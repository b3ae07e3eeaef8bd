"""Throughput of batches (mtb_render_batch) against one call per frame, on the C3 scene (two lights, depth 5) and its
orbit yaw = C3 yaw + 2 degrees * k.

    python tools/batch_throughput.py [--devices 0[,1,..]] [--out FILE] [--reps 3]
                                     [--supersample | --debug-planes | --subframes | --device-output | --lens | --panorama]

480x270, 64 frames: (a) one render_chunk per frame, megakernel forced; (b) one render_chunk per frame, automatic
pipeline choice (after the 13 frames it needs to decide); (c) render_batch in batches of 1, 4, 16, 64.
1920x1080, 8 frames: one render_chunk per frame against one batch of 8; 960x540, 32 frames, likewise.
Then the work per ray of each size from the counting build (box tests and triangle tests per ray; not timed).
With several devices also: a 64-frame batch on all of them against per-frame strip rendering on the same devices.

Per mode: frames/s from a host clock around the synchronous calls (median of --reps passes), summed kernel_ms (CUDA
events of each call), Mrays/s (rays / summed kernel time) and the SHA-256 of every frame; every mode of one shape must
give the same frames.  Every shape is warmed up before it is timed.  The card's name, power limit and max SM clock
are read in the same run.  Prints one JSON document (and writes it to --out).

--supersample measures supersampled batches instead (render_batch(..., samples_per_axis=s)), 16 views of the orbit:
1920x1080 plain (the rays of every row below), 960x540 with s = 2, 480x270 with s = 4, 240x135 with s = 8, and plain
480x270 (the same output with 16x fewer rays).  Each s is also rendered the way a caller has to without it: render_batch
at s*W x s*H plus the block mean in numpy (frames/s end to end).  Per mode: median kernel_ms per call over --reps calls,
Mrays/s, frames/s, and whether every view equals the block mean of the 1920x1080 views.  Then the work per ray of each
mode from the counting build (not timed).

--debug-planes measures batches that also return per-pixel planes (render_batch(..., debug=True / taps=True)): 64 C3
views at 480x270 and 8 at 1920x1080, each with neither, with debug, with taps and with both, against one
render_chunk(debug=True) per frame (megakernel).  Per mode: median kernel_ms per call (summed over the calls of a
pass for render_chunk), frames/s end to end, Mrays/s and the bytes copied back per view; whether the RGB equals that of
the batch without planes, and whether the planes of the first and the last view equal render_chunk's.

--subframes measures accumulated batches (render_batch(..., subframes=k)): output view f of the orbit is the mean of k
sub-frames at yaw + 2 degrees * (f + j / k).  Shapes: 16 outputs x k = 8 at 480x270 (s = 1), 4 x k = 4 at 1920x1080
(s = 1) and 16 x k = 4 at 480x270 with s = 4.  Each against the plain batch of the same sub-frames at the same s (the
same rays; kernel time), and against the way a caller has to do it without the feature: render_batch of the sub-frames
at s*W x s*H plus the mean in numpy (frames/s end to end).  Per mode: median kernel_ms per call over --reps calls,
Mrays/s, output frames/s, and whether the output equals the numpy mean of the sub-frames.

--device-output measures batches that leave their outputs in device memory (render_batch(..., device=True),
mtb_render_batch_device) against the same batch into host memory: 64 views at 480x270; the same with debug and taps;
16 views at 480x270 with s = 4; 4 outputs x k = 4 sub-frames at 1920x1080.  Per row: frames/s end to end of both forms
(median of --reps calls; the host form is synchronous, the device form is timed with a host clock around the call and
torch.cuda.synchronize()), the median kernel_ms per call of both (CUDA events of the library: the device form's come from
mtb_render_batch_device called with stats, in calls of their own), the bytes the host form copies back per output, and
whether the device outputs, copied back, equal the host outputs byte for byte (RGB and every plane).

--lens measures thin-lens batches (render_batch(..., lenses=...), mtb_render_batch_lens): 16 outputs x k = 8 at 480x270
and 4 x k = 4 at 1920x1080, both on the orbit sub-frames of --subframes.  Three modes per shape, timed in turn in every
pass: the accumulated batch without lenses; the same with centred lens samples (0, 0, f), which trace the same rays
(its output must equal the first's); and a disc aperture (seeded concentric-disc samples of radius 4 focused at 150),
which traces different rays.  Per mode: median kernel_ms per call over --reps passes, Mrays/s, output frames/s, and the
kernel time over that of the batch without lenses.

--panorama measures panorama batches (render_batch(..., panorama=(360, 180)), mtb_render_batch_pano) against pinhole
batches of the same primary-ray count (same views, grid and s): 8 equirectangular C3 panoramas of the orbit at
4096x2048; an omni-directional stereo pair from the C3 camera at 4096x2048 (eye offsets -/+0.032 x the scene's
diagonal); 16 panoramas of the orbit at 1024x512 with s = 2.  Pinhole and panorama are timed in turn in every pass.  Per
mode: median kernel_ms per call over --reps passes, Mrays/s, output frames/s, and the kernel time over the pinhole's.
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

from mythtracer_b200 import MTB_FLAG_COUNT_WORK, MTB_FLAG_MEGAKERNEL, Light, MythTracer, scenegen  # noqa: E402


def _card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()
        return out
    except Exception as e:  # (the numbers below are still device-timed; the card is then unknown)
        return ["nvidia-smi failed: %s" % e]


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _orbit(cam, n):
    out = []
    for k in range(n):
        c = list(cam)
        c[4] += 2.0 * k
        out.append(tuple(c))
    return out


def _singles(mt, cams, w, h, reps):
    """One synchronous render_chunk per frame."""
    buf = np.zeros((h, w, 3), np.uint8)
    walls, kernel_ms, rays, shas = [], 0.0, 0, []
    for rep in range(reps):
        kms, nr, hs = 0.0, 0, []
        t0 = time.perf_counter()
        for cam in cams:
            r = mt.render_chunk(cam, w, h, 0, 0, w, h, out=buf)
            kms += r["stats"]["kernel_ms"]
            nr += r["stats"]["rays"]
            if rep == 0:
                hs.append(_sha(buf))
        walls.append(time.perf_counter() - t0)
        if rep == 0:
            kernel_ms, rays, shas = kms, nr, hs
    return walls, kernel_ms, rays, shas


def _batches(mt, cams, w, h, per_call, reps):
    """render_batch in calls of `per_call` views (the last one may be partial)."""
    buf = np.zeros((per_call, h, w, 3), np.uint8)
    walls, kernel_ms, rays, shas = [], 0.0, 0, []
    for rep in range(reps):
        kms, nr, hs = 0.0, 0, []
        t0 = time.perf_counter()
        for b in range(0, len(cams), per_call):
            part = cams[b:b + per_call]
            out = buf if len(part) == per_call else np.zeros((len(part), h, w, 3), np.uint8)
            r = mt.render_batch(part, w, h, out=out)
            kms += r["stats"]["kernel_ms"]
            nr += r["stats"]["rays"]
            if rep == 0:
                hs.extend(_sha(out[v]) for v in range(len(part)))
        walls.append(time.perf_counter() - t0)
        if rep == 0:
            kernel_ms, rays, shas = kms, nr, hs
    return walls, kernel_ms, rays, shas


def _record(name, n_frames, res):
    walls, kernel_ms, rays, shas = res
    wall = statistics.median(walls)
    rec = dict(mode=name, frames=n_frames, frames_per_s=round(n_frames / wall, 1), wall_s_all=[round(x, 4) for x in walls],
               kernel_ms_sum=round(kernel_ms, 3), rays=rays, mrays_per_s=round(rays / kernel_ms / 1e3, 1) if kernel_ms > 0 else None,
               frame_sha256=shas)
    print("%-34s %5d frames  %8.1f frames/s  kernel %9.3f ms  %8.1f Mrays/s" % (name, n_frames, rec["frames_per_s"], kernel_ms,
                                                                           rec["mrays_per_s"] or 0.0), file=sys.stderr, flush=True)
    return rec


def _block_mean(frames, s):
    f = frames.astype(np.uint32)
    h, w = f.shape[-3] // s, f.shape[-2] // s
    blocks = f.reshape(f.shape[:-3] + (h, s, w, s, 3)).sum(axis=(-4, -2))
    return ((blocks + s * s // 2) // (s * s)).astype(np.uint8)


def _timed_calls(fn, reps):
    """fn() -> stats of one synchronous call; wall and kernel time of each of `reps` calls after one warm-up call."""
    fn()
    walls, kms = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        st = fn()
        walls.append(time.perf_counter() - t0)
        kms.append(st["kernel_ms"])
    return walls, kms, st["rays"]


def _ss_record(name, n_frames, w, h, s, walls, kms, rays, equal, base_kernel_ms=None):
    wall, kms_med = statistics.median(walls), statistics.median(kms)
    rec = dict(mode=name, width=w, height=h, samples_per_axis=s, frames=n_frames, frames_per_s=round(n_frames / wall, 1),
               wall_s_all=[round(x, 4) for x in walls], kernel_ms=round(kms_med, 3), kernel_ms_all=[round(x, 3) for x in kms], rays=rays,
               mrays_per_s=round(rays / kms_med / 1e3, 1) if kms_med > 0 else None, equals_block_mean_of_1080p=equal)
    if base_kernel_ms:
        rec["kernel_ms_over_1080p_batch"] = round(kms_med / base_kernel_ms, 4)
    print("%-42s %8.1f frames/s  kernel %8.3f ms  %8.1f Mrays/s  %s" % (name, rec["frames_per_s"], kms_med, rec["mrays_per_s"] or 0.0,
                                                                     "" if base_kernel_ms is None else "x%.4f of 1080p" % (kms_med / base_kernel_ms)),
          file=sys.stderr, flush=True)
    return rec


def supersample(mt, files, cfg, reps):
    """The --supersample measurements (see the module docstring)."""
    n = 16
    W, H = cfg["width"], cfg["height"]
    cams = _orbit(files.camera, n)
    hi = np.zeros((n, H, W, 3), np.uint8)
    walls, kms, rays = _timed_calls(lambda: mt.render_batch(cams, W, H, out=hi)["stats"], reps)
    hi_frames = hi.copy()
    base = statistics.median(kms)
    recs = [_ss_record("render_batch %dx%d" % (W, H), n, W, H, 1, walls, kms, rays, True)]
    for s in (2, 4, 8):
        w, h = W // s, H // s
        out = np.zeros((n, h, w, 3), np.uint8)
        walls, kms, rays = _timed_calls(lambda: mt.render_batch(cams, w, h, out=out, samples_per_axis=s)["stats"], reps)
        equal = bool(np.array_equal(out, _block_mean(hi_frames, s)))
        recs.append(_ss_record("render_batch %dx%d, %d samples per axis" % (w, h, s), n, w, h, s, walls, kms, rays, equal, base))

        def hi_then_mean():
            st = mt.render_batch(cams, W, H, out=hi)["stats"]
            out[...] = _block_mean(hi, s)
            return st
        walls, kms, rays = _timed_calls(hi_then_mean, reps)
        equal = bool(np.array_equal(out, _block_mean(hi_frames, s)))
        recs.append(_ss_record("render_batch %dx%d + numpy block mean to %dx%d" % (W, H, w, h), n, w, h, s, walls, kms, rays, equal, base))
    w, h = W // 4, H // 4
    out = np.zeros((n, h, w, 3), np.uint8)
    walls, kms, rays = _timed_calls(lambda: mt.render_batch(cams, w, h, out=out)["stats"], reps)
    recs.append(_ss_record("render_batch %dx%d, one ray per pixel" % (w, h), n, w, h, 1, walls, kms, rays, None, base))

    mt.set_flags(MTB_FLAG_MEGAKERNEL | MTB_FLAG_COUNT_WORK)
    work = []
    for (ww, hh, s) in ((W, H, 1), (W // 2, H // 2, 2), (W // 4, H // 4, 4), (W // 8, H // 8, 8), (W // 4, H // 4, 1)):
        st = mt.render_batch(cams, ww, hh, samples_per_axis=s)["stats"]
        work.append(dict(width=ww, height=hh, samples_per_axis=s, views=n, rays_per_sample=round(st["rays"] / (n * ww * hh * s * s), 3),
                         bvh_box_tests_per_ray=round(st["n_bvh"] / st["rays"], 2), triangle_tests_per_ray=round(st["n_mt"] / st["rays"], 2),
                         rays_over_512_visits=st["n_long512_rays"]))
        print(json.dumps(work[-1]), file=sys.stderr, flush=True)
    mt.set_flags(MTB_FLAG_MEGAKERNEL)
    return dict(shape="C3 orbit, %d views" % n, modes=recs, work_per_ray=work)


def _accum_mean(frames, k, s):
    """(n_out * k, s*H, s*W, 3) -> (n_out, H, W, 3): the rounded mean of the k * s * s samples of every output channel."""
    n_out, sh, sw = frames.shape[0] // k, frames.shape[1], frames.shape[2]
    sums = frames.reshape(n_out, k, sh // s, s, sw // s, s, 3).sum(axis=(1, 3, 5), dtype=np.uint32)
    n = k * s * s
    return ((sums + n // 2) // n).astype(np.uint8)


def subframes(mt, files, cfg, reps):
    """The --subframes measurements (see the module docstring)."""
    groups = []
    for n_out, k, w, h, s in ((16, 8, 480, 270, 1), (4, 4, cfg["width"], cfg["height"], 1), (16, 4, 480, 270, 4)):
        cams = [c for f in range(n_out) for c in _orbit_subframes(files.camera, f, k)]
        out = np.zeros((n_out, h, w, 3), np.uint8)
        walls, kms, rays = _timed_calls(lambda: mt.render_batch(cams, w, h, out=out, samples_per_axis=s, subframes=k)["stats"], reps)
        got = out.copy()
        hi = np.zeros((n_out * k, s * h, s * w, 3), np.uint8)
        mt.render_batch(cams, s * w, s * h, out=hi)
        want = _accum_mean(hi, k, s)
        equal = bool(np.array_equal(got, want))
        recs = [_ss_record("render_batch %d x %d subframes, %dx%d, s = %d" % (n_out, k, w, h, s), n_out, w, h, s, walls, kms, rays, equal)]
        plain = np.zeros((n_out * k, h, w, 3), np.uint8)
        walls, kms_p, rays_p = _timed_calls(lambda: mt.render_batch(cams, w, h, out=plain, samples_per_axis=s)["stats"], reps)
        base_kms = statistics.median(kms_p)
        recs.append(_ss_record("render_batch %d views (the sub-frames), %dx%d, s = %d" % (n_out * k, w, h, s), n_out * k, w, h, s, walls, kms_p,
                               rays_p, None))

        def hi_then_mean():
            st = mt.render_batch(cams, s * w, s * h, out=hi)["stats"]
            out[...] = _accum_mean(hi, k, s)
            return st
        walls, kms_h, rays_h = _timed_calls(hi_then_mean, reps)
        recs.append(_ss_record("render_batch %d views at %dx%d + numpy mean" % (n_out * k, s * w, s * h), n_out, w, h, s, walls, kms_h, rays_h,
                               bool(np.array_equal(out, want))))
        for r in recs:
            r["equals_numpy_mean"] = r.pop("equals_block_mean_of_1080p")
        recs[0]["kernel_ms_over_plain_batch"] = round(statistics.median(kms) / base_kms, 4)
        print("accumulated / plain kernel time: x%.4f" % recs[0]["kernel_ms_over_plain_batch"], file=sys.stderr, flush=True)
        groups.append(dict(shape="C3 orbit, %d outputs x %d subframes at %dx%d, %d samples per axis" % (n_out, k, w, h, s), outputs=n_out,
                           subframes=k, modes=recs))
    return groups


def _disc_lenses(n, radius, focus, seed):
    """n seeded thin-lens samples (u, v, focus) on a disc of `radius` (Shirley-Chiu concentric mapping)."""
    out = []
    for a, b in 2.0 * np.random.default_rng(seed).random((n, 2)) - 1.0:
        if abs(a) > abs(b):
            r, phi = a, np.pi / 4 * (b / a)
        elif b != 0.0:
            r, phi = b, np.pi / 2 - np.pi / 4 * (a / b)
        else:
            r, phi = 0.0, 0.0
        out.append((radius * r * np.cos(phi), radius * r * np.sin(phi), focus))
    return np.array(out)


def lens(mt, files, cfg, reps):
    """The --lens measurements (see the module docstring)."""
    groups = []
    for n_out, k, w, h in ((16, 8, 480, 270), (4, 4, cfg["width"], cfg["height"])):
        cams = [c for f in range(n_out) for c in _orbit_subframes(files.camera, f, k)]
        modes = (("render_batch %d x %d subframes, no lenses" % (n_out, k), None),
                 ("render_batch %d x %d subframes, centred lens samples" % (n_out, k), np.array([(0.0, 0.0, 150.0)] * len(cams))),
                 ("render_batch %d x %d subframes, disc aperture r = 4, focus 150" % (n_out, k), _disc_lenses(len(cams), 4.0, 150.0, 7)))
        outs = [np.zeros((n_out, h, w, 3), np.uint8) for _ in modes]
        call = [lambda i=i: mt.render_batch(cams, w, h, out=outs[i], subframes=k, lenses=modes[i][1])["stats"] for i in range(len(modes))]
        for c in call:
            c()  # warm-up of this shape
        walls, kms, rays = [[] for _ in modes], [[] for _ in modes], [0] * len(modes)
        for _ in range(reps):  # the modes alternate within every pass
            for i, c in enumerate(call):
                t0 = time.perf_counter()
                st = c()
                walls[i].append(time.perf_counter() - t0)
                kms[i].append(st["kernel_ms"])
                rays[i] = st["rays"]
        base = statistics.median(kms[0])
        recs = []
        for i, (name, _) in enumerate(modes):
            rec = _ss_record(name, n_out, w, h, 1, walls[i], kms[i], rays[i], None)
            rec.pop("equals_block_mean_of_1080p")
            rec["kernel_ms_over_no_lenses"] = round(statistics.median(kms[i]) / base, 4)
            recs.append(rec)
        recs[1]["equals_no_lenses"] = bool(np.array_equal(outs[1], outs[0]))
        recs[2]["differs_from_no_lenses"] = not np.array_equal(outs[2], outs[0])
        print("centred / no lenses kernel time: x%.4f, disc / no lenses: x%.4f" % (recs[1]["kernel_ms_over_no_lenses"],
                                                                                 recs[2]["kernel_ms_over_no_lenses"]), file=sys.stderr, flush=True)
        groups.append(dict(shape="C3 orbit, %d outputs x %d subframes at %dx%d" % (n_out, k, w, h), outputs=n_out, subframes=k, modes=recs))
    return groups


def panorama(mt, files, cfg, reps):
    """The --panorama measurements (see the module docstring)."""
    box = mt.scene_info()
    scale = float(np.linalg.norm(np.array(box["aabb_max"]) - np.array(box["aabb_min"])))
    groups = []
    for title, n, w, h, s, eyes in (("8 equirectangular panoramas", 8, 4096, 2048, 1, None),
                                    ("ODS stereo pair, e = -/+0.032 x scene diagonal", 2, 4096, 2048, 1, [-0.032 * scale, 0.032 * scale]),
                                    ("16 panoramas, s = 2", 16, 1024, 512, 2, None)):
        cams = _orbit(files.camera, n) if eyes is None else [files.camera] * n
        modes = (("pinhole batch", {}), ("panorama 360 x 180", dict(panorama=(360.0, 180.0), eye_offsets=eyes)))
        outs = [np.zeros((n, h, w, 3), np.uint8) for _ in modes]
        call = [lambda i=i: mt.render_batch(cams, w, h, out=outs[i], samples_per_axis=s, **modes[i][1])["stats"] for i in range(len(modes))]
        for c in call:
            c()  # warm-up of this shape
        walls, kms, rays = [[] for _ in modes], [[] for _ in modes], [0] * len(modes)
        for _ in range(reps):  # the modes alternate within every pass
            for i, c in enumerate(call):
                t0 = time.perf_counter()
                st = c()
                walls[i].append(time.perf_counter() - t0)
                kms[i].append(st["kernel_ms"])
                rays[i] = st["rays"]
        base = statistics.median(kms[0])
        recs = []
        for i, (name, _) in enumerate(modes):
            rec = _ss_record(name, n, w, h, s, walls[i], kms[i], rays[i], None)
            rec.pop("equals_block_mean_of_1080p")
            rec["primary_rays"] = n * w * h * s * s
            rec["kernel_ms_over_pinhole"] = round(statistics.median(kms[i]) / base, 4)
            recs.append(rec)
        recs[1]["differs_from_pinhole"] = not np.array_equal(outs[1], outs[0])
        if eyes is not None:
            recs[1]["eyes_differ"] = not np.array_equal(outs[1][0], outs[1][1])
        print("%s: panorama / pinhole kernel time x%.4f" % (title, recs[1]["kernel_ms_over_pinhole"]), file=sys.stderr, flush=True)
        groups.append(dict(shape="C3, %s at %dx%d" % (title, w, h), views=n, samples_per_axis=s, eye_offsets=eyes, modes=recs))
    return groups


def _orbit_subframes(cam, f, k):
    """The k sub-frames of output frame f of the orbit: yaw + 2 degrees * (f + j / k)."""
    out = []
    for j in range(k):
        c = list(cam)
        c[4] += 2.0 * f + 2.0 * j / k
        out.append(tuple(c))
    return out


PLANE_KEYS = ("debug", "sig_hits", "sig_shadow", "n_rays")


def _walls(fn, reps):
    """Host wall time of each of `reps` calls of fn() after one warm-up call."""
    fn()
    walls = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        walls.append(time.perf_counter() - t0)
    return walls


def _device_kernel_ms(mt, cams, n_out, k, w, h, s, planes, reps):
    """kernel_ms of mtb_render_batch_device with stats (the call then waits for its batch), into fresh CUDA tensors, on
    the context's lights: median over `reps` calls after one warm-up call."""
    import ctypes

    import torch

    from mythtracer_b200 import api
    cam_arr = np.zeros(len(cams), api.CAMERA_DTYPE)
    for i, c in enumerate(cams):
        cam_arr[i] = api.Camera.from_tuple(c).as_array()
    rgb = torch.empty((n_out, h, w, 3), dtype=torch.uint8, device="cuda:%d" % mt._device0)
    plane = len(cams) * s * s * w * h
    dbg = torch.empty(plane * 32 if planes else 0, dtype=torch.uint8, device=rgb.device)
    tap = torch.empty(plane * 20 if planes else 0, dtype=torch.uint8, device=rgb.device)
    taps = api._TapsStruct(tap.data_ptr(), tap.data_ptr() + 8 * plane, tap.data_ptr() + 16 * plane) if planes else None
    stats = np.zeros((), api.STATS_DTYPE)
    kms = []
    for rep in range(reps + 1):
        rc = mt._lib.mtb_render_batch_device(mt._ctx, cam_arr.ctypes.data_as(ctypes.c_void_p), n_out, k, None, 0, w, h, s, mt.max_depth,
                                             ctypes.c_void_p(rgb.data_ptr()), ctypes.c_void_p(dbg.data_ptr()) if planes else None,
                                             ctypes.cast(ctypes.pointer(taps), ctypes.c_void_p) if planes else None, None,
                                             stats.ctypes.data_as(ctypes.c_void_p))
        mt._check(rc, "mtb_render_batch_device")
        if rep > 0:
            kms.append(float(stats["kernel_ms"]))
    return kms


def device_output(mt, files, cfg, reps):
    """The --device-output measurements (see the module docstring)."""
    import torch
    rows = []
    W, H = cfg["width"], cfg["height"]
    for n_out, k, w, h, s, planes in ((64, 1, 480, 270, 1, False), (64, 1, 480, 270, 1, True), (16, 1, 480, 270, 4, False),
                                      (4, 4, W, H, 1, False)):
        cams = [c for f in range(n_out) for c in _orbit_subframes(files.camera, f, k)]
        kw = dict(samples_per_axis=s, subframes=k, debug=planes, taps=planes)
        host, dev = {}, {}

        def host_call():
            host.update(mt.render_batch(cams, w, h, **kw))
            return host["stats"]
        walls_h, kms_h, rays = _timed_calls(host_call, reps)

        def device_call():
            dev.update(mt.render_batch(cams, w, h, device=True, **kw))
            torch.cuda.synchronize()
        walls_d = _walls(device_call, reps)
        kms_d = _device_kernel_ms(mt, cams, n_out, k, w, h, s, planes, reps)
        equal = bool(np.array_equal(dev["rgb"].cpu().numpy(), host["rgb"]))
        if planes:
            equal &= dev["debug"].cpu().numpy().tobytes() == host["debug"].tobytes()
            equal &= all(np.array_equal(dev[key].cpu().numpy(), host[key]) for key in ("sig_hits", "sig_shadow", "n_rays"))
        wh, wd = statistics.median(walls_h), statistics.median(walls_d)
        name = "%d x %dx%d, s = %d%s%s" % (n_out, w, h, s, ", k = %d" % k if k > 1 else "", ", debug + taps" if planes else "")
        rec = dict(mode=name, outputs=n_out, subframes=k, width=w, height=h, samples_per_axis=s, debug=planes, taps=planes, rays=rays,
                   host_frames_per_s=round(n_out / wh, 1), device_frames_per_s=round(n_out / wd, 1),
                   host_kernel_ms=round(statistics.median(kms_h), 3), device_kernel_ms=round(statistics.median(kms_d), 3),
                   host_wall_s_all=[round(x, 4) for x in walls_h], device_wall_s_all=[round(x, 4) for x in walls_d],
                   host_kernel_ms_all=[round(x, 3) for x in kms_h], device_kernel_ms_all=[round(x, 3) for x in kms_d],
                   host_bytes_copied_per_output=w * h * 3 + (k * s * s * w * h * (32 + 20) if planes else 0), device_equals_host=equal)
        print("%-40s host %8.1f frames/s  device %8.1f frames/s  kernel %8.3f / %8.3f ms  %s" % (
            name, rec["host_frames_per_s"], rec["device_frames_per_s"], rec["host_kernel_ms"], rec["device_kernel_ms"],
            "equal" if equal else "DIFFERENT"), file=sys.stderr, flush=True)
        rows.append(rec)
        host.clear()
        dev.clear()
    return rows


def debug_planes(mt, files, cfg, reps):
    """The --debug-planes measurements (see the module docstring)."""
    groups = []
    for w, h, n in ((480, 270, 64), (cfg["width"], cfg["height"], 8)):
        cams = _orbit(files.camera, n)
        recs, rgb0 = [], None
        for debug, taps in ((False, False), (True, False), (False, True), (True, True)):
            last = {}

            def call():
                last.update(mt.render_batch(cams, w, h, debug=debug, taps=taps))
                return last["stats"]
            walls, kms, rays = _timed_calls(call, reps)
            if rgb0 is None:
                rgb0 = last["rgb"].copy()
            per_view = w * h * (3 + (32 if debug else 0) + (20 if taps else 0))
            name = "render_batch %d x %dx%d, %s" % (n, w, h, {(False, False): "no planes", (True, False): "debug", (False, True): "taps",
                                                           (True, True): "debug + taps"}[(debug, taps)])
            rec = _ss_record(name, n, w, h, 1, walls, kms, rays, None)
            del rec["equals_block_mean_of_1080p"]
            rec.update(debug=debug, taps=taps, bytes_copied_per_view=per_view, rgb_equals_no_planes=bool(np.array_equal(last["rgb"], rgb0)))
            if debug or taps:
                same = True
                for v in (0, n - 1):
                    single = mt.render_chunk(cams[v], w, h, 0, 0, w, h, debug=True, taps=True)
                    same &= all(last[k][v].tobytes() == single[k].tobytes() for k in PLANE_KEYS if k in last)
                rec["planes_equal_render_chunk"] = bool(same)
            recs.append(rec)

        def singles():
            kms, nr = 0.0, 0
            for cam in cams:
                st = mt.render_chunk(cam, w, h, 0, 0, w, h, debug=True)["stats"]
                kms += st["kernel_ms"]
                nr += st["rays"]
            return dict(kernel_ms=kms, rays=nr)
        walls, kms, rays = _timed_calls(singles, reps)
        rec = _ss_record("render_chunk(debug=True) x %d, %dx%d" % (n, w, h), n, w, h, 1, walls, kms, rays, None)
        del rec["equals_block_mean_of_1080p"]
        rec.update(debug=True, taps=False, bytes_copied_per_view=w * h * (3 + 32))
        recs.append(rec)
        groups.append(dict(shape="C3 orbit, %d views at %dx%d" % (n, w, h), modes=recs))
    return groups


def _group(title, w, h, recs):
    first = recs[0]["frame_sha256"]
    same = all(r["frame_sha256"] == first for r in recs)
    return dict(shape=title, width=w, height=h, frames_identical_across_modes=same, modes=recs)


def _emit(doc, out):
    text = json.dumps(doc, indent=1)
    print(text)
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            f.write(text + "\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--devices", default="0")
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--supersample", action="store_true")
    ap.add_argument("--debug-planes", action="store_true")
    ap.add_argument("--subframes", action="store_true")
    ap.add_argument("--device-output", action="store_true")
    ap.add_argument("--lens", action="store_true")
    ap.add_argument("--panorama", action="store_true")
    args = ap.parse_args()
    devices = [int(x) for x in args.devices.split(",")]
    files, cfg = scenegen.generate_config("C3", os.environ.get("MTB_SCENE_DIR", "/tmp/mtb_scenes"))
    depth = cfg["depth"]
    doc = dict(tool="tools/batch_throughput.py", scene="C3", triangles=files.n_triangles, lights=len(files.lights), depth=depth,
               card=_card(), reps=args.reps, groups=[])

    mt = MythTracer(devices=devices[:1], max_depth=depth, flags=MTB_FLAG_MEGAKERNEL)
    assert mt.LoadObj(files.obj_path), mt.last_error()
    mt.GetScene().lights = [Light.from_tuple(l) for l in files.lights]

    if args.debug_planes:
        doc["debug_planes"] = debug_planes(mt, files, cfg, args.reps)
        mt.close()
        _emit(doc, args.out)
        modes = [r for g in doc["debug_planes"] for r in g["modes"]]
        if not all(r.get("rgb_equals_no_planes", True) and r.get("planes_equal_render_chunk", True) for r in modes):
            sys.exit("a batch with planes differs from the batch without planes or from render_chunk")
        return

    if args.device_output:
        doc["device_output"] = device_output(mt, files, cfg, args.reps)
        mt.close()
        _emit(doc, args.out)
        if not all(r["device_equals_host"] for r in doc["device_output"]):
            sys.exit("a batch into device memory differs from the same batch into host memory")
        return

    if args.lens:
        doc["lens"] = lens(mt, files, cfg, args.reps)
        mt.close()
        _emit(doc, args.out)
        if not all(g["modes"][1]["equals_no_lenses"] for g in doc["lens"]):
            sys.exit("centred lens samples differ from the batch without lenses")
        return

    if args.panorama:
        doc["panorama"] = panorama(mt, files, cfg, args.reps)
        mt.close()
        _emit(doc, args.out)
        if not all(g["modes"][1]["differs_from_pinhole"] and g["modes"][1].get("eyes_differ", True) for g in doc["panorama"]):
            sys.exit("a panorama gave the pinhole frames, or both eyes gave the same frame")
        return

    if args.subframes:
        doc["subframes"] = subframes(mt, files, cfg, args.reps)
        mt.close()
        _emit(doc, args.out)
        if not all(r["equals_numpy_mean"] is not False for g in doc["subframes"] for r in g["modes"]):
            sys.exit("an accumulated batch differs from the numpy mean of its sub-frames")
        return

    if args.supersample:
        doc["supersample"] = supersample(mt, files, cfg, args.reps)
        mt.close()
        _emit(doc, args.out)
        if not all(r["equals_block_mean_of_1080p"] is not False for r in doc["supersample"]["modes"]):
            sys.exit("a supersampled mode differs from the block means of the 1080p views")
        return

    # ---- 480x270, 64 frames ----
    w, h = 480, 270
    cams = _orbit(files.camera, 64)
    recs = []
    mt.set_flags(MTB_FLAG_MEGAKERNEL)
    _singles(mt, cams[:4], w, h, 1)  # warm-up
    recs.append(_record("(a) render_chunk, megakernel", 64, _singles(mt, cams, w, h, args.reps)))
    mt.set_flags(0)
    _singles(mt, cams[:14], w, h, 1)  # the automatic choice decides on frame 13 of a geometry
    auto = _record("(b) render_chunk, automatic", 64, _singles(mt, cams, w, h, args.reps))
    auto["pipeline"] = mt.pipeline_in_use()[0]
    recs.append(auto)
    mt.set_flags(MTB_FLAG_MEGAKERNEL)
    for n in (1, 4, 16, 64):
        _batches(mt, cams[:n], w, h, n, 1)  # warm-up of this shape
        recs.append(_record("(c) render_batch, %d per call" % n, 64, _batches(mt, cams, w, h, n, args.reps)))
    doc["groups"].append(_group("480x270 x 64", w, h, recs))

    # ---- 1920x1080, 8 frames ----
    W, H = cfg["width"], cfg["height"]
    cams8 = _orbit(files.camera, 8)
    _singles(mt, cams8[:1], W, H, 1)
    _batches(mt, cams8, W, H, 8, 1)
    recs = [_record("render_chunk, megakernel", 8, _singles(mt, cams8, W, H, args.reps)),
            _record("render_batch, 8 per call", 8, _batches(mt, cams8, W, H, 8, args.reps))]
    doc["groups"].append(_group("1920x1080 x 8", W, H, recs))

    # ---- between the two: 960x540, 32 frames ----
    cams32 = _orbit(files.camera, 32)
    _singles(mt, cams32[:2], 960, 540, 1)
    _batches(mt, cams32, 960, 540, 32, 1)
    recs = [_record("render_chunk, megakernel", 32, _singles(mt, cams32, 960, 540, args.reps)),
            _record("render_batch, 32 per call", 32, _batches(mt, cams32, 960, 540, 32, args.reps))]
    doc["groups"].append(_group("960x540 x 32", 960, 540, recs))

    # ---- work per ray by resolution (counting build of the kernels; not timed) ----
    mt.set_flags(MTB_FLAG_MEGAKERNEL | MTB_FLAG_COUNT_WORK)
    work = []
    for (ww, hh, n) in ((480, 270, 64), (960, 540, 32), (W, H, 8)):
        s = mt.render_batch(_orbit(files.camera, n), ww, hh)["stats"]
        work.append(dict(width=ww, height=hh, views=n, rays_per_pixel=round(s["rays"] / (n * ww * hh), 3),
                         bvh_box_tests_per_ray=round(s["n_bvh"] / s["rays"], 2), triangle_tests_per_ray=round(s["n_mt"] / s["rays"], 2),
                         rays_over_512_visits=s["n_long512_rays"]))
        print(json.dumps(work[-1]), file=sys.stderr, flush=True)
    doc["work_per_ray"] = work
    mt.close()

    # ---- several devices: whole views per device against strips of every frame ----
    if len(devices) > 1:
        many = MythTracer(devices=devices, max_depth=depth, flags=MTB_FLAG_MEGAKERNEL)
        assert many.LoadObj(files.obj_path), many.last_error()
        many.GetScene().lights = [Light.from_tuple(l) for l in files.lights]
        _singles(many, cams[:4], w, h, 1)
        _batches(many, cams, w, h, 64, 1)
        recs = [_record("render_chunk strips, %d devices" % len(devices), 64, _singles(many, cams, w, h, args.reps)),
                _record("render_batch 64, %d devices" % len(devices), 64, _batches(many, cams, w, h, 64, args.reps))]
        doc["groups"].append(_group("480x270 x 64 on devices %s" % args.devices, w, h, recs))
        many.close()

    _emit(doc, args.out)
    if not all(g["frames_identical_across_modes"] for g in doc["groups"]):
        sys.exit("frames differ between modes")


if __name__ == "__main__":
    main()
