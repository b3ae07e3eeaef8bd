"""Throughput of batches (mtb_render_batch) against one call per frame, on the C3 scene (two lights, depth 5) and its
orbit yaw = C3 yaw + 2 degrees * k.

    python tools/batch_throughput.py [--devices 0[,1,..]] [--out FILE] [--reps 3] [--supersample]

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


def _group(title, w, h, recs):
    first = recs[0]["frame_sha256"]
    same = all(r["frame_sha256"] == first for r in recs)
    return dict(shape=title, width=w, height=h, frames_identical_across_modes=same, modes=recs)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--devices", default="0")
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--supersample", action="store_true")
    args = ap.parse_args()
    devices = [int(x) for x in args.devices.split(",")]
    files, cfg = scenegen.generate_config("C3", os.environ.get("MTB_SCENE_DIR", "/tmp/mtb_scenes"))
    depth = cfg["depth"]
    doc = dict(tool="tools/batch_throughput.py", scene="C3", triangles=files.n_triangles, lights=len(files.lights), depth=depth,
               card=_card(), reps=args.reps, groups=[])

    mt = MythTracer(devices=devices[:1], max_depth=depth, flags=MTB_FLAG_MEGAKERNEL)
    assert mt.LoadObj(files.obj_path), mt.last_error()
    mt.GetScene().lights = [Light.from_tuple(l) for l in files.lights]

    if args.supersample:
        doc["supersample"] = supersample(mt, files, cfg, args.reps)
        mt.close()
        text = json.dumps(doc, indent=1)
        print(text)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(text + "\n")
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

    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    if not all(g["frames_identical_across_modes"] for g in doc["groups"]):
        sys.exit("frames differ between modes")


if __name__ == "__main__":
    main()
