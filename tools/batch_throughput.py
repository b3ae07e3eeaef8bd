"""Throughput of batches (mtb_render_batch) against one call per frame, on the C3 scene (two lights, depth 5) and its
orbit yaw = C3 yaw + 2 degrees * k.

    python tools/batch_throughput.py [--devices 0[,1,..]] [--out FILE] [--reps 3]

480x270, 64 frames: (a) one render_chunk per frame, megakernel forced; (b) one render_chunk per frame, automatic
pipeline choice (after the 13 frames it needs to decide); (c) render_batch in batches of 1, 4, 16, 64.
1920x1080, 8 frames: one render_chunk per frame against one batch of 8; 960x540, 32 frames, likewise.
Then the work per ray of each size from the counting build (box tests and triangle tests per ray; not timed).
With several devices also: a 64-frame batch on all of them against per-frame strip rendering on the same devices.

Per mode: frames/s from a host clock around the synchronous calls (median of --reps passes), summed kernel_ms (CUDA
events of each call), Mrays/s (rays / summed kernel time) and the SHA-256 of every frame; every mode of one shape must
give the same frames.  Every shape is warmed up before it is timed.  The card's name, power limit and max SM clock
are read in the same run.  Prints one JSON document (and writes it to --out).
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


def _group(title, w, h, recs):
    first = recs[0]["frame_sha256"]
    same = all(r["frame_sha256"] == first for r in recs)
    return dict(shape=title, width=w, height=h, frames_identical_across_modes=same, modes=recs)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--devices", default="0")
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    devices = [int(x) for x in args.devices.split(",")]
    files, cfg = scenegen.generate_config("C3", os.environ.get("MTB_SCENE_DIR", "/tmp/mtb_scenes"))
    depth = cfg["depth"]
    doc = dict(tool="tools/batch_throughput.py", scene="C3", triangles=files.n_triangles, lights=len(files.lights), depth=depth,
               card=_card(), reps=args.reps, groups=[])

    mt = MythTracer(devices=devices[:1], max_depth=depth, flags=MTB_FLAG_MEGAKERNEL)
    assert mt.LoadObj(files.obj_path), mt.last_error()
    mt.GetScene().lights = [Light.from_tuple(l) for l in files.lights]

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
