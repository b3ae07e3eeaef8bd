"""Quick device timing of the BASELINE configs (development aid; bench.py is the measured contract)."""
import sys, os, time, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from mythtracer_b200 import MythTracer, Light, scenegen, MTB_FLAG_COUNT_WORK, MTB_FLAG_NO_LIST_BVH

names = sys.argv[1].split(",") if len(sys.argv) > 1 else ["C1", "C2", "C3"]
modes = sys.argv[2].split(",") if len(sys.argv) > 2 else ["bvh"]
out = []
for name in names:
    files, cfg = scenegen.generate_config(name, "/tmp/mtb_scenes")
    for mode in modes:
        base_flags = {"bvh": 16, "nobvh": MTB_FLAG_NO_LIST_BVH | 16, "auto": 0, "noorder": 16 | 32, "exact": 16 | 128, "devbvh": 16 | 4096, "queue": 8192}.get(mode, 0)
        mt = MythTracer(max_depth=cfg["depth"], flags=base_flags)
        t0 = time.time(); assert mt.LoadObj(files.obj_path); t_load = time.time() - t0
        mt.GetScene().lights = [Light.from_tuple(l) for l in files.lights]
        w, h = cfg["width"], cfg["height"]
        best = None
        all_ms = []
        for it in range(8):
            r = mt.render_chunk(files.camera, w, h, 0, 0, w, h)
            s = r["stats"]
            all_ms.append(round(s["kernel_ms"], 3))
            if best is None or s["kernel_ms"] < best["kernel_ms"]: best = s
        mt.set_flags(MTB_FLAG_COUNT_WORK | base_flags)
        c = mt.render_chunk(files.camera, w, h, 0, 0, w, h)["stats"]
        rays = best["rays"]
        rec = dict(kernel_ms=round(best["kernel_ms"], 3), config=name, mode=mode, tris=files.n_triangles, w=w, h=h, load_s=round(t_load, 2),
                   total_ms=round(best["total_ms"], 3), rays=rays, mrays_s=round(rays / best["kernel_ms"] / 1e3, 1),
                   per_ray=dict(slab=round(c["n_slab"] / rays, 1), visit=round(c["n_visit"] / rays, 1), triaabb=round(c["n_triaabb"] / rays, 1),
                                bvh=round(c["n_bvh"] / rays, 1), mt=round(c["n_mt"] / rays, 2), hit=round(c["n_hit"] / rays, 2), shade=round(c["n_shade"] / rays, 2)),
                   literal=c["n_literal"], fast=c["n_fast"], fallback=c["n_fallback"], count_kernel_ms=round(c["kernel_ms"], 1), all_ms=all_ms,
                   long128=dict(rays=c["n_long128_rays"], visits=c["n_long128_visits"]), long512=dict(rays=c["n_long512_rays"], visits=c["n_long512_visits"]),
                   total_visits=c["n_bvh"] // 2, load=mt.load_timing())
        print(json.dumps(rec), flush=True)
        out.append(rec)
        mt.close()
os.makedirs("gpurun_out", exist_ok=True)
json.dump(out, open("gpurun_out/quick_time.json", "w"), indent=1)
