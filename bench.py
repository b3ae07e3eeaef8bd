#!/usr/bin/env python
"""bench.py -- the measured contract of mythtracer_b200 (see DESIGN.md, "Measurement").

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA kernels through the C ABI)
    python bench.py --impl reference --steps K --warmup W    # the reference's own CPU renderer (oracle/_ref)

Workload: BASELINE.json configs[2] ("C3": ~500k-triangle synthetic interior, 1920x1080, 2 lights, depth 5,
the configuration the 1080p metric is quoted on; it fits one GPU).  A step = one full frame of the fixed
BASELINE camera = one pass of the hot path (MythTracer::RayTrace, mythtracer.cc:280-312).

metric   Mrays/s, rays = OctTree::IntersectRay-equivalent queries (primary + shadow segments + reflection
         + refraction rays), counted on the device; identical to the reference's count (parity tests).
value    whole-job Mrays/s with everything resident in HBM: K frames rendered into device memory (N > 1:
         every rank renders its strips of the same frame -- strong scaling -- and its kernels store the tiles
         straight into rank 0's frame over NVLink), CUDA events, max over ranks.
e2e      the same metric through the reference-facing call with HOST buffers (mtb_render_chunk: lights
         and camera go host->device, the RGB24 frame comes back into pinned host memory), per step, L2 flushed
         before every step as in the device-resident loop.
frame_sha  sha256 of the last timed frame as it stands in rank 0's HBM -- the same at every N, and equal to the
         reference's own render of the frame (tests/golden/full_C3.npz -> reference_frame_sha).
roofline algorithmic bytes of one frame (SURVEY.md 8d formula over the kernel's own work counters, from
         the counting build run outside the timed region) / the kernel time measured inside the timed loop,
         against the measured HBM copy bandwidth of MEASURED_PEAKS.json; dram_frac = ncu DRAM bytes / time / peak.
cpu_baseline  the unmodified reference (oracle/_ref) on all host cores, on a bounded sample of the same
         frame (full-width row bands), rays of the sample counted by the oracle restatement.
config.other_workloads  the other GPU configurations of BASELINE.json (C2, C4, C5) on the same GPU, 3 frames each.

--dump-outputs DIR writes the frame of the last timed step (what a caller of the timed path receives) to
DIR/frame.npy as float32 (H, W, 3); the scene, camera and lights are seeded, so two builds can be compared output for
output.  The benchmark runs the library as it was built and writes nothing into the source tree.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # no __pycache__ in the tree

WORKLOAD = "C3"
SCENE_DIR = os.environ.get("MTB_SCENE_DIR", "/tmp/mtb_scenes")
L2_FLUSH_BYTES = 256 << 20
FALLBACK_HBM_GBS = 6650.0  # B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            with open(path) as f:
                return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "B200_PROFILING.md fallback"


def alg_flops(stats) -> float:
    """SURVEY.md 8(d): 24 flops per box test, 57 per Moller-Trumbore, 400 per shaded hit."""
    return (24.0 * (stats["n_slab"] + stats["n_triaabb"] + stats.get("n_bvh", 0)) + 57.0 * stats["n_mt"] +
            400.0 * stats["n_shade"])


def measured_fp64_peak():
    """FP64 separate add / mul issue rate (the code is built with --fmad=false), tools/fp_peak.cu on this pool."""
    path = os.path.join(ROOT, "profiles", "fp_peaks.json")
    try:
        with open(path) as f:
            return float(json.load(f)["fp64_addmul_tflops"]), "profiles/fp_peaks.json fp64_addmul_tflops (tools/fp_peak.cu, measured)"
    except Exception:
        return None, "unmeasured"


def alg_bytes(stats) -> float:
    """SURVEY.md 8(d): operands the arithmetic consumes: 48-byte FP64 boxes for octree slab tests and exact triangle
    pre-tests, 24-byte FP32 boxes for the conservative BVH culls (scene BVH / list BVH), 72 bytes of vertices per
    Moller-Trumbore evaluation, 384 bytes per shaded hit."""
    return (48.0 * (stats["n_slab"] + stats["n_triaabb"]) + 24.0 * stats.get("n_bvh", 0) + 72.0 * stats["n_mt"] +
            384.0 * stats["n_shade"])


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        self.index = index
        self.samples = []
        self.proc = None
        self.thread = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 7:
                self.samples.append(parts)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for p in self.samples:
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
            except ValueError:
                continue
            for n, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def load_workload():
    from mythtracer_b200 import scenegen
    files, cfg = scenegen.generate_config(WORKLOAD, SCENE_DIR)
    return files, cfg


def config_dict(files, cfg, n_gpus, extra=None):
    d = {"workload": "%s: %d-triangle synthetic interior (seed %d), %dx%d, %d lights, depth %d, fixed BASELINE camera" % (
        WORKLOAD, files.n_triangles, cfg["seed"], cfg["width"], cfg["height"], cfg["n_lights"], cfg["depth"]),
        "triangles": files.n_triangles, "width": cfg["width"], "height": cfg["height"], "lights": cfg["n_lights"],
        "max_depth": cfg["depth"], "partition": "strips of 8 rows, round-robin over %d GPU(s)" % n_gpus,
        "l2": "256 MiB device memset between steps (inside the timed region) flushes the 126 MB L2"}
    if extra:
        d.update(extra)
    return d


# ----------------------------------------------------------------------------------------------------
# reference arm / cpu baseline
# ----------------------------------------------------------------------------------------------------

def sample_bands(height, width, n_bands, rows_per_band):
    """Full-width row bands spread evenly over the frame (the reference renders rectangles only)."""
    bands = []
    for i in range(n_bands):
        y = int((i + 0.5) * height / n_bands) - rows_per_band // 2
        y = max(0, min(height - rows_per_band, y))
        bands.append((0, y, width, rows_per_band))
    return bands


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def time_reference(files, cfg, target_seconds, steps, warmup, min_bands=3):
    """Times the unmodified reference (oracle/_ref) on a bounded sample of the frame, on ALL host cores (a launcher
    such as torch.distributed.run exports OMP_NUM_THREADS=1; the team size is set explicitly).  Returns dict."""
    from oracle import oracle_py
    if not oracle_py.Reference.available():
        return None
    ref = oracle_py.Reference(files.obj_path)
    ref.set_lights(files.lights)
    ref.set_threads(host_cores())
    threads = ref.threads()
    W, H = cfg["width"], cfg["height"]
    # probe: one band, rows = thread count (static OpenMP schedule over rows, mythtracer.cc:292-295)
    rows = max(8, min(H, threads))
    probe = ref.render(files.camera, W, H, chunk=(0, H // 2, W, rows), depth=cfg["depth"], debug=False)
    per_row = probe["seconds"] / rows
    total_rows = max(rows * min_bands, int(target_seconds / max(per_row, 1e-9)))
    n_bands = max(min_bands, min(8, total_rows // rows))
    rows_per_band = max(rows, min(H // n_bands, total_rows // n_bands))
    bands = sample_bands(H, W, n_bands, rows_per_band)
    # rays of the sample: counted by the oracle restatement (bit-identical to the reference, see tests/)
    orc = oracle_py.Oracle.from_obj(files.obj_path)
    orc.set_lights(files.lights)
    orc.set_threads(host_cores())
    rays = 0
    for b in bands:
        rays += orc.render(files.camera, W, H, chunk=b, depth=cfg["depth"], debug=False)["stats"]["rays"]
    times = []
    for it in range(warmup + steps):
        t = 0.0
        for b in bands:
            t += ref.render(files.camera, W, H, chunk=b, depth=cfg["depth"], debug=False)["seconds"]
        if it >= warmup:
            times.append(t)
    sec = sum(times) / len(times)
    px = sum(b[2] * b[3] for b in bands)
    return {"seconds_per_step": sec, "rays_per_step": rays, "pixels": px, "threads": threads,
            "mrays_s": rays / sec / 1e6,
            "sample": "%d full-width bands of %d rows spread over the frame height (%d of %d pixels, %.2f%% of the frame)" % (
                n_bands, rows_per_band, px, W * H, 100.0 * px / (W * H)),
            "frame_ms_extrapolated": sec * 1e3 * (W * H) / px}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    files, cfg = load_workload()
    warm = min(args.warmup, 1)  # a warm-up pass of the sample costs as much as a timed one: one is run, and reported
    res = time_reference(files, cfg, target_seconds=6.0, steps=max(1, min(args.steps, 3)), warmup=warm)
    if res is None:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref is not built and /root/reference is absent"}))
        return 0
    line = {
        "impl": "reference", "metric": "Mrays/s", "value": res["mrays_s"], "unit": "Mrays/s", "n_gpus": args.gpus,
        "steps": max(1, min(args.steps, 3)), "warmup": warm, "ms_per_step": res["seconds_per_step"] * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_dict(files, cfg, args.gpus, {"step": "bounded sample: " + res["sample"],
                                                     "frame_ms_extrapolated": res["frame_ms_extrapolated"],
                                                     "host_cores": host_cores(), "omp_threads": res["threads"]}),
        "cpu_baseline": {"value": res["mrays_s"], "unit": "Mrays/s", "cores": res["threads"], "kind": "reference",
                         "sample": res["sample"]},
        "e2e": {"value": res["mrays_s"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ----------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------

def run_ours(args):
    # NCCL / the loader may print to stdout; the contract is ONE JSON line there, so everything else goes to
    # stderr until the final print
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        line = _run_ours(args)
    finally:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        os.close(saved_stdout)
    if line is not None:
        print(json.dumps(line), flush=True)
    return 0


def golden_frame_sha():
    """sha256 of the reference's own render of the C3 frame (tests/golden/full_C3.npz, made by oracle/_ref)."""
    path = os.path.join(ROOT, "tests", "golden", "full_%s.npz" % WORKLOAD)
    try:
        import numpy as np
        with np.load(path) as z:
            return str(z["rgb_sha256"])
    except Exception:
        return None


def git_head():
    """Commit of the tree: from git where there is one, else the stamp mythtracer_b200/build.py left next to the
    built library (the GPU box gets a snapshot without .git)."""
    try:
        return subprocess.check_output(["git", "-C", ROOT, "rev-parse", "--short", "HEAD"], stderr=subprocess.DEVNULL, text=True).strip()
    except Exception:
        pass
    try:
        with open(os.path.join(ROOT, "mythtracer_b200", "build", "commit.txt")) as f:
            return f.read().strip() or None
    except Exception:
        return None


def time_other_workloads(names, steps):
    """The other GPU configurations of BASELINE.json on this GPU (after the C3 timed region): frame ms (CUDA events
    around mtb_render_chunk_device, L2 flushed before every frame), Mrays/s, rays per frame, the pipeline the library
    chose, time to the first frame split by stage."""
    import hashlib
    import torch
    from mythtracer_b200 import Light, MythTracer, scenegen
    out = {}
    dev = torch.device("cuda", torch.cuda.current_device())
    stream = torch.cuda.current_stream()
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
    for name in names:
        try:
            t0 = time.time()
            files, cfg = scenegen.generate_config(name, SCENE_DIR)
            gen_s = time.time() - t0
            W, H = cfg["width"], cfg["height"]
            mt = MythTracer(devices=[dev.index], max_depth=cfg["depth"], flags=0)
            t0 = time.time()
            if not mt.LoadObj(files.obj_path):
                raise RuntimeError(mt.last_error())
            load_s = time.time() - t0
            mt.GetScene().lights = [Light.from_tuple(l) for l in files.lights]
            mt.push_lights()
            d_frame = torch.zeros((H, W, 3), dtype=torch.uint8, device=dev)
            t0 = time.time()
            mt.render_device(files.camera, W, H, d_frame.data_ptr(), stream.cuda_stream)
            torch.cuda.synchronize(dev)
            first_frame_s = time.time() - t0
            for _ in range(14):  # automatic pipeline choice: twelve measuring frames
                mt.render_device(files.camera, W, H, d_frame.data_ptr(), stream.cuda_stream)
            torch.cuda.synchronize(dev)
            mt.read_counters()
            evs = []
            for _ in range(steps):
                flush.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream)
                mt.render_device(files.camera, W, H, d_frame.data_ptr(), stream.cuda_stream)
                b.record(stream)
                evs.append((a, b))
            torch.cuda.synchronize(dev)
            ms = sum(a.elapsed_time(b) for a, b in evs) / len(evs)
            rays = mt.read_counters()["rays"] / steps
            # the same frame as the unmodified reference rendered it (tests/golden/full_<cfg>.npz: whole frame or bands)
            equals_ref, ref_rows = None, 0
            gpath = os.path.join(ROOT, "tests", "golden", "full_%s.npz" % name)
            frame_np = d_frame.cpu().numpy()
            if os.path.exists(gpath):
                try:
                    import numpy as np
                    with np.load(gpath) as z:
                        rows = z["rows"]
                        ref_rows = int(len(rows))
                        equals_ref = bool(int(z["width"]) == W and int(z["height"]) == H and np.array_equal(frame_np[rows], z["rgb"]))
                except Exception:
                    equals_ref = None
            out[name] = {"equals_reference": equals_ref, "reference_rows_compared": ref_rows, "triangles": files.n_triangles, "width": W, "height": H, "lights": cfg["n_lights"], "max_depth": cfg["depth"],
                         "ms_per_frame": ms, "mrays_s": rays / ms / 1e3, "rays_per_frame": rays, "pipeline": mt.pipeline_in_use()[0],
                         "steps": steps, "scene_generate_s": gen_s, "scene_load_s": load_s, "first_frame_s": first_frame_s,
                         "time_to_first_frame_s": load_s + first_frame_s, "load_stages_ms": mt.load_timing(),
                         "frame_sha256": hashlib.sha256(frame_np.tobytes()).hexdigest()}
            mt.close()
            del d_frame
        except Exception as e:  # reported, never required
            out[name] = {"error": repr(e)}
    return out


def _run_ours(args):
    import hashlib

    import numpy as np
    import torch
    import torch.distributed as dist

    from mythtracer_b200 import Light, MythTracer, MTB_FLAG_COUNT_WORK, MTB_FLAG_HYBRID, MTB_FLAG_MEGAKERNEL, MTB_FLAG_QUEUE, MTB_FLAG_WAVEFRONT, tiles

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        log("warning: WORLD_SIZE %d != --gpus %d; using WORLD_SIZE" % (world, args.gpus))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    if world > 1:
        dist.barrier()
    files, cfg = (load_workload() if rank == 0 else (None, None))
    if world > 1:
        dist.barrier()
        if rank != 0:
            files, cfg = load_workload()  # reuses the files rank 0 wrote
    W, H, depth = cfg["width"], cfg["height"], cfg["depth"]

    base_flags = {"wavefront": MTB_FLAG_WAVEFRONT, "mega": MTB_FLAG_MEGAKERNEL, "hybrid": MTB_FLAG_HYBRID, "queue": MTB_FLAG_QUEUE, "auto": 0}[args.pipeline]
    # Launched plainly (no torchrun) with --gpus N > 1: ONE process, one context over N devices -- the
    # in-process form (strips interleaved over the devices, tiles stored straight into device 0's frame over NVLink).
    inproc = 1
    if world == 1 and args.gpus > 1:
        inproc = min(args.gpus, torch.cuda.device_count())
    mt = MythTracer(devices=[local_rank] if inproc == 1 else list(range(inproc)), max_depth=depth, flags=base_flags)
    t0 = time.time()
    if not mt.LoadObj(files.obj_path):
        raise SystemExit("LoadObj failed: " + mt.last_error())
    load_s = time.time() - t0
    load_stages = mt.load_timing()
    mt.GetScene().lights = [Light.from_tuple(l) for l in files.lights]
    mt.push_lights()
    mt.set_partition(rank, world)
    info = mt.scene_info()

    # a real (non-default) stream: its handle goes through the C ABI, so that the kernels, torch's copies /
    # collectives and the timing events are all on one stream (torch.cuda.Event only sees torch's stream)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    frame_bytes = W * H * 3
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
    h_frame = torch.empty((H, W, 3), dtype=torch.uint8).pin_memory()
    sync_word = torch.zeros(1, dtype=torch.int32, device=dev)

    # ---- where the frame lives ----
    # N = 1: a torch tensor.  N > 1 under torchrun, gather "peer" (default): rank 0 owns TWO frames (double buffer)
    # allocated by the library, the other ranks map them (cudaIpc*) and every rank's kernels store the tiles it
    # owns straight into rank 0's HBM over NVLink; the only collective of a step is a 4-byte all-reduce that orders
    # "all tiles are in" before rank 0 reads the frame.  gather "nccl": every rank renders into its own frame and
    # the strips are gathered with one NCCL gather (round 1's path, kept for the A/B).
    gather = args.gather if world > 1 else "none"
    shared = [None, None]
    d_local = None
    d_frame_nccl = None
    if world == 1 or inproc > 1:
        d_local = torch.zeros((H, W, 3), dtype=torch.uint8, device=dev)
    elif gather == "peer":
        handles = [None, None]
        if rank == 0:
            for k in range(2):
                shared[k], handles[k] = mt.frame_create(frame_bytes)
        box = [handles]
        dist.broadcast_object_list(box, src=0)
        if rank != 0:
            for k in range(2):
                shared[k] = mt.frame_open(box[0][k])
    else:
        hp = tiles.padded_height(H, world)
        d_local = torch.zeros((hp, W, 3), dtype=torch.uint8, device=dev)
        d_frame_nccl = torch.zeros((hp, W, 3), dtype=torch.uint8, device=dev) if rank == 0 else None

    step_no = [0]

    def step_device():
        """One step: L2 flush, this rank's tiles, and (N > 1) whatever makes the frame complete on rank 0."""
        flush.zero_()
        if world == 1:
            mt.render_device(files.camera, W, H, d_local.data_ptr(), stream.cuda_stream)
            return d_local.data_ptr()
        if gather == "peer":
            target = shared[step_no[0] & 1]
            step_no[0] += 1
            mt.render_device(files.camera, W, H, target, stream.cuda_stream)
            dist.all_reduce(sync_word)  # orders every rank's stores before rank 0's next read of this frame
            return target
        mt.render_device(files.camera, W, H, d_local.data_ptr(), stream.cuda_stream)
        fr = tiles.gather_frame(d_local, H, W, rank, world, 0, out=d_frame_nccl)
        return fr.data_ptr() if fr is not None else 0

    def read_frame(ptr):
        """The frame of the last step as host bytes (rank 0)."""
        torch.cuda.synchronize(dev)
        if world > 1 and gather == "peer":
            return mt.frame_read(ptr, frame_bytes)
        src = d_local if world == 1 else d_frame_nccl
        return src[:H].contiguous().cpu().numpy().reshape(-1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- warm-up, then K timed steps (device-resident).  The automatic pipeline choice measures the megakernel, the
    # queue pipeline and the hybrid split during the first 12 frames of a geometry and decides at the 13th, so the
    # warm-up covers at least 14 (reported as "warmup" in the JSON line) ----
    n_warm = max(args.warmup, 14 if args.pipeline == "auto" else (10 if args.pipeline == "hybrid" else 3))
    for _ in range(n_warm):
        step_device()
    barrier()
    mt.read_counters()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k_events = []
    barrier()
    launches0 = mt.launch_count()
    ev0.record(stream)
    last_ptr = 0
    for _ in range(args.steps):
        # (the per-step kernel time is measured INSIDE the timed loop: events around this rank's render call)
        flush.zero_()
        ka, kb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ka.record(stream)
        if world == 1:
            mt.render_device(files.camera, W, H, d_local.data_ptr(), stream.cuda_stream)
            kb.record(stream)
            last_ptr = d_local.data_ptr()
        elif gather == "peer":
            target = shared[step_no[0] & 1]
            step_no[0] += 1
            mt.render_device(files.camera, W, H, target, stream.cuda_stream)
            kb.record(stream)
            dist.all_reduce(sync_word)
            last_ptr = target
        else:
            mt.render_device(files.camera, W, H, d_local.data_ptr(), stream.cuda_stream)
            kb.record(stream)
            fr = tiles.gather_frame(d_local, H, W, rank, world, 0, out=d_frame_nccl)
            last_ptr = fr.data_ptr() if fr is not None else 0
        k_events.append((ka, kb))
    ev1.record(stream)
    barrier()
    launches = mt.launch_count() - launches0
    elapsed_ms = ev0.elapsed_time(ev1)
    kernel_ms_mean = sum(a.elapsed_time(b) for a, b in k_events) / len(k_events)
    counters = mt.read_counters()
    frame = read_frame(last_ptr) if rank == 0 else None
    frame_sha = hashlib.sha256(frame.tobytes()).hexdigest() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        # 1920 x 1080 x 3 float32 = 25 MB: the whole frame, exact (uint8 values)
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "frame.npy"), frame.reshape(H, W, 3).astype(np.float32))
        log("bench.py: wrote the last timed frame to %s" % os.path.join(args.dump_outputs, "frame.npy"))
    t = torch.tensor([elapsed_ms, float(counters["rays"]), float(launches), kernel_ms_mean], dtype=torch.float64, device=dev)
    kernel_ms_max = kernel_ms_mean
    kernel_ms_ranks = [kernel_ms_mean]
    if world > 1:
        per_rank = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(per_rank, t[3:4].clone())
        kernel_ms_ranks = [round(float(x[0]), 4) for x in per_rank]
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        elapsed_ms, total_rays, launches, kernel_ms_max = float(tmax[0]), float(tsum[1]), int(tsum[2]), float(tmax[3])
    else:
        total_rays = float(t[1])
    rays_per_frame = total_rays / args.steps
    value = total_rays / (elapsed_ms * 1e-3) / 1e6

    pipeline_used, tune_mega_ms, tune_wf_ms = mt.pipeline_in_use()

    # ---- end to end through the host-buffer call (lights + camera H2D, frame D2H into pinned memory), L2 flushed
    # before every step like the device-resident loop ----
    h_np = h_frame.numpy()
    for _ in range(2):
        if world == 1:
            mt.render_chunk(files.camera, W, H, 0, 0, W, H, out=h_np)
    barrier()
    e0 = time.perf_counter()
    for _ in range(args.steps):
        flush.zero_()
        if world == 1:
            stream.synchronize()
            mt.render_chunk(files.camera, W, H, 0, 0, W, H, out=h_np)
        else:
            mt.push_lights()
            if gather == "peer":
                target = shared[step_no[0] & 1]
                step_no[0] += 1
                mt.render_device(files.camera, W, H, target, stream.cuda_stream)
                dist.all_reduce(sync_word)
                if rank == 0:
                    mt.frame_read(target, frame_bytes, out=h_np.reshape(-1))  # D2H into the pinned frame
            else:
                mt.render_device(files.camera, W, H, d_local.data_ptr(), stream.cuda_stream)
                fr = tiles.gather_frame(d_local, H, W, rank, world, 0, out=d_frame_nccl)
                if rank == 0:
                    h_frame.copy_(fr, non_blocking=True)
            torch.cuda.synchronize(dev)
    barrier()
    e2e_s = time.perf_counter() - e0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s = float(te[0])
    e2e_value = rays_per_frame * args.steps / e2e_s / 1e6
    e2e_sha = hashlib.sha256(h_np.tobytes()).hexdigest() if rank == 0 else None
    clocks = sampler.stop() if rank == 0 else None

    # ---- work counters of one frame (counting build, not timed) -> algorithmic bytes ----
    mt.read_counters()  # reset
    mt.set_flags(MTB_FLAG_COUNT_WORK | base_flags)
    scratch = d_local.data_ptr() if d_local is not None else shared[0]
    mt.render_device(files.camera, W, H, scratch, stream.cuda_stream)
    torch.cuda.synchronize(dev)
    work = mt.read_counters()
    mt.set_flags(base_flags)
    keys = ("n_slab", "n_triaabb", "n_bvh", "n_mt", "n_shade", "n_visit", "n_hit", "rays", "n_fast", "n_fallback", "n_literal")
    wt = torch.tensor([float(work[k]) for k in keys], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(wt, op=dist.ReduceOp.SUM)
    work_all = dict(zip(keys, [float(x) for x in wt]))
    my_alg = alg_bytes(work)
    my_flops = alg_flops(work)

    if rank != 0:
        if world > 1:
            barrier()
            dist.destroy_process_group()
        return None

    peak, peak_src = measured_peak()
    fp_peak, fp_src = measured_fp64_peak()
    # (one context over several devices counts the work of all of them, the kernel time is one device's: its share)
    my_alg /= inproc
    my_flops /= inproc
    achieved = my_alg / (kernel_ms_mean * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            with open(tpath) as f:
                tj = json.load(f)
            if tj.get("workload") == WORKLOAD and tj.get("n_gpus", 1) == world * inproc and pipeline_used == "mega":
                traffic = tj.get("dram_bytes_per_launch")
                traffic_src = "%s; captured at commit %s (not measured in this run)" % (tj.get("source"), tj.get("commit"))
        except Exception:
            pass
    golden = golden_frame_sha()
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src,
                "dram_frac": (traffic / (kernel_ms_mean * 1e-3) / 1e9 / peak) if traffic else None,
                "kernel": {"mega": "RenderMega", "hybrid": "RenderMega + wavefront kernels on the most expensive tiles, concurrently",
                           "queue": "WfQueue (one persistent kernel over the device-side ray queue; + WfResolveTree)"}.get(pipeline_used, "wavefront pipeline (WfTrace + WfShadow dominate)"),
                "kernel_ms": kernel_ms_mean, "kernel_ms_max_over_ranks": kernel_ms_max, "kernel_ms_per_rank": kernel_ms_ranks,
                "kernel_ms_how": "mean over the K timed steps of CUDA events recorded around this rank's render call inside the timed loop (after the L2 flush)",
                "algorithmic_bytes_per_launch": my_alg, "peak_source": peak_src,
                "note": "frac counts ALGORITHMIC operand bytes (SURVEY 8d), most of which are served by L1/L2 (the BVH top and neighbouring rays' nodes are shared); dram_frac = ncu DRAM bytes of the same launch / time / peak is the HBM utilisation proper",
                "fp": {"bound": "fp64 add/mul issue", "achieved": my_flops / (kernel_ms_mean * 1e-3) / 1e12, "peak": fp_peak,
                       "unit": "Tflop/s", "frac": (my_flops / (kernel_ms_mean * 1e-3) / 1e12 / fp_peak) if fp_peak else None,
                       "peak_source": fp_src, "algorithmic_flops_per_launch": my_flops},
                "per_ray": {k: work_all[k] / max(work_all["rays"], 1.0) for k in ("n_slab", "n_visit", "n_triaabb", "n_bvh", "n_mt", "n_hit", "n_shade")},
                "traversal": {"fast": work_all["n_fast"], "exact_fallback": work_all["n_fallback"], "literal": work_all["n_literal"]}}

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            r = time_reference(files, cfg, target_seconds=12.0, steps=1, warmup=0)
            if r is not None:
                cpu = {"value": r["mrays_s"], "unit": "Mrays/s", "cores": r["threads"], "kind": "reference",
                       "sample": r["sample"], "frame_ms_extrapolated": r["frame_ms_extrapolated"]}
        except Exception as e:  # the baseline is reported, never required
            log("cpu_baseline failed:", repr(e))

    others = None
    if world == 1 and inproc == 1 and not args.no_other_workloads:
        others = time_other_workloads(["C2", "C4", "C5"], 3)

    launch = ("one process per GPU (torchrun); " + ("tiles stored straight into rank 0's frame over NVLink (cudaIpc mapping), one 4-byte all-reduce per step"
                                                   if gather == "peer" else "NCCL gather of the strips")) if world > 1 else (
        "one process, one context over %d devices, tiles stored straight into device 0's frame" % inproc if inproc > 1 else "one process, one GPU")
    lights_bytes = 96 * len(files.lights)
    line = {
        "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": world * inproc, "steps": args.steps, "warmup": n_warm,
        "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": config_dict(files, cfg, world * inproc, {"launch": launch, "gather": gather,
                                                           "pipeline": pipeline_used, "pipeline_choice": args.pipeline, "hybrid_share": mt.hybrid_share(), "autotune_ms": {"mega": tune_mega_ms, "queue": tune_wf_ms},
                                                           "rays_per_frame": rays_per_frame, "scene_load_s": load_s, "load_stages_ms": load_stages,
                                                           "octree_nodes": info["n_nodes"], "tree_depth": info["tree_depth"],
                                                           "device_scene_bytes": info["device_bytes"], "commit": git_head(),
                                                           "other_workloads": others}),
        "frame_sha": frame_sha, "e2e_frame_sha": e2e_sha, "reference_frame_sha": golden,
        "frame_equals_reference": (frame_sha == golden) if golden else None,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "e2e": {"value": e2e_value, "unit": "Mrays/s", "ms_per_step": e2e_s * 1e3 / args.steps,
                "h2d_bytes_per_step": lights_bytes + 256, "d2h_bytes_per_step": W * H * 3,
                "l2": "256 MiB device memset before every step, inside the timed region"},
        "gpu_launches": int(launches),
        "clocks": clocks,
    }
    if world > 1:
        barrier()
        dist.destroy_process_group()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-workloads", action="store_true", default=os.environ.get("MTB_BENCH_OTHERS", "1") == "0")
    ap.add_argument("--pipeline", default=os.environ.get("MTB_PIPELINE", "auto"), choices=["auto", "mega", "wavefront", "hybrid", "queue"])
    ap.add_argument("--gather", default=os.environ.get("MTB_GATHER", "peer"), choices=["peer", "nccl"],
                    help="N > 1 under torchrun: direct peer stores into rank 0's frame (default) or an NCCL gather (A/B)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the frame of the last timed step to DIR/frame.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
