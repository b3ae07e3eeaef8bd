"""Is a small share of the frame latency-bound or throughput-bound?  Two contexts on ONE GPU render two different 1/16
shares of the C3 frame, first one after the other, then at the same time (two streams); if the concurrent pair takes
about as long as one alone, the kernels of a share do not fill the machine (development aid)."""
import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from mythtracer_b200 import MythTracer, Light, scenegen, tiles
world = int(sys.argv[1]) if len(sys.argv) > 1 else 16
mode = sys.argv[2] if len(sys.argv) > 2 else "queue"
flags = {"queue": 8192, "mega": 16, "auto": 0}[mode]
files, cfg = scenegen.generate_config("C3", "/tmp/mtb_scenes")
W, H = cfg["width"], cfg["height"]
mts, streams, bufs = [], [], []
for r in range(2):
    mt = MythTracer(max_depth=cfg["depth"], flags=flags)
    assert mt.LoadObj(files.obj_path)
    mt.GetScene().lights = [Light.from_tuple(l) for l in files.lights]; mt.push_lights()
    mt.set_partition(r, world)
    mts.append(mt); streams.append(torch.cuda.Stream()); bufs.append(torch.zeros((tiles.padded_height(H, world), W, 3), dtype=torch.uint8, device="cuda"))
def run(which):
    for r in which:
        mts[r].render_device(files.camera, W, H, bufs[r].data_ptr(), streams[r].cuda_stream)
for _ in range(16):
    run([0, 1]); torch.cuda.synchronize()
res = {}
for name, which in (("rank0 alone", [0]), ("rank1 alone", [1]), ("both at once", [0, 1])):
    ts = []
    for _ in range(8):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(torch.cuda.default_stream())
        for r in which: streams[r].wait_event(e0)
        run(which)
        for r in which: torch.cuda.default_stream().wait_stream(streams[r])
        e1.record(torch.cuda.default_stream())
        torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1))
    res[name] = round(min(ts), 3)
print(json.dumps(dict(world=world, mode=mode, **res)))
