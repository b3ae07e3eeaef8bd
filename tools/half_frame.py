"""Times the queue pipeline / megakernel on a 1/world partition of the C3 frame on ONE GPU (scaling diagnosis).
   half_frame.py <world> <mega|queue|auto> [rank,rank,...]   (default: ranks 0 and 1)"""
import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from mythtracer_b200 import MythTracer, Light, scenegen, tiles
world = int(sys.argv[1]); mode = sys.argv[2]
files, cfg = scenegen.generate_config("C3", "/tmp/mtb_scenes")
mt = MythTracer(max_depth=cfg["depth"], flags={"mega": 16, "queue": 8192, "auto": 0}[mode])
assert mt.LoadObj(files.obj_path)
mt.GetScene().lights = [Light.from_tuple(l) for l in files.lights]; mt.push_lights()
W, H = cfg["width"], cfg["height"]
s = torch.cuda.Stream(); torch.cuda.set_stream(s)
buf = torch.zeros((tiles.padded_height(H, world), W, 3), dtype=torch.uint8, device="cuda")
ranks = [int(x) for x in sys.argv[3].split(",")] if len(sys.argv) > 3 else list(range(min(world, 2)))
for rank in ranks:
    mt.set_partition(rank, world)
    ts = []
    for it in range(16):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record(s)
        mt.render_device(files.camera, W, H, buf.data_ptr(), s.cuda_stream)
        e1.record(s); torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1))
    c = mt.read_counters()
    print(json.dumps(dict(mode=mode, world=world, rank=rank, ms=round(min(ts[8:]), 2), first=round(ts[1], 2), rays_per_frame=c["rays"] // 16)))
