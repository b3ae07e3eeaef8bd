"""One GPU renders 1/world of the C3 frame with the queue pipeline or the megakernel (development aid for launch lists)."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from mythtracer_b200 import MythTracer, Light, scenegen, MTB_FLAG_QUEUE, tiles
world = int(sys.argv[1]); mode = sys.argv[2]
files, cfg = scenegen.generate_config("C3", "/tmp/mtb_scenes")
mt = MythTracer(max_depth=cfg["depth"], flags=MTB_FLAG_QUEUE if mode == "queue" else 16)
assert mt.LoadObj(files.obj_path)
mt.GetScene().lights = [Light.from_tuple(l) for l in files.lights]; mt.push_lights()
W, H = cfg["width"], cfg["height"]
buf = torch.zeros((tiles.padded_height(H, world), W, 3), dtype=torch.uint8, device="cuda")
mt.set_partition(0, world)
for it in range(3):
    mt.render_device(files.camera, W, H, buf.data_ptr(), 0)
    torch.cuda.synchronize()
