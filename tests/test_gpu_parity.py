"""GPU parity tests proper: the CUDA path, called through the C ABI, against the CPU oracle on the same inputs.

Bars (BASELINE.json north_star): primary-hit ids, hit points, every shadow decision and every ray count
must agree exactly; RGB is compared byte for byte too -- the one place that can legitimately differ is pow()
(mythtracer.cc:174: CUDA and glibc differ by <= 2 ulp), so RGB is allowed MAX_RGB_DIFF = 1 LSB on at most
MAX_RGB_FRACTION of the channels (stated tolerance; north_star allows <= 2/255).  In practice it is 0.
"""
import numpy as np
import pytest

from tests import scenes

pytestmark = pytest.mark.gpu

MAX_RGB_DIFF = 1
MAX_RGB_FRACTION = 1e-5


def _tracer(product_lib, depth, flags=0, devices=None):
    """flags without a pipeline bit: force the megakernel (small test frames would auto-select the queue pipeline)."""
    from mythtracer_b200 import MTB_FLAG_MEGAKERNEL, MTB_FLAG_WAVEFRONT, MythTracer
    from mythtracer_b200 import MTB_FLAG_QUEUE
    if not flags & (MTB_FLAG_WAVEFRONT | MTB_FLAG_MEGAKERNEL | MTB_FLAG_QUEUE):
        flags |= MTB_FLAG_MEGAKERNEL
    return MythTracer(devices=devices, max_depth=depth, flags=flags)


def _oracle_for(oracle_mod, mt):
    """Oracle over exactly the arrays the product loader produced."""
    tris, mtls = mt.scene_arrays()
    return tris, mtls


def _load_pair(product_lib, oracle_mod, files, depth, flags=0):
    from mythtracer_b200 import Light
    mt = _tracer(product_lib, depth, flags)
    assert mt.LoadObj(files.obj_path), mt.last_error()
    mt.GetScene().lights = [Light.from_tuple(l) for l in files.lights]
    orc = oracle_mod.Oracle.from_obj(files.obj_path)
    orc.set_lights(files.lights)
    return mt, orc


def _assert_render_equal(gpu, cpu, what):
    assert np.array_equal(gpu["line_no"], cpu["line_no"]), "%s: primary hit ids differ at %d pixels" % (
        what, int((gpu["line_no"] != cpu["line_no"]).sum()))
    assert np.array_equal(gpu["points"], cpu["points"], equal_nan=True), "%s: hit points differ" % what
    assert np.array_equal(gpu["n_rays"], cpu["n_rays"]), "%s: per-pixel ray counts differ" % what
    assert np.array_equal(gpu["sig_hits"], cpu["sig_hits"]), "%s: secondary hit ids differ" % what
    assert np.array_equal(gpu["sig_shadow"], cpu["sig_shadow"]), "%s: shadow decisions differ" % what
    diff = np.abs(gpu["rgb"].astype(np.int16) - cpu["rgb"].astype(np.int16))
    assert diff.max() <= MAX_RGB_DIFF, "%s: max RGB error %d" % (what, diff.max())
    assert (diff > 0).mean() <= MAX_RGB_FRACTION, "%s: %d channels differ" % (what, int((diff > 0).sum()))
    for k in ("rays", "primary", "shadow", "reflect", "refract"):
        if gpu["stats"][k] or k == "rays":
            assert gpu["stats"][k] == cpu["stats"][k], "%s: %s count %d != %d" % (what, k, gpu["stats"][k], cpu["stats"][k])


def test_c1_full_frame(product_lib, oracle_mod, scene_dir):
    """BASELINE config C1 (2k triangles, 320x240, 1 light, depth 2), every tap compared."""
    from mythtracer_b200 import MTB_FLAG_COUNT_WORK
    files, cfg = scenes.config_scene("C1", scene_dir)
    mt, orc = _load_pair(product_lib, oracle_mod, files, cfg["depth"], MTB_FLAG_COUNT_WORK)
    w, h = cfg["width"], cfg["height"]
    gpu = mt.render_chunk(files.camera, w, h, 0, 0, w, h, debug=True, taps=True)
    cpu = orc.render(files.camera, w, h, depth=cfg["depth"], taps=True)
    _assert_render_equal(gpu, cpu, "C1")
    assert gpu["stats"]["n_shade"] == cpu["stats"]["n_shade"]
    # the fast build (no counters) must give the same bytes
    from mythtracer_b200 import MTB_FLAG_MEGAKERNEL
    mt.set_flags(MTB_FLAG_MEGAKERNEL)
    fast = mt.render_chunk(files.camera, w, h, 0, 0, w, h)
    assert np.array_equal(fast["rgb"], gpu["rgb"])
    assert fast["stats"]["rays"] == cpu["stats"]["rays"]
    mt.set_flags(0)  # automatic choice: same bytes
    auto = mt.render_chunk(files.camera, w, h, 0, 0, w, h)
    assert np.array_equal(auto["rgb"], gpu["rgb"]) and auto["stats"]["rays"] == cpu["stats"]["rays"]


def test_c1_depths_and_lights(product_lib, oracle_mod, scene_dir):
    """Recursion depth 0..8 and 0..4 lights (main_local.cc's four-light rig) on the C1 scene."""
    from mythtracer_b200 import Light
    files, cfg = scenes.config_scene("C1", scene_dir)
    mt, orc = _load_pair(product_lib, oracle_mod, files, 5)
    w, h = 160, 120
    for depth, n_lights in [(0, 1), (1, 2), (3, 0), (5, 4), (8, 3)]:
        lights = scenes.LIGHT_RIG[:n_lights]
        mt.max_depth = depth
        mt.GetScene().lights = [Light.from_tuple(l) for l in lights]
        orc.set_lights(lights)
        gpu = mt.render_chunk(files.camera, w, h, 0, 0, w, h, debug=True, taps=True)
        cpu = orc.render(files.camera, w, h, depth=depth, taps=True)
        _assert_render_equal(gpu, cpu, "C1 depth %d lights %d" % (depth, n_lights))


def test_c2_textured(product_lib, oracle_mod, scene_dir):
    """BASELINE config C2 (100k triangles, map_Ka textures, 2 lights, depth 3) at a test-size resolution."""
    files, cfg = scenes.config_scene("C2", scene_dir)
    mt, orc = _load_pair(product_lib, oracle_mod, files, cfg["depth"])
    w, h = 320, 180
    gpu = mt.render_chunk(files.camera, w, h, 0, 0, w, h, debug=True, taps=True)
    cpu = orc.render(files.camera, w, h, depth=cfg["depth"], taps=True)
    _assert_render_equal(gpu, cpu, "C2")
    info = mt.scene_info()
    assert info["n_textures"] == 3 and info["n_triangles"] == len(orc.tris)


def test_c3_tile_of_full_frame(product_lib, oracle_mod, scene_dir):
    """BASELINE config C3 (500k triangles, depth 5): WorkChunk tiles of the 1920x1080 frame
    (main_net_master.cc:24-25 uses 128x128 tiles), compared with the oracle's render of the same tiles."""
    files, cfg = scenes.config_scene("C3", scene_dir)
    mt, orc = _load_pair(product_lib, oracle_mod, files, cfg["depth"])
    W, H = cfg["width"], cfg["height"]
    for (cx, cy, cw, ch) in [(896, 512, 128, 128), (1792, 1024, 128, 56)]:
        gpu = mt.render_chunk(files.camera, W, H, cx, cy, cw, ch, debug=True, taps=True)
        cpu = orc.render(files.camera, W, H, chunk=(cx, cy, cw, ch), depth=cfg["depth"], taps=True)
        _assert_render_equal(gpu, cpu, "C3 tile %d,%d" % (cx, cy))


def test_c3_full_frame_properties(product_lib, oracle_mod, scene_dir):
    """Full BASELINE size (C3, 1920x1080): properties that do not need the oracle to render 2M pixels --
    determinism, tiles == whole frame (the master/worker contract), and a random sample of pixels against the
    oracle rendering them as 1x1 chunks."""
    files, cfg = scenes.config_scene("C3", scene_dir)
    mt, orc = _load_pair(product_lib, oracle_mod, files, cfg["depth"])
    W, H = cfg["width"], cfg["height"]
    full = mt.render_chunk(files.camera, W, H, 0, 0, W, H, debug=True)
    again = mt.render_chunk(files.camera, W, H, 0, 0, W, H)
    assert np.array_equal(full["rgb"], again["rgb"])
    assert full["stats"]["rays"] == again["stats"]["rays"]
    # 128x128 tiles, clipped at the edges (main_net_master.cc:202-217)
    rng = np.random.default_rng(7)
    tiles = [(x, y) for y in range(0, H, 128) for x in range(0, W, 128)]
    for i in rng.choice(len(tiles), 12, replace=False):
        x, y = tiles[i]
        cw, ch = min(128, W - x), min(128, H - y)
        tile = mt.render_chunk(files.camera, W, H, x, y, cw, ch)
        assert np.array_equal(tile["rgb"], full["rgb"][y:y + ch, x:x + cw])
    for _ in range(400):
        x, y = int(rng.integers(0, W)), int(rng.integers(0, H))
        cpu = orc.render(files.camera, W, H, chunk=(x, y, 1, 1), depth=cfg["depth"])
        assert cpu["line_no"][0, 0] == full["line_no"][y, x]
        assert np.array_equal(cpu["points"][0, 0], full["points"][y, x], equal_nan=True)
        assert np.abs(cpu["rgb"][0, 0].astype(int) - full["rgb"][y, x].astype(int)).max() <= MAX_RGB_DIFF


def test_lattice_nan_paths(product_lib, oracle_mod, scene_dir):
    """On-axis camera over integer-lattice boxes: zero direction components, origins on box planes
    (0 * inf = NaN slab tests), shared-edge ties, transparent stacks.  Exercises the literal traversal."""
    from mythtracer_b200 import Light, MTB_FLAG_COUNT_WORK
    path, cam, lights = scenes.lattice_scene(scene_dir)
    mt = _tracer(product_lib, 5, MTB_FLAG_COUNT_WORK)
    assert mt.LoadObj(path)
    mt.GetScene().lights = [Light.from_tuple(l) for l in lights]
    orc = oracle_mod.Oracle.from_obj(path)
    orc.set_lights(lights)
    for (w, h) in [(65, 49), (64, 48)]:   # odd width: the centre column has dir.x == 0 exactly
        gpu = mt.render_chunk(cam, w, h, 0, 0, w, h, debug=True, taps=True)
        cpu = orc.render(cam, w, h, depth=5, taps=True)
        _assert_render_equal(gpu, cpu, "lattice %dx%d" % (w, h))
    assert gpu["stats"]["n_literal"] >= 0
    odd = mt.render_chunk(cam, 65, 49, 0, 0, 65, 49)
    assert odd["stats"]["n_literal"] > 0, "the on-axis column must take the literal traversal"


def test_intersect_rays_random(product_lib, oracle_mod, scene_dir):
    """Batched OctTree::IntersectRay on random interior rays, axis-parallel rays and rays from outside."""
    files, cfg = scenes.config_scene("C2", scene_dir, scale=0.2)
    mt, orc = _load_pair(product_lib, oracle_mod, files, 3)
    rng = np.random.default_rng(11)
    o, d = scenes.random_rays(rng, orc.aabb(), 40000)
    # axis-parallel directions (zero components -> +-inf inverse) and un-normalised directions
    d[:2000] = np.eye(3)[rng.integers(0, 3, 2000)] * rng.choice([-1.0, 1.0], (2000, 1))
    d[2000:4000] *= rng.uniform(0.1, 7.0, (2000, 1))
    o[4000:6000] += 1000.0
    gpu = mt.intersect_rays(o, d)
    cpu = orc.intersect(o, d)
    assert np.array_equal(gpu["tri"], cpu["tri"])
    hit = cpu["tri"] >= 0
    assert hit.sum() > 10000
    assert np.array_equal(gpu["t"][hit], cpu["t"][hit])
    assert np.array_equal(gpu["point"][hit], cpu["point"][hit])


def test_list_bvh_is_transparent(product_lib, oracle_mod, scene_dir):
    """The list-BVH only prunes work: with and without it the results are byte identical."""
    from mythtracer_b200 import MTB_FLAG_COUNT_WORK, MTB_FLAG_MEGAKERNEL, MTB_FLAG_NO_LIST_BVH
    files, cfg = scenes.config_scene("C2", scene_dir, scale=0.2)
    mt, orc = _load_pair(product_lib, oracle_mod, files, 3, MTB_FLAG_COUNT_WORK | MTB_FLAG_MEGAKERNEL)
    w, h = 256, 144
    a = mt.render_chunk(files.camera, w, h, 0, 0, w, h, debug=True, taps=True)
    mt.set_flags(MTB_FLAG_COUNT_WORK | MTB_FLAG_MEGAKERNEL | MTB_FLAG_NO_LIST_BVH)
    b = mt.render_chunk(files.camera, w, h, 0, 0, w, h, debug=True, taps=True)
    for k in ("rgb", "line_no", "n_rays", "sig_hits", "sig_shadow"):
        assert np.array_equal(a[k], b[k]), k
    cpu = orc.render(files.camera, w, h, depth=3, taps=True)
    _assert_render_equal(b, cpu, "no list BVH")
    # without the BVH the traversal does exactly the reference's triangle tests
    assert b["stats"]["n_triaabb"] == cpu["stats"]["n_triaabb"]
    assert b["stats"]["n_mt"] == cpu["stats"]["n_mt"]
    assert b["stats"]["n_hit"] == cpu["stats"]["n_hit"]
    assert a["stats"]["n_triaabb"] < b["stats"]["n_triaabb"]


def test_reference_octtree_known_answers(product_lib):
    """The reference's own octtree_test vectors (octtree_test.cc:14-72, with CacheAABB as the loader does)."""
    from mythtracer_b200 import MythTracer
    from mythtracer_b200.api import MTL_DTYPE, TRI_DTYPE
    tris = np.zeros(2, TRI_DTYPE)
    tris[0]["vertex"] = [1, 1, 0, 1, 0, 0, 0, 0, 0]
    tris[1]["vertex"] = [1, 1, 1, 1, 0, 1, 0, 0, 1]
    tris["material"] = -1
    mt = MythTracer()
    mt.upload(tris, np.zeros(0, MTL_DTYPE))
    r = mt.intersect_rays([[0.9, 0.9, -10.0], [0.9, 0.9, 10.0], [5.0, 5.0, 5.0]],
                          [[0.0, 0.0, 1.0], [0.0, 0.0, -1.0], [0.0, 0.0, 1.0]])
    assert r["tri"].tolist() == [0, 1, -1]
    assert r["t"][0] == 10.0 and r["t"][1] == 9.0
    tri, point, dist = mt.GetScene().tree.IntersectRay([0.9, 0.9, -10.0], [0.0, 0.0, 1.0])
    assert tri == 0 and dist == 10.0 and point.tolist() == [0.9, 0.9, 0.0]


def test_missing_material_and_no_normals(product_lib, oracle_mod, scene_dir):
    """`usemtl` of an unknown name (mtl == nullptr -> grey n.v shading, mythtracer.cc:49-52) and faces
    without normals (zero normal vector, primitive_triangle.cc:60)."""
    from mythtracer_b200 import Light
    text = "mtllib odd.mtl\n"
    text += "v 0 0 5\nv 4 0 5\nv 4 4 5\nv 0 4 5\nv 0 0 9\nv 4 0 9\nv 4 4 9\nv 0 4 9\nvn 0 0 -1\n"
    text += "usemtl matte\nf 1 2 3 \nf 3 4 1 \n"           # no normals
    text += "usemtl does_not_exist\nf 5//1 6//1 7//1 8//1 \n"  # a quad without material, behind
    path = scenes.write_obj(scene_dir + "/odd.obj", text, scenes.BASIC_MTL)
    mt = _tracer(product_lib, 3)
    assert mt.LoadObj(path)
    orc = oracle_mod.Oracle.from_obj(path)
    cam = (2.1, 2.2, -3.0, 0.0, 3.0, 0.0, 100.0)
    for lights in ([], [(2.0, 2.0, 0.0, 0.2, 0.2, 0.2, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0)]):
        mt.GetScene().lights = [Light.from_tuple(l) for l in lights]
        orc.set_lights(lights)
        gpu = mt.render_chunk(cam, 96, 64, 0, 0, 96, 64, debug=True, taps=True)
        cpu = orc.render(cam, 96, 64, depth=3, taps=True)
        _assert_render_equal(gpu, cpu, "odd scene, %d lights" % len(lights))


def test_errors_are_reported(product_lib):
    from mythtracer_b200 import MythTracer, MythTracerError
    mt = MythTracer()
    assert mt.LoadObj("/nonexistent/file.obj") is False
    assert "not found" in mt.last_error()
    assert mt.RayTrace(32, 32, (0, 0, 0, 0, 0, 0, 90)) is None      # no scene
    with pytest.raises(MythTracerError):
        mt.render_chunk((0, 0, 0, 0, 0, 0, 90), 32, 32, 0, 0, 32, 32)


def test_partition_is_the_tile_contract(product_lib, scene_dir):
    """mtb_set_partition: each part renders only its strips of 8 rows and leaves the rest untouched; the union
    of the parts is the single-context frame (the master/worker contract, main_net_master.cc:195-236)."""
    import torch
    from mythtracer_b200 import Light, tiles
    files, cfg = scenes.config_scene("C1", scene_dir)
    W, H = 200, 141   # neither a multiple of 8
    mt = _tracer(product_lib, 2)
    assert mt.LoadObj(files.obj_path)
    mt.GetScene().lights = [Light.from_tuple(l) for l in files.lights]
    full = mt.render_chunk(files.camera, W, H, 0, 0, W, H)["rgb"]
    for world in (2, 3):
        acc = np.zeros_like(full)
        for rank in range(world):
            mt.set_partition(rank, world)
            buf = torch.full((H, W, 3), 9, dtype=torch.uint8, device="cuda")
            mt.push_lights()
            mt.render_device(files.camera, W, H, buf.data_ptr(), torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            got = buf.cpu().numpy()
            rows = tiles.owned_rows(H, rank, world)
            others = sorted(set(range(H)) - set(rows))
            assert np.array_equal(got[rows], full[rows])
            assert (got[others] == 9).all()
            acc[rows] = got[rows]
        assert np.array_equal(acc, full)
    mt.set_partition(0, 1)


def test_golden_fixtures_on_gpu(product_lib):
    """The CUDA path against fixtures produced by the unmodified reference (tests/golden/make_golden.py)."""
    import os
    from mythtracer_b200 import Light
    golden = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    for name in ("room_small", "room_textured", "lattice"):
        z = np.load(os.path.join(golden, name + ".npz"))
        mt = _tracer(product_lib, int(z["depth"]))
        assert mt.LoadObj(os.path.join(golden, name + ".obj")), mt.last_error()
        mt.GetScene().lights = [Light.from_tuple(l) for l in z["lights"].tolist()]
        w, h = int(z["width"]), int(z["height"])
        out = mt.render_chunk(z["camera"].tolist(), w, h, 0, 0, w, h, debug=True)
        assert np.array_equal(out["line_no"], z["line_no"]), name
        np.testing.assert_allclose(out["points"], z["points"], rtol=0, atol=1e-9, equal_nan=True)
        diff = np.abs(out["rgb"].astype(int) - z["rgb"].astype(int))
        assert diff.max() <= MAX_RGB_DIFF and (diff > 0).mean() <= 1e-4, (name, diff.max(), (diff > 0).sum())
        hits = mt.intersect_rays(z["ray_o"], z["ray_d"])
        tris, _ = mt.scene_arrays()
        line_no = np.where(hits["tri"] >= 0, tris["line_no"][np.maximum(hits["tri"], 0)], -1)
        assert np.array_equal(line_no, z["ray_line_no"]), name
        hit = z["ray_line_no"] >= 0
        assert np.array_equal(hits["t"][hit], z["ray_t"][hit])
        assert np.array_equal(hits["point"][hit], z["ray_point"][hit])


def test_multi_device_context(product_lib, scene_dir):
    """In-process multi-GPU: strips interleaved over the devices of one context, gathered by peer copies;
    the frame must be byte-identical to the single-GPU frame, through either pipeline."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from mythtracer_b200 import Light, MTB_FLAG_MEGAKERNEL, MTB_FLAG_QUEUE
    files, cfg = scenes.config_scene("C1", scene_dir)
    W, H = 320, 243
    one = _tracer(product_lib, 2)
    assert one.LoadObj(files.obj_path)
    one.GetScene().lights = [Light.from_tuple(l) for l in files.lights]
    ref = one.render_chunk(files.camera, W, H, 0, 0, W, H, debug=True, taps=True)
    n = min(torch.cuda.device_count(), 8)
    for flags in (MTB_FLAG_MEGAKERNEL, MTB_FLAG_QUEUE):
        many = _tracer(product_lib, 2, flags, devices=list(range(n)))
        assert many.LoadObj(files.obj_path)
        many.GetScene().lights = [Light.from_tuple(l) for l in files.lights]
        got = many.render_chunk(files.camera, W, H, 0, 0, W, H, debug=True, taps=True)
        for k in ("rgb", "line_no", "points", "n_rays", "sig_hits", "sig_shadow"):
            assert np.array_equal(got[k], ref[k], equal_nan=(k == "points")), (flags, k)
        assert got["stats"]["rays"] == ref["stats"]["rays"]
        many.close()


@pytest.mark.parametrize("name,scale,w,h", [("C1", 1.0, 320, 240), ("C2", 0.3, 256, 144)])
def test_queue_pipeline_parity(product_lib, oracle_mod, scene_dir, name, scale, w, h):
    """The queue pipeline (MTB_FLAG_QUEUE: one persistent kernel over a single ray queue) against the oracle, every
    tap, in the plain and the counting build, and against the megakernel's bytes."""
    from mythtracer_b200 import MTB_FLAG_COUNT_WORK, MTB_FLAG_MEGAKERNEL, MTB_FLAG_QUEUE
    files, cfg = scenes.config_scene(name, scene_dir, scale)
    mt, orc = _load_pair(product_lib, oracle_mod, files, cfg["depth"], MTB_FLAG_QUEUE | MTB_FLAG_COUNT_WORK)
    gpu = mt.render_chunk(files.camera, w, h, 0, 0, w, h, debug=True, taps=True)
    cpu = orc.render(files.camera, w, h, depth=cfg["depth"], taps=True)
    _assert_render_equal(gpu, cpu, name + " queue (counting build)")
    mt.set_flags(MTB_FLAG_QUEUE)
    for it in range(3):  # the epoch of the ready flags moves on from frame to frame
        fast = mt.render_chunk(files.camera, w, h, 0, 0, w, h, debug=True, taps=True)
        _assert_render_equal(fast, cpu, name + " queue frame %d" % it)
    mt.set_flags(MTB_FLAG_MEGAKERNEL)
    mega = mt.render_chunk(files.camera, w, h, 0, 0, w, h)
    assert np.array_equal(fast["rgb"], mega["rgb"]) and np.array_equal(fast["rgb"], gpu["rgb"])
    assert fast["stats"]["rays"] == mega["stats"]["rays"] == cpu["stats"]["rays"]


def test_queue_pipeline_depths_lights_lattice_and_tiles(product_lib, oracle_mod, scene_dir):
    from mythtracer_b200 import Light, MTB_FLAG_QUEUE
    files, cfg = scenes.config_scene("C1", scene_dir)
    mt, orc = _load_pair(product_lib, oracle_mod, files, 5, MTB_FLAG_QUEUE)
    w, h = 160, 120
    for depth, n_lights in [(0, 1), (2, 0), (5, 4), (8, 2)]:
        lights = scenes.LIGHT_RIG[:n_lights]
        mt.max_depth = depth
        mt.GetScene().lights = [Light.from_tuple(l) for l in lights]
        orc.set_lights(lights)
        gpu = mt.render_chunk(files.camera, w, h, 0, 0, w, h, debug=True, taps=True)
        cpu = orc.render(files.camera, w, h, depth=depth, taps=True)
        _assert_render_equal(gpu, cpu, "queue depth %d lights %d" % (depth, n_lights))
    mt.max_depth = 3
    gpu = mt.render_chunk(files.camera, 333, 211, 100, 37, 77, 45, debug=True, taps=True)
    cpu = orc.render(files.camera, 333, 211, chunk=(100, 37, 77, 45), depth=3, taps=True)
    _assert_render_equal(gpu, cpu, "queue tile")
    path, cam, lights = scenes.lattice_scene(scene_dir)
    mt2 = _tracer(product_lib, 5, MTB_FLAG_QUEUE)
    assert mt2.LoadObj(path)
    mt2.GetScene().lights = [Light.from_tuple(l) for l in lights]
    orc2 = oracle_mod.Oracle.from_obj(path)
    orc2.set_lights(lights)
    gpu = mt2.render_chunk(cam, 65, 49, 0, 0, 65, 49, debug=True, taps=True)
    cpu = orc2.render(cam, 65, 49, depth=5, taps=True)
    _assert_render_equal(gpu, cpu, "queue lattice")


def test_megakernel_launch_forms(product_lib, oracle_mod, scene_dir):
    """The megakernel against the oracle, every tap: the plain and the counting build, with and without the
    cost-aware tile order, with the retired flag bits set (accepted and ignored) -- on a full frame, a
    clipped odd-sized tile (rows that cannot leave the block as aligned 8-byte stores), a partitioned render and
    two consecutive frames (warm tile order).  MTB_FLAG_WAVEFRONT is the queue pipeline."""
    from mythtracer_b200 import (MTB_FLAG_COUNT_WORK, MTB_FLAG_HYBRID, MTB_FLAG_MEGAKERNEL, MTB_FLAG_NO_TILE_ORDER, MTB_FLAG_PACKING,
                                 MTB_FLAG_PERSISTENT, MTB_FLAG_QUEUE, MTB_FLAG_RESUME, MTB_FLAG_WARP_SYNC, MTB_FLAG_WAVEFRONT)
    files, cfg = scenes.config_scene("C2", scene_dir, 0.3)
    mt, orc = _load_pair(product_lib, oracle_mod, files, cfg["depth"], MTB_FLAG_MEGAKERNEL)
    w, h = 250, 141
    cpu = orc.render(files.camera, w, h, depth=cfg["depth"], taps=True)
    cpu_tile = orc.render(files.camera, 333, 211, chunk=(100, 37, 77, 45), depth=cfg["depth"], taps=True)
    cpu_w8 = orc.render(files.camera, 256, 100, chunk=(0, 0, 256, 100), depth=cfg["depth"], taps=True)
    for flags in (MTB_FLAG_MEGAKERNEL, MTB_FLAG_MEGAKERNEL | MTB_FLAG_COUNT_WORK, MTB_FLAG_MEGAKERNEL | MTB_FLAG_NO_TILE_ORDER,
                  MTB_FLAG_MEGAKERNEL | MTB_FLAG_PACKING | MTB_FLAG_PERSISTENT | MTB_FLAG_RESUME | MTB_FLAG_WARP_SYNC | MTB_FLAG_HYBRID):
        mt.set_flags(flags)
        for frame in range(2):
            gpu = mt.render_chunk(files.camera, w, h, 0, 0, w, h, debug=True, taps=True)
            _assert_render_equal(gpu, cpu, "flags %d frame %d" % (flags, frame))
        full = gpu["rgb"].copy()
        gpu = mt.render_chunk(files.camera, 333, 211, 100, 37, 77, 45, debug=True, taps=True)
        _assert_render_equal(gpu, cpu_tile, "flags %d tile" % flags)
        # a width that is a multiple of 8 (whole tile rows leave the block as aligned 8-byte stores) with a clipped
        # last strip (100 = 12 * 8 + 4 rows)
        gpu = mt.render_chunk(files.camera, 256, 100, 0, 0, 256, 100, debug=True, taps=True)
        _assert_render_equal(gpu, cpu_w8, "flags %d 256x100" % flags)
        # two partitions of the frame: each fills only its own strips, together they are the frame
        parts = []
        for rank in range(2):
            mt.set_partition(rank, 2)
            parts.append(mt.render_chunk(files.camera, w, h, 0, 0, w, h)["rgb"].copy())
        mt.set_partition(0, 1)
        rows = np.arange(h)
        own0 = ((rows // 8) % 2) == 0
        assert np.array_equal(parts[0][own0], full[own0]) and np.array_equal(parts[1][~own0], full[~own0])
    assert mt.pipeline_in_use()[0] == "mega" and mt.hybrid_share() == 0.0
    outs = {}
    for flags in (MTB_FLAG_QUEUE, MTB_FLAG_WAVEFRONT):
        mt.set_flags(flags)
        outs[flags] = mt.render_chunk(files.camera, w, h, 0, 0, w, h, debug=True, taps=True)
        assert mt.pipeline_in_use()[0] == "queue"
        _assert_render_equal(outs[flags], cpu, "flags %d" % flags)
    for k in ("rgb", "line_no", "n_rays", "sig_hits", "sig_shadow"):
        assert np.array_equal(outs[MTB_FLAG_WAVEFRONT][k], outs[MTB_FLAG_QUEUE][k]), k


@pytest.mark.parametrize("pipeline", ["mega", "queue"])
def test_textured_light_terms_in_isolation(product_lib, oracle_mod, scene_dir, pipeline):
    """Ambient-only, diffuse-only and specular-only lights on the textured scene, both pipelines: each Phong
    term (mythtracer.cc:83-84,163-167,169-177) is compared on its own, so a wrong surface colour cannot hide
    behind the other terms.  (A register-capped build of the megakernel once lost one bilinear tap here.)"""
    from mythtracer_b200 import Light, MTB_FLAG_MEGAKERNEL, MTB_FLAG_QUEUE
    files, cfg = scenes.config_scene("C2", scene_dir, 0.1)
    flags = MTB_FLAG_MEGAKERNEL if pipeline == "mega" else MTB_FLAG_QUEUE
    mt, orc = _load_pair(product_lib, oracle_mod, files, 2, flags)
    w, h = 200, 112
    pos = (200.0, 100.0, 160.0)
    zero, one = (0.0, 0.0, 0.0), (1.0, 1.0, 1.0)
    for amb, dif, spe in [(one, zero, zero), (zero, one, zero), (zero, zero, one), ((0.2, 0.3, 0.4), (0.9, 0.8, 0.7), (0.5, 0.6, 0.7))]:
        rig = [pos + amb + dif + spe, (120.0, 100.0, 250.0) + zero + dif + spe]
        mt.GetScene().lights = [Light.from_tuple(l) for l in rig]
        orc.set_lights(rig)
        gpu = mt.render_chunk(files.camera, w, h, 0, 0, w, h, debug=True, taps=True)
        cpu = orc.render(files.camera, w, h, depth=2, taps=True)
        _assert_render_equal(gpu, cpu, "%s terms %s" % (pipeline, (amb, dif, spe)))


def test_automatic_pipeline_choice_decides_at_frame_5(product_lib, oracle_mod, scene_dir):
    """flags = 0: the library times the megakernel and the queue pipeline on the first four frames of a geometry and
    keeps the faster from frame 5 on; every one of those frames must carry the same bytes (the choice is invisible in
    the output)."""
    from mythtracer_b200 import Light, MythTracer
    files, cfg = scenes.config_scene("C1", scene_dir)
    mt = MythTracer(max_depth=cfg["depth"])
    assert mt.LoadObj(files.obj_path)
    mt.GetScene().lights = [Light.from_tuple(l) for l in files.lights]
    orc = oracle_mod.Oracle.from_obj(files.obj_path)
    orc.set_lights(files.lights)
    w, h = 320, 240
    cpu = orc.render(files.camera, w, h, depth=cfg["depth"])
    states = []
    for _ in range(8):
        out = mt.render_chunk(files.camera, w, h, 0, 0, w, h)
        assert np.array_equal(out["rgb"], cpu["rgb"])
        assert out["stats"]["rays"] == cpu["stats"]["rays"]
        states.append(mt.pipeline_in_use()[0])
    assert states[:4] == ["measuring"] * 4 and states[4] in ("mega", "queue") and len(set(states[4:])) == 1
    _, mega_ms, wf_ms = mt.pipeline_in_use()
    assert mega_ms > 0 and wf_ms > 0
    assert states[-1] == ("queue" if wf_ms < mega_ms else "mega")
    # a different geometry starts measuring again
    mt.render_chunk(files.camera, w, h, 0, 0, w // 2, h)
    assert mt.pipeline_in_use()[0] == "measuring"


def _pair_from_loader(product_lib, oracle_mod, files, depth, lights):
    """Product + oracle over the arrays the product loader parsed (a Python re-parse of 2 M faces is slow)."""
    from mythtracer_b200 import Light
    mt = _tracer(product_lib, depth)
    assert mt.LoadObj(files.obj_path), mt.last_error()
    mt.GetScene().lights = [Light.from_tuple(l) for l in lights]
    tris, mtls = mt.scene_arrays()
    orc = oracle_mod.Oracle(tris, mtls, [])
    orc.set_lights(lights)
    return mt, orc


def test_c4_stress_scene_tiles(product_lib, oracle_mod, scene_dir):
    """BASELINE config C4: ~2 M triangles (dense clusters of tiny triangles + long thin sticks that straddle the
    top octree planes), 1920x1080, depth 5 -- WorkChunk tiles against the oracle, plus the octree shape."""
    files, cfg = scenes.config_scene("C4", scene_dir)
    mt, orc = _pair_from_loader(product_lib, oracle_mod, files, cfg["depth"], files.lights)
    info, tree = mt.scene_info(), orc.tree_info()
    assert info["n_triangles"] > 1900000
    assert (info["n_nodes"], info["tree_depth"], info["biggest_list"]) == (tree["nodes"], tree["depth"], tree["biggest_list"])
    W, H = cfg["width"], cfg["height"]
    for (cx, cy, cw, ch) in [(300, 420, 96, 64), (1500, 200, 64, 48)]:
        gpu = mt.render_chunk(files.camera, W, H, cx, cy, cw, ch, debug=True, taps=True)
        cpu = orc.render(files.camera, W, H, chunk=(cx, cy, cw, ch), depth=cfg["depth"], taps=True)
        _assert_render_equal(gpu, cpu, "C4 tile %d,%d" % (cx, cy))


def test_c5_4k_depth8_four_lights_tiles(product_lib, oracle_mod, scene_dir):
    """BASELINE config C5: the 500 k-triangle interior at 3840x2160, 4 lights, depth 8 -- tiles against the oracle
    with both pipelines."""
    from mythtracer_b200 import MTB_FLAG_MEGAKERNEL, MTB_FLAG_QUEUE
    files, cfg = scenes.config_scene("C5", scene_dir)
    assert len(files.lights) == 4 and cfg["depth"] == 8
    mt, orc = _pair_from_loader(product_lib, oracle_mod, files, cfg["depth"], files.lights)
    W, H = cfg["width"], cfg["height"]
    for flags, (cx, cy, cw, ch) in [(MTB_FLAG_MEGAKERNEL, (1800, 1100, 96, 64)), (MTB_FLAG_QUEUE, (2600, 1500, 80, 48))]:
        mt.set_flags(flags)
        gpu = mt.render_chunk(files.camera, W, H, cx, cy, cw, ch, debug=True, taps=True)
        cpu = orc.render(files.camera, W, H, chunk=(cx, cy, cw, ch), depth=cfg["depth"], taps=True)
        _assert_render_equal(gpu, cpu, "C5 tile %d,%d" % (cx, cy))


def test_edge_scenes(product_lib, oracle_mod, scene_dir):
    """Empty scene, a single triangle, zero-area and needle triangles, all triangles in one unsplit node, a ray
    batch of size 0 -- both pipelines."""
    from mythtracer_b200 import Light, MythTracer, MTB_FLAG_MEGAKERNEL, MTB_FLAG_QUEUE
    from mythtracer_b200.api import MTL_DTYPE, TRI_DTYPE
    cam = (0.3, 0.4, -6.0, 2.0, 5.0, 1.0, 70.0)
    lights = [(1.0, 5.0, -4.0, 0.2, 0.2, 0.2, 1.0, 1.0, 1.0, 0.8, 0.8, 0.8)]
    mtl = np.zeros(1, MTL_DTYPE)
    mtl["ambient"], mtl["diffuse"], mtl["specular"] = (0.4, 0.5, 0.6), (0.7, 0.6, 0.5), (0.5, 0.5, 0.5)
    mtl["specular_exp"], mtl["reflectance"], mtl["transparency"], mtl["texture"] = 30.0, 0.4, 0.3, -1
    mtl["transmission_filter"] = (0.9, 0.8, 0.7)
    rng = np.random.default_rng(2)
    cases = {"empty": np.zeros(0, TRI_DTYPE)}
    one = np.zeros(1, TRI_DTYPE)
    one["vertex"] = [-3, -3, 2, 4, -3, 2.5, 0, 4, 3]
    one["normal"] = [0, 0, -1, 0.1, 0, -1, 0, 0.1, -1]
    cases["single"] = one
    few = np.zeros(15, TRI_DTYPE)   # below SPLIT_BOUNDARY: the root is never split; includes degenerate triangles
    few["vertex"] = rng.uniform(-3, 3, (15, 9))
    few["normal"] = rng.normal(size=(15, 9))
    few["vertex"][3] = [1, 1, 1, 1, 1, 1, 1, 1, 1]                 # a point
    few["vertex"][4] = [0, 0, 1, 1, 1, 2, 2, 2, 3]                 # collinear
    few["vertex"][5][3:] = few["vertex"][5][:6] + 1e-9             # a needle
    cases["few"] = few
    for name, tris in cases.items():
        tris["material"] = 0
        tris["line_no"] = np.arange(len(tris))
        orc = oracle_mod.Oracle(tris, mtl, [])
        orc.set_lights(lights)
        cpu = orc.render(cam, 96, 64, depth=4, taps=True)
        for flags in (MTB_FLAG_MEGAKERNEL, MTB_FLAG_QUEUE):
            mt = MythTracer(max_depth=4, flags=flags)
            mt.upload(tris, mtl)
            mt.GetScene().lights = [Light.from_tuple(l) for l in lights]
            gpu = mt.render_chunk(cam, 96, 64, 0, 0, 96, 64, debug=True, taps=True)
            _assert_render_equal(gpu, cpu, "%s flags %d" % (name, flags))
            r = mt.intersect_rays(np.zeros((0, 3)), np.zeros((0, 3)))
            assert len(r["tri"]) == 0


def test_fast_traversal_and_exact_octree_agree(product_lib, oracle_mod, scene_dir):
    """Regular rays are answered by the certified fast traversal (scene BVH, DESIGN.md section 4) by default and
    by the exact octree recursion under MTB_FLAG_EXACT_OCTREE.  Both against the oracle, every tap, both pipelines,
    on C1 (full frame), textured C2 and a C3 tile; the counters must show which traversal ran."""
    from mythtracer_b200 import MTB_FLAG_COUNT_WORK, MTB_FLAG_EXACT_OCTREE, MTB_FLAG_MEGAKERNEL, MTB_FLAG_QUEUE
    for name, scale, (W, H), chunk in [("C1", 1.0, (320, 240), (0, 0, 320, 240)), ("C2", 0.3, (320, 180), (0, 0, 320, 180)),
                                        ("C3", 0.2, (1920, 1080), (900, 500, 128, 64))]:
        files, cfg = scenes.config_scene(name, scene_dir, scale)
        mt, orc = _load_pair(product_lib, oracle_mod, files, cfg["depth"], MTB_FLAG_MEGAKERNEL)
        cpu = orc.render(files.camera, W, H, chunk=chunk, depth=cfg["depth"], taps=True)
        for pipe in (MTB_FLAG_MEGAKERNEL, MTB_FLAG_QUEUE):
            for exact in (0, MTB_FLAG_EXACT_OCTREE):
                mt.set_flags(pipe | exact | MTB_FLAG_COUNT_WORK)
                gpu = mt.render_chunk(files.camera, W, H, *chunk, debug=True, taps=True)
                _assert_render_equal(gpu, cpu, "%s pipe %d exact %d" % (name, pipe, exact))
                st = gpu["stats"]
                assert st["n_fast"] + st["n_fallback"] + st["n_literal"] == st["rays"] or exact
                if exact:
                    assert st["n_fast"] == 0 and st["n_fallback"] == 0
                else:
                    assert st["n_fast"] > 0.99 * st["rays"], "the fast traversal should answer nearly every ray"
                mt.set_flags(pipe | exact)
                fast = mt.render_chunk(files.camera, W, H, *chunk)
                assert np.array_equal(fast["rgb"], gpu["rgb"])


def test_ambiguous_hits_fall_back_to_the_exact_recursion(product_lib, oracle_mod, scene_dir):
    """Coincident triangles (exact ties in t: the reference's list order decides, octtree.cc:186-195), triangles that
    differ by 1e-13 (hits inside each other's error bound) and a grazing, ill-conditioned triangle: the fast
    traversal must declare these rays ambiguous and the exact recursion must give the reference's answer."""
    from mythtracer_b200 import Light, MythTracer, MTB_FLAG_COUNT_WORK, MTB_FLAG_MEGAKERNEL, MTB_FLAG_QUEUE
    from mythtracer_b200.api import MTL_DTYPE, TRI_DTYPE
    cam = (0.3, 0.4, -6.0, 2.0, 5.0, 1.0, 70.0)
    lights = [(1.0, 5.0, -4.0, 0.2, 0.2, 0.2, 1.0, 1.0, 1.0, 0.8, 0.8, 0.8)]
    mtl = np.zeros(3, MTL_DTYPE)
    for i, ka in enumerate([(0.9, 0.1, 0.1), (0.1, 0.9, 0.1), (0.1, 0.1, 0.9)]):
        mtl["ambient"][i], mtl["diffuse"][i], mtl["specular"][i] = ka, (0.5, 0.5, 0.5), (0.3, 0.3, 0.3)
        mtl["specular_exp"][i], mtl["texture"][i] = 20.0, -1
    mtl["transparency"][2], mtl["transmission_filter"][2], mtl["reflectance"][1] = 0.5, (0.9, 0.9, 0.9), 0.5
    rng = np.random.default_rng(7)
    base = np.zeros(40, TRI_DTYPE)
    base["vertex"] = rng.uniform(-4, 4, (40, 9))
    base["vertex"][:, 2::3] += 3.0
    base["normal"] = rng.normal(size=(40, 9))
    tris = np.concatenate([base, base, base])           # every triangle three times: exact ties everywhere
    tris["vertex"][80:] += 1e-13                         # the third copy is displaced by less than the error bound
    tris["material"] = np.repeat([0, 1, 2], 40)
    graze = np.zeros(1, TRI_DTYPE)                       # nearly edge-on from the camera: tiny determinant
    graze["vertex"] = [0.3, 0.4, -5.0, 0.3 + 1e-7, 3.0, 6.0, 0.3 - 1e-7, -3.0, 6.0]
    graze["normal"] = [1, 0, 0] * 3
    tris = np.concatenate([tris, graze])
    tris["line_no"] = np.arange(len(tris))
    orc = oracle_mod.Oracle(tris, mtl, [])
    orc.set_lights(lights)
    cpu = orc.render(cam, 128, 96, depth=3, taps=True)
    for flags in (MTB_FLAG_MEGAKERNEL, MTB_FLAG_QUEUE):
        mt = MythTracer(max_depth=3, flags=flags | MTB_FLAG_COUNT_WORK)
        mt.upload(tris, mtl)
        mt.GetScene().lights = [Light.from_tuple(l) for l in lights]
        gpu = mt.render_chunk(cam, 128, 96, 0, 0, 128, 96, debug=True, taps=True)
        _assert_render_equal(gpu, cpu, "ties flags %d" % flags)
        assert gpu["stats"]["n_fallback"] > 0, "tied hits must be handed to the exact recursion"
    # the same through the batched OctTree::IntersectRay
    o = np.tile(np.array(cam[:3]), (2000, 1))
    d = rng.normal(size=(2000, 3))
    d[:, 2] = np.abs(d[:, 2]) + 0.5
    got = mt.intersect_rays(o, d)
    ref = orc.intersect(o, d)
    assert np.array_equal(got["tri"], ref["tri"])
    hit = got["tri"] >= 0
    assert hit.sum() > 100 and np.array_equal(got["t"][hit], ref["t"][hit])


def test_fast_traversal_equals_exact_octree_at_full_size(product_lib, scene_dir):
    """BASELINE sizes: the certified fast traversal and the exact octree recursion (MTB_FLAG_EXACT_OCTREE) must give
    the same bytes and the same taps (hit ids, hit points, per-pixel ray counts, secondary-hit and shadow-decision
    signatures) on the whole C3 frame (22.5 M rays), on a 4K band of C5 (depth 8, 4 lights) and on a tile of the C4
    stress scene; the number of rays that needed the exact recursion is reported by the counters."""
    from mythtracer_b200 import MTB_FLAG_COUNT_WORK, MTB_FLAG_EXACT_OCTREE, MTB_FLAG_MEGAKERNEL, MTB_FLAG_QUEUE
    for name, chunk in [("C3", None), ("C5", (0, 1000, 3840, 96)), ("C4", (800, 500, 160, 64))]:
        files, cfg = scenes.config_scene(name, scene_dir)
        W, H = cfg["width"], cfg["height"]
        chunk = chunk or (0, 0, W, H)
        from mythtracer_b200 import Light
        mt = _tracer(product_lib, cfg["depth"], MTB_FLAG_MEGAKERNEL | MTB_FLAG_EXACT_OCTREE)
        assert mt.LoadObj(files.obj_path), mt.last_error()
        mt.GetScene().lights = [Light.from_tuple(l) for l in files.lights]
        exact = mt.render_chunk(files.camera, W, H, *chunk, debug=True, taps=True)
        for pipe in (MTB_FLAG_MEGAKERNEL, MTB_FLAG_QUEUE):
            mt.set_flags(pipe | MTB_FLAG_COUNT_WORK)
            fast = mt.render_chunk(files.camera, W, H, *chunk, debug=True, taps=True)
            for k in ("rgb", "line_no", "points", "n_rays", "sig_hits", "sig_shadow"):
                assert np.array_equal(fast[k], exact[k], equal_nan=(k == "points")), "%s pipe %d: %s differs" % (name, pipe, k)
            st = fast["stats"]
            assert st["rays"] == exact["stats"]["rays"]
            assert st["n_fast"] + st["n_fallback"] + st["n_literal"] == st["rays"]
            assert st["n_fallback"] < 1e-4 * st["rays"], "%s: %d rays fell back" % (name, st["n_fallback"])
        mt.close()


def test_sibling_entry_tie_on_the_device(product_lib, oracle_mod):
    """Round 1's stated edge case (a), closed: for the constructed ray through an octree grid edge
    (tests/test_certification_math.py has the construction and the reference's side of it) the reference returns the
    FARTHER triangle (octtree.cc:244-246 stops behind a sibling whose entry distance ties).  The default traversal
    must return exactly that -- the winner of its closest-hit search lies in an octree node the ray only touches
    (DegeneratePassage, device_core.cuh), so the ray is handed to the exact recursion -- as must MTB_FLAG_EXACT_OCTREE."""
    from mythtracer_b200 import MythTracer, MTB_FLAG_COUNT_WORK, MTB_FLAG_EXACT_OCTREE
    from mythtracer_b200.api import MTL_DTYPE, TRI_DTYPE
    tris = []

    def tri(a, b, c):
        tris.append([*a, *b, *c])
    tri((1, 3, 1.0), (3, 1, 1.0), (2.2, 2.2, 3.9))
    tri((4, 4, 2.0), (4, 4, 3.25), (6, 2, 2.5))
    tri((0, 0, 0), (0.3, 0, 0), (0, 0.3, 0))
    tri((8, 8, 8), (7.7, 8, 8), (8, 7.7, 8))
    rng = np.random.default_rng(1)
    for _ in range(14):
        c = np.array([6.5, 1.0, 6.5]) + rng.uniform(-0.4, 0.4, 3)
        tri(c, c + [0.2, 0, 0], c + [0, 0.2, 0])
    arr = np.zeros(len(tris), TRI_DTYPE)
    arr["vertex"] = np.array(tris, float)
    arr["material"] = -1
    arr["line_no"] = np.arange(len(tris))
    # the tie ray, and two neighbours of it that pass the grid edge at a distance (no tie: the nearer triangle wins)
    o = np.array([[7.0, 7.0, 3.0], [7.0, 7.0, 3.0], [7.0, 7.0, 3.0]])
    d = np.array([[-1.0, -1.0, -0.125], [-1.0, -0.99, -0.125], [-0.99, -1.0, -0.125]])
    ref = oracle_mod.Oracle(arr, np.zeros(0, MTL_DTYPE), []).intersect(o, d)
    assert ref["tri"][0] == 0
    for flags in (MTB_FLAG_EXACT_OCTREE, 0, MTB_FLAG_COUNT_WORK):
        mt = MythTracer(flags=flags)
        mt.upload(arr, np.zeros(0, MTL_DTYPE))
        got = mt.intersect_rays(o, d, want_stats=True)
        assert np.array_equal(got["tri"], ref["tri"]), (flags, got["tri"], ref["tri"])
        hit = ref["tri"] >= 0
        assert np.array_equal(got["t"][hit], ref["t"][hit])
        if flags == MTB_FLAG_COUNT_WORK:
            assert got["stats"]["n_fallback"] >= 1 and got["stats"]["n_fast"] >= 1
        mt.close()


def test_retired_pair_and_chain_flags_change_nothing(product_lib, oracle_mod, scene_dir):
    """MTB_FLAG_PAIR_RAYS and MTB_FLAG_CHAIN_RAYS (retired two-rays-per-thread forms of mtb_intersect_rays) are accepted and
    ignored: the answers match the oracle and, with the integer stats, the same call without the two bits.  Random rays,
    axis-parallel ones (literal path), rays from outside, and an odd count."""
    from mythtracer_b200 import MTB_FLAG_CHAIN_RAYS, MTB_FLAG_COUNT_WORK, MTB_FLAG_PAIR_RAYS
    files, cfg = scenes.config_scene("C2", scene_dir, scale=0.2)
    mt, orc = _load_pair(product_lib, oracle_mod, files, 3)
    rng = np.random.default_rng(12)
    o, d = scenes.random_rays(rng, orc.aabb(), 20001)
    d[:1000] = np.eye(3)[rng.integers(0, 3, 1000)] * rng.choice([-1.0, 1.0], (1000, 1))
    o[1000:2000] += 1000.0
    cpu = orc.intersect(o, d)
    hit = cpu["tri"] >= 0
    assert hit.sum() > 5000
    plain = {}
    for flags in (0, MTB_FLAG_COUNT_WORK):
        mt.set_flags(flags)
        plain[flags] = mt.intersect_rays(o, d, want_stats=True)
    for flags in (MTB_FLAG_PAIR_RAYS, MTB_FLAG_PAIR_RAYS | MTB_FLAG_COUNT_WORK, MTB_FLAG_CHAIN_RAYS, MTB_FLAG_CHAIN_RAYS | MTB_FLAG_COUNT_WORK,
                  MTB_FLAG_CHAIN_RAYS | MTB_FLAG_PAIR_RAYS):
        mt.set_flags(flags)
        gpu = mt.intersect_rays(o, d, want_stats=True)
        assert np.array_equal(gpu["tri"], cpu["tri"]), flags
        assert np.array_equal(gpu["t"][hit], cpu["t"][hit]), flags
        assert np.array_equal(gpu["point"][hit], cpu["point"][hit]), flags
        assert np.isnan(gpu["t"][~hit]).all()
        if flags & MTB_FLAG_COUNT_WORK:
            assert gpu["stats"]["rays"] == len(o) and gpu["stats"]["n_literal"] >= 1000
        ref = plain[flags & MTB_FLAG_COUNT_WORK]
        for k in ("tri", "t", "point"):
            assert np.array_equal(gpu[k], ref[k], equal_nan=True), (flags, k)
        assert {k: v for k, v in gpu["stats"].items() if isinstance(v, int)} == {k: v for k, v in ref["stats"].items() if isinstance(v, int)}, flags
