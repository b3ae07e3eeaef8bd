"""Full-size parity on the GPU against fixtures the UNMODIFIED reference produced (tests/golden/full_*.npz, made by
tests/golden/make_golden_full.py in the build container with oracle/_ref):

* C3 (the configuration the headline metric is quoted on): the WHOLE 1920x1080 frame -- every primary hit id and
  every RGB byte (RGB within the stated pow() tolerance, in practice 0 differing bytes), for every pipeline;
* C2 (textured, 720p), C4 (2 M triangles incl. the room-spanning sticks that the scene BVH references through
  several pre-split pieces) and C5 (4K, depth 8, 4 lights, 160 M rays): the whole frame as well.

Plus the paths that only matter at scale: a queue-pipeline frame whose activation table overflows (repaired on the
device, taps and counters exact), and frames shared between processes (tiles stored straight into another process's frame).
"""
import hashlib
import multiprocessing as mp
import os

import numpy as np
import pytest

from tests import scenes

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
MAX_RGB_DIFF = 1
MAX_RGB_FRACTION = 1e-5


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _file_sha(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for blk in iter(lambda: f.read(1 << 20), b""):
            h.update(blk)
    return h.hexdigest()


def _golden(name, scene_dir):
    path = os.path.join(HERE, "golden", "full_%s.npz" % name)
    if not os.path.exists(path):
        pytest.fail("missing fixture %s (python tests/golden/make_golden_full.py %s)" % (path, name))
    z = np.load(path)
    files, cfg = scenes.config_scene(name, scene_dir)
    # the scene generator is seeded; the fixture belongs to exactly these bytes
    assert _file_sha(files.obj_path) == str(z["obj_sha256"]), "generated %s scene differs from the fixture's scene" % name
    assert _file_sha(files.mtl_path) == str(z["mtl_sha256"])
    assert int(z["width"]) == cfg["width"] and int(z["height"]) == cfg["height"] and int(z["depth"]) == cfg["depth"]
    return z, files, cfg


def _compare(got_rgb, got_line_no, z, what):
    rows = z["rows"]
    assert np.array_equal(got_line_no[rows], z["line_no"]), "%s: %d primary hit ids differ from the reference" % (
        what, int((got_line_no[rows] != z["line_no"]).sum()))
    diff = np.abs(got_rgb[rows].astype(np.int16) - z["rgb"].astype(np.int16))
    assert diff.max() <= MAX_RGB_DIFF, "%s: max RGB error %d" % (what, diff.max())
    assert (diff > 0).mean() <= MAX_RGB_FRACTION, "%s: %d channels differ" % (what, int((diff > 0).sum()))
    return int((diff > 0).sum())


def test_c3_full_frame_equals_the_reference(product_lib, scene_dir):
    """Every pixel of the 1920x1080 C3 frame against the reference's own render: megakernel and queue pipeline."""
    from mythtracer_b200 import Light, MythTracer, MTB_FLAG_MEGAKERNEL, MTB_FLAG_QUEUE
    z, files, cfg = _golden("C3", scene_dir)
    W, H = cfg["width"], cfg["height"]
    assert len(z["rows"]) == H
    mt = MythTracer(max_depth=cfg["depth"], flags=MTB_FLAG_MEGAKERNEL)
    assert mt.LoadObj(files.obj_path), mt.last_error()
    mt.GetScene().lights = [Light.from_tuple(l) for l in files.lights]
    shas = set()
    for name, flags in (("megakernel", MTB_FLAG_MEGAKERNEL), ("queue", MTB_FLAG_QUEUE)):
        mt.set_flags(flags)
        for frame in range(2):  # (the second frame: warm tile order)
            got = mt.render_chunk(files.camera, W, H, 0, 0, W, H, debug=True)
        differing = _compare(got["rgb"], got["line_no"], z, "C3 " + name)
        assert _sha(got["line_no"]) == str(z["line_no_sha256"])
        assert _sha(got["points"]) == str(z["points_sha256"]), "C3 %s: hit points differ from the reference's" % name
        if differing == 0:
            assert _sha(got["rgb"]) == str(z["rgb_sha256"])
        shas.add(_sha(got["rgb"]))
    assert len(shas) == 1, "the pipelines disagree with each other"
    mt.close()


def test_c2_textured_full_frame_equals_the_reference(product_lib, scene_dir):
    """Every pixel of the textured 1280x720 C2 frame (depth 3, bilinear texture fetches in every shaded hit) against the
    reference's own render, megakernel and queue pipeline."""
    from mythtracer_b200 import Light, MythTracer, MTB_FLAG_MEGAKERNEL, MTB_FLAG_QUEUE
    z, files, cfg = _golden("C2", scene_dir)
    W, H = cfg["width"], cfg["height"]
    assert len(z["rows"]) == H
    mt = MythTracer(max_depth=cfg["depth"], flags=MTB_FLAG_MEGAKERNEL)
    assert mt.LoadObj(files.obj_path), mt.last_error()
    assert mt.scene_info()["n_textures"] > 0
    mt.GetScene().lights = [Light.from_tuple(l) for l in files.lights]
    for name, flags in (("megakernel", MTB_FLAG_MEGAKERNEL), ("queue", MTB_FLAG_QUEUE)):
        mt.set_flags(flags)
        for frame in range(2):
            got = mt.render_chunk(files.camera, W, H, 0, 0, W, H, debug=True)
        differing = _compare(got["rgb"], got["line_no"], z, "C2 " + name)
        assert _sha(got["points"]) == str(z["points_sha256"]), "C2 %s: hit points differ from the reference's" % name
        if differing == 0:
            assert _sha(got["rgb"]) == str(z["rgb_sha256"])
    mt.close()


@pytest.mark.parametrize("name", ["C4", "C5"])
def test_c4_c5_full_frames_equal_the_reference(product_lib, scene_dir, name):
    """The whole C4 and C5 frames against the reference's render, megakernel and queue pipeline."""
    from mythtracer_b200 import Light, MythTracer, MTB_FLAG_MEGAKERNEL, MTB_FLAG_QUEUE
    z, files, cfg = _golden(name, scene_dir)
    W, H = cfg["width"], cfg["height"]
    assert len(z["rows"]) >= 0.05 * H
    assert len(z["rows"]) == H
    mt = MythTracer(max_depth=cfg["depth"], flags=MTB_FLAG_MEGAKERNEL)
    assert mt.LoadObj(files.obj_path), mt.last_error()
    mt.GetScene().lights = [Light.from_tuple(l) for l in files.lights]
    for pipeline, flags in (("megakernel", MTB_FLAG_MEGAKERNEL), ("queue", MTB_FLAG_QUEUE)):
        mt.set_flags(flags)
        got = mt.render_chunk(files.camera, W, H, 0, 0, W, H, debug=True)
        _compare(got["rgb"], got["line_no"], z, "%s %s" % (name, pipeline))
        assert _sha(got["points"][z["rows"]]) == str(z["points_sha256"]), "%s %s: hit points" % (name, pipeline)
    mt.close()


def test_wavefront_queue_overflow_is_repaired_on_the_device(product_lib, oracle_mod, scene_dir, monkeypatch):
    """An activation table sized for one ray per pixel overflows at the first bounce of a reflective + transparent
    scene: the frame must still be exact in every tap and counter (the repair launch renders it), and the table must
    have grown by the time a later frame goes through the queue pipeline's kernels themselves."""
    from mythtracer_b200 import Light, MythTracer, MTB_FLAG_COUNT_WORK, MTB_FLAG_QUEUE
    monkeypatch.setenv("MTB_WF_ACT_FACTOR", "1")
    files, cfg = scenes.config_scene("C1", scene_dir)
    w, h = 200, 120
    orc = oracle_mod.Oracle.from_obj(files.obj_path)
    orc.set_lights(files.lights)
    cpu = orc.render(files.camera, w, h, depth=4, taps=True)
    assert cpu["stats"]["reflect"] + cpu["stats"]["refract"] > 0
    for flags in (MTB_FLAG_QUEUE, MTB_FLAG_QUEUE | MTB_FLAG_COUNT_WORK):
        mt = MythTracer(max_depth=4, flags=flags)
        assert mt.LoadObj(files.obj_path), mt.last_error()
        mt.GetScene().lights = [Light.from_tuple(l) for l in files.lights]
        for frame in range(5):
            gpu = mt.render_chunk(files.camera, w, h, 0, 0, w, h, debug=True, taps=True)
            for k in ("line_no", "n_rays", "sig_hits", "sig_shadow"):
                assert np.array_equal(gpu[k], cpu[k]), "frame %d: %s" % (frame, k)
            assert np.array_equal(gpu["points"], cpu["points"], equal_nan=True)
            assert np.abs(gpu["rgb"].astype(int) - cpu["rgb"].astype(int)).max() <= MAX_RGB_DIFF
            for k in ("rays", "shadow", "reflect", "refract") if flags & MTB_FLAG_COUNT_WORK else ("rays",):
                assert gpu["stats"][k] == cpu["stats"][k], "frame %d: %s %d != %d" % (frame, k, gpu["stats"][k], cpu["stats"][k])
        mt.close()


def _shared_frame_worker(rank, world, obj_path, camera, lights, w, h, depth, conn):
    import torch  # noqa: F401  (initialises CUDA the way the other tests do)
    from mythtracer_b200 import Light, MythTracer, MTB_FLAG_MEGAKERNEL
    try:
        mt = MythTracer(max_depth=depth, flags=MTB_FLAG_MEGAKERNEL)
        assert mt.LoadObj(obj_path), mt.last_error()
        mt.GetScene().lights = [Light.from_tuple(l) for l in lights]
        mt.push_lights()
        mt.set_partition(rank, world)
        handle = conn.recv()
        ptr = mt.frame_open(handle)
        mt.render_device(camera, w, h, ptr, 0)
        mt.wait()
        mt.frame_release(ptr)
        mt.close()
        conn.send("done")
    except Exception as e:  # pragma: no cover
        conn.send("error: %r" % (e,))


def test_tiles_stored_into_another_process_frame(product_lib, scene_dir):
    """One process per partition (the torchrun form): the other process maps this process's frame (mtb_frame_open)
    and its kernels store the strips it owns straight into it; the result must be the single-process frame."""
    from mythtracer_b200 import Light, MythTracer, MTB_FLAG_MEGAKERNEL
    files, cfg = scenes.config_scene("C1", scene_dir)
    w, h, depth = 320, 240, 2
    mt = MythTracer(max_depth=depth, flags=MTB_FLAG_MEGAKERNEL)
    assert mt.LoadObj(files.obj_path), mt.last_error()
    mt.GetScene().lights = [Light.from_tuple(l) for l in files.lights]
    mt.push_lights()
    ref = mt.render_chunk(files.camera, w, h, 0, 0, w, h)["rgb"]
    ptr, handle = mt.frame_create(w * h * 3)
    ctx = mp.get_context("spawn")
    parent, child = ctx.Pipe()
    proc = ctx.Process(target=_shared_frame_worker, args=(1, 2, files.obj_path, files.camera, files.lights, w, h, depth, child))
    proc.start()
    parent.send(handle)
    mt.set_partition(0, 2)
    mt.render_device(files.camera, w, h, ptr, 0)
    mt.wait()
    assert parent.poll(300), "the second process did not answer"
    msg = parent.recv()
    proc.join(60)
    assert msg == "done", msg
    got = mt.frame_read(ptr, w * h * 3).reshape(h, w, 3)
    assert np.array_equal(got, ref)
    mt.frame_release(ptr)
    mt.close()


def test_device_built_scene_bvh(product_lib, oracle_mod, scene_dir):
    """SURVEY section 8 f1: with MTB_FLAG_DEVICE_BVH the scene BVH is built ON the device (PLOC,
    csrc/device_build.cu).  The tree read back from the device must have the properties the certified traversal
    relies on (every triangle referenced, child boxes contain what is below them, split references cover their
    triangle); a render over it must be the oracle's, and the same bytes as over the host-built tree - which tree is
    walked can only change the speed.  (The full-size C3 frame over the device-built tree is compared with the
    reference's render in test_c3_device_built_tree_equals_the_reference.)"""
    from mythtracer_b200 import Light, MythTracer, MTB_FLAG_DEVICE_BVH, MTB_FLAG_MEGAKERNEL
    from tests.bvh_check import check_scene_bvh
    for name, scale in (("C1", 1.0), ("C4", 0.02)):
        files, cfg = scenes.config_scene(name, scene_dir, scale)
        mt = MythTracer(max_depth=cfg["depth"], flags=MTB_FLAG_MEGAKERNEL | MTB_FLAG_DEVICE_BVH)
        assert mt.LoadObj(files.obj_path), mt.last_error()
        timing = mt.load_timing()
        assert timing["scene_bvh_on_device"] and timing["scene_bvh_device_ms"] > 0.0
        check_scene_bvh(mt, mt.scene_arrays()[0], expect_splits=True)
        mt.GetScene().lights = [Light.from_tuple(l) for l in files.lights]
        w, h = 160, 120
        dev = mt.render_chunk(files.camera, w, h, 0, 0, w, h, debug=True, taps=True)
        orc = oracle_mod.Oracle.from_obj(files.obj_path)
        orc.set_lights(files.lights)
        cpu = orc.render(files.camera, w, h, depth=cfg["depth"], taps=True)
        for k in ("line_no", "n_rays", "sig_hits", "sig_shadow"):
            assert np.array_equal(dev[k], cpu[k]), (name, k)
        assert np.abs(dev["rgb"].astype(int) - cpu["rgb"].astype(int)).max() <= MAX_RGB_DIFF
        mt.set_flags(MTB_FLAG_MEGAKERNEL)
        assert not mt.load_timing()["scene_bvh_on_device"]
        host = mt.render_chunk(files.camera, w, h, 0, 0, w, h, debug=True, taps=True)
        for k in ("rgb", "line_no", "n_rays", "sig_hits", "sig_shadow"):
            assert np.array_equal(dev[k], host[k]), (name, k)
        mt.close()


def test_c3_device_built_tree_equals_the_reference(product_lib, scene_dir):
    """The whole C3 frame rendered over the DEVICE-built scene BVH against the reference's own render."""
    from mythtracer_b200 import Light, MythTracer, MTB_FLAG_DEVICE_BVH, MTB_FLAG_MEGAKERNEL
    z, files, cfg = _golden("C3", scene_dir)
    W, H = cfg["width"], cfg["height"]
    mt = MythTracer(max_depth=cfg["depth"], flags=MTB_FLAG_MEGAKERNEL | MTB_FLAG_DEVICE_BVH)
    assert mt.LoadObj(files.obj_path), mt.last_error()
    assert mt.load_timing()["scene_bvh_on_device"]
    mt.GetScene().lights = [Light.from_tuple(l) for l in files.lights]
    got = mt.render_chunk(files.camera, W, H, 0, 0, W, H, debug=True)
    _compare(got["rgb"], got["line_no"], z, "C3 over the device-built tree")
    assert _sha(got["points"]) == str(z["points_sha256"])
    mt.close()
