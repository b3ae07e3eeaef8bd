"""Batches (mtb_render_batch / MythTracer.render_batch): N whole frames, one camera and one light set per view, in one
megakernel launch per device.  Every view must be exactly the frame mtb_render_chunk renders with that camera and those
lights - the path that is pinned to the oracle and to the reference's own frames - and a batch must leave the
single-frame path's state alone."""
import ctypes
import hashlib
import os
import shutil
import subprocess

import numpy as np
import pytest

from tests import scenes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
MAX_RGB_DIFF = 1
MAX_RGB_FRACTION = 1e-5


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _yawed(cam, dyaw):
    c = list(cam)
    c[4] += dyaw
    return tuple(c)


def _tracer(path, depth, flags=0, devices=None):
    from mythtracer_b200 import MythTracer
    mt = MythTracer(devices=devices, max_depth=depth, flags=flags)
    assert mt.LoadObj(path), mt.last_error()
    return mt


def _singles(mt, cams, w, h, light_sets=None):
    """mtb_render_chunk of every view with its own lights (None: the scene's lights)."""
    from mythtracer_b200 import Light
    keep = list(mt.GetScene().lights)
    out = []
    for i, cam in enumerate(cams):
        if light_sets is not None:
            mt.GetScene().lights = [Light.from_tuple(l) for l in light_sets[i]]
        out.append(mt.render_chunk(cam, w, h, 0, 0, w, h))
    mt.GetScene().lights = keep
    return out


def _lights(rows):
    from mythtracer_b200 import Light
    return [Light.from_tuple(l) for l in rows]


# ---------------------------------------------------------------------------------------------- CPU


def test_batch_has_no_cpu_fallback(product_lib):
    from mythtracer_b200 import MythTracer, MythTracerError
    files, cfg = scenes.config_scene("C1", "/tmp/mtb_scenes")
    mt = MythTracer(host_only=True)
    assert mt.LoadObj(files.obj_path)
    with pytest.raises(MythTracerError, match="no CPU fallback"):
        mt.render_batch([files.camera, files.camera], 16, 16)
    with pytest.raises(MythTracerError, match="no CPU fallback"):
        mt.render_batch([files.camera], 16, 16, lights=[_lights(scenes.LIGHT_RIG[:2])])


def test_batch_arguments_are_checked_in_python(product_lib):
    from mythtracer_b200 import MythTracer, MythTracerError
    files, cfg = scenes.config_scene("C1", "/tmp/mtb_scenes")
    mt = MythTracer(host_only=True)
    assert mt.LoadObj(files.obj_path)
    cams = [files.camera, files.camera]
    with pytest.raises(MythTracerError, match="no cameras"):
        mt.render_batch([], 16, 16)
    with pytest.raises(MythTracerError, match="same number of lights"):
        mt.render_batch(cams, 16, 16, lights=[_lights(scenes.LIGHT_RIG[:2]), _lights(scenes.LIGHT_RIG[:1])])
    with pytest.raises(MythTracerError, match="one per view"):
        mt.render_batch(cams, 16, 16, lights=[_lights(scenes.LIGHT_RIG[:2])])
    with pytest.raises(MythTracerError, match="out must be"):
        mt.render_batch(cams, 16, 16, out=np.zeros((2, 16, 15, 3), np.uint8))


# ---------------------------------------------------------------------------------------------- GPU


@pytest.mark.gpu
def test_views_vary_camera_and_lights(product_lib, oracle_mod, scene_dir):
    """C1 at 150x97 (edge tiles, byte stores), depth 5, five views with their own yaw and their own two lights."""
    from mythtracer_b200 import MTB_FLAG_MEGAKERNEL
    files, cfg = scenes.config_scene("C1", scene_dir)
    w, h, depth = 150, 97, 5
    rig = scenes.LIGHT_RIG
    cams = [_yawed(files.camera, 6.0 * k - 12.0) for k in range(5)]
    light_sets = [[rig[k % 4], rig[(k + 1) % 4]] for k in range(5)]
    mt = _tracer(files.obj_path, depth, MTB_FLAG_MEGAKERNEL)
    got = mt.render_batch(cams, w, h, lights=[_lights(ls) for ls in light_sets])
    assert got["rgb"].shape == (5, h, w, 3)
    for flags in (MTB_FLAG_MEGAKERNEL, 0):
        mt.set_flags(flags)
        for v, single in enumerate(_singles(mt, cams, w, h, light_sets)):
            assert np.array_equal(got["rgb"][v], single["rgb"]), "view %d differs from its single render (flags %d)" % (v, flags)
    orc = oracle_mod.Oracle.from_obj(files.obj_path)
    rays = 0
    for v in range(5):
        orc.set_lights(light_sets[v])
        cpu = orc.render(cams[v], w, h, depth=depth)
        diff = np.abs(got["rgb"][v].astype(np.int16) - cpu["rgb"].astype(np.int16))
        assert diff.max() <= MAX_RGB_DIFF and (diff > 0).mean() <= MAX_RGB_FRACTION, "view %d against the oracle" % v
        rays += cpu["stats"]["rays"]
    assert got["stats"]["rays"] == rays
    assert got["stats"]["kernel_ms"] > 0.0


@pytest.mark.gpu
def test_light_and_depth_edge_cases(product_lib, scene_dir):
    """lights=None (the scene's lights), no lights at all, depths 0 and 8, one view and 64 views."""
    from mythtracer_b200 import MTB_FLAG_MEGAKERNEL
    files, cfg = scenes.config_scene("C1", scene_dir)
    w, h = 40, 27
    mt = _tracer(files.obj_path, 5, MTB_FLAG_MEGAKERNEL)
    mt.GetScene().lights = _lights(scenes.LIGHT_RIG[:3])
    for depth in (0, 8):
        mt.max_depth = depth
        for n in (1, 64):
            cams = [_yawed(files.camera, 1.5 * k) for k in range(n)]
            singles = _singles(mt, cams, w, h)
            got = mt.render_batch(cams, w, h)
            for v in range(n):
                assert np.array_equal(got["rgb"][v], singles[v]["rgb"]), "depth %d, %d views: view %d" % (depth, n, v)
            assert got["stats"]["rays"] == sum(s["stats"]["rays"] for s in singles)
            # no lights: the views are lit by nothing, whatever the scene's lights are
            dark = mt.render_batch(cams, w, h, lights=[[] for _ in cams])
            dark_singles = _singles(mt, cams, w, h, [[] for _ in cams])
            for v in range(n):
                assert np.array_equal(dark["rgb"][v], dark_singles[v]["rgb"]), "no lights, depth %d, %d views: view %d" % (depth, n, v)


@pytest.mark.gpu
def test_counters_are_the_sum_of_the_views(product_lib, scene_dir):
    from mythtracer_b200 import MTB_FLAG_COUNT_WORK, MTB_FLAG_MEGAKERNEL
    files, cfg = scenes.config_scene("C1", scene_dir)
    w, h = 96, 64
    cams = [_yawed(files.camera, 4.0 * k) for k in range(4)]
    light_sets = [scenes.LIGHT_RIG[k:k + 2] for k in range(4)]
    light_sets[3] = scenes.LIGHT_RIG[:1] + scenes.LIGHT_RIG[3:]
    mt = _tracer(files.obj_path, 4, MTB_FLAG_COUNT_WORK | MTB_FLAG_MEGAKERNEL)
    got = mt.render_batch(cams, w, h, lights=[_lights(ls) for ls in light_sets])
    singles = _singles(mt, cams, w, h, light_sets)
    for k, value in got["stats"].items():
        if k.endswith("_ms"):
            continue
        assert value == sum(s["stats"][k] for s in singles), "counter %s" % k
    assert got["stats"]["n_bvh"] > 0 and got["stats"]["shadow"] > 0


@pytest.mark.gpu
def test_textured_views(product_lib, scene_dir):
    from mythtracer_b200 import MTB_FLAG_MEGAKERNEL
    files, cfg = scenes.config_scene("C2", scene_dir)
    w, h = 320, 180
    mt = _tracer(files.obj_path, cfg["depth"], MTB_FLAG_MEGAKERNEL)
    assert mt.scene_info()["n_textures"] > 0
    mt.GetScene().lights = _lights(files.lights)
    cams = [_yawed(files.camera, d) for d in (-3.0, 0.0, 5.0)]
    got = mt.render_batch(cams, w, h)
    for v, single in enumerate(_singles(mt, cams, w, h)):
        assert np.array_equal(got["rgb"][v], single["rgb"]), "C2 view %d" % v


@pytest.mark.gpu
def test_full_size_views_equal_the_reference(product_lib, scene_dir):
    """C3 at 1920x1080: views 0 and 2 are the reference's own frame (tests/golden/full_C3.npz), view 1 (yaw + 2 degrees)
    its single render."""
    from mythtracer_b200 import MTB_FLAG_MEGAKERNEL
    z = np.load(os.path.join(HERE, "golden", "full_C3.npz"))
    files, cfg = scenes.config_scene("C3", scene_dir)
    W, H = cfg["width"], cfg["height"]
    assert int(z["width"]) == W and int(z["height"]) == H and int(z["depth"]) == cfg["depth"] and len(z["rows"]) == H
    mt = _tracer(files.obj_path, cfg["depth"], MTB_FLAG_MEGAKERNEL)
    mt.GetScene().lights = _lights(files.lights)
    cams = [files.camera, _yawed(files.camera, 2.0), files.camera]
    got = mt.render_batch(cams, W, H)
    for v in (0, 2):
        diff = np.abs(got["rgb"][v].astype(np.int16) - z["rgb"].astype(np.int16))
        if diff.max() == 0:
            assert _sha(got["rgb"][v]) == str(z["rgb_sha256"])
        assert diff.max() <= MAX_RGB_DIFF and (diff > 0).mean() <= MAX_RGB_FRACTION, "C3 view %d against the reference" % v
    assert np.array_equal(got["rgb"][1], _singles(mt, cams[1:2], W, H)[0]["rgb"])


@pytest.mark.gpu
def test_batch_leaves_the_single_frame_state_alone(product_lib, scene_dir):
    files, cfg = scenes.config_scene("C1", scene_dir)
    w, h = 160, 120
    mt = _tracer(files.obj_path, 3)  # automatic pipeline choice
    mt.GetScene().lights = _lights(scenes.LIGHT_RIG[:2])
    before = [mt.render_chunk(files.camera, w, h, 0, 0, w, h)["rgb"] for _ in range(14)]  # past the 13 deciding frames
    pipeline = mt.pipeline_in_use()
    assert pipeline[0] != "measuring"
    mt.max_depth = 7
    mt.render_batch([_yawed(files.camera, 10.0)] * 3, 64, 48, lights=[_lights(scenes.LIGHT_RIG[1:4])] * 3)
    mt.max_depth = 3
    after = mt.render_chunk(files.camera, w, h, 0, 0, w, h)["rgb"]
    assert np.array_equal(after, before[-1])
    assert mt.pipeline_in_use() == pipeline


@pytest.mark.gpu
def test_views_split_over_devices(product_lib, scene_dir):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from mythtracer_b200 import MTB_FLAG_MEGAKERNEL
    files, cfg = scenes.config_scene("C1", scene_dir)
    w, h = 150, 97
    cams = [_yawed(files.camera, 3.0 * k) for k in range(5)]
    light_sets = [_lights(scenes.LIGHT_RIG[k % 3:k % 3 + 2]) for k in range(5)]
    one = _tracer(files.obj_path, 5, MTB_FLAG_MEGAKERNEL).render_batch(cams, w, h, lights=light_sets)
    n = min(torch.cuda.device_count(), 8)
    many = _tracer(files.obj_path, 5, MTB_FLAG_MEGAKERNEL, devices=list(range(n)))
    assert many.device_count() == n
    got = many.render_batch(cams, w, h, lights=light_sets)
    assert np.array_equal(got["rgb"], one["rgb"])
    assert got["stats"]["rays"] == one["stats"]["rays"]


@pytest.mark.gpu
def test_bad_batch_arguments(product_lib, scene_dir):
    """Each refused call returns MTB_ERR_ARG and leaves a message in mtb_last_error."""
    from mythtracer_b200 import MythTracer, api
    MTB_OK, MTB_ERR_ARG = 0, -1
    files, cfg = scenes.config_scene("C1", scene_dir)
    mt = MythTracer(max_depth=3)
    assert mt.LoadObj(files.obj_path)
    cams = np.zeros(1, api.CAMERA_DTYPE)
    cams[0] = api.Camera.from_tuple(files.camera).as_array()
    cam_ptr = cams.ctypes.data_as(ctypes.c_void_p)
    rgb = np.zeros(8 * 8 * 3, np.uint8)

    def call(cams, n_views, depth=3):
        rc = product_lib.mtb_render_batch(mt._ctx, cams, n_views, None, 0, 8, 8, depth, rgb.ctypes.data_as(ctypes.c_void_p), None)
        return rc, product_lib.mtb_last_error(mt._ctx).decode()

    assert call(cam_ptr, 1)[0] == MTB_OK
    for args, words in (((cam_ptr, 0), "n_views"), ((cam_ptr, 65536), "n_views"), ((cam_ptr, 1, 17), "render arguments"),
                        ((None, 1), "cams")):
        rc, msg = call(*args)
        assert rc == MTB_ERR_ARG and words in msg, (args, rc, msg)
    mt.set_partition(1, 2)
    rc, msg = call(cam_ptr, 1)
    assert rc == MTB_ERR_ARG and "partition" in msg
    mt.set_partition(0, 1)
    assert call(cam_ptr, 1)[0] == MTB_OK


@pytest.mark.gpu
def test_animation_driver_in_batches(product_lib, scene_dir, tmp_path):
    """Frames 74..80 with frames_per_call 4: two batch calls (the second one partial) through RayTraceBatchAsync, two
    pinned batch buffers in rotation; every file equals MythTracer.RayTrace of its frame."""
    from mythtracer_b200 import Camera, Light, MythTracer
    if shutil.which("g++") is None or shutil.which("make") is None:
        pytest.skip("g++/make not available")
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "apps")], stdout=subprocess.DEVNULL)
    files, cfg = scenes.config_scene("C1", scene_dir)
    out_dir = tmp_path / "anim"
    W, H = 160, 90
    res = subprocess.run([os.path.join(ROOT, "apps", "_build", "mythtracer_local_b200"), files.obj_path, str(W), str(H), "74", "80",
                          str(out_dir), "4"], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stdout[-1500:] + res.stderr[-1500:]
    assert "in 2 calls" in res.stdout
    assert sorted(os.listdir(out_dir)) == ["dump_%05d.raw" % f for f in range(74, 81)]
    mt = MythTracer(max_depth=5)
    assert mt.LoadObj(files.obj_path)
    rig = [(231.82174, 81.69966, -27.78259, 0.3, 0.3, 0.3, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0)] + [
        (200.0, 80.0, z, 0.0, 0.0, 0.0, 0.3, 0.3, 0.3, 0.3, 0.3, 0.3) for z in (0.0, 80.0, 160.0)]
    mt.GetScene().lights = [Light.from_tuple(l) for l in rig]
    for frame in range(74, 81):   # main_local.cc:51,72-76: angle = 2 * frame, yaw = angle + 90
        cam = Camera((300.0, 107.0, 40.0), 30.0, 2.0 * frame + 90, 0.0, 110.0)
        got = np.fromfile(out_dir / ("dump_%05d.raw" % frame), np.uint8).reshape(H, W, 3)
        assert np.array_equal(got, mt.RayTrace(W, H, cam)), "frame %d" % frame
