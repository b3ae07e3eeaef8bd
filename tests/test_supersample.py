"""Supersampled batches (mtb_render_batch_ss / render_batch(..., samples_per_axis=s)): every output pixel is the rounded
mean of the s x s pixels of the same view rendered at (s*W) x (s*H), formed in the kernel.  The samples are the
reference's own pixels, so the expected output is fully determined by a frame the reference renders: the block means of
render_batch at s*W x s*H, and of the reference's stored full frames (tests/golden/full_C*.npz)."""
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
MTB_OK, MTB_ERR_ARG = 0, -1


def _block_mean(frames, s):
    """(..., s*H, s*W, 3) uint8 -> (..., H, W, 3): (sum of each s x s block + s*s/2) / (s*s), integer division."""
    f = np.asarray(frames, np.uint32)
    h, w = f.shape[-3] // s, f.shape[-2] // s
    blocks = f.reshape(f.shape[:-3] + (h, s, w, s, 3)).sum(axis=(-4, -2))
    return ((blocks + s * s // 2) // (s * s)).astype(np.uint8)


def _yawed(cam, dyaw):
    c = list(cam)
    c[4] += dyaw
    return tuple(c)


def _lights(rows):
    from mythtracer_b200 import Light
    return [Light.from_tuple(l) for l in rows]


def _tracer(path, depth, flags=0, devices=None):
    from mythtracer_b200 import MythTracer
    mt = MythTracer(devices=devices, max_depth=depth, flags=flags)
    assert mt.LoadObj(path), mt.last_error()
    return mt


def _file_sha(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for blk in iter(lambda: f.read(1 << 20), b""):
            h.update(blk)
    return h.hexdigest()


def _check_ss(mt, cams, w, h, s, lights=None):
    """render_batch at w x h with s samples per axis against the block means of render_batch at s*w x s*h."""
    got = mt.render_batch(cams, w, h, lights=lights, samples_per_axis=s)
    hi = mt.render_batch(cams, s * w, s * h, lights=lights)
    assert got["rgb"].shape == (len(cams), h, w, 3)
    want = _block_mean(hi["rgb"], s)
    for v in range(len(cams)):
        assert np.array_equal(got["rgb"][v], want[v]), "s = %d, %dx%d, view %d of %d" % (s, w, h, v, len(cams))
    assert got["stats"]["rays"] == hi["stats"]["rays"]
    return got


# ---------------------------------------------------------------------------------------------- CPU


def test_supersampling_has_no_cpu_fallback(product_lib):
    from mythtracer_b200 import MythTracer, MythTracerError
    files, cfg = scenes.config_scene("C1", "/tmp/mtb_scenes")
    mt = MythTracer(host_only=True)
    assert mt.LoadObj(files.obj_path)
    with pytest.raises(MythTracerError, match="no CPU fallback"):
        mt.render_batch([files.camera, files.camera], 16, 16, samples_per_axis=2)


def test_supersampling_arguments_are_checked_in_python(product_lib):
    from mythtracer_b200 import MythTracer, MythTracerError
    files, cfg = scenes.config_scene("C1", "/tmp/mtb_scenes")
    mt = MythTracer(host_only=True)
    assert mt.LoadObj(files.obj_path)
    cams = [files.camera, files.camera]
    for s in (0, 3, 16, -2, 2.0, True):
        with pytest.raises(MythTracerError, match="samples_per_axis"):
            mt.render_batch(cams, 16, 16, samples_per_axis=s)
    # out holds the output pixels, not the samples
    with pytest.raises(MythTracerError, match="out must be"):
        mt.render_batch(cams, 16, 16, out=np.zeros((2, 32, 32, 3), np.uint8), samples_per_axis=2)
    with pytest.raises(MythTracerError, match="one per view"):
        mt.render_batch(cams, 16, 16, lights=[_lights(scenes.LIGHT_RIG[:2])], samples_per_axis=4)
    with pytest.raises(MythTracerError, match="same number of lights"):
        mt.render_batch(cams, 16, 16, lights=[_lights(scenes.LIGHT_RIG[:2]), _lights(scenes.LIGHT_RIG[:1])], samples_per_axis=8)


def test_block_mean_rounds_half_up():
    f = np.zeros((4, 4, 3), np.uint8)
    f[:2, :2, 0] = [[1, 1], [0, 0]]     # mean 0.5 -> 1
    f[:2, 2:, 0] = [[1, 0], [0, 0]]     # mean 0.25 -> 0
    f[2:, :2, 1] = [[255, 255], [255, 254]]  # mean 254.75 -> 255
    f[2:, 2:, 2] = [[3, 4], [5, 6]]     # mean 4.5 -> 5
    m = _block_mean(f, 2)
    assert m[0, 0, 0] == 1 and m[0, 1, 0] == 0 and m[1, 0, 1] == 255 and m[1, 1, 2] == 5


# ---------------------------------------------------------------------------------------------- GPU


@pytest.mark.gpu
@pytest.mark.parametrize("s", [2, 4, 8])
def test_views_equal_the_block_means_of_the_high_resolution_batch(product_lib, scene_dir, s):
    """C1 at 75x49 (the sample grid has partial edge tiles for s = 2 and 4), depth 5, five views with their own yaw and
    their own two lights."""
    from mythtracer_b200 import MTB_FLAG_MEGAKERNEL
    files, cfg = scenes.config_scene("C1", scene_dir)
    rig = scenes.LIGHT_RIG
    cams = [_yawed(files.camera, 6.0 * k - 12.0) for k in range(5)]
    light_sets = [_lights([rig[k % 4], rig[(k + 1) % 4]]) for k in range(5)]
    mt = _tracer(files.obj_path, 5, MTB_FLAG_MEGAKERNEL)
    got = _check_ss(mt, cams, 75, 49, s, lights=light_sets)
    assert got["stats"]["kernel_ms"] > 0.0
    # the anti-aliased view is not the one-ray-per-pixel view
    assert not np.array_equal(got["rgb"], mt.render_batch(cams, 75, 49, lights=light_sets)["rgb"])


@pytest.mark.gpu
@pytest.mark.parametrize("s", [2, 4, 8])
def test_light_and_depth_edge_cases(product_lib, scene_dir, s):
    """lights=None (the scene's lights), no lights at all, depths 0 and 8, one view and 64 views."""
    files, cfg = scenes.config_scene("C1", scene_dir)
    w, h = 24, 17
    mt = _tracer(files.obj_path, 5)
    mt.GetScene().lights = _lights(scenes.LIGHT_RIG[:3])
    for depth in (0, 8):
        mt.max_depth = depth
        for n in (1, 64):
            cams = [_yawed(files.camera, 1.5 * k) for k in range(n)]
            _check_ss(mt, cams, w, h, s)
            _check_ss(mt, cams, w, h, s, lights=[[] for _ in cams])


@pytest.mark.gpu
@pytest.mark.parametrize("s", [2, 4, 8])
def test_textured_views(product_lib, scene_dir, s):
    files, cfg = scenes.config_scene("C2", scene_dir, 0.1)
    mt = _tracer(files.obj_path, cfg["depth"])
    assert mt.scene_info()["n_textures"] > 0
    mt.GetScene().lights = _lights(files.lights)
    _check_ss(mt, [_yawed(files.camera, d) for d in (-3.0, 0.0, 5.0)], 80, 45, s)


@pytest.mark.gpu
@pytest.mark.parametrize("name,sizes", [("C3", ((960, 540, 2), (480, 270, 4), (240, 135, 8))), ("C5", ((1920, 1080, 2),)),
                                        ("C2", ((640, 360, 2),)), ("C4", ((960, 540, 2),))])
def test_views_equal_the_block_means_of_the_reference_frame(product_lib, scene_dir, name, sizes):
    """The reference's own full frame (tests/golden/full_<name>.npz) at s*W x s*H is exactly the sample grid of a
    W x H view with s samples per axis: its block means are the expected bytes."""
    z = np.load(os.path.join(HERE, "golden", "full_%s.npz" % name))
    files, cfg = scenes.config_scene(name, scene_dir)
    assert _file_sha(files.obj_path) == str(z["obj_sha256"]), "generated %s scene differs from the fixture's scene" % name
    assert _file_sha(files.mtl_path) == str(z["mtl_sha256"])
    assert int(z["depth"]) == cfg["depth"] and len(z["rows"]) == int(z["height"])
    mt = _tracer(files.obj_path, cfg["depth"])
    mt.GetScene().lights = _lights(files.lights)
    for w, h, s in sizes:
        assert (s * w, s * h) == (int(z["width"]), int(z["height"]))
        got = mt.render_batch([files.camera], w, h, samples_per_axis=s)
        want = _block_mean(z["rgb"], s)
        assert np.array_equal(got["rgb"][0], want), "%s at %dx%d, s = %d: %d channels differ from the reference's block means" % (
            name, w, h, s, int((got["rgb"][0] != want).sum()))
    mt.close()


@pytest.mark.gpu
def test_oracle(product_lib, oracle_mod, scene_dir):
    """C1 at 40x27 with s = 2 against the block means of the CPU oracle's 80x54 frame (the oracle and the GPU may differ
    in the last ulp of pow(): at most 1 per channel)."""
    files, cfg = scenes.config_scene("C1", scene_dir)
    w, h, s, depth = 40, 27, 2, 5
    lights = scenes.LIGHT_RIG[:2]
    mt = _tracer(files.obj_path, depth)
    mt.GetScene().lights = _lights(lights)
    got = mt.render_batch([files.camera], w, h, samples_per_axis=s)
    orc = oracle_mod.Oracle.from_obj(files.obj_path)
    orc.set_lights(lights)
    cpu = orc.render(files.camera, s * w, s * h, depth=depth)
    diff = np.abs(got["rgb"][0].astype(np.int16) - _block_mean(cpu["rgb"], s).astype(np.int16))
    assert diff.max() <= 1
    assert got["stats"]["rays"] == cpu["stats"]["rays"]


@pytest.mark.gpu
@pytest.mark.parametrize("s", [2, 4, 8])
def test_counters_equal_those_of_the_high_resolution_batch(product_lib, scene_dir, s):
    from mythtracer_b200 import MTB_FLAG_COUNT_WORK
    files, cfg = scenes.config_scene("C1", scene_dir)
    w, h = 48, 32
    cams = [_yawed(files.camera, 4.0 * k) for k in range(3)]
    light_sets = [_lights(scenes.LIGHT_RIG[k:k + 2]) for k in range(3)]
    mt = _tracer(files.obj_path, 4, MTB_FLAG_COUNT_WORK)
    got = _check_ss(mt, cams, w, h, s, lights=light_sets)["stats"]
    hi = mt.render_batch(cams, s * w, s * h, lights=light_sets)["stats"]
    for k, value in got.items():
        if not k.endswith("_ms"):
            assert value == hi[k], "counter %s" % k
    assert got["n_bvh"] > 0 and got["shadow"] > 0


@pytest.mark.gpu
def test_async_into_pinned_memory(product_lib, scene_dir):
    """mtb_render_batch_ss_async into mtb_host_alloc memory, then mtb_wait: the bytes of the synchronous call."""
    from mythtracer_b200 import api
    files, cfg = scenes.config_scene("C1", scene_dir)
    w, h, s, n = 64, 40, 4, 3
    mt = _tracer(files.obj_path, 5)
    mt.GetScene().lights = _lights(scenes.LIGHT_RIG[:2])
    cams = [_yawed(files.camera, 5.0 * k) for k in range(n)]
    want = mt.render_batch(cams, w, h, samples_per_axis=s)["rgb"]
    cam_arr = np.zeros(n, api.CAMERA_DTYPE)
    for i, c in enumerate(cams):
        cam_arr[i] = api.Camera.from_tuple(c).as_array()
    product_lib.mtb_host_alloc.restype = ctypes.c_void_p
    product_lib.mtb_host_alloc.argtypes = [ctypes.c_size_t]
    product_lib.mtb_host_free.argtypes = [ctypes.c_void_p]
    nbytes = n * h * w * 3
    buf = product_lib.mtb_host_alloc(nbytes)
    assert buf
    try:
        ctypes.memset(buf, 0, nbytes)
        mt.push_lights()
        rc = product_lib.mtb_render_batch_ss_async(mt._ctx, cam_arr.ctypes.data_as(ctypes.c_void_p), n, None, 0, w, h, s, mt.max_depth,
                                                   ctypes.c_void_p(buf))
        assert rc == MTB_OK, product_lib.mtb_last_error(mt._ctx)
        mt.wait()
        got = np.ctypeslib.as_array((ctypes.c_uint8 * nbytes).from_address(buf)).reshape(n, h, w, 3).copy()
    finally:
        product_lib.mtb_host_free(ctypes.c_void_p(buf))
    assert np.array_equal(got, want)


@pytest.mark.gpu
def test_supersampling_leaves_the_single_frame_state_alone(product_lib, scene_dir):
    files, cfg = scenes.config_scene("C1", scene_dir)
    w, h = 160, 120
    mt = _tracer(files.obj_path, 3)  # automatic pipeline choice
    mt.GetScene().lights = _lights(scenes.LIGHT_RIG[:2])
    before = [mt.render_chunk(files.camera, w, h, 0, 0, w, h)["rgb"] for _ in range(14)]  # past the 13 deciding frames
    pipeline = mt.pipeline_in_use()
    assert pipeline[0] != "measuring"
    mt.max_depth = 7
    for s in (2, 4, 8):
        mt.render_batch([_yawed(files.camera, 10.0)] * 3, 64, 48, lights=[_lights(scenes.LIGHT_RIG[1:4])] * 3, samples_per_axis=s)
    mt.max_depth = 3
    after = mt.render_chunk(files.camera, w, h, 0, 0, w, h)["rgb"]
    assert np.array_equal(after, before[-1])
    assert mt.pipeline_in_use() == pipeline


@pytest.mark.gpu
def test_bad_samples_per_axis(product_lib, scene_dir):
    """Each refused call returns MTB_ERR_ARG and leaves a message in mtb_last_error; s = 1 is mtb_render_batch."""
    from mythtracer_b200 import MythTracer, api
    files, cfg = scenes.config_scene("C1", scene_dir)
    mt = MythTracer(max_depth=3)
    assert mt.LoadObj(files.obj_path)
    mt.GetScene().lights = _lights(scenes.LIGHT_RIG[:2])
    mt.push_lights()
    cams = np.zeros(1, api.CAMERA_DTYPE)
    cams[0] = api.Camera.from_tuple(files.camera).as_array()
    cam_ptr = cams.ctypes.data_as(ctypes.c_void_p)
    rgb = np.zeros(16 * 8 * 3, np.uint8)

    def call(s, w=16, h=8):
        rc = product_lib.mtb_render_batch_ss(mt._ctx, cam_ptr, 1, None, 0, w, h, s, 3, rgb.ctypes.data_as(ctypes.c_void_p), None)
        return rc, product_lib.mtb_last_error(mt._ctx).decode()

    for s in (0, 3, 5, 16, -1):
        rc, msg = call(s)
        assert rc == MTB_ERR_ARG and "samples_per_axis" in msg, (s, rc, msg)
    rc, msg = call(8, w=8193)
    assert rc == MTB_ERR_ARG and "sample grid" in msg, (rc, msg)
    assert call(1)[0] == MTB_OK
    one = rgb.copy()
    assert product_lib.mtb_render_batch(mt._ctx, cam_ptr, 1, None, 0, 16, 8, 3, rgb.ctypes.data_as(ctypes.c_void_p), None) == MTB_OK
    assert np.array_equal(rgb, one)


@pytest.mark.gpu
@pytest.mark.parametrize("per_call", [1, 4])
def test_animation_driver_supersampled(product_lib, scene_dir, tmp_path, per_call):
    """Frames 74..80 with samples_per_axis 2: through the batch path even with frames_per_call 1; every file equals
    render_batch(..., samples_per_axis=2) of the orbit camera of its frame."""
    from mythtracer_b200 import Camera, Light, MythTracer
    if shutil.which("g++") is None or shutil.which("make") is None:
        pytest.skip("g++/make not available")
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "apps")], stdout=subprocess.DEVNULL)
    files, cfg = scenes.config_scene("C1", scene_dir)
    out_dir = tmp_path / "anim"
    W, H = 160, 90
    res = subprocess.run([os.path.join(ROOT, "apps", "_build", "mythtracer_local_b200"), files.obj_path, str(W), str(H), "74", "80",
                          str(out_dir), str(per_call), "2"], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stdout[-1500:] + res.stderr[-1500:]
    assert "in %d calls" % (7 if per_call == 1 else 2) in res.stdout
    assert sorted(os.listdir(out_dir)) == ["dump_%05d.raw" % f for f in range(74, 81)]
    mt = MythTracer(max_depth=5)
    assert mt.LoadObj(files.obj_path)
    rig = [(231.82174, 81.69966, -27.78259, 0.3, 0.3, 0.3, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0)] + [
        (200.0, 80.0, z, 0.0, 0.0, 0.0, 0.3, 0.3, 0.3, 0.3, 0.3, 0.3) for z in (0.0, 80.0, 160.0)]
    mt.GetScene().lights = [Light.from_tuple(l) for l in rig]
    cams = [Camera((300.0, 107.0, 40.0), 30.0, 2.0 * frame + 90, 0.0, 110.0) for frame in range(74, 81)]
    want = mt.render_batch(cams, W, H, samples_per_axis=2)["rgb"]
    for i, frame in enumerate(range(74, 81)):
        got = np.fromfile(out_dir / ("dump_%05d.raw" % frame), np.uint8).reshape(H, W, 3)
        assert np.array_equal(got, want[i]), "frame %d" % frame


@pytest.mark.gpu
def test_supersampled_views_split_over_devices(product_lib, scene_dir):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    files, cfg = scenes.config_scene("C1", scene_dir)
    w, h = 75, 49
    cams = [_yawed(files.camera, 3.0 * k) for k in range(5)]
    light_sets = [_lights(scenes.LIGHT_RIG[k % 3:k % 3 + 2]) for k in range(5)]
    n = min(torch.cuda.device_count(), 8)
    one = _tracer(files.obj_path, 5)
    many = _tracer(files.obj_path, 5, devices=list(range(n)))
    assert many.device_count() == n
    for s in (2, 4, 8):
        a = one.render_batch(cams, w, h, lights=light_sets, samples_per_axis=s)
        b = many.render_batch(cams, w, h, lights=light_sets, samples_per_axis=s)
        assert np.array_equal(b["rgb"], a["rgb"]), "s = %d" % s
        assert b["stats"]["rays"] == a["stats"]["rays"]
