"""Accumulated batches (mtb_render_batch_accum / render_batch(..., subframes=k)): every output view is the rounded mean
of all k * s * s quantised samples of its k sub-frames (one camera and one light set each), formed in the kernel.  The
sub-frames are frames the reference renders, so the expected bytes are fixed by render_batch of the sub-frames at
(s*W) x (s*H), itself pinned to the reference, and by the reference's stored full frames (tests/golden/full_C3.npz)."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from tests import scenes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
MTB_OK, MTB_ERR_ARG = 0, -1


def _accum_mean(frames, k, s):
    """(n_out * k, s*H, s*W, 3) uint8 -> (n_out, H, W, 3): per output view, (sum of the k * s * s samples of each output
    channel + k*s*s/2) / (k*s*s), integer division."""
    f = np.asarray(frames)
    n_out, sh, sw = f.shape[0] // k, f.shape[1], f.shape[2]
    out = np.zeros((n_out, sh // s, sw // s, 3), np.uint8)
    n = k * s * s
    for v in range(n_out):
        acc = np.zeros((sh, sw, 3), np.uint32)
        for j in range(k):
            acc += f[v * k + j]
        blocks = acc.reshape(sh // s, s, sw // s, s, 3).sum(axis=(1, 3))
        out[v] = ((blocks + n // 2) // n).astype(np.uint8)
    return out


def _yawed(cam, dyaw):
    c = list(cam)
    c[4] += dyaw
    return tuple(c)


def _orbit_subframes(cam, n_out, k):
    """Output view f at yaw + 2 degrees * f (the C3 orbit of tools/batch_throughput.py), its sub-frame j at
    + 2 * j / k: a shutter open for one frame interval."""
    return [_yawed(cam, 2.0 * f + 2.0 * j / k) for f in range(n_out) for j in range(k)]


def _lights(rows):
    from mythtracer_b200 import Light
    return [Light.from_tuple(l) for l in rows]


def _tracer(path, depth, flags=0, devices=None):
    from mythtracer_b200 import MythTracer
    mt = MythTracer(devices=devices, max_depth=depth, flags=flags)
    assert mt.LoadObj(path), mt.last_error()
    return mt


def _check_accum(mt, cams, w, h, k, s, lights=None):
    """render_batch(..., subframes=k) at w x h against the formula over render_batch of the sub-frames at s*w x s*h."""
    got = mt.render_batch(cams, w, h, lights=lights, samples_per_axis=s, subframes=k)
    assert got["rgb"].shape == (len(cams) // k, h, w, 3)
    hi = mt.render_batch(cams, s * w, s * h, lights=lights)
    want = _accum_mean(hi["rgb"], k, s)
    for v in range(len(cams) // k):
        assert np.array_equal(got["rgb"][v], want[v]), "k = %d, s = %d, %dx%d, output view %d: %d channels differ" % (
            k, s, w, h, v, int((got["rgb"][v] != want[v]).sum()))
    assert got["stats"]["rays"] == hi["stats"]["rays"]
    return got, hi


def _c3(scene_dir):
    files, cfg = scenes.config_scene("C3", scene_dir)
    mt = _tracer(files.obj_path, cfg["depth"])
    mt.GetScene().lights = _lights(files.lights)
    return files, cfg, mt


def _jittered_lights(base, k, radius, seed):
    """k light sets: every light of `base` moved to a seeded random point of a disc of `radius` in its horizontal
    plane (an area light sampled at k positions)."""
    rng = np.random.default_rng(seed)
    sets = []
    for _ in range(k):
        ls = []
        for l in base:
            r, a = radius * np.sqrt(rng.random()), 2.0 * np.pi * rng.random()
            row = list(l)
            row[0] += r * np.cos(a)
            row[2] += r * np.sin(a)
            ls.append(tuple(row))
        sets.append(_lights(ls))
    return sets


# ---------------------------------------------------------------------------------------------- CPU


def test_accumulation_has_no_cpu_fallback(product_lib):
    from mythtracer_b200 import MythTracer, MythTracerError
    files, cfg = scenes.config_scene("C1", "/tmp/mtb_scenes")
    mt = MythTracer(host_only=True)
    assert mt.LoadObj(files.obj_path)
    with pytest.raises(MythTracerError, match="no CPU fallback"):
        mt.render_batch([files.camera] * 4, 16, 16, subframes=2)


def test_accumulation_arguments_are_checked_in_python(product_lib):
    from mythtracer_b200 import MythTracer, MythTracerError
    files, cfg = scenes.config_scene("C1", "/tmp/mtb_scenes")
    mt = MythTracer(host_only=True)
    assert mt.LoadObj(files.obj_path)
    cams = [files.camera] * 6
    for k in (0, -1, 2.0, True, False, "2", None):
        with pytest.raises(MythTracerError, match="subframes"):
            mt.render_batch(cams, 16, 16, subframes=k)
    # the cameras are whole output views of k sub-frames
    for k in (4, 5, 7):
        with pytest.raises(MythTracerError, match="whole number of output views"):
            mt.render_batch(cams, 16, 16, subframes=k)
    # out holds the output views, not the sub-frames
    with pytest.raises(MythTracerError, match="out must be"):
        mt.render_batch(cams, 16, 16, out=np.zeros((6, 16, 16, 3), np.uint8), subframes=3)
    with pytest.raises(MythTracerError, match="out must be"):
        mt.render_batch(cams, 16, 16, out=np.zeros((2, 32, 32, 3), np.uint8), subframes=3, samples_per_axis=2)
    # no planes of an accumulated view
    for kw in (dict(debug=True), dict(taps=True), dict(debug=True, taps=True)):
        with pytest.raises(MythTracerError, match="debug and taps"):
            mt.render_batch(cams, 16, 16, subframes=2, **kw)
    # one light set per sub-frame
    with pytest.raises(MythTracerError, match="one per view"):
        mt.render_batch(cams, 16, 16, lights=[_lights(scenes.LIGHT_RIG[:2])] * 2, subframes=3)
    with pytest.raises(MythTracerError, match="samples_per_axis"):
        mt.render_batch(cams, 16, 16, samples_per_axis=3, subframes=2)


def test_accumulated_mean_rounds_half_up_over_all_samples():
    f = np.zeros((3, 2, 2, 3), np.uint8)  # one output view of k = 3 sub-frames, s = 2: 12 samples
    f[0, 0, 0, 0] = 6                     # 6 / 12 = 0.5 -> 1
    f[:, :, :, 1] = 200
    f[2, 1, 1, 1] = 205                   # (12 * 200 + 5) / 12 = 200.42 -> 200
    f[0, :, :, 2] = 10                    # 40 / 12 = 3.33 -> 3 (the mean of the sub-frame means, 10/3, would round the same)
    f[1, 0, 0, 2] = 5                     # 45 / 12 = 3.75 -> 4
    m = _accum_mean(f, 3, 2)
    assert m.shape == (1, 1, 1, 3)
    assert m[0, 0, 0].tolist() == [1, 200, 4]
    # not a mean of means: two sub-frames of s = 2 whose rounded block means are 1 (sum 2) and 0 (sum 0); their rounded
    # mean would be 1, the mean of the 8 samples is 2 / 8 -> 0
    g = np.zeros((2, 2, 2, 3), np.uint8)
    g[0, 0, :, 0] = 1
    assert _accum_mean(g, 2, 2)[0, 0, 0, 0] == 0
    # k = 1 is the block mean of supersampling
    h = np.arange(4 * 4 * 3, dtype=np.uint8).reshape(1, 4, 4, 3)
    blocks = h[0].astype(np.uint32).reshape(2, 2, 2, 2, 3).sum(axis=(1, 3))
    assert np.array_equal(_accum_mean(h, 1, 2)[0], ((blocks + 2) // 4).astype(np.uint8))


# ---------------------------------------------------------------------------------------------- GPU


@pytest.mark.gpu
def test_identical_subframes_equal_the_reference_frame(product_lib, scene_dir):
    """k = 4 identical sub-frames of the C3 camera: at 1920x1080 with s = 1 the bytes of the reference's stored frame,
    at 960x540 with s = 2 its block means."""
    z = np.load(os.path.join(HERE, "golden", "full_C3.npz"))
    files, cfg, mt = _c3(scene_dir)
    W, H = int(z["width"]), int(z["height"])
    assert (W, H) == (cfg["width"], cfg["height"]) and int(z["depth"]) == cfg["depth"]
    got = mt.render_batch([files.camera] * 4, W, H, subframes=4)
    assert np.array_equal(got["rgb"][0], z["rgb"]), "%d channels differ from full_C3" % int((got["rgb"][0] != z["rgb"]).sum())
    got = mt.render_batch([files.camera] * 4, W // 2, H // 2, samples_per_axis=2, subframes=4)
    assert np.array_equal(got["rgb"][0], _accum_mean(z["rgb"][None], 1, 2)[0])
    mt.close()


@pytest.mark.gpu
@pytest.mark.parametrize("s", [1, 2, 4, 8])
@pytest.mark.parametrize("k", [3, 5, 8])
def test_motion_blur_of_the_c3_orbit(product_lib, scene_dir, k, s):
    """3 output frames of the C3 orbit at 480x270, each the mean of k sub-frames spread over the frame interval."""
    files, cfg, mt = _c3(scene_dir)
    cams = _orbit_subframes(files.camera, 3, k)
    got, hi = _check_accum(mt, cams, 480, 270, k, s)
    if s == 1:
        # a blurred frame is not its first sub-frame
        assert not np.array_equal(got["rgb"][0], hi["rgb"][0])
    mt.close()


@pytest.mark.gpu
@pytest.mark.parametrize("s", [1, 4])
def test_soft_shadows_from_jittered_lights(product_lib, scene_dir, s):
    """One C3 camera, k = 8 sub-frames with seeded jittered light positions (two output views with their own jitter);
    then lights=None, where every sub-frame uses the scene's lights."""
    files, cfg, mt = _c3(scene_dir)
    k, w, h = 8, 240, 135
    light_sets = _jittered_lights(files.lights, k, 25.0, seed=11) + _jittered_lights(files.lights, k, 25.0, seed=12)
    got, hi = _check_accum(mt, [files.camera] * (2 * k), w, h, k, s, lights=light_sets)
    assert not np.array_equal(got["rgb"][0], got["rgb"][1])
    got, hi = _check_accum(mt, [files.camera] * k, w, h, k, s)
    # identical sub-frames: the mean is the supersampled view itself
    assert np.array_equal(got["rgb"][0], mt.render_batch([files.camera], w, h, samples_per_axis=s)["rgb"][0])
    mt.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name,scale,w,h,k,s", [("C2", 0.1, 100, 75, 3, 2), ("C4", 1.0, 96, 64, 4, 1), ("C5", 1.0, 64, 40, 3, 4),
                                               ("C1", 1.0, 75, 49, 6, 8)])
def test_other_scenes(product_lib, scene_dir, name, scale, w, h, k, s):
    """C2 (textured), C4 (stress), C5 (4 lights, depth 8), C1 at sizes that are not multiples of 8; two output views of
    the orbit with a light set per sub-frame."""
    files, cfg = scenes.config_scene(name, scene_dir, scale)
    mt = _tracer(files.obj_path, cfg["depth"])
    cams = _orbit_subframes(files.camera, 2, k)
    rig = files.lights if len(files.lights) >= 2 else scenes.LIGHT_RIG[:2]
    light_sets = [_lights(rig) for _ in cams]
    light_sets[1] = _lights(scenes.LIGHT_RIG[:len(rig)])
    _check_accum(mt, cams, w, h, k, s, lights=light_sets)
    mt.close()


@pytest.mark.gpu
@pytest.mark.parametrize("s", [1, 2, 8])
def test_stats_equal_those_of_the_subframes(product_lib, scene_dir, s):
    from mythtracer_b200 import MTB_FLAG_COUNT_WORK
    files, cfg = scenes.config_scene("C1", scene_dir)
    w, h, k = 48, 32, 3
    cams = _orbit_subframes(files.camera, 2, k)
    light_sets = [_lights(scenes.LIGHT_RIG[j % 3:j % 3 + 2]) for j in range(len(cams))]
    mt = _tracer(files.obj_path, 4)
    got, hi = _check_accum(mt, cams, w, h, k, s, lights=light_sets)
    assert got["stats"]["kernel_ms"] > 0.0
    mt = _tracer(files.obj_path, 4, MTB_FLAG_COUNT_WORK)
    got, hi = _check_accum(mt, cams, w, h, k, s, lights=light_sets)
    for key, value in got["stats"].items():
        if not key.endswith("_ms"):
            assert value == hi["stats"][key], "counter %s" % key
    assert got["stats"]["n_bvh"] > 0 and got["stats"]["shadow"] > 0


@pytest.mark.gpu
def test_c_abi_k1_and_argument_errors(product_lib, scene_dir):
    """mtb_render_batch_accum with k = 1 is mtb_render_batch_ss; refused calls return MTB_ERR_ARG with a message."""
    from mythtracer_b200 import api
    files, cfg = scenes.config_scene("C1", scene_dir)
    mt = _tracer(files.obj_path, 3)
    mt.GetScene().lights = _lights(scenes.LIGHT_RIG[:2])
    mt.push_lights()
    n = 4
    cams = np.zeros(n, api.CAMERA_DTYPE)
    for i in range(n):
        cams[i] = api.Camera.from_tuple(_yawed(files.camera, 2.0 * i)).as_array()
    cam_ptr = cams.ctypes.data_as(ctypes.c_void_p)
    w, h = 40, 24
    rgb = np.zeros((n, h, w, 3), np.uint8)

    def call(n_out, k, s=1, w=w, h=h, depth=3):
        rc = product_lib.mtb_render_batch_accum(mt._ctx, cam_ptr, n_out, k, None, 0, w, h, s, depth, rgb.ctypes.data_as(ctypes.c_void_p), None)
        return rc, product_lib.mtb_last_error(mt._ctx).decode()

    for s in (1, 2, 4, 8):
        assert call(n, 1, s)[0] == MTB_OK
        want = np.zeros((n, h, w, 3), np.uint8)
        assert product_lib.mtb_render_batch_ss(mt._ctx, cam_ptr, n, None, 0, w, h, s, 3, want.ctypes.data_as(ctypes.c_void_p), None) == MTB_OK
        assert np.array_equal(rgb, want), "s = %d" % s
        assert np.array_equal(mt.render_batch([_yawed(files.camera, 2.0 * i) for i in range(n)], w, h, samples_per_axis=s, subframes=1)["rgb"], want)
    for args, words in (((1, 0), "subframes"), ((1, -3), "subframes"), ((0, 2), "n_out"), ((-1, 2), "n_out"), ((32768, 2), "n_out"),
                        ((2, 32768), "n_out"), ((2, 2, 3), "samples_per_axis"), ((2, 2, 8, 8193), "sample grid"),
                        ((2, 2, 1, w, h, 17), "render arguments")):
        rc, msg = call(*args)
        assert rc == MTB_ERR_ARG and words in msg, (args, rc, msg)
    assert call(2, 2)[0] == MTB_OK


@pytest.mark.gpu
def test_back_to_back_calls_of_different_shapes(product_lib, scene_dir):
    """Calls of different n_out, k, s and sizes in a row, each checked: the sums and arrival counters start from zero
    every time (a larger call first, then smaller ones that reuse its buffers)."""
    files, cfg = scenes.config_scene("C1", scene_dir)
    mt = _tracer(files.obj_path, 5)
    mt.GetScene().lights = _lights(scenes.LIGHT_RIG[:2])
    for n_out, k, s, w, h in ((4, 6, 2, 64, 48), (1, 2, 1, 64, 48), (3, 3, 4, 40, 30), (2, 7, 1, 33, 17), (4, 6, 2, 64, 48),
                              (5, 2, 8, 20, 12), (4, 6, 2, 64, 48)):
        _check_accum(mt, _orbit_subframes(files.camera, n_out, k), w, h, k, s)
    # the same call twice gives the same bytes (nothing left over from the first)
    cams = _orbit_subframes(files.camera, 2, 4)
    a = mt.render_batch(cams, 50, 30, subframes=4)["rgb"].copy()
    b = mt.render_batch(cams, 50, 30, subframes=4)["rgb"]
    assert np.array_equal(a, b)


@pytest.mark.gpu
def test_async_calls_into_pinned_memory(product_lib, scene_dir):
    """Two mtb_render_batch_accum_async calls of different shapes queued into two pinned buffers before one mtb_wait:
    both equal the synchronous results."""
    from mythtracer_b200 import api
    files, cfg = scenes.config_scene("C1", scene_dir)
    mt = _tracer(files.obj_path, 5)
    mt.GetScene().lights = _lights(scenes.LIGHT_RIG[:2])
    shapes = ((3, 4, 2, 64, 40), (2, 5, 1, 72, 36))
    product_lib.mtb_host_alloc.restype = ctypes.c_void_p
    product_lib.mtb_host_alloc.argtypes = [ctypes.c_size_t]
    product_lib.mtb_host_free.argtypes = [ctypes.c_void_p]
    wants, bufs, keep = [], [], []
    try:
        for n_out, k, s, w, h in shapes:
            cams = _orbit_subframes(files.camera, n_out, k)
            wants.append(mt.render_batch(cams, w, h, samples_per_axis=s, subframes=k)["rgb"].copy())
        mt.push_lights()
        for (n_out, k, s, w, h) in shapes:
            nbytes = n_out * h * w * 3
            buf = product_lib.mtb_host_alloc(nbytes)
            assert buf
            bufs.append(buf)
            ctypes.memset(buf, 0, nbytes)
            cam_arr = np.zeros(n_out * k, api.CAMERA_DTYPE)
            for i, c in enumerate(_orbit_subframes(files.camera, n_out, k)):
                cam_arr[i] = api.Camera.from_tuple(c).as_array()
            keep.append(cam_arr)
            rc = product_lib.mtb_render_batch_accum_async(mt._ctx, cam_arr.ctypes.data_as(ctypes.c_void_p), n_out, k, None, 0, w, h, s,
                                                          mt.max_depth, ctypes.c_void_p(buf))
            assert rc == MTB_OK, product_lib.mtb_last_error(mt._ctx)
        mt.wait()
        for (n_out, k, s, w, h), buf, want in zip(shapes, bufs, wants):
            nbytes = n_out * h * w * 3
            got = np.ctypeslib.as_array((ctypes.c_uint8 * nbytes).from_address(buf)).reshape(n_out, h, w, 3).copy()
            assert np.array_equal(got, want), (n_out, k, s, w, h)
    finally:
        for buf in bufs:
            product_lib.mtb_host_free(ctypes.c_void_p(buf))


@pytest.mark.gpu
def test_accumulation_leaves_the_single_frame_state_alone(product_lib, scene_dir):
    files, cfg = scenes.config_scene("C1", scene_dir)
    w, h = 160, 120
    mt = _tracer(files.obj_path, 3)  # automatic pipeline choice
    mt.GetScene().lights = _lights(scenes.LIGHT_RIG[:2])
    before = [mt.render_chunk(files.camera, w, h, 0, 0, w, h)["rgb"] for _ in range(8)]  # past the deciding frames
    pipeline = mt.pipeline_in_use()
    assert pipeline[0] != "measuring"
    mt.max_depth = 7
    for s in (1, 2, 8):
        mt.render_batch(_orbit_subframes(files.camera, 2, 3), 64, 48, lights=[_lights(scenes.LIGHT_RIG[1:4])] * 6, samples_per_axis=s,
                        subframes=3)
    mt.max_depth = 3
    after = mt.render_chunk(files.camera, w, h, 0, 0, w, h)["rgb"]
    assert np.array_equal(after, before[-1])
    assert mt.pipeline_in_use() == pipeline


@pytest.mark.gpu
def test_accumulated_views_split_over_devices(product_lib, scene_dir):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    files, cfg = scenes.config_scene("C1", scene_dir)
    w, h = 75, 49
    n = min(torch.cuda.device_count(), 8)
    one = _tracer(files.obj_path, 5)
    many = _tracer(files.obj_path, 5, devices=list(range(n)))
    assert many.device_count() == n
    for n_out, k, s in ((n + 3, 3, 1), (1, 5, 2), (n - 1, 4, 8), (2 * n, 2, 4)):
        cams = _orbit_subframes(files.camera, n_out, k)
        light_sets = [_lights(scenes.LIGHT_RIG[j % 3:j % 3 + 2]) for j in range(len(cams))]
        a = one.render_batch(cams, w, h, lights=light_sets, samples_per_axis=s, subframes=k)
        b = many.render_batch(cams, w, h, lights=light_sets, samples_per_axis=s, subframes=k)
        assert np.array_equal(b["rgb"], a["rgb"]), (n_out, k, s)
        assert b["stats"]["rays"] == a["stats"]["rays"]


def _build_apps():
    if shutil.which("g++") is None or shutil.which("make") is None:
        pytest.skip("g++/make not available")
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "apps")], stdout=subprocess.DEVNULL)


def _driver_rig():
    from mythtracer_b200 import Light
    rig = [(231.82174, 81.69966, -27.78259, 0.3, 0.3, 0.3, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0)] + [
        (200.0, 80.0, z, 0.0, 0.0, 0.0, 0.3, 0.3, 0.3, 0.3, 0.3, 0.3) for z in (0.0, 80.0, 160.0)]
    return [Light.from_tuple(l) for l in rig]


def _run_driver(obj, out_dir, W, H, extra):
    res = subprocess.run([os.path.join(ROOT, "apps", "_build", "mythtracer_local_b200"), obj, str(W), str(H), "74", "80", str(out_dir)] + extra,
                         capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stdout[-1500:] + res.stderr[-1500:]
    assert sorted(os.listdir(out_dir)) == ["dump_%05d.raw" % f for f in range(74, 81)]
    return res


@pytest.mark.gpu
@pytest.mark.parametrize("per_call,s", [(1, 1), (4, 2)])
def test_animation_driver_motion_blur(product_lib, scene_dir, tmp_path, per_call, s):
    """Frames 74..80 with subframes 4: every file equals render_batch(..., subframes=4) of the orbit cameras at the
    frame's angle a + 2 * j / 4 degrees."""
    from mythtracer_b200 import Camera, MythTracer
    _build_apps()
    files, cfg = scenes.config_scene("C1", scene_dir)
    W, H, k = 160, 90, 4
    res = _run_driver(files.obj_path, tmp_path / "anim", W, H, [str(per_call), str(s), str(k)])
    assert "in %d calls" % (7 if per_call == 1 else 2) in res.stdout
    mt = MythTracer(max_depth=5)
    assert mt.LoadObj(files.obj_path)
    mt.GetScene().lights = _driver_rig()
    cams = [Camera((300.0, 107.0, 40.0), 30.0, (2.0 * frame + 2.0 * j / k) + 90, 0.0, 110.0) for frame in range(74, 81) for j in range(k)]
    want = mt.render_batch(cams, W, H, samples_per_axis=s, subframes=k)["rgb"]
    for i, frame in enumerate(range(74, 81)):
        got = np.fromfile(tmp_path / "anim" / ("dump_%05d.raw" % frame), np.uint8).reshape(H, W, 3)
        assert np.array_equal(got, want[i]), "frame %d" % frame


@pytest.mark.gpu
def test_animation_driver_with_one_subframe_writes_the_frames_of_today(product_lib, scene_dir, tmp_path):
    """subframes 1 through the batch path (frames_per_call 4) and through the single-frame path (frames_per_call 1)
    writes the same files as without the argument, and they equal render_batch of the orbit cameras."""
    from mythtracer_b200 import Camera, MythTracer
    _build_apps()
    files, cfg = scenes.config_scene("C1", scene_dir)
    W, H = 120, 72
    outs = {}
    for name, extra in (("none", []), ("k1", ["1", "1", "1"]), ("batch_none", ["4"]), ("batch_k1", ["4", "1", "1"])):
        _run_driver(files.obj_path, tmp_path / name, W, H, extra)
        outs[name] = [(tmp_path / name / ("dump_%05d.raw" % f)).read_bytes() for f in range(74, 81)]
    assert outs["k1"] == outs["none"] and outs["batch_k1"] == outs["batch_none"] == outs["none"]
    mt = MythTracer(max_depth=5)
    assert mt.LoadObj(files.obj_path)
    mt.GetScene().lights = _driver_rig()
    want = mt.render_batch([Camera((300.0, 107.0, 40.0), 30.0, 2.0 * frame + 90, 0.0, 110.0) for frame in range(74, 81)], W, H)["rgb"]
    for i in range(7):
        assert outs["none"][i] == want[i].tobytes(), "frame %d" % (74 + i)


@pytest.mark.gpu
@pytest.mark.parametrize("s,k", [(1, 3), (2, 4)])
def test_cpp_shim_accumulated_batches(product_lib, scene_dir, tmp_path, s, k):
    """RayTraceBatch / RayTraceBatchAsync with subframes, called from C++ (tests/cpp/accum_check.cc): the output
    equals render_batch(..., subframes=k) of the same sub-frames."""
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    exe = str(tmp_path / "accum_check")
    lib_dir = os.path.join(ROOT, "mythtracer_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                           os.path.join(HERE, "cpp", "accum_check.cc"), "-L", lib_dir, "-lmythtracer_b200", "-Wl,-rpath," + lib_dir, "-o", exe])
    files, cfg = scenes.config_scene("C2", scene_dir, 0.1)
    W, H = 60, 36
    prefix = str(tmp_path / "out")
    res = subprocess.run([exe, files.obj_path, prefix, str(W), str(H), str(s), str(k)], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    assert "accum ok" in res.stdout
    mt = _tracer(files.obj_path, 3)
    mt.GetScene().lights = _lights([(231.82174, 81.69966, 27.78259, 0.3, 0.3, 0.3, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0),
                                    (200.0, 95.0, 160.0, 0.0, 0.0, 0.0, 0.3, 0.3, 0.3, 0.3, 0.3, 0.3)])
    cams = [(301.37, 57.21, 161.13, 4.0, 243.0 + 3.0 * v + 0.5 * j, 0.0, 110.0) for v in range(2) for j in range(k)]
    want = mt.render_batch(cams, W, H, samples_per_axis=s, subframes=k)["rgb"]
    got = np.fromfile(prefix + ".rgb", np.uint8).reshape(2, H, W, 3)
    assert np.array_equal(got, want)
    # and the formula over the sub-frames
    assert np.array_equal(want, _accum_mean(mt.render_batch(cams, s * W, s * H)["rgb"], k, s))
