"""Batches with per-pixel planes (mtb_render_batch_debug / render_batch(..., debug=True, taps=True)): for every view of a
batch with s samples per axis, the debug info (line_no and point of the primary hit) and the taps (sig_hits, sig_shadow,
n_rays) on the view's (s*W) x (s*H) sample grid.  Entry (x, y) of view v must be exactly what render_chunk returns for
pixel (x, y) of an (s*W) x (s*H) frame with that view's camera and lights - the planes the single-frame path is pinned
to the oracle and to the reference's own frames with - and asking for planes must not change the RGB or the stats."""
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
TAPS = ("sig_hits", "sig_shadow", "n_rays")


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _file_sha(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for blk in iter(lambda: f.read(1 << 20), b""):
            h.update(blk)
    return h.hexdigest()


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


def _singles(mt, cams, w, h, light_sets=None):
    """render_chunk(debug=True, taps=True) of every view with its own lights (None: the scene's lights)."""
    keep = list(mt.GetScene().lights)
    out = []
    for i, cam in enumerate(cams):
        if light_sets is not None:
            mt.GetScene().lights = _lights(light_sets[i])
        out.append(mt.render_chunk(cam, w, h, 0, 0, w, h, debug=True, taps=True))
    mt.GetScene().lights = keep
    return out


def _assert_planes_equal(got, want, what):
    """Every plane of `got` (one view) equals `want`'s; points bit for bit (NaN on a miss included)."""
    assert np.array_equal(got["line_no"], want["line_no"]), "%s: %d primary hit ids differ" % (
        what, int((got["line_no"] != want["line_no"]).sum()))
    assert got["points"].tobytes() == want["points"].tobytes(), "%s: hit points differ" % what
    assert got["debug"].tobytes() == want["debug"].tobytes(), "%s: debug records differ" % what
    for k in TAPS:
        assert np.array_equal(got[k], want[k]), "%s: %s differs" % (what, k)


def _view(res, v):
    return {k: res[k][v] for k in ("debug", "line_no", "points") + TAPS if k in res}


def _assert_same_render(a, b, what):
    """RGB byte for byte and every stat but the timings."""
    assert np.array_equal(a["rgb"], b["rgb"]), "%s: RGB differs" % what
    for k, value in a["stats"].items():
        if not k.endswith("_ms"):
            assert value == b["stats"][k], "%s: stat %s" % (what, k)


# ---------------------------------------------------------------------------------------------- CPU


def test_batch_planes_have_no_cpu_fallback(product_lib):
    from mythtracer_b200 import MythTracer, MythTracerError
    files, cfg = scenes.config_scene("C1", "/tmp/mtb_scenes")
    mt = MythTracer(host_only=True)
    assert mt.LoadObj(files.obj_path)
    for kw in (dict(debug=True), dict(taps=True), dict(debug=True, taps=True, samples_per_axis=2)):
        with pytest.raises(MythTracerError, match="no CPU fallback"):
            mt.render_batch([files.camera, files.camera], 16, 16, **kw)


def test_batch_plane_arguments_are_checked_in_python(product_lib):
    from mythtracer_b200 import MythTracer, MythTracerError
    files, cfg = scenes.config_scene("C1", "/tmp/mtb_scenes")
    mt = MythTracer(host_only=True)
    assert mt.LoadObj(files.obj_path)
    cams = [files.camera, files.camera]
    for bad in (1, 0, "yes", None, np.array([True])):
        with pytest.raises(MythTracerError, match="debug must be True or False"):
            mt.render_batch(cams, 16, 16, debug=bad)
        with pytest.raises(MythTracerError, match="taps must be True or False"):
            mt.render_batch(cams, 16, 16, taps=bad)
    # the checks of the call without planes still apply
    with pytest.raises(MythTracerError, match="samples_per_axis"):
        mt.render_batch(cams, 16, 16, samples_per_axis=3, debug=True)
    with pytest.raises(MythTracerError, match="out must be"):
        mt.render_batch(cams, 16, 16, out=np.zeros((2, 32, 32, 3), np.uint8), samples_per_axis=2, taps=True)
    with pytest.raises(MythTracerError, match="one per view"):
        mt.render_batch(cams, 16, 16, lights=[_lights(scenes.LIGHT_RIG[:2])], debug=True)
    with pytest.raises(MythTracerError, match="no cameras"):
        mt.render_batch([], 16, 16, debug=True, taps=True)


# ---------------------------------------------------------------------------------------------- GPU


@pytest.mark.gpu
def test_planes_of_every_view_equal_render_chunk_and_the_oracle(product_lib, oracle_mod, scene_dir):
    """C1 at 150x97 (edge tiles), depth 5, five views with their own yaw and their own two lights."""
    from mythtracer_b200 import MTB_FLAG_MEGAKERNEL
    files, cfg = scenes.config_scene("C1", scene_dir)
    w, h, depth = 150, 97, 5
    rig = scenes.LIGHT_RIG
    cams = [_yawed(files.camera, 6.0 * k - 12.0) for k in range(5)]
    light_sets = [[rig[k % 4], rig[(k + 1) % 4]] for k in range(5)]
    mt = _tracer(files.obj_path, depth, MTB_FLAG_MEGAKERNEL)
    lights = [_lights(ls) for ls in light_sets]
    got = mt.render_batch(cams, w, h, lights=lights, debug=True, taps=True)
    for k in ("line_no", "points", "debug") + TAPS:
        assert got[k].shape[:3] == (5, h, w), k
    _assert_same_render(got, mt.render_batch(cams, w, h, lights=lights), "planes vs no planes")
    # one of the two kinds at a time returns the same planes
    only_dbg = mt.render_batch(cams, w, h, lights=lights, debug=True)
    only_taps = mt.render_batch(cams, w, h, lights=lights, taps=True)
    assert not any(k in only_dbg for k in TAPS) and "debug" not in only_taps
    assert only_dbg["debug"].tobytes() == got["debug"].tobytes()
    for k in TAPS:
        assert np.array_equal(only_taps[k], got[k]), k
    assert (got["line_no"] >= 0).any()
    for v, single in enumerate(_singles(mt, cams, w, h, light_sets)):
        _assert_planes_equal(_view(got, v), single, "view %d against render_chunk" % v)
    orc = oracle_mod.Oracle.from_obj(files.obj_path)
    for v in range(5):
        orc.set_lights(light_sets[v])
        cpu = orc.render(cams[v], w, h, depth=depth, taps=True)
        assert np.array_equal(got["line_no"][v], cpu["line_no"]), "view %d: primary hit ids against the oracle" % v
        assert np.array_equal(got["points"][v], cpu["points"], equal_nan=True), "view %d: hit points against the oracle" % v
        for k in TAPS:
            assert np.array_equal(got[k][v], cpu[k]), "view %d: %s against the oracle" % (v, k)


@pytest.mark.gpu
@pytest.mark.parametrize("s", [2, 4, 8])
def test_sample_grid_planes_equal_those_of_the_high_resolution_batch(product_lib, scene_dir, s):
    """C1 at 75x49 (odd sides; partial edge tiles of the sample grid for s = 2 and 4), per-view lights, depth 5."""
    files, cfg = scenes.config_scene("C1", scene_dir)
    w, h = 75, 49
    rig = scenes.LIGHT_RIG
    cams = [_yawed(files.camera, 6.0 * k - 12.0) for k in range(5)]
    lights = [_lights([rig[k % 4], rig[(k + 1) % 4]]) for k in range(5)]
    mt = _tracer(files.obj_path, 5)
    got = mt.render_batch(cams, w, h, lights=lights, samples_per_axis=s, debug=True, taps=True)
    assert got["rgb"].shape == (5, h, w, 3)
    for k in ("line_no", "points", "debug") + TAPS:
        assert got[k].shape[:3] == (5, s * h, s * w), k
    _assert_same_render(got, mt.render_batch(cams, w, h, lights=lights, samples_per_axis=s), "s = %d: planes vs no planes" % s)
    hi = mt.render_batch(cams, s * w, s * h, lights=lights, debug=True, taps=True)
    for v in range(5):
        _assert_planes_equal(_view(got, v), _view(hi, v), "s = %d, view %d against the %dx%d batch" % (s, v, s * w, s * h))
    # ... and view 0 against render_chunk of the sample grid
    one = _singles(mt, cams[:1], s * w, s * h, [[scenes.LIGHT_RIG[0], scenes.LIGHT_RIG[1]]])[0]
    _assert_planes_equal(_view(got, 0), one, "s = %d, view 0 against render_chunk" % s)


def _golden(name, scene_dir):
    z = np.load(os.path.join(HERE, "golden", "full_%s.npz" % name))
    files, cfg = scenes.config_scene(name, scene_dir)
    assert _file_sha(files.obj_path) == str(z["obj_sha256"]), "generated %s scene differs from the fixture's scene" % name
    assert _file_sha(files.mtl_path) == str(z["mtl_sha256"])
    assert int(z["depth"]) == cfg["depth"] and len(z["rows"]) == int(z["height"])
    return z, files, cfg


def _assert_reference_planes(line_no, points, z, what):
    rows = z["rows"]
    assert np.array_equal(line_no[rows], z["line_no"]), "%s: %d primary hit ids differ from the reference's" % (
        what, int((line_no[rows] != z["line_no"]).sum()))
    assert _sha(line_no[rows]) == str(z["line_no_sha256"])
    assert _sha(points[rows]) == str(z["points_sha256"]), "%s: hit points differ from the reference's" % what


@pytest.mark.gpu
def test_c3_views_carry_the_reference_planes(product_lib, scene_dir):
    """A 1080p C3 batch of 4 views with the reference's camera as view 2 (tests/golden/full_C3.npz), and C3 at 960x540
    with s = 2, whose sample grid is the reference's 1080p frame."""
    z, files, cfg = _golden("C3", scene_dir)
    W, H = int(z["width"]), int(z["height"])
    mt = _tracer(files.obj_path, cfg["depth"])
    mt.GetScene().lights = _lights(files.lights)
    cams = [_yawed(files.camera, -4.0), _yawed(files.camera, 2.0), files.camera, _yawed(files.camera, 7.0)]
    got = mt.render_batch(cams, W, H, debug=True)
    _assert_reference_planes(got["line_no"][2], got["points"][2], z, "C3 batch view 2")
    assert not np.array_equal(got["line_no"][1], got["line_no"][2])
    ss = mt.render_batch([files.camera], W // 2, H // 2, samples_per_axis=2, debug=True)
    assert ss["line_no"].shape == (1, H, W)
    _assert_reference_planes(ss["line_no"][0], ss["points"][0], z, "C3 960x540, s = 2")
    mt.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["C2", "C4", "C5"])
def test_one_view_batches_carry_the_reference_planes(product_lib, scene_dir, name):
    z, files, cfg = _golden(name, scene_dir)
    mt = _tracer(files.obj_path, cfg["depth"])
    mt.GetScene().lights = _lights(files.lights)
    got = mt.render_batch([files.camera], int(z["width"]), int(z["height"]), debug=True)
    _assert_reference_planes(got["line_no"][0], got["points"][0], z, name)
    mt.close()


@pytest.mark.gpu
def test_light_depth_and_view_count_edge_cases(product_lib, scene_dir):
    """lights=None (the scene's lights), no lights at all, depths 0 and 8, one view and 64 views."""
    files, cfg = scenes.config_scene("C1", scene_dir)
    w, h = 40, 27
    mt = _tracer(files.obj_path, 5)
    mt.GetScene().lights = _lights(scenes.LIGHT_RIG[:3])
    for depth in (0, 8):
        mt.max_depth = depth
        for n in (1, 64):
            cams = [_yawed(files.camera, 1.5 * k) for k in range(n)]
            for light_sets in (None, [[] for _ in cams]):
                lights = None if light_sets is None else [_lights(ls) for ls in light_sets]
                what = "depth %d, %d views, %s" % (depth, n, "scene lights" if light_sets is None else "no lights")
                got = mt.render_batch(cams, w, h, lights=lights, debug=True, taps=True)
                _assert_same_render(got, mt.render_batch(cams, w, h, lights=lights), what)
                for v, single in enumerate(_singles(mt, cams, w, h, light_sets)):
                    _assert_planes_equal(_view(got, v), single, "%s: view %d" % (what, v))


@pytest.mark.gpu
def test_textured_views(product_lib, scene_dir):
    files, cfg = scenes.config_scene("C2", scene_dir)
    w, h = 320, 180
    mt = _tracer(files.obj_path, cfg["depth"])
    assert mt.scene_info()["n_textures"] > 0
    mt.GetScene().lights = _lights(files.lights)
    cams = [_yawed(files.camera, d) for d in (-3.0, 0.0, 5.0)]
    got = mt.render_batch(cams, w, h, debug=True, taps=True)
    _assert_same_render(got, mt.render_batch(cams, w, h), "C2")
    for v, single in enumerate(_singles(mt, cams, w, h)):
        _assert_planes_equal(_view(got, v), single, "C2 view %d" % v)


@pytest.mark.gpu
@pytest.mark.parametrize("s", [1, 2])
def test_counting_build(product_lib, scene_dir, s):
    """MTB_FLAG_COUNT_WORK: the planes are those of the fast build, and every counter equals the plain batch's."""
    from mythtracer_b200 import MTB_FLAG_COUNT_WORK
    files, cfg = scenes.config_scene("C1", scene_dir)
    w, h = 48, 32
    cams = [_yawed(files.camera, 4.0 * k) for k in range(4)]
    rig = scenes.LIGHT_RIG
    lights = [_lights([rig[k % 4], rig[(k + 1) % 4]]) for k in range(4)]
    fast = _tracer(files.obj_path, 4).render_batch(cams, w, h, lights=lights, samples_per_axis=s, debug=True, taps=True)
    mt = _tracer(files.obj_path, 4, MTB_FLAG_COUNT_WORK)
    got = mt.render_batch(cams, w, h, lights=lights, samples_per_axis=s, debug=True, taps=True)
    _assert_same_render(got, mt.render_batch(cams, w, h, lights=lights, samples_per_axis=s), "counting build, s = %d" % s)
    assert got["stats"]["n_bvh"] > 0 and got["stats"]["shadow"] > 0
    assert np.array_equal(got["rgb"], fast["rgb"])
    for v in range(len(cams)):
        _assert_planes_equal(_view(got, v), _view(fast, v), "counting build, s = %d, view %d" % (s, v))


@pytest.mark.gpu
def test_batch_planes_leave_the_single_frame_state_alone(product_lib, scene_dir):
    """Both ways: render_chunk's planes are the same before and after a batch with planes, and a batch without planes
    after one with planes returns what it returned before (its kernel gets no planes)."""
    files, cfg = scenes.config_scene("C1", scene_dir)
    w, h = 160, 120
    mt = _tracer(files.obj_path, 3)  # automatic pipeline choice
    mt.GetScene().lights = _lights(scenes.LIGHT_RIG[:2])
    before = [mt.render_chunk(files.camera, w, h, 0, 0, w, h, debug=True, taps=True) for _ in range(6)]  # past the deciding frames
    pipeline = mt.pipeline_in_use()
    assert pipeline[0] != "measuring"
    bcams = [_yawed(files.camera, 10.0)] * 3
    blights = [_lights(scenes.LIGHT_RIG[1:4])] * 3
    plain_before = mt.render_batch(bcams, 64, 48, lights=blights)
    mt.max_depth = 7
    big = mt.render_batch([files.camera] * 4, 200, 150, lights=blights[:1] * 4, debug=True, taps=True)
    mt.max_depth = 3
    after = mt.render_chunk(files.camera, w, h, 0, 0, w, h, debug=True, taps=True)
    assert np.array_equal(after["rgb"], before[-1]["rgb"])
    _assert_planes_equal(after, before[-1], "render_chunk after a batch with planes")
    assert mt.pipeline_in_use() == pipeline
    plain_after = mt.render_batch(bcams, 64, 48, lights=blights)
    _assert_same_render(plain_after, plain_before, "plain batch after a batch with planes")
    # a smaller batch with planes into the grown buffers
    small = mt.render_batch(bcams, 64, 48, lights=blights, debug=True, taps=True)
    _assert_same_render(small, plain_before, "smaller batch with planes")
    singles = _singles(mt, bcams[:1], 64, 48, [scenes.LIGHT_RIG[1:4]])
    _assert_planes_equal(_view(small, 0), singles[0], "smaller batch with planes, view 0")
    assert big["line_no"].shape == (4, 150, 200)


@pytest.mark.gpu
def test_bad_batch_debug_arguments(product_lib, scene_dir):
    """The C ABI: each refused call returns MTB_ERR_ARG with a message; NULL planes (or a taps struct of NULL pointers)
    make the call mtb_render_batch_ss; a single tap plane may be asked for alone."""
    from mythtracer_b200 import MythTracer, api
    files, cfg = scenes.config_scene("C1", scene_dir)
    mt = MythTracer(max_depth=3)
    assert mt.LoadObj(files.obj_path)
    mt.GetScene().lights = _lights(scenes.LIGHT_RIG[:2])
    mt.push_lights()
    cams = np.zeros(2, api.CAMERA_DTYPE)
    for v in range(2):
        cams[v] = api.Camera.from_tuple(_yawed(files.camera, 5.0 * v)).as_array()
    cam_ptr = cams.ctypes.data_as(ctypes.c_void_p)
    w, h = 16, 8
    rgb = np.zeros((2, h, w, 3), np.uint8)

    def ptr(a):
        return None if a is None else a.ctypes.data_as(ctypes.c_void_p)

    def call(s=2, n=2, cam=cam_ptr, ww=w, depth=3, out=rgb, dbg=None, taps=None):
        tap_ptr = None if taps is None else ctypes.cast(ctypes.pointer(taps), ctypes.c_void_p)
        rc = product_lib.mtb_render_batch_debug(mt._ctx, cam, n, None, 0, ww, h, s, depth, ptr(out), ptr(dbg), tap_ptr, None)
        return rc, product_lib.mtb_last_error(mt._ctx).decode()

    dbg = np.zeros((2, 2 * h, 2 * w), api.DEBUG_DTYPE)
    for kw, words in ((dict(n=0), "n_views"), (dict(n=65536), "n_views"), (dict(depth=17), "render arguments"),
                      (dict(cam=None), "cams"), (dict(out=None), "rgb_out"), (dict(s=3), "samples_per_axis"),
                      (dict(s=0), "samples_per_axis"), (dict(s=8, ww=8193), "sample grid")):
        rc, msg = call(dbg=dbg, **kw)
        assert rc == MTB_ERR_ARG and words in msg, (kw, rc, msg)
    mt.set_partition(1, 2)
    rc, msg = call(dbg=dbg)
    assert rc == MTB_ERR_ARG and "partition" in msg
    mt.set_partition(0, 1)

    # with every plane NULL the call is mtb_render_batch_ss
    want = np.zeros_like(rgb)
    assert product_lib.mtb_render_batch_ss(mt._ctx, cam_ptr, 2, None, 0, w, h, 2, 3, ptr(want), None) == MTB_OK
    assert call()[0] == MTB_OK and np.array_equal(rgb, want)
    rgb[:] = 0
    assert call(taps=api._TapsStruct(None, None, None))[0] == MTB_OK and np.array_equal(rgb, want)
    full = mt.render_batch([_yawed(files.camera, 5.0 * v) for v in range(2)], w, h, samples_per_axis=2, debug=True, taps=True)
    assert np.array_equal(full["rgb"], want)
    assert call(dbg=dbg)[0] == MTB_OK and dbg.tobytes() == full["debug"].tobytes()
    for k in TAPS:
        plane = np.zeros_like(full[k])
        fields = {f: (plane.ctypes.data if f == k else None) for f in TAPS}
        rc, msg = call(taps=api._TapsStruct(fields["sig_hits"], fields["sig_shadow"], fields["n_rays"]))
        assert rc == MTB_OK, msg
        assert np.array_equal(plane, full[k]), k


@pytest.mark.gpu
def test_batch_planes_split_over_devices(product_lib, scene_dir):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    files, cfg = scenes.config_scene("C1", scene_dir)
    w, h = 75, 49
    cams = [_yawed(files.camera, 3.0 * k) for k in range(5)]
    lights = [_lights(scenes.LIGHT_RIG[k % 3:k % 3 + 2]) for k in range(5)]
    n = min(torch.cuda.device_count(), 8)
    one = _tracer(files.obj_path, 5)
    many = _tracer(files.obj_path, 5, devices=list(range(n)))
    assert many.device_count() == n
    for s in (1, 2):
        a = one.render_batch(cams, w, h, lights=lights, samples_per_axis=s, debug=True, taps=True)
        b = many.render_batch(cams, w, h, lights=lights, samples_per_axis=s, debug=True, taps=True)
        assert np.array_equal(b["rgb"], a["rgb"]), "s = %d" % s
        assert b["stats"]["rays"] == a["stats"]["rays"]
        for v in range(len(cams)):
            _assert_planes_equal(_view(b, v), _view(a, v), "s = %d, view %d on %d devices" % (s, v, n))


@pytest.mark.gpu
@pytest.mark.parametrize("s", [1, 2])
def test_cpp_batch_debug_overload(product_lib, scene_dir, tmp_path, s):
    """RayTraceBatch(..., std::vector<PerPixelDebugInfo> *) of include/mythtracer/mythtracer.h, from a program of its
    own (tests/cpp/batch_debug_check.cc): its outputs equal render_batch(debug=True) of the same views."""
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    exe = str(tmp_path / "batch_debug_check")
    lib_dir = os.path.join(ROOT, "mythtracer_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                           os.path.join(HERE, "cpp", "batch_debug_check.cc"), "-L", lib_dir, "-lmythtracer_b200",
                           "-Wl,-rpath," + lib_dir, "-o", exe])
    files, cfg = scenes.config_scene("C2", scene_dir, 0.1)
    W, H = 60, 36
    prefix = str(tmp_path / "out")
    res = subprocess.run([exe, files.obj_path, prefix, str(W), str(H), str(s)], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    assert "batch debug ok" in res.stdout
    from mythtracer_b200 import api
    mt = _tracer(files.obj_path, 3)
    mt.GetScene().lights = _lights([(231.82174, 81.69966, 27.78259, 0.3, 0.3, 0.3, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0),
                                    (200.0, 95.0, 160.0, 0.0, 0.0, 0.0, 0.3, 0.3, 0.3, 0.3, 0.3, 0.3)])
    cams = [(301.37, 57.21, 161.13, 4.0, 243.0 + 3.0 * v, 0.0, 110.0) for v in range(3)]
    want = mt.render_batch(cams, W, H, samples_per_axis=s, debug=True)
    got_rgb = np.fromfile(prefix + ".rgb", np.uint8).reshape(3, H, W, 3)
    got_dbg = np.fromfile(prefix + ".dbg", api.DEBUG_DTYPE).reshape(3, s * H, s * W)
    assert np.array_equal(got_rgb, want["rgb"])
    assert got_dbg.tobytes() == want["debug"].tobytes()
