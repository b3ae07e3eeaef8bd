"""Thin-lens batches (mtb_render_batch_lens / render_batch(..., lenses=...)): depth of field as the mean of sub-frames
whose primary rays start on a lens point and pass through a common focal plane.  The lens rays are restated here in
numpy from the oracle's sensor and the formula of include/mythtracer_b200.h, and mto_render_rays (tests/cpp/oracle_rays.cc:
the oracle's per-pixel body with the primary ray given) traces them with the reference's TraceRay; a centred sample is
the pinhole ray, so it is also pinned to the plain batches and to the reference's stored frame
(tests/golden/full_C3.npz)."""
import ctypes
import math
import os
import shutil
import subprocess

import numpy as np
import pytest

from tests import scenes
from tests.test_accumulate import _accum_mean, _jittered_lights, _lights, _orbit_subframes, _tracer, _yawed

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")
MTB_OK, MTB_ERR_ARG = 0, -1
TAPS = ("sig_hits", "sig_shadow", "n_rays")
# the shading's pow() of CUDA and of glibc differ by <= 2 ulp (tests/test_gpu_parity.py): RGB may differ by one LSB
MAX_RGB_DIFF, MAX_RGB_FRACTION = 1, 1e-4


# ---------------------------------------------------------------------------------------------- the restatement


def _cross(t, a):
    return (t[1] * a[2] - t[2] * a[1], t[2] * a[0] - t[0] * a[2], t[0] * a[1] - t[1] * a[0])


def _dot(a, b):
    return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]


def _normalized(a):
    n = math.sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2])
    return (a[0] / n, a[1] / n, a[2] / n)


def _pinhole_dirs(sensor, w, h):
    """Normalized(S + Dy * Y + Dx * X) for every sample (X, Y) of a w x h grid, FP64 in the kernel's order: (h, w) arrays
    of the three components."""
    S, Dy, Dx = sensor
    Y, X = np.arange(h, dtype=np.float64)[:, None], np.arange(w, dtype=np.float64)[None, :]
    p = [(S[a] + Dy[a] * Y) + Dx[a] * X for a in range(3)]
    n = np.sqrt((p[0] * p[0] + p[1] * p[1]) + p[2] * p[2])
    return [p[a] / n for a in range(3)]


def _lens_rays(cam, sensor, w, h, lens):
    """(origins, dirs), each (h, w, 3): the primary rays of one sub-frame with lens sample (u, v, f)."""
    u, v, f = lens
    S, Dy, Dx = (tuple(float(x) for x in r) for r in sensor)
    O = tuple(float(x) for x in cam[0:3])
    d = _pinhole_dirs((S, Dy, Dx), w, h)
    if u == 0.0 and v == 0.0:
        return np.broadcast_to(np.array(O), (h, w, 3)).copy(), np.stack(d, axis=-1)
    n = _normalized(_cross(Dy, Dx))
    if _dot(n, S) < 0:
        n = tuple(-x for x in n)
    ex = _normalized(Dx)
    ey = _cross(n, ex)
    if _dot(ey, Dy) < 0:
        ey = tuple(-x for x in ey)
    L = tuple(ex[a] * u + ey[a] * v for a in range(3))
    t = f / ((d[0] * n[0] + d[1] * n[1]) + d[2] * n[2])
    q = [d[a] * t - L[a] for a in range(3)]
    norm = np.sqrt((q[0] * q[0] + q[1] * q[1]) + q[2] * q[2])
    origin = tuple(O[a] + L[a] for a in range(3))
    return np.broadcast_to(np.array(origin), (h, w, 3)).copy(), np.stack([q[a] / norm for a in range(3)], axis=-1)


def _disc(rng, n, radius):
    """n seeded points of a disc of `radius` (Shirley-Chiu concentric mapping of the unit square)."""
    out = []
    for a, b in 2.0 * rng.random((n, 2)) - 1.0:
        if a == 0.0 and b == 0.0:
            out.append((0.0, 0.0))
            continue
        if abs(a) > abs(b):
            r, phi = a, math.pi / 4 * (b / a)
        else:
            r, phi = b, math.pi / 2 - math.pi / 4 * (a / b)
        out.append((radius * r * math.cos(phi), radius * r * math.sin(phi)))
    return out


def _aperture(rng, n, radius, focus):
    return [(u, v, focus) for u, v in _disc(rng, n, radius)]


def _scale(orc):
    box = orc.aabb()
    return float(np.linalg.norm(box[3:] - box[:3]))


@pytest.fixture(scope="module")
def rays_oracle(oracle_mod, tmp_path_factory):
    """oracle_py.Oracle on a library built from tests/cpp/oracle_rays.cc (the oracle's source with mto_render_rays),
    with the flags of oracle/Makefile, in a temporary directory; its render_rays(origins, dirs, ...) returns what
    render(...) returns, one pixel per given primary ray."""
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    so = str(tmp_path_factory.mktemp("oracle_rays") / "liboracle_rays.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fopenmp", "-fPIC", "-ffp-contract=off", "-Wall", "-Wextra", "-D_USE_MATH_DEFINES",
                           # (mt_oracle.cc is an included file here, which makes g++ warn about its anonymous-namespace members)
                           "-Wno-subobject-linkage",
                           "-shared", "-I", os.path.join(ROOT, "oracle"), os.path.join(HERE, "cpp", "oracle_rays.cc"), "-o", so])
    lib = ctypes.CDLL(so)
    vp = ctypes.c_void_p
    lib.mto_create.restype = vp
    lib.mto_create.argtypes = [vp, ctypes.c_int64, vp, ctypes.c_int32, vp, ctypes.c_int32]
    lib.mto_destroy.argtypes = [vp]
    lib.mto_set_lights.argtypes = [vp, vp, ctypes.c_int32]
    lib.mto_scene_aabb.argtypes = [vp, vp]
    lib.mto_render.argtypes = [vp, vp] + [ctypes.c_int] * 7 + [vp] * 5
    lib.mto_camera_sensor.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp]
    lib.mto_camera_ray.argtypes = [vp] + [ctypes.c_int] * 4 + [vp]
    lib.mto_render_rays.argtypes = [vp, ctypes.c_int64, vp, vp, ctypes.c_int] + [vp] * 5

    class RaysOracle(oracle_mod.Oracle):
        _lib = lib

        def render_rays(self, origins, dirs, depth=5, taps=False):
            o = np.ascontiguousarray(origins, np.float64)
            d = np.ascontiguousarray(dirs, np.float64)
            assert o.shape == d.shape and o.shape[-1] == 3, (o.shape, d.shape)
            shape = o.shape[:-1]
            rgb = np.zeros(shape + (3,), np.uint8)
            line_no = np.zeros(shape, np.int32)
            points = np.zeros(shape + (3,), np.float64)
            stats = np.zeros(len(oracle_mod.STATS_FIELDS), np.uint64)
            res, tap_ptr = {}, None
            if taps:
                res["sig_hits"] = np.zeros(shape, np.uint64)
                res["sig_shadow"] = np.zeros(shape, np.uint64)
                res["n_rays"] = np.zeros(shape, np.uint32)
                tap_struct = oracle_mod.TapsStruct(res["sig_hits"].ctypes.data, res["sig_shadow"].ctypes.data, res["n_rays"].ctypes.data)
                tap_ptr = ctypes.cast(ctypes.pointer(tap_struct), vp)
            ptr = lambda a: a.ctypes.data_as(vp)  # noqa: E731
            rc = lib.mto_render_rays(self.handle, int(np.prod(shape)), ptr(o), ptr(d), depth, ptr(rgb), ptr(line_no), ptr(points), tap_ptr,
                                     ptr(stats))
            assert rc == 0
            res.update(rgb=rgb, line_no=line_no, points=points, stats=dict(zip(oracle_mod.STATS_FIELDS, [int(x) for x in stats])))
            return res

    return RaysOracle


def _golden_case(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    return z, os.path.join(GOLDEN, name + ".obj")


# ---------------------------------------------------------------------------------------------- CPU


@pytest.mark.parametrize("name", ["room_small", "lattice", "room_textured"])
def test_render_rays_with_the_pinhole_rays_is_render(oracle_mod, rays_oracle, name):
    """mto_render_rays fed a camera's own primary rays (restated in numpy) gives the oracle's mto_render bytes, hit ids,
    points, taps and work counters."""
    z, obj = _golden_case(name)
    ref = oracle_mod.Oracle.from_obj(obj)
    ref.set_lights(z["lights"].tolist())
    cam, w, h, depth = z["camera"].tolist(), int(z["width"]), int(z["height"]), int(z["depth"])
    want = ref.render(cam, w, h, depth=depth, taps=True)
    orc = rays_oracle.from_obj(obj)
    orc.set_lights(z["lights"].tolist())
    o, d = _lens_rays(cam, oracle_mod.Oracle.camera_sensor(cam, w, h), w, h, (0.0, 0.0, 1.0))
    for y, x in ((0, 0), (h // 2, w // 3), (h - 1, w - 1)):
        assert np.array_equal(d[y, x], orc.camera_ray(cam, w, h, x, y))
    got = orc.render_rays(o, d, depth=depth, taps=True)
    assert np.array_equal(got["rgb"], want["rgb"]) and np.array_equal(got["rgb"], z["rgb"])
    assert np.array_equal(got["line_no"], want["line_no"])
    assert np.array_equal(got["points"], want["points"], equal_nan=True)
    for k in TAPS:
        assert np.array_equal(got[k], want[k]), k
    assert got["stats"] == want["stats"]


def test_lens_rays_of_the_restatement():
    """The formula's geometry: every lens ray of a sub-frame meets its pinhole ray on the focal plane, and a centred
    sample is the pinhole ray itself."""
    from oracle import oracle_py
    cam = (10.0, 5.0, -3.0, 12.0, 40.0, 3.0, 80.0)
    w, h, f = 24, 16, 37.5
    sensor = oracle_py.Oracle.camera_sensor(cam, w, h)
    o0, d0 = _lens_rays(cam, sensor, w, h, (0.0, 0.0, f))
    o1, d1 = _lens_rays(cam, sensor, w, h, (1.5, -0.75, f))
    assert np.array_equal(o0[0, 0], np.array(cam[:3])) and not np.array_equal(d0, d1)
    n = np.cross(sensor[1], sensor[2])
    n /= np.linalg.norm(n)
    n = n if np.dot(n, sensor[0]) > 0 else -n
    focal0 = o0 + d0 * (f / (d0 @ n))[..., None]
    focal1 = o1 + d1 * ((f - (o1 - o0) @ n) / (d1 @ n))[..., None]
    np.testing.assert_allclose(focal1, focal0, rtol=0, atol=1e-9)
    # the lens point lies in the plane of the sensor axes, u along the image's right and v along its down direction
    L = o1[0, 0] - np.array(cam[:3])
    assert abs(np.dot(L, n)) < 1e-12
    assert np.dot(L, sensor[2]) > 0 and np.dot(L, sensor[1]) < 0


def test_lenses_have_no_cpu_fallback(product_lib):
    from mythtracer_b200 import MythTracer, MythTracerError
    files, cfg = scenes.config_scene("C1", "/tmp/mtb_scenes")
    mt = MythTracer(host_only=True)
    assert mt.LoadObj(files.obj_path)
    with pytest.raises(MythTracerError, match="no CPU fallback"):
        mt.render_batch([files.camera] * 2, 16, 16, lenses=[(0.5, 0.0, 10.0)] * 2, subframes=2)


def test_lens_arguments_are_checked_in_python(product_lib):
    from mythtracer_b200 import MythTracer, MythTracerError
    files, cfg = scenes.config_scene("C1", "/tmp/mtb_scenes")
    mt = MythTracer(host_only=True)
    assert mt.LoadObj(files.obj_path)
    cams = [files.camera] * 4
    good = [(0.5, -0.5, 10.0)] * 4
    for lenses, words in ((good[:3], "shape"), (good + good[:1], "shape"), ([(0.5, 10.0)] * 4, "shape"), (np.zeros((4, 3, 1)), "shape"),
                          ([0.5, 0.5, 10.0, 1.0], "shape"), ("abc", "sequence"), ([("a", 0.0, 1.0)] * 4, "numbers"),
                          ([(float("nan"), 0.0, 1.0)] + good[1:], "finite"), ([(0.0, float("inf"), 1.0)] + good[1:], "finite"),
                          (good[:3] + [(0.0, 0.0, float("inf"))], "finite"), (good[:3] + [(0.0, 0.0, 0.0)], "focus_distance"),
                          ([(0.0, 0.0, -2.0)] * 4, "focus_distance")):
        for device in (False, True):
            with pytest.raises(MythTracerError, match=words):
                mt.render_batch(cams, 16, 16, lenses=lenses, subframes=2, device=device)
    # the other argument rules hold with lenses too
    with pytest.raises(MythTracerError, match="debug and taps"):
        mt.render_batch(cams, 16, 16, lenses=good, subframes=2, debug=True)
    with pytest.raises(MythTracerError, match="samples_per_axis"):
        mt.render_batch(cams, 16, 16, lenses=good, samples_per_axis=3)


# ---------------------------------------------------------------------------------------------- GPU


def _assert_like_oracle(got, v, cpu, what):
    assert np.array_equal(got["line_no"][v], cpu["line_no"]), "%s: %d primary hit ids differ" % (
        what, int((got["line_no"][v] != cpu["line_no"]).sum()))
    assert np.array_equal(got["points"][v], cpu["points"], equal_nan=True), "%s: hit points differ" % what
    for k in TAPS:
        assert np.array_equal(got[k][v], cpu[k]), "%s: %s differs" % (what, k)
    diff = np.abs(got["rgb"][v].astype(int) - cpu["rgb"].astype(int))
    assert diff.max() <= MAX_RGB_DIFF and (diff > 0).mean() <= MAX_RGB_FRACTION, "%s: RGB (max %d, %d channels)" % (
        what, diff.max(), int((diff > 0).sum()))


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 3])
@pytest.mark.parametrize("s", [1, 2, 4, 8])
def test_centred_samples_are_the_pinhole(product_lib, scene_dir, s, k):
    """Samples (0, 0, f) for assorted f give the bytes, planes and ray counts of render_batch without lenses."""
    files, cfg = scenes.config_scene("C1", scene_dir)
    mt = _tracer(files.obj_path, 5)
    mt.GetScene().lights = _lights(scenes.LIGHT_RIG[:2])
    w, h = 75, 49
    cams = _orbit_subframes(files.camera, 2, k)
    lenses = [(0.0, 0.0, f) for f in np.geomspace(0.01, 1e6, len(cams))]
    got = mt.render_batch(cams, w, h, samples_per_axis=s, subframes=k, lenses=lenses)
    want = mt.render_batch(cams, w, h, samples_per_axis=s, subframes=k)
    assert np.array_equal(got["rgb"], want["rgb"])
    assert got["stats"]["rays"] == want["stats"]["rays"]
    if k == 1:
        got = mt.render_batch(cams, w, h, samples_per_axis=s, lenses=lenses, debug=True, taps=True)
        want = mt.render_batch(cams, w, h, samples_per_axis=s, debug=True, taps=True)
        assert got["debug"].tobytes() == want["debug"].tobytes()
        for key in TAPS:
            assert np.array_equal(got[key], want[key]), key
    mt.close()


@pytest.mark.gpu
def test_centred_c3_sample_is_the_reference_frame(product_lib, scene_dir):
    z = np.load(os.path.join(GOLDEN, "full_C3.npz"))
    files, cfg = scenes.config_scene("C3", scene_dir)
    mt = _tracer(files.obj_path, cfg["depth"])
    mt.GetScene().lights = _lights(files.lights)
    W, H = int(z["width"]), int(z["height"])
    got = mt.render_batch([files.camera], W, H, lenses=[(0.0, 0.0, 250.0)])
    assert np.array_equal(got["rgb"][0], z["rgb"]), "%d channels differ from full_C3" % int((got["rgb"][0] != z["rgb"]).sum())
    mt.close()


def _oracle_case(name, scene_dir, oracle_mod):
    """(obj path, camera, lights, w, h, depth) of the golden scenes and of C1 / C2 at small sizes."""
    if name in ("room_small", "lattice", "room_textured"):
        z, obj = _golden_case(name)
        return obj, z["camera"].tolist(), z["lights"].tolist(), int(z["width"]), int(z["height"]), int(z["depth"])
    files, cfg = scenes.config_scene(name, scene_dir, 0.1 if name == "C2" else 1.0)
    rig = files.lights if len(files.lights) >= 2 else scenes.LIGHT_RIG[:2]
    w, h = (75, 49) if name == "C1" else (100, 75)
    return files.obj_path, tuple(files.camera), [tuple(l) for l in rig], w, h, cfg["depth"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["room_small", "lattice", "room_textured", "C1", "C2"])
def test_off_centre_samples_are_the_reference_trace(product_lib, oracle_mod, rays_oracle, scene_dir, name):
    """k = 1, s = 1: four views with disc samples at two focus distances and one centred view; each view's RGB, hit ids,
    hit points and taps against the oracle's TraceRay of the restated lens rays, and the ray count against the oracle's."""
    obj, cam, rig, w, h, depth = _oracle_case(name, scene_dir, oracle_mod)
    orc = rays_oracle.from_obj(obj)
    orc.set_lights(rig)
    size = _scale(orc)
    rng = np.random.default_rng(17)
    lenses = _aperture(rng, 2, 0.03 * size, 0.2 * size) + _aperture(rng, 2, 0.05 * size, 0.6 * size) + [(0.0, 0.0, 0.3 * size)]
    cams = [cam] * len(lenses)
    mt = _tracer(obj, depth)
    mt.GetScene().lights = _lights(rig)
    got = mt.render_batch(cams, w, h, lenses=lenses, debug=True, taps=True)
    sensor = oracle_mod.Oracle.camera_sensor(cam, w, h)
    rays = 0
    for v, lens in enumerate(lenses):
        o, d = _lens_rays(cam, sensor, w, h, lens)
        cpu = orc.render_rays(o, d, depth=depth, taps=True)
        _assert_like_oracle(got, v, cpu, "%s view %d %s" % (name, v, lens))
        rays += cpu["stats"]["rays"]
    assert got["stats"]["rays"] == rays
    assert not np.array_equal(got["line_no"][0], got["line_no"][4]), "the aperture changed no primary hit"
    mt.close()


@pytest.mark.gpu
def test_off_centre_c3_samples_on_a_1080p_view(product_lib, oracle_mod, rays_oracle, scene_dir):
    """C3 at 1920x1080 with two off-centre lens samples: 3000 seeded pixels of each view against the oracle."""
    files, cfg = scenes.config_scene("C3", scene_dir)
    W, H, depth = cfg["width"], cfg["height"], cfg["depth"]
    orc = rays_oracle.from_obj(files.obj_path)
    orc.set_lights(files.lights)
    size = _scale(orc)
    lenses = [(0.02 * size, -0.01 * size, 0.25 * size), (-0.005 * size, 0.03 * size, 0.5 * size)]
    mt = _tracer(files.obj_path, depth)
    mt.GetScene().lights = _lights(files.lights)
    got = mt.render_batch([files.camera] * 2, W, H, lenses=lenses, debug=True, taps=True)
    sensor = oracle_mod.Oracle.camera_sensor(files.camera, W, H)
    rng = np.random.default_rng(5)
    ys, xs = rng.integers(0, H, 3000), rng.integers(0, W, 3000)
    for v, lens in enumerate(lenses):
        o, d = _lens_rays(files.camera, sensor, W, H, lens)
        cpu = orc.render_rays(o[ys, xs], d[ys, xs], depth=depth, taps=True)
        picked = {k: got[k][v][ys, xs][None] for k in ("rgb", "line_no", "points") + TAPS}
        _assert_like_oracle(picked, 0, cpu, "C3 view %d" % v)
    mt.close()


@pytest.mark.gpu
@pytest.mark.parametrize("s", [1, 2, 4, 8])
@pytest.mark.parametrize("k", [3, 5, 8])
def test_depth_of_field_is_the_mean_of_the_lens_subframes(product_lib, scene_dir, k, s):
    """Two C3 output views (orbit cameras) of k disc samples each: the accumulated output equals _accum_mean of the
    k = 1 lens sub-frames rendered at s*W x s*H."""
    files, cfg = scenes.config_scene("C3", scene_dir)
    mt = _tracer(files.obj_path, cfg["depth"])
    mt.GetScene().lights = _lights(files.lights)
    w, h = 160, 90
    cams = [_yawed(files.camera, 2.0 * v) for v in range(2) for _ in range(k)]
    lenses = _aperture(np.random.default_rng(100 + k), 2 * k, 6.0, 150.0)
    got = mt.render_batch(cams, w, h, samples_per_axis=s, subframes=k, lenses=lenses)
    hi = mt.render_batch(cams, s * w, s * h, lenses=lenses)
    assert np.array_equal(got["rgb"], _accum_mean(hi["rgb"], k, s))
    assert got["stats"]["rays"] == hi["stats"]["rays"]
    assert not np.array_equal(got["rgb"], mt.render_batch(cams, w, h, samples_per_axis=s, subframes=k)["rgb"])
    mt.close()


@pytest.mark.gpu
def test_motion_blur_soft_shadows_and_depth_of_field_in_one_call(product_lib, scene_dir):
    """A camera path, jittered lights and lens samples in one accumulated call, against the formula over the sub-frames."""
    files, cfg = scenes.config_scene("C3", scene_dir)
    mt = _tracer(files.obj_path, cfg["depth"])
    k, s, w, h = 6, 2, 120, 68
    cams = _orbit_subframes(files.camera, 2, k)
    light_sets = _jittered_lights(files.lights, k, 25.0, seed=3) + _jittered_lights(files.lights, k, 25.0, seed=4)
    lenses = np.array(_aperture(np.random.default_rng(9), 2 * k, 5.0, 120.0))
    got = mt.render_batch(cams, w, h, lights=light_sets, samples_per_axis=s, subframes=k, lenses=lenses)
    hi = mt.render_batch(cams, s * w, s * h, lights=light_sets, lenses=lenses)
    assert np.array_equal(got["rgb"], _accum_mean(hi["rgb"], k, s))
    mt.close()


@pytest.mark.gpu
@pytest.mark.parametrize("s,k", [(1, 1), (2, 1), (1, 3), (2, 3)])
def test_device_form_equals_the_host_form(product_lib, scene_dir, s, k):
    import torch
    files, cfg = scenes.config_scene("C1", scene_dir)
    mt = _tracer(files.obj_path, 5)
    mt.GetScene().lights = _lights(scenes.LIGHT_RIG[:2])
    w, h = 75, 49
    cams = _orbit_subframes(files.camera, 3, k)
    lenses = _aperture(np.random.default_rng(21), len(cams), 8.0, 90.0)
    planes = dict(debug=True, taps=True) if k == 1 else {}
    host = mt.render_batch(cams, w, h, samples_per_axis=s, subframes=k, lenses=lenses, **planes)
    dev = mt.render_batch(cams, w, h, samples_per_axis=s, subframes=k, lenses=lenses, device=True, **planes)
    torch.cuda.current_stream().synchronize()
    assert np.array_equal(dev["rgb"].cpu().numpy(), host["rgb"])
    if k == 1:
        assert dev["debug"].cpu().numpy().tobytes() == host["debug"].tobytes()
        for key in TAPS:
            assert np.array_equal(dev[key].cpu().numpy(), host[key]), key
    mt.close()


@pytest.mark.gpu
def test_lens_batches_split_over_devices(product_lib, scene_dir):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    files, cfg = scenes.config_scene("C1", scene_dir)
    n = min(torch.cuda.device_count(), 8)
    one = _tracer(files.obj_path, 5)
    many = _tracer(files.obj_path, 5, devices=list(range(n)))
    for n_out, k, s in ((n + 3, 3, 1), (n - 1, 4, 2), (2 * n, 1, 1)):
        cams = _orbit_subframes(files.camera, n_out, k)
        lenses = _aperture(np.random.default_rng(n_out), len(cams), 8.0, 90.0)
        a = one.render_batch(cams, 75, 49, samples_per_axis=s, subframes=k, lenses=lenses)
        b = many.render_batch(cams, 75, 49, samples_per_axis=s, subframes=k, lenses=lenses)
        assert np.array_equal(b["rgb"], a["rgb"]), (n_out, k, s)
        assert b["stats"]["rays"] == a["stats"]["rays"]
        d = many.render_batch(cams, 75, 49, samples_per_axis=s, subframes=k, lenses=lenses, device=True)
        torch.cuda.synchronize()
        assert np.array_equal(d["rgb"].cpu().numpy(), a["rgb"]), (n_out, k, s)


@pytest.mark.gpu
def test_c_abi_argument_errors_queue_nothing(product_lib, scene_dir):
    """Every refused call returns MTB_ERR_ARG with a message and launches nothing, in both forms."""
    import torch
    from mythtracer_b200 import api
    files, cfg = scenes.config_scene("C1", scene_dir)
    mt = _tracer(files.obj_path, 3)
    mt.GetScene().lights = _lights(scenes.LIGHT_RIG[:2])
    mt.push_lights()
    n, w, h = 4, 40, 24
    cams = np.zeros(n, api.CAMERA_DTYPE)
    for i in range(n):
        cams[i] = api.Camera.from_tuple(_yawed(files.camera, 2.0 * i)).as_array()
    rgb = np.zeros((n, h, w, 3), np.uint8)
    d_rgb = torch.zeros((n, h, w, 3), dtype=torch.uint8, device="cuda:0")
    vp = ctypes.c_void_p

    def call(lenses, cam_arr=cams, device=False, n_out=2, k=2, w=w, h=h):
        lp = None if lenses is None else np.ascontiguousarray(lenses, np.float64).ctypes.data_as(vp)
        if device:
            rc = product_lib.mtb_render_batch_lens_device(mt._ctx, cam_arr.ctypes.data_as(vp), lp, n_out, k, None, 0, w, h, 1, 3,
                                                          vp(d_rgb.data_ptr()), None, None, None, None)
        else:
            rc = product_lib.mtb_render_batch_lens(mt._ctx, cam_arr.ctypes.data_as(vp), lp, n_out, k, None, 0, w, h, 1, 3,
                                                   rgb.ctypes.data_as(vp), None, None, None)
        return rc, product_lib.mtb_last_error(mt._ctx).decode()

    good = np.array([(0.5, -0.25, 30.0)] * n)
    # the corner rule: a degenerate sensor (aov 0), and aov 180 on a portrait grid, whose corner rays leave the half-space
    # in front of the focal plane
    flat, wide = cams.copy(), cams.copy()
    flat[2]["aov"] = 0.0
    wide[0]["aov"] = 180.0
    nan, inf = float("nan"), float("inf")
    cases = [(None, {}, "lenses is NULL")]
    for i, row in enumerate([(nan, 0.0, 1.0), (0.0, inf, 1.0), (0.0, 0.0, nan), (0.0, 0.0, -inf), (1.0, 0.0, 0.0), (0.0, 0.0, -1.0)]):
        bad = good.copy()
        bad[i % n] = row
        cases.append((bad, {}, "lenses[%d]" % (i % n)))
    cases.append((good, dict(cam_arr=flat), "lenses[2]: the sub-frame's corner rays"))
    cases.append((good[:1], dict(n_out=1, k=1, cam_arr=wide[:1], w=h, h=w), "lenses[0]: the sub-frame's corner rays"))
    cases.append((good, dict(n_out=0), "n_out"))
    for device in (False, True):
        for lenses, kw, words in cases:
            before = mt.launch_count()
            rc, msg = call(lenses, device=device, **kw)
            assert rc == MTB_ERR_ARG and words in msg, (device, lenses, kw, rc, msg)
            assert mt.launch_count() == before
        assert call(good, device=device)[0] == MTB_OK
    torch.cuda.synchronize()
    assert np.array_equal(d_rgb[:2].cpu().numpy(), rgb[:2])


@pytest.mark.gpu
def test_pinhole_renders_are_unchanged_after_a_lens_batch(product_lib, scene_dir):
    files, cfg = scenes.config_scene("C1", scene_dir)
    mt = _tracer(files.obj_path, 5)
    mt.GetScene().lights = _lights(scenes.LIGHT_RIG[:2])
    cams = _orbit_subframes(files.camera, 3, 2)
    before_batch = mt.render_batch(cams, 64, 48, subframes=2)["rgb"].copy()
    before_chunk = mt.render_chunk(files.camera, 96, 64, 0, 0, 96, 64)["rgb"].copy()
    mt.render_batch(cams, 128, 96, samples_per_axis=2, subframes=2, lenses=_aperture(np.random.default_rng(1), 6, 10.0, 80.0))
    mt.render_batch(cams[:4], 64, 48, lenses=[(3.0, 1.0, 50.0)] * 4, debug=True)
    assert np.array_equal(mt.render_batch(cams, 64, 48, subframes=2)["rgb"], before_batch)
    assert np.array_equal(mt.render_chunk(files.camera, 96, 64, 0, 0, 96, 64)["rgb"], before_chunk)


@pytest.mark.gpu
@pytest.mark.parametrize("s,k", [(1, 4), (2, 3)])
def test_cpp_shim_lens_batches(product_lib, scene_dir, tmp_path, s, k):
    """RayTraceBatch with lens samples, called from C++ (tests/cpp/lens_check.cc): the output equals render_batch(...,
    lenses=...) of the same sub-frames."""
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    exe = str(tmp_path / "lens_check")
    lib_dir = os.path.join(ROOT, "mythtracer_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                           os.path.join(HERE, "cpp", "lens_check.cc"), "-L", lib_dir, "-lmythtracer_b200", "-Wl,-rpath," + lib_dir, "-o", exe])
    files, cfg = scenes.config_scene("C2", scene_dir, 0.1)
    W, H = 60, 36
    prefix = str(tmp_path / "out")
    res = subprocess.run([exe, files.obj_path, prefix, str(W), str(H), str(s), str(k)], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    assert "lens ok" in res.stdout
    mt = _tracer(files.obj_path, 3)
    mt.GetScene().lights = _lights([(231.82174, 81.69966, 27.78259, 0.3, 0.3, 0.3, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0),
                                    (200.0, 95.0, 160.0, 0.0, 0.0, 0.0, 0.3, 0.3, 0.3, 0.3, 0.3, 0.3)])
    cams = [(301.37, 57.21, 161.13, 4.0, 243.0 + 3.0 * v, 0.0, 110.0) for v in range(2) for j in range(k)]
    lenses = [(4.0 * math.cos(2.0 * math.pi * j / k), 4.0 * math.sin(2.0 * math.pi * j / k), 150.0) for v in range(2) for j in range(k)]
    want = mt.render_batch(cams, W, H, samples_per_axis=s, subframes=k, lenses=lenses)["rgb"]
    got = np.fromfile(prefix + ".rgb", np.uint8).reshape(2, H, W, 3)
    assert np.array_equal(got, want)
