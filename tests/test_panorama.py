"""Panorama batches (mtb_render_batch_pano / render_batch(..., panorama=(h_fov, v_fov), eye_offsets=...)):
equirectangular and omni-directional stereo views.  The panorama rays are restated here in plain Python from the
formula of include/mythtracer_b200.h (math.sin / math.cos per table entry, the C library's functions like the
library's), pinned to mtb_panorama_rays bit for bit, and traced with the reference's TraceRay by mto_render_rays
(tests/cpp/oracle_rays.cc, through test_lens.py's rays_oracle fixture)."""
import ctypes
import math
import os
import shutil
import subprocess

import numpy as np
import pytest

from tests import scenes
from tests.test_accumulate import _accum_mean, _jittered_lights, _lights, _orbit_subframes, _tracer, _yawed
from tests.test_lens import TAPS, _assert_like_oracle, _oracle_case, _scale, rays_oracle  # noqa: F401 (rays_oracle: a fixture)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
MTB_OK, MTB_ERR_ARG = 0, -1
FULL = (360.0, 180.0)

# (x, y, z, pitch, yaw, roll, aov): level, pitched and rolled, negative yaw, steep
CAMERAS = [(0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 60.0), (10.0, 5.0, -3.0, 12.0, 40.0, 3.0, 80.0), (-2.5, 1.0, 7.0, -30.0, -135.0, 20.0, 60.0),
           (1.0, 2.0, 3.0, 85.0, -270.0, -45.0, 45.0)]


# ---------------------------------------------------------------------------------------------- the restatement


def _rot(axis, deg):
    a = (deg * math.pi) / 180.0
    c, s = math.cos(a), math.sin(a)
    if axis == "x":
        return [[1.0, 0.0, 0.0, 0.0], [0.0, c, -s, 0.0], [0.0, s, c, 0.0], [0.0, 0.0, 0.0, 1.0]]
    if axis == "y":
        return [[c, 0.0, s, 0.0], [0.0, 1.0, 0.0, 0.0], [-s, 0.0, c, 0.0], [0.0, 0.0, 0.0, 1.0]]
    return [[c, -s, 0.0, 0.0], [s, c, 0.0, 0.0], [0.0, 0.0, 1.0, 0.0], [0.0, 0.0, 0.0, 1.0]]


def _mul(a, b):
    return [[a[j][0] * b[0][i] + a[j][1] * b[1][i] + a[j][2] * b[2][i] + a[j][3] * b[3][i] for i in range(4)] for j in range(4)]


def _apply(m, v):
    # (the reference adds m[0][3] to every row, math3d.h:210-216)
    return tuple(m[r][0] * v[0] + m[r][1] * v[1] + m[r][2] * v[2] + m[0][3] for r in range(3))


def _basis(cam):
    """(F, R, U) of a camera: aim = Mul(Mul(RotY(yaw), RotX(pitch)), RotZ(roll)) applied to (0, 0, 1), (-1, 0, 0), (0, 1, 0)."""
    aim = _mul(_mul(_rot("y", cam[4]), _rot("x", cam[3])), _rot("z", cam[5]))
    return _apply(aim, (0.0, 0.0, 1.0)), _apply(aim, (-1.0, 0.0, 0.0)), _apply(aim, (0.0, 1.0, 0.0))


def _tables(w, h, h_fov, v_fov):
    """(cl, sl) per column and (cp, sp) per row, float64 arrays, one math.cos / math.sin call per entry."""
    lon = [(float(2 * x + 1 - w) / float(2 * w)) * (h_fov * (math.pi / 180.0)) for x in range(w)]
    lat = [(float(h - 2 * y - 1) / float(2 * h)) * (v_fov * (math.pi / 180.0)) for y in range(h)]
    arr = lambda f, angles: np.array([f(a) for a in angles], np.float64)  # noqa: E731
    return arr(math.cos, lon), arr(math.sin, lon), arr(math.cos, lat), arr(math.sin, lat)


def _pano_rays(cam, w, h, h_fov, v_fov, e=0.0):
    """(origins, dirs), each (h, w, 3): the formula of mtb_render_batch_pano, FP64 in its order (numpy's + * / sqrt are
    IEEE operations; only the trigonometry comes from math)."""
    F, R, U = _basis(cam)
    cl, sl, cp, sp = _tables(w, h, h_fov, v_fov)
    cl, sl, cp, sp = cl[None, :], sl[None, :], cp[:, None], sp[:, None]
    q = [(F[a] * cl + R[a] * sl) * cp + U[a] * sp for a in range(3)]
    n = np.sqrt((q[0] * q[0] + q[1] * q[1]) + q[2] * q[2])
    dirs = np.stack([q[a] / n for a in range(3)], axis=-1)
    O = [float(x) for x in cam[0:3]]
    if e == 0.0:
        origins = np.broadcast_to(np.array(O), (h, w, 3)).copy()
    else:
        origins = np.stack([np.broadcast_to(O[a] + (R[a] * cl - F[a] * sl) * e, (h, w)) for a in range(3)], axis=-1)
    return origins, dirs


# ---------------------------------------------------------------------------------------------- CPU


@pytest.mark.parametrize("e", [0.0, 0.03, -0.03])
@pytest.mark.parametrize("fov", [FULL, (90.0, 45.0), (1.0, 1.0)])
@pytest.mark.parametrize("w,h", [(17, 9), (16, 8), (1, 1)])
def test_panorama_rays_are_the_restatement(product_lib, w, h, fov, e):
    from mythtracer_b200 import Camera, panorama_rays
    for cam in CAMERAS:
        want_o, want_d = _pano_rays(cam, w, h, fov[0], fov[1], e)
        o, d = panorama_rays(cam, w, h, fov[0], fov[1], eye_offset=e)
        assert o.shape == d.shape == (h, w, 3) and o.dtype == d.dtype == np.float64
        assert np.array_equal(d, want_d), (cam, int((d != want_d).sum()))
        assert np.array_equal(o, want_o), (cam, int((o != want_o).sum()))
        # the C ABI with origins == NULL writes the same directions
        d2 = np.zeros((h, w, 3))
        c = Camera.from_tuple(cam).as_array()
        assert product_lib.mtb_panorama_rays(c.ctypes.data, w, h, fov[0], fov[1], e, None, d2.ctypes.data) == MTB_OK
        assert np.array_equal(d2, want_d)


def test_panorama_geometry_of_the_restatement():
    """A full panorama's directions are unit vectors whose longitude and latitude follow the grid, the seam columns
    meet behind the camera, and an eye offset moves each column's origin along its tangent, perpendicular to it."""
    cam = CAMERAS[2]
    w, h, e = 36, 18, 0.5
    F, R, U = (np.array(v) for v in _basis(cam))
    o, d = _pano_rays(cam, w, h, 360.0, 180.0, e)
    np.testing.assert_allclose(np.linalg.norm(d, axis=-1), 1.0, atol=1e-15)
    lat = np.arcsin(np.clip(d @ U, -1, 1))
    np.testing.assert_allclose(lat[:, 0], (h - 2 * np.arange(h) - 1) / (2 * h) * np.pi, atol=1e-12)
    lon = np.arctan2(d @ R, d @ F)
    np.testing.assert_allclose(lon[h // 2], (2 * np.arange(w) + 1 - w) / (2 * w) * 2 * np.pi, atol=1e-12)
    # the left and right edge columns are one column apart across the seam (-180 degrees = +180 degrees)
    np.testing.assert_allclose(lon[h // 2, 0] + 2 * np.pi - lon[h // 2, -1], 2 * np.pi / w, atol=1e-12)
    shift = o - np.array(cam[:3])
    np.testing.assert_allclose(np.linalg.norm(shift, axis=-1), abs(e), atol=1e-12)
    assert np.abs((shift * d).sum(-1)[h // 2]).max() < 1e-12  # on the horizon the offset is perpendicular to the ray
    assert np.abs(shift @ U).max() < 1e-12


@pytest.mark.parametrize("cam", CAMERAS)
def test_panorama_basis_signs_match_the_pinhole_sensor(product_lib, cam):
    """R points along the pinhole sensor's delta_pixel, U against its delta_scanline, F at the sensor's centre."""
    from mythtracer_b200 import Camera
    F, R, U = (np.array(v) for v in _basis(cam))
    c = list(cam)
    c[6] = 60.0
    w, h = 64, 48
    S, Dy, Dx = Camera.from_tuple(c).GetSensor(w, h)
    assert np.dot(R, Dx) > 0 and np.dot(U, Dy) < 0
    assert np.dot(F, S + Dy * (h / 2) + Dx * (w / 2)) > 0
    # and the basis is the sensor's frame: F along the centre direction, R and U along the sensor's axes
    centre = S + Dy * (h / 2) + Dx * (w / 2)
    np.testing.assert_allclose(F, centre / np.linalg.norm(centre), atol=1e-12)
    np.testing.assert_allclose(R, Dx / np.linalg.norm(Dx), atol=1e-12)
    np.testing.assert_allclose(U, -Dy / np.linalg.norm(Dy), atol=1e-12)


def test_panorama_rays_arguments_are_checked(product_lib):
    from mythtracer_b200 import Camera, MythTracerError, panorama_rays
    cam = CAMERAS[1]
    nan, inf = float("nan"), float("inf")
    for args, kw, words in (((0, 8, 360.0, 180.0), {}, "w must be"), ((8, 65537, 360.0, 180.0), {}, "h must be"),
                            ((8, 8, 0.0, 180.0), {}, "h_fov"), ((8, 8, 360.5, 180.0), {}, "h_fov"), ((8, 8, nan, 180.0), {}, "h_fov"),
                            ((8, 8, 360.0, 0.0), {}, "v_fov"), ((8, 8, 360.0, 180.5), {}, "v_fov"), ((8, 8, 360.0, -inf), {}, "v_fov"),
                            ((8, 8, "360", 180.0), {}, "h_fov"), ((8, 8, 360.0, 180.0), dict(eye_offset=inf), "eye_offset"),
                            ((8, 8, 360.0, 180.0), dict(eye_offset=nan), "eye_offset")):
        with pytest.raises(MythTracerError, match=words):
            panorama_rays(cam, *args, **kw)
    c = Camera.from_tuple(cam).as_array()
    d = np.zeros((4, 4, 3))
    for w, h, hf, vf, e in ((0, 4, 360.0, 180.0, 0.0), (4, 4, 0.0, 180.0, 0.0), (4, 4, 360.0, 181.0, 0.0), (4, 4, 360.0, 180.0, nan)):
        assert product_lib.mtb_panorama_rays(c.ctypes.data, w, h, hf, vf, e, None, d.ctypes.data) == MTB_ERR_ARG
    assert product_lib.mtb_panorama_rays(c.ctypes.data, 4, 4, 360.0, 180.0, 0.0, None, None) == MTB_ERR_ARG
    assert product_lib.mtb_panorama_rays(None, 4, 4, 360.0, 180.0, 0.0, None, d.ctypes.data) == MTB_ERR_ARG


def test_panoramas_have_no_cpu_fallback(product_lib):
    from mythtracer_b200 import MythTracer, MythTracerError
    files, cfg = scenes.config_scene("C1", "/tmp/mtb_scenes")
    mt = MythTracer(host_only=True)
    assert mt.LoadObj(files.obj_path)
    for device in (False, True):
        with pytest.raises(MythTracerError, match="no CPU fallback"):
            mt.render_batch([files.camera] * 2, 16, 8, panorama=FULL, eye_offsets=[-0.1, 0.1], device=device)


def test_panorama_arguments_are_checked_in_python(product_lib):
    from mythtracer_b200 import MythTracer, MythTracerError
    files, cfg = scenes.config_scene("C1", "/tmp/mtb_scenes")
    mt = MythTracer(host_only=True)
    assert mt.LoadObj(files.obj_path)
    cams = [files.camera] * 4
    nan, inf = float("nan"), float("inf")
    cases = [(dict(panorama=360.0), "pair"), (dict(panorama=(360.0,)), "pair"), (dict(panorama="ab"), "pair"),
             (dict(panorama=(0.0, 180.0)), "h_fov"), (dict(panorama=(400.0, 180.0)), "h_fov"), (dict(panorama=(nan, 180.0)), "h_fov"),
             (dict(panorama=(-1.0, 180.0)), "h_fov"), (dict(panorama=(True, 180.0)), "h_fov"), (dict(panorama=(360.0, 0.0)), "v_fov"),
             (dict(panorama=(360.0, 180.1)), "v_fov"), (dict(panorama=(360.0, inf)), "v_fov"),
             (dict(panorama=FULL, eye_offsets=[0.1] * 3), "shape"), (dict(panorama=FULL, eye_offsets=[[0.1]] * 4), "shape"),
             (dict(panorama=FULL, eye_offsets="abcd"), "sequence"), (dict(panorama=FULL, eye_offsets=["a"] * 4), "numbers"),
             (dict(panorama=FULL, eye_offsets=[0.1, nan, 0.0, 0.0]), "finite"), (dict(panorama=FULL, eye_offsets=[0.0, 0.0, 0.0, -inf]), "finite"),
             (dict(eye_offsets=[0.1] * 4), "need a panorama"), (dict(panorama=FULL, lenses=[(0.0, 0.0, 1.0)] * 4), "cannot be combined")]
    for kw, words in cases:
        for device in (False, True):
            with pytest.raises(MythTracerError, match=words):
                mt.render_batch(cams, 16, 8, subframes=2, device=device, **kw)
    # the other argument rules hold with a panorama too
    with pytest.raises(MythTracerError, match="debug and taps"):
        mt.render_batch(cams, 16, 8, panorama=FULL, subframes=2, debug=True)
    with pytest.raises(MythTracerError, match="samples_per_axis"):
        mt.render_batch(cams, 16, 8, panorama=FULL, samples_per_axis=3)


def _c_call(lib, ctx, cams, device, eye=None, n_out=2, k=2, h_fov=360.0, v_fov=180.0, w=16, h=8, rgb=None, d_rgb=None, planes=(None, None)):
    """mtb_render_batch_pano(_device) with the given arguments: (return code, mtb_last_error)."""
    vp = ctypes.c_void_p
    ep = None if eye is None else np.ascontiguousarray(eye, np.float64).ctypes.data_as(vp)
    cp = cams.ctypes.data_as(vp)
    if device:
        rc = lib.mtb_render_batch_pano_device(ctx, cp, ep, n_out, k, h_fov, v_fov, None, 0, w, h, 1, 3, d_rgb, planes[0], planes[1], None, None)
    else:
        rc = lib.mtb_render_batch_pano(ctx, cp, ep, n_out, k, h_fov, v_fov, None, 0, w, h, 1, 3, rgb, planes[0], planes[1], None)
    return rc, lib.mtb_last_error(ctx).decode()


def _refusal_cases(n):
    nan, inf = float("nan"), float("inf")
    cases = []
    for hf in (0.0, -5.0, 360.0000001, nan, inf):
        cases.append((dict(h_fov=hf), "h_fov must be finite and in (0, 360]"))
    for vf in (0.0, 180.0000001, nan, -inf):
        cases.append((dict(v_fov=vf), "v_fov must be finite and in (0, 180]"))
    for i, bad in enumerate((nan, inf, -inf)):
        eye = np.zeros(n)
        eye[(i + 1) % n] = bad
        cases.append((dict(eye=eye), "eye_offsets[%d] must be finite" % ((i + 1) % n)))
    return cases


def test_c_abi_panorama_refusals_on_a_host_only_context(product_lib):
    """The panorama rules are checked before anything else, so a host-only context reports them too."""
    from mythtracer_b200 import MythTracer, api
    mt = MythTracer(host_only=True)
    cams = np.zeros(4, api.CAMERA_DTYPE)
    for i in range(4):
        cams[i] = api.Camera.from_tuple(CAMERAS[i]).as_array()
    rgb = np.zeros((2, 8, 16, 3), np.uint8)
    for device in (False, True):
        for kw, words in _refusal_cases(4):
            rc, msg = _c_call(product_lib, mt._ctx, cams, device, rgb=rgb.ctypes.data, **kw)
            assert rc == MTB_ERR_ARG and words in msg, (device, kw, rc, msg)
        rc, msg = _c_call(product_lib, mt._ctx, cams, device, rgb=rgb.ctypes.data, eye=np.zeros(4))
        assert rc != MTB_OK and "no CPU fallback" in msg, (rc, msg)
    assert product_lib.mtb_render_batch_pano(None, cams.ctypes.data, None, 2, 2, 360.0, 180.0, None, 0, 16, 8, 1, 3, rgb.ctypes.data, None,
                                             None, None) == MTB_ERR_ARG


# ---------------------------------------------------------------------------------------------- GPU


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["room_small", "lattice", "room_textured", "C1", "C2"])
def test_full_panoramas_are_the_reference_trace(product_lib, oracle_mod, rays_oracle, scene_dir, name):  # noqa: F811
    """k = 1, s = 1: a full panorama and an ODS pair (e = -/+0.032 * scene scale) from each scene's camera; each view's
    RGB, hit ids, hit points and taps against the oracle's TraceRay of mtb_panorama_rays' rays, and the ray count."""
    from mythtracer_b200 import panorama_rays
    obj, cam, rig, w, h, depth = _oracle_case(name, scene_dir, oracle_mod)
    w, h = 2 * w, w  # (2:1, the equirectangular aspect)
    orc = rays_oracle.from_obj(obj)
    orc.set_lights(rig)
    eyes = [0.0, -0.032 * _scale(orc), 0.032 * _scale(orc)]
    mt = _tracer(obj, depth)
    mt.GetScene().lights = _lights(rig)
    got = mt.render_batch([cam] * 3, w, h, panorama=FULL, eye_offsets=eyes, debug=True, taps=True)
    rays = 0
    for v, e in enumerate(eyes):
        o, d = panorama_rays(cam, w, h, *FULL, eye_offset=e)
        assert np.array_equal(d, _pano_rays(cam, w, h, *FULL, e)[1])
        cpu = orc.render_rays(o, d, depth=depth, taps=True)
        _assert_like_oracle(got, v, cpu, "%s eye %g" % (name, e))
        rays += cpu["stats"]["rays"]
    assert got["stats"]["rays"] == rays
    assert not np.array_equal(got["line_no"][1], got["line_no"][2]), "the two eyes saw the same hits"
    mt.close()


@pytest.mark.gpu
def test_c3_panorama_at_4096x2048(product_lib, oracle_mod, rays_oracle, scene_dir):  # noqa: F811
    """A full 4096x2048 C3 panorama from the C3 origin: 3000 seeded pixels against the oracle."""
    from mythtracer_b200 import panorama_rays
    files, cfg = scenes.config_scene("C3", scene_dir)
    W, H, depth = 4096, 2048, cfg["depth"]
    orc = rays_oracle.from_obj(files.obj_path)
    orc.set_lights(files.lights)
    mt = _tracer(files.obj_path, depth)
    mt.GetScene().lights = _lights(files.lights)
    got = mt.render_batch([files.camera], W, H, panorama=FULL, debug=True, taps=True)
    o, d = panorama_rays(files.camera, W, H, *FULL)
    rng = np.random.default_rng(11)
    ys, xs = rng.integers(0, H, 3000), rng.integers(0, W, 3000)
    cpu = orc.render_rays(o[ys, xs], d[ys, xs], depth=depth, taps=True)
    picked = {k: got[k][0][ys, xs][None] for k in ("rgb", "line_no", "points") + TAPS}
    _assert_like_oracle(picked, 0, cpu, "C3 panorama")
    assert (got["line_no"][0] >= 0).mean() > 0.5, "the panorama hit little of the scene"
    mt.close()


@pytest.mark.gpu
def test_exact_zero_direction_components_take_the_literal_path(product_lib, oracle_mod, rays_oracle, scene_dir):  # noqa: F811
    """An axis-aligned camera with an odd grid: the centre column and the horizon row have exact zero direction
    components.  The counting build shows literal traversals, and every output equals the oracle's."""
    from mythtracer_b200 import MTB_FLAG_COUNT_WORK, panorama_rays
    files, cfg = scenes.config_scene("C1", scene_dir)
    cam = tuple(files.camera[:3]) + (0.0, 0.0, 0.0, 60.0)
    w, h = 75, 49
    o, d = panorama_rays(cam, w, h, 120.0, 60.0)
    assert (d[h // 2, :, 1] == 0.0).all() and (d[:, w // 2, 0] == 0.0).all()
    assert np.array_equal(d[h // 2, w // 2], [0.0, 0.0, 1.0])
    orc = rays_oracle.from_obj(files.obj_path)
    rig = scenes.LIGHT_RIG[:2]
    orc.set_lights(rig)
    cpu = orc.render_rays(o, d, depth=cfg["depth"], taps=True)
    for flags in (0, MTB_FLAG_COUNT_WORK):
        mt = _tracer(files.obj_path, cfg["depth"], flags=flags)
        mt.GetScene().lights = _lights(rig)
        got = mt.render_batch([cam], w, h, panorama=(120.0, 60.0), debug=True, taps=True)
        _assert_like_oracle(got, 0, cpu, "axis-aligned panorama, flags %d" % flags)
        assert got["stats"]["rays"] == cpu["stats"]["rays"]
        if flags:
            assert got["stats"]["n_literal"] > 0
        mt.close()


@pytest.mark.gpu
@pytest.mark.parametrize("s", [2, 4, 8])
def test_supersampled_panorama_is_the_mean_of_the_fine_grid(product_lib, scene_dir, s):
    files, cfg = scenes.config_scene("C3", scene_dir)
    mt = _tracer(files.obj_path, cfg["depth"])
    mt.GetScene().lights = _lights(files.lights)
    w, h = 96, 48
    cams = [files.camera, _yawed(files.camera, 37.0)]
    eyes = [-0.5, 0.5]
    got = mt.render_batch(cams, w, h, samples_per_axis=s, panorama=FULL, eye_offsets=eyes)
    hi = mt.render_batch(cams, s * w, s * h, panorama=FULL, eye_offsets=eyes)
    assert np.array_equal(got["rgb"], _accum_mean(hi["rgb"], 1, s))
    assert got["stats"]["rays"] == hi["stats"]["rays"]
    mt.close()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [3, 5])
@pytest.mark.parametrize("s", [1, 2])
def test_accumulated_panorama_is_the_mean_of_its_subframes(product_lib, scene_dir, k, s):
    files, cfg = scenes.config_scene("C3", scene_dir)
    mt = _tracer(files.obj_path, cfg["depth"])
    mt.GetScene().lights = _lights(files.lights)
    w, h = 80, 40
    cams = _orbit_subframes(files.camera, 2, k)
    eyes = list(np.random.default_rng(k).uniform(-1.0, 1.0, len(cams)))
    got = mt.render_batch(cams, w, h, samples_per_axis=s, subframes=k, panorama=(300.0, 150.0), eye_offsets=eyes)
    hi = mt.render_batch(cams, s * w, s * h, panorama=(300.0, 150.0), eye_offsets=eyes)
    assert np.array_equal(got["rgb"], _accum_mean(hi["rgb"], k, s))
    assert got["stats"]["rays"] == hi["stats"]["rays"]
    mt.close()


@pytest.mark.gpu
def test_camera_path_jittered_lights_and_eye_offsets_in_one_call(product_lib, scene_dir):
    files, cfg = scenes.config_scene("C3", scene_dir)
    mt = _tracer(files.obj_path, cfg["depth"])
    k, s, w, h = 4, 2, 64, 32
    cams = _orbit_subframes(files.camera, 2, k)
    light_sets = _jittered_lights(files.lights, k, 25.0, seed=5) + _jittered_lights(files.lights, k, 25.0, seed=6)
    eyes = np.array([-0.8] * k + [0.8] * k)
    got = mt.render_batch(cams, w, h, lights=light_sets, samples_per_axis=s, subframes=k, panorama=FULL, eye_offsets=eyes)
    hi = mt.render_batch(cams, s * w, s * h, lights=light_sets, panorama=FULL, eye_offsets=eyes)
    assert np.array_equal(got["rgb"], _accum_mean(hi["rgb"], k, s))
    mt.close()


@pytest.mark.gpu
@pytest.mark.parametrize("s,k", [(1, 1), (2, 1), (1, 3), (2, 3)])
def test_device_form_equals_the_host_form(product_lib, scene_dir, s, k):
    import torch
    files, cfg = scenes.config_scene("C1", scene_dir)
    mt = _tracer(files.obj_path, 5)
    mt.GetScene().lights = _lights(scenes.LIGHT_RIG[:2])
    w, h = 64, 32
    cams = _orbit_subframes(files.camera, 3, k)
    eyes = np.random.default_rng(4).uniform(-2.0, 2.0, len(cams))
    planes = dict(debug=True, taps=True) if k == 1 else {}
    host = mt.render_batch(cams, w, h, samples_per_axis=s, subframes=k, panorama=FULL, eye_offsets=eyes, **planes)
    dev = mt.render_batch(cams, w, h, samples_per_axis=s, subframes=k, panorama=FULL, eye_offsets=eyes, device=True, **planes)
    torch.cuda.current_stream().synchronize()
    assert np.array_equal(dev["rgb"].cpu().numpy(), host["rgb"])
    if k == 1:
        assert dev["debug"].cpu().numpy().tobytes() == host["debug"].tobytes()
        for key in TAPS:
            assert np.array_equal(dev[key].cpu().numpy(), host[key]), key
    mt.close()


@pytest.mark.gpu
def test_panorama_batches_split_over_devices(product_lib, scene_dir):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    files, cfg = scenes.config_scene("C1", scene_dir)
    n = min(torch.cuda.device_count(), 8)
    one = _tracer(files.obj_path, 5)
    many = _tracer(files.obj_path, 5, devices=list(range(n)))
    for n_out, k, s in ((n + 3, 3, 1), (n - 1, 4, 2), (2 * n, 1, 1)):
        cams = _orbit_subframes(files.camera, n_out, k)
        eyes = np.random.default_rng(n_out).uniform(-2.0, 2.0, len(cams))
        a = one.render_batch(cams, 64, 32, samples_per_axis=s, subframes=k, panorama=FULL, eye_offsets=eyes)
        b = many.render_batch(cams, 64, 32, samples_per_axis=s, subframes=k, panorama=FULL, eye_offsets=eyes)
        assert np.array_equal(b["rgb"], a["rgb"]), (n_out, k, s)
        assert b["stats"]["rays"] == a["stats"]["rays"]
        d = many.render_batch(cams, 64, 32, samples_per_axis=s, subframes=k, panorama=FULL, eye_offsets=eyes, device=True)
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
    n, w, h = 4, 16, 8
    cams = np.zeros(n, api.CAMERA_DTYPE)
    for i in range(n):
        cams[i] = api.Camera.from_tuple(_yawed(files.camera, 2.0 * i)).as_array()
    rgb = np.zeros((n, h, w, 3), np.uint8)
    d_rgb = torch.zeros((n, h, w, 3), dtype=torch.uint8, device="cuda:0")
    dbg = np.zeros((n, h, w), api.DEBUG_DTYPE)
    for device in (False, True):
        cases = _refusal_cases(n) + [(dict(n_out=0), "n_out"), (dict(n_out=40000), "n_out"), (dict(k=0), "subframes must be >= 1")]
        if not device:
            cases.append((dict(planes=(dbg.ctypes.data, None)), "no debug or tap planes"))
        for kw, words in cases:
            before = mt.launch_count()
            rc, msg = _c_call(product_lib, mt._ctx, cams, device, rgb=rgb.ctypes.data, d_rgb=d_rgb.data_ptr(), **kw)
            assert rc == MTB_ERR_ARG and words in msg, (device, kw, rc, msg)
            assert mt.launch_count() == before
        rc, msg = _c_call(product_lib, mt._ctx, cams, device, rgb=rgb.ctypes.data, d_rgb=d_rgb.data_ptr(), eye=[0.1, -0.1, 0.1, -0.1])
        assert rc == MTB_OK, msg
    torch.cuda.synchronize()
    assert np.array_equal(d_rgb[:2].cpu().numpy(), rgb[:2])


@pytest.mark.gpu
def test_other_paths_are_unchanged_after_a_panorama_batch(product_lib, scene_dir):
    files, cfg = scenes.config_scene("C1", scene_dir)
    mt = _tracer(files.obj_path, 5)
    mt.GetScene().lights = _lights(scenes.LIGHT_RIG[:2])
    cams = _orbit_subframes(files.camera, 3, 2)
    lenses = [(1.5, -0.5, 60.0)] * len(cams)
    before_batch = mt.render_batch(cams, 64, 48, subframes=2)["rgb"].copy()
    before_lens = mt.render_batch(cams, 64, 48, subframes=2, lenses=lenses)["rgb"].copy()
    before_chunk = mt.render_chunk(files.camera, 96, 64, 0, 0, 96, 64)["rgb"].copy()
    mt.render_batch(cams, 128, 64, samples_per_axis=2, subframes=2, panorama=FULL, eye_offsets=[0.3] * len(cams))
    mt.render_batch(cams[:4], 64, 32, panorama=(90.0, 45.0), debug=True)
    assert np.array_equal(mt.render_batch(cams, 64, 48, subframes=2)["rgb"], before_batch)
    assert np.array_equal(mt.render_batch(cams, 64, 48, subframes=2, lenses=lenses)["rgb"], before_lens)
    assert np.array_equal(mt.render_chunk(files.camera, 96, 64, 0, 0, 96, 64)["rgb"], before_chunk)
    mt.close()


@pytest.mark.gpu
@pytest.mark.parametrize("s,k", [(1, 2), (2, 3)])
def test_cpp_shim_panorama_batches(product_lib, scene_dir, tmp_path, s, k):
    """RayTraceBatch with panorama parameters, called from C++ (tests/cpp/pano_check.cc): the output equals
    render_batch(..., panorama=..., eye_offsets=...) of the same sub-frames."""
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    exe = str(tmp_path / "pano_check")
    lib_dir = os.path.join(ROOT, "mythtracer_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                           os.path.join(HERE, "cpp", "pano_check.cc"), "-L", lib_dir, "-lmythtracer_b200", "-Wl,-rpath," + lib_dir, "-o", exe])
    files, cfg = scenes.config_scene("C2", scene_dir, 0.1)
    W, H = 64, 32
    prefix = str(tmp_path / "out")
    res = subprocess.run([exe, files.obj_path, prefix, str(W), str(H), str(s), str(k)], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    assert "pano ok" in res.stdout
    mt = _tracer(files.obj_path, 3)
    mt.GetScene().lights = _lights([(231.82174, 81.69966, 27.78259, 0.3, 0.3, 0.3, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0),
                                    (200.0, 95.0, 160.0, 0.0, 0.0, 0.0, 0.3, 0.3, 0.3, 0.3, 0.3, 0.3)])
    cams = [(301.37, 57.21, 161.13, 4.0, 243.0 + 3.0 * v, 0.0, 110.0) for v in range(2) for j in range(k)]
    eyes = [(-3.2 if v == 0 else 3.2) for v in range(2) for j in range(k)]
    want = mt.render_batch(cams, W, H, samples_per_axis=s, subframes=k, panorama=FULL, eye_offsets=eyes)["rgb"]
    got = np.fromfile(prefix + ".rgb", np.uint8).reshape(2, H, W, 3)
    assert np.array_equal(got, want)
