"""The oracle (CPU restatement) against the unmodified reference.

Where the reference library oracle/_ref is built (oracle/build_ref.sh, from the reference's own sources) it is run
live; otherwise the tests that have one compare with what the reference rendered for the same inputs, stored under
tests/golden/ by tests/golden/make_golden.py and make_golden_full.py.  The C1 frame and the random rays have no
stored answer: those two tests skip without the library (test_oracle_golden.py pins the oracle on other scenes)."""
import hashlib
import os

import numpy as np
import pytest

from tests import scenes

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def ref_cls(oracle_mod):
    if not oracle_mod.Reference.available():
        pytest.skip("the unmodified reference library (oracle/_ref) is not built")
    return oracle_mod.Reference


def _file_sha(path):
    with open(path, "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()


def _compare_with_fixture(oracle_mod, fixture, obj, cam, lights, w, h, depth, chunk=None):
    """The oracle's render against the reference's render of the same frame stored in tests/golden/<fixture>.npz
    (the whole frame; a chunk is compared with the same pixels of it)."""
    z = np.load(os.path.join(GOLDEN, fixture + ".npz"))
    assert np.array_equal(np.array(cam), z["camera"]) and np.array_equal(np.array(lights), z["lights"])
    assert (w, h, depth) == (int(z["width"]), int(z["height"]), int(z["depth"])) and z["line_no"].shape == (h, w)
    orc = oracle_mod.Oracle.from_obj(obj)
    orc.set_lights(lights)
    out = orc.render(cam, w, h, chunk=chunk, depth=depth)
    x, y, cw, ch = chunk or (0, 0, w, h)
    assert np.array_equal(out["line_no"], z["line_no"][y:y + ch, x:x + cw])
    assert np.array_equal(out["rgb"], z["rgb"][y:y + ch, x:x + cw])
    return orc, out, z


def _compare(oracle_mod, ref_cls, obj, cam, lights, w, h, depth, chunk=None):
    orc = oracle_mod.Oracle.from_obj(obj)
    orc.set_lights(lights)
    ref = ref_cls(obj)
    ref.set_lights(lights)
    a = orc.render(cam, w, h, chunk=chunk, depth=depth)
    b = ref.render(cam, w, h, chunk=chunk, depth=depth)
    assert np.array_equal(a["line_no"], b["line_no"])
    assert np.array_equal(a["points"], b["points"], equal_nan=True)
    assert np.array_equal(a["rgb"], b["rgb"])
    assert np.array_equal(orc.aabb(), ref.aabb())
    return orc, ref


def test_c1_bit_identical(oracle_mod, ref_cls, scene_dir):
    files, cfg = scenes.config_scene("C1", scene_dir)
    _compare(oracle_mod, ref_cls, files.obj_path, files.camera, files.lights, cfg["width"], cfg["height"], cfg["depth"])


def test_c2_textured_tile(oracle_mod, scene_dir):
    files, cfg = scenes.config_scene("C2", scene_dir)
    assert _file_sha(files.obj_path) == str(np.load(os.path.join(GOLDEN, "full_C2.npz"))["obj_sha256"])
    args = (files.obj_path, files.camera, files.lights, cfg["width"], cfg["height"], cfg["depth"])
    chunk = (500, 300, 96, 64)
    _compare_with_fixture(oracle_mod, "full_C2", *args, chunk=chunk)
    if oracle_mod.Reference.available():
        _compare(oracle_mod, oracle_mod.Reference, *args, chunk=chunk)


def test_lattice_nan_column(oracle_mod, scene_dir):
    path, cam, lights = scenes.lattice_scene(scene_dir)
    assert _file_sha(path) == _file_sha(os.path.join(GOLDEN, "lattice.obj"))
    orc, out, z = _compare_with_fixture(oracle_mod, "lattice", path, cam, lights, 65, 49, 5)
    assert np.array_equal(orc.aabb(), z["aabb"])
    # the fixture was made on another host: a 1-ulp difference of libm's sin/cos in the camera basis moves hit
    # points by ~1e-13 (the live comparison below is bit for bit)
    np.testing.assert_allclose(out["points"], z["points"], rtol=0, atol=1e-9, equal_nan=True)
    if oracle_mod.Reference.available():
        _compare(oracle_mod, oracle_mod.Reference, path, cam, lights, 65, 49, 5)


def test_depth_8_four_lights(oracle_mod, scene_dir):
    """A tile of the C5 frame (the C3 scene at 3840x2160, depth 8, the four-light rig)."""
    files, cfg = scenes.config_scene("C5", scene_dir)
    assert cfg["depth"] == 8 and np.array_equal(np.array(files.lights), np.array(scenes.LIGHT_RIG))
    assert _file_sha(files.obj_path) == str(np.load(os.path.join(GOLDEN, "full_C5.npz"))["obj_sha256"])
    args = (files.obj_path, files.camera, files.lights, cfg["width"], cfg["height"], cfg["depth"])
    chunk = (1800, 1000, 96, 72)
    _compare_with_fixture(oracle_mod, "full_C5", *args, chunk=chunk)
    if oracle_mod.Reference.available():
        _compare(oracle_mod, oracle_mod.Reference, *args, chunk=chunk)


def test_random_rays(oracle_mod, ref_cls, scene_dir):
    files, cfg = scenes.config_scene("C1", scene_dir)
    orc = oracle_mod.Oracle.from_obj(files.obj_path)
    ref = ref_cls(files.obj_path)
    rng = np.random.default_rng(5)
    o, d = scenes.random_rays(rng, orc.aabb(), 20000)
    d[:1000] = np.eye(3)[rng.integers(0, 3, 1000)]
    d[1000:2000] *= 3.7
    a = orc.intersect(o, d)
    b = ref.intersect(o, d)
    line_no = np.where(a["tri"] >= 0, orc.tris["line_no"][np.maximum(a["tri"], 0)], -1)
    assert np.array_equal(line_no, b["line_no"])
    hit = b["line_no"] >= 0
    assert np.array_equal(a["t"][hit], b["t"][hit])
    assert np.array_equal(a["point"][hit], b["point"][hit])
