"""Batches into device memory (mtb_render_batch_device / render_batch(..., device=True)): every batch form with its outputs
left in HBM of device 0, ordered on the caller's stream.  The bytes must be exactly those of the host form with the same
arguments - which the other batch tests pin to render_chunk, the oracle and the reference's stored frames - and the
ordering must hold without any synchronisation between the caller's work and the batch."""
import ctypes
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from tests import scenes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
MTB_OK, MTB_ERR_ARG, MTB_ERR_CUDA = 0, -1, -2
TAPS = ("sig_hits", "sig_shadow", "n_rays")


def _yawed(cam, dyaw):
    c = list(cam)
    c[4] += dyaw
    return tuple(c)


def _orbit(cam, n, step=2.0):
    return [_yawed(cam, step * i) for i in range(n)]


def _lights(rows):
    from mythtracer_b200 import Light
    return [Light.from_tuple(l) for l in rows]


def _light_sets(n):
    """A different light set of two lights for every view."""
    return [_lights(scenes.LIGHT_RIG[j % 3:j % 3 + 2]) for j in range(n)]


def _tracer(path, depth, flags=0, devices=None):
    from mythtracer_b200 import MythTracer
    mt = MythTracer(devices=devices, max_depth=depth, flags=flags)
    assert mt.LoadObj(path), mt.last_error()
    return mt


def _c1(scene_dir, depth=5, flags=0, devices=None):
    files, cfg = scenes.config_scene("C1", scene_dir)
    mt = _tracer(files.obj_path, depth, flags, devices)
    mt.GetScene().lights = _lights(scenes.LIGHT_RIG[:2])
    return files, mt


def _host(t):
    return t.cpu().numpy()


def _assert_device_equals_host(mt, cams, w, h, s=1, k=1, lights=None, debug=False, taps=False, out=None):
    """render_batch(..., device=True) copied back equals render_batch(...) byte for byte, every plane included."""
    import torch
    want = mt.render_batch(cams, w, h, lights=lights, samples_per_axis=s, subframes=k, debug=debug, taps=taps)
    stats_before = mt.last_stats
    got = mt.render_batch(cams, w, h, lights=lights, samples_per_axis=s, subframes=k, debug=debug, taps=taps, out=out, device=True)
    torch.cuda.synchronize()
    assert got["stats"] is None and mt.last_stats is stats_before
    assert got["rgb"].dtype == torch.uint8 and got["rgb"].device == torch.device("cuda", 0)
    assert tuple(got["rgb"].shape) == want["rgb"].shape == (len(cams) // k, h, w, 3)
    if out is not None:
        assert got["rgb"] is out
    rgb = _host(got["rgb"])
    assert np.array_equal(rgb, want["rgb"]), "rgb: %d channels differ" % int((rgb != want["rgb"]).sum())
    if debug:
        plane = (len(cams), s * h, s * w)
        assert tuple(got["debug"].shape) == plane + (32,)
        assert _host(got["debug"]).tobytes() == want["debug"].tobytes()
        assert np.array_equal(_host(got["line_no"]), want["line_no"])
        assert _host(got["points"]).tobytes() == np.ascontiguousarray(want["points"]).tobytes()
    else:
        assert "debug" not in got
    for key, dtype in zip(TAPS, (torch.uint64, torch.uint64, torch.uint32)):
        if taps:
            assert got[key].dtype == dtype
            assert np.array_equal(_host(got[key]), want[key]), key
        else:
            assert key not in got
    return got, want


# ---------------------------------------------------------------------------------------------- CPU


def test_host_only_context_returns_err_cuda(product_lib):
    from mythtracer_b200 import MythTracer, MythTracerError, api
    files, cfg = scenes.config_scene("C1", "/tmp/mtb_scenes")
    mt = MythTracer(host_only=True)
    assert mt.LoadObj(files.obj_path)
    cams = np.zeros(2, api.CAMERA_DTYPE)
    cams[0] = cams[1] = api.Camera.from_tuple(files.camera).as_array()
    fake = ctypes.c_void_p(1 << 20)  # (never dereferenced: the context has no device)
    rc = product_lib.mtb_render_batch_device(mt._ctx, cams.ctypes.data_as(ctypes.c_void_p), 2, 1, None, 0, 16, 16, 1, 3, fake, None, None,
                                             None, None)
    assert rc == MTB_ERR_CUDA and "no CPU fallback" in mt.last_error()
    pytest.importorskip("torch")
    for kw in (dict(), dict(debug=True, taps=True), dict(subframes=2), dict(samples_per_axis=4)):
        with pytest.raises(MythTracerError, match="no CPU fallback"):
            mt.render_batch([files.camera, files.camera], 16, 16, device=True, **kw)


def test_device_arguments_are_checked_in_python(product_lib):
    torch = pytest.importorskip("torch")
    from mythtracer_b200 import MythTracer, MythTracerError
    files, cfg = scenes.config_scene("C1", "/tmp/mtb_scenes")
    mt = MythTracer(host_only=True)
    assert mt.LoadObj(files.obj_path)
    cams = [files.camera] * 4
    for bad in (1, 0, "yes", None, np.array([True]), "cuda"):
        with pytest.raises(MythTracerError, match="device must be True or False"):
            mt.render_batch(cams, 16, 8, device=bad)
    # device=True takes a uint8 CUDA tensor of the output shape on devices[0], C-contiguous
    for out in (np.zeros((4, 8, 16, 3), np.uint8),                              # numpy
                torch.zeros((4, 8, 16, 3), dtype=torch.uint8),                   # host tensor
                torch.zeros((4, 8, 16, 3), dtype=torch.uint8, device="meta"),    # not a CUDA tensor
                torch.zeros((4, 8, 16, 3), dtype=torch.int8),                    # dtype
                torch.zeros((4, 16, 8, 3), dtype=torch.uint8),                   # shape
                torch.zeros((4, 8, 16, 4), dtype=torch.uint8)[..., :3],          # not contiguous
                [0] * 4):
        with pytest.raises(MythTracerError, match="out must be a C-contiguous uint8 torch tensor"):
            mt.render_batch(cams, 16, 8, out=out, device=True)
    # with subframes the output views, not the sub-frames
    with pytest.raises(MythTracerError, match="out must be"):
        mt.render_batch(cams, 16, 8, out=torch.zeros((4, 8, 16, 3), dtype=torch.uint8), subframes=2, device=True)
    # device=False takes numpy only
    with pytest.raises(MythTracerError, match="out must be a numpy array"):
        mt.render_batch(cams, 16, 8, out=torch.zeros((4, 8, 16, 3), dtype=torch.uint8))
    # the checks of the host form apply
    with pytest.raises(MythTracerError, match="samples_per_axis"):
        mt.render_batch(cams, 16, 8, samples_per_axis=3, device=True)
    with pytest.raises(MythTracerError, match="subframes"):
        mt.render_batch(cams, 16, 8, subframes=0, device=True)
    with pytest.raises(MythTracerError, match="debug and taps"):
        mt.render_batch(cams, 16, 8, subframes=2, debug=True, device=True)
    with pytest.raises(MythTracerError, match="one per view"):
        mt.render_batch(cams, 16, 8, lights=[_lights(scenes.LIGHT_RIG[:2])], device=True)
    with pytest.raises(MythTracerError, match="no cameras"):
        mt.render_batch([], 16, 8, device=True)


def test_package_imports_without_torch():
    """device=True imports torch lazily: the package itself does not."""
    code = ("import sys; sys.modules['torch'] = None; sys.path.insert(0, %r); import mythtracer_b200; from mythtracer_b200 import api; "
            "assert 'torch' not in [m for m in sys.modules if sys.modules[m] is not None]; print('ok')" % ROOT)
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0 and "ok" in res.stdout, res.stdout + res.stderr


# ---------------------------------------------------------------------------------------------- GPU


CASES = {
    # name: (views, w, h, s, k, lights per view, debug, taps)
    "s1": (8, 96, 64, 1, 1, False, False, False),
    "s2": (8, 96, 64, 2, 1, False, False, False),
    "s4": (4, 64, 40, 4, 1, True, False, False),
    "s8": (4, 40, 24, 8, 1, False, False, False),
    "accum_k3_s1": (6, 96, 64, 1, 3, True, False, False),
    "accum_k3_s2": (6, 64, 40, 2, 3, False, False, False),
    "planes_s1": (6, 96, 64, 1, 1, True, True, True),
    "planes_s2": (4, 64, 40, 2, 1, False, True, True),
    "debug_only": (3, 72, 40, 1, 1, False, True, False),
    "taps_only": (3, 72, 40, 2, 1, True, False, True),
    "one_view": (1, 96, 64, 1, 1, False, False, False),
    "one_view_planes": (1, 48, 32, 2, 1, True, True, True),
    "64_views": (64, 64, 40, 1, 1, True, False, False),
    "64_views_s2_planes": (64, 32, 24, 2, 1, False, True, True),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_device_output_equals_the_host_form(product_lib, scene_dir, case):
    n, w, h, s, k, per_view, debug, taps = CASES[case]
    files, mt = _c1(scene_dir)
    cams = _orbit(files.camera, n)
    _assert_device_equals_host(mt, cams, w, h, s, k, _light_sets(n) if per_view else None, debug, taps)
    mt.close()


@pytest.mark.gpu
@pytest.mark.parametrize("s,k", [(1, 1), (2, 1), (1, 3), (4, 2)])
def test_odd_size_into_a_tensor_offset_by_one_byte(product_lib, scene_dir, s, k):
    """75x49 (not a multiple of 8) into `out`, a view that starts 1 byte into a larger tensor: the plain epilogue falls
    back to byte stores, and the bytes around the output are left alone."""
    import torch
    files, mt = _c1(scene_dir)
    w, h, n_out = 75, 49, 3
    nbytes = n_out * h * w * 3
    big = torch.full((nbytes + 16,), 0xA5, dtype=torch.uint8, device="cuda:0")
    out = big[1:1 + nbytes].view(n_out, h, w, 3)
    assert out.is_contiguous() and out.data_ptr() % 8 == 1
    cams = _orbit(files.camera, n_out * k, 0.7)
    _assert_device_equals_host(mt, cams, w, h, s, k, _light_sets(n_out * k), out=out)
    rest = _host(big)
    assert rest[0] == 0xA5 and np.all(rest[1 + nbytes:] == 0xA5)


@pytest.mark.gpu
def test_full_size_c3_view_equals_the_reference(product_lib, scene_dir):
    import torch
    z = np.load(os.path.join(HERE, "golden", "full_C3.npz"))
    files, cfg = scenes.config_scene("C3", scene_dir)
    mt = _tracer(files.obj_path, cfg["depth"])
    mt.GetScene().lights = _lights(files.lights)
    W, H = int(z["width"]), int(z["height"])
    assert (W, H) == (cfg["width"], cfg["height"]) and int(z["depth"]) == cfg["depth"]
    got = mt.render_batch([files.camera], W, H, device=True)
    torch.cuda.synchronize()
    rgb = _host(got["rgb"])[0]
    assert np.array_equal(rgb, z["rgb"]), "%d channels differ from full_C3" % int((rgb != z["rgb"]).sum())
    mt.close()


@pytest.mark.gpu
def test_ordering_on_a_torch_stream(product_lib, scene_dir):
    """On a non-default torch stream: a fill of `out` queued before the call behind a long device sleep does not land
    on the frame, the call returns while the sleep still runs, and a reduction queued right after the call, without any
    synchronisation, sees the finished frame."""
    import torch
    files, mt = _c1(scene_dir)
    w, h, n = 96, 64, 4
    cams = _orbit(files.camera, n)
    want = mt.render_batch(cams, w, h)["rgb"]
    stream = torch.cuda.Stream(device=0)
    with torch.cuda.stream(stream):
        out = torch.empty((n, h, w, 3), dtype=torch.uint8, device="cuda:0")
        mt.render_batch(cams, w, h, out=out, device=True)  # (grows the context's buffers, so that the timed call does not)
        stream.synchronize()
        torch.cuda._sleep(500_000_000)
        out.fill_(7)
        mt.render_batch(cams, w, h, out=out, device=True)
        still_sleeping = not stream.query()
        total = out.to(torch.int64).sum()
        first = out[0].clone()
    torch.cuda.synchronize()
    assert still_sleeping, "the call waited for the caller's stream"
    assert np.array_equal(_host(out), want)
    assert int(total.item()) == int(want.astype(np.int64).sum())
    assert np.array_equal(_host(first), want[0])


@pytest.mark.gpu
def test_two_calls_on_two_streams(product_lib, scene_dir):
    """Two calls of different shapes queued back to back on two streams into two tensors: both right after one
    synchronise."""
    import torch
    files, mt = _c1(scene_dir)
    a_cams, b_cams = _orbit(files.camera, 5), _orbit(_yawed(files.camera, 1.0), 6)
    want_a = mt.render_batch(a_cams, 96, 64, samples_per_axis=2)["rgb"]
    want_b = mt.render_batch(b_cams, 72, 40, lights=_light_sets(6), subframes=3)["rgb"]
    sa, sb = torch.cuda.Stream(device=0), torch.cuda.Stream(device=0)
    with torch.cuda.stream(sa):
        a = mt.render_batch(a_cams, 96, 64, samples_per_axis=2, device=True)["rgb"]
    with torch.cuda.stream(sb):
        b = mt.render_batch(b_cams, 72, 40, lights=_light_sets(6), subframes=3, device=True)["rgb"]
    torch.cuda.synchronize()
    assert np.array_equal(_host(a), want_a)
    assert np.array_equal(_host(b), want_b)


def _c_call(lib, mt, cams, w, h, rgb_ptr, s=1, k=1, dbg_ptr=None, taps=None, stream=None, stats=None, lights=None):
    """mtb_render_batch_device through the C ABI; taps: (sig_hits, sig_shadow, n_rays) pointers or None."""
    from mythtracer_b200 import api
    cam_arr = np.zeros(len(cams), api.CAMERA_DTYPE)
    for i, c in enumerate(cams):
        cam_arr[i] = api.Camera.from_tuple(c).as_array()
    light_arr, n_lights = None, 0
    if lights is not None:
        n_lights = len(lights[0])
        light_arr = api._lights_array([l for ls in lights for l in ls])
    tap_ptr = None
    if taps is not None:
        tap_struct = api._TapsStruct(*taps)
        tap_ptr = ctypes.cast(ctypes.pointer(tap_struct), ctypes.c_void_p)
    rc = lib.mtb_render_batch_device(mt._ctx, cam_arr.ctypes.data_as(ctypes.c_void_p), len(cams) // max(k, 1), k,
                                     None if light_arr is None else light_arr.ctypes.data_as(ctypes.c_void_p), n_lights, w, h, s, mt.max_depth,
                                     None if rgb_ptr is None else ctypes.c_void_p(rgb_ptr), None if dbg_ptr is None else ctypes.c_void_p(dbg_ptr),
                                     tap_ptr, None if stream is None else ctypes.c_void_p(stream),
                                     None if stats is None else stats.ctypes.data_as(ctypes.c_void_p))
    return rc, mt.last_error()


@pytest.mark.gpu
def test_refused_arguments_launch_nothing(product_lib, scene_dir):
    import torch
    files, mt = _c1(scene_dir, depth=3)
    mt.push_lights()
    w, h, n = 40, 24, 4
    cams = _orbit(files.camera, n)
    plane = n * h * w
    rgb = torch.zeros((n, h, w, 3), dtype=torch.uint8, device="cuda:0")
    dbg = torch.zeros(plane * 32 + 8, dtype=torch.uint8, device="cuda:0")
    hits = torch.zeros(plane + 1, dtype=torch.int64, device="cuda:0")
    rays = torch.zeros(plane + 1, dtype=torch.int32, device="cuda:0")
    pinned = torch.zeros(n * h * w * 3, dtype=torch.uint8).pin_memory()
    pageable = np.zeros(n * h * w * 3, np.uint8)
    ok_taps = (hits.data_ptr(), hits.data_ptr(), rays.data_ptr())
    assert _c_call(product_lib, mt, cams, w, h, rgb.data_ptr(), dbg_ptr=dbg.data_ptr(), taps=ok_taps)[0] == MTB_OK
    torch.cuda.synchronize()
    cases = [
        (dict(rgb_ptr=None), "d_rgb is NULL"),
        (dict(rgb_ptr=pageable.ctypes.data), "d_rgb is not device memory"),
        (dict(rgb_ptr=pinned.data_ptr()), "d_rgb is not device memory"),
        (dict(dbg_ptr=pinned.data_ptr()), "d_dbg is not device memory"),
        (dict(dbg_ptr=dbg.data_ptr() + 4), "d_dbg must be 8-byte aligned"),
        (dict(taps=(hits.data_ptr() + 4, None, None)), "sig_hits must be 8-byte aligned"),
        (dict(taps=(None, hits.data_ptr() + 2, None)), "sig_shadow must be 8-byte aligned"),
        (dict(taps=(None, None, rays.data_ptr() + 2)), "n_rays must be 4-byte aligned"),
        (dict(taps=(None, None, pageable.ctypes.data)), "n_rays is not device memory"),
        (dict(k=2, dbg_ptr=dbg.data_ptr()), "no debug or tap planes of accumulated views"),
        (dict(k=2, taps=(None, None, rays.data_ptr())), "no debug or tap planes of accumulated views"),
        (dict(s=3), "samples_per_axis"),
        (dict(k=0), "subframes"),
    ]
    for kw, words in cases:
        launches = mt.launch_count()
        args = dict(rgb_ptr=rgb.data_ptr())
        args.update(kw)
        rc, msg = _c_call(product_lib, mt, cams, w, h, **args)
        assert rc == MTB_ERR_ARG and words in msg, (kw, rc, msg)
        assert mt.launch_count() == launches, kw
    # the partition must be (0, 1)
    mt.set_partition(1, 2)
    launches = mt.launch_count()
    rc, msg = _c_call(product_lib, mt, cams, w, h, rgb.data_ptr())
    assert rc == MTB_ERR_ARG and "partition" in msg and mt.launch_count() == launches
    mt.set_partition(0, 1)
    # a stream that is being captured into a graph
    graph, side = torch.cuda.CUDAGraph(), torch.cuda.Stream(device=0)
    x = torch.zeros(4, device="cuda:0")
    launches = mt.launch_count()
    with torch.cuda.graph(graph, stream=side, capture_error_mode="relaxed"):
        x += 1
        rc, msg = _c_call(product_lib, mt, cams, w, h, rgb.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
    assert rc == MTB_ERR_ARG and "captured" in msg and mt.launch_count() == launches
    # memory of another device
    if torch.cuda.device_count() >= 2:
        other = torch.zeros((n, h, w, 3), dtype=torch.uint8, device="cuda:1")
        rc, msg = _c_call(product_lib, mt, cams, w, h, other.data_ptr())
        assert rc == MTB_ERR_ARG and "not of the context's device 0" in msg and mt.launch_count() == launches
        from mythtracer_b200 import MythTracerError
        with pytest.raises(MythTracerError, match="out must be"):
            mt.render_batch(cams, w, h, out=other, device=True)
    # a CUDA tensor is not an output of the host form
    from mythtracer_b200 import MythTracerError
    with pytest.raises(MythTracerError, match="out must be a numpy array"):
        mt.render_batch(cams, w, h, out=rgb)
    # and the context still renders
    want = mt.render_batch(cams, w, h)["rgb"]
    assert _c_call(product_lib, mt, cams, w, h, rgb.data_ptr())[0] == MTB_OK
    torch.cuda.synchronize()
    assert np.array_equal(_host(rgb), want)


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, 1], ids=["timed", "count_work"])
def test_stats_equal_those_of_the_host_form(product_lib, scene_dir, flags):
    import torch
    from mythtracer_b200.api import STATS_DTYPE
    files, mt = _c1(scene_dir, depth=4, flags=flags)
    mt.push_lights()
    for n, s, k, planes in ((4, 1, 1, False), (6, 2, 3, False), (3, 2, 1, True)):
        w, h = 48, 32
        cams = _orbit(files.camera, n)
        lights = _light_sets(n)
        want = mt.render_batch(cams, w, h, lights=lights, samples_per_axis=s, subframes=k, debug=planes, taps=planes)
        rgb = torch.zeros((n // k, h, w, 3), dtype=torch.uint8, device="cuda:0")
        size = n * s * s * w * h
        dbg = torch.zeros(size * 32, dtype=torch.uint8, device="cuda:0") if planes else None
        hits = torch.zeros(2 * size, dtype=torch.int64, device="cuda:0") if planes else None
        rays = torch.zeros(size, dtype=torch.int32, device="cuda:0") if planes else None
        stats = np.zeros((), STATS_DTYPE)
        rc, msg = _c_call(product_lib, mt, cams, w, h, rgb.data_ptr(), s, k, None if dbg is None else dbg.data_ptr(),
                          (hits.data_ptr(), hits.data_ptr() + 8 * size, rays.data_ptr()) if planes else None, stats=stats, lights=lights)
        assert rc == MTB_OK, msg
        # stats != NULL waits for the batch: the outputs are there without any further synchronisation of the stream
        assert np.array_equal(_host(rgb), want["rgb"])
        for key in STATS_DTYPE.names:
            if not key.endswith("_ms"):
                assert stats[key] == want["stats"][key], (n, s, k, key)
        assert stats["kernel_ms"] > 0.0 and stats["total_ms"] >= stats["kernel_ms"]
        if planes:
            assert _host(dbg).tobytes() == want["debug"].tobytes()
            assert _host(hits[:size]).view(np.uint64).tobytes() == want["sig_hits"].tobytes()
            assert _host(rays).view(np.uint32).tobytes() == want["n_rays"].tobytes()
        if flags:
            assert stats["n_bvh"] > 0 and stats["shadow"] > 0


@pytest.mark.gpu
def test_device_batches_leave_the_single_frame_state_alone(product_lib, scene_dir):
    import torch
    files, cfg = scenes.config_scene("C1", scene_dir)
    w, h = 160, 120
    mt = _tracer(files.obj_path, 3)  # automatic pipeline choice
    mt.GetScene().lights = _lights(scenes.LIGHT_RIG[:2])
    before = [mt.render_chunk(files.camera, w, h, 0, 0, w, h)["rgb"] for _ in range(8)]  # past the deciding frames
    pipeline = mt.pipeline_in_use()
    assert pipeline[0] != "measuring"
    mt.max_depth = 7
    for kw in (dict(), dict(samples_per_axis=2, debug=True, taps=True), dict(subframes=3, samples_per_axis=4)):
        mt.render_batch(_orbit(files.camera, 6), 64, 48, lights=[_lights(scenes.LIGHT_RIG[1:4])] * 6, device=True, **kw)
    mt.render_batch(_orbit(files.camera, 2), 64, 48, device=True)
    torch.cuda.synchronize()
    mt.max_depth = 3
    after = mt.render_chunk(files.camera, w, h, 0, 0, w, h)["rgb"]
    assert np.array_equal(after, before[-1])
    assert mt.pipeline_in_use() == pipeline


@pytest.mark.gpu
def test_split_over_devices_equals_one_device(product_lib, scene_dir):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    files, cfg = scenes.config_scene("C1", scene_dir)
    w, h = 75, 49
    n = min(torch.cuda.device_count(), 8)
    one = _tracer(files.obj_path, 5)
    many = _tracer(files.obj_path, 5, devices=list(range(n)))
    assert many.device_count() == n
    for n_out, k, s, planes in ((n + 3, 1, 1, True), (1, 1, 2, False), (n - 1, 4, 8, False), (2 * n, 2, 4, False), (2 * n + 1, 1, 2, True)):
        cams = _orbit(files.camera, n_out * k, 0.9)
        lights = _light_sets(len(cams))
        want = one.render_batch(cams, w, h, lights=lights, samples_per_axis=s, subframes=k, debug=planes, taps=planes)
        got = many.render_batch(cams, w, h, lights=lights, samples_per_axis=s, subframes=k, debug=planes, taps=planes, device=True)
        torch.cuda.synchronize()
        assert got["rgb"].device == torch.device("cuda", 0)
        assert np.array_equal(_host(got["rgb"]), want["rgb"]), (n_out, k, s)
        if planes:
            assert _host(got["debug"]).tobytes() == want["debug"].tobytes()
            for key in TAPS:
                assert np.array_equal(_host(got[key]), want[key]), key


@pytest.mark.gpu
@pytest.mark.parametrize("s,k", [(1, 1), (2, 3)])
def test_cpp_shim_batches_into_device_memory(product_lib, scene_dir, tmp_path, s, k):
    """RayTraceBatchDevice from C++ (tests/cpp/batch_device_check.cc) into a cudaMalloc buffer: the output equals
    render_batch of the same views."""
    nvcc = os.environ.get("NVCC", "nvcc")
    if shutil.which(nvcc) is None:
        pytest.skip("nvcc not available")
    exe = str(tmp_path / "batch_device_check")
    lib_dir = os.path.join(ROOT, "mythtracer_b200")
    subprocess.check_call([nvcc, "-std=c++17", "-O1", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-Wall,-Wextra,-Werror",
                           "-I", os.path.join(ROOT, "include"), os.path.join(HERE, "cpp", "batch_device_check.cc"), "-L", lib_dir,
                           "-lmythtracer_b200", "-Xlinker", "-rpath," + lib_dir, "-o", exe])
    files, cfg = scenes.config_scene("C2", scene_dir, 0.1)
    W, H = 60, 36
    prefix = str(tmp_path / "out")
    res = subprocess.run([exe, files.obj_path, prefix, str(W), str(H), str(s), str(k)], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    assert "device ok" in res.stdout
    mt = _tracer(files.obj_path, 3)
    mt.GetScene().lights = _lights([(231.82174, 81.69966, 27.78259, 0.3, 0.3, 0.3, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0),
                                    (200.0, 95.0, 160.0, 0.0, 0.0, 0.0, 0.3, 0.3, 0.3, 0.3, 0.3, 0.3)])
    cams = [(301.37, 57.21, 161.13, 4.0, 243.0 + 3.0 * v + 0.5 * j, 0.0, 110.0) for v in range(2) for j in range(k)]
    want = mt.render_batch(cams, W, H, samples_per_axis=s, subframes=k)["rgb"]
    got = np.fromfile(prefix + ".rgb", np.uint8).reshape(2, H, W, 3)
    assert np.array_equal(got, want)
