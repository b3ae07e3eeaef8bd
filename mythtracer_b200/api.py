"""Python mirror of the reference's renderer API on top of the C ABI (include/mythtracer_b200.h).

Names, argument meaning and error behaviour follow the reference's public C++ interface for this path:

    reference (VerStarting/)                      here
    ------------------------------------------    -------------------------------------------
    Camera{origin,pitch,yaw,roll,aov}  camera.h:31-33     Camera
    Light{position,ambient,diffuse,specular} light.h:8-14 Light
    WorkChunk  mythtracer.h:18-53                 WorkChunk (output_bitmap / output_debug filled by RayTrace)
    MythTracer::LoadObj            mythtracer.cc:247      MythTracer.LoadObj            -> bool
    MythTracer::GetScene()->lights scene.h:14             MythTracer.GetScene().lights  (plain list, re-read per call)
    MythTracer::RayTrace(w,h,cam,out) mythtracer.cc:258   MythTracer.RayTrace(w, h, cam) -> bytes-like RGB24 or None
    MythTracer::RayTrace(WorkChunk*)  mythtracer.cc:280   MythTracer.RayTrace(chunk)     -> bool
    OctTree::IntersectRay          octtree.cc:26          MythTracer.GetScene().tree.IntersectRays (batched)

The work is done by the CUDA kernels of libmythtracer_b200.so.  There is no CPU fallback: importing works
anywhere (so the host-side logic can be tested), but creating a MythTracer without the built library or
without a CUDA device raises.
"""
from __future__ import annotations

import ctypes
import os
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MTB_LIB_PATH", os.path.join(HERE, "libmythtracer_b200.so"))  # override: development A/B builds

MTB_OK = 0
MTB_FLAG_COUNT_WORK = 1
MTB_FLAG_NO_LIST_BVH = 2
MTB_FLAG_WAVEFRONT = 4
MTB_FLAG_RAY_SORT = 8
MTB_FLAG_MEGAKERNEL = 16
MTB_FLAG_NO_TILE_ORDER = 32
MTB_FLAG_PERSISTENT = 64
MTB_FLAG_EXACT_OCTREE = 128
MTB_FLAG_PACKING = 256
MTB_FLAG_WARP_SYNC = 512
MTB_FLAG_RESUME = 1024
MTB_FLAG_HYBRID = 2048
MTB_FLAG_DEVICE_BVH = 4096
MTB_FLAG_QUEUE = 8192
MTB_FLAG_PAIR_RAYS = 16384
MTB_FLAG_CHAIN_RAYS = 32768
MAX_RECURSION_LEVEL = 5  # reference mythtracer.h:11 (a run-time argument here)
FRAME_HANDLE_BYTES = 64

TRI_DTYPE = np.dtype([("vertex", "f8", (9,)), ("normal", "f8", (9,)), ("uvw", "f8", (9,)),
                      ("material", "i4"), ("line_no", "i4")], align=True)
MTL_DTYPE = np.dtype([("ambient", "f8", (3,)), ("diffuse", "f8", (3,)), ("specular", "f8", (3,)),
                      ("specular_exp", "f8"), ("reflectance", "f8"), ("transparency", "f8"),
                      ("transmission_filter", "f8", (3,)), ("refraction_index", "f8"),
                      ("texture", "i4"), ("pad_", "i4")], align=True)
LIGHT_DTYPE = np.dtype([("position", "f8", (3,)), ("ambient", "f8", (3,)), ("diffuse", "f8", (3,)),
                        ("specular", "f8", (3,))], align=True)
CAMERA_DTYPE = np.dtype([("origin", "f8", (3,)), ("pitch", "f8"), ("yaw", "f8"), ("roll", "f8"), ("aov", "f8")],
                        align=True)
DEBUG_DTYPE = np.dtype([("line_no", "i4"), ("pad_", "i4"), ("point", "f8", (3,))], align=True)
STATS_DTYPE = np.dtype([(n, "u8") for n in ("rays", "primary", "shadow", "reflect", "refract", "n_slab", "n_visit",
                                            "n_triaabb", "n_mt", "n_hit", "n_shade", "n_bvh", "n_literal", "n_fast",
                                            "n_fallback", "n_long128_rays", "n_long128_visits", "n_long512_rays", "n_long512_visits")] +
                       [("kernel_ms", "f8"), ("total_ms", "f8")], align=True)
SUMMARY_DTYPE = np.dtype([("n_triangles", "i8"), ("n_nodes", "i8"), ("n_bvh_nodes", "i8"), ("tree_depth", "i4"),
                          ("n_materials", "i4"), ("n_textures", "i4"), ("n_lights", "i4"), ("root_list", "i8"),
                          ("biggest_list", "i8"), ("interior_triangles", "i8"), ("aabb_min", "f8", (3,)),
                          ("aabb_max", "f8", (3,)), ("device_bytes", "i8"), ("n_scene_refs", "i8")], align=True)
BVH2_DTYPE = np.dtype([("lbox", "f4", (6,)), ("rbox", "f4", (6,)), ("left", "i4"), ("right", "i4"), ("pad_", "i4", (2,))])
assert BVH2_DTYPE.itemsize == 64
assert TRI_DTYPE.itemsize == 224 and MTL_DTYPE.itemsize == 136 and DEBUG_DTYPE.itemsize == 32

# every symbol include/mythtracer_b200.h declares (tests check the library exports all of them)
EXPORTED_SYMBOLS = [
    "mtb_create", "mtb_create_host", "mtb_destroy", "mtb_last_error", "mtb_device_count", "mtb_scene_upload", "mtb_load_obj",
    "mtb_set_lights", "mtb_scene_info", "mtb_scene_read", "mtb_scene_material_name", "mtb_scene_texture_name", "mtb_scene_texture", "mtb_load_mtl",
    "mtb_scene_triangle_nodes", "mtb_scene_bvh", "mtb_set_flags", "mtb_set_partition", "mtb_render_chunk",
    "mtb_render_chunk_device", "mtb_render_chunk_async", "mtb_wait", "mtb_host_alloc", "mtb_host_free", "mtb_read_counters", "mtb_launch_count", "mtb_pipeline_in_use", "mtb_intersect_rays", "mtb_camera_sensor", "mtb_version",
    "mtb_frame_create", "mtb_frame_open", "mtb_frame_release", "mtb_frame_read", "mtb_load_timing", "mtb_hybrid_share",
    "mtb_render_batch", "mtb_render_batch_async", "mtb_render_batch_ss", "mtb_render_batch_ss_async",
]


class _TextureStruct(ctypes.Structure):
    _fields_ = [("width", ctypes.c_int32), ("height", ctypes.c_int32), ("rgba", ctypes.c_void_p)]


class _TapsStruct(ctypes.Structure):
    _fields_ = [("sig_hits", ctypes.c_void_p), ("sig_shadow", ctypes.c_void_p), ("n_rays", ctypes.c_void_p)]


class MythTracerError(RuntimeError):
    pass


_lib = None


def load_library():
    """Loads libmythtracer_b200.so; raises if it has not been built (no fallback of any kind)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MythTracerError("%s is missing: run `python -m mythtracer_b200.build` (nvcc, sm_100a)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    vp, i32, i64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64
    lib.mtb_create.argtypes = [ctypes.POINTER(vp), vp, i32]
    lib.mtb_create_host.argtypes = [ctypes.POINTER(vp)]
    lib.mtb_scene_triangle_nodes.argtypes = [vp, vp, vp]
    lib.mtb_scene_bvh.argtypes = [vp, vp, vp, vp, vp]
    lib.mtb_scene_material_name.argtypes = [vp, ctypes.c_int32]
    lib.mtb_scene_material_name.restype = ctypes.c_char_p
    lib.mtb_scene_texture_name.argtypes = [vp, ctypes.c_int32]
    lib.mtb_scene_texture_name.restype = ctypes.c_char_p
    lib.mtb_scene_texture.argtypes = [vp, ctypes.c_int32, vp]
    lib.mtb_load_mtl.argtypes = [vp, ctypes.c_char_p]
    lib.mtb_destroy.argtypes = [vp]
    lib.mtb_destroy.restype = None
    lib.mtb_last_error.argtypes = [vp]
    lib.mtb_last_error.restype = ctypes.c_char_p
    lib.mtb_device_count.argtypes = [vp]
    lib.mtb_scene_upload.argtypes = [vp, vp, i64, vp, ctypes.c_int32, vp, ctypes.c_int32]
    lib.mtb_load_obj.argtypes = [vp, ctypes.c_char_p]
    lib.mtb_set_lights.argtypes = [vp, vp, ctypes.c_int32]
    lib.mtb_scene_info.argtypes = [vp, vp]
    lib.mtb_scene_read.argtypes = [vp, vp, vp]
    lib.mtb_set_flags.argtypes = [vp, ctypes.c_uint32]
    lib.mtb_set_partition.argtypes = [vp, i32, i32]
    lib.mtb_render_chunk.argtypes = [vp, vp] + [i32] * 7 + [vp, vp, vp, vp]
    lib.mtb_render_chunk_device.argtypes = [vp, vp] + [i32] * 7 + [vp, vp, vp]
    lib.mtb_render_batch.argtypes = [vp, vp, ctypes.c_int32, vp, ctypes.c_int32, i32, i32, i32, vp, vp]
    lib.mtb_render_batch_async.argtypes = [vp, vp, ctypes.c_int32, vp, ctypes.c_int32, i32, i32, i32, vp]
    lib.mtb_render_batch_ss.argtypes = [vp, vp, ctypes.c_int32, vp, ctypes.c_int32, i32, i32, i32, i32, vp, vp]
    lib.mtb_render_batch_ss_async.argtypes = [vp, vp, ctypes.c_int32, vp, ctypes.c_int32, i32, i32, i32, i32, vp]
    lib.mtb_read_counters.argtypes = [vp, vp]
    lib.mtb_pipeline_in_use.argtypes = [vp, vp, vp]
    lib.mtb_launch_count.argtypes = [vp]
    lib.mtb_launch_count.restype = ctypes.c_uint64
    lib.mtb_intersect_rays.argtypes = [vp, i64, vp, vp, vp, vp, vp, vp]
    lib.mtb_camera_sensor.argtypes = [vp, i32, i32, vp]
    lib.mtb_wait.argtypes = [vp]
    lib.mtb_hybrid_share.argtypes = [vp]
    lib.mtb_hybrid_share.restype = ctypes.c_float
    lib.mtb_load_timing.argtypes = [vp, vp]
    lib.mtb_frame_create.argtypes = [vp, ctypes.c_size_t, ctypes.POINTER(vp), vp]
    lib.mtb_frame_open.argtypes = [vp, vp, ctypes.POINTER(vp)]
    lib.mtb_frame_release.argtypes = [vp, vp]
    lib.mtb_frame_read.argtypes = [vp, vp, ctypes.c_size_t, ctypes.c_size_t, vp]
    lib.mtb_version.restype = ctypes.c_char_p
    _lib = lib
    return lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


@dataclass
class Camera:
    """reference camera.h:12-46"""
    origin: Sequence[float] = (0.0, 0.0, 0.0)
    pitch: float = 0.0
    yaw: float = 0.0
    roll: float = 0.0
    aov: float = 90.0

    kSerializedSize = 56  # camera.h:38-43

    def as_array(self) -> np.ndarray:
        c = np.zeros((), CAMERA_DTYPE)
        c["origin"] = self.origin
        c["pitch"], c["yaw"], c["roll"], c["aov"] = self.pitch, self.yaw, self.roll, self.aov
        return c

    def Serialize(self) -> bytes:  # camera.cc:71-81
        return self.as_array().tobytes()

    @classmethod
    def Deserialize(cls, data: bytes) -> Optional["Camera"]:  # camera.cc:83-96
        if len(data) != cls.kSerializedSize:
            return None
        v = np.frombuffer(data, np.float64)
        return cls(tuple(v[0:3]), float(v[3]), float(v[4]), float(v[5]), float(v[6]))

    def GetSensor(self, width: int, height: int) -> np.ndarray:
        """start_point, delta_scanline, delta_pixel as rows of a 3x3 array (camera.cc:27-63)."""
        out = np.zeros(9)
        rc = load_library().mtb_camera_sensor(_ptr(self.as_array()), width, height, _ptr(out))
        if rc != MTB_OK:
            raise MythTracerError("bad sensor arguments")
        return out.reshape(3, 3)

    @classmethod
    def from_tuple(cls, t) -> "Camera":
        return cls(tuple(t[0:3]), t[3], t[4], t[5], t[6])


@dataclass
class Light:
    """reference light.h:8-14"""
    position: Sequence[float] = (0.0, 0.0, 0.0)
    ambient: Sequence[float] = (0.0, 0.0, 0.0)
    diffuse: Sequence[float] = (0.0, 0.0, 0.0)
    specular: Sequence[float] = (0.0, 0.0, 0.0)

    @classmethod
    def from_tuple(cls, t) -> "Light":
        return cls(tuple(t[0:3]), tuple(t[3:6]), tuple(t[6:9]), tuple(t[9:12]))


def _lights_array(lights) -> np.ndarray:
    arr = np.zeros(len(lights), LIGHT_DTYPE)
    for i, l in enumerate(lights):
        if not isinstance(l, Light):
            l = Light.from_tuple(l)
        arr[i]["position"], arr[i]["ambient"] = l.position, l.ambient
        arr[i]["diffuse"], arr[i]["specular"] = l.diffuse, l.specular
    return arr


@dataclass
class WorkChunk:
    """reference mythtracer.h:18-53: one tile of a frame plus its output."""
    image_width: int = 0
    image_height: int = 0
    chunk_x: int = 0
    chunk_y: int = 0
    chunk_width: int = 0
    chunk_height: int = 0
    camera: Camera = field(default_factory=Camera)
    output_bitmap: Optional[np.ndarray] = None   # uint8 [chunk_height, chunk_width, 3]
    output_debug: Optional[np.ndarray] = None    # DEBUG_DTYPE [chunk_height, chunk_width]; set want_debug
    want_debug: bool = False

    kSerializedInputSize = 24  # mythtracer.h:28-34

    def SerializeInput(self) -> bytes:  # mythtracer.cc:314-333
        return np.array([self.image_width, self.image_height, self.chunk_x, self.chunk_y, self.chunk_width,
                         self.chunk_height], np.uint32).tobytes()

    def DeserializeInput(self, data: bytes) -> bool:  # mythtracer.cc:335-381
        if len(data) != self.kSerializedInputSize:
            return False
        iw, ih, cx, cy, cw, ch = (int(x) for x in np.frombuffer(data, np.uint32))
        if (iw > 100000 or ih > 100000 or cx > iw or cy > ih or cw > iw or ch > ih or cx + cw > iw or cy + ch > ih or
                iw == 0 or ih == 0 or cw == 0 or ch == 0):
            return False
        self.image_width, self.image_height, self.chunk_x, self.chunk_y = iw, ih, cx, cy
        self.chunk_width, self.chunk_height = cw, ch
        return True

    def SerializeOutput(self) -> Optional[bytes]:  # mythtracer.cc:383-397
        if self.output_bitmap is None:
            return None
        raw = np.ascontiguousarray(self.output_bitmap, np.uint8).tobytes()
        return np.array([len(raw)], np.uint32).tobytes() + raw

    def DeserializeOutput(self, data: bytes) -> bool:  # mythtracer.cc:399-429
        if len(data) < 4:
            return False
        sz = int(np.frombuffer(data[:4], np.uint32)[0])
        partial = self.chunk_width * self.chunk_height
        if sz // 3 != partial or sz % 3 != 0 or len(data) - 4 < sz:
            return False
        self.output_bitmap = np.frombuffer(data[4:4 + sz], np.uint8).reshape(self.chunk_height, self.chunk_width, 3).copy()
        return True


class OctTree:
    """The scene's acceleration structure as the reference exposes it (octtree.h:14-39), GPU resident."""

    def __init__(self, owner: "MythTracer"):
        self._owner = owner

    def GetAABB(self):
        info = self._owner.scene_info()
        return np.array(info["aabb_min"]), np.array(info["aabb_max"])

    def IntersectRays(self, origins, directions, want_stats: bool = False):
        """Batched OctTree::IntersectRay: returns dict(tri=insertion index or -1, t, point[, stats])."""
        return self._owner.intersect_rays(origins, directions, want_stats)

    def IntersectRay(self, origin, direction):
        """OctTree::IntersectRay for one ray: (triangle index or None, point, distance)."""
        r = self._owner.intersect_rays(np.asarray(origin, np.float64)[None], np.asarray(direction, np.float64)[None])
        if r["tri"][0] < 0:
            return None, None, None
        return int(r["tri"][0]), r["point"][0], float(r["t"][0])


class Scene:
    """reference scene.h:9-15 (materials / textures live on the device; `lights` is the caller's list)."""

    def __init__(self, owner: "MythTracer"):
        self.tree = OctTree(owner)
        self.lights: List[Light] = []


class MythTracer:
    """reference mythtracer.h:55-66, backed by the CUDA kernels."""

    def __init__(self, devices: Optional[Sequence[int]] = None, max_depth: int = MAX_RECURSION_LEVEL, flags: int = 0,
                 host_only: bool = False):
        self._lib = load_library()
        self._ctx = ctypes.c_void_p()
        dev_arr = None
        n = 0
        if devices is not None:
            dev_arr = np.ascontiguousarray(devices, np.int32)
            n = len(dev_arr)
        if host_only:  # loader / octree builder inspection only; rendering raises (no CPU fallback)
            rc = self._lib.mtb_create_host(ctypes.byref(self._ctx))
        else:
            rc = self._lib.mtb_create(ctypes.byref(self._ctx), _ptr(dev_arr), n)
        if rc != MTB_OK:
            raise MythTracerError("mtb_create failed: %s" % self._lib.mtb_last_error(None).decode())
        self.max_depth = max_depth
        self._scene = Scene(self)
        self._flags = 0
        if flags:
            self.set_flags(flags)
        self.last_stats = None

    # -- life cycle --
    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx:
            self._lib.mtb_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != MTB_OK:
            raise MythTracerError("%s failed (%d): %s" % (what, rc, self._lib.mtb_last_error(self._ctx).decode()))

    def last_error(self) -> str:
        return self._lib.mtb_last_error(self._ctx).decode()

    # -- reference API --
    def GetScene(self) -> Scene:
        return self._scene

    def LoadObj(self, fname: str) -> bool:
        return self._lib.mtb_load_obj(self._ctx, os.fsencode(fname)) == MTB_OK

    def RayTrace(self, *args):
        """RayTrace(chunk: WorkChunk) -> bool   or   RayTrace(width, height, camera) -> uint8[h, w, 3] | None."""
        if len(args) == 1:
            chunk = args[0]
            out = self.render_chunk(chunk.camera, chunk.image_width, chunk.image_height, chunk.chunk_x, chunk.chunk_y,
                                    chunk.chunk_width, chunk.chunk_height, debug=chunk.want_debug, _raise=False)
            if out is None:
                return False
            chunk.output_bitmap = out["rgb"]
            chunk.output_debug = out.get("debug")
            return True
        width, height, camera = args
        out = self.render_chunk(camera, width, height, 0, 0, width, height, _raise=False)
        return None if out is None else out["rgb"]

    # -- extended API --
    def set_flags(self, flags: int):
        self._check(self._lib.mtb_set_flags(self._ctx, flags), "mtb_set_flags")
        self._flags = flags

    def set_partition(self, index: int, count: int):
        self._check(self._lib.mtb_set_partition(self._ctx, index, count), "mtb_set_partition")

    def device_count(self) -> int:
        return self._lib.mtb_device_count(self._ctx)

    def upload(self, tris, mtls, textures=()):
        tris = np.ascontiguousarray(tris, TRI_DTYPE)
        mtls = np.ascontiguousarray(mtls, MTL_DTYPE)
        keep = [np.ascontiguousarray(t, np.uint8) for t in textures]
        tex_arr = (_TextureStruct * max(1, len(keep)))()
        for i, t in enumerate(keep):
            tex_arr[i].width, tex_arr[i].height, tex_arr[i].rgba = t.shape[1], t.shape[0], t.ctypes.data
        self._check(self._lib.mtb_scene_upload(self._ctx, _ptr(tris), len(tris), _ptr(mtls), len(mtls),
                                               ctypes.cast(tex_arr, ctypes.c_void_p), len(keep)), "mtb_scene_upload")

    def scene_info(self) -> dict:
        s = np.zeros((), SUMMARY_DTYPE)
        self._check(self._lib.mtb_scene_info(self._ctx, _ptr(s)), "mtb_scene_info")
        return {k: (s[k].tolist()) for k in SUMMARY_DTYPE.names}

    def scene_arrays(self):
        info = self.scene_info()
        tris = np.zeros(info["n_triangles"], TRI_DTYPE)
        mtls = np.zeros(info["n_materials"], MTL_DTYPE)
        self._check(self._lib.mtb_scene_read(self._ctx, _ptr(tris), _ptr(mtls)), "mtb_scene_read")
        return tris, mtls

    def triangle_nodes(self):
        n = self.scene_info()["n_triangles"]
        box = np.zeros((n, 6))
        depth = np.zeros(n, np.int32)
        self._check(self._lib.mtb_scene_triangle_nodes(self._ctx, _ptr(box), _ptr(depth)), "mtb_scene_triangle_nodes")
        return box, depth

    def LoadMtl(self, path: str) -> bool:
        """MtlFileReader::ReadMtlFile (objreader.cc:472-549): materials and their map_Ka textures only."""
        return self._lib.mtb_load_mtl(self._ctx, os.fsencode(path)) == 0

    def texture_name(self, index: int) -> str:
        name = self._lib.mtb_scene_texture_name(self._ctx, index)
        return name.decode() if name is not None else ""

    def texture(self, index: int) -> np.ndarray:
        """The decoded RGBA32 texels of texture `index` as the loader keeps them: uint8 [height, width, 4]."""
        t = _TextureStruct()
        self._check(self._lib.mtb_scene_texture(self._ctx, index, ctypes.byref(t)), "mtb_scene_texture")
        n = t.width * t.height * 4
        buf = (ctypes.c_uint8 * n).from_address(t.rgba)
        return np.frombuffer(buf, np.uint8).reshape(t.height, t.width, 4).copy()

    def scene_bvh(self):
        """mtb_scene_bvh: (nodes as a structured array, depth, leaf_order = insertion index per leaf position)."""
        n = ctypes.c_int64(0)
        depth = ctypes.c_int32(0)
        self._check(self._lib.mtb_scene_bvh(self._ctx, ctypes.byref(n), ctypes.byref(depth), None, None), "mtb_scene_bvh")
        nodes = np.zeros(n.value, BVH2_DTYPE)
        order = np.zeros(self.scene_info()["n_scene_refs"] if n.value else 0, np.int32)
        self._check(self._lib.mtb_scene_bvh(self._ctx, None, None, _ptr(nodes), _ptr(order)), "mtb_scene_bvh")
        return nodes, depth.value, order

    def _push_lights(self):
        arr = _lights_array(self._scene.lights)
        self._check(self._lib.mtb_set_lights(self._ctx, _ptr(arr), len(arr)), "mtb_set_lights")

    def render_chunk(self, camera, image_w, image_h, chunk_x, chunk_y, chunk_w, chunk_h, debug=False, taps=False,
                     out: Optional[np.ndarray] = None, _raise=True):
        """mtb_render_chunk with host buffers; returns dict(rgb[, debug, sig_hits, sig_shadow, n_rays], stats)."""
        if not isinstance(camera, Camera):
            camera = Camera.from_tuple(camera)
        self._push_lights()
        rgb = out if out is not None else np.zeros((chunk_h, chunk_w, 3), np.uint8)
        dbg = np.zeros((chunk_h, chunk_w), DEBUG_DTYPE) if debug else None
        res = {}
        tap_ptr = None
        if taps:
            res["sig_hits"] = np.zeros((chunk_h, chunk_w), np.uint64)
            res["sig_shadow"] = np.zeros((chunk_h, chunk_w), np.uint64)
            res["n_rays"] = np.zeros((chunk_h, chunk_w), np.uint32)
            tap_struct = _TapsStruct(res["sig_hits"].ctypes.data, res["sig_shadow"].ctypes.data, res["n_rays"].ctypes.data)
            tap_ptr = ctypes.cast(ctypes.pointer(tap_struct), ctypes.c_void_p)
        stats = np.zeros((), STATS_DTYPE)
        rc = self._lib.mtb_render_chunk(self._ctx, _ptr(camera.as_array()), image_w, image_h, chunk_x, chunk_y, chunk_w,
                                        chunk_h, self.max_depth, _ptr(rgb), _ptr(dbg), tap_ptr, _ptr(stats))
        if rc != MTB_OK:
            if _raise:
                self._check(rc, "mtb_render_chunk")
            return None
        res["rgb"] = rgb
        if debug:
            res["debug"] = dbg
            res["line_no"] = dbg["line_no"]
            res["points"] = dbg["point"]
        res["stats"] = {k: stats[k].item() for k in STATS_DTYPE.names}
        self.last_stats = res["stats"]
        return res

    def render_batch(self, cameras, width: int, height: int, lights=None, out: Optional[np.ndarray] = None, samples_per_axis: int = 1):
        """mtb_render_batch: len(cameras) whole frames in one launch per device, at depth self.max_depth.

        lights: None (every view uses GetScene().lights) or one list of Light per view, all of the same length.
        samples_per_axis: 1, 2, 4 or 8.  s > 1 renders anti-aliased views through mtb_render_batch_ss: each output pixel
        is the rounded mean of the s x s pixels of the same view rendered at (s*width) x (s*height).
        Returns dict(rgb=uint8[n, height, width, 3], stats) with the stats summed over the views (those of the
        s*width x s*height samples)."""
        ss = samples_per_axis
        if isinstance(ss, bool) or not isinstance(ss, (int, np.integer)) or ss not in (1, 2, 4, 8):
            raise MythTracerError("render_batch: samples_per_axis must be 1, 2, 4 or 8 (got %r)" % (ss,))
        ss = int(ss)
        cams = [c if isinstance(c, Camera) else Camera.from_tuple(c) for c in cameras]
        if not cams:
            raise MythTracerError("render_batch: no cameras")
        cam_arr = np.zeros(len(cams), CAMERA_DTYPE)
        for i, c in enumerate(cams):
            cam_arr[i] = c.as_array()
        light_arr, n_lights = None, 0
        if lights is None:
            self._push_lights()
        else:
            lights = list(lights)
            if len(lights) != len(cams):
                raise MythTracerError("render_batch: %d light sets for %d cameras (one per view)" % (len(lights), len(cams)))
            sizes = {len(ls) for ls in lights}
            if len(sizes) != 1:
                raise MythTracerError("render_batch: every view needs the same number of lights (got %s)" % sorted(sizes))
            n_lights = sizes.pop()
            # (n_lights = 0 still passes a non-NULL array: no lights at all, not "the scene's lights")
            light_arr = _lights_array([l for ls in lights for l in ls]) if n_lights else np.zeros(1, LIGHT_DTYPE)
        shape = (len(cams), height, width, 3)
        if out is None:
            rgb = np.zeros(shape, np.uint8)
        else:
            if out.shape != shape or out.dtype != np.uint8 or not out.flags["C_CONTIGUOUS"]:
                raise MythTracerError("render_batch: out must be a C-contiguous uint8 array of shape %s" % (shape,))
            rgb = out
        stats = np.zeros((), STATS_DTYPE)
        if ss == 1:
            self._check(self._lib.mtb_render_batch(self._ctx, _ptr(cam_arr), len(cams), _ptr(light_arr), n_lights, width, height,
                                                   self.max_depth, _ptr(rgb), _ptr(stats)), "mtb_render_batch")
        else:
            self._check(self._lib.mtb_render_batch_ss(self._ctx, _ptr(cam_arr), len(cams), _ptr(light_arr), n_lights, width, height,
                                                      ss, self.max_depth, _ptr(rgb), _ptr(stats)), "mtb_render_batch_ss")
        res = {"rgb": rgb, "stats": {k: stats[k].item() for k in STATS_DTYPE.names}}
        self.last_stats = res["stats"]
        return res

    def render_device(self, camera, image_w, image_h, d_rgb_ptr: int, stream: int = 0, chunk=None):
        """mtb_render_chunk_device: asynchronous render into device memory (lights must already be pushed)."""
        if not isinstance(camera, Camera):
            camera = Camera.from_tuple(camera)
        cx, cy, cw, ch = chunk if chunk is not None else (0, 0, image_w, image_h)
        rc = self._lib.mtb_render_chunk_device(self._ctx, _ptr(camera.as_array()), image_w, image_h, cx, cy, cw, ch,
                                               self.max_depth, ctypes.c_void_p(d_rgb_ptr), ctypes.c_void_p(stream), None)
        self._check(rc, "mtb_render_chunk_device")

    def push_lights(self):
        self._push_lights()

    def load_timing(self) -> dict:
        """Stages of the last scene load in milliseconds (mtb_load_timing)."""
        out = np.zeros(8)
        self._check(self._lib.mtb_load_timing(self._ctx, _ptr(out)), "mtb_load_timing")
        return {"parse_ms": out[0], "octree_ms": out[1], "flatten_ms": out[2], "scene_bvh_host_ms": out[3],
                "scene_bvh_device_ms": out[4], "upload_ms": out[5], "scene_bvh_on_device": bool(out[6]),
                "scene_bvh_host_thread_ms": out[7]}

    def wait(self):
        """mtb_wait: everything queued on the context's devices has finished."""
        self._check(self._lib.mtb_wait(self._ctx), "mtb_wait")

    # -- frames shared between processes (one process per GPU; include/mythtracer_b200.h) --
    def frame_create(self, n_bytes: int):
        """-> (device pointer, 64-byte handle other processes pass to frame_open)."""
        ptr = ctypes.c_void_p()
        handle = (ctypes.c_ubyte * FRAME_HANDLE_BYTES)()
        self._check(self._lib.mtb_frame_create(self._ctx, n_bytes, ctypes.byref(ptr), handle), "mtb_frame_create")
        return int(ptr.value), bytes(handle)

    def frame_open(self, handle: bytes) -> int:
        ptr = ctypes.c_void_p()
        buf = (ctypes.c_ubyte * FRAME_HANDLE_BYTES).from_buffer_copy(bytes(handle))
        self._check(self._lib.mtb_frame_open(self._ctx, buf, ctypes.byref(ptr)), "mtb_frame_open")
        return int(ptr.value)

    def frame_release(self, ptr: int):
        self._check(self._lib.mtb_frame_release(self._ctx, ctypes.c_void_p(ptr)), "mtb_frame_release")

    def frame_read(self, ptr: int, n_bytes: int, offset: int = 0, out: Optional[np.ndarray] = None) -> np.ndarray:
        """Copies n_bytes of a frame to the host (waits for the context's queued work first)."""
        if out is None:
            out = np.zeros(n_bytes, np.uint8)
        assert out.dtype == np.uint8 and out.flags["C_CONTIGUOUS"] and out.size >= n_bytes
        self._check(self._lib.mtb_frame_read(self._ctx, ctypes.c_void_p(ptr), offset, n_bytes, _ptr(out)), "mtb_frame_read")
        return out

    def pipeline_in_use(self):
        """('mega' | 'wavefront' | 'hybrid' | 'queue' | 'measuring', mega_ms, queue_ms) on device 0."""
        a, b = ctypes.c_float(0), ctypes.c_float(0)
        rc = self._lib.mtb_pipeline_in_use(self._ctx, ctypes.cast(ctypes.byref(a), ctypes.c_void_p),
                                           ctypes.cast(ctypes.byref(b), ctypes.c_void_p))
        return {0: "mega", 1: "wavefront", 2: "hybrid", 3: "queue"}.get(rc, "measuring"), a.value, b.value

    def hybrid_share(self) -> float:
        return float(self._lib.mtb_hybrid_share(self._ctx))

    def launch_count(self) -> int:
        return int(self._lib.mtb_launch_count(self._ctx))

    def read_counters(self) -> dict:
        stats = np.zeros((), STATS_DTYPE)
        self._check(self._lib.mtb_read_counters(self._ctx, _ptr(stats)), "mtb_read_counters")
        return {k: stats[k].item() for k in STATS_DTYPE.names}

    def intersect_rays(self, origins, directions, want_stats=False):
        o = np.ascontiguousarray(origins, np.float64).reshape(-1, 3)
        d = np.ascontiguousarray(directions, np.float64).reshape(-1, 3)
        n = o.shape[0]
        tri = np.full(n, -1, np.int32)
        t = np.zeros(n)
        p = np.zeros((n, 3))
        stats = np.zeros((), STATS_DTYPE)
        self._check(self._lib.mtb_intersect_rays(self._ctx, n, _ptr(o), _ptr(d), _ptr(tri), _ptr(t), _ptr(p), _ptr(stats)),
                    "mtb_intersect_rays")
        res = dict(tri=tri, t=t, point=p)
        if want_stats:
            res["stats"] = {k: stats[k].item() for k in STATS_DTYPE.names}
        return res
