"""mythtracer_b200: a B200-native (sm_100a) replacement for MythTracer's per-pixel ray-casting hot path.

The product is libmythtracer_b200.so (hand-written CUDA kernels behind the C ABI of
include/mythtracer_b200.h); this package is the Python mirror of the reference's renderer API on top of it
plus the seeded synthetic-scene generator.  There is no CPU fallback.
"""
from .api import (Camera, Light, MythTracer, MythTracerError, OctTree, Scene, WorkChunk, load_library, panorama_rays,
                  MAX_RECURSION_LEVEL, MTB_FLAG_COUNT_WORK, MTB_FLAG_MEGAKERNEL, MTB_FLAG_NO_LIST_BVH, MTB_FLAG_WAVEFRONT,
                  MTB_FLAG_RAY_SORT, MTB_FLAG_NO_TILE_ORDER, MTB_FLAG_PERSISTENT, MTB_FLAG_EXACT_OCTREE, MTB_FLAG_PACKING, MTB_FLAG_WARP_SYNC, MTB_FLAG_RESUME, MTB_FLAG_HYBRID, MTB_FLAG_DEVICE_BVH, MTB_FLAG_QUEUE, MTB_FLAG_PAIR_RAYS, MTB_FLAG_CHAIN_RAYS)

__all__ = ["Camera", "Light", "MythTracer", "MythTracerError", "OctTree", "Scene", "WorkChunk", "load_library", "panorama_rays",
           "MAX_RECURSION_LEVEL", "MTB_FLAG_COUNT_WORK", "MTB_FLAG_MEGAKERNEL", "MTB_FLAG_NO_LIST_BVH", "MTB_FLAG_WAVEFRONT",
           "MTB_FLAG_RAY_SORT", "MTB_FLAG_NO_TILE_ORDER", "MTB_FLAG_PERSISTENT", "MTB_FLAG_EXACT_OCTREE", "MTB_FLAG_PACKING", "MTB_FLAG_WARP_SYNC", "MTB_FLAG_RESUME", "MTB_FLAG_HYBRID", "MTB_FLAG_DEVICE_BVH", "MTB_FLAG_QUEUE", "MTB_FLAG_PAIR_RAYS", "MTB_FLAG_CHAIN_RAYS"]
