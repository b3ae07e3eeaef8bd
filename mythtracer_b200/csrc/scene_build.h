// Host-side scene preparation: reference-exact octree + flattened, cache-line-aligned device records.
//
// Replaces OctTree::AddPrimitive / Finalize / Node::AttemptSplit (reference octtree.cc:8-24,46-135),
// Triangle::CacheAABB (primitive_triangle.cc:18-24) and the AoS `Triangle` / `Node` objects
// (primitive_triangle.h:26-29, octtree.h:47-52) with flat arrays that are uploaded to HBM as they are.
#pragma once
#include <stdint.h>

#include <string>
#include <vector>

#include "mythtracer_b200.h"

namespace mtb {

// Threaded (stackless) BVH over one long node list, records in depth-first order: on a box hit go to
// the next record, on a miss jump to `skip`.  A record is a CONSERVATIVE cull only: its FP32 box is the
// union of the exact FP64 triangle AABBs below it, rounded outwards, and every triangle it lets through is
// still decided by the exact FP64 reference tests.  32 bytes: four records per 128-byte line.
struct alignas(32) BvhRec {
  float box[6];    // lo.xyz rounded down, hi.xyz rounded up
  int32_t skip;
  uint32_t leaf;   // leaf: (first_slot << 3) | count (count 1..kBvhLeafSize); inner record: 0
};
static_assert(sizeof(BvhRec) == 32, "BvhRec must be a quarter of a cache line");

// Scene BVH of the certified fast traversal (device_core.cuh, TraceFast): one binary BVH over ALL triangles, a
// node holds the boxes of its two children (FP32, grown by SceneBvhBuilder::pad = 2^-16 R and rounded outwards) = 64 bytes,
// half a line, four 128-bit loads.  Measured alternatives that did not pay (same bytes, DESIGN.md section 5): the
// tree collapsed to four children per node (128-byte nodes, commit e83e983) and four-wide nodes with 8-bit
// quantised boxes (64 bytes for four children, commit 5e4af88).
// Like BvhRec it is a CONSERVATIVE cull only: the triangles of a leaf are decided by the exact FP64 reference tests.
struct alignas(64) Bvh2Node {
  float lbox[6];   // left child: lo.xyz rounded down, hi.xyz rounded up
  float rbox[6];   // right child
  int32_t left;    // >= 0: inner node index; < 0: leaf, ~left = (first_gslot << 3) | count (count 0..7)
  int32_t right;
  int32_t pad_[2];
};
static_assert(sizeof(Bvh2Node) == 64, "Bvh2Node must be half a cache line");

// One octree node = one 128-byte line.  The 8 children of a node are contiguous (first_child .. +7) and
// their boxes are exactly {lo,c} / {c,hi} per axis (octtree.cc:61-100), so a node carries the three
// planes per axis once instead of eight child boxes.
struct alignas(128) NodeRec {
  double planes[9];     // lo.xyz, c.xyz (centre, octtree.cc:46-50), hi.xyz
  uint32_t child_mask;  // bit k: the subtree of child k holds at least one triangle      (offset 72)
  int32_t bvh_end;      // one past the last list-BVH record of this list
  int32_t first_child;  // -1: never split (octtree.cc:53-55)                             (offset 80, int4)
  int32_t list_first;   // first slot of this node's own primitive list
  int32_t list_count;
  int32_t bvh_root;     // first list-BVH record of this list, -1: scan the list linearly
  BvhRec root_rec;      // copy of bvh[bvh_root]: the first box test of a visit needs no second dependent load
};
static_assert(sizeof(NodeRec) == 128, "NodeRec must be one cache line");

// One triangle as the traversal sees it (exact FP64 AABB + vertices) = one 128-byte line.  Slots of one
// node list are contiguous; inside a list they are in list-BVH leaf order (or list order without a BVH).
struct alignas(128) SlotRec {
  double box[6];   // cached_aabb: lo.xyz, hi.xyz
  double vert[9];
  int32_t tri;     // insertion index (decides ties: later in the reference's list order wins)
  int32_t canon;   // slot index in FlatScene::slots / ::shade (identity there; the gslots copies point back)
};
static_assert(sizeof(SlotRec) == 128, "SlotRec must be one cache line");

// Shading attributes of the triangle in the same slot = one 128-byte line.
struct alignas(128) ShadeRec {
  double normal[9];
  double uv[6];     // u,v of uvw[3] (w is never read downstream: mythtracer.cc:61-62)
  int32_t material;
  int32_t line_no;
};
static_assert(sizeof(ShadeRec) == 128, "ShadeRec must be one cache line");

struct FlatScene {
  std::vector<NodeRec> nodes;
  std::vector<SlotRec> slots;
  std::vector<ShadeRec> shade;
  std::vector<BvhRec> bvh;
  std::vector<int32_t> list_order;  // list_order[list_first + k] = slot of the k-th entry in reference order
  std::vector<int32_t> slot_node;   // octree node whose own list holds the slot (TraceFast's degenerate-passage check)
  std::vector<Bvh2Node> gnodes;     // scene BVH, node 0 = root (empty: no fast traversal)
  std::vector<SlotRec> gslots;      // copies of `slots` in scene-BVH leaf order: one per REFERENCE (a triangle much larger
                                    // than the scene's grain is referenced from several leaves, see SplitTriangle)
  int64_t n_split_refs = 0;         // references - triangles
  // What a DEVICE-side build of the scene BVH needs (device_build.cu): the exact FP64 box of every reference
  // (6 doubles each), the canonical slot of the triangle behind it, and the padding of the stored boxes.
  std::vector<double> ref_box;
  std::vector<int32_t> ref_slot;
  double bvh_pad = 0.0;
  // host stages of the last build, milliseconds (time to first frame, SURVEY.md section 8 f1)
  // (the scene BVH's tree is built on its own thread WHILE the octree is split and flattened: ms_scene_bvh is what was
  // left to wait for afterwards plus the leaf-record gather, ms_scene_bvh_thread the build itself, ms_total the wall
  // time of the whole host build)
  double ms_octree = 0.0, ms_flatten = 0.0, ms_scene_bvh = 0.0, ms_scene_bvh_thread = 0.0, ms_total = 0.0;
  int32_t gbvh_depth = 0;
  int32_t depth = 0;
  int64_t root_list = 0, biggest_list = 0, interior = 0;
  double aabb[6] = {0, 0, 0, 0, 0, 0};
  double max_abs_coord = 0.0;  // largest |coordinate| of the scene box (bounds the FP32 cull error)
  double max_tri_extent = 0.0; // largest extent of a triangle box along an axis
};

#ifndef MTB_BVH_LEAF
#define MTB_BVH_LEAF 2
#endif
#ifndef MTB_BVH_MIN_LIST
#define MTB_BVH_MIN_LIST 3
#endif
#ifndef MTB_SCENE_BVH_LEAF
#define MTB_SCENE_BVH_LEAF 2
#endif
constexpr int kSceneBvhLeafSize = MTB_SCENE_BVH_LEAF;  // <= 7
constexpr int kSceneBvhMaxDepth = 88;                   // deeper trees (never seen) disable the fast traversal
constexpr int kBvhLeafSize = MTB_BVH_LEAF;      // <= 7 (3-bit count in BvhRec::leaf)
constexpr int kBvhMinList = MTB_BVH_MIN_LIST;  // shorter lists are scanned linearly
// measured on B200, C3 frame (megakernel / wavefront ms): leaf 4 min 12: 39.4 / 46.5; leaf 2 min 6: 36.5 / 42.7;
// leaf 2 min 3: 35.5 / 41.8; leaf 3 min 4: 35.6 / 42.0; leaf 1 min 2: 37.9 / 44.9; leaf 6 min 16: 43.7 / 51.4

// Returns MTB_OK or an error code with text in *err.
// scene_bvh: kSceneBvhNone, kSceneBvhHost (binned SAH on the host threads: gnodes / gslots are filled) or kSceneBvhRefs
// (only the references are prepared; the tree is built on the device).
enum SceneBvhMode { kSceneBvhNone = 0, kSceneBvhHost = 1, kSceneBvhRefs = 2 };
int BuildFlatScene(const mtb_triangle *tris, int64_t n, bool use_list_bvh, SceneBvhMode scene_bvh, FlatScene *out,
                   std::string *err);

// Camera::GetSensor / Sensor::Reset (camera.cc:17-63): out9 = start_point, delta_scanline, delta_pixel.
void ComputeSensor(const mtb_camera &cam, int image_w, int image_h, double out9[9]);
// The panorama basis of a camera (mtb_render_batch_pano): aim (ComputeSensor's rotation) applied to (0, 0, 1),
// (-1, 0, 0) and (0, 1, 0).  right points along the pinhole sensor's delta_pixel and up against its delta_scanline.
void ComputePanoramaBasis(const mtb_camera &cam, double forward[3], double right[3], double up[3]);

// ObjFileReader::ReadObjFile + MtlFileReader::ReadMtlFile (objreader.cc:201-274,472-549) + own decoders
// for Texture::LoadFromFile (texture.cc:60-109; SDL2_image is not available offline).
struct LoadedTexture {
  int32_t width = 0, height = 0;
  std::vector<uint8_t> rgba;
};
struct LoadedScene {
  std::vector<mtb_triangle> triangles;
  std::vector<mtb_material> materials;
  std::vector<std::string> material_names;
  std::vector<LoadedTexture> textures;
  std::vector<std::string> texture_names;
};
// Texture::LoadFromFile's decoding step (texture.cc:60-99) without SDL2_image: PPM, PNG, BMP, TGA -> RGBA32
// (image_decode.cc).
bool DecodeImageFile(const std::string &path, LoadedTexture *tex);
bool LoadObjFile(const char *path, LoadedScene *scene, std::string *err);
bool LoadMtlFile(const char *path, LoadedScene *scene, std::string *err);

}  // namespace mtb
