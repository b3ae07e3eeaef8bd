// Device core shared by the megakernel (megakernel.cu) and the wavefront pipeline (wavefront.cu):
// hand-written sm_100a code for MythTracer's ray-casting path.
//
// Everything that DECIDES a result (which triangle is hit, shadowed or not, the hit point) is computed in
// FP64 with the reference's operation order and without FMA contraction (build with --fmad=false; the
// reference binary contains no FMA, SURVEY.md fact 4), so hit ids, shadow decisions and colours are
// reproduced bit for bit except for pow() (mythtracer.cc:174; CUDA's and glibc's differ by <= 2 ulp).
//
// Reference functions replaced here:
//   OctTree::IntersectRay                      octtree.cc:26-40        -> Trace: TraceFast / TraceRegular / TraceLiteral
//   Node::NodeIntersectRay                     octtree.cc:138-167      -> the slab tests inside them
//   Node::PrimitiveIntersectRay                octtree.cc:169-257      -> the explicit frame stack
//   Triangle::IntersectRay                     primitive_triangle.cc:81-143 -> TestSlot*
//   Triangle::GetNormal / GetUVW               primitive_triangle.cc:27-79  -> Barycentric
//   Texture::GetColorAt                        texture.cc:11-58        -> SampleTexture
//   Sensor::GetRay                             camera.cc:65-69         -> PixelDirection
//   MythTracer::TraceRayWorker + shadow walk   mythtracer.cc:13-228    -> the state machine of RenderMega
//   MythTracer::V3DtoRGB                       mythtracer.cc:235-241   -> Quantize
//   the OpenMP row loop                        mythtracer.cc:292-305   -> the CUDA grid (8x8 pixel tiles)
//
// Three traversals exist, chosen per ray in Trace().  Rays whose direction has a zero / non-finite component
// ("irregular": the NaN producing cases of SURVEY.md fact 9) take TraceLiteral, a literal restatement of the
// octree recursion including std::min/max NaN behaviour and libstdc++'s insertion sort.  All other rays first
// take TraceFast, a certified closest-hit search over one BVH of all triangles (conservative FP32 boxes, the
// exact FP64 reference tests at the leaves, a forward error bound on every accepted hit); if it cannot certify
// that its answer is the recursion's - two hits closer together than their error bounds - the ray is decided by
// TraceRegular, the octree recursion itself (explicit frame stack, reference order), which may use any
// evaluation order that yields the same VALUES when no NaN can occur: sign-selected near/far planes instead of
// pairwise min/max, the three shared planes of the eight children, skipping empty subtrees, and a conservative
// threaded BVH over long node lists whose candidates are decided by the exact reference tests with the
// reference's tie rule (later list entry wins on equal t).  DESIGN.md section 4 has the argument.
#pragma once
#include <math_constants.h>

#include "device_scene.h"

namespace mtb {
namespace {

constexpr int kMaxTreeStack = MTB_MAX_TREE_DEPTH + 2;
constexpr int kMaxRayStack = MTB_MAX_RAY_DEPTH + 2;
constexpr int kTile = 8;            // 8x8 pixel tiles, one per 64-thread block; a warp covers 8x4 pixels
constexpr int kBlockThreads = 64;

// ---------------------------------------------------------------------------------------------------
// math3d.h:31-136 with the operand order spelled out
// ---------------------------------------------------------------------------------------------------
struct D3 {
  double x, y, z;
};
__device__ __forceinline__ D3 Mk(double x, double y, double z) { return D3{x, y, z}; }
__device__ __forceinline__ D3 Add(const D3 &a, const D3 &b) { return Mk(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ D3 Sub(const D3 &a, const D3 &b) { return Mk(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ D3 Neg(const D3 &a) { return Mk(-a.x, -a.y, -a.z); }
__device__ __forceinline__ D3 MulV(const D3 &a, const D3 &b) { return Mk(a.x * b.x, a.y * b.y, a.z * b.z); }
__device__ __forceinline__ D3 MulS(const D3 &a, double s) { return Mk(a.x * s, a.y * s, a.z * s); }
__device__ __forceinline__ D3 DivS(const D3 &a, double s) { return Mk(a.x / s, a.y / s, a.z / s); }
__device__ __forceinline__ double Dot(const D3 &a, const D3 &b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
// this.Cross(a), math3d.h:120-126
__device__ __forceinline__ D3 Cross(const D3 &t, const D3 &a) {
  return Mk(t.y * a.z - t.z * a.y, t.z * a.x - t.x * a.z, t.x * a.y - t.y * a.x);
}
__device__ __forceinline__ double SqrLen(const D3 &a) { return a.x * a.x + a.y * a.y + a.z * a.z; }
__device__ __forceinline__ double SqrDist(const D3 &t, const D3 &a) {
  const double dx = a.x - t.x, dy = a.y - t.y, dz = a.z - t.z;
  return dx * dx + dy * dy + dz * dz;
}
__device__ __forceinline__ double Dist(const D3 &t, const D3 &a) { return sqrt(SqrDist(t, a)); }
__device__ __forceinline__ D3 Normalized(const D3 &a) {
  const double l = sqrt(SqrLen(a));
  return Mk(a.x / l, a.y / l, a.z / l);
}
__device__ __forceinline__ D3 Load3(const double *p) { return Mk(p[0], p[1], p[2]); }
__device__ __forceinline__ void Store3(double *p, const D3 &v) {
  p[0] = v.x;
  p[1] = v.y;
  p[2] = v.z;
}

// std::min / std::max of libstdc++ (NaN behaviour is contract, SURVEY.md appendix A.7)
__device__ __forceinline__ double SMin(double a, double b) { return (b < a) ? b : a; }
__device__ __forceinline__ double SMax(double a, double b) { return (a < b) ? b : a; }
__device__ __forceinline__ double SMin3(double a, double b, double c) {
  double r = a;
  if (b < r) r = b;
  if (c < r) r = c;
  return r;
}
__device__ __forceinline__ double SMax3(double a, double b, double c) {
  double r = a;
  if (r < b) r = b;
  if (r < c) r = c;
  return r;
}

template <bool DBG>
__device__ __forceinline__ void Count(unsigned long long *cnt, int which, unsigned long long n = 1) {
  if (DBG) cnt[which] += n;
}

// 128-bit read-only loads of the 16-byte aligned records
__device__ __forceinline__ double2 Ld2(const double *p) { return __ldg(reinterpret_cast<const double2 *>(p)); }

struct Ray {
  D3 o, d, inv;
  bool sx, sy, sz;  // inv component negative (regular rays only)
  // FP32 conservative cull of list-BVH boxes (CullBox); valid when cull32
  bool cull32;
  float ox, oy, oz, ix, iy, iz, px, py, pz;  // origin, inverse direction, absolute slack per axis (in t)
};

// ---------------------------------------------------------------------------------------------------
// Literal slab test: Node::NodeIntersectRay (octtree.cc:138-167) == the triangle pre-test
// (primitive_triangle.cc:85-108).  Used for irregular rays.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool SlabLiteral(const double lo[3], const double hi[3], const Ray &r, double *tmin_out) {
  const double t1 = (lo[0] - r.o.x) * r.inv.x;
  const double t2 = (hi[0] - r.o.x) * r.inv.x;
  const double t3 = (lo[1] - r.o.y) * r.inv.y;
  const double t4 = (hi[1] - r.o.y) * r.inv.y;
  const double t5 = (lo[2] - r.o.z) * r.inv.z;
  const double t6 = (hi[2] - r.o.z) * r.inv.z;
  const double tmax = SMin3(SMax(t1, t2), SMax(t3, t4), SMax(t5, t6));
  if (tmax < 0.0) return false;
  const double tmin = SMax3(SMin(t1, t2), SMin(t3, t4), SMin(t5, t6));
  if (tmin > tmax) return false;
  *tmin_out = tmin;
  return true;
}

// Regular rays (finite non-zero inverse direction, finite origin): no NaN can arise, and since
// lo <= hi and FP64 subtraction / multiplication are monotonic, min(t_lo, t_hi) is t of the plane the
// direction sign selects.  Same values as SlabLiteral, fewer FP64 compares.
__device__ __forceinline__ bool SlabRegular(double lox, double loy, double loz, double hix, double hiy, double hiz,
                                            const Ray &r, double *tmin_out) {
  const double nx = ((r.sx ? hix : lox) - r.o.x) * r.inv.x;
  const double fx = ((r.sx ? lox : hix) - r.o.x) * r.inv.x;
  const double ny = ((r.sy ? hiy : loy) - r.o.y) * r.inv.y;
  const double fy = ((r.sy ? loy : hiy) - r.o.y) * r.inv.y;
  const double nz = ((r.sz ? hiz : loz) - r.o.z) * r.inv.z;
  const double fz = ((r.sz ? loz : hiz) - r.o.z) * r.inv.z;
  const double tmax = SMin3(fx, fy, fz);
  if (tmax < 0.0) return false;
  const double tmin = SMax3(nx, ny, nz);
  if (tmin > tmax) return false;
  *tmin_out = tmin;
  return true;
}

// Conservative FP32 cull of a list-BVH box: returns true whenever the exact FP64 pre-test
// (primitive_triangle.cc:85-108, == SlabRegular) passes for ANY triangle box inside the record's box.
// The record's float box contains the FP64 union box (rounded outwards), which only moves the near plane
// nearer and the far plane farther.  For every plane, with R = cull_radius >= |box coordinate| and a ray
// with |origin| <= 8R, the FP32 value differs from the FP64 one by at most
//     2^-24 * 8R * |inv|      (origin rounded to float)            -> absolute slack p = 2^-20 * R * |inv|
//   + ~4 * 2^-24 * |t|        (inverse direction, subtraction, fma) -> relative slack 2^-21
// so near planes are pushed down and far planes up by (p + 2^-21 |t|); both margins are >= 2x the bound.
// min/max over lower / upper bounds stay lower / upper bounds, hence the test can only over-accept.
__device__ __forceinline__ bool CullBox32(float lox, float loy, float loz, float hix, float hiy, float hiz, const Ray &r) {
  const float kRel = 4.76837158203125e-07f;  // 2^-21
  float nx = __fmaf_rn((r.sx ? hix : lox) - r.ox, r.ix, -r.px);
  float fx = __fmaf_rn((r.sx ? lox : hix) - r.ox, r.ix, r.px);
  float ny = __fmaf_rn((r.sy ? hiy : loy) - r.oy, r.iy, -r.py);
  float fy = __fmaf_rn((r.sy ? loy : hiy) - r.oy, r.iy, r.py);
  float nz = __fmaf_rn((r.sz ? hiz : loz) - r.oz, r.iz, -r.pz);
  float fz = __fmaf_rn((r.sz ? loz : hiz) - r.oz, r.iz, r.pz);
  nx = __fmaf_rn(-kRel, fabsf(nx), nx);
  ny = __fmaf_rn(-kRel, fabsf(ny), ny);
  nz = __fmaf_rn(-kRel, fabsf(nz), nz);
  fx = __fmaf_rn(kRel, fabsf(fx), fx);
  fy = __fmaf_rn(kRel, fabsf(fy), fy);
  fz = __fmaf_rn(kRel, fabsf(fz), fz);
  const float tmax = fminf(fminf(fx, fy), fz);
  const float tmin = fmaxf(fmaxf(nx, ny), nz);
  return !(tmax < 0.0f) && !(tmin > tmax);
}

// The same cull for rays outside the FP32 error model (far-away origin, extreme direction): the float box
// is evaluated with the exact FP64 slab arithmetic; box32 contains box64, so this over-accepts too.
__device__ __forceinline__ bool CullBox64(float lox, float loy, float loz, float hix, float hiy, float hiz, const Ray &r) {
  double unused;
  return SlabRegular((double)lox, (double)loy, (double)loz, (double)hix, (double)hiy, (double)hiz, r, &unused);
}

// Moller-Trumbore exactly as primitive_triangle.cc:111-142.
__device__ __forceinline__ bool MollerTrumbore(const double *vert, const Ray &r, double *t_out) {
  const double2 a = Ld2(vert + 0), b = Ld2(vert + 2), c = Ld2(vert + 4), d = Ld2(vert + 6);
  const double v22 = __ldg(vert + 8);
  const D3 v0 = Mk(a.x, a.y, b.x), v1 = Mk(b.y, c.x, c.y), v2 = Mk(d.x, d.y, v22);
  const D3 e1 = Sub(v1, v0);
  const D3 e2 = Sub(v2, v0);
  const D3 pvec = Cross(r.d, e2);
  const double det = Dot(e1, pvec);
  if (det >= -0.00000001 && det < 0.00000001) return false;
  const double inv_det = 1.0 / det;
  const D3 tvec = Sub(r.o, v0);
  const double u = Dot(tvec, pvec) * inv_det;
  if (u < 0.0 || u > 1.0) return false;
  const D3 qvec = Cross(tvec, e1);
  const double v = Dot(r.d, qvec) * inv_det;
  if (v < 0.0 || u + v > 1.0) return false;
  const double t = Dot(e2, qvec) * inv_det;
  if (t < 0.0) return false;
  *t_out = t;
  return true;
}

// One list entry for a regular ray; candidates arrive in arbitrary order, so the reference's sequential
// "replace unless strictly farther" (octtree.cc:186-195) becomes: nearer wins, on equal t the entry that is
// later in the reference's list (= larger insertion index) wins.
template <bool DBG>
__device__ __forceinline__ void TestSlotRegular(const DeviceScene &sc, int slot, const Ray &r, double *best_t,
                                                int *best_slot, unsigned long long *cnt) {
  const SlotRec *rec = sc.slots + slot;
  const double2 b0 = Ld2(rec->box + 0), b1 = Ld2(rec->box + 2), b2 = Ld2(rec->box + 4);
  Count<DBG>(cnt, kTriAabb);
  double unused;
  if (!SlabRegular(b0.x, b0.y, b1.x, b1.y, b2.x, b2.y, r, &unused)) return;
  Count<DBG>(cnt, kMt);
  double t;
  if (!MollerTrumbore(rec->vert, r, &t)) return;
  Count<DBG>(cnt, kHit);
  if (*best_slot >= 0) {
    if (t > *best_t) return;
    if (t == *best_t && __ldg(&rec->tri) < __ldg(&sc.slots[*best_slot].tri)) return;
  }
  *best_t = t;
  *best_slot = slot;
}

// ---------------------------------------------------------------------------------------------------
// Regular traversal
// ---------------------------------------------------------------------------------------------------
template <bool DBG>
__device__ int TraceRegular(const DeviceScene &sc, const Ray &r, double *t_out, unsigned long long *cnt) {
  int f_child[kMaxTreeStack];
  unsigned f_order[kMaxTreeStack];
  double f_t[kMaxTreeStack];
  int f_slot[kMaxTreeStack];

  {  // the root gate (octtree.cc:34-37)
    const NodeRec *root = sc.nodes;
    double unused;
    Count<DBG>(cnt, kSlab);
    if (!SlabRegular(__ldg(&root->planes[0]), __ldg(&root->planes[1]), __ldg(&root->planes[2]), __ldg(&root->planes[6]),
                     __ldg(&root->planes[7]), __ldg(&root->planes[8]), r, &unused)) {
      return -1;
    }
  }

  int sp = 0;
  int cur = 0;
  // current frame in registers
  double c_t = 0.0;
  int c_slot = -1;
  unsigned c_order = 0;
  int c_child = -1;
  for (;;) {
    // ---- enter node `cur`: own list first (octtree.cc:177-196) ----
    const NodeRec *node = (sc.nodes + cur);
    const int4 info = __ldg(reinterpret_cast<const int4 *>(&node->first_child));  // first_child, list_first, list_count, bvh_root
    const int2 info2 = __ldg(reinterpret_cast<const int2 *>(&node->child_mask));  // child_mask, bvh_end
    Count<DBG>(cnt, kVisit);
    c_t = 0.0;
    c_slot = -1;
    c_order = 0;
    c_child = info.x;
    if (info.w < 0) {
      for (int s = info.y, e = info.y + info.z; s < e; s++) TestSlotRegular<DBG>(sc, s, r, &c_t, &c_slot, cnt);
    } else {
      // Two phases per list ("while-while"): first walk the BVH with the cheap FP32 cull only and park
      // the leaves it lets through, then run the exact FP64 triangle tests of the parked leaves back to
      // back.  Lanes of a warp reach leaves at different iterations; testing triangles inside the walk
      // would make every other lane wait for each of them.
      constexpr int kPend = 6;
      unsigned pend[kPend];
      int n_pend = 0;
      int i = info.w;
      const int end = info2.y;
      const BvhRec *b = &node->root_rec;  // the list's first record travels in the node's own cache line
      while (i < end) {
        const float4 q0 = __ldg(reinterpret_cast<const float4 *>(b->box));      // lo.xyz hi.x
        const float4 q1 = __ldg(reinterpret_cast<const float4 *>(b->box) + 1);  // hi.yz skip leaf
        Count<DBG>(cnt, kBvh);
        const bool pass = r.cull32 ? CullBox32(q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, r)
                                   : CullBox64(q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, r);
        i = pass ? i + 1 : __float_as_int(q1.z);
        b = sc.bvh + i;
        const unsigned leaf = __float_as_uint(q1.w);
        if (pass && leaf != 0u) {
          pend[n_pend++] = leaf;
          if (n_pend == kPend) {
            for (int j = 0; j < kPend; j++) {
              for (int s = (int)(pend[j] >> 3), e = s + (int)(pend[j] & 7u); s < e; s++) TestSlotRegular<DBG>(sc, s, r, &c_t, &c_slot, cnt);
            }
            n_pend = 0;
          }
        }
      }
      for (int j = 0; j < n_pend; j++) {
        for (int s = (int)(pend[j] >> 3), e = s + (int)(pend[j] & 7u); s < e; s++) TestSlotRegular<DBG>(sc, s, r, &c_t, &c_slot, cnt);
      }
    }
    // ---- children that the ray enters, ordered by entry distance (octtree.cc:200-216) ----
    const unsigned mask = (unsigned)info2.x;
    if (info.x >= 0 && mask != 0u) {
      const double2 p0 = __ldg(reinterpret_cast<const double2 *>(node->planes + 0)), p1 = __ldg(reinterpret_cast<const double2 *>(node->planes + 2)),
                    p2 = __ldg(reinterpret_cast<const double2 *>(node->planes + 4)), p3 = __ldg(reinterpret_cast<const double2 *>(node->planes + 6));
      const double hz = __ldg(&node->planes[8]);
      // planes: lo = (p0.x p0.y p1.x), c = (p1.y p2.x p2.y), hi = (p3.x p3.y hz)
      const double tx0 = (p0.x - r.o.x) * r.inv.x, tx1 = (p1.y - r.o.x) * r.inv.x, tx2 = (p3.x - r.o.x) * r.inv.x;
      const double ty0 = (p0.y - r.o.y) * r.inv.y, ty1 = (p2.x - r.o.y) * r.inv.y, ty2 = (p3.y - r.o.y) * r.inv.y;
      const double tz0 = (p1.x - r.o.z) * r.inv.z, tz1 = (p2.y - r.o.z) * r.inv.z, tz2 = (hz - r.o.z) * r.inv.z;
      // near / far per axis for the lower [lo,c] and upper [c,hi] halves
      const double nx[2] = {r.sx ? tx1 : tx0, r.sx ? tx2 : tx1}, fx[2] = {r.sx ? tx0 : tx1, r.sx ? tx1 : tx2};
      const double ny[2] = {r.sy ? ty1 : ty0, r.sy ? ty2 : ty1}, fy[2] = {r.sy ? ty0 : ty1, r.sy ? ty1 : ty2};
      const double nz[2] = {r.sz ? tz1 : tz0, r.sz ? tz2 : tz1}, fz[2] = {r.sz ? tz0 : tz1, r.sz ? tz1 : tz2};
      double key[8];
      unsigned pass = 0;
#pragma unroll
      for (int k = 0; k < 8; k++) {
        const int xh = k & 1, zh = (k >> 1) & 1, yh = (k >> 2) & 1;  // octtree.cc:61-100
        const double tmax = SMin3(fx[xh], fy[yh], fz[zh]);
        const double tmin = SMax3(nx[xh], ny[yh], nz[zh]);
        key[k] = tmin;
        if ((mask >> k) & 1u) {
          Count<DBG>(cnt, kSlab);
          if (!(tmax < 0.0) && !(tmin > tmax)) pass |= 1u << k;
        }
      }
      // stable order by key: child j precedes child k (j < k) iff key[j] <= key[k].  A line pierces at
      // most four octants, usually one or two: those cases skip the general ranking.
      const int n_pass = __popc(pass);
      if (n_pass == 1) {
        c_order = 8u | (unsigned)(__ffs((int)pass) - 1);
      } else if (n_pass == 2) {
        const unsigned k0 = (unsigned)(__ffs((int)pass) - 1), k1 = 31u - (unsigned)__clz((int)pass);
        double a = key[0], b = key[7];
#pragma unroll
        for (int k = 1; k < 7; k++) {
          a = (k0 == (unsigned)k) ? key[k] : a;
          b = (k1 == (unsigned)k) ? key[k] : b;
        }
        a = (k0 == 0u) ? key[0] : a;
        b = (k1 == 7u) ? key[7] : b;
        c_order = (a <= b) ? ((8u | k0) | ((8u | k1) << 4)) : ((8u | k1) | ((8u | k0) << 4));
      } else if (n_pass > 2) {
        unsigned rank[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
        for (int j = 0; j < 8; j++) {
#pragma unroll
          for (int k = j + 1; k < 8; k++) {
            const bool both = ((pass >> j) & (pass >> k) & 1u) != 0u;
            const bool j_first = key[j] <= key[k];
            rank[k] += (both && j_first) ? 1u : 0u;
            rank[j] += (both && !j_first) ? 1u : 0u;
          }
        }
#pragma unroll
        for (int k = 0; k < 8; k++) {
          if ((pass >> k) & 1u) c_order |= (8u | (unsigned)k) << (4u * rank[k]);
        }
      }
    }
    // ---- visit children nearest first; unwind finished frames (octtree.cc:219-256) ----
    for (;;) {
      const unsigned e = c_order & 15u;
      if (e != 0u) {
        c_order >>= 4;
        f_child[sp] = c_child;
        f_order[sp] = c_order;
        f_t[sp] = c_t;
        f_slot[sp] = c_slot;
        sp++;
        cur = c_child + (int)(e & 7u);
        break;  // enter the child
      }
      if (sp == 0) {
        if (c_slot < 0) return -1;
        *t_out = c_t;
        return c_slot;
      }
      // return (c_t, c_slot) to the parent frame
      sp--;
      const double rt = c_t;
      const int rs = c_slot;
      c_child = f_child[sp];
      c_order = f_order[sp];
      c_t = f_t[sp];
      c_slot = f_slot[sp];
      if (rs >= 0 && !(c_slot >= 0 && rt > c_t)) {
        c_t = rt;
        c_slot = rs;
        c_order = 0;  // `break`: nodes were sorted by distance (octtree.cc:244-246)
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// Literal traversal for irregular rays: no shortcut of any kind.
// ---------------------------------------------------------------------------------------------------
template <bool DBG>
__device__ __noinline__ int TraceLiteral(const DeviceScene &sc, const Ray &r, double *t_out, unsigned long long *cnt) {
  int f_node[kMaxTreeStack];
  unsigned f_order[kMaxTreeStack];
  double f_t[kMaxTreeStack];
  int f_slot[kMaxTreeStack];
  Count<DBG>(cnt, kLiteral);
  {
    const NodeRec *root = sc.nodes;
    double unused;
    Count<DBG>(cnt, kSlab);
    if (!SlabLiteral(root->planes, root->planes + 6, r, &unused)) return -1;
  }
  int sp = 0;
  int cur = 0;
  for (;;) {
    const NodeRec *node = sc.nodes + cur;
    Count<DBG>(cnt, kVisit);
    double bt = 0.0;
    int bs = -1;
    for (int k = 0; k < node->list_count; k++) {  // reference list order
      const int slot = sc.list_order[node->list_first + k];
      const SlotRec *rec = sc.slots + slot;
      double unused, t;
      Count<DBG>(cnt, kTriAabb);
      if (!SlabLiteral(rec->box, rec->box + 3, r, &unused)) continue;
      Count<DBG>(cnt, kMt);
      if (!MollerTrumbore(rec->vert, r, &t)) continue;
      Count<DBG>(cnt, kHit);
      if (bs >= 0 && t > bt) continue;
      bt = t;
      bs = slot;
    }
    unsigned order = 0;
    if (node->first_child >= 0) {
      int idx[8];
      double key[8];
      int n = 0;
      for (int k = 0; k < 8; k++) {
        const NodeRec *ch = sc.nodes + node->first_child + k;
        double d;
        Count<DBG>(cnt, kSlab);
        if (!SlabLiteral(ch->planes, ch->planes + 6, r, &d)) continue;
        idx[n] = k;
        key[n] = d;
        n++;
      }
      // libstdc++ __insertion_sort (std::sort on <= 16 elements), comparator a.second < b.second
      for (int i = 1; i < n; i++) {
        const int vi = idx[i];
        const double vk = key[i];
        if (vk < key[0]) {
          for (int j = i; j > 0; j--) {
            idx[j] = idx[j - 1];
            key[j] = key[j - 1];
          }
          idx[0] = vi;
          key[0] = vk;
        } else {
          int j = i;
          while (vk < key[j - 1]) {
            idx[j] = idx[j - 1];
            key[j] = key[j - 1];
            j--;
          }
          idx[j] = vi;
          key[j] = vk;
        }
      }
      for (int i = 0; i < n; i++) order |= (8u | (unsigned)idx[i]) << (4u * i);
    }
    f_node[sp] = cur;
    f_order[sp] = order;
    f_t[sp] = bt;
    f_slot[sp] = bs;
    for (;;) {
      const unsigned e = f_order[sp] & 15u;
      if (e != 0u) {
        f_order[sp] >>= 4;
        cur = sc.nodes[f_node[sp]].first_child + (int)(e & 7u);
        sp++;
        break;
      }
      if (sp == 0) {
        if (f_slot[0] < 0) return -1;
        *t_out = f_t[0];
        return f_slot[0];
      }
      const double rt = f_t[sp];
      const int rs = f_slot[sp];
      sp--;
      if (rs >= 0 && !(f_slot[sp] >= 0 && rt > f_t[sp])) {
        f_t[sp] = rt;
        f_slot[sp] = rs;
        f_order[sp] = 0;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// Certified fast traversal for regular rays.
//
// The octree recursion of the reference returns the closest accepted triangle (SURVEY.md appendix A.7); what
// makes it expensive is the shape of the search, not the answer: every own list of every node on the ray's
// path is examined and nothing is pruned by distance.  TraceFast searches the SAME candidate set - every
// triangle whose exact FP64 reference test (primitive_triangle.cc:81-143) accepts the ray - through one
// binary BVH over all triangles, nearest child first, skipping subtrees that start behind the best hit.  The
// boxes are a conservative FP32 cull (as CullBox32); a triangle is only ever accepted, and its t only ever
// computed, by the exact reference arithmetic, so t, the hit point and everything downstream are the
// reference's bits.
//
// Where the two searches could disagree is which triangle wins when two accepted hits are closer together than
// the rounding error of their t (the reference then decides by list / sibling order).  So every accepted hit
// carries a forward error bound e of its t (MollerTrumboreBound), the search keeps the best hit (t*, e*) and
// lo2 = min (t - e) over all other accepted hits, and
//   * prunes a subtree only if its conservative entry distance exceeds t* + 2 e* + 2^-20 t*,
//   * declares the ray AMBIGUOUS if lo2 <= t* + e* (two hits whose error intervals touch, an exact tie, or an
//     ill-conditioned winner), in which case the caller discards the answer and runs the exact octree recursion.
// Why an unambiguous answer is the reference's: (1) the reference evaluates the winner h* (it only stops early
// behind a sibling that was entered EARLIER, and any accepted hit there has a true distance <= the separating
// plane <= h*'s; with disjoint error intervals its computed t would be smaller than t*: contradiction), (2) every
// comparison the recursion makes between two evaluated hits picks the smaller t, ties aside, (3) a pruned
// triangle's box starts behind t* + 2 e*, so it cannot lie in an earlier sibling either.  Left over, and stated
// in DESIGN.md section 4: an exact tie of two sibling octants' entry distances (a ray through an octree edge in
// computed arithmetic), and a pruned, never evaluated triangle whose own computed t is off by more than the
// pruning margin (Moller-Trumbore determinant within ~1e3 of the reference's rejection threshold 1e-8).
// ---------------------------------------------------------------------------------------------------
constexpr int kFastStack = kSceneBvhMaxDepth + 8;
constexpr int kFastExit = (int)0x80000000;

// Moller-Trumbore exactly as MollerTrumbore() above (same operations, same order -> same bits) plus a forward
// error bound of t against the exact ray-plane parameter: with u = 2^-53 and |x| meaning component-wise
// magnitudes, det carries at most 7u * D, D = |e1| . (|d| x |e2|), the numerator at most 8u * N,
// N = |e2| . (|tvec| x |e1|), and the final quotient 2u |t|; the bound uses 16u, 16u and 8u.
struct TriVerts {
  double2 a, b, c, d;
  double v22;
};
__device__ __forceinline__ bool MollerTrumboreBound(const TriVerts &tv, const Ray &r, double *t_out, double *e_out) {
  const D3 v0 = Mk(tv.a.x, tv.a.y, tv.b.x), v1 = Mk(tv.b.y, tv.c.x, tv.c.y), v2 = Mk(tv.d.x, tv.d.y, tv.v22);
  const D3 e1 = Sub(v1, v0);
  const D3 e2 = Sub(v2, v0);
  const D3 pvec = Cross(r.d, e2);
  const double det = Dot(e1, pvec);
  if (det >= -0.00000001 && det < 0.00000001) return false;
  const D3 tvec = Sub(r.o, v0);
  const double un = Dot(tvec, pvec);
  {
    // Most candidates are far misses (u far outside [0, 1]).  Their rejection by the reference's `u < 0 || u > 1`
    // can be decided without the division: |det| >= 1e-8, so inv_det = fl(1 / det) is a normal number with det's
    // sign and u = fl(un * inv_det) (a) is a non-zero negative number whenever un and det have opposite signs and
    // |un| > 1e-200 (no underflow to -0, which would NOT be < 0), (b) exceeds 1 whenever un / det > 1 + 1e-10
    // (two roundings of 2^-53 cannot bring it back to <= 1).  Anything closer goes through the division below.
    const double us = det > 0.0 ? un : -un;
    if (us < -1e-200 || us > fabs(det) * 1.0000000001) return false;
  }
  const double inv_det = 1.0 / det;
  const double u = un * inv_det;
  if (u < 0.0 || u > 1.0) return false;
  const D3 qvec = Cross(tvec, e1);
  const double v = Dot(r.d, qvec) * inv_det;
  if (v < 0.0 || u + v > 1.0) return false;
  const double t = Dot(e2, qvec) * inv_det;
  if (t < 0.0) return false;
  *t_out = t;
  const D3 ad = Mk(fabs(r.d.x), fabs(r.d.y), fabs(r.d.z)), a1 = Mk(fabs(e1.x), fabs(e1.y), fabs(e1.z)),
           a2 = Mk(fabs(e2.x), fabs(e2.y), fabs(e2.z)), at = Mk(fabs(tvec.x), fabs(tvec.y), fabs(tvec.z));
  const double D = a1.x * (ad.y * a2.z + ad.z * a2.y) + a1.y * (ad.z * a2.x + ad.x * a2.z) + a1.z * (ad.x * a2.y + ad.y * a2.x);
  const double N = a2.x * (at.y * a1.z + at.z * a1.y) + a2.y * (at.z * a1.x + at.x * a1.z) + a2.z * (at.x * a1.y + at.y * a1.x);
  const double e_det = 0x1p-49 * D, e_num = 0x1p-49 * N;
  const double den = fabs(det) - e_det;
  *e_out = den > 0.0 ? (e_num + t * e_det) / den + 0x1p-50 * t : CUDART_INF;
  return true;
}

// What the LEAVES need of a ray and of the search so far: the FP64 ray (the exact tests run in the reference's FP64
// arithmetic) and the best hit with its error bound - twelve doubles per thread that are written once per ray and
// read at every leaf visit.  The node loop runs on FP32 values only (FastRay); keeping the 18 registers of the FP64
// ray and the 6 of the best hit alive across it made the register allocator spill and rematerialise inside the loop
// (3 local loads + 3 F2F + 3 DSETP per node visit under the 64-register cap).
//
// The twelve doubles live in shared memory, laid out [field][thread] (conflict-free 64-bit accesses).  ncu on the
// local-memory form: the leaf reloads were 44 % of the kernel's local-memory bytes, half of them missed L1 (the per-SM
// working set of 1024 threads' local memory is larger than L1) and went to L2 next to the BVH nodes.  The best hit
// (kFmT, kFmE, kFmLo2) is touched by only 0.5 accepted hits per ray, but keeping it in local memory instead, so that
// sixteen 64-thread blocks fit a smaller shared-memory carve-out, measured neutral (DESIGN.md section 5, row "best hit
// (t, e, lo2) in local memory"): L1 capacity is not what the walk waits for.
//
// Fields: o.xyz, d.xyz, inv.xyz, best t, its error bound e, lo2 = min (t - e) over all other accepted hits.
enum FastField { kFmO = 0, kFmD = 3, kFmInv = 6, kFmT = 9, kFmE = 10, kFmLo2 = 11, kFmWords = 12 };
// MTB_FAST_BARRIER: a compiler barrier whose operand is the address of a per-ray local FastMem.  Nothing reads or
// writes the struct (the fields are in shared memory), but dropping the operand changes the code ptxas generates for
// every kernel that traces, so the struct stays as the barrier's anchor.
struct alignas(16) FastMem {
  double w[kFmWords];
};
#define MTB_FAST_BARRIER(m) asm volatile("" : : "l"(m) : "memory")

// Per-thread handles of the fast traversal's scratch memory.
struct FastCtx {
  unsigned ray_base;  // shared-space address of this thread's column of the fields (field f at + f * stride_bytes)
  int stride_bytes;   // threads per block * 8
};
#define MTB_DECLARE_FAST_CTX(threads)                                                            \
  __shared__ unsigned long long s_fast_scratch[kFmWords * (threads)];                            \
  const FastCtx fctx{(unsigned)__cvta_generic_to_shared(s_fast_scratch + threadIdx.x), (threads) * 8}

// `field` is a constant at every call site.
__device__ __forceinline__ double FmLoad(const FastCtx &fc, int field) {
  double v;
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(fc.ray_base + (unsigned)(field * fc.stride_bytes)));
  return v;
}
__device__ __forceinline__ void FmStore(const FastCtx &fc, int field, double v) {
  asm volatile("st.shared.f64 [%0], %1;" : : "r"(fc.ray_base + (unsigned)(field * fc.stride_bytes)), "d"(v));
}
__device__ __forceinline__ D3 FmLoad3(const FastCtx &fc, int field) {
  return Mk(FmLoad(fc, field), FmLoad(fc, field + 1), FmLoad(fc, field + 2));
}

struct FastRay {
  float ix, iy, iz, nox, noy, noz;  // FP32 inverse direction and -(origin * inverse direction)
};

// One triangle of a scene-BVH leaf: the reference's exact FP64 pre-test and Moller-Trumbore.  `r` carries the FP64
// origin and inverse direction (loaded once per leaf visit); the direction is fetched when the pre-test passes.
// *slot / *prune are the canonical slot of the best hit so far (-1: none) and the FP32 pruning distance.
template <bool DBG>
__device__ __forceinline__ void TestSlotFast(const SlotRec *rec, Ray &r, const FastCtx &fc, int *slot, float *prune,
                                             unsigned long long *cnt) {
  // the whole 128-byte record (box, vertices, ids) in four 256-bit loads: one memory round trip per candidate instead
  // of two for the 58 % of the candidates that pass the pre-test
  double2 b0, b1, b2;
  TriVerts tv;
  double ids_word;
  {
    asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(b0.x), "=d"(b0.y), "=d"(b1.x), "=d"(b1.y) : "l"(rec));
    asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(b2.x), "=d"(b2.y), "=d"(tv.a.x), "=d"(tv.a.y) : "l"(reinterpret_cast<const char *>(rec) + 32));
    asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(tv.b.x), "=d"(tv.b.y), "=d"(tv.c.x), "=d"(tv.c.y) : "l"(reinterpret_cast<const char *>(rec) + 64));
    asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(tv.d.x), "=d"(tv.d.y), "=d"(tv.v22), "=d"(ids_word) : "l"(reinterpret_cast<const char *>(rec) + 96));
  }
  Count<DBG>(cnt, kTriAabb);
  double unused;
  if (!SlabRegular(b0.x, b0.y, b1.x, b1.y, b2.x, b2.y, r, &unused)) return;  // primitive_triangle.cc:85-108
  Count<DBG>(cnt, kMt);
  r.d = FmLoad3(fc, kFmD);
  double t, e;
  if (!MollerTrumboreBound(tv, r, &t, &e)) return;
  Count<DBG>(cnt, kHit);
  const int canon = __double2hiint(ids_word);  // SlotRec: tri (low word), canon (high word) behind the vertices
  if (canon == *slot) return;  // the best hit itself, met again through another of its references (spatial splits)
  if (*slot >= 0) {
    const double bt = FmLoad(fc, kFmT), lo2 = FmLoad(fc, kFmLo2);
    if (!(t < bt)) {
      FmStore(fc, kFmLo2, fmin(lo2, t - e));
      return;
    }
    FmStore(fc, kFmLo2, fmin(lo2, bt - FmLoad(fc, kFmE)));
  }
  FmStore(fc, kFmT, t);
  FmStore(fc, kFmE, e);
  *slot = canon;
  *prune = fminf(*prune, __double2float_ru(t + 2.0 * e + t * 0x1p-20));
}

// Conservative FP32 slab test of one child box; *tn_out = lower bound of the entry distance.  With u = 2^-24,
// of = fl(o), if = fl(1/d), nox = -fl(of if) and t32 = fma(b, if, nox):
//   t32 = [ (b - o) i (1 + a2) - o i (1 + a2) ((1 + a1)(1 + a3) - 1) ] (1 + a4),  |a_k| <= u,
// so |t32 - (b - o) i| <= (2u |b - o| + 2u |o|) |i| (1 + 3u): IN SPACE (divide by |i|) the error is at most
// 2^-23 (|b - o| + |o|) <= 2^-23 * 17 R = 2^-18.9 R for |o| <= 8R, |b| <= R, whatever the ray.  It is therefore paid
// once, at build time: every stored box is grown by 2^-16 R on all sides (SceneBvhBuilder::pad, 7.5x the bound), which
// moves every near plane down and every far plane up PER AXIS.  (Per axis matters: a slack shared between the axes
// made rays almost perpendicular to one axis - huge |i| - pass every box of the scene.  Round 1 paid the |b - o| part
// with two extra FMAs per box in the node loop; folding it into the padding removes them, at 0.006 units of padding
// in the 400-unit C3 room.)  The min / max of per-plane lower / upper bounds are bounds of the true min / max.
__device__ __forceinline__ bool FastBox(float lox, float loy, float loz, float hix, float hiy, float hiz, const FastRay &r,
                                        float prune, float *tn_out) {
  // near / far plane per axis = min / max of the two plane distances (the same two values a sign select picks:
  // the inverse direction is finite and non-zero here, so no NaN can arise) - no predicate per axis to keep alive
  const float ax = __fmaf_rn(lox, r.ix, r.nox), bx = __fmaf_rn(hix, r.ix, r.nox);
  const float ay = __fmaf_rn(loy, r.iy, r.noy), by = __fmaf_rn(hiy, r.iy, r.noy);
  const float az = __fmaf_rn(loz, r.iz, r.noz), bz = __fmaf_rn(hiz, r.iz, r.noz);
  const float tn = fmaxf(fmaxf(fminf(ax, bx), fminf(ay, by)), fminf(az, bz));
  const float tf = fminf(fminf(fmaxf(ax, bx), fmaxf(ay, by)), fmaxf(az, bz));
  *tn_out = tn;
  return tf >= 0.0f && tn <= tf && tn <= prune;
}

// t_limit: the caller discards every hit with t > t_limit (a shadow segment only asks about occluders in front of
// the light, mythtracer.cc:115-118; +inf otherwise), so subtrees that start behind t_limit + M need not be
// searched.  M must cover the rounding error of the t the reference would compute for a triangle that is never
// evaluated here.  Worst case over every triangle the reference could accept (|det| >= 1e-8, component extents
// <= L = sc.max_tri_extent) whose box the ray enters at distance T: |tvec_i| <= |d_i| T + L, so
// N <= 6 L^2 (dmax T + L), D <= 6 dmax L^2 and, as in MollerTrumboreBound (with twice its constants),
//   e <= 2^-48 * 6 L^2 (2 dmax T + L) / (1e-8 - 2^-48 * 6 dmax L^2) + 2^-49 T =: M(T).
// M grows by far less than 1 per unit of T, so a triangle entered behind t_limit + M(t_limit) cannot come out in
// front of t_limit.  If the denominator is not comfortably positive (huge triangles) nothing is pruned by limit.
__device__ __forceinline__ float LimitPrune(const DeviceScene &sc, const D3 &d, double t_limit) {
  if (!(t_limit < CUDART_INF)) return CUDART_INF_F;
  const double L = (double)sc.max_tri_extent;
  const double dmax = fmax(fmax(fabs(d.x), fabs(d.y)), fabs(d.z));
  const double k = 0x1p-48 * 6.0 * L * L;
  const double den = 0.00000001 - k * dmax;
  if (!(den > 0.000000005)) return CUDART_INF_F;
  const double m = k * (2.0 * dmax * t_limit + L) / den + 0x1p-49 * t_limit;
  return __double2float_ru(t_limit + 2.0 * m + t_limit * 0x1p-20);
}

// Closing stated edge case (a) of round 1 (DESIGN.md section 4).  The recursion stops at the first child, in
// entry-distance order, that returns a hit (octtree.cc:244-246).  Octants have disjoint interiors, so along a regular
// ray an octant B that is entered AFTER a sibling A is entered only when A has been left: a hit in A cannot be
// farther than a hit in B, and stopping behind A loses nothing - unless the computed entry keys of A and B tie or
// flip although B really comes first.  Then in(B) <= out(B) <= in(A) <= in(B) + (rounding of the two keys): the
// ray's passage through B, and through every octree node inside B, is degenerate - it touches B in an edge or a
// corner.  (If instead A really comes first, a hit in A is at most as far as the winner, and the error-interval rule
// above already calls that ray ambiguous.)  So for the final hit the passage of the ray through the octree node H
// that HOLDS the winning triangle is measured with the reference's own FP64 slab arithmetic, and a passage shorter
// than 2^-40 relative (keys carry ~2^-52) hands the ray to the exact recursion.  The test ray of round 1
// (o = (7,7,3), d = (-1,-1,-1/8) through the edge x = y = 4 of a [0,8]^3 root) is such a ray.
__device__ __forceinline__ bool DegeneratePassage(const DeviceScene &sc, int slot, const FastCtx &fc) {
  Ray r;
  r.o = FmLoad3(fc, kFmO);
  r.inv = FmLoad3(fc, kFmInv);
  r.sx = r.inv.x < 0.0;
  r.sy = r.inv.y < 0.0;
  r.sz = r.inv.z < 0.0;
  const NodeRec *h = sc.nodes + __ldg(sc.slot_node + slot);
  const double2 p0 = Ld2(h->planes + 0), p1 = Ld2(h->planes + 2), p3 = Ld2(h->planes + 6);
  const double hz = __ldg(&h->planes[8]);
  // planes: lo = (p0.x p0.y p1.x), hi = (p3.x p3.y hz)
  const double nx = ((r.sx ? p3.x : p0.x) - r.o.x) * r.inv.x, fx = ((r.sx ? p0.x : p3.x) - r.o.x) * r.inv.x;
  const double ny = ((r.sy ? p3.y : p0.y) - r.o.y) * r.inv.y, fy = ((r.sy ? p0.y : p3.y) - r.o.y) * r.inv.y;
  const double nz = ((r.sz ? hz : p1.x) - r.o.z) * r.inv.z, fz = ((r.sz ? p1.x : hz) - r.o.z) * r.inv.z;
  const double tmin = SMax3(nx, ny, nz), tmax = SMin3(fx, fy, fz);
  return !(tmax - tmin > 0x1p-40 * (fabs(tmin) + fabs(tmax)));
}

// The FP64 ray has been stored by the caller (fields kFmO .. kFmInv); `prune0` = LimitPrune.  Returns the canonical
// slot of the closest accepted hit (-1: none) with its distance in *t_out.
template <bool DBG>
__device__ __forceinline__ int TraceFast(const DeviceScene &sc, FastMem *m, const FastRay &r_in, float prune0, double *t_out, bool *ambiguous,
                                         unsigned long long *cnt, const FastCtx &fc) {
  // Traversal stack, in the thread's local memory.  An entry is 64 bits: conservative entry distance (FP32 bits) << 32 |
  // child reference, so a pop can discard a subtree behind the pruning distance without touching its node.  Its first
  // entries in shared memory measured slower: the carve-out costs L1 (DESIGN.md section 5, row "first 8 stack entries").
  unsigned long long stack[kFastStack];
  int sp = 0;
  int slot = -1;
  float prune = prune0;
  FmStore(fc, kFmLo2, CUDART_INF);
  int node = 0;
  unsigned visits = 0;  // (counting build only)
  // next subtree from the stack that still starts in front of the pruning distance; kFastExit when there is none
#define MTB_FAST_POP()                                                   \
  do {                                                                   \
    node = kFastExit;                                                    \
    while (sp > 0) {                                                     \
      const unsigned long long top__ = stack[--sp];                      \
      if (__uint_as_float((unsigned)(top__ >> 32)) <= prune) {           \
        node = (int)(unsigned)top__;                                     \
        break;                                                           \
      }                                                                  \
    }                                                                    \
  } while (0)
  // The FP32 ray is only needed in the node loop, the leaf tests in between are where the register pressure peaks
  // (FP64 Moller-Trumbore).  Left to itself ptxas keeps the six floats "live" across the leaf phase by spilling them and
  // puts the reloads INSIDE the node loop (three LDL per node visit at 64 registers).  So the live range is split by
  // hand: the ray stays in memory behind a laundered pointer and is loaded once per entry into the node loop - the
  // barrier of the leaf phase (memory clobber) forces exactly that.
  const FastRay *r_mem = &r_in;
  asm volatile("" : "+l"(r_mem) : : "memory");
  for (;;) {
    const FastRay r = *r_mem;
    while (node >= 0) {
      if (DBG) visits++;
      // one 64-byte node = two 256-bit loads (LDG.E.256, new with sm_100): half the L1 requests / wavefronts of four
      // 128-bit loads when the lanes of a warp are at different nodes
      float4 q0, q1, q2;
      int2 kids;
      {
        const Bvh2Node *np_ = sc.gnodes + node;
        float w8, w9, w10, w11;
        asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=f"(q0.x), "=f"(q0.y), "=f"(q0.z), "=f"(q0.w), "=f"(q1.x), "=f"(q1.y), "=f"(q1.z), "=f"(q1.w)
                     : "l"(np_));
        asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=f"(q2.x), "=f"(q2.y), "=f"(q2.z), "=f"(q2.w), "=f"(w8), "=f"(w9), "=f"(w10), "=f"(w11)
                     : "l"(reinterpret_cast<const char *>(np_) + 32));
        kids.x = __float_as_int(w8);
        kids.y = __float_as_int(w9);
      }
      Count<DBG>(cnt, kBvh, 2);
      float tl, tr;
      const bool hl = FastBox(q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, r, prune, &tl);
      const bool hr = FastBox(q1.z, q1.w, q2.x, q2.y, q2.z, q2.w, r, prune, &tr);
      if (hl && hr) {
        const bool right_first = tr < tl;
        stack[sp++] = ((unsigned long long)__float_as_uint(right_first ? tl : tr) << 32) | (unsigned)(right_first ? kids.x : kids.y);
        node = right_first ? kids.y : kids.x;
      } else if (hl) {
        node = kids.x;
      } else if (hr) {
        node = kids.y;
      } else {
        MTB_FAST_POP();
      }
    }
    if (node == kFastExit) break;
    {
      MTB_FAST_BARRIER(m);
      Ray rr;  // FP64 origin and inverse direction: once per leaf visit
      rr.o = FmLoad3(fc, kFmO);
      rr.inv = FmLoad3(fc, kFmInv);
      rr.sx = rr.inv.x < 0.0;
      rr.sy = rr.inv.y < 0.0;
      rr.sz = rr.inv.z < 0.0;
      const unsigned leaf = ~(unsigned)node;
      for (unsigned s = leaf >> 3, e = s + (leaf & 7u); s < e; s++) TestSlotFast<DBG>(sc.gslots + s, rr, fc, &slot, &prune, cnt);
      MTB_FAST_BARRIER(m);
    }
    MTB_FAST_POP();
  }
#undef MTB_FAST_POP
  if (DBG) {
    if (visits > 128u) Count<DBG>(cnt, kLongRays128), Count<DBG>(cnt, kLongVisits128, visits);
    if (visits > 512u) Count<DBG>(cnt, kLongRays512), Count<DBG>(cnt, kLongVisits512, visits);
  }
  bool amb = false;
  if (slot >= 0) {
    MTB_FAST_BARRIER(m);
    const double t = FmLoad(fc, kFmT);
    amb = FmLoad(fc, kFmLo2) <= t + FmLoad(fc, kFmE) || DegeneratePassage(sc, slot, fc);
    *t_out = t;
  }
  *ambiguous = amb;
  return slot;
}

// The ray record of the exact traversals (TraceRegular / TraceLiteral): inverse direction, signs, FP32 cull values.
__device__ __forceinline__ void MakeRay(const DeviceScene &sc, const D3 &o, const D3 &d, Ray *out, bool *regular) {
  Ray &r = *out;
  r.o = o;
  r.d = d;
  r.inv = Mk(1.0 / d.x, 1.0 / d.y, 1.0 / d.z);
  r.sx = r.inv.x < 0.0;
  r.sy = r.inv.y < 0.0;
  r.sz = r.inv.z < 0.0;
  *regular = isfinite(r.inv.x) && isfinite(r.inv.y) && isfinite(r.inv.z) && r.inv.x != 0.0 && r.inv.y != 0.0 &&
             r.inv.z != 0.0 && isfinite(o.x) && isfinite(o.y) && isfinite(o.z);
  // FP32 cull preconditions (see CullBox32 / FastBox): origin within 8R, |inv| within [2^-100, 2^100]
  const float R = sc.cull_radius;
  const double ao = fmax(fmax(fabs(o.x), fabs(o.y)), fabs(o.z));
  const double ai_max = fmax(fmax(fabs(r.inv.x), fabs(r.inv.y)), fabs(r.inv.z));
  const double ai_min = fmin(fmin(fabs(r.inv.x), fabs(r.inv.y)), fabs(r.inv.z));
  r.cull32 = *regular && R > 0.0f && ao <= 8.0 * (double)R && ai_max <= 0x1p100 && ai_min >= 0x1p-100;
  r.ox = (float)o.x;
  r.oy = (float)o.y;
  r.oz = (float)o.z;
  r.ix = (float)r.inv.x;
  r.iy = (float)r.inv.y;
  r.iz = (float)r.inv.z;
  const float pr = R * 9.5367431640625e-07f;  // 2^-20 * R
  r.px = pr * fabsf(r.ix);
  r.py = pr * fabsf(r.iy);
  r.pz = pr * fabsf(r.iz);
}

// Rays the fast traversal does not answer: irregular rays (literal recursion), rays outside the FP32 error model or
// scenes without a scene BVH, and rays whose fast answer could not be certified (exact recursion).
template <bool DBG>
__device__ __noinline__ int TraceExactCold(const DeviceScene &sc, const D3 &o, const D3 &d, double *t_out, unsigned long long *cnt) {
  Ray r;
  bool regular;
  MakeRay(sc, o, d, &r, &regular);
  if (regular) return TraceRegular<DBG>(sc, r, t_out, cnt);
  return TraceLiteral<DBG>(sc, r, t_out, cnt);
}

// OctTree::IntersectRay (octtree.cc:26-40): inverse direction, then one of the traversals.
// t_limit: results with t > t_limit are of no use to the caller (it may then get -1 or any such hit); CUDART_INF
// for a plain closest-hit query.
template <bool DBG>
__device__ __forceinline__ int Trace(const DeviceScene &sc, const D3 &o, const D3 &d, double t_limit, double *t_out,
                                     unsigned long long *cnt, const FastCtx &fc) {
  Count<DBG>(cnt, kRays);
  FastMem mem;
  bool fast;
  FastRay fr;
  float prune0;
  {
    const D3 inv = Mk(1.0 / d.x, 1.0 / d.y, 1.0 / d.z);
    const bool regular = isfinite(inv.x) && isfinite(inv.y) && isfinite(inv.z) && inv.x != 0.0 && inv.y != 0.0 &&
                         inv.z != 0.0 && isfinite(o.x) && isfinite(o.y) && isfinite(o.z);
    const float R = sc.cull_radius;
    const double ao = fmax(fmax(fabs(o.x), fabs(o.y)), fabs(o.z));
    const double ai_max = fmax(fmax(fabs(inv.x), fabs(inv.y)), fabs(inv.z));
    const double ai_min = fmin(fmin(fabs(inv.x), fabs(inv.y)), fabs(inv.z));
    fast = regular && sc.gnodes != nullptr && R > 0.0f && ao <= 8.0 * (double)R && ai_max <= 0x1p100 && ai_min >= 0x1p-100;
    FmStore(fc, kFmO + 0, o.x), FmStore(fc, kFmO + 1, o.y), FmStore(fc, kFmO + 2, o.z);
    FmStore(fc, kFmD + 0, d.x), FmStore(fc, kFmD + 1, d.y), FmStore(fc, kFmD + 2, d.z);
    FmStore(fc, kFmInv + 0, inv.x), FmStore(fc, kFmInv + 1, inv.y), FmStore(fc, kFmInv + 2, inv.z);
    fr.ix = (float)inv.x;
    fr.iy = (float)inv.y;
    fr.iz = (float)inv.z;
    fr.nox = -((float)o.x * fr.ix);
    fr.noy = -((float)o.y * fr.iy);
    fr.noz = -((float)o.z * fr.iz);
    prune0 = LimitPrune(sc, d, t_limit);
  }
  if (fast) {
    MTB_FAST_BARRIER(&mem);
    bool ambiguous;
    const int slot = TraceFast<DBG>(sc, &mem, fr, prune0, t_out, &ambiguous, cnt, fc);
    if (!ambiguous) {
      Count<DBG>(cnt, kFast);
      return slot;
    }
    Count<DBG>(cnt, kFallback);
  }
  MTB_FAST_BARRIER(&mem);
  return TraceExactCold<DBG>(sc, FmLoad3(fc, kFmO), FmLoad3(fc, kFmD), t_out, cnt);
}

// ---------------------------------------------------------------------------------------------------
// shading helpers
// ---------------------------------------------------------------------------------------------------
// primitive_triangle.cc:27-40
__device__ __forceinline__ double Heron(double a, double b, double c) {
  const double p = (a + b + c) / 2.0;
  const double area_sqr = p * (p - a) * (p - b) * (p - c);
  if (area_sqr < 0.0) return 0.0;
  return sqrt(area_sqr);
}

struct BaryWeights {
  double n0, n1, n2, n;
};
// primitive_triangle.cc:45-57 (shared by GetNormal and GetUVW)
__device__ __forceinline__ BaryWeights Barycentric(const D3 &v0, const D3 &v1, const D3 &v2, const D3 &point) {
  const double a = Dist(v0, v1);
  const double b = Dist(v1, v2);
  const double c = Dist(v2, v0);
  const double p0 = Dist(point, v0);
  const double p1 = Dist(point, v1);
  const double p2 = Dist(point, v2);
  BaryWeights w;
  w.n0 = Heron(b, p2, p1);
  w.n1 = Heron(c, p0, p2);
  w.n2 = Heron(a, p1, p0);
  w.n = w.n0 + w.n1 + w.n2;
  return w;
}

// texture.cc:11-58 with point fetches of the 8-bit texels; px / 255.0 as texture.cc:100-104.  A texel is one
// 32-bit word (R | G << 8 | B << 16 | A << 24) of layer `layer` of the scene's single layered texture object.
__device__ __forceinline__ D3 Texel(cudaTextureObject_t atlas, int layer, size_t x, size_t y) {
  const unsigned p = tex2DLayered<unsigned>(atlas, (float)x + 0.5f, (float)y + 0.5f, layer);
  return Mk((double)(p & 255u) / 255.0, (double)((p >> 8) & 255u) / 255.0, (double)((p >> 16) & 255u) / 255.0);
}
__device__ __noinline__ D3 SampleTexture(cudaTextureObject_t tex, int layer, int2 dim, double u, double v) {
  u = fmod(u, 1.0);
  v = fmod(v, 1.0);
  if (u < 0.0) u += 1.0;
  if (v < 0.0) v += 1.0;
  v = 1.0 - v;
  const size_t width = (size_t)dim.x, height = (size_t)dim.y;
  const double x = u * (double)(width - 1);
  const double y = v * (double)(height - 1);
  size_t bx = (size_t)x;
  size_t by = (size_t)y;
  // (size_t)NaN is undefined upstream (vector::at would throw); stay inside the texture here
  if (bx >= width) bx = width - 1;
  if (by >= height) by = height - 1;
  const size_t bx1 = (bx + 1 == width) ? bx : bx + 1;
  const size_t by1 = (by + 1 == height) ? by : by + 1;
  const D3 c0 = Texel(tex, layer, bx, by), c1 = Texel(tex, layer, bx1, by), c2 = Texel(tex, layer, bx, by1), c3 = Texel(tex, layer, bx1, by1);
  const double dx = fmod(x, 1.0);
  const double dy = fmod(y, 1.0);
  const double a0 = (1.0 - dx) * (1.0 - dy);
  const double a1 = dx * (1.0 - dy);
  const double a2 = (1.0 - dx) * dy;
  const double a3 = dx * dy;
  return Add(Add(Add(MulS(c0, a0), MulS(c1, a1)), MulS(c2, a2)), MulS(c3, a3));
}

// mythtracer.cc:235-241.  (uint8_t)(NaN * 255) is 0 on x86-64; restated explicitly.
__device__ __forceinline__ unsigned char QuantizeChannel(double v) {
  if (v > 1.0) return 255;
  if (v < 0.0) return 0;
  if (v != v) return 0;
  return (unsigned char)(int)(v * 255);
}

__device__ __forceinline__ unsigned long long Mix64(unsigned long long path, unsigned long long kind,
                                                    unsigned long long value) {
  unsigned long long z = path * 0x9E3779B97F4A7C15ull + kind * 0xC2B2AE3D27D4EB4Full +
                         value * 0x165667B19E3779F9ull + 0x27D4EB2F165667C5ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}


}  // namespace
}  // namespace mtb
