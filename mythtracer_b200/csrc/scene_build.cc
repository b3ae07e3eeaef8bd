// Reference-exact octree construction, flattened for the GPU (see scene_build.h).
//
// What must be identical to the reference, because it decides results:
//   * triangle boxes = exact min/max of the three vertices      (primitive_triangle.cc:18-24, aabb.cc:42-47)
//   * the root box grows from {0,0,0}-{0,0,0}                    (math3d.h:141, octtree.cc:12-13)
//   * a node is split iff it holds >= 16 primitives, no depth cap (octtree.h:43, octtree.cc:53-55)
//   * centre = lo + (hi - lo) / 2.0                               (octtree.cc:46-50)
//   * child k: bit0 -> upper x half, bit1 -> upper z half, bit2 -> upper y half   (octtree.cc:61-100)
//   * a primitive moves to the FIRST child whose closed box holds both corners of its box, otherwise it
//     stays; order inside every list = insertion order             (octtree.cc:106-129, aabb.cc:5-7,29-33)
// What is free (it only affects speed): the order of nodes in memory, the order of slots inside a list
// (ties are decided by the insertion index stored in every slot) and the list-BVH.
#include "scene_build.h"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <numeric>
#include <thread>

namespace mtb {
namespace {

struct Box3 {
  double lo[3], hi[3];
};

struct BuildNode {
  Box3 box;
  double c[3] = {0, 0, 0};
  int32_t first_child = -1;
  int32_t level = 0;
  std::vector<int32_t> list;  // insertion indices, ascending
};

inline bool HoldsBox(const Box3 &outer, const Box3 &inner) {
  for (int a = 0; a < 3; a++) {
    if (!(inner.lo[a] >= outer.lo[a] && inner.lo[a] <= outer.hi[a])) return false;
    if (!(inner.hi[a] >= outer.lo[a] && inner.hi[a] <= outer.hi[a])) return false;
  }
  return true;
}

// Work-list formulation of Node::AttemptSplit: nodes are appended to `nodes`, eight at a time.
int SplitAll(const std::vector<Box3> &tri_box, std::vector<BuildNode> *nodes, int32_t *depth, std::string *err) {
  std::vector<int32_t> todo;
  todo.push_back(0);
  std::vector<int32_t> keep;
  while (!todo.empty()) {
    const int32_t idx = todo.back();
    todo.pop_back();
    if ((*nodes)[idx].level > *depth) *depth = (*nodes)[idx].level;
    if ((*nodes)[idx].list.size() < 16) continue;
    if ((*nodes)[idx].level >= MTB_MAX_TREE_DEPTH) {
      *err = "octree deeper than MTB_MAX_TREE_DEPTH (16 or more coincident primitives?)";
      return MTB_ERR_LIMIT;
    }
    const int32_t first = (int32_t)nodes->size();
    nodes->resize(nodes->size() + 8);
    BuildNode &n = (*nodes)[idx];
    n.first_child = first;
    for (int a = 0; a < 3; a++) n.c[a] = n.box.lo[a] + (n.box.hi[a] - n.box.lo[a]) / 2.0;
    for (int k = 0; k < 8; k++) {
      BuildNode &ch = (*nodes)[first + k];
      ch.level = n.level + 1;
      const int upper[3] = {k & 1, (k >> 2) & 1, (k >> 1) & 1};  // x <- bit0, y <- bit2, z <- bit1
      for (int a = 0; a < 3; a++) {
        ch.box.lo[a] = upper[a] ? n.c[a] : n.box.lo[a];
        ch.box.hi[a] = upper[a] ? n.box.hi[a] : n.c[a];
      }
    }
    keep.clear();
    for (int32_t t : n.list) {
      int k = 0;
      for (; k < 8; k++) {
        if (HoldsBox((*nodes)[first + k].box, tri_box[t])) break;
      }
      if (k < 8) {
        (*nodes)[first + k].list.push_back(t);
      } else {
        keep.push_back(t);
      }
    }
    n.list.assign(keep.begin(), keep.end());
    n.list.shrink_to_fit();
    for (int k = 7; k >= 0; k--) todo.push_back(first + k);
  }
  return MTB_OK;
}

inline double HalfArea(const Box3 &b) {
  const double dx = b.hi[0] - b.lo[0], dy = b.hi[1] - b.lo[1], dz = b.hi[2] - b.lo[2];
  return dx * dy + dy * dz + dz * dx;
}

// double -> float, rounded towards -inf / +inf (the float box must contain the double box)
inline float RoundDown(double x) {
  float f = (float)x;
  if ((double)f > x) f = std::nextafterf(f, -INFINITY);
  return f;
}
inline float RoundUp(double x) {
  float f = (float)x;
  if ((double)f < x) f = std::nextafterf(f, INFINITY);
  return f;
}

// Bounds of ids[b, e): union box `u` and the bounds clo/chi of the doubled centroids (lo + hi).
inline void RangeBounds(const std::vector<Box3> &tri_box, const std::vector<int32_t> &ids, int32_t b, int32_t e, Box3 *u,
                        double clo[3], double chi[3]) {
  for (int a = 0; a < 3; a++) {
    u->lo[a] = clo[a] = INFINITY;
    u->hi[a] = chi[a] = -INFINITY;
  }
  for (int32_t i = b; i < e; i++) {
    const Box3 &tb = tri_box[ids[i]];
    for (int a = 0; a < 3; a++) {
      u->lo[a] = std::min(u->lo[a], tb.lo[a]);
      u->hi[a] = std::max(u->hi[a], tb.hi[a]);
      const double cc = tb.lo[a] + tb.hi[a];
      clo[a] = std::min(clo[a], cc);
      chi[a] = std::max(chi[a], cc);
    }
  }
}

// Partitions ids[b, e) in place and returns the split position (b < mid < e for e - b >= 2): binned surface-area
// heuristic over the centroids (16 bins per axis); object median along the widest axis when SAH finds no split
// (or `median_only`).  The summed surface area of the descendants is proportional to the expected number of box
// tests of a ray that is not pruned by distance: what SAH minimises.
int32_t SahPartition(const std::vector<Box3> &tri_box, std::vector<int32_t> &ids, int32_t b, int32_t e, const double clo[3],
                     const double chi[3], bool median_only) {
  constexpr int kBins = 16;  // 8 / 16 / 32 / 64 bins: SAH cost of the C3 scene BVH 52.6 / 51.8 / 51.2 / 51.1 expected node visits
  int best_axis = -1, best_bin = -1;
  double best_cost = INFINITY;
  for (int axis = 0; axis < 3 && !median_only; axis++) {
    const double lo = clo[axis], ext = chi[axis] - clo[axis];
    if (!(ext > 0.0)) continue;
    Box3 bin_box[kBins];
    int bin_n[kBins];
    for (int k = 0; k < kBins; k++) {
      bin_n[k] = 0;
      for (int a = 0; a < 3; a++) {
        bin_box[k].lo[a] = INFINITY;
        bin_box[k].hi[a] = -INFINITY;
      }
    }
    for (int32_t i = b; i < e; i++) {
      const Box3 &tb = tri_box[ids[i]];
      int k = (int)(((tb.lo[axis] + tb.hi[axis]) - lo) / ext * kBins);
      k = k < 0 ? 0 : (k >= kBins ? kBins - 1 : k);
      bin_n[k]++;
      for (int a = 0; a < 3; a++) {
        bin_box[k].lo[a] = std::min(bin_box[k].lo[a], tb.lo[a]);
        bin_box[k].hi[a] = std::max(bin_box[k].hi[a], tb.hi[a]);
      }
    }
    double right_area[kBins];
    int right_n[kBins];
    Box3 acc;
    int n_acc = 0;
    for (int a = 0; a < 3; a++) {
      acc.lo[a] = INFINITY;
      acc.hi[a] = -INFINITY;
    }
    for (int k = kBins - 1; k > 0; k--) {
      if (bin_n[k] > 0) {
        for (int a = 0; a < 3; a++) {
          acc.lo[a] = std::min(acc.lo[a], bin_box[k].lo[a]);
          acc.hi[a] = std::max(acc.hi[a], bin_box[k].hi[a]);
        }
        n_acc += bin_n[k];
      }
      right_area[k] = n_acc > 0 ? HalfArea(acc) : 0.0;
      right_n[k] = n_acc;
    }
    n_acc = 0;
    for (int a = 0; a < 3; a++) {
      acc.lo[a] = INFINITY;
      acc.hi[a] = -INFINITY;
    }
    for (int k = 0; k + 1 < kBins; k++) {
      if (bin_n[k] > 0) {
        for (int a = 0; a < 3; a++) {
          acc.lo[a] = std::min(acc.lo[a], bin_box[k].lo[a]);
          acc.hi[a] = std::max(acc.hi[a], bin_box[k].hi[a]);
        }
        n_acc += bin_n[k];
      }
      if (n_acc == 0 || right_n[k + 1] == 0) continue;
      const double cost = HalfArea(acc) * n_acc + right_area[k + 1] * right_n[k + 1];
      if (cost < best_cost) {
        best_cost = cost;
        best_axis = axis;
        best_bin = k;
      }
    }
  }
  int32_t mid = b;  // all centroids coincide
  if (best_axis >= 0) {
    const double lo = clo[best_axis], ext = chi[best_axis] - clo[best_axis];
    auto bin_of = [&](int32_t t) {
      int k = (int)(((tri_box[t].lo[best_axis] + tri_box[t].hi[best_axis]) - lo) / ext * kBins);
      return k < 0 ? 0 : (k >= kBins ? kBins - 1 : k);
    };
    mid = (int32_t)(std::partition(ids.begin() + b, ids.begin() + e, [&](int32_t t) { return bin_of(t) <= best_bin; }) - ids.begin());
  }
  if (mid == b || mid == e) {
    int axis = 0;
    if (chi[1] - clo[1] > chi[axis] - clo[axis]) axis = 1;
    if (chi[2] - clo[2] > chi[axis] - clo[axis]) axis = 2;
    mid = b + (e - b) / 2;
    std::nth_element(ids.begin() + b, ids.begin() + mid, ids.begin() + e, [&](int32_t x, int32_t y) {
      const double cx = tri_box[x].lo[axis] + tri_box[x].hi[axis];
      const double cy = tri_box[y].lo[axis] + tri_box[y].hi[axis];
      return cx < cy || (cx == cy && x < y);
    });
  }
  return mid;
}

// SAH BVH over `ids[b, e)` of ONE node list; emits threaded records depth first and the slot order of the triangles.
struct BvhBuilder {
  const std::vector<Box3> &tri_box;
  std::vector<BvhRec> *out;
  std::vector<int32_t> ids;  // triangles of the current list; permuted in place into leaf order
  int32_t slot_base = 0;

  void Build(int32_t b, int32_t e) {
    const int32_t me = (int32_t)out->size();
    out->emplace_back();
    Box3 u;
    double clo[3], chi[3];
    RangeBounds(tri_box, ids, b, e, &u, clo, chi);
    BvhRec rec;
    memset(&rec, 0, sizeof(rec));
    for (int a = 0; a < 3; a++) {
      rec.box[a] = RoundDown(u.lo[a]);
      rec.box[3 + a] = RoundUp(u.hi[a]);
    }
    if (e - b <= kBvhLeafSize) {
      rec.leaf = ((uint32_t)(slot_base + b) << 3) | (uint32_t)(e - b);
      rec.skip = me + 1;
      (*out)[me] = rec;
      return;
    }
    const int32_t mid = SahPartition(tri_box, ids, b, e, clo, chi, false);
    Build(b, mid);
    Build(mid, e);
    rec.skip = (int32_t)out->size();
    (*out)[me] = rec;
  }
};

// Spatial pre-splitting of large triangles for the scene BVH ("early split clipping").  A long thin triangle that
// crosses the room diagonally has an AABB the size of the room: every ray passes its box, the reference's exact
// pre-test passes too, and the triangle has to be given its exact Moller-Trumbore evaluation by almost every ray
// (round 1, C4: 2835 evaluations per ray).  Here such a triangle enters the scene BVH as several REFERENCES, each with
// the bounds of the piece of the triangle inside one cell of a recursive midpoint split of its box; a ray then reaches
// the triangle only through the pieces it actually passes.  What is evaluated at a leaf is unchanged - the whole
// triangle, by the reference's exact pre-test and Moller-Trumbore - so the set of accepted hits can only shrink by
// hits whose computed position lies outside every padded piece box, i.e. off the triangle by more than the padding:
// that needs a ray parallel to the triangle's plane to within rounding (|det| a few ulps above the reference's 1e-8
// threshold), the extension of stated edge case (b) of DESIGN.md section 4 to split triangles.
struct Poly {
  int n = 0;
  double v[10][3];
};

// Sutherland-Hodgman against the half space x[axis] <= p (keep_low) or >= p; points on the plane get x[axis] = p.
inline void ClipPoly(const Poly &in, int axis, double p, bool keep_low, Poly *out) {
  out->n = 0;
  for (int i = 0; i < in.n; i++) {
    const double *a = in.v[i], *b = in.v[(i + 1) % in.n];
    const bool ina = keep_low ? a[axis] <= p : a[axis] >= p;
    const bool inb = keep_low ? b[axis] <= p : b[axis] >= p;
    if (ina && out->n < 10) {
      for (int k = 0; k < 3; k++) out->v[out->n][k] = a[k];
      out->n++;
    }
    if (ina != inb && out->n < 10) {
      const double t = (p - a[axis]) / (b[axis] - a[axis]);
      for (int k = 0; k < 3; k++) out->v[out->n][k] = a[k] + t * (b[k] - a[k]);
      out->v[out->n][axis] = p;
      out->n++;
    }
  }
}

// References of triangle `tri` (box `tb`) with pieces no longer than `max_extent` along any axis, appended to the
// lists.  Every piece box is grown by `guard` (the clipping arithmetic rounds) and clipped to the triangle's box.
inline void SplitTriangle(const double vert[9], const Box3 &tb, int32_t tri, double max_extent, double guard,
                          std::vector<Box3> *ref_box, std::vector<int32_t> *ref_tri) {
  struct Item {
    Poly poly;
    Box3 cell;
    int depth;
  };
  std::vector<Item> stack(1);
  stack[0].poly.n = 3;
  for (int i = 0; i < 3; i++) {
    for (int k = 0; k < 3; k++) stack[0].poly.v[i][k] = vert[i * 3 + k];
  }
  stack[0].cell = tb;
  stack[0].depth = 0;
  while (!stack.empty()) {
    Item it = stack.back();
    stack.pop_back();
    // bounds of the piece, inside its cell
    Box3 pb;
    for (int a = 0; a < 3; a++) {
      pb.lo[a] = INFINITY;
      pb.hi[a] = -INFINITY;
      for (int i = 0; i < it.poly.n; i++) {
        pb.lo[a] = std::min(pb.lo[a], it.poly.v[i][a]);
        pb.hi[a] = std::max(pb.hi[a], it.poly.v[i][a]);
      }
      pb.lo[a] = std::max(pb.lo[a], it.cell.lo[a]);
      pb.hi[a] = std::min(pb.hi[a], it.cell.hi[a]);
    }
    int axis = 0;
    for (int a = 1; a < 3; a++) {
      if (pb.hi[a] - pb.lo[a] > pb.hi[axis] - pb.lo[axis]) axis = a;
    }
    const double ext = pb.hi[axis] - pb.lo[axis];
    if (!(ext > max_extent) || it.depth >= 24) {
      Box3 out;
      for (int a = 0; a < 3; a++) {
        out.lo[a] = std::max(pb.lo[a] - guard, tb.lo[a]);
        out.hi[a] = std::min(pb.hi[a] + guard, tb.hi[a]);
      }
      ref_box->push_back(out);
      ref_tri->push_back(tri);
      continue;
    }
    const double mid = pb.lo[axis] + 0.5 * ext;
    for (int side = 0; side < 2; side++) {
      Item child;
      ClipPoly(it.poly, axis, mid, side == 0, &child.poly);
      if (child.poly.n < 3) continue;
      child.cell = pb;
      (side == 0 ? child.cell.hi[axis] : child.cell.lo[axis]) = mid;
      child.depth = it.depth + 1;
      stack.push_back(child);
    }
  }
}

// The top levels of the scene BVH are ranges of hundreds of thousands of references handled by ONE node at a time;
// in round 1 the calling thread binned and partitioned them alone (0.10 of the 0.15 s of the C3 build on 24 cores).
// These helpers spread one such pass over the host threads.  Results do not depend on the number of threads: the
// bounds and bins are min / max / counts (order-free), the partition is STABLE (a unique result).
constexpr int32_t kParallelRange = 1 << 15;

template <typename F>
void ParallelSlices(int32_t b, int32_t e, unsigned n_threads, F fn) {  // fn(slice index, slice begin, slice end)
  const int32_t n = e - b;
  const unsigned slices = n_threads < 1 ? 1 : n_threads;
  if (slices == 1) {
    fn(0u, b, e);
    return;
  }
  std::vector<std::thread> pool;
  for (unsigned k = 1; k < slices; k++) {
    pool.emplace_back([=]() { fn(k, b + (int32_t)((int64_t)n * k / slices), b + (int32_t)((int64_t)n * (k + 1) / slices)); });
  }
  fn(0u, b, b + (int32_t)((int64_t)n / slices));
  for (std::thread &t : pool) t.join();
}

inline void ParallelRangeBounds(const std::vector<Box3> &tri_box, const std::vector<int32_t> &ids, int32_t b, int32_t e, unsigned n_threads,
                                Box3 *u, double clo[3], double chi[3]) {
  struct Part {
    Box3 u;
    double clo[3], chi[3];
  };
  std::vector<Part> part(n_threads < 1 ? 1 : n_threads);
  ParallelSlices(b, e, n_threads, [&](unsigned k, int32_t sb, int32_t se) { RangeBounds(tri_box, ids, sb, se, &part[k].u, part[k].clo, part[k].chi); });
  for (int a = 0; a < 3; a++) {
    u->lo[a] = clo[a] = INFINITY;
    u->hi[a] = chi[a] = -INFINITY;
  }
  for (const Part &p : part) {
    for (int a = 0; a < 3; a++) {
      u->lo[a] = std::min(u->lo[a], p.u.lo[a]);
      u->hi[a] = std::max(u->hi[a], p.u.hi[a]);
      clo[a] = std::min(clo[a], p.clo[a]);
      chi[a] = std::max(chi[a], p.chi[a]);
    }
  }
}

// SahPartition for a big range: the same 16 bins per axis and the same cost, every pass spread over the threads.
int32_t ParallelSahPartition(const std::vector<Box3> &tri_box, std::vector<int32_t> &ids, std::vector<int32_t> &scratch, int32_t b, int32_t e,
                             const double clo[3], const double chi[3], unsigned n_threads) {
  constexpr int kBins = 16;
  struct Bins {
    Box3 box[3][kBins];
    int n[3][kBins];
  };
  const unsigned T = n_threads < 1 ? 1 : n_threads;
  std::vector<Bins> part(T);
  ParallelSlices(b, e, T, [&](unsigned k, int32_t sb, int32_t se) {
    Bins &bn = part[k];
    for (int axis = 0; axis < 3; axis++) {
      for (int q = 0; q < kBins; q++) {
        bn.n[axis][q] = 0;
        for (int a = 0; a < 3; a++) {
          bn.box[axis][q].lo[a] = INFINITY;
          bn.box[axis][q].hi[a] = -INFINITY;
        }
      }
    }
    for (int32_t i = sb; i < se; i++) {
      const Box3 &tb = tri_box[ids[i]];
      for (int axis = 0; axis < 3; axis++) {
        const double ext = chi[axis] - clo[axis];
        if (!(ext > 0.0)) continue;
        int q = (int)(((tb.lo[axis] + tb.hi[axis]) - clo[axis]) / ext * kBins);
        q = q < 0 ? 0 : (q >= kBins ? kBins - 1 : q);
        bn.n[axis][q]++;
        for (int a = 0; a < 3; a++) {
          bn.box[axis][q].lo[a] = std::min(bn.box[axis][q].lo[a], tb.lo[a]);
          bn.box[axis][q].hi[a] = std::max(bn.box[axis][q].hi[a], tb.hi[a]);
        }
      }
    }
  });
  int best_axis = -1, best_bin = -1;
  double best_cost = INFINITY;
  for (int axis = 0; axis < 3; axis++) {
    if (!(chi[axis] - clo[axis] > 0.0)) continue;
    Box3 bin_box[kBins];
    int bin_n[kBins];
    for (int q = 0; q < kBins; q++) {
      bin_n[q] = 0;
      for (int a = 0; a < 3; a++) {
        bin_box[q].lo[a] = INFINITY;
        bin_box[q].hi[a] = -INFINITY;
      }
      for (const Bins &bn : part) {
        bin_n[q] += bn.n[axis][q];
        for (int a = 0; a < 3; a++) {
          bin_box[q].lo[a] = std::min(bin_box[q].lo[a], bn.box[axis][q].lo[a]);
          bin_box[q].hi[a] = std::max(bin_box[q].hi[a], bn.box[axis][q].hi[a]);
        }
      }
    }
    double right_area[kBins];
    int right_n[kBins];
    Box3 acc;
    int n_acc = 0;
    for (int a = 0; a < 3; a++) {
      acc.lo[a] = INFINITY;
      acc.hi[a] = -INFINITY;
    }
    for (int q = kBins - 1; q > 0; q--) {
      if (bin_n[q] > 0) {
        for (int a = 0; a < 3; a++) {
          acc.lo[a] = std::min(acc.lo[a], bin_box[q].lo[a]);
          acc.hi[a] = std::max(acc.hi[a], bin_box[q].hi[a]);
        }
        n_acc += bin_n[q];
      }
      right_area[q] = n_acc > 0 ? HalfArea(acc) : 0.0;
      right_n[q] = n_acc;
    }
    n_acc = 0;
    for (int a = 0; a < 3; a++) {
      acc.lo[a] = INFINITY;
      acc.hi[a] = -INFINITY;
    }
    for (int q = 0; q + 1 < kBins; q++) {
      if (bin_n[q] > 0) {
        for (int a = 0; a < 3; a++) {
          acc.lo[a] = std::min(acc.lo[a], bin_box[q].lo[a]);
          acc.hi[a] = std::max(acc.hi[a], bin_box[q].hi[a]);
        }
        n_acc += bin_n[q];
      }
      if (n_acc == 0 || right_n[q + 1] == 0) continue;
      const double cost = HalfArea(acc) * n_acc + right_area[q + 1] * right_n[q + 1];
      if (cost < best_cost) {
        best_cost = cost;
        best_axis = axis;
        best_bin = q;
      }
    }
  }
  if (best_axis < 0) return SahPartition(tri_box, ids, b, e, clo, chi, true);  // all centroids coincide: median
  // stable partition through the scratch array: lefts of all slices first, then the rights, each in input order
  const double lo = clo[best_axis], ext = chi[best_axis] - clo[best_axis];
  auto is_left = [&](int32_t t) {
    int q = (int)(((tri_box[t].lo[best_axis] + tri_box[t].hi[best_axis]) - lo) / ext * kBins);
    q = q < 0 ? 0 : (q >= kBins ? kBins - 1 : q);
    return q <= best_bin;
  };
  std::vector<int32_t> n_left(T + 1, 0), s_begin(T, b), s_end(T, b);
  ParallelSlices(b, e, T, [&](unsigned k, int32_t sb, int32_t se) {
    int32_t c = 0;
    for (int32_t i = sb; i < se; i++) c += is_left(ids[i]) ? 1 : 0;
    n_left[k + 1] = c;
    s_begin[k] = sb;
    s_end[k] = se;
  });
  for (unsigned k = 0; k < T; k++) n_left[k + 1] += n_left[k];
  const int32_t mid = b + n_left[T];
  if (mid == b || mid == e) return SahPartition(tri_box, ids, b, e, clo, chi, true);
  if (scratch.size() < ids.size()) scratch.resize(ids.size());
  ParallelSlices(b, e, T, [&](unsigned k, int32_t sb, int32_t se) {
    int32_t l = b + n_left[k], r = mid + (sb - b) - n_left[k];
    for (int32_t i = sb; i < se; i++) {
      const int32_t t = ids[i];
      if (is_left(t)) {
        scratch[(size_t)l++] = t;
      } else {
        scratch[(size_t)r++] = t;
      }
    }
  });
  ParallelSlices(b, e, T, [&](unsigned, int32_t sb, int32_t se) { memcpy(&ids[(size_t)sb], &scratch[(size_t)sb], (size_t)(se - sb) * sizeof(int32_t)); });
  return mid;
}

// Scene BVH (Bvh2Node, scene_build.h) over ALL triangles: the acceleration structure of the certified fast
// traversal.  ids ends up in leaf order = the order of the `gslots` copies.  The top of the tree is split by the
// calling thread; every range of at most `grain` triangles below it is an independent job for a pool of threads
// (each job builds into its own vector, the vectors are appended and their indices rebased afterwards), so the
// result does not depend on the number of threads.
struct SceneBvhBuilder {
  const std::vector<Box3> &tri_box;
  std::vector<int32_t> ids;
  int32_t max_depth = 0;
  // every stored box is grown by `pad` on all sides: the FP32 slab test's whole error bound is a constant
  // 2^-18.9 R in space, whatever the ray (FastBox, device_core.cuh); pad = 2^-16 R
  double pad = 0.0;

  unsigned par_threads = 1;
  std::vector<int32_t> scratch;  // ParallelSahPartition

  struct Job {
    int32_t b, e, depth;
    int32_t parent, side;  // where the finished subtree hangs
    std::vector<Bvh2Node> nodes;
    int32_t ref = 0;       // subtree root: local node index (>= 0) or leaf (< 0)
    Box3 box;
    int32_t deepest = 0;
  };
  std::vector<Job> jobs;

  void SetChild(Bvh2Node *n, int side, int32_t ref, const Box3 &box) const {
    float *dst = side == 0 ? n->lbox : n->rbox;
    for (int a = 0; a < 3; a++) {
      dst[a] = RoundDown(box.lo[a] - pad);
      dst[3 + a] = RoundUp(box.hi[a] + pad);
    }
    (side == 0 ? n->left : n->right) = ref;
  }

  // Builds ids[b, e) into *out; ranges of at most `grain` triangles become jobs when jobs_out is given.
  // Returns the child reference (>= 0 inner node, < 0 leaf) and the FP64 union box.
  int32_t Build(std::vector<Bvh2Node> *out, int32_t b, int32_t e, int32_t depth, Box3 *box, int32_t *deepest, int32_t grain,
                int32_t parent, int side) {
    if (grain > 0 && e - b <= grain && parent >= 0) {
      Job j;
      j.b = b;
      j.e = e;
      j.depth = depth;
      j.parent = parent;
      j.side = side;
      jobs.push_back(std::move(j));
      return 0;  // patched when the job is done
    }
    double clo[3], chi[3];
    const bool wide = grain > 0 && e - b >= kParallelRange;  // (only the calling thread's top of the tree has grain > 0)
    if (wide) {
      ParallelRangeBounds(tri_box, ids, b, e, par_threads, box, clo, chi);
    } else {
      RangeBounds(tri_box, ids, b, e, box, clo, chi);
    }
    if (depth > *deepest) *deepest = depth;
    if (e - b <= kSceneBvhLeafSize) return ~(int32_t)(((uint32_t)b << 3) | (uint32_t)(e - b));
    const int32_t me = (int32_t)out->size();
    out->emplace_back();
    memset(&out->back(), 0, sizeof(Bvh2Node));
    const int32_t mid = wide && depth < 40 ? ParallelSahPartition(tri_box, ids, scratch, b, e, clo, chi, par_threads)
                                           : SahPartition(tri_box, ids, b, e, clo, chi, depth >= 40);
    Box3 lb, rb;
    const int32_t l = Build(out, b, mid, depth + 1, &lb, deepest, grain, me, 0);
    const int32_t r = Build(out, mid, e, depth + 1, &rb, deepest, grain, me, 1);
    // (a deferred child leaves garbage here; it is overwritten when its job is merged)
    SetChild(&(*out)[(size_t)me], 0, l, lb);
    SetChild(&(*out)[(size_t)me], 1, r, rb);
    return me;
  }

  void Run(std::vector<Bvh2Node> *out, int32_t n) {
    unsigned n_threads = std::thread::hardware_concurrency();
    if (n_threads == 0) n_threads = 1;
    if (n_threads > 32) n_threads = 32;
    // (the grain does not depend on the thread count: the tree must not either)
    const int32_t grain = n >= 65536 ? std::max<int32_t>(4096, n / 256) : 0;
    par_threads = n_threads;
    Box3 whole;
    for (int a = 0; a < 3; a++) whole.lo[a] = whole.hi[a] = 0.0;
    Build(out, 0, n, 0, &whole, &max_depth, grain, -1, 0);
    if (jobs.empty()) return;
    std::atomic<size_t> next(0);
    auto worker = [&]() {
      for (;;) {
        const size_t k = next.fetch_add(1);
        if (k >= jobs.size()) return;
        Job &j = jobs[k];
        j.deepest = j.depth;
        j.ref = Build(&j.nodes, j.b, j.e, j.depth, &j.box, &j.deepest, 0, -1, 0);
      }
    };
    std::vector<std::thread> pool;
    for (unsigned t = 1; t < n_threads; t++) pool.emplace_back(worker);
    worker();
    for (std::thread &t : pool) t.join();
    for (Job &j : jobs) {
      const int32_t base = (int32_t)out->size();
      for (Bvh2Node nd : j.nodes) {
        if (nd.left >= 0) nd.left += base;
        if (nd.right >= 0) nd.right += base;
        out->push_back(nd);
      }
      SetChild(&(*out)[(size_t)j.parent], j.side, j.ref >= 0 ? j.ref + base : j.ref, j.box);
      if (j.deepest > max_depth) max_depth = j.deepest;
    }
    jobs.clear();
  }
};

}  // namespace

int BuildFlatScene(const mtb_triangle *tris, int64_t n, bool use_list_bvh, SceneBvhMode scene_bvh, FlatScene *out,
                   std::string *err) {
  const bool use_scene_bvh = scene_bvh != kSceneBvhNone;
  if (n < 0 || n > 0x3fffffff) {
    *err = "triangle count out of range";
    return MTB_ERR_ARG;
  }
  std::vector<Box3> tri_box((size_t)n);
  std::vector<BuildNode> nodes(1);
  for (int a = 0; a < 3; a++) nodes[0].box.lo[a] = nodes[0].box.hi[a] = 0.0;
  nodes[0].list.resize((size_t)n);
  for (int64_t i = 0; i < n; i++) {
    Box3 &b = tri_box[(size_t)i];
    const double *v = tris[i].vertex;
    for (int a = 0; a < 3; a++) {
      // std::min(a, b) = (b < a) ? b : a and std::max(a, b) = (a < b) ? b : a (aabb.cc:42-47)
      double lo = v[a], hi = v[a];
      for (int k = 1; k < 3; k++) {
        const double x = v[k * 3 + a];
        lo = (x < lo) ? x : lo;
        hi = (hi < x) ? x : hi;
      }
      b.lo[a] = lo;
      b.hi[a] = hi;
      nodes[0].box.lo[a] = (lo < nodes[0].box.lo[a]) ? lo : nodes[0].box.lo[a];
      nodes[0].box.hi[a] = (nodes[0].box.hi[a] < hi) ? hi : nodes[0].box.hi[a];
    }
    nodes[0].list[(size_t)i] = (int32_t)i;
  }
  out->max_tri_extent = 0.0;
  for (const Box3 &b : tri_box) {
    for (int a = 0; a < 3; a++) out->max_tri_extent = std::max(out->max_tri_extent, b.hi[a] - b.lo[a]);
  }
  out->depth = 0;
  const bool timing = getenv("MTB_TIMING") != nullptr;
  auto t0 = std::chrono::steady_clock::now();
  auto lap = [&](const char *what, double *record) {
    const auto t1 = std::chrono::steady_clock::now();
    const double ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
    if (timing) fprintf(stderr, "[mtb] %-28s %8.1f ms\n", what, ms);
    if (record != nullptr) *record = ms;
    t0 = t1;
  };
  const auto t_build0 = std::chrono::steady_clock::now();
  out->max_abs_coord = 0.0;
  for (int a = 0; a < 3; a++) {
    out->aabb[a] = nodes[0].box.lo[a];
    out->aabb[3 + a] = nodes[0].box.hi[a];
    out->max_abs_coord = std::max(out->max_abs_coord, std::max(std::fabs(nodes[0].box.lo[a]), std::fabs(nodes[0].box.hi[a])));
  }

  // ---- scene BVH of the certified fast traversal, part 1: references and (host build) the tree.  It needs nothing
  // of the octree, so on big scenes it runs on its own thread while the octree is split and flattened below. ----
  out->gnodes.clear();
  out->gslots.clear();
  out->gbvh_depth = 0;
  out->ref_box.clear();
  out->ref_slot.clear();
  out->n_split_refs = 0;
  out->bvh_pad = 0x1p-16 * out->max_abs_coord * 1.000001;
  std::vector<Box3> ref_box;
  std::vector<int32_t> ref_tri;
  SceneBvhBuilder sb{ref_box, {}, 0, out->bvh_pad, {}};
  double ms_tree = 0.0;
  auto build_tree = [&]() {
    const auto tt0 = std::chrono::steady_clock::now();
    // references: one per triangle, several for triangles much larger than the scene's grain (see SplitTriangle)
    {
      double scene_ext = 0.0;
      for (int a = 0; a < 3; a++) scene_ext = std::max(scene_ext, out->aabb[3 + a] - out->aabb[a]);
      const char *env = getenv("MTB_SPLIT_DIV");  // development knob: pieces of at most scene extent / div (0: no splitting)
      const double div = env != nullptr ? atof(env) : 64.0;  // measured on C4 (B200): 16 -> 20.8 ms, 32 -> 12.1, 64 -> 7.6 (no splitting: 438)
      double max_extent = div > 0.0 ? scene_ext / div : INFINITY;
      const double guard = 1e-9 * std::max(out->max_abs_coord, 1e-30);
      for (int attempt = 0; attempt < 8; attempt++) {
        ref_box.clear();
        ref_tri.clear();
        ref_box.reserve((size_t)n + (size_t)n / 4);
        ref_tri.reserve((size_t)n + (size_t)n / 4);
        for (int64_t i = 0; i < n; i++) {
          const Box3 &tb = tri_box[(size_t)i];
          const double dx = tb.hi[0] - tb.lo[0], dy = tb.hi[1] - tb.lo[1], dz = tb.hi[2] - tb.lo[2];
          const double ext = std::max(std::max(dx, dy), dz);
          // Only boxes that are mostly empty are worth several references: a long triangle that runs diagonally
          // through its box (area far below the box's cross sections).  A big axis-aligned wall triangle fills half
          // of its flat box; splitting those only deepens the tree (measured on C3: +4 % node visits, no gain).
          bool wasteful = false;
          if (ext > max_extent) {
            const double *v = tris[i].vertex;
            const double e1[3] = {v[3] - v[0], v[4] - v[1], v[5] - v[2]}, e2[3] = {v[6] - v[0], v[7] - v[1], v[8] - v[2]};
            const double cx = e1[1] * e2[2] - e1[2] * e2[1], cy = e1[2] * e2[0] - e1[0] * e2[2], cz = e1[0] * e2[1] - e1[1] * e2[0];
            const double tri_area = 0.5 * std::sqrt(cx * cx + cy * cy + cz * cz);
            wasteful = tri_area < 0.125 * (dx * dy + dy * dz + dz * dx);
          }
          if (!wasteful) {
            ref_box.push_back(tb);
            ref_tri.push_back((int32_t)i);
          } else {
            SplitTriangle(tris[i].vertex, tb, (int32_t)i, max_extent, guard, &ref_box, &ref_tri);
          }
        }
        // budget: at most half as many extra references as there are triangles (+ 4096 for small scenes with big walls)
        if (ref_box.size() <= (size_t)n + (size_t)n / 2 + 4096 && ref_box.size() < 0x0fffffffu) break;
        max_extent *= 2.0;
      }
    }
    const int64_t n_refs = (int64_t)ref_box.size();
    out->n_split_refs = n_refs - n;
    if (scene_bvh == kSceneBvhHost) {
      sb.ids.resize((size_t)n_refs);
      std::iota(sb.ids.begin(), sb.ids.end(), 0);
      Box3 whole;
      if (n_refs <= kSceneBvhLeafSize) {
        // a single leaf: the root holds it as its left child and an empty leaf on the right
        double clo[3], chi[3];
        RangeBounds(ref_box, sb.ids, 0, (int32_t)n_refs, &whole, clo, chi);
        Bvh2Node root;
        memset(&root, 0, sizeof(root));
        for (int a = 0; a < 3; a++) {
          root.lbox[a] = root.rbox[a] = RoundDown(whole.lo[a] - sb.pad);
          root.lbox[3 + a] = root.rbox[3 + a] = RoundUp(whole.hi[a] + sb.pad);
        }
        root.left = ~(int32_t)(uint32_t)n_refs;  // first_gslot 0, count n_refs
        root.right = ~0;                         // count 0
        out->gnodes.push_back(root);
      } else {
        sb.Run(&out->gnodes, (int32_t)n_refs);
      }
      out->gbvh_depth = sb.max_depth;
      if (sb.max_depth > kSceneBvhMaxDepth) out->gnodes.clear();
    }
    ms_tree = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tt0).count();
  };
  std::thread tree_thread;
  const bool tree_wanted = use_scene_bvh && n > 0;
  if (tree_wanted && n >= 65536 && std::thread::hardware_concurrency() > 2) tree_thread = std::thread(build_tree);
  struct Joiner {  // (an error return below must not leave the thread running)
    std::thread *t;
    ~Joiner() {
      if (t->joinable()) t->join();
    }
  } joiner{&tree_thread};

  const int rc = SplitAll(tri_box, &nodes, &out->depth, err);
  if (rc != MTB_OK) return rc;
  lap("octree (AttemptSplit)", &out->ms_octree);

  // ---- flatten ----
  out->nodes.assign(nodes.size(), NodeRec{});
  out->slots.assign((size_t)n, SlotRec{});
  out->shade.assign((size_t)n, ShadeRec{});
  out->list_order.assign((size_t)n, 0);
  out->slot_node.assign((size_t)n, 0);
  out->bvh.clear();
  out->root_list = (int64_t)nodes[0].list.size();
  out->biggest_list = 0;
  out->interior = 0;
  std::vector<int32_t> slot_of((size_t)n, -1);
  // Every node's list is independent (its slots, its list-BVH), so the nodes are handed out in batches to a pool of
  // threads; each thread builds its list-BVHs into its own arena, and the arenas are stitched together in node
  // order afterwards (record indices rebased), so the result does not depend on the number of threads.
  std::vector<int32_t> cursor_of(nodes.size() + 1, 0);
  for (size_t i = 0; i < nodes.size(); i++) {
    cursor_of[i + 1] = cursor_of[i] + (int32_t)nodes[i].list.size();
    out->biggest_list = std::max<int64_t>(out->biggest_list, (int64_t)nodes[i].list.size());
    if (nodes[i].first_child >= 0) out->interior += (int64_t)nodes[i].list.size();
  }
  struct Piece {
    int32_t thread = -1, offset = 0, count = 0;  // this node's list-BVH records inside the thread's arena
  };
  std::vector<Piece> piece(nodes.size());
  unsigned n_threads = std::thread::hardware_concurrency();
  if (n_threads == 0) n_threads = 1;
  if (n_threads > 32) n_threads = 32;
  if (n < 20000) n_threads = 1;
  std::vector<std::vector<BvhRec>> arena(n_threads);
  std::atomic<size_t> next_batch(0);
  constexpr size_t kBatch = 64;
  auto flatten_worker = [&](unsigned tid) {
    BvhBuilder bb{tri_box, &arena[tid], {}, 0};
    for (;;) {
      const size_t first = next_batch.fetch_add(kBatch);
      if (first >= nodes.size()) return;
      const size_t last = std::min(nodes.size(), first + kBatch);
      for (size_t i = first; i < last; i++) {
        const BuildNode &bn = nodes[i];
        NodeRec &nr = out->nodes[i];
        memset(&nr, 0, sizeof(nr));
        for (int a = 0; a < 3; a++) {
          nr.planes[a] = bn.box.lo[a];
          nr.planes[3 + a] = bn.c[a];
          nr.planes[6 + a] = bn.box.hi[a];
        }
        const int32_t cursor = cursor_of[i];
        nr.first_child = bn.first_child;
        nr.list_first = cursor;
        nr.list_count = (int32_t)bn.list.size();
        nr.bvh_root = -1;
        nr.bvh_end = -1;
        const std::vector<int32_t> *order = &bn.list;
        if (use_list_bvh && nr.list_count >= kBvhMinList) {
          bb.ids = bn.list;
          bb.slot_base = cursor;
          piece[i].thread = (int32_t)tid;
          piece[i].offset = (int32_t)arena[tid].size();
          bb.Build(0, nr.list_count);
          piece[i].count = (int32_t)arena[tid].size() - piece[i].offset;
          order = &bb.ids;
        }
        for (int32_t k = 0; k < nr.list_count; k++) {
          const int32_t t = (*order)[(size_t)k];
          const int32_t sidx = cursor + k;
          slot_of[(size_t)t] = sidx;
          out->slot_node[(size_t)sidx] = (int32_t)i;
          SlotRec &sr = out->slots[(size_t)sidx];
          for (int a = 0; a < 3; a++) {
            sr.box[a] = tri_box[(size_t)t].lo[a];
            sr.box[3 + a] = tri_box[(size_t)t].hi[a];
          }
          memcpy(sr.vert, tris[t].vertex, sizeof(sr.vert));
          sr.tri = t;
          sr.canon = sidx;
          ShadeRec &sh = out->shade[(size_t)sidx];
          memcpy(sh.normal, tris[t].normal, sizeof(sh.normal));
          for (int v = 0; v < 3; v++) {
            sh.uv[v * 2 + 0] = tris[t].uvw[v * 3 + 0];
            sh.uv[v * 2 + 1] = tris[t].uvw[v * 3 + 1];
          }
          sh.material = tris[t].material;
          sh.line_no = tris[t].line_no;
        }
        for (int32_t k = 0; k < nr.list_count; k++) out->list_order[(size_t)(cursor + k)] = slot_of[(size_t)bn.list[(size_t)k]];
      }
    }
  };
  {
    std::vector<std::thread> pool;
    for (unsigned t = 1; t < n_threads; t++) pool.emplace_back(flatten_worker, t);
    flatten_worker(0);
    for (std::thread &t : pool) t.join();
  }
  size_t total_records = 0;
  for (const std::vector<BvhRec> &a : arena) total_records += a.size();
  out->bvh.reserve(total_records);
  for (size_t i = 0; i < nodes.size(); i++) {
    const Piece &pc = piece[i];
    if (pc.thread < 0) continue;
    NodeRec &nr = out->nodes[i];
    const int32_t base = (int32_t)out->bvh.size();
    nr.bvh_root = base;
    for (int32_t k = 0; k < pc.count; k++) {
      BvhRec rec = arena[(size_t)pc.thread][(size_t)(pc.offset + k)];
      rec.skip = rec.skip - pc.offset + base;
      out->bvh.push_back(rec);
    }
    nr.bvh_end = (int32_t)out->bvh.size();
    nr.root_rec = out->bvh[(size_t)base];
  }
  // subtree occupancy, children always have larger indices than their parent
  std::vector<int64_t> subtree(nodes.size(), 0);
  for (size_t i = nodes.size(); i-- > 0;) {
    int64_t total = (int64_t)nodes[i].list.size();
    uint32_t mask = 0;
    if (nodes[i].first_child >= 0) {
      for (int k = 0; k < 8; k++) {
        const int64_t sub = subtree[(size_t)nodes[i].first_child + k];
        if (sub > 0) mask |= 1u << k;
        total += sub;
      }
    }
    out->nodes[i].child_mask = mask;
    subtree[i] = total;
  }

  lap("flatten + list BVHs", &out->ms_flatten);
  // ---- scene BVH, part 2: what needs both the tree and the slot order of the octree lists ----
  if (tree_wanted) {
    if (tree_thread.joinable()) {
      tree_thread.join();
    } else {
      build_tree();
    }
    const int64_t n_refs = (int64_t)ref_box.size();
    if (scene_bvh == kSceneBvhRefs) {
      out->ref_box.resize((size_t)n_refs * 6);
      out->ref_slot.resize((size_t)n_refs);
      for (int64_t r = 0; r < n_refs; r++) {
        for (int a = 0; a < 3; a++) {
          out->ref_box[(size_t)r * 6 + a] = ref_box[(size_t)r].lo[a];
          out->ref_box[(size_t)r * 6 + 3 + a] = ref_box[(size_t)r].hi[a];
        }
        out->ref_slot[(size_t)r] = slot_of[(size_t)ref_tri[(size_t)r]];
      }
    } else if (!out->gnodes.empty()) {
      out->gslots.resize((size_t)n_refs);
      ParallelSlices(0, (int32_t)n_refs, n_refs >= 65536 ? sb.par_threads : 1u, [&](unsigned, int32_t sb_, int32_t se_) {
        for (int32_t i = sb_; i < se_; i++) out->gslots[(size_t)i] = out->slots[(size_t)slot_of[(size_t)ref_tri[(size_t)sb.ids[(size_t)i]]]];
      });
    }
  }
  if (timing && !out->gnodes.empty()) {
    auto harea = [](const float *b) {
      const double dx = (double)b[3] - b[0], dy = (double)b[4] - b[1], dz = (double)b[5] - b[2];
      return dx * dy + dy * dz + dz * dx;
    };
    double root = 0.0, inner = 0.0, leaf = 0.0;
    {
      float rb[6];
      for (int a = 0; a < 3; a++) {
        rb[a] = std::min(out->gnodes[0].lbox[a], out->gnodes[0].rbox[a]);
        rb[3 + a] = std::max(out->gnodes[0].lbox[3 + a], out->gnodes[0].rbox[3 + a]);
      }
      root = harea(rb);
    }
    for (const Bvh2Node &g : out->gnodes) {
      for (int side = 0; side < 2; side++) {
        const int32_t ref = side == 0 ? g.left : g.right;
        const double ar = harea(side == 0 ? g.lbox : g.rbox);
        if (ref >= 0) {
          inner += ar;
        } else {
          leaf += ar * (double)((~(uint32_t)ref) & 7u);
        }
      }
    }
    fprintf(stderr, "[mtb] scene BVH SAH: expected node visits %.2f, expected triangle tests %.2f per random ray\n",
            1.0 + inner / root, leaf / root);
  }
  lap(scene_bvh == kSceneBvhRefs ? "scene BVH references (join)" : "scene BVH (join + leaf records)", &out->ms_scene_bvh);
  out->ms_scene_bvh_thread = ms_tree;
  out->ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_build0).count();
  if (timing) fprintf(stderr, "[mtb] %-28s %8.1f ms (on its own thread, overlapping the octree stages)\n", "  scene BVH tree build", ms_tree);
  return MTB_OK;
}

// ---------------------------------------------------------------------------------------------------
// Camera::GetSensor / Sensor::Reset (camera.cc:17-63).  Matrix products keep the reference's operand
// order and left-to-right sums (math3d.h:188-216) so the three vectors come out bit-identical.
// ---------------------------------------------------------------------------------------------------
namespace {

struct Mat4 {
  double m[4][4];
};

Mat4 Mul(const Mat4 &a, const Mat4 &b) {
  Mat4 r;
  for (int j = 0; j < 4; j++) {
    for (int i = 0; i < 4; i++) {
      r.m[j][i] = a.m[j][0] * b.m[0][i] + a.m[j][1] * b.m[1][i] + a.m[j][2] * b.m[2][i] + a.m[j][3] * b.m[3][i];
    }
  }
  return r;
}

void Apply(const Mat4 &a, const double in[3], double out[3]) {
  // math3d.h:210-216 adds m[0][3] to every row; it is always 0 for rotations.
  const double x = in[0], y = in[1], z = in[2];
  out[0] = a.m[0][0] * x + a.m[0][1] * y + a.m[0][2] * z + a.m[0][3];
  out[1] = a.m[1][0] * x + a.m[1][1] * y + a.m[1][2] * z + a.m[0][3];
  out[2] = a.m[2][0] * x + a.m[2][1] * y + a.m[2][2] * z + a.m[0][3];
}

double Rad(double deg) { return (deg * M_PI) / 180.0; }

Mat4 RotX(double deg) {
  const double a = Rad(deg);
  return Mat4{{{1.0, 0.0, 0.0, 0.0}, {0.0, cos(a), -sin(a), 0.0}, {0.0, sin(a), cos(a), 0.0}, {0.0, 0.0, 0.0, 1.0}}};
}
Mat4 RotY(double deg) {
  const double a = Rad(deg);
  return Mat4{{{cos(a), 0.0, sin(a), 0.0}, {0.0, 1.0, 0.0, 0.0}, {-sin(a), 0.0, cos(a), 0.0}, {0.0, 0.0, 0.0, 1.0}}};
}
Mat4 RotZ(double deg) {
  const double a = Rad(deg);
  return Mat4{{{cos(a), -sin(a), 0.0, 0.0}, {sin(a), cos(a), 0.0, 0.0}, {0.0, 0.0, 1.0, 0.0}, {0.0, 0.0, 0.0, 1.0}}};
}

// The camera's rotation (camera.cc:48-51): the one matrix both the pinhole sensor and the panorama basis turn by.
Mat4 Aim(const mtb_camera &cam) { return Mul(Mul(RotY(cam.yaw), RotX(cam.pitch)), RotZ(cam.roll)); }

}  // namespace

void ComputeSensor(const mtb_camera &cam, int image_w, int image_h, double out9[9]) {
  const double vertical = (double(image_h) / double(image_w)) * cam.aov;  // camera.cc:29
  const Mat4 left = RotY(cam.aov / 2.0), right = RotY(-cam.aov / 2.0);
  const Mat4 top = RotZ(vertical / 2.0), bottom = RotZ(-vertical / 2.0);
  const Mat4 corner_tl = Mul(top, left);
  const Mat4 corner_tr = Mul(bottom, right);  // the reference pairs "right" with the bottom rotation (camera.cc:38)
  const Mat4 corner_bl = Mul(bottom, left);
  const double fwd[3] = {0.0, 0.0, 1.0};
  double tl[3], tr[3], bl[3];
  Apply(corner_tl, fwd, tl);
  Apply(corner_tr, fwd, tr);
  Apply(corner_bl, fwd, bl);
  const Mat4 aim = Aim(cam);
  Apply(aim, tl, tl);
  Apply(aim, tr, tr);
  Apply(aim, bl, bl);
  for (int a = 0; a < 3; a++) {
    out9[a] = tl[a];                                  // start_point
    out9[3 + a] = (bl[a] - tl[a]) / double(image_h);  // delta_scanline
    out9[6 + a] = (tr[a] - tl[a]) / double(image_w);  // delta_pixel
  }
}

void ComputePanoramaBasis(const mtb_camera &cam, double forward[3], double right[3], double up[3]) {
  const Mat4 aim = Aim(cam);
  const double f[3] = {0.0, 0.0, 1.0}, r[3] = {-1.0, 0.0, 0.0}, u[3] = {0.0, 1.0, 0.0};
  Apply(aim, f, forward);
  Apply(aim, r, right);
  Apply(aim, u, up);
}

}  // namespace mtb
