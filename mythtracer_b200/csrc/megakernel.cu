// RenderMega (per-pixel megakernel) and the batched intersect kernel; see device_core.cuh for the traversal.
#include <type_traits>

#include "device_core.cuh"

namespace mtb {
namespace {

// One suspended TraceRayWorker activation waiting for its reflection / refraction child.
struct ShadeFrame {
  double color[3];
  double point[3];
  double dir[3];  // ray.direction of this activation (the refraction child continues along it)
  double coef;    // current_reflection_coef
  unsigned long long path;
  int material;
  unsigned char stage;  // 0: reflection child pending, 1: refraction child pending
  unsigned char do_refract;
  unsigned char in_object;
  unsigned char pad_;
};

// Everything of a pixel that has to survive a traversal, in the thread's local memory.
//
// Round 1 kept this state in C++ variables under a 64-register cap, and the register allocator spread 1.3 KB of
// spill stores and 1.4 KB of spill loads over every ray (ncu: 57 % of the kernel's L1 sectors were local memory,
// 5.4 GB of DRAM writes per frame for 6 MB of output).  Here the placement is explicit: the traversal runs with
// little more than its own registers live, and what the shading code needs afterwards is loaded where it is used - a
// shadow ray that misses reads ~20 doubles and writes 3, instead of the whole state going out and coming back.
// MTB_STATE_BARRIER() makes the struct's address escape through an empty asm with a memory clobber, so the compiler
// can neither promote it to registers (and spill it again) nor carry loaded values across the Trace call.
struct alignas(16) PixelState {
  double m_o[3], m_d[3];                                         // ray of the current activation
  double P[3], normal[3], surface[3], reflected[3], color[3];    // its shading context (mythtracer.cc:38-76)
  double ldir[3], seg_start[3], power[3];                        // shadow walk of the current light (mythtracer.cc:86-156)
  double coef;                                                   // current_reflection_coef
  double light_distance;                                         // of the shadow segment in flight (mythtracer.cc:101-102)
  unsigned long long path, sig_hits, sig_shadow;
  // small integers that are only touched between two traversals (a register each across the node loop would push
  // the FP32 ray of TraceFast into spill slots at 64 registers)
  int level, li, material;
  unsigned segments, n_rays;
};
#define MTB_STATE_BARRIER() asm volatile("" : : "l"(&st) : "memory")

// ---------------------------------------------------------------------------------------------------
// RenderMega: one thread = one pixel = the whole TraceRay recursion, evaluated in the reference's
// post-order so that colour sums associate identically.  Every loop iteration issues exactly one
// OctTree::IntersectRay-equivalent query (a primary / reflection / refraction ray or one shadow segment),
// so the lanes of a warp reconverge at the single Trace call site.  One block = one 8x8 pixel tile (a warp =
// 8x4 pixels); a finished warp writes its 4 rows as 12 aligned 8-byte stores (the frame buffer may be the
// peer-mapped frame of another GPU, api.cu) and exits without waiting for the other warp.
//
// Retired launch forms of round 1, all bit-identical and all measured slower on B200 (DESIGN.md section 5):
// persistent lane refill, block-level ray packing, forced warp re-convergence, suspendable walks.
// ---------------------------------------------------------------------------------------------------
#ifndef MTB_MEGA_MIN_BLOCKS
// Blocks per SM = registers per thread.  The frame time falls with every warp in flight as long as the node loop of
// TraceFast stays free of spill code (B200, C3, ms): 10 blocks (96 registers) 10.50, 12 (80) 9.66, 14 (72) 9.07 - and,
// once the FP32 ray's live range was split by hand (TraceFast, device_core.cuh) and the small per-pixel integers
// moved into PixelState, so that 64 registers no longer put reloads into the node loop - 16 (64) 8.88, 18 (56) 9.00,
// 20 (48) 9.14.  With the leaf's FP64 ray read from shared memory at each use (fewer leaf spills below 64 registers;
// DESIGN.md section 5): 16 8.83, 20 8.83, 24 (40) 9.32 - the optimum is not set by the leaf spills alone.
#define MTB_MEGA_MIN_BLOCKS 16
#endif

constexpr unsigned kShadowMode = 1u, kInObject = 2u, kInShadow = 4u, kThrough = 8u;

// The lights of this block's view.  A batch launch (BATCH) renders view blockIdx.y with lights
// sc.lights[blockIdx.y * n_lights ..]; blockIdx.y is re-read at every use, so nothing per view stays live in a register
// across a traversal.
template <bool BATCH>
__device__ __forceinline__ const mtb_light *ViewLights(const DeviceScene &sc) {
  return BATCH ? sc.lights + (size_t)blockIdx.y * sc.n_lights : sc.lights;
}
// ... and where its pixels go (view-major frames of chunk_w x chunk_h RGB24).
template <bool BATCH>
__device__ __forceinline__ uint8_t *ViewFrame(const RenderParams &rp) {
  return BATCH ? rp.rgb + (size_t)blockIdx.y * rp.chunk_w * rp.chunk_h * 3 : rp.rgb;
}
// ... and the entry of pixel (px, py) in its debug and tap planes (view-major planes of chunk_w x chunk_h entries: for a
// supersampled batch, the sample grid).
template <bool BATCH>
__device__ __forceinline__ size_t PlaneIndex(const RenderParams &rp, int px, int py) {
  return (BATCH ? (size_t)blockIdx.y * rp.chunk_w * rp.chunk_h : 0) + (size_t)py * rp.chunk_w + px;
}

// Averaged batch: the output pixel is the rounded mean of n quantised samples.
//
// Supersampled (SS = 2, 4, 8 samples per axis): the tile is a tile of the (SS*W) x (SS*H) sample grid (rp.chunk_w x
// rp.chunk_h), every thread traces one sample exactly as a pixel of that frame, and the epilogue writes the (8/SS)^2
// output pixels of the tile, each the mean of its SS x SS samples, to view-major W x H frames.  W = chunk_w / SS: the
// sample grid's sides are multiples of SS, so an output pixel inside the frame has all its samples live, and its SS x SS
// block never straddles a tile (SS divides 8).
//
// Accumulated (ACC, SS = 1, 2, 4, 8): block row u traces sub-frame u of output view v = u / k exactly as view u of a
// batch, and the output pixel is the mean of all k * SS * SS samples of its k sub-frames.  Every warp adds the
// per-output-channel sums of its half tile (SS = 8: the warp that finishes second, for the whole tile) into acc.sum of
// view v, fences, and bumps the arrival counter of (v, tile, warp half).  The warp whose arrival is the k-th reads the
// completed sums from L2 and stores the bytes.  The sums are integers, so the bytes do not depend on the order in which
// the sub-frames finish.
//
// No block barrier after the trace, for the reason of the plain epilogue (RenderMega).  SS = 1, 2 and 4: a warp (8x4
// samples) holds whole blocks, so the sum stays warp-level like the plain epilogue.
// SS = 8: the one output pixel of a tile spans both warps.  Each warp reduces its 32 samples with shuffles; the warp
// that finishes first leaves its partial sums in shared memory and exits, the last one adds them and finishes the pixel.
// A block barrier there instead holds the first warp's slot until the other is done: 1.3 % more kernel time for 16 C3
// views at 240x135 (B200, DESIGN.md section 13).
template <int SS, bool ACC>
__device__ __forceinline__ void AverageEpilogue(const RenderParams &rp, const AccumParams &acc, const unsigned char *s_rgb, int tile_id,
                                                int strip, unsigned *s_ss8) {
  const int out_w = rp.chunk_w / SS, out_h = rp.chunk_h / SS;
  const unsigned view = ACC ? blockIdx.y / (unsigned)acc.subframes : blockIdx.y;
  const size_t view_base = (size_t)view * out_w * out_h * 3;
  uint32_t *const sum = acc.sum + view_base;
  uint8_t *const frame = rp.rgb + view_base;
  const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const unsigned n = (ACC ? (unsigned)acc.subframes : 1u) * (SS * SS);
  uint32_t *const arrive = acc.arrive + ((size_t)view * gridDim.x + tile_id) * 2;
  if constexpr (SS == 8) {
    // the tile is one output pixel, and every sample of it is live (tiles_x = W, 8 rows of tiles per output row)
    const unsigned char *mine = s_rgb + threadIdx.x * 3;
    unsigned r = mine[0], g = mine[1], b = mine[2];
    for (int off = 16; off > 0; off >>= 1) {
      r += __shfl_down_sync(0xffffffffu, r, off);
      g += __shfl_down_sync(0xffffffffu, g, off);
      b += __shfl_down_sync(0xffffffffu, b, off);
    }
    // s_ss8: [0] warps done (zeroed before the trace), [1 + 3 * warp ..] that warp's three sums
    volatile unsigned *part = s_ss8 + 1;
    if (lane != 0u) return;
    part[warp * 3 + 0] = r;
    part[warp * 3 + 1] = g;
    part[warp * 3 + 2] = b;
    __threadfence_block();
    if (atomicAdd(s_ss8, 1u) != 1u) return;  // the other warp's sums are not in place yet
    __threadfence_block();
    const unsigned o = (warp ^ 1u) * 3;
    const size_t at = (size_t)tile_id * 3;  // tile (x, y) = output pixel (x, y): tiles_x = out_w
    if constexpr (ACC) {
      atomicAdd(sum + at + 0, r + part[o + 0]);
      atomicAdd(sum + at + 1, g + part[o + 1]);
      atomicAdd(sum + at + 2, b + part[o + 2]);
      __threadfence();
      if (atomicAdd(arrive, 1u) != (unsigned)acc.subframes - 1u) return;
      __threadfence();
      for (int c = 0; c < 3; c++) frame[at + c] = (uint8_t)((__ldcg(sum + at + c) + n / 2) / n);
    } else {
      frame[at + 0] = (uint8_t)((r + part[o + 0] + n / 2) / n);
      frame[at + 1] = (uint8_t)((g + part[o + 1] + n / 2) / n);
      frame[at + 2] = (uint8_t)((b + part[o + 2] + n / 2) / n);
    }
  } else {
    // the output channels this lane owns: SS = 1, the 3 of its own pixel; SS = 2, 4, one of the warp's (8/SS) x (4/SS)
    // output pixels (lane = 3 * pixel + channel)
    constexpr int kPer = SS == 1 ? 3 : 1;
    long long at = -1;  // this lane's first channel in the view's frame; -1: none
    unsigned val[kPer];
    if constexpr (SS == 1) {
      const int tx = (int)(threadIdx.x & 7u), ty = (int)(threadIdx.x >> 3);
      const int px = (tile_id % rp.tiles_x) * kTile + tx, py = strip * kTile + ty;
      if (px < out_w && py < out_h) {
        at = ((long long)py * out_w + px) * 3;
        const unsigned char *src = s_rgb + ((ty * kTile) + tx) * 3;
        for (int c = 0; c < 3; c++) val[c] = src[c];
      }
    } else {
      constexpr int kCols = kTile / SS, kRows = 4 / SS;
      if (lane < (unsigned)(kCols * kRows * 3)) {
        const int k = (int)lane / 3, c = (int)lane % 3, i = k % kCols, j = k / kCols;
        const int ox = (tile_id % rp.tiles_x) * kCols + i, oy = (strip * kTile + (int)warp * 4) / SS + j;
        if (ox < out_w && oy < out_h) {
          at = ((long long)oy * out_w + ox) * 3 + c;
          const unsigned char *src = s_rgb + warp * (4 * kTile * 3) + (j * SS * kTile + i * SS) * 3 + c;
          unsigned s = 0;
#pragma unroll
          for (int a = 0; a < SS; a++) {
#pragma unroll
            for (int b = 0; b < SS; b++) s += src[(a * kTile + b) * 3];
          }
          val[0] = s;
        }
      }
    }
    if (at < 0 && !ACC) return;  // (an accumulating lane without a channel still takes part in the warp's arrival)
    if constexpr (ACC) {
      if (at >= 0) {
        for (int c = 0; c < kPer; c++) atomicAdd(sum + at + c, val[c]);
      }
      __threadfence();
      __syncwarp();
      unsigned last = 0u;
      if (lane == 0u) last = atomicAdd(arrive + warp, 1u) == (unsigned)acc.subframes - 1u ? 1u : 0u;
      if (__shfl_sync(0xffffffffu, last, 0) == 0u) return;
      __threadfence();
    }
    if (at >= 0) {
      for (int c = 0; c < kPer; c++) frame[at + c] = (uint8_t)(((ACC ? __ldcg(sum + at + c) : val[c]) + n / 2) / n);
    }
  }
}

// BATCH: grid (tiles per view, views), block b of row v renders tile b of view v in scanline order; the camera comes from
// views[v] and the pixels go to rp.rgb + v * chunk_w * chunk_h * 3.  A batch launch passes NULL for tile_order,
// tile_cost and run_if; its debug and tap planes (NULL unless the caller asked for them) are view-major, view v's entries
// start at v * chunk_w * chunk_h (PlaneIndex).  Without BATCH, `views` is unused and every `BATCH ? :`
// folds away: the single-view kernels compile to the code they had before the batch form existed.  SS > 1 (BATCH only):
// the supersampled batch, see AverageEpilogue; with SS = 1 every `SS` branch folds away.  ACC (BATCH only): the
// accumulated batch, see AverageEpilogue; `acc` is unused without it.  LENS (BATCH only): thin-lens views, the
// primary ray of grid row u starts on the lens point of lens[u] and passes through the focal-plane point of the pinhole
// ray (LensRec); `lens` is unused without it, and only the primary ray differs.  PANO (BATCH only, never with LENS):
// panoramas, the primary ray of sample (X, Y) of grid row u is made from pano.rec[u] and the {cos, sin} entries
// pano.lon[X] and pano.lat[Y] with + * / sqrt only (PanoRec; the host computes the trigonometry, so the rays match
// its restatement bit for bit); `pano` is unused without it, and only the primary ray differs.
// `sc` is __grid_constant__: the exact traversals take it by reference (TraceExactCold is not inlined), and a plain
// by-value parameter whose address is taken is copied to local memory at kernel start (112 B), after which the scene
// pointers (nodes, leaf records, shading records, materials, lights) are loaded from that copy.  A grid constant's
// address points at the parameter bank itself, so the fields are constant-bank operands: C3 8.86 ->
// 8.56 ms, C5 49.1 -> 47.7 ms, C4 7.73-7.79 -> 7.59-7.61 ms (B200, 1000 W, 1965 MHz max SM clock; DESIGN.md section 5).
template <bool DBG, bool BATCH, int SS, bool ACC, bool LENS, bool PANO>
__global__ void __launch_bounds__(kBlockThreads, MTB_MEGA_MIN_BLOCKS) RenderMega(const __grid_constant__ DeviceScene sc, RenderParams rp, const ViewRec *views,
                                                                                 AccumParams acc, const LensRec *lens, PanoParams pano) {
  static_assert(SS == 1 || (BATCH && (SS == 2 || SS == 4 || SS == 8)), "supersampling is a batch form with 2, 4 or 8 samples per axis");
  static_assert(!ACC || BATCH, "accumulation is a batch form");
  static_assert(!LENS || BATCH, "thin-lens views are a batch form");
  static_assert(!PANO || (BATCH && !LENS), "panoramas are a batch form without thin lenses");
  MTB_DECLARE_FAST_CTX(kBlockThreads);
  // (SS = 8: 7 more words behind the samples for the epilogue's counter and partial sums)
  __shared__ __align__(8) unsigned char s_rgb[kTile * kTile * 3 + (SS == 8 ? 7 * 4 : 0)];
  unsigned *const s_ss8 = reinterpret_cast<unsigned *>(s_rgb + kTile * kTile * 3);
  if constexpr (SS == 8) {
    if (threadIdx.x == 0) s_ss8[0] = 0u;
    __syncthreads();  // (both warps start together: unlike a barrier after the trace, this holds nobody's slot)
  }
  // repair launch of a wavefront frame whose activation table did not overflow: nothing to do
  if (rp.run_if != nullptr && __ldg(rp.run_if) == 0u) return;
  unsigned long long cnt_store[DBG ? kNumCounters : 1];
  unsigned long long *cnt = cnt_store;
  if (DBG) {
    for (int i = 0; i < kNumCounters; i++) cnt[i] = 0;
  }

  // block -> 8x8 tile of one of this launch's strips (a strip = 8 image rows; strips are interleaved
  // across devices / processes, the in-box form of the reference's master/worker tiling)
  const int tile_id = rp.tile_order != nullptr ? rp.tile_order[blockIdx.x] : (int)blockIdx.x;
  const int strip = rp.strip_first + (tile_id / rp.tiles_x) * rp.strip_stride;
  const int tx = (int)(threadIdx.x & 7u), ty = (int)(threadIdx.x >> 3);
  const int px = (tile_id % rp.tiles_x) * kTile + tx;
  const int py = strip * kTile + ty;
  const bool live = px < rp.chunk_w && py < rp.chunk_h;
  const bool want_sig = rp.sig_hits != nullptr || rp.sig_shadow != nullptr;
  unsigned n_rays = 0;

  if (live) {
    PixelState st;
    ShadeFrame frames[kMaxRayStack];
    // what stays in registers across a traversal
    int sp = 0;
    unsigned flags = 0;
    st.level = 0;
    st.li = 0;
    st.material = -1;
    st.segments = 0;
    st.n_rays = 0;

    if constexpr (PANO) {  // panorama (PanoRec): longitude X and latitude Y of the sample grid, from the row's basis
      const PanoRec &pr = pano.rec[blockIdx.y];
      const double2 lon = reinterpret_cast<const double2 *>(pano.lon)[rp.chunk_x + px];  // {cos, sin}
      const double2 lat = reinterpret_cast<const double2 *>(pano.lat)[rp.chunk_y + py];
      const D3 fwd = Load3(pr.forward), right = Load3(pr.right);
      Store3(st.m_d, Normalized(Add(MulS(Add(MulS(fwd, lon.x), MulS(right, lon.y)), lat.x), MulS(Load3(pr.up), lat.y))));
      const D3 o = Load3(views[blockIdx.y].origin);
      Store3(st.m_o, pr.eye == 0.0 ? o : Add(o, MulS(Sub(MulS(right, lon.x), MulS(fwd, lon.y)), pr.eye)));
    } else {  // Sensor::GetRay (camera.cc:65-69) with full-image pixel coordinates (mythtracer.cc:298)
      const double *sensor = BATCH ? views[blockIdx.y].sensor : rp.sensor;
      const D3 start = Load3(sensor), d_scan = Load3(sensor + 3), d_pixel = Load3(sensor + 6);
      if constexpr (LENS) {
        // thin lens (LensRec): from O + L towards the point where the pinhole ray d meets the focal plane, O + d * t
        const D3 o = Load3(views[blockIdx.y].origin);
        const D3 d = Normalized(Add(Add(start, MulS(d_scan, (double)(rp.chunk_y + py))), MulS(d_pixel, (double)(rp.chunk_x + px))));
        const LensRec &ln = lens[blockIdx.y];
        if (ln.centred != 0u) {
          Store3(st.m_o, o);
          Store3(st.m_d, d);
        } else {
          const D3 shift = Load3(ln.shift);
          const double t = ln.focus / Dot(d, Load3(ln.axis));
          Store3(st.m_o, Add(o, shift));
          Store3(st.m_d, Normalized(Sub(MulS(d, t), shift)));
        }
      } else {
        Store3(st.m_o, Load3(BATCH ? views[blockIdx.y].origin : rp.origin));
        Store3(st.m_d, Normalized(Add(Add(start, MulS(d_scan, (double)(rp.chunk_y + py))), MulS(d_pixel, (double)(rp.chunk_x + px)))));
      }
    }
    st.coef = 1.0;
    st.path = 1ull;
    st.sig_hits = 0ull;
    st.sig_shadow = 0ull;
    Count<DBG>(cnt, kPrimary);

    for (;;) {
      int slot;
      double t = 0.0;
      {
        D3 to, td;
        double limit = CUDART_INF;
        if (flags & kShadowMode) {
          const D3 seg = Load3(st.seg_start);
          td = Load3(st.ldir);
          to = Add(seg, MulS(td, 0.00001));                                    // mythtracer.cc:95-99
          limit = Dist(seg, Load3(ViewLights<BATCH>(sc)[st.li].position));  // mythtracer.cc:101-102
          st.light_distance = limit;
          Count<DBG>(cnt, kShadow);
        } else {
          to = Load3(st.m_o);
          td = Load3(st.m_d);
        }
        MTB_STATE_BARRIER();
        slot = Trace<DBG>(sc, to, td, limit, &t, cnt, fctx);
        MTB_STATE_BARRIER();
      }
      st.n_rays++;

      bool have_ret = false;
      D3 ret = Mk(0.0, 0.0, 0.0);
      if (flags & kShadowMode) {
        bool light_done = false;
        st.segments++;
        if (slot < 0) {
          light_done = true;  // mythtracer.cc:109-112
        } else if (t > st.light_distance) {
          light_done = true;  // mythtracer.cc:115-118
        } else {
          const int smtl = __ldg(&sc.shade[slot].material);
          // mtl is dereferenced unconditionally upstream (mythtracer.cc:121); a missing material acts opaque
          const double str = smtl >= 0 ? __ldg(&sc.materials[smtl].transparency) : 0.0;
          if (str == 0.0) {
            Store3(st.power, Mk(0.0, 0.0, 0.0));
            flags |= kInShadow;
            light_done = true;
          } else {
            D3 power = Load3(st.power);
            if (!(flags & kThrough)) {  // light_power *= Tf * Tr (mythtracer.cc:129-132)
              const D3 tf = Load3(sc.materials[smtl].transmission_filter);
              power = MulV(power, MulS(tf, str));
              Store3(st.power, power);
            }
            flags ^= kThrough;
            const D3 ldir = Load3(st.ldir);
            const D3 to = Add(Load3(st.seg_start), MulS(ldir, 0.00001));
            const D3 hit_point = Add(to, MulS(ldir, t));                 // primitive_triangle.cc:141
            const D3 seg_start = Add(hit_point, MulS(ldir, 0.0000001));  // mythtracer.cc:137
            Store3(st.seg_start, seg_start);
            const D3 P = Load3(st.P);
            if (SqrDist(P, seg_start) > SqrDist(P, Load3(ViewLights<BATCH>(sc)[st.li].position))) {  // mythtracer.cc:141-145
              light_done = true;
            } else if (power.x <= 0.001 && power.y <= 0.001 && power.z <= 0.001) {
              Store3(st.power, Mk(0.0, 0.0, 0.0));
              flags |= kInShadow;
              light_done = true;
            }
          }
        }
        if (!light_done) continue;  // next segment of the same light

        // ---- this light is settled: Phong terms (mythtracer.cc:159-177) ----
        const mtb_light *lt = ViewLights<BATCH>(sc) + st.li;
        const mtb_material *m = sc.materials + st.material;
        const bool in_shadow = (flags & kInShadow) != 0u;
        if (want_sig) {
          st.sig_shadow += Mix64(st.path, 2ull + (unsigned long long)st.li, (in_shadow ? 1ull : 0ull) | ((unsigned long long)st.segments << 1));
        }
        const D3 lamb = Load3(lt->ambient);
        D3 power = Load3(st.power);
        power.x = SMax(power.x, lamb.x);
        power.y = SMax(power.y, lamb.y);
        power.z = SMax(power.z, lamb.z);
        const D3 surface = Load3(st.surface);
        D3 color = Load3(st.color);
        color = Add(color, MulV(MulV(MulS(MulV(Load3(m->diffuse), surface), Dot(Load3(st.normal), Load3(st.ldir))), Load3(lt->diffuse)), power));
        if (!in_shadow) {
          const double refl_dot = Dot(Neg(Load3(st.m_d)), Load3(st.reflected));
          if (refl_dot > 0) {
            color = Add(color, MulV(MulS(MulV(Load3(m->specular), surface), pow(refl_dot, m->specular_exp)), Load3(lt->specular)));
          }
        }
        Store3(st.color, color);
        st.li++;
      } else {
        // ---- result of a primary / reflection / refraction ray (mythtracer.cc:13-76) ----
        if (slot < 0) {
          if (st.level == 0 && rp.dbg != nullptr) {
            mtb_debug *dbg = rp.dbg + PlaneIndex<BATCH>(rp, px, py);
            dbg->line_no = -1;
            dbg->pad_ = 0;
            dbg->point[0] = dbg->point[1] = dbg->point[2] = CUDART_NAN;
          }
          have_ret = true;  // background colour {0,0,0}
        } else {
          const ShadeRec *sh = sc.shade + slot;
          const SlotRec *sr = sc.slots + slot;
          const D3 m_d = Load3(st.m_d);
          const D3 P = Add(Load3(st.m_o), MulS(m_d, t));
          const int line_no = __ldg(&sh->line_no);
          if (st.level == 0 && rp.dbg != nullptr) {
            mtb_debug *dbg = rp.dbg + PlaneIndex<BATCH>(rp, px, py);
            dbg->line_no = line_no;
            dbg->pad_ = 0;
            dbg->point[0] = P.x;
            dbg->point[1] = P.y;
            dbg->point[2] = P.z;
          }
          if (want_sig) st.sig_hits += Mix64(st.path, 1ull, (unsigned long long)(long long)line_no);
          Count<DBG>(cnt, kShade);
          const D3 v0 = Load3(sr->vert), v1 = Load3(sr->vert + 3), v2 = Load3(sr->vert + 6);
          const BaryWeights w = Barycentric(v0, v1, v2, P);
          // (normal[0]*n0 + normal[1]*n1 + normal[2]*n2) / n, not normalised (primitive_triangle.cc:60)
          D3 normal = DivS(Add(Add(MulS(Load3(sh->normal), w.n0), MulS(Load3(sh->normal + 3), w.n1)), MulS(Load3(sh->normal + 6), w.n2)), w.n);
          const D3 towards_camera = Neg(m_d);
          double normal_ray_dot = Dot(towards_camera, normal);
          if (normal_ray_dot < 0.0) {
            normal = Neg(normal);
            normal_ray_dot = Dot(towards_camera, normal);
          }
          st.material = __ldg(&sh->material);
          if (st.material < 0) {  // mythtracer.cc:49-52
            normal_ray_dot = (normal_ray_dot + 1.0) * 0.5;
            ret = Mk(normal_ray_dot, normal_ray_dot, normal_ray_dot);
            have_ret = true;
          } else {
            const mtb_material *m = sc.materials + st.material;
            D3 surface = Load3(m->ambient);
            const int tex = m->texture;
            if (tex >= 0) {  // mythtracer.cc:59-64
              const double u = (sh->uv[0] * w.n0 + sh->uv[2] * w.n1 + sh->uv[4] * w.n2) / w.n;
              const double v = (sh->uv[1] * w.n0 + sh->uv[3] * w.n1 + sh->uv[5] * w.n2) / w.n;
              surface = MulV(surface, SampleTexture(sc.tex_atlas, tex, sc.texture_dim[tex], u, v));
            }
            Store3(st.P, P);
            Store3(st.normal, normal);
            Store3(st.surface, surface);
            // ray.direction - normal * (2 * ray.direction.Dot(normal)) (mythtracer.cc:68-69)
            Store3(st.reflected, Sub(m_d, MulS(normal, 2 * Dot(normal, m_d))));
            Store3(st.color, Mk(0.0, 0.0, 0.0));
            st.li = 0;
          }
        }
      }

      if (!have_ret) {
        if (st.li < sc.n_lights) {
          // ---- start the shadow walk of light li (mythtracer.cc:79-94) ----
          const mtb_light *lt = ViewLights<BATCH>(sc) + st.li;
          const D3 P = Load3(st.P);
          Store3(st.ldir, Normalized(Sub(Load3(lt->position), P)));
          Store3(st.color, Add(Load3(st.color), MulV(Load3(lt->ambient), Load3(st.surface))));  // mythtracer.cc:83-84
          Store3(st.power, Mk(1.0, 1.0, 1.0));
          Store3(st.seg_start, P);
          flags = (flags & kInObject) | kShadowMode;  // in_shadow = through = false
          st.segments = 0;
          continue;
        }
        // ---- all lights done: secondary rays (mythtracer.cc:181-225) ----
        flags &= kInObject;
        const mtb_material *m = sc.materials + st.material;
        const double refl = m->reflectance, tr = m->transparency;
        const double coef = st.coef;
        const bool in_object = (flags & kInObject) != 0u;
        const bool do_reflect = st.level < rp.max_depth && refl > 0.0 && coef > 0.01 && !in_object;
        const bool do_refract = st.level < rp.max_depth && tr > 0.0;
        if (do_reflect || do_refract) {
          const D3 P = Load3(st.P), m_d = Load3(st.m_d);
          ShadeFrame &f = frames[sp];
          Store3(f.color, Load3(st.color));
          Store3(f.point, P);
          Store3(f.dir, m_d);
          f.coef = coef;
          f.path = st.path;
          f.material = st.material;
          f.stage = do_reflect ? 0 : 1;
          f.do_refract = do_refract ? 1 : 0;
          f.in_object = in_object ? 1 : 0;
          sp++;
          st.level++;
          if (do_reflect) {
            Count<DBG>(cnt, kReflect);
            const D3 reflected = Load3(st.reflected);
            Store3(st.m_o, Add(P, MulS(reflected, 0.0001)));  // mythtracer.cc:70-75
            Store3(st.m_d, reflected);
            st.coef = coef * refl;
            st.path = st.path * 2ull;
          } else {
            Count<DBG>(cnt, kRefract);
            const D3 rdir = Normalized(m_d);           // mythtracer.cc:208-212
            Store3(st.m_o, Add(P, MulS(rdir, 0.00001)));  // mythtracer.cc:214-218
            Store3(st.m_d, rdir);
            flags ^= kInObject;
            st.path = st.path * 2ull + 1ull;
          }
          continue;
        }
        ret = Load3(st.color);
      }

      // ---- an activation returned `ret`: fold it into suspended parents (mythtracer.cc:185-189,220-224) ----
      bool finished = false;
      for (;;) {
        if (sp == 0) {
          finished = true;
          break;
        }
        ShadeFrame &f = frames[sp - 1];
        const mtb_material *m = sc.materials + f.material;
        if (f.stage == 0) {
          const D3 c = Add(Load3(f.color), MulS(ret, m->reflectance));
          if (f.do_refract) {
            Store3(f.color, c);
            f.stage = 1;
            Count<DBG>(cnt, kRefract);
            const D3 rdir = Normalized(Load3(f.dir));
            Store3(st.m_o, Add(Load3(f.point), MulS(rdir, 0.00001)));
            Store3(st.m_d, rdir);
            flags = f.in_object != 0 ? 0u : kInObject;  // in_object toggled; not in a shadow walk
            st.coef = f.coef;
            st.path = f.path * 2ull + 1ull;
            st.level = sp;
            break;  // trace the refraction child
          }
          ret = c;
          sp--;
        } else {
          // (c * Tf) * Tr (mythtracer.cc:224)
          ret = Add(Load3(f.color), MulS(MulV(ret, Load3(m->transmission_filter)), m->transparency));
          sp--;
        }
      }
      if (!finished) continue;

      // ---- the pixel is done (mythtracer.cc:301) ----
      unsigned char *out = s_rgb + ((ty * kTile) + tx) * 3;
      out[0] = QuantizeChannel(ret.x);
      out[1] = QuantizeChannel(ret.y);
      out[2] = QuantizeChannel(ret.z);
      const size_t pix = PlaneIndex<BATCH>(rp, px, py);
      if (rp.sig_hits != nullptr) rp.sig_hits[pix] = st.sig_hits;
      if (rp.sig_shadow != nullptr) rp.sig_shadow[pix] = st.sig_shadow;
      n_rays = st.n_rays;
      if (rp.n_rays != nullptr) rp.n_rays[pix] = n_rays;
      break;
    }
  }

  // ---- the warp's half of the tile (4 rows of 24 bytes) leaves as aligned 8-byte stores when the layout allows it.
  // Warp-level on purpose: with a block-wide barrier here the warp that finishes first kept its slot on the SM until
  // the other one was done (ncu: 9 % of all warp samples sat in that barrier); now it exits and a warp of the next
  // tile takes its registers (DESIGN.md section 5, the warp-level epilogue row). ----
  __syncwarp();
  if constexpr (ACC || SS > 1) {
    AverageEpilogue<SS, ACC>(rp, acc, s_rgb, tile_id, strip, s_ss8);
  } else {
    const int px0 = (tile_id % rp.tiles_x) * kTile, py0 = strip * kTile + (int)(threadIdx.x >> 5) * 4;
    const unsigned lane = threadIdx.x & 31u;
    const unsigned char *half = s_rgb + (threadIdx.x >> 5) * (4 * kTile * 3);
    // (a view of a batch starts at a multiple of 24 bytes when chunk_w is a multiple of 8: rp.rgb's alignment decides)
    const bool whole_rows = px0 + kTile <= rp.chunk_w && (rp.chunk_w & 7) == 0 && (reinterpret_cast<uintptr_t>(rp.rgb) & 7u) == 0u;
    if (whole_rows) {
      if (lane < 12u) {
        const int row = (int)lane / 3, seg = (int)lane % 3;
        if (py0 + row < rp.chunk_h) {
          const uint2 v = *reinterpret_cast<const uint2 *>(half + row * 24 + seg * 8);
          *reinterpret_cast<uint2 *>(ViewFrame<BATCH>(rp) + ((size_t)(py0 + row) * rp.chunk_w + px0) * 3 + seg * 8) = v;
        }
      }
    } else if (live) {
      unsigned char *dst = ViewFrame<BATCH>(rp) + ((size_t)py * rp.chunk_w + px) * 3;
      const unsigned char *src = s_rgb + ((ty * kTile) + tx) * 3;
      dst[0] = src[0];
      dst[1] = src[1];
      dst[2] = src[2];
    }
  }

  // what this tile cost, for the next frame's launch order
  if (rp.tile_cost != nullptr) {
    unsigned v = n_rays;
    for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
    if ((threadIdx.x & 31u) == 0u) atomicAdd(rp.tile_cost + tile_id, v);
  }
  // (FlushCounters of wavefront.cu does the same; called here instead, it reschedules the single-frame kernels: 8 more
  // instructions in RenderMega<false, false, 1, false, false>)
  if (DBG && rp.counters != nullptr) {
    for (int i = 0; i < kNumCounters; i++) {
      unsigned long long v = cnt[i];
      for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
      if ((threadIdx.x & 31u) == 0u && v != 0ull) atomicAdd(rp.counters + i, v);
    }
  } else if (rp.counters != nullptr) {
    // the fast build still reports the ray count (the metric's numerator)
    unsigned long long v = n_rays;
    for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
    if ((threadIdx.x & 31u) == 0u && v != 0ull) atomicAdd(rp.counters + kRays, v);
  }
}

// Batched OctTree::IntersectRay (octtree.cc:26-40), one ray per thread.
template <bool DBG>
__global__ void __launch_bounds__(128) IntersectKernel(const __grid_constant__ DeviceScene sc, IntersectParams ip) {
  MTB_DECLARE_FAST_CTX(128);
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long cnt_store[DBG ? kNumCounters : 1];
  unsigned long long *cnt = cnt_store;
  if (DBG) {
    for (int k = 0; k < kNumCounters; k++) cnt[k] = 0;
  }
  if (i < ip.n) {
    const D3 o = Load3(ip.origins + i * 3), d = Load3(ip.dirs + i * 3);
    double t = 0.0;
    const int slot = Trace<DBG>(sc, o, d, CUDART_INF, &t, cnt, fctx);
    if (slot < 0) {
      // miss contract (include/mythtracer_b200.h): tri_index -1, t and point NaN - the scratch buffers are reused
      // between queries, so a miss must not leave an earlier query's values behind
      ip.tri_index[i] = -1;
      if (ip.t != nullptr) ip.t[i] = CUDART_NAN;
      if (ip.point != nullptr) ip.point[i * 3 + 0] = ip.point[i * 3 + 1] = ip.point[i * 3 + 2] = CUDART_NAN;
    } else {
      ip.tri_index[i] = sc.slots[slot].tri;
      if (ip.t != nullptr) ip.t[i] = t;
      if (ip.point != nullptr) {
        const D3 p = Add(o, MulS(d, t));
        ip.point[i * 3 + 0] = p.x;
        ip.point[i * 3 + 1] = p.y;
        ip.point[i * 3 + 2] = p.z;
      }
    }
  }
  if (DBG && ip.counters != nullptr) {
    for (int k = 0; k < kNumCounters; k++) {
      unsigned long long v = cnt[k];
      for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
      if ((threadIdx.x & 31u) == 0u && v != 0ull) atomicAdd(ip.counters + k, v);
    }
  }
}

// Counting sort of the tiles by cost bucket (log2 of the ray count, most expensive first).  One block.
__global__ void __launch_bounds__(1024) BuildTileOrder(uint32_t *tile_cost, int32_t *tile_order, int n_tiles) {
  __shared__ unsigned hist[33];
  __shared__ unsigned offset[33];
  // Every warp counts into its own copy (atomics on one address are serialised; 1024 threads on two or three hot
  // buckets took 33 us in round 1).
  __shared__ unsigned w_hist[32][33];
  for (int i = threadIdx.x; i < 32 * 33; i += blockDim.x) (&w_hist[0][0])[i] = 0;
  __syncthreads();
  // warp w owns the contiguous tiles [w * chunk, (w + 1) * chunk): inside a bucket the launch order then stays in
  // tile order, i.e. blocks that run at the same time render neighbouring tiles
  const unsigned warp = threadIdx.x >> 5;
  const int chunk = (n_tiles + 31) / 32;
  const int t_begin = (int)warp * chunk + (int)(threadIdx.x & 31u), t_end = min(n_tiles, ((int)warp + 1) * chunk);
  for (int t = t_begin; t < t_end; t += 32) {
    const unsigned c = tile_cost[t];
    const int b = c == 0u ? 0 : 32 - __clz((int)c);
    atomicAdd(&w_hist[warp][b], 1u);
  }
  __syncthreads();
  if (threadIdx.x < 33) {
    unsigned h = 0;
    for (int w = 0; w < 32; w++) h += w_hist[w][threadIdx.x];
    hist[threadIdx.x] = h;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned run = 0;
    for (int b = 32; b >= 0; b--) {
      offset[b] = run;
      run += hist[b];
    }
  }
  __syncthreads();
  // positions: a bucket's range is cut into one piece per warp (what that warp counted), filled with warp-local atomics
  if (threadIdx.x < 33) {
    unsigned run = offset[threadIdx.x];
    for (int w = 0; w < 32; w++) {
      const unsigned h = w_hist[w][threadIdx.x];
      w_hist[w][threadIdx.x] = run;
      run += h;
    }
  }
  __syncthreads();
  for (int t = t_begin; t < t_end; t += 32) {
    const unsigned c = tile_cost[t];
    const unsigned pos = atomicAdd(&w_hist[warp][c == 0u ? 0 : 32 - __clz((int)c)], 1u);
    tile_order[pos] = t;
    tile_cost[t] = 0;
  }
}

}  // namespace

void LaunchBuildTileOrder(uint32_t *tile_cost, int32_t *tile_order, int n_tiles, cudaStream_t stream) {
  if (n_tiles <= 0) return;
  BuildTileOrder<<<1, 1024, 0, stream>>>(tile_cost, tile_order, n_tiles);
}

// n_blocks = number of 8x8 tiles of the launch.
void LaunchRenderMega(const DeviceScene &sc, const RenderParams &rp, int n_blocks, bool debug_build, cudaStream_t stream) {
  if (n_blocks <= 0) return;
  if (debug_build) {
    RenderMega<true, false, 1, false, false, false><<<n_blocks, kBlockThreads, 0, stream>>>(sc, rp, nullptr, AccumParams{}, nullptr, PanoParams{});
  } else {
    RenderMega<false, false, 1, false, false, false><<<n_blocks, kBlockThreads, 0, stream>>>(sc, rp, nullptr, AccumParams{}, nullptr, PanoParams{});
  }
}

// Calls f(std::true_type{}) or f(std::false_type{}): a run-time flag as a template argument.
template <class F>
void WithBool(bool b, const F &f) {
  if (b) {
    f(std::true_type{});
  } else {
    f(std::false_type{});
  }
}

// One of the 48 batch kernels: DBG x SS (1, 2, 4, 8) x ACC x primary ray (pinhole, thin lens, panorama).
void LaunchRenderMegaBatch(const DeviceScene &sc, const RenderParams &rp, const ViewRec *views, int tiles_per_view, int n_views,
                           int samples_per_axis, const AccumParams &acc, const LensRec *lens, const PanoParams &pano, bool debug_build,
                           cudaStream_t stream) {
  if (tiles_per_view <= 0 || n_views <= 0) return;
  const dim3 grid((unsigned)tiles_per_view, (unsigned)n_views);
  // f(lens, panorama) as two type flags, never both true
  const auto with_primary_ray = [&](const auto &f) {
    if (lens != nullptr) {
      f(std::true_type{}, std::false_type{});
    } else {
      WithBool(pano.rec != nullptr, [&](auto panorama) { f(std::false_type{}, panorama); });
    }
  };
  WithBool(debug_build, [&](auto dbg) {
    WithBool(acc.subframes > 1, [&](auto accum) {
      with_primary_ray([&](auto thin_lens, auto panorama) {
        const auto launch = [&](auto ss) {
          RenderMega<decltype(dbg)::value, true, decltype(ss)::value, decltype(accum)::value, decltype(thin_lens)::value,
                     decltype(panorama)::value><<<grid, kBlockThreads, 0, stream>>>(sc, rp, views, acc, lens, pano);
        };
        switch (samples_per_axis) {
          case 1: launch(std::integral_constant<int, 1>{}); break;
          case 2: launch(std::integral_constant<int, 2>{}); break;
          case 4: launch(std::integral_constant<int, 4>{}); break;
          case 8: launch(std::integral_constant<int, 8>{}); break;
          default: break;  // (the host API admits 1, 2, 4 and 8 only)
        }
      });
    });
  });
}

void LaunchIntersect(const DeviceScene &sc, const IntersectParams &ip, bool debug_build, cudaStream_t stream) {
  if (ip.n <= 0) return;
  const int blocks = (int)((ip.n + 127) / 128);
  if (debug_build) {
    IntersectKernel<true><<<blocks, 128, 0, stream>>>(sc, ip);
  } else {
    IntersectKernel<false><<<blocks, 128, 0, stream>>>(sc, ip);
  }
}

}  // namespace mtb
