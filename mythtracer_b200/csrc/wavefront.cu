// Wavefront pipeline (the queue pipeline): the recursive TraceRayWorker (mythtracer.cc:13-228) as activations taken
// from ONE device-side ray queue by a persistent kernel, then a per-pixel fold.  Four kernels per frame:
//
//   WfQueueBegin   resets the queue, the overflow flag and the frame's work counters
//   WfQueue        traces every activation of every level, queues its reflection / refraction children, walks its
//                  shadow segments and sums its Phong terms (mythtracer.cc:13-178)
//   WfResolveTree  per pixel: parent += child * Refl, then parent += (child * Tf) * Tr -- the same two additions, in the
//                  same order, as the recursion performs on return -- and V3DtoRGB (mythtracer.cc:235-241)
//   WfCommit       work counters of the frame -> the context's counters; overflow flag -> pinned host words
//
// Nothing is read back to the host while a frame is in flight.  An activation table that overflows sets
// WfBuffers::ctrl[0]; every warp then leaves, and a RenderMega launch that is always queued behind the frame
// (RenderParams::run_if) renders the same pixels instead - both pipelines produce the same bytes - while the host
// enlarges the table for the next frame.
//
// Because every activation keeps its own colour and the fold replays the reference's additions in the
// reference's order, the result is bit-identical to the megakernel (and to the reference, up to pow()).
#include "device_core.cuh"

namespace mtb {
namespace {

template <bool DBG>
__device__ __forceinline__ void FlushCounters(unsigned long long *cnt, unsigned long long *global, unsigned n_rays) {
  if (global == nullptr) return;
  if (DBG) {
    for (int i = 0; i < kNumCounters; i++) {
      unsigned long long v = cnt[i];
      for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
      if ((threadIdx.x & 31u) == 0u && v != 0ull) atomicAdd(global + i, v);
    }
  } else {
    unsigned long long v = n_rays;
    for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
    if ((threadIdx.x & 31u) == 0u && v != 0ull) atomicAdd(global + kRays, v);
  }
}

// ---------------------------------------------------------------------------------------------------
// WfQueue: ONE persistent kernel for all levels
// ---------------------------------------------------------------------------------------------------
// A kernel per level would pay one kernel boundary per level on its critical path (a level's trace kernel ends with
// its slowest ray before the first ray of the next level starts) and write the whole shading context of every
// activation to HBM for separate shadow / light kernels.  Here a task is ONE ACTIVATION from beginning to end:
// a warp takes up to 32 consecutive entries of a single ray queue (entry id = activation id; ids below `slots` are
// the primary rays), traces them, shades the hits, appends their reflection / refraction children to the queue
// (warp ballots + prefix counts, one atomic per warp) and publishes them BEFORE it walks its own shadow segments -
// so the chain primary -> child -> grandchild runs ahead on other warps while the shadow walks fill the machine -
// and then does the shadow walks and the Phong sum of its hits in registers (nothing but colour, material and the two
// child links of an activation is ever stored).  The lanes of a warp are in phase by construction: all trace, then
// all walk towards light 0, then light 1, ... (the megakernel's lanes drift apart because every pixel follows its own
// tree).  The fold happens afterwards, per pixel, in the reference's order (WfResolveTree).
//
// Queue protocol.  qctl[kQTail] is advanced by producers (reservation), then the entries are written, then - after a
// __threadfence() - act_ready[id] = epoch marks each one complete.  A consumer takes [head, head + n) with one
// compare-and-swap on qctl[kQHead] (never beyond the reserved tail), and a lane whose entry is not complete yet spins
// on its flag; the producer never waits for anything in between, so the wait is short.  Queue fields are read with
// ld.global.cg: they were written by another SM during this kernel and L1 is not coherent.  qctl[kQPending] counts
// activations that are not finished; a warp that finds the queue empty leaves when it is zero.  Overflow of the
// activation table, or a wait that lasts absurdly long, sets ctrl[0]: every warp leaves and the repair launch
// (RenderMega, same bytes) renders the frame.
#ifndef MTB_QUEUE_MIN_BLOCKS
#define MTB_QUEUE_MIN_BLOCKS 16  // 64-thread blocks at 64 registers, the megakernel's shape (14 / 16 / 18 / 20 blocks: C3 9.77 / 9.36 / 9.38 / 9.42 ms)
#endif
constexpr unsigned kQueueSpinLimit = 1u << 22;
#ifndef MTB_QUEUE_MIN_TICKET
#define MTB_QUEUE_MIN_TICKET 4
#endif
#ifndef MTB_QUEUE_DRAIN
#define MTB_QUEUE_DRAIN 1  // 0: tickets are always 32 wide
#endif

__device__ __forceinline__ unsigned LdVolatile(const uint32_t *p) {
  unsigned v;
  asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ D3 LdCg3(const double *p) { return Mk(__ldcg(p), __ldcg(p + 1), __ldcg(p + 2)); }

// What an activation keeps across a traversal (local memory, explicit; cf. PixelState in megakernel.cu).
struct alignas(16) QueueState {
  double m_o[3], m_d[3];                                       // its ray
  double P[3], normal[3], surface[3], reflected[3], color[3];  // shading context (mythtracer.cc:38-76)
  double ldir[3], seg_start[3], power[3];                      // shadow walk of the current light (mythtracer.cc:86-156)
  double coef, light_distance;
  unsigned long long path, sig;
  int level, pixel, material, child_refl, child_refr, in_object;
  unsigned segments, rays;
};
#define MTB_QSTATE_BARRIER() asm volatile("" : : "l"(&st) : "memory")
__device__ __forceinline__ D3 Ld3q(const double *p) { return Mk(p[0], p[1], p[2]); }
__device__ __forceinline__ void St3q(double *p, const D3 &v) {
  p[0] = v.x;
  p[1] = v.y;
  p[2] = v.z;
}

__global__ void WfQueueBegin(WfBuffers wf, int slots) {
  const int i = (int)threadIdx.x;
  if (i < 2) wf.ctrl[i] = 0u;
  if (i < kNumCounters) wf.work[i] = 0ull;
  if (i < kQWords) wf.qctl[i] = (i == kQTail || i == kQPending) ? (uint32_t)slots : 0u;
}

// (`sc` is __grid_constant__ for the reason given at RenderMega: no local copy of the scene record.)
template <bool DBG>
__global__ void __launch_bounds__(kBlockThreads, MTB_QUEUE_MIN_BLOCKS) WfQueue(const __grid_constant__ DeviceScene sc, RenderParams rp, WfBuffers wf, int slots, unsigned epoch) {
  MTB_DECLARE_FAST_CTX(kBlockThreads);
  unsigned long long cnt_store[DBG ? kNumCounters : 1];
  unsigned long long *cnt = cnt_store;
  if (DBG) {
    for (int k = 0; k < kNumCounters; k++) cnt[k] = 0;
  }
  const unsigned lane = threadIdx.x & 31u, below = (1u << lane) - 1u;
  unsigned traced = 0;
  // The warp's ticket: it owns activations [ticket, ticket + tsize) and has handed `done` of them to its lanes so far.
  // Tickets are 32 wide (primary rays: whole groups of 8x4 pixels) until the queue runs dry at the very end of the
  // frame: when fewer rays are queued than MTB_QUEUE_DRAIN per warp of the grid, a warp takes 16, 8 or 4, so that the
  // last rays spread over more, emptier warps - a warp runs as long as its slowest ray, and the kernel as long as its
  // last warp.  Measured on C3, share 1/8 of the frame: always 32 wide 1.67 ms; this rule 1.50; thresholds 4x higher
  // 1.67, 6x higher 1.86 (small tickets any earlier cost more than they gain); tickets down to 2 or 1: 1.49.
  const unsigned n_warps = gridDim.x * (kBlockThreads / 32);
  unsigned ticket = 0, tsize = 32, done = 32;
  for (;;) {
    if (done >= tsize) {
      if (lane == 0u) {
        const unsigned head = LdVolatile(wf.qctl + kQHead);
        tsize = 32u;
        if (head >= (unsigned)slots) {  // (the head only grows: a ticket taken now lies behind the primary rays too)
          const unsigned tail = LdVolatile(wf.qctl + kQTail);
          const unsigned backlog = tail > head ? tail - head : 0u;
          const unsigned unit = n_warps * MTB_QUEUE_DRAIN;
          tsize = backlog >= 4u * unit ? 32u : (backlog >= 2u * unit ? 16u : (backlog >= unit ? 8u : 4u));
          if (MTB_QUEUE_MIN_TICKET < 4 && backlog < unit / 2u) tsize = backlog >= unit / 4u ? 2u : (unsigned)MTB_QUEUE_MIN_TICKET;
        }
        ticket = atomicAdd(wf.qctl + kQHead, tsize);  // fetch-and-add: never fails, never retried
      }
      ticket = __shfl_sync(0xffffffffu, ticket, 0);
      tsize = __shfl_sync(0xffffffffu, tsize, 0);
      done = 0;
    }
    if (ticket >= (unsigned)wf.act_cap) break;  // beyond the table: such entries are never produced (overflow is flagged)
    // ---- how many of the ticket's entries exist by now?  Primary rays always do; queued ones once the tail has
    // passed them.  A partly filled ticket is not waited for for long: what is there goes out to the first lanes
    // (late in a frame that spreads the few remaining rays over many warps by itself) ----
    unsigned n = tsize - done;
    bool over = false;
    if (ticket >= (unsigned)slots) {
      unsigned waited = 0;
      for (;;) {
        unsigned tail = 0, pending = 1, stop = 0;
        if (lane == 0u) {
          tail = LdVolatile(wf.qctl + kQTail);
          pending = LdVolatile(wf.qctl + kQPending);
          stop = LdVolatile(wf.ctrl);
          if (pending == 0u) tail = LdVolatile(wf.qctl + kQTail);  // nothing is in flight any more: this tail is final
        }
        tail = __shfl_sync(0xffffffffu, tail, 0);
        pending = __shfl_sync(0xffffffffu, pending, 0);
        stop = __shfl_sync(0xffffffffu, stop, 0);
        const unsigned first = ticket + done;
        const unsigned avail = tail > first ? (tail - first < tsize - done ? tail - first : tsize - done) : 0u;
        if (stop != 0u || (avail == 0u && pending == 0u)) {
          over = true;
          break;
        }
        if (avail == tsize - done || (avail > 0u && waited >= 2u)) {
          n = avail;
          break;
        }
        __nanosleep(waited < 16u ? 250u : 2000u);
        if (++waited > kQueueSpinLimit) {
          if (lane == 0u) wf.ctrl[0] = 1u;
          over = true;
          break;
        }
      }
    }
    if (over) break;

    // ---- the batch: lane k < n owns activation ticket + done + k ----
    const bool mine = lane < n;
    const int act = (int)(ticket + done + lane);
    done += n;
    bool live = mine, failed = false;
    // what has to survive a traversal lives in `st` (local memory, explicit - see PixelState in megakernel.cu for why),
    // including the scalars that are only touched between two traversals: a register each across the node loop is
    // what pushes other values into spill slots at 64 registers
    QueueState st;
    st.in_object = 0;
    st.level = 0;
    st.pixel = -1;
    st.coef = 1.0;
    st.path = 1ull;
    D3 o = Mk(0.0, 0.0, 0.0), d = Mk(0.0, 0.0, 0.0);
    if (mine) {
      if (act < slots) {
        // 8x8 pixel tiles (a warp = 8x4 pixels) of this launch's strips, as in RenderMega
        const int tile = act >> 6, t = act & 63;
        const int strip = rp.strip_first + (tile / rp.tiles_x) * rp.strip_stride;
        const int px = (tile % rp.tiles_x) * 8 + (t & 7);
        const int py = strip * 8 + (t >> 3);
        live = px < rp.chunk_w && py < rp.chunk_h;
        st.pixel = live ? py * rp.chunk_w + px : -1;
        const D3 start = Load3(rp.sensor), d_scan = Load3(rp.sensor + 3), d_pixel = Load3(rp.sensor + 6);
        o = Load3(rp.origin);
        d = Normalized(Add(Add(start, MulS(d_scan, (double)(rp.chunk_y + py))), MulS(d_pixel, (double)(rp.chunk_x + px))));
        if (live) Count<DBG>(cnt, kPrimary);
      } else {
        // reserved, and being written by the warp that spawned it: a short wait
        unsigned spins = 0;
        while (LdVolatile(wf.act_ready + act) != epoch) {
          if (++spins > kQueueSpinLimit || ((spins & 255u) == 0u && LdVolatile(wf.ctrl) != 0u)) {
            failed = true;
            break;
          }
          __nanosleep(40u);
        }
        __threadfence();
        if (!failed) {
          o = LdCg3(wf.act_point + (size_t)act * 3);
          d = LdCg3(wf.act_dir + (size_t)act * 3);
          st.coef = __ldcg(wf.act_coef + act);
          st.path = __ldcg(wf.act_path + act);
          st.pixel = __ldcg(wf.act_pixel + act);
          const int info = __ldcg(wf.act_info + act);
          st.level = info & 0xff;
          st.in_object = (info >> 8) != 0;
        }
      }
    }
    if (__any_sync(0xffffffffu, failed)) {
      if (lane == 0u) wf.ctrl[0] = 1u;
      break;
    }

    // ---- one traversal per loop iteration, as in RenderMega: iteration 0 traces the activations' own rays, then the
    // hits are shaded and their children queued (warp-wide), then every further iteration is one shadow segment of
    // the lanes that still walk.  What has to survive a traversal lives in `st` (local memory, explicit - see
    // PixelState in megakernel.cu for why); a handful of scalars stay in registers ----
    St3q(st.m_o, o);
    St3q(st.m_d, d);
    St3q(st.color, Mk(0.0, 0.0, 0.0));
    bool walking = live, main_phase = true, lit = false, in_shadow = false, through = false;
    int li = 0;
    st.material = -2;
    st.child_refl = -1;
    st.child_refr = -1;
    st.segments = 0;
    st.rays = 0;
    st.sig = 0ull;
    bool stop_all = false;
    for (;;) {
      int slot = -1;
      double t = 0.0;
      if (walking) {
        D3 to, td;
        double limit = CUDART_INF;
        if (main_phase) {
          to = Ld3q(st.m_o);
          td = Ld3q(st.m_d);
        } else {
          const D3 seg = Ld3q(st.seg_start);
          td = Ld3q(st.ldir);
          to = Add(seg, MulS(td, 0.00001));                                     // mythtracer.cc:95-99
          limit = Dist(seg, Load3(sc.lights[li].position));   // mythtracer.cc:101-102
          st.light_distance = limit;
          Count<DBG>(cnt, kShadow);
        }
        MTB_QSTATE_BARRIER();
        slot = Trace<DBG>(sc, to, td, limit, &t, cnt, fctx);
        MTB_QSTATE_BARRIER();
        st.rays++;
      }
      if (main_phase) {
        // ---- results of the activations' own rays (mythtracer.cc:13-76); every lane of the warp is here ----
        main_phase = false;
        bool do_reflect = false, do_refract = false;
        double refl = 0.0;
        if (walking) {
          walking = false;
          if (slot < 0) {
            if (st.level == 0 && rp.dbg != nullptr) {
              mtb_debug *dbg = rp.dbg + st.pixel;
              dbg->line_no = -1;
              dbg->pad_ = 0;
              dbg->point[0] = dbg->point[1] = dbg->point[2] = CUDART_NAN;
            }
          } else {
            const ShadeRec *sh = sc.shade + slot;
            const SlotRec *sr = sc.slots + slot;
            const D3 m_d = Ld3q(st.m_d);
            const D3 P = Add(Ld3q(st.m_o), MulS(m_d, t));
            const int line_no = __ldg(&sh->line_no);
            if (st.level == 0 && rp.dbg != nullptr) {
              mtb_debug *dbg = rp.dbg + st.pixel;
              dbg->line_no = line_no;
              dbg->pad_ = 0;
              dbg->point[0] = P.x;
              dbg->point[1] = P.y;
              dbg->point[2] = P.z;
            }
            if (rp.sig_hits != nullptr) {
              atomicAdd(reinterpret_cast<unsigned long long *>(rp.sig_hits) + st.pixel, Mix64(st.path, 1ull, (unsigned long long)(long long)line_no));
            }
            Count<DBG>(cnt, kShade);
            const D3 v0 = Load3(sr->vert), v1 = Load3(sr->vert + 3), v2 = Load3(sr->vert + 6);
            const BaryWeights w = Barycentric(v0, v1, v2, P);
            D3 normal = DivS(Add(Add(MulS(Load3(sh->normal), w.n0), MulS(Load3(sh->normal + 3), w.n1)), MulS(Load3(sh->normal + 6), w.n2)), w.n);
            const D3 towards_camera = Neg(m_d);
            double normal_ray_dot = Dot(towards_camera, normal);
            if (normal_ray_dot < 0.0) {
              normal = Neg(normal);
              normal_ray_dot = Dot(towards_camera, normal);
            }
            const int mtl = __ldg(&sh->material);
            if (mtl < 0) {  // mythtracer.cc:49-52
              normal_ray_dot = (normal_ray_dot + 1.0) * 0.5;
              St3q(st.color, Mk(normal_ray_dot, normal_ray_dot, normal_ray_dot));
            } else {
              const mtb_material *m = sc.materials + mtl;
              D3 surface = Load3(m->ambient);
              const int tex = m->texture;
              if (tex >= 0) {
                const double u = (sh->uv[0] * w.n0 + sh->uv[2] * w.n1 + sh->uv[4] * w.n2) / w.n;
                const double v = (sh->uv[1] * w.n0 + sh->uv[3] * w.n1 + sh->uv[5] * w.n2) / w.n;
                surface = MulV(surface, SampleTexture(sc.tex_atlas, tex, sc.texture_dim[tex], u, v));
              }
              const D3 reflected = Sub(m_d, MulS(normal, 2 * Dot(normal, m_d)));
              St3q(st.P, P);
              St3q(st.normal, normal);
              St3q(st.surface, surface);
              St3q(st.reflected, reflected);
              st.material = mtl;
              lit = true;
              if (st.level < rp.max_depth) {
                refl = m->reflectance;
                do_reflect = refl > 0.0 && st.coef > 0.01 && !st.in_object;  // mythtracer.cc:181-184
                do_refract = m->transparency > 0.0;                    // mythtracer.cc:192
              }
            }
          }
        }
        // ---- children -> queue, published before this warp walks its shadow segments.  The warp's reflection
        // children are stored first, then its refraction children: neighbouring entries (= the lanes of some warp
        // later) are rays of the same kind from neighbouring pixels ----
        const unsigned refl_mask = __ballot_sync(0xffffffffu, do_reflect);
        const unsigned refr_mask = __ballot_sync(0xffffffffu, do_refract);
        const unsigned n_refl = (unsigned)__popc(refl_mask), total = n_refl + (unsigned)__popc(refr_mask);
        if (total != 0u) {
          unsigned base = 0;
          if (lane == 0u) {
            atomicAdd(wf.qctl + kQPending, total);  // counted before they can be seen: the count never runs low
            base = atomicAdd(wf.qctl + kQTail, total);
          }
          base = __shfl_sync(0xffffffffu, base, 0);
          if ((unsigned long long)base + total > (unsigned long long)wf.act_cap) {
            stop_all = true;
          } else {
            if (do_reflect || do_refract) {
              const D3 P = Ld3q(st.P), m_d = Ld3q(st.m_d);
              if (do_reflect) {
                const int c = (int)(base + (unsigned)__popc(refl_mask & below));
                const D3 reflected = Ld3q(st.reflected);
                Count<DBG>(cnt, kReflect);
                Store3(wf.act_point + (size_t)c * 3, Add(P, MulS(reflected, 0.0001)));  // mythtracer.cc:70-75
                Store3(wf.act_dir + (size_t)c * 3, reflected);
                wf.act_coef[c] = st.coef * refl;
                wf.act_path[c] = st.path * 2ull;
                wf.act_pixel[c] = st.pixel;
                wf.act_info[c] = (st.level + 1) | (st.in_object ? 256 : 0);
                st.child_refl = c;
              }
              if (do_refract) {
                const int c = (int)(base + n_refl + (unsigned)__popc(refr_mask & below));
                Count<DBG>(cnt, kRefract);
                const D3 rdir = Normalized(m_d);                                      // mythtracer.cc:208-212
                Store3(wf.act_point + (size_t)c * 3, Add(P, MulS(rdir, 0.00001)));    // mythtracer.cc:214-218
                Store3(wf.act_dir + (size_t)c * 3, rdir);
                wf.act_coef[c] = st.coef;
                wf.act_path[c] = st.path * 2ull + 1ull;
                wf.act_pixel[c] = st.pixel;
                wf.act_info[c] = (st.level + 1) | (st.in_object ? 0 : 256);
                st.child_refr = c;
              }
              __threadfence();
              if (st.child_refl >= 0) asm volatile("st.volatile.global.u32 [%0], %1;" : : "l"(wf.act_ready + st.child_refl), "r"(epoch) : "memory");
              if (st.child_refr >= 0) asm volatile("st.volatile.global.u32 [%0], %1;" : : "l"(wf.act_ready + st.child_refr), "r"(epoch) : "memory");
            }
          }
        }
        if (stop_all) break;
        // this batch's activations spawn nothing else: they leave the count (their children are in it already)
        if (lane == 0u) atomicAdd(wf.qctl + kQPending, 0u - n);
        // the links and the material are final now
        if (mine) {
          wf.act_mtl[act] = st.material;
          wf.act_refl[act] = st.child_refl;
          wf.act_refr[act] = st.child_refr;
        }
        walking = lit && sc.n_lights > 0;
      } else if (walking) {
        // ---- one shadow segment came back (mythtracer.cc:104-156) ----
        bool light_done = false;
        st.segments++;
        if (slot < 0) {
          light_done = true;
        } else if (t > st.light_distance) {
          light_done = true;
        } else {
          const int smtl = __ldg(&sc.shade[slot].material);
          const double str = smtl >= 0 ? __ldg(&sc.materials[smtl].transparency) : 0.0;
          if (str == 0.0) {
            St3q(st.power, Mk(0.0, 0.0, 0.0));
            in_shadow = true;
            light_done = true;
          } else {
            D3 power = Ld3q(st.power);
            if (!through) {
              power = MulV(power, MulS(Load3(sc.materials[smtl].transmission_filter), str));
              St3q(st.power, power);
            }
            through = !through;
            const D3 ldir = Ld3q(st.ldir);
            const D3 to = Add(Ld3q(st.seg_start), MulS(ldir, 0.00001));
            const D3 seg_start = Add(Add(to, MulS(ldir, t)), MulS(ldir, 0.0000001));  // mythtracer.cc:137
            St3q(st.seg_start, seg_start);
            const D3 P = Ld3q(st.P);
            if (SqrDist(P, seg_start) > SqrDist(P, Load3(sc.lights[li].position))) {  // mythtracer.cc:141-145
              light_done = true;
            } else if (power.x <= 0.001 && power.y <= 0.001 && power.z <= 0.001) {
              St3q(st.power, Mk(0.0, 0.0, 0.0));
              in_shadow = true;
              light_done = true;
            }
          }
        }
        if (light_done) {
          // ---- this light is settled: Phong terms (mythtracer.cc:159-177) ----
          const mtb_light *lt = sc.lights + li;
          const mtb_material *m = sc.materials + st.material;
          st.sig += Mix64(st.path, 2ull + (unsigned long long)li, (in_shadow ? 1ull : 0ull) | ((unsigned long long)st.segments << 1));
          const D3 lamb = Load3(lt->ambient);
          D3 power = Ld3q(st.power);
          power.x = SMax(power.x, lamb.x);
          power.y = SMax(power.y, lamb.y);
          power.z = SMax(power.z, lamb.z);
          const D3 surface = Ld3q(st.surface);
          D3 color = Ld3q(st.color);
          color = Add(color, MulV(MulV(MulS(MulV(Load3(m->diffuse), surface), Dot(Ld3q(st.normal), Ld3q(st.ldir))), Load3(lt->diffuse)), power));
          if (!in_shadow) {
            const double refl_dot = Dot(Neg(Ld3q(st.m_d)), Ld3q(st.reflected));
            if (refl_dot > 0) {
              color = Add(color, MulV(MulS(MulV(Load3(m->specular), surface), pow(refl_dot, m->specular_exp)), Load3(lt->specular)));
            }
          }
          St3q(st.color, color);
          li++;
          walking = li < sc.n_lights;
        } else {
          continue;  // next segment of the same light
        }
      }
      if (!walking) break;
      // ---- start the shadow walk of light li (mythtracer.cc:79-94) ----
      {
        const mtb_light *lt = sc.lights + li;
        const D3 P = Ld3q(st.P);
        St3q(st.ldir, Normalized(Sub(Load3(lt->position), P)));
        St3q(st.color, Add(Ld3q(st.color), MulV(Load3(lt->ambient), Ld3q(st.surface))));  // mythtracer.cc:83-84
        St3q(st.power, Mk(1.0, 1.0, 1.0));
        St3q(st.seg_start, P);
        in_shadow = false;
        through = false;
        st.segments = 0;
      }
    }
    if (__any_sync(0xffffffffu, stop_all)) {
      if (lane == 0u) wf.ctrl[0] = 1u;
      break;
    }
    if (mine) {
      Store3(wf.act_color + (size_t)act * 3, Ld3q(st.color));
      if (live) {
        traced += st.rays;
        if (lit && rp.sig_shadow != nullptr && sc.n_lights > 0) atomicAdd(reinterpret_cast<unsigned long long *>(rp.sig_shadow) + st.pixel, st.sig);
        if (rp.n_rays != nullptr) atomicAdd(rp.n_rays + st.pixel, st.rays);
      }
    }
  }
  FlushCounters<DBG>(cnt, wf.work, traced);
}

// Per-pixel fold of the activation tree in the reference's order - parent += child * Refl, then
// parent += (child * Tf) * Tr (mythtracer.cc:185-189, 220-224), children before parents - followed by V3DtoRGB
// (mythtracer.cc:235-241).  One block = one 8x8 tile (slots pos * 64 ..), written like RenderMega writes its tiles.
__global__ void __launch_bounds__(kBlockThreads) WfResolveTree(const __grid_constant__ DeviceScene sc, RenderParams rp, WfBuffers wf, int slots) {
  __shared__ __align__(8) unsigned char s_rgb[kTile * kTile * 3];
  if (wf.ctrl[0] != 0u) return;
  const int tile = (int)blockIdx.x, root = tile * 64 + (int)threadIdx.x;
  if (root >= slots) return;
  const int strip = rp.strip_first + (tile / rp.tiles_x) * rp.strip_stride;
  const int tx = (int)(threadIdx.x & 7u), ty = (int)(threadIdx.x >> 3);
  const int px = (tile % rp.tiles_x) * kTile + tx, py = strip * kTile + ty;
  const bool live = px < rp.chunk_w && py < rp.chunk_h;
  {
    int f_act[MTB_MAX_RAY_DEPTH + 2];
    unsigned char f_stage[MTB_MAX_RAY_DEPTH + 2];  // 0: nothing folded yet, 1: reflection child in progress / done, 2: refraction child
    D3 f_color[MTB_MAX_RAY_DEPTH + 2];
    int sp = 0;
    D3 ret = Mk(0.0, 0.0, 0.0);
    if (live) {
      f_act[0] = root;
      f_stage[0] = 0;
      f_color[0] = Load3(wf.act_color + (size_t)root * 3);
      sp = 1;
    }
    while (sp > 0) {
      const int a = f_act[sp - 1];
      int child = -1;
      if (f_stage[sp - 1] == 0) {
        f_stage[sp - 1] = 1;
        child = wf.act_refl[a];
      }
      if (child < 0 && f_stage[sp - 1] == 1) {
        f_stage[sp - 1] = 2;
        child = wf.act_refr[a];
      }
      if (child >= 0 && sp < MTB_MAX_RAY_DEPTH + 2) {
        f_act[sp] = child;
        f_stage[sp] = 0;
        f_color[sp] = Load3(wf.act_color + (size_t)child * 3);
        sp++;
        continue;
      }
      ret = f_color[sp - 1];
      sp--;
      if (sp == 0) break;
      const mtb_material *m = sc.materials + wf.act_mtl[f_act[sp - 1]];
      if (f_stage[sp - 1] == 1) {
        f_color[sp - 1] = Add(f_color[sp - 1], MulS(ret, m->reflectance));
      } else {
        f_color[sp - 1] = Add(f_color[sp - 1], MulS(MulV(ret, Load3(m->transmission_filter)), m->transparency));
      }
    }
    unsigned char *out = s_rgb + ((ty * kTile) + tx) * 3;
    out[0] = QuantizeChannel(ret.x);
    out[1] = QuantizeChannel(ret.y);
    out[2] = QuantizeChannel(ret.z);
  }
  __syncwarp();
  {
    const int px0 = (tile % rp.tiles_x) * kTile, py0 = strip * kTile + (int)(threadIdx.x >> 5) * 4;
    const unsigned lane = threadIdx.x & 31u;
    const unsigned char *half = s_rgb + (threadIdx.x >> 5) * (4 * kTile * 3);
    const bool whole_rows = px0 + kTile <= rp.chunk_w && (rp.chunk_w & 7) == 0 && (reinterpret_cast<uintptr_t>(rp.rgb) & 7u) == 0u;
    if (whole_rows) {
      if (lane < 12u) {
        const int row = (int)lane / 3, seg = (int)lane % 3;
        if (py0 + row < rp.chunk_h) {
          const uint2 v = *reinterpret_cast<const uint2 *>(half + row * 24 + seg * 8);
          *reinterpret_cast<uint2 *>(rp.rgb + ((size_t)(py0 + row) * rp.chunk_w + px0) * 3 + seg * 8) = v;
        }
      }
    } else if (live) {
      unsigned char *dst = rp.rgb + ((size_t)py * rp.chunk_w + px) * 3;
      const unsigned char *src = s_rgb + ((ty * kTile) + tx) * 3;
      dst[0] = src[0];
      dst[1] = src[1];
      dst[2] = src[2];
    }
  }
}

// Last kernel of a frame.  The work counters of a frame that overflowed are dropped (the repair launch counts its
// own rays); host_copy (pinned, nullable) receives the overflow flag for the next frame's table capacity - written by
// the device, never waited for by the host.
__global__ void WfCommit(WfBuffers wf, unsigned long long *global, uint32_t *host_copy) {
  const int i = (int)threadIdx.x;
  const bool overflow = wf.ctrl[0] != 0u;
  if (!overflow && global != nullptr && i < kNumCounters && wf.work[i] != 0ull) atomicAdd(global + i, wf.work[i]);
  if (host_copy != nullptr) {
    if (i == 0) host_copy[kWfHostOverflow] = overflow ? 1u : 0u;
    __syncwarp();
    __threadfence_system();
    if (i == 0) host_copy[kWfHostSequence] += 1u;  // frames completed so far
  }
}

}  // namespace

void LaunchWfQueueBegin(const WfBuffers &wf, int slots, cudaStream_t stream) { WfQueueBegin<<<1, 32, 0, stream>>>(wf, slots); }

void LaunchWfQueue(const DeviceScene &sc, const RenderParams &rp, const WfBuffers &wf, int slots, unsigned epoch, int sm_count, bool debug_build,
                   cudaStream_t stream) {
  // persistent: what the device can hold, but not more warps than the frame has groups of 32 primary rays
  long long blocks = (long long)sm_count * MTB_QUEUE_MIN_BLOCKS;
  const long long need = ((long long)slots / 32 + 1) / 2;
  if (blocks > need) blocks = need < 1 ? 1 : need;
  if (debug_build) {
    WfQueue<true><<<(int)blocks, kBlockThreads, 0, stream>>>(sc, rp, wf, slots, epoch);
  } else {
    WfQueue<false><<<(int)blocks, kBlockThreads, 0, stream>>>(sc, rp, wf, slots, epoch);
  }
}

void LaunchWfResolveTree(const DeviceScene &sc, const RenderParams &rp, const WfBuffers &wf, int slots, cudaStream_t stream) {
  if (slots <= 0) return;
  WfResolveTree<<<slots / 64, kBlockThreads, 0, stream>>>(sc, rp, wf, slots);
}

void LaunchWfCommit(const WfBuffers &wf, unsigned long long *global, uint32_t *host_copy, cudaStream_t stream) {
  WfCommit<<<1, 32, 0, stream>>>(wf, global, host_copy);
}

}  // namespace mtb
