// TEST INFRASTRUCTURE ONLY: the CPU oracle (oracle/mt_oracle.cc, compiled here unchanged into the same translation
// unit) with one more entry point, mto_render_rays: the per-pixel body of render_impl with the primary ray given
// instead of made from a camera - the same trace(...) call, the same quantisation, debug info and taps, and no shading
// code of its own.  tests/test_lens.py builds it into a temporary library and traces the thin-lens rays of the product's
// mtb_render_batch_lens with it, restated in numpy.  Every other mto_* function of the library is the oracle's.
//
// Build: g++ -O2 -std=c++17 -fopenmp -fPIC -ffp-contract=off -shared -I oracle tests/cpp/oracle_rays.cc (the flags of
// oracle/Makefile).
#include "mt_oracle.cc"

extern "C" {

// Pixel i is TraceRay(origins[i], dirs[i]) at depth max_depth (mythtracer.cc:297-301 with the primary ray given).
// rgb: n*3; dbg_line_no n, dbg_point n*3 and taps (n entries each) may be NULL.
int mto_render_rays(const mto_scene *s, int64_t n, const double *origins, const double *dirs, int max_depth, uint8_t *rgb,
                    int32_t *dbg_line_no, double *dbg_point, const mto_taps *taps, mto_stats *stats) {
  if (s == nullptr || n < 0 || (n > 0 && (origins == nullptr || dirs == nullptr))) return -1;
  mto_stats total;
  memset(&total, 0, sizeof(total));
  const int nthreads = g_threads > 0 ? g_threads : omp_get_max_threads();
#pragma omp parallel num_threads(nthreads)
  {
    Counters cn;
    memset(&cn, 0, sizeof(cn));
#pragma omp for schedule(dynamic, 64)
    for (int64_t i = 0; i < n; i++) {
      const size_t px = (size_t)i;
      PixelTap tap;
      tap.want_dbg = (dbg_line_no != nullptr || dbg_point != nullptr);
      cn.s.primary++;
      const V3 o = mk(origins[i * 3], origins[i * 3 + 1], origins[i * 3 + 2]);
      const V3 d = mk(dirs[i * 3], dirs[i * 3 + 1], dirs[i * 3 + 2]);
      const V3 c = trace(s, o, d, 0, false, 1.0, max_depth, 1, &tap, &cn);
      if (rgb != nullptr) quantize(c, rgb + px * 3);
      if (dbg_line_no != nullptr) dbg_line_no[px] = tap.dbg_line;
      if (dbg_point != nullptr) memcpy(dbg_point + px * 3, tap.dbg_point.v, sizeof(tap.dbg_point.v));
      if (taps != nullptr) {
        if (taps->sig_hits) taps->sig_hits[px] = tap.sig_hits;
        if (taps->sig_shadow) taps->sig_shadow[px] = tap.sig_shadow;
        if (taps->n_rays) taps->n_rays[px] = tap.n_rays;
      }
    }
#pragma omp critical
    add_stats(&total, cn.s);
  }
  if (stats != nullptr) *stats = total;
  return 0;
}

}  // extern "C"
