// Host build of csrc/gemm_plan.cuh -- TEST INFRASTRUCTURE.  tests/test_cpu_gemm_plan.py compiles this with g++ and checks which kernel, tile
// width, grid and shared-memory size dsb_gemm_ex launches for a descriptor, without a GPU.
#include <cstdarg>
#include <cstdio>

#include "gemm_plan.cuh"

namespace {
char g_err[512];
}

void dsb::set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// The plan in plain ints (mirrored by a ctypes.Structure in the test)
struct PlanOut {
  int kernel, block_n, grid, smem_bytes, w_box_rows, l2_promo_128;
  int tiles_m, tiles_n, n_pad, a_stages, f3_nsp, lo_a, lo_w;
  unsigned tap_share_mask;
  int tap_shift[dsb::MAX_TAPS], tap_acol[dsb::MAX_TAPS], tap_wcol[dsb::MAX_TAPS];
};

extern "C" int plan_gemm_host(const dsb_gemm_desc* d, int sms, PlanOut* o) {
  g_err[0] = 0;
  dsb::GemmPlan g;
  if (const int rc = dsb::plan_gemm(*d, sms, &g)) return rc;
  const dsb::GemmParams& p = g.p;
  *o = PlanOut{g.kernel, g.block_n, g.grid, g.smem_bytes, g.w_box_rows, g.l2_promo_128,
               p.tiles_m, p.tiles_n, p.n_pad, p.a_stages, p.f3_nsp, p.lo_a, p.lo_w, p.tap_share_mask, {}, {}, {}};
  for (int i = 0; i < dsb::MAX_TAPS; ++i) {
    o->tap_shift[i] = p.tap_shift[i];
    o->tap_acol[i] = p.tap_acol[i];
    o->tap_wcol[i] = p.tap_wcol[i];
  }
  return 0;
}

extern "C" const char* plan_gemm_error() { return g_err; }
