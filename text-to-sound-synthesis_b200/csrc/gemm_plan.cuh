// Kernel choice of dsb_gemm_ex: descriptor checks, tile width, which of the four tcgen05 GEMM kernels runs, its parameters and its launch
// geometry.  Everything here depends on the descriptor and the SM count only and makes no CUDA call, so the host compiler builds this header
// too: tests/native/gemm_plan_host.cpp pins the choices without a GPU.
#pragma once
#include "diffsound_b200.h"
#include "error.cuh"

namespace dsb {

constexpr int BLOCK_M = 128;
constexpr int ROW_BYTES = 128;  // one swizzle-128B row of K per operand row
constexpr int MAX_TAPS = 32;

struct GemmParams {
  int M, N, batch;
  int tiles_m, tiles_n;
  int kb_per_tap;  // ceil(Kc / BLOCK_K)
  int block_k;     // elements per k-block (32 tf32 / 64 bf16)
  int num_taps;
  int tap_shift[MAX_TAPS];
  int tap_acol[MAX_TAPS];
  int tap_wcol[MAX_TAPS];  // W column offset per tap (default tap * Kc)
  unsigned tap_a2_mask;    // bit i set: tap i reads the SECOND A tensor map (a fused GEMM over two activation buffers)
  unsigned tap_share_mask; // resident-W kernel: bit i set: tap i multiplies the A box tap i-1 staged (same shift / column / operand)
  int n_pad;               // resident-W kernel: rows of one W box = the MMA's N (N rounded up to 16)
  int a_stages;            // resident-W kernel: depth of the A-box ring (whatever shared memory the resident weights leave, <= 12)
  // fused split-fp16 pair kernel: f3_nsp spatial taps j, each with row shift tap_shift[j], hi-half columns tap_acol[j] (A) / tap_wcol[j] (W);
  // the lo halves sit lo_a / lo_w columns further right
  int f3_nsp, lo_a, lo_w;
  long long split_off;     // DSB_GEMM_OUT_F16_SPLIT: offset of the lo half inside an output row
  long long dual_off;      // DSB_GEMM_DUAL_LRELU: offset of the LeakyReLU(0.2) copy (hi at +dual_off, lo at +dual_off+split_off)
  int ocg, ocg_stride;     // output column groups: logical column n lives at (n / ocg) * ocg_stride + n % ocg (0 = plain)
  float* amax_out;         // optional: atomic max of |value stored| over the whole output (calibration of fp16 activation scales)
  int kc;          // channels per tap
  int b_batched;
  const float* bias;
  const float* residual;
  long long ld_res, res_bstride;
  void* out;
  long long ldo, out_bstride;
  int flags;
  // optional row mask (padded conv geometry): row r -> p = r % geo_P; y = p / geo_Wp; x = p % geo_Wp;
  // rows outside [y0,y1) x [x0,x1) are written as zeros.  geo_P == 0 disables.
  int geo_P, geo_Wp, geo_y0, geo_y1, geo_x0, geo_x1;
  float alpha;     // scale applied to the accumulator before bias (1.0 for Linear)
  // MN-major operands (2-byte types, one tap): the operand lies in HBM as (K rows, MN columns) -- e.g. dY and X of a weight-gradient GEMM
  // dW = dY^T X, which contract over the token dimension.  Loaded as 64-column x 64-row TMA boxes (SWIZZLE_128B), consumed through MN-major
  // UMMA descriptors: no transposed copies.
  int a_mn, b_mn;
};

// Shared-memory layouts of the four kernels (gemm_tcgen05.cu)
template <int BLOCK_N>
struct GemmSmem {
  static constexpr int A_BYTES = BLOCK_M * ROW_BYTES;
  static constexpr int B_BYTES = BLOCK_N * ROW_BYTES;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = (BLOCK_N == 256) ? 4 : 6;
  static constexpr int TOTAL = STAGES * STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/ + 8 * 32 * 32 * 4 /*epilogue transpose tiles*/;
};

struct PairSmem {
  static constexpr int BLOCK_N = 256;
  static constexpr int A_BYTES = BLOCK_M * ROW_BYTES;        // this CTA's 128 rows of A
  static constexpr int B_BYTES = (BLOCK_N / 2) * ROW_BYTES;  // this CTA's half of the B tile
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = 6;
  static constexpr int TOTAL = STAGES * STAGE_BYTES + 1024 + 256 + 8 * 32 * 32 * 4;
};

template <int BN>
struct PairSplitSmem {
  static constexpr int BLOCK_N = BN;
  static constexpr int TILE_A = BLOCK_M * ROW_BYTES;     // 16 KB: this CTA's 128 rows x 64 halves of A (hi or lo)
  static constexpr int TILE_B = (BN / 2) * ROW_BYTES;    // this CTA's half of the W tile (hi or lo)
  static constexpr int STAGE_BYTES = 2 * TILE_A + 2 * TILE_B;  // A hi | A lo | W hi | W lo
  static constexpr int STAGES = BN == 256 ? 3 : 4;
  static constexpr int TOTAL = STAGES * STAGE_BYTES + 1024 + 256 + 8 * 32 * 32 * 4;
};

struct ResidentSmem {
  static constexpr int A_BYTES = BLOCK_M * ROW_BYTES;
  static constexpr int MAX_STAGES = 12;
  static constexpr int W_MAX = 96 * 1024;
  static constexpr int BAR_BYTES = 512;
  static constexpr int EPI_BYTES = 8 * 32 * 32 * 4;
  static constexpr int BUDGET = 227 * 1024 - 1024 /*static smem of the epilogue*/;
  static constexpr int FIXED = 1024 /*align slack*/ + BAR_BYTES + EPI_BYTES;
};

enum GemmKernel {
  GEMM_1CTA = 0,        // gemm_tcgen05_kernel<block_n, dtype>
  GEMM_PAIR = 1,        // gemm_tcgen05_pair_kernel<dtype>: 256 x 256 tiles on a CTA pair
  GEMM_F16X3_PAIR = 2,  // gemm_f16x3_pair_kernel<block_n>: the three split-fp16 passes off one staged copy, 256-row pair tiles
  CONV_RESIDENT = 3,    // conv_resident_kernel<dtype>: every tap's W box resident in shared memory
};

struct GemmPlan {
  GemmParams p;
  int kernel;        // GemmKernel
  int block_n;       // output tile width (the resident-W kernel: n_pad)
  int grid;          // CTAs launched (pair kernels: twice the pairs)
  int smem_bytes;    // dynamic shared memory per CTA
  int w_box_rows;    // rows of one W TMA box: block_n, half of it on a CTA pair, n_pad for the resident-W kernel
  int l2_promo_128;  // the A maps promote 128-byte L2 lines instead of 256-byte ones
};

// Checks the descriptor (non-zero return and the error message on a malformed one) and fills *out with what dsb_gemm_ex launches on a GPU
// with `sms` SMs.
inline int plan_gemm(const dsb_gemm_desc& d, int sms, GemmPlan* out) {
  DSB_REQUIRE(d.M > 0 && d.N > 0 && d.K > 0 && d.batch > 0, "dsb_gemm_ex: bad shape M=%d N=%d K=%d batch=%d", d.M, d.N, d.K, d.batch);
  DSB_REQUIRE(d.num_taps >= 1 && d.num_taps <= MAX_TAPS, "dsb_gemm_ex: num_taps=%d out of range", d.num_taps);
  DSB_REQUIRE(d.dtype == DSB_DTYPE_TF32 || d.dtype == DSB_DTYPE_BF16 || d.dtype == DSB_DTYPE_F16,
              "dsb_gemm_ex: dtype must be TF32, BF16 or F16 (use dsb_gemm_f32 for exact fp32)");
  const int kind = d.dtype;
  const int block_k = kind == DSB_DTYPE_TF32 ? 32 : 64;
  GemmPlan g{};
  GemmParams& p = g.p;
  p.M = d.M; p.N = d.N; p.batch = d.batch;
  p.tiles_m = (d.M + BLOCK_M - 1) / BLOCK_M;
  p.kb_per_tap = (d.K + block_k - 1) / block_k;
  p.block_k = block_k;
  p.num_taps = d.num_taps;
  for (int i = 0; i < MAX_TAPS; ++i) {
    p.tap_shift[i] = i < d.num_taps ? d.tap_shift[i] : 0;
    p.tap_acol[i] = i < d.num_taps ? d.tap_acol[i] : 0;
    p.tap_wcol[i] = i < d.num_taps ? (d.use_tap_wcol ? d.tap_wcol[i] : i * d.K) : 0;
  }
  {
    const int es_ = kind == DSB_DTYPE_TF32 ? 4 : 2;
    for (int i = 0; i < d.num_taps; ++i)
      DSB_REQUIRE((p.tap_acol[i] * es_) % 16 == 0 && (p.tap_wcol[i] * es_) % 16 == 0,
                  "dsb_gemm_ex: tap %d starts at A column %d / W column %d: TMA box coordinates must be multiples of 16 bytes", i, p.tap_acol[i], p.tap_wcol[i]);
  }
  p.split_off = d.split_off > 0 ? d.split_off : d.N;
  p.dual_off = d.dual_off;
  p.amax_out = d.amax_out;
  p.ocg = d.out_col_group; p.ocg_stride = d.out_col_group_stride;
  p.tap_a2_mask = 0;
  if (d.A2) {
    for (int i = 0; i < d.num_taps; ++i)
      if (d.tap_a2[i]) p.tap_a2_mask |= 1u << i;
  }
  DSB_REQUIRE(!(d.flags & DSB_GEMM_DUAL_LRELU) || ((d.flags & DSB_GEMM_OUT_F16_SPLIT) && d.dual_off > 0),
              "dsb_gemm_ex: DSB_GEMM_DUAL_LRELU needs DSB_GEMM_OUT_F16_SPLIT and dual_off > 0");
  DSB_REQUIRE(d.out_col_group == 0 || ((d.flags & DSB_GEMM_OUT_F16_SPLIT) && d.out_col_group % 4 == 0 && d.out_col_group_stride % 4 == 0 && !d.residual),
              "dsb_gemm_ex: output column groups need the split-fp16 output, multiples of 4 and no residual");
  p.kc = d.K;
  p.b_batched = d.w_batch_stride != 0;
  p.bias = d.bias; p.residual = d.residual; p.ld_res = d.ld_res; p.res_bstride = d.res_batch_stride;
  p.out = d.out; p.ldo = d.ldo; p.out_bstride = d.out_batch_stride;
  p.flags = d.flags;
  p.geo_P = d.geo_P; p.geo_Wp = d.geo_Wp; p.geo_y0 = d.geo_y0; p.geo_y1 = d.geo_y1; p.geo_x0 = d.geo_x0; p.geo_x1 = d.geo_x1;
  p.alpha = d.alpha == 0.0f ? 1.0f : d.alpha;
  p.a_mn = d.a_mn_major != 0;
  p.b_mn = d.b_mn_major != 0;
  const bool any_mn = p.a_mn || p.b_mn;
  DSB_REQUIRE(!any_mn || (kind != DSB_DTYPE_TF32 && d.num_taps == 1 && d.tap_shift[0] == 0 && d.tap_acol[0] == 0),
              "dsb_gemm_ex: MN-major operands need a 2-byte dtype and a single unshifted tap");
  const int max_ctas = d.max_ctas > 0 ? d.max_ctas : sms;

  if (d.resident_w) {
    DSB_REQUIRE(kind != DSB_DTYPE_TF32 && !any_mn && !p.b_batched && d.K == 64 && d.N <= 128 && d.use_tap_wcol,
                "dsb_gemm_ex: resident_w needs a 2-byte dtype, K-major operands, K == 64 per tap, N <= 128, explicit tap_wcol and an unbatched W");
    p.n_pad = (d.N + 15) / 16 * 16;
    const int w_bytes = d.num_taps * p.n_pad * ROW_BYTES;
    DSB_REQUIRE(w_bytes <= ResidentSmem::W_MAX, "dsb_gemm_ex: resident_w: %d taps x %d rows do not fit the %d KB weight area", d.num_taps, p.n_pad, ResidentSmem::W_MAX >> 10);
    p.tap_share_mask = 0;
    for (int i = 1; i < d.num_taps; ++i)
      if (p.tap_shift[i] == p.tap_shift[i - 1] && p.tap_acol[i] == p.tap_acol[i - 1] && (((p.tap_a2_mask >> i) ^ (p.tap_a2_mask >> (i - 1))) & 1u) == 0)
        p.tap_share_mask |= 1u << i;
    p.tiles_n = 1;
    p.a_stages = (ResidentSmem::BUDGET - ResidentSmem::FIXED - w_bytes) / ResidentSmem::A_BYTES;
    if (p.a_stages > ResidentSmem::MAX_STAGES) p.a_stages = ResidentSmem::MAX_STAGES;
    const int tiles = p.tiles_m * p.batch;
    g.kernel = CONV_RESIDENT;
    g.block_n = p.n_pad;
    g.grid = tiles < max_ctas ? tiles : max_ctas;
    g.smem_bytes = ResidentSmem::FIXED + w_bytes + p.a_stages * ResidentSmem::A_BYTES;
    g.w_box_rows = p.n_pad;
    g.l2_promo_128 = 1;
    *out = g;
    return 0;
  }

  // CTA pairs (cta_group::2, 256 x 256 tiles) pay ~1 us of extra prologue (cluster barriers) and win once the mainloop dominates
  // (K >= 2048: 33.3 -> 31.3 us at N=1024, K=4096; tools/gemm_microbench.py)
  const bool pair_shape = !any_mn && d.M > BLOCK_M && (long long)d.K * d.num_taps >= 2048;
  // tile-N choice: fewest waves, then the wider tile (less A re-read)
  int block_n = d.block_n;
  if (block_n == 0) {
    if (d.N <= 128) block_n = 128;
    else {
      const long long t256 = (long long)p.tiles_m * ((d.N + 255) / 256) * d.batch;
      const long long t128 = (long long)p.tiles_m * ((d.N + 127) / 128) * d.batch;
      const long long cost256 = ((t256 + sms - 1) / sms) * 2, cost128 = ((t128 + sms - 1) / sms);
      // where the 256-wide choice leads to the CTA-pair / fused split-fp16 kernels, 128-wide tiles only when they save at least a fifth of the
      // waves: the pair tile has twice the arithmetic intensity per staged byte.  (A bare "fewer waves" rule picked the 1-CTA 128-wide kernel for 29 vs 30 waves
      // at M = 67 840 and ran the N = 1024 / 4096 layers of a 256-clip batch at half the fused kernel's rate: tools/batch_scaling.py.)
      const bool pair_possible = pair_shape && d.cta_pair >= 0;
      block_n = (pair_possible ? cost128 * 5 < cost256 * 4 : cost128 < cost256) ? 128 : 256;
    }
  }
  DSB_REQUIRE(block_n == 128 || block_n == 256, "dsb_gemm_ex: block_n must be 0, 128 or 256");
  DSB_REQUIRE(!(any_mn && d.cta_pair > 0), "dsb_gemm_ex: the cta_group::2 kernel takes K-major operands only");
  DSB_REQUIRE(!(any_mn && p.tap_a2_mask), "dsb_gemm_ex: a second A operand is K-major only");
  // pairs by default whenever the library chose 256-wide tiles for a pair-worthy shape
  const bool use_pair = !any_mn && (d.cta_pair > 0 || (d.cta_pair == 0 && d.block_n == 0 && block_n == 256 && pair_shape));
  // split-fp16 tap list -- per spatial tap j the triple (shift_j, A lo, W hi), (shift_j, A hi, W lo), (shift_j, A hi, W hi) with constant hi -> lo column
  // distances: run the three passes off ONE staged copy of the four tiles (Linear layers: one unshifted triple; convs: 9 / 3 / 2 shifted triples)
  bool f3_pattern = kind == DSB_DTYPE_F16 && d.num_taps % 3 == 0 && !p.tap_a2_mask && !p.b_batched && !any_mn && d.K % 64 == 0 && d.M > BLOCK_M;
  int f3_lo_a = 0, f3_lo_w = 0;
  if (f3_pattern) {
    f3_lo_a = p.tap_acol[0] - p.tap_acol[1];
    f3_lo_w = p.tap_wcol[1] - p.tap_wcol[0];
    for (int j = 0; j < d.num_taps && f3_pattern; j += 3)
      f3_pattern = p.tap_shift[j] == p.tap_shift[j + 1] && p.tap_shift[j] == p.tap_shift[j + 2] && p.tap_acol[j + 1] == p.tap_acol[j + 2] &&
                   p.tap_acol[j] - p.tap_acol[j + 1] == f3_lo_a && p.tap_wcol[j] == p.tap_wcol[j + 2] && p.tap_wcol[j + 1] - p.tap_wcol[j] == f3_lo_w;
    f3_pattern = f3_pattern && f3_lo_a > 0 && f3_lo_w > 0;
  }
  const bool f3_linear = f3_pattern && d.num_taps == 3 && p.tap_shift[0] == 0 && d.batch == 1;  // the denoiser's Linear layers (any N)
  // conv form: whenever the caller left tile shape and pairing to the library
  const bool f3_conv = f3_pattern && !f3_linear && d.block_n == 0 && d.cta_pair == 0;
  const bool fused3 = f3_pattern && ((use_pair && f3_linear) || f3_conv);
  const bool pair_tiles = use_pair || fused3;
  if (pair_tiles) {
    block_n = fused3 && d.N <= 128 ? 128 : 256;
    p.tiles_m = (d.M + 2 * BLOCK_M - 1) / (2 * BLOCK_M);
  }
  p.tiles_n = (d.N + block_n - 1) / block_n;
  const long long tiles = (long long)p.tiles_m * p.tiles_n * p.batch;
  if (pair_tiles) {
    int pairs = max_ctas / 2;
    if (pairs < 1) pairs = 1;
    if (tiles < pairs) pairs = (int)tiles;
    g.grid = 2 * pairs;
  } else {
    g.grid = tiles < max_ctas ? (int)tiles : max_ctas;
  }
  if (fused3) {
    p.f3_nsp = d.num_taps / 3;
    p.lo_a = f3_lo_a;
    p.lo_w = f3_lo_w;
    for (int j = 0; j < p.f3_nsp; ++j) {  // triple j -> spatial tap j: (row shift, hi-half column of A, hi-half column of W)
      const int sh = p.tap_shift[3 * j], ac = p.tap_acol[3 * j + 1], wc = p.tap_wcol[3 * j];
      p.tap_shift[j] = sh; p.tap_acol[j] = ac; p.tap_wcol[j] = wc;
    }
    g.kernel = GEMM_F16X3_PAIR;
    g.smem_bytes = block_n == 256 ? PairSplitSmem<256>::TOTAL : PairSplitSmem<128>::TOTAL;
  } else if (use_pair) {
    g.kernel = GEMM_PAIR;
    g.smem_bytes = PairSmem::TOTAL;
  } else {
    g.kernel = GEMM_1CTA;
    g.smem_bytes = block_n == 256 ? GemmSmem<256>::TOTAL : GemmSmem<128>::TOTAL;
  }
  g.block_n = block_n;
  g.w_box_rows = pair_tiles ? block_n / 2 : block_n;
  *out = g;
  return 0;
}

}  // namespace dsb
