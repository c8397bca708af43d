// TMA + tcgen05 GEMM for sm_100a:  out[b][M,N] = epilogue( sum_tap A[b][m + shift_tap, :Kc] . W[n, tap*Kc : (tap+1)*Kc]^T )
//
// * A and W are K-contiguous ("TN"), i.e. torch.nn.Linear's activation (M,K) and weight (N,K) as they lie in HBM.
// * operands: TF32 (fp32 containers, kind::tf32) or BF16 (kind::f16); accumulation fp32 in TMEM.
// * "taps": the K loop runs over (tap, channel-block); each tap reads A rows shifted by shift_tap.  With one tap this is
//   a plain Linear layer (Text2ImageTransformer, reference transformer_utils.py:45-57,95-108,248-253,345-348); with 9 / 3 / 7
//   taps on zero-padded channels-last buffers it is the implicit-GEMM form of the SpecVQGAN decoder's 3x3 convs (reference
//   specvqgan/modules/diffusionmodules/model.py:92-151) and the MelGAN convs (reference vocoder/modules.py:72-126).
// * warp-specialised persistent kernel: warp0 = TMA producer, warp1 = tcgen05.mma issuer (+TMEM owner), warps2-5 = epilogue
//   (TMEM -> registers -> bias / GELU2 / residual / tf32-round -> HBM); smem ring of kStages, 2 TMEM accumulator stages.
#include "common.cuh"
#include "gemm_plan.cuh"
#include <cuda_bf16.h>
#include <cuda_fp16.h>

namespace dsb {

constexpr int MN_BOX_BYTES_C = 64 * 128;
constexpr int GEMM_THREADS = 320;  // warp0 TMA, warp1 MMA, warps 2..9 epilogue
constexpr int MN_BOX_BYTES = 64 * ROW_BYTES;  // one MN-major TMA box: 64 K rows x 64 two-byte columns
constexpr int EPI_LD = 36;  // padded row stride (floats) of the epilogue transpose tile: 16-byte aligned rows, conflict-free

// SW128 MN-major UMMA descriptor (canonical layout ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte units): a 64-column block is 64 K rows of
// 128 bytes; LBO = distance between 64-column blocks (one TMA box, 8 KB), SBO = distance between groups of 8 K rows (1 KB).
__device__ __forceinline__ uint64_t make_sw128_mnmajor_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(MN_BOX_BYTES_C >> 4) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

// One output tile's epilogue for one warp: TMEM -> registers -> XOR-swizzled smem transpose -> bias / activation / residual ->
// coalesced global stores.  Shared by the 1-CTA and the CTA-pair kernels (row_base = first row of this warp's 32-row slab).
template <int BLOCK_N>
__device__ __forceinline__ void epilogue_tile(const GemmParams& p, float* sw, uint32_t tmem_acc, uint64_t* tmem_full_bar, uint32_t aphase,
                                              int row_base, int n_blk, int b, int q, int half, int lane) {
  const bool has_geo = p.geo_P > 0;
  const int out_mode = (p.flags & DSB_GEMM_OUT_F16_SPLIT) ? 3 : ((p.flags & DSB_GEMM_OUT_F16) ? 1 : ((p.flags & DSB_GEMM_OUT_BF16) ? 2 : 0));
  const int act = (p.flags & DSB_GEMM_GELU2) ? 1 : ((p.flags & DSB_GEMM_LRELU) ? 2 : ((p.flags & DSB_GEMM_TANH) ? 3 : 0));
  const bool do_round = (p.flags & DSB_GEMM_ROUND_TF32) != 0;
  const bool dual = (p.flags & DSB_GEMM_DUAL_LRELU) != 0;
  const bool res_first = (p.flags & DSB_GEMM_RES_BEFORE_ACT) != 0;
  const int out_es = out_mode ? 2 : 4;
  const bool vec_ok = ((p.ldo & 3) == 0) && ((p.out_bstride & 3) == 0) && ((p.split_off & 3) == 0) && ((p.dual_off & 3) == 0) && ((p.ocg & 3) == 0) &&
                      ((p.ocg_stride & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.out) & (4 * out_es - 1)) == 0) &&
                      (!p.residual || (((p.ld_res & 3) == 0) && ((p.res_bstride & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.residual) & 15) == 0))) &&
                      (!p.bias || ((reinterpret_cast<uintptr_t>(p.bias) & 15) == 0));
  const int c4 = lane & 7;    // float4 column slot inside the 32-column chunk
  const int rsub = lane >> 3; // row inside each group of 4 rows
      uint32_t ok_mask = 0, in_mask = 0;  // bit i: row (row_base + i*4 + rsub) exists / is an interior row
#pragma unroll 1
  for (int i = 0; i < 8; ++i) {
    const int row = row_base + i * 4 + rsub;
    if (row < p.M) ok_mask |= 1u << i;
    bool interior = true;
    if (has_geo) {
      const int pp = row % p.geo_P;
      const int y = pp / p.geo_Wp, x = pp - y * p.geo_Wp;
      interior = (y >= p.geo_y0) && (y < p.geo_y1) && (x >= p.geo_x0) && (x < p.geo_x1);
    }
    if (interior) in_mask |= 1u << i;
  }
  const uint32_t t_row = tmem_acc + (static_cast<uint32_t>(q * 32) << 16);
  const long long out_boff = (long long)b * p.out_bstride;
  const float* res_b = p.residual ? p.residual + (long long)b * p.res_bstride : nullptr;
  const int n_chunks = min(BLOCK_N / 32, (p.N - n_blk * BLOCK_N + 31) / 32);

  // bias + residual are fetched one chunk ahead (the first one while the mainloop still runs)
  float4 rz_next[8];
  float4 bz_next = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int i = 0; i < 8; ++i) rz_next[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  auto prefetch = [&](int c) {
    const int col = n_blk * BLOCK_N + c * 32 + c4 * 4;
    if (vec_ok && (col + 3 < p.N)) {  // tail / unaligned chunks fetch inside the slow path instead
      if (p.bias) bz_next = __ldg(reinterpret_cast<const float4*>(p.bias + col));
      if (res_b) {
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if ((ok_mask >> i) & 1u) rz_next[i] = *reinterpret_cast<const float4*>(res_b + (long long)(row_base + i * 4 + rsub) * p.ld_res + col);
      }
    }
  };
  if (half < n_chunks) prefetch(half);
  mbar_wait(tmem_full_bar, aphase);
  tc_fence_after();
#pragma unroll 1
  for (int c = half; c < n_chunks; c += 2) {
    const int col0 = n_blk * BLOCK_N + c * 32;
    {
      uint32_t v[32];
      tmem_ld_32x32(t_row + c * 32, v);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 8; ++j)
    *reinterpret_cast<uint4*>(sw + lane * 32 + ((j ^ (lane & 7)) << 2)) = make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    }
    __syncwarp();
    const int col = col0 + c4 * 4;
    if (vec_ok && (col0 + 32 <= p.N)) {
      // ---------------- fast path: whole chunk in range, 16-byte aligned everywhere
      float x[32];
      float4 rz_cur[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
    const int r = i * 4 + rsub;
    const float4 a4 = *reinterpret_cast<const float4*>(sw + r * 32 + ((c4 ^ (r & 7)) << 2));
    rz_cur[i] = rz_next[i];
    x[4 * i + 0] = fmaf(a4.x, p.alpha, bz_next.x); x[4 * i + 1] = fmaf(a4.y, p.alpha, bz_next.y);
    x[4 * i + 2] = fmaf(a4.z, p.alpha, bz_next.z); x[4 * i + 3] = fmaf(a4.w, p.alpha, bz_next.w);
      }
      if (c + 2 < n_chunks) prefetch(c + 2);  // issued before this chunk's stores (out may alias residual)
      if (res_b && res_first) {
#pragma unroll
    for (int i = 0; i < 8; ++i) { x[4 * i] += rz_cur[i].x; x[4 * i + 1] += rz_cur[i].y; x[4 * i + 2] += rz_cur[i].z; x[4 * i + 3] += rz_cur[i].w; }
      }
      if (act == 1) {
#pragma unroll
    for (int e = 0; e < 32; ++e) x[e] = __fdividef(x[e], 1.0f + __expf(-1.702f * x[e]));
      } else if (act == 2) {
#pragma unroll
    for (int e = 0; e < 32; ++e) x[e] = x[e] > 0.f ? x[e] : 0.2f * x[e];
      } else if (act == 3) {
#pragma unroll
    for (int e = 0; e < 32; ++e) {  // tanh(x) = 1 - 2 / (1 + exp(2x)), clamped so exp stays finite
      const float z = fminf(fmaxf(x[e], -15.f), 15.f);
      x[e] = 1.0f - __fdividef(2.0f, 1.0f + __expf(2.0f * z));
    }
      }
      if (res_b && !res_first) {
#pragma unroll
    for (int i = 0; i < 8; ++i) { x[4 * i] += rz_cur[i].x; x[4 * i + 1] += rz_cur[i].y; x[4 * i + 2] += rz_cur[i].z; x[4 * i + 3] += rz_cur[i].w; }
      }
      if (do_round) {
#pragma unroll
    for (int e = 0; e < 32; ++e) x[e] = round_tf32(x[e]);
      }
      if (has_geo) {
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (!((in_mask >> i) & 1u)) { x[4 * i] = 0.f; x[4 * i + 1] = 0.f; x[4 * i + 2] = 0.f; x[4 * i + 3] = 0.f; }
      }
      if (p.amax_out) {  // calibration runs only: largest magnitude this launch would store
    float m = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if ((ok_mask >> i) & 1u) m = fmaxf(m, fmaxf(fmaxf(fabsf(x[4 * i]), fabsf(x[4 * i + 1])), fmaxf(fabsf(x[4 * i + 2]), fabsf(x[4 * i + 3]))));
    int mi = __float_as_int(m);  // non-negative floats (and +inf, NaN payloads) order like their bit patterns
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mi = max(mi, __shfl_xor_sync(0xffffffffu, mi, o));
    if (lane == 0) atomicMax(reinterpret_cast<int*>(p.amax_out), mi);
      }
      if (p.flags & DSB_GEMM_NO_STORE) {
      } else if (out_mode == 0) {
    float* op = reinterpret_cast<float*>(p.out) + out_boff + (long long)(row_base + rsub) * p.ldo + col;
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if ((ok_mask >> i) & 1u) *reinterpret_cast<float4*>(op + (long long)i * 4 * p.ldo) = make_float4(x[4 * i], x[4 * i + 1], x[4 * i + 2], x[4 * i + 3]);
      } else if (out_mode == 1) {
    __half* op = reinterpret_cast<__half*>(p.out) + out_boff + (long long)(row_base + rsub) * p.ldo + col;
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if ((ok_mask >> i) & 1u) {
        __half2 h0 = __floats2half2_rn(x[4 * i], x[4 * i + 1]), h1 = __floats2half2_rn(x[4 * i + 2], x[4 * i + 3]);
        uint2 u;
        u.x = *reinterpret_cast<uint32_t*>(&h0); u.y = *reinterpret_cast<uint32_t*>(&h1);
        *reinterpret_cast<uint2*>(op + (long long)i * 4 * p.ldo) = u;
      }
      } else if (out_mode == 3) {  // fp16 (hi | lo) pair: the A operand of a split-fp16 GEMM / attention
    const int ocol = p.ocg > 0 ? (col / p.ocg) * p.ocg_stride + col % p.ocg : col;
    __half* op = reinterpret_cast<__half*>(p.out) + out_boff + (long long)(row_base + rsub) * p.ldo + ocol;
#pragma unroll 1
    for (int pass = 0; pass < (dual ? 2 : 1); ++pass) {
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if ((ok_mask >> i) & 1u) {
          const __half2 h0 = __floats2half2_rn(x[4 * i], x[4 * i + 1]), h1 = __floats2half2_rn(x[4 * i + 2], x[4 * i + 3]);
          const __half2 l0 = __floats2half2_rn(x[4 * i] - __low2float(h0), x[4 * i + 1] - __high2float(h0));
          const __half2 l1 = __floats2half2_rn(x[4 * i + 2] - __low2float(h1), x[4 * i + 3] - __high2float(h1));
          uint2 u, w;
          u.x = *reinterpret_cast<const uint32_t*>(&h0); u.y = *reinterpret_cast<const uint32_t*>(&h1);
          w.x = *reinterpret_cast<const uint32_t*>(&l0); w.y = *reinterpret_cast<const uint32_t*>(&l1);
          *reinterpret_cast<uint2*>(op + (long long)i * 4 * p.ldo) = u;
          *reinterpret_cast<uint2*>(op + (long long)i * 4 * p.ldo + p.split_off) = w;
        }
      if (dual) {  // second copy: LeakyReLU(0.2) of the value just stored (the next conv's input; the raw copy feeds the 1x1 shortcut)
#pragma unroll
        for (int e = 0; e < 32; ++e) x[e] = x[e] > 0.f ? x[e] : 0.2f * x[e];
        op += p.dual_off;
      }
    }
      } else {
    __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(p.out) + out_boff + (long long)(row_base + rsub) * p.ldo + col;
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if ((ok_mask >> i) & 1u) {
        __nv_bfloat162 h0 = __floats2bfloat162_rn(x[4 * i], x[4 * i + 1]), h1 = __floats2bfloat162_rn(x[4 * i + 2], x[4 * i + 3]);
        uint2 u;
        u.x = *reinterpret_cast<uint32_t*>(&h0); u.y = *reinterpret_cast<uint32_t*>(&h1);
        *reinterpret_cast<uint2*>(op + (long long)i * 4 * p.ldo) = u;
      }
      }
    } else {
      // ---------------- slow path (N tail, unaligned leading dimensions): rolled scalar loops, rarely taken
      if (c + 2 < n_chunks) prefetch(c + 2);
#pragma unroll 1
      for (int i = 0; i < 8; ++i) {
    if (!((ok_mask >> i) & 1u)) continue;
    const int r = i * 4 + rsub;
    const long long row = row_base + r;
    const float4 a4 = *reinterpret_cast<const float4*>(sw + r * 32 + ((c4 ^ (r & 7)) << 2));
    const float av[4] = {a4.x, a4.y, a4.z, a4.w};
#pragma unroll 1
    for (int k = 0; k < 4; ++k) {
      if (col + k >= p.N) break;
      float xv = av[k] * p.alpha + (p.bias ? __ldg(p.bias + col + k) : 0.f);
      const float rv = res_b ? res_b[row * p.ld_res + col + k] : 0.f;
      if (res_first) xv += rv;
      if (act == 1) xv = __fdividef(xv, 1.0f + __expf(-1.702f * xv));
      else if (act == 2) xv = xv > 0.f ? xv : 0.2f * xv;
      else if (act == 3) { const float z = fminf(fmaxf(xv, -15.f), 15.f); xv = 1.0f - __fdividef(2.0f, 1.0f + __expf(2.0f * z)); }
      if (!res_first) xv += rv;
      if (do_round) xv = round_tf32(xv);
      if (!((in_mask >> i) & 1u)) xv = 0.f;
      const long long o = out_boff + row * p.ldo + col + k;
      if (p.amax_out) atomicMax(reinterpret_cast<int*>(p.amax_out), __float_as_int(fabsf(xv)));
      if (p.flags & DSB_GEMM_NO_STORE) continue;
      if (out_mode == 0) reinterpret_cast<float*>(p.out)[o] = xv;
      else if (out_mode == 1) reinterpret_cast<__half*>(p.out)[o] = __float2half_rn(xv);
      else if (out_mode == 3) {
        const int cc = col + k;
        const long long o3 = out_boff + row * p.ldo + (p.ocg > 0 ? (cc / p.ocg) * p.ocg_stride + cc % p.ocg : cc);
        __half hv = __float2half_rn(xv);
        reinterpret_cast<__half*>(p.out)[o3] = hv;
        reinterpret_cast<__half*>(p.out)[o3 + p.split_off] = __float2half_rn(xv - __half2float(hv));
        if (dual) {
          const float yv = xv > 0.f ? xv : 0.2f * xv;
          hv = __float2half_rn(yv);
          reinterpret_cast<__half*>(p.out)[o3 + p.dual_off] = hv;
          reinterpret_cast<__half*>(p.out)[o3 + p.dual_off + p.split_off] = __float2half_rn(yv - __half2float(hv));
        }
      }
      else reinterpret_cast<__nv_bfloat16*>(p.out)[o] = __float2bfloat16(xv);
    }
      }
    }
    __syncwarp();  // the smem tile is rewritten by the next chunk
  }
}

template <int BLOCK_N, int KIND>  // KIND = DSB_DTYPE_*
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_a2, const __grid_constant__ CUtensorMap tmap_b,
                    const __grid_constant__ GemmParams p) {
  using S = GemmSmem<BLOCK_N>;
  constexpr int STAGES = S::STAGES;
  constexpr uint32_t TMEM_COLS = 2 * BLOCK_N;  // 2 accumulator stages; 256 or 512 (power of two)
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * S::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full = empty_bar + STAGES;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  float* epi_smem = reinterpret_cast<float*>(smem + STAGES * S::STAGE_BYTES + 256);  // 8 warps x 32 x 32 floats (XOR-swizzled)

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_tiles = p.tiles_m * p.tiles_n * p.batch;
  const int num_kb = p.kb_per_tap * p.num_taps;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmap_a);
    prefetch_tmap(&tmap_a2);
    prefetch_tmap(&tmap_b);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full[s], 1);
      mbar_init(&tmem_empty[s], 8);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr, TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  // everything above (barrier init, TMEM allocation, tensor-map prefetch) overlapped the predecessor's tail
  pdl_wait();
  pdl_trigger();

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int m_blk = tile % p.tiles_m;
        const int n_blk = (tile / p.tiles_m) % p.tiles_n;
        const int b = tile / (p.tiles_m * p.tiles_n);
        for (int kb = 0; kb < num_kb; ++kb) {
          const int tap = kb / p.kb_per_tap;
          const int c0 = (kb - tap * p.kb_per_tap) * p.block_k;
          mbar_wait(&empty_bar[stage], phase ^ 1);
          mbar_arrive_expect_tx(&full_bar[stage], S::STAGE_BYTES);
          uint8_t* sa = smem + stage * S::STAGE_BYTES;
          if (p.a_mn) {
#pragma unroll
            for (int j = 0; j < BLOCK_M / 64; ++j) tma_load_3d(&tmap_a, &full_bar[stage], sa + j * MN_BOX_BYTES, m_blk * BLOCK_M + j * 64, c0, b);
          } else {
            tma_load_3d(((p.tap_a2_mask >> tap) & 1u) ? &tmap_a2 : &tmap_a, &full_bar[stage], sa, c0 + p.tap_acol[tap], m_blk * BLOCK_M + p.tap_shift[tap], b);
          }
          if (p.b_mn) {
#pragma unroll
            for (int j = 0; j < BLOCK_N / 64; ++j)
              tma_load_3d(&tmap_b, &full_bar[stage], sa + S::A_BYTES + j * MN_BOX_BYTES, n_blk * BLOCK_N + j * 64, c0, p.b_batched ? b : 0);
          } else {
            tma_load_3d(&tmap_b, &full_bar[stage], sa + S::A_BYTES, p.tap_wcol[tap] + c0, n_blk * BLOCK_N, p.b_batched ? b : 0);
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer (one thread)
    if (lane == 0) {
      const uint32_t idesc = make_idesc(KIND, BLOCK_M, BLOCK_N) | (p.a_mn ? (1u << 15) : 0u) | (p.b_mn ? (1u << 16) : 0u);
      // descriptor step per 16-element K slice: K-major = 32 bytes inside the swizzle row, MN-major = 16 rows of 128 bytes
      const uint32_t a_step = p.a_mn ? (16 * ROW_BYTES) >> 4 : 2, b_step = p.b_mn ? (16 * ROW_BYTES) >> 4 : 2;
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
        const int as = it & 1;
        const uint32_t aphase = (it >> 1) & 1;
        mbar_wait(&tmem_empty[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BLOCK_N;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * S::STAGE_BYTES);
          const uint64_t da = p.a_mn ? make_sw128_mnmajor_desc(sa) : make_sw128_kmajor_desc(sa);
          const uint64_t db = p.b_mn ? make_sw128_mnmajor_desc(sa + S::A_BYTES) : make_sw128_kmajor_desc(sa + S::A_BYTES);
#pragma unroll
          for (int k = 0; k < 4; ++k)  // 4 K slices (16 elements of 2 bytes / 8 of 4 bytes) per 64-deep k-block
            umma<KIND == DSB_DTYPE_TF32>(d_tmem, da + a_step * k, db + b_step * k, idesc, (kb | k) != 0 ? 1u : 0u);
          umma_commit(&empty_bar[stage]);  // frees the smem slot once these MMAs retire
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tmem_full[as]);
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue warps (2..9): TMEM lane quadrant = warp % 4,
    // two warps per quadrant splitting the 32-column chunks (even / odd).
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;  // 0: even chunks, 1: odd chunks
    float* sw = epi_smem + (warp - 2) * (32 * 32);
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      const int m_blk = tile % p.tiles_m;
      const int n_blk = (tile / p.tiles_m) % p.tiles_n;
      const int b = tile / (p.tiles_m * p.tiles_n);
      const int as = it & 1;
      const uint32_t aphase = (it >> 1) & 1;
      epilogue_tile<BLOCK_N>(p, sw, tmem_base + as * BLOCK_N, &tmem_full[as], aphase, m_blk * BLOCK_M + q * 32, n_blk, b, q, half, lane);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[as]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------ CTA-pair (cta_group::2) kernel
// Two CTAs of a cluster (one TPC) cooperate on a 256 x 256 output tile: CTA r loads its own 128 rows of A and HALF of the
// B tile (128 of the 256 N rows); the leader (rank 0) issues tcgen05.mma.cta_group::2 with M = 256, which reads A / B halves
// from both CTAs' shared memory and accumulates rows [128 r, 128 r + 128) into CTA r's TMEM.  Per k-block each SM now moves
// 32 KB in + 32 KB out of shared memory instead of 48 + 48 KB -- the 1-CTA kernel is bound by exactly that (760 vs 542
// cycles per k-block).  Protocol: both producers' TMA loads complete_tx on the LEADER's full barrier (.cta_group::2 form);
// MMA completion is multicast to both CTAs' empty / tmem_full barriers; epilogue warps of both CTAs arrive on the leader's
// tmem_empty barrier.
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t map_to_cta(uint32_t smem_addr, uint32_t rank) {  // same smem offset in CTA `rank` of the cluster
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void tma_load_3d_2sm(const CUtensorMap* m, uint32_t bar_cluster_addr, void* dst, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
template <bool kTf32>
__device__ __forceinline__ void umma_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  if constexpr (kTf32) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
  } else {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
  }
}
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar) {  // arrives on `bar` (same offset) in both CTAs of the pair
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar_cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster_addr) : "memory");
}

template <int KIND>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GEMM_THREADS, 1)
gemm_tcgen05_pair_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_a2, const __grid_constant__ CUtensorMap tmap_b,
                         const __grid_constant__ GemmParams p) {
  using S = PairSmem;
  constexpr int BLOCK_N = S::BLOCK_N;
  constexpr int STAGES = S::STAGES;
  constexpr uint32_t TMEM_COLS = 2 * BLOCK_N;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * S::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full = empty_bar + STAGES;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  float* epi_smem = reinterpret_cast<float*>(smem + STAGES * S::STAGE_BYTES + 256);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int num_tiles = p.tiles_m * p.tiles_n * p.batch;  // tiles_m counts 256-row pair tiles
  const int num_kb = p.kb_per_tap * p.num_taps;
  const int pair_id = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmap_a);
    prefetch_tmap(&tmap_a2);
    prefetch_tmap(&tmap_b);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);   // leader's copy is the one in use: its producer arms expect_tx for both CTAs' bytes
      mbar_init(&empty_bar[s], 1);  // one multicast tcgen05.commit per phase
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full[s], 1);
      mbar_init(&tmem_empty[s], 16);  // 8 epilogue warps x 2 CTAs (leader's copy is the one in use)
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // both CTAs' barriers are initialised before any remote arrive / multicast commit / peer TMA signal
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  pdl_wait();
  pdl_trigger();

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer (both CTAs)
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = pair_id; tile < num_tiles; tile += num_pairs) {
        const int m_blk = tile % p.tiles_m;
        const int n_blk = (tile / p.tiles_m) % p.tiles_n;
        const int b = tile / (p.tiles_m * p.tiles_n);
        const int row0 = m_blk * (2 * BLOCK_M) + (int)rank * BLOCK_M;
        const int nrow0 = n_blk * BLOCK_N + (int)rank * (BLOCK_N / 2);
        for (int kb = 0; kb < num_kb; ++kb) {
          const int tap = kb / p.kb_per_tap;
          const int c0 = (kb - tap * p.kb_per_tap) * p.block_k;
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (leader) mbar_arrive_expect_tx(&full_bar[stage], 2 * S::STAGE_BYTES);
          const uint32_t bar = map_to_cta(smem_u32(&full_bar[stage]), 0);
          uint8_t* sa = smem + stage * S::STAGE_BYTES;
          tma_load_3d_2sm(((p.tap_a2_mask >> tap) & 1u) ? &tmap_a2 : &tmap_a, bar, sa, c0 + p.tap_acol[tap], row0 + p.tap_shift[tap], b);
          tma_load_3d_2sm(&tmap_b, bar, sa + S::A_BYTES, p.tap_wcol[tap] + c0, nrow0, p.b_batched ? b : 0);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer: one thread of the leader CTA
    if (leader && lane == 0) {
      constexpr uint32_t idesc = make_idesc(KIND, 2 * BLOCK_M, BLOCK_N);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int tile = pair_id; tile < num_tiles; tile += num_pairs, ++it) {
        const int as = it & 1;
        const uint32_t aphase = (it >> 1) & 1;
        mbar_wait(&tmem_empty[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BLOCK_N;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * S::STAGE_BYTES);
          const uint64_t da = make_sw128_kmajor_desc(sa);
          const uint64_t db = make_sw128_kmajor_desc(sa + S::A_BYTES);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_2sm<KIND == DSB_DTYPE_TF32>(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
          umma_commit_2sm(&empty_bar[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit_2sm(&tmem_full[as]);
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue warps of both CTAs (rows [128 rank, 128 rank + 128) of the pair tile)
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    float* sw = epi_smem + (warp - 2) * (32 * 32);
    int it = 0;
    for (int tile = pair_id; tile < num_tiles; tile += num_pairs, ++it) {
      const int m_blk = tile % p.tiles_m;
      const int n_blk = (tile / p.tiles_m) % p.tiles_n;
      const int b = tile / (p.tiles_m * p.tiles_n);
      const int as = it & 1;
      const uint32_t aphase = (it >> 1) & 1;
      epilogue_tile<BLOCK_N>(p, sw, tmem_base + as * BLOCK_N, &tmem_full[as], aphase, m_blk * (2 * BLOCK_M) + (int)rank * BLOCK_M + q * 32, n_blk, b, q,
                             half, lane);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(map_to_cta(smem_u32(&tmem_empty[as]), 0));
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // nobody leaves (or frees TMEM) while the peer may still signal / read
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------------------------------ fused split-fp16 ("f16x3") CTA-pair kernel
// out = epi(alpha * (Alo Whi^T + Ahi Wlo^T + Ahi Whi^T) + bias) with A = (M, 2K) [hi | lo] and W = (N, 2K) [hi | lo].  The tap form of the same
// product streams every operand tile once PER PASS (3 x (32 KB in + 32 KB out of shared memory per SM and 64-deep k-block): exactly the MMA time,
// no slack).  Here one pipeline stage holds the four tiles of a k-block (A hi, A lo, W hi half, W lo half: 64 KB per CTA) and the issuer runs the
// three passes off them: 64 KB in + 96 KB out per 1536 MMA cycles, so the shared-memory port is no longer co-critical and L2 traffic drops by a third.
// BN = 256: 256 x 256 pair tiles (best MMA shape).  BN = 128: 256 x 128 pair tiles for N <= 128 (the decoder's 128-channel convs).
template <int BN>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GEMM_THREADS, 1)
gemm_f16x3_pair_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, const __grid_constant__ GemmParams p) {
  using S = PairSplitSmem<BN>;
  constexpr int BLOCK_N = S::BLOCK_N;
  constexpr int STAGES = S::STAGES;
  constexpr uint32_t TMEM_COLS = 2 * BLOCK_N;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * S::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full = empty_bar + STAGES;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  float* epi_smem = reinterpret_cast<float*>(smem + STAGES * S::STAGE_BYTES + 256);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int num_tiles = p.tiles_m * p.tiles_n * p.batch;  // tiles_m counts 256-row pair tiles
  const int num_kb = p.kb_per_tap;                        // k-blocks of the ORIGINAL reduction length K
  const int pair_id = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;
  const int lo_a = p.lo_a, lo_w = p.lo_w;                 // column distance from a hi half to its lo half
  const int nsp = p.f3_nsp;                               // spatial taps (1 = a Linear layer; 9 / 3 / 2 = conv taps over padded rows)

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmap_a);
    prefetch_tmap(&tmap_b);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full[s], 1);
      mbar_init(&tmem_empty[s], 16);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  pdl_wait();
  pdl_trigger();

  if (warp == 0) {
    if (lane == 0) {  // ------------------------------------------------------------ TMA producer (both CTAs): four boxes per k-block
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = pair_id; tile < num_tiles; tile += num_pairs) {
        const int m_blk = tile % p.tiles_m;
        const int n_blk = (tile / p.tiles_m) % p.tiles_n;
        const int b = tile / (p.tiles_m * p.tiles_n);
        const int row0 = m_blk * (2 * BLOCK_M) + (int)rank * BLOCK_M;
        const int nrow0 = n_blk * BLOCK_N + (int)rank * (BLOCK_N / 2);
        for (int j = 0; j < nsp; ++j) {
          const int arow = row0 + p.tap_shift[j], acol = p.tap_acol[j], wcol = p.tap_wcol[j];
          for (int kb = 0; kb < num_kb; ++kb) {
            const int c0 = kb * 64;
            mbar_wait(&empty_bar[stage], phase ^ 1);
            if (leader) mbar_arrive_expect_tx(&full_bar[stage], 2 * S::STAGE_BYTES);
            const uint32_t bar = map_to_cta(smem_u32(&full_bar[stage]), 0);
            uint8_t* sa = smem + stage * S::STAGE_BYTES;
            tma_load_3d_2sm(&tmap_a, bar, sa, acol + c0, arow, b);
            tma_load_3d_2sm(&tmap_a, bar, sa + S::TILE_A, acol + lo_a + c0, arow, b);
            tma_load_3d_2sm(&tmap_b, bar, sa + 2 * S::TILE_A, wcol + c0, nrow0, 0);
            tma_load_3d_2sm(&tmap_b, bar, sa + 2 * S::TILE_A + S::TILE_B, wcol + lo_w + c0, nrow0, 0);
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (leader && lane == 0) {  // ---------------------------------------------------- MMA issuer: lo*hi, hi*lo, hi*hi per 16-element K slice
      constexpr uint32_t idesc = make_idesc(DSB_DTYPE_F16, 2 * BLOCK_M, BLOCK_N);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int tile = pair_id; tile < num_tiles; tile += num_pairs, ++it) {
        const int as = it & 1;
        const uint32_t aphase = (it >> 1) & 1;
        mbar_wait(&tmem_empty[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BLOCK_N;
        const int num_kbt = num_kb * nsp;
        for (int kb = 0; kb < num_kbt; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * S::STAGE_BYTES);
          const uint64_t dah = make_sw128_kmajor_desc(sa), dal = make_sw128_kmajor_desc(sa + S::TILE_A);
          const uint64_t dbh = make_sw128_kmajor_desc(sa + 2 * S::TILE_A), dbl = make_sw128_kmajor_desc(sa + 2 * S::TILE_A + S::TILE_B);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            umma_2sm<false>(d_tmem, dal + 2 * k, dbh + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
            umma_2sm<false>(d_tmem, dah + 2 * k, dbl + 2 * k, idesc, 1u);
            umma_2sm<false>(d_tmem, dah + 2 * k, dbh + 2 * k, idesc, 1u);
          }
          umma_commit_2sm(&empty_bar[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit_2sm(&tmem_full[as]);
      }
    }
  } else {
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    float* sw = epi_smem + (warp - 2) * (32 * 32);
    int it = 0;
    for (int tile = pair_id; tile < num_tiles; tile += num_pairs, ++it) {
      const int m_blk = tile % p.tiles_m;
      const int n_blk = (tile / p.tiles_m) % p.tiles_n;
      const int b = tile / (p.tiles_m * p.tiles_n);
      const int as = it & 1;
      const uint32_t aphase = (it >> 1) & 1;
      epilogue_tile<BLOCK_N>(p, sw, tmem_base + as * BLOCK_N, &tmem_full[as], aphase, m_blk * (2 * BLOCK_M) + (int)rank * BLOCK_M + q * 32, n_blk, b, q,
                             half, lane);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(map_to_cta(smem_u32(&tmem_empty[as]), 0));
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------------------------------ resident-W narrow-channel kernel
// MelGAN's last stages are convs over 32 / 64 channels and millions of time rows (reference vocoder/modules.py:104-126): the generic kernel
// re-streams every tap's W box and a 64-column A box per (tap, pass) for each 128-row tile -- 288 KB of L2 -> smem traffic per tile of
// 16 KB of state, and measures L2-bound (7.2 TB/s, 0.12 of the HBM roofline).  Here each tap is one 64-deep k-block; ALL taps' W boxes
// (num_taps x n_pad rows x 128 B, <= 96 KB) are loaded once per CTA and stay in shared memory, and consecutive taps that read the same A box
// (the hi*hi / hi*lo passes of one spatial tap, or the folded [hi | lo] . [Wh | Wh], [hi | lo] . [Wl | 0] pair of a 32-channel row) share one
// staged copy.  MMA N = n_pad (16..128), accumulators 2 x 128 TMEM columns, epilogue shared with the generic kernel.
template <int KIND>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
conv_resident_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_a2, const __grid_constant__ CUtensorMap tmap_b,
                     const __grid_constant__ GemmParams p) {
  using S = ResidentSmem;
  // 4 accumulator stages: the MMA issuer runs up to three tiles ahead of the epilogue, so staged A boxes are consumed (and their ring slots
  // re-armed) as they land instead of waiting for an epilogue -- the launch is a stream of 16 KB boxes with a few microseconds of latency each
  constexpr uint32_t ACC_COLS = 128, ACC_STAGES = 4, TMEM_COLS = ACC_COLS * ACC_STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int STAGES = p.a_stages;
  const int wbox = p.n_pad * ROW_BYTES;
  uint8_t* w_smem = smem + STAGES * S::A_BYTES;
  uint8_t* tail = w_smem + p.num_taps * wbox;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(tail);
  uint64_t* empty_bar = full_bar + S::MAX_STAGES;
  uint64_t* tmem_full = empty_bar + S::MAX_STAGES;
  uint64_t* tmem_empty = tmem_full + ACC_STAGES;
  uint64_t* w_bar = tmem_empty + ACC_STAGES;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(w_bar + 1);
  float* epi_smem = reinterpret_cast<float*>(tail + S::BAR_BYTES);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_tiles = p.tiles_m * p.batch;
  // N <= 32 is a single 32-column chunk: the two epilogue warps of a TMEM lane quadrant then alternate TILES instead of chunks
  const bool alt_tiles = p.N <= 32;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmap_a);
    prefetch_tmap(&tmap_a2);
    prefetch_tmap(&tmap_b);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < (int)ACC_STAGES; ++s) {
      mbar_init(&tmem_full[s], 1);
      mbar_init(&tmem_empty[s], alt_tiles ? 4 : 8);
    }
    mbar_init(w_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr, TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  pdl_wait();
  pdl_trigger();

  if (warp == 0) {
    if (lane == 0) {
      mbar_arrive_expect_tx(w_bar, static_cast<uint32_t>(p.num_taps * wbox));
      for (int t = 0; t < p.num_taps; ++t) tma_load_3d(&tmap_b, w_bar, w_smem + t * wbox, p.tap_wcol[t], 0, 0);
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int m_blk = tile % p.tiles_m;
        const int b = tile / p.tiles_m;
        for (int t = 0; t < p.num_taps; ++t) {
          if ((p.tap_share_mask >> t) & 1u) continue;
          mbar_wait(&empty_bar[stage], phase ^ 1);
          mbar_arrive_expect_tx(&full_bar[stage], S::A_BYTES);
          tma_load_3d(((p.tap_a2_mask >> t) & 1u) ? &tmap_a2 : &tmap_a, &full_bar[stage], smem + stage * S::A_BYTES, p.tap_acol[t],
                      m_blk * BLOCK_M + p.tap_shift[t], b);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = make_idesc(KIND, BLOCK_M, p.n_pad);
      const uint32_t w_addr = smem_u32(w_smem);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      mbar_wait(w_bar, 0);
      tc_fence_after();
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
        const int as = it & (ACC_STAGES - 1);
        const uint32_t aphase = (it / ACC_STAGES) & 1;
        mbar_wait(&tmem_empty[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * ACC_COLS;
        for (int t = 0; t < p.num_taps; ++t) {
          if (!((p.tap_share_mask >> t) & 1u)) {
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after();
          }
          const uint64_t da = make_sw128_kmajor_desc(smem_u32(smem + stage * S::A_BYTES));
          const uint64_t db = make_sw128_kmajor_desc(w_addr + t * wbox);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma<false>(d_tmem, da + 2 * k, db + 2 * k, idesc, (t | k) != 0 ? 1u : 0u);
          if (t + 1 == p.num_taps || !((p.tap_share_mask >> (t + 1)) & 1u)) {
            umma_commit(&empty_bar[stage]);  // this A box has no further reader
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
        umma_commit(&tmem_full[as]);
      }
    }
  } else {
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    float* sw = epi_smem + (warp - 2) * (32 * 32);
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      if (alt_tiles && (it & 1) != half) continue;
      const int as = it & (ACC_STAGES - 1);
      const int m_blk = tile % p.tiles_m;
      const int b = tile / p.tiles_m;
      const uint32_t aphase = (it / ACC_STAGES) & 1;
      epilogue_tile<128>(p, sw, tmem_base + as * ACC_COLS, &tmem_full[as], aphase, m_blk * BLOCK_M + q * 32, 0, b, q, alt_tiles ? 0 : half, lane);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[as]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------ host side
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  return fn;
}

// 3-D map (K, rows, batch) over a K-contiguous matrix; box = (128 bytes of K, box_rows, 1); SWIZZLE_128B; OOB -> 0
int make_operand_map(CUtensorMap* map, const void* ptr, int kind, long long kdim, long long rows, long long batch,
                            long long ld_elems, long long bstride_elems, int box_rows, int l2_promo_128) {
  PFN_encodeTiled enc = get_encode();
  DSB_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled entry point unavailable (no CUDA driver?)");
  const int es = kind == DSB_DTYPE_TF32 ? 4 : 2;
  DSB_REQUIRE((reinterpret_cast<uintptr_t>(ptr) & 15) == 0, "GEMM operand pointer must be 16-byte aligned");
  DSB_REQUIRE((ld_elems * es) % 16 == 0, "GEMM operand leading dimension must be a multiple of 16 bytes (ld=%lld)", ld_elems);
  DSB_REQUIRE(batch == 1 || (bstride_elems * es) % 16 == 0, "GEMM batch stride must be a multiple of 16 bytes");
  cuuint64_t gdim[3] = {(cuuint64_t)kdim, (cuuint64_t)rows, (cuuint64_t)batch};
  cuuint64_t gstr[2] = {(cuuint64_t)(ld_elems * es), (cuuint64_t)((batch == 1 ? ld_elems * rows : bstride_elems) * es)};
  cuuint32_t box[3] = {(cuuint32_t)(ROW_BYTES / es), (cuuint32_t)box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, kind == DSB_DTYPE_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : (kind == DSB_DTYPE_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32), 3, const_cast<void*>(ptr), gdim, gstr,
                   box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   // state rows [raw pair | activated pair] are read one 128-byte half at a time: a 256-byte promotion would fetch the other half too
                   l2_promo_128 ? CU_TENSOR_MAP_L2_PROMOTION_L2_128B : CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  DSB_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (%d): k=%lld rows=%lld batch=%lld ld=%lld", (int)r, kdim, rows, batch, ld_elems);
  return 0;
}

// 3-D map (MN, K rows, batch) over an MN-contiguous operand; box = (64 columns = 128 bytes, 64 K rows, 1); SWIZZLE_128B; OOB -> 0
int make_operand_map_mn(CUtensorMap* map, const void* ptr, int kind, long long mn, long long krows, long long batch, long long ld_elems,
                        long long bstride_elems) {
  PFN_encodeTiled enc = get_encode();
  DSB_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled entry point unavailable (no CUDA driver?)");
  DSB_REQUIRE(kind != DSB_DTYPE_TF32, "MN-major GEMM operands are implemented for the 2-byte types only");
  DSB_REQUIRE((reinterpret_cast<uintptr_t>(ptr) & 15) == 0, "GEMM operand pointer must be 16-byte aligned");
  DSB_REQUIRE((ld_elems * 2) % 16 == 0, "GEMM operand leading dimension must be a multiple of 16 bytes (ld=%lld)", ld_elems);
  DSB_REQUIRE(batch == 1 || (bstride_elems * 2) % 16 == 0, "GEMM batch stride must be a multiple of 16 bytes");
  cuuint64_t gdim[3] = {(cuuint64_t)mn, (cuuint64_t)krows, (cuuint64_t)batch};
  cuuint64_t gstr[2] = {(cuuint64_t)(ld_elems * 2), (cuuint64_t)((batch == 1 ? ld_elems * krows : bstride_elems) * 2)};
  cuuint32_t box[3] = {64, 64, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, kind == DSB_DTYPE_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(ptr), gdim, gstr,
                   box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  DSB_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (MN-major) failed (%d): mn=%lld k=%lld batch=%lld ld=%lld", (int)r, mn, krows, batch, ld_elems);
  return 0;
}

// One PDL launch of `Kern` with the plan's grid and shared memory; the first launch of each kernel raises its dynamic shared-memory limit
// to `smem_limit`.
template <auto Kern, typename... Maps>
static int launch(const GemmPlan& g, int smem_limit, cudaStream_t st, const Maps&... maps) {
  static bool attr_done = false;
  if (!attr_done) {
    DSB_CHECK_CUDA(cudaFuncSetAttribute(Kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_limit));
    attr_done = true;
  }
  DSB_CHECK_CUDA(launch_pdl(Kern, dim3(g.grid), dim3(GEMM_THREADS), g.smem_bytes, st, maps..., g.p));
  return 0;
}

static int launch_plan(const GemmPlan& g, int kind, const CUtensorMap& ma, const CUtensorMap& ma2, const CUtensorMap& mb, cudaStream_t st) {
  constexpr int TF32 = DSB_DTYPE_TF32, BF16 = DSB_DTYPE_BF16, F16 = DSB_DTYPE_F16;
  switch (g.kernel) {
    case CONV_RESIDENT:  // the A ring depth varies per launch: the limit covers every depth
      return kind == BF16 ? launch<conv_resident_kernel<BF16>>(g, ResidentSmem::BUDGET, st, ma, ma2, mb)
                          : launch<conv_resident_kernel<F16>>(g, ResidentSmem::BUDGET, st, ma, ma2, mb);
    case GEMM_F16X3_PAIR:
      return g.block_n == 128 ? launch<gemm_f16x3_pair_kernel<128>>(g, g.smem_bytes, st, ma, mb)
                              : launch<gemm_f16x3_pair_kernel<256>>(g, g.smem_bytes, st, ma, mb);
    case GEMM_PAIR:
      if (kind == TF32) return launch<gemm_tcgen05_pair_kernel<TF32>>(g, g.smem_bytes, st, ma, ma2, mb);
      if (kind == BF16) return launch<gemm_tcgen05_pair_kernel<BF16>>(g, g.smem_bytes, st, ma, ma2, mb);
      return launch<gemm_tcgen05_pair_kernel<F16>>(g, g.smem_bytes, st, ma, ma2, mb);
    default:  // GEMM_1CTA
      if (g.block_n == 256) {
        if (kind == TF32) return launch<gemm_tcgen05_kernel<256, TF32>>(g, g.smem_bytes, st, ma, ma2, mb);
        if (kind == BF16) return launch<gemm_tcgen05_kernel<256, BF16>>(g, g.smem_bytes, st, ma, ma2, mb);
        return launch<gemm_tcgen05_kernel<256, F16>>(g, g.smem_bytes, st, ma, ma2, mb);
      }
      if (kind == TF32) return launch<gemm_tcgen05_kernel<128, TF32>>(g, g.smem_bytes, st, ma, ma2, mb);
      if (kind == BF16) return launch<gemm_tcgen05_kernel<128, BF16>>(g, g.smem_bytes, st, ma, ma2, mb);
      return launch<gemm_tcgen05_kernel<128, F16>>(g, g.smem_bytes, st, ma, ma2, mb);
  }
}

}  // namespace dsb

using namespace dsb;

extern "C" int dsb_gemm_ex(const dsb_gemm_desc* d, void* stream) {
  DSB_REQUIRE(d != nullptr, "dsb_gemm_ex: null descriptor");
  GemmPlan g;
  if (const int rc = plan_gemm(*d, sm_count(), &g)) return rc;
  const GemmParams& p = g.p;
  const int kind = d->dtype;
  CUtensorMap ma, mb;
  const long long a_rows = d->a_rows > 0 ? d->a_rows : d->M;
  if (p.a_mn) {
    if (make_operand_map_mn(&ma, d->A, kind, a_rows, d->K, d->batch, d->lda, d->a_batch_stride)) return 3;
  } else if (make_operand_map(&ma, d->A, kind, d->a_cols > 0 ? d->a_cols : d->K, a_rows, d->batch, d->lda, d->a_batch_stride, BLOCK_M, g.l2_promo_128)) return 3;
  if (p.b_mn) {
    if (make_operand_map_mn(&mb, d->W, kind, d->N, d->K, p.b_batched ? d->batch : 1, d->ldw, d->w_batch_stride)) return 3;
  } else if (make_operand_map(&mb, d->W, kind, d->w_cols > 0 ? d->w_cols : (long long)d->K * d->num_taps, d->N, p.b_batched ? d->batch : 1, d->ldw,
                              d->w_batch_stride, g.w_box_rows)) return 3;
  CUtensorMap ma2 = ma;
  if (p.tap_a2_mask && make_operand_map(&ma2, d->A2, kind, d->a2_cols > 0 ? d->a2_cols : d->K, d->a2_rows > 0 ? d->a2_rows : d->M, d->batch, d->lda2,
                                        d->a2_batch_stride, BLOCK_M, g.l2_promo_128))
    return 3;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  return launch_plan(g, kind, ma, ma2, mb, st);
}
