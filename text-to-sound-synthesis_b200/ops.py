"""torch-tensor front end of the C-ABI kernels: pointer extraction, shape checks, current-stream plumbing.

PyTorch is used here only for device memory and streams; all arithmetic happens in libdiffsound_b200.so.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import torch

from . import _lib

TF32, BF16, F16 = 0, 1, 2
GELU2, ROUND_TF32, OUT_BF16, LRELU, TANH, GN_SWISH, GN_COMPACT, RES_BEFORE_ACT, OUT_F16, SPLIT_OUT = 1, 2, 4, 8, 16, 32, 64, 128, 256, 512
OUT_F16_SPLIT = 2048
DUAL_LRELU = 4096
SPLIT_OUT_F16 = 8192
NO_STORE = 16384


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("diffsound_b200 ops need CUDA tensors: this path has no CPU fallback")


def device_info():
    s, a, b = C.c_int(), C.c_int(), C.c_int()
    _lib.check(_lib.lib().dsb_device_info(C.byref(s), C.byref(a), C.byref(b)), "dsb_device_info")
    return s.value, a.value, b.value


def round_tf32(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _need_cuda(x)
    x = x.contiguous()
    out = torch.empty_like(x) if out is None else out
    _lib.check(_lib.lib().dsb_round_tf32(x.data_ptr(), out.data_ptr(), x.numel(), _stream()), "dsb_round_tf32")
    return out


def to_bf16(x: torch.Tensor) -> torch.Tensor:
    _need_cuda(x)
    x = x.contiguous()
    out = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    _lib.check(_lib.lib().dsb_f32_to_bf16(x.data_ptr(), out.data_ptr(), x.numel(), _stream()), "dsb_f32_to_bf16")
    return out


def to_f16(x: torch.Tensor) -> torch.Tensor:
    _need_cuda(x)
    x = x.contiguous()
    out = torch.empty(x.shape, dtype=torch.float16, device=x.device)
    _lib.check(_lib.lib().dsb_f32_to_f16(x.data_ptr(), out.data_ptr(), x.numel(), _stream()), "dsb_f32_to_f16")
    return out


def split_tf32(x: torch.Tensor, w_format: bool = False) -> torch.Tensor:
    """(..., C) fp32 -> (..., 2*Cp) [hi | lo] split-TF32 A operand (or (..., 3*Cp) [hi | hi | lo] W operand), Cp = C rounded up to 32."""
    _need_cuda(x)
    C = x.shape[-1]
    Cp = (C + 31) // 32 * 32
    x2 = x.reshape(-1, C) if x.is_contiguous() else x
    if x2.dim() != 2:
        raise RuntimeError("split_tf32 needs a contiguous tensor or a 2-D row-strided view")
    nb = 3 if w_format else 2
    out = torch.empty(*x.shape[:-1], nb * Cp, dtype=torch.float32, device=x.device)
    _lib.check(_lib.lib().dsb_split_tf32(x2.data_ptr(), x2.stride(0), out.data_ptr(), nb * Cp, x2.shape[0], C, Cp, 1 if w_format else 0, _stream()),
               "dsb_split_tf32")
    return out


def pack_split_weight(w: torch.Tensor, ntaps: int) -> torch.Tensor:
    """(N, ntaps*C) fp32 tap-major weight -> (N, 3*ntaps*Cp): per tap [Whi | Whi | Wlo] (pairs with gemm_split's tap list)."""
    N = w.shape[0]
    C = w.shape[1] // ntaps
    Cp = (C + 31) // 32 * 32
    w3 = w.reshape(N, ntaps, C).float()
    hi = round_tf32(w3.contiguous())
    lo = round_tf32((w3 - hi).contiguous())
    out = torch.zeros(N, ntaps, 3, Cp, dtype=torch.float32, device=w.device)
    out[:, :, 0, :C] = hi
    out[:, :, 1, :C] = hi
    out[:, :, 2, :C] = lo
    return out.reshape(N, ntaps * 3 * Cp).contiguous()


def gemm_split(a_split: torch.Tensor, w_split: torch.Tensor, bias=None, residual=None, out=None, *, taps=None, **kw) -> torch.Tensor:
    """3xTF32 GEMM: a_split from split_tf32 (.., 2*Cp), w_split from pack_split_weight; same epilogue options as gemm()."""
    Cp = a_split.shape[-1] // 2
    taps = list(taps) if taps is not None else [0]
    t3, ac = [], []
    for s_ in taps:
        t3 += [s_, s_, s_]
        ac += [0, Cp, 0]  # hi*Whi, lo*Whi, hi*Wlo
    return gemm(a_split, w_split, bias, residual, out, dtype=TF32, taps=t3, tap_acol=ac, k_per_tap=Cp, **kw)


def split_f16(x: torch.Tensor, scale: float = 1.0, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(rows, C) fp32 -> (rows, 2C) fp16 [hi | lo] with hi = f16(scale*x), lo = f16(scale*x - hi): one operand of a split-fp16 ("f16x3") GEMM."""
    _need_cuda(x)
    if x.dim() != 2 or x.stride(1) != 1:
        raise RuntimeError("split_f16 needs a 2-D tensor contiguous in its last dimension")
    rows, Cc = x.shape
    if out is None:
        out = torch.empty(rows, 2 * Cc, dtype=torch.float16, device=x.device)
    _lib.check(_lib.lib().dsb_split_f16(x.data_ptr(), x.stride(0), out.data_ptr(), out.stride(0), Cc, rows, Cc, float(scale), _stream()), "dsb_split_f16")
    return out


def gemm_f16x3(a_pair: torch.Tensor, w_pair: torch.Tensor, bias=None, residual=None, out=None, *, alpha: float = 1.0, gelu: bool = False,
               split_out: bool = False, **kw) -> torch.Tensor:
    """Split-fp16 GEMM at fp32-class accuracy on tcgen05: a_pair (M, 2K) [Ahi | Alo], w_pair (N, 2K) [Whi | Wlo] (both from split_f16 or a
    split_out producer); out = epi(alpha * (Alo Whi^T + Ahi Wlo^T + Ahi Whi^T) + bias) (+ residual), fp32 accumulation over all three passes.
    split_out: write the result as an fp16 (hi | lo) pair (M, 2N) for the next split GEMM / attention instead of fp32."""
    K = a_pair.shape[-1] // 2
    if w_pair.shape[-1] != 2 * K:
        raise RuntimeError(f"gemm_f16x3: W pair has {w_pair.shape[-1]} columns, expected {2 * K}")
    N = w_pair.shape[0]
    M = a_pair.shape[0]
    if out is None:
        out = torch.empty(M, 2 * N, dtype=torch.float16, device=a_pair.device) if split_out else torch.empty(M, N, dtype=torch.float32, device=a_pair.device)
    return gemm(a_pair, w_pair, bias, residual, out, dtype=F16, taps=[0, 0, 0], tap_acol=[K, 0, 0], tap_wcol=[0, K, 0], k_per_tap=K, alpha=alpha,
                gelu=gelu, split_out=split_out, **kw)


def silu(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _need_cuda(x, out)
    x = x.contiguous()
    out = torch.empty_like(x) if out is None else out
    _lib.check(_lib.lib().dsb_silu(x.data_ptr(), out.data_ptr(), x.numel(), _stream()), "dsb_silu")
    return out


def gemm(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None,
         out: Optional[torch.Tensor] = None, *, dtype: int = TF32, gelu: bool = False, round_out: bool = False, out_bf16: bool = False, out_f16: bool = False,
         lrelu: bool = False, tanh: bool = False, res_before_act: bool = False, taps: Optional[Sequence[int]] = None,
         tap_acol: Optional[Sequence[int]] = None, k_per_tap: Optional[int] = None, out_rows: Optional[int] = None, geo: Optional[Sequence[int]] = None, alpha: float = 1.0,
         block_n: int = 0, max_ctas: int = 0, cta_pair: int = 0, a_mn: bool = False, w_mn: bool = False,
         tap_wcol: Optional[Sequence[int]] = None, split_out: bool = False) -> torch.Tensor:
    """out = epi(alpha * A @ W^T + bias) (+ residual) on tcgen05.  a: (M,K) or (batch,M,K); w: (N, taps*K) or (batch,N,K).
    a_mn / w_mn: that operand is given MN-major, i.e. as it lies in memory with the reduction dimension as rows -- a: (K, M), w: (K, N)
    (2-byte dtypes): out = a^T @ w with no transposed copies."""
    _need_cuda(a, w, bias, residual, out)
    batched = a.dim() == 3
    if a.stride(-1) != 1 or w.stride(-1) != 1:
        raise RuntimeError("gemm operands must be contiguous in their last dimension")
    ntaps = 1 if taps is None else len(taps)
    batch = a.shape[0] if batched else 1
    a_rows, a_cols = (a.shape[-1], a.shape[-2]) if a_mn else (a.shape[-2], a.shape[-1])  # (M, K)
    K = a_cols if k_per_tap is None else k_per_tap  # reduction length per tap (A may hold several K blocks side by side)
    N = w.shape[-1] if w_mn else w.shape[-2]
    if tap_wcol is None and (w.shape[-2] if w_mn else w.shape[-1]) != K * ntaps:
        raise RuntimeError(f"gemm: W has reduction length {w.shape[-2] if w_mn else w.shape[-1]}, expected {K}*{ntaps}")
    M = a_rows if out_rows is None else out_rows
    odt = torch.bfloat16 if out_bf16 else (torch.float16 if out_f16 else torch.float32)
    if out is None:
        out = torch.empty((batch, M, N) if batched else (M, N), dtype=odt, device=a.device)
    out_f16 = out.dtype == torch.float16 and not split_out
    out_bf16 = out.dtype == torch.bfloat16
    if split_out and (out.dtype != torch.float16 or batched):
        raise RuntimeError("gemm: split_out writes an fp16 (hi | lo) pair and is not batched")
    flags = (GELU2 if gelu else 0) | (ROUND_TF32 if round_out else 0) | (OUT_BF16 if out_bf16 else 0) | (LRELU if lrelu else 0) | (TANH if tanh else 0) | (RES_BEFORE_ACT if res_before_act else 0) | (OUT_F16 if out_f16 else 0) | (OUT_F16_SPLIT if split_out else 0)
    tap_list = [(s, tap_acol[i] if tap_acol is not None else 0, tap_wcol[i] if tap_wcol is not None else 0, 0) for i, s in enumerate(taps or [0])]
    gemm_desc(A=a.data_ptr(), W=w.data_ptr(), out=out.data_ptr(), M=M, N=N, K=K, batch=batch, dtype=dtype, flags=flags, alpha=alpha, taps=tap_list,
              use_tap_wcol=int(tap_wcol is not None), w_cols=w.shape[-1] if tap_wcol is not None else 0,
              a_rows=a_rows, a_cols=a_cols, lda=a.stride(-2), ldw=w.stride(-2), ldo=out.stride(-2),
              a_batch_stride=a.stride(0) if batched else 0, w_batch_stride=w.stride(0) if w.dim() == 3 else 0, out_batch_stride=out.stride(0) if batched else 0,
              bias=bias, residual=_ptr(residual), ld_res=residual.stride(-2) if residual is not None else 0,
              res_batch_stride=residual.stride(0) if (residual is not None and batched) else 0, split_off=N if split_out else 0, geo=geo,
              block_n=block_n, max_ctas=max_ctas, cta_pair=cta_pair, a_mn=a_mn, w_mn=w_mn)
    return out


def gemm_desc(*, A, W, out, M, N, K, taps, lda, ldw, ldo, dtype=F16, batch=1, a_rows=0, a_cols=0, a_batch_stride=0, w_cols=0, out_batch_stride=0,
              bias=None, flags=0, alpha=1.0, split_off=0, dual_off=0, out_col_group=0, out_col_group_stride=0, A2=None, lda2=0, a2_rows=0, a2_cols=0,
              a2_batch_stride=0, block_n=0, cta_pair=0, residual=None, ld_res=0, geo=None, amax_out=None, resident_w=0, w_batch_stride=0,
              res_batch_stride=0, max_ctas=0, a_mn=False, w_mn=False, use_tap_wcol=1):
    """Descriptor front end of dsb_gemm_ex, for callers that lay out their own buffers (the MelGAN / SpecVQGAN state buffers) and for gemm(): A / W /
    out / A2 / residual are raw device addresses (ints: tensor.data_ptr() plus a byte offset), sizes and strides in elements;
    taps = [(row_shift, a_col, w_col, use_a2), ...]; use_tap_wcol=0 ignores w_col and reads W columns [i*K, (i+1)*K) for tap i."""
    d = _lib.GemmDesc()
    d.A, d.W, d.out, d.bias, d.A2 = A, W, out, _ptr(bias), A2
    d.M, d.N, d.K, d.batch = M, N, K, batch
    d.a_rows, d.a_cols, d.lda, d.ldw, d.ldo = a_rows, a_cols, lda, ldw, ldo
    d.a_batch_stride, d.w_batch_stride, d.out_batch_stride = a_batch_stride, w_batch_stride, out_batch_stride
    d.dtype, d.flags, d.alpha = dtype, flags, alpha
    d.num_taps = len(taps)
    d.use_tap_wcol, d.w_cols = use_tap_wcol, w_cols
    for i, (sh, ac, wc, a2) in enumerate(taps):
        d.tap_shift[i], d.tap_acol[i], d.tap_wcol[i], d.tap_a2[i] = int(sh), int(ac), int(wc), int(a2)
    d.split_off, d.dual_off, d.out_col_group, d.out_col_group_stride = split_off, dual_off, out_col_group, out_col_group_stride
    d.lda2, d.a2_rows, d.a2_cols, d.a2_batch_stride = lda2, a2_rows, a2_cols, a2_batch_stride
    d.block_n, d.max_ctas, d.cta_pair = block_n, max_ctas, cta_pair
    d.a_mn_major, d.b_mn_major = int(a_mn), int(w_mn)
    d.residual, d.ld_res, d.res_batch_stride = residual, ld_res, res_batch_stride
    d.amax_out = _ptr(amax_out)
    d.resident_w = int(resident_w)
    if geo is not None:
        d.geo_P, d.geo_Wp, d.geo_y0, d.geo_y1, d.geo_x0, d.geo_x1 = [int(v) for v in geo]
    _lib.check(_lib.lib().dsb_gemm_ex(C.byref(d), _stream()), "dsb_gemm_ex")


def mel_pack_f16(mel, pad, Kp):
    """mel (B, Cm, T) fp32 -> (B, T + 2 pad, 2 Kp) fp16 (hi | lo), reflection-padded in time."""
    _need_cuda(mel)
    B, Cm, T = mel.shape
    out = torch.empty(B, T + 2 * pad, 2 * Kp, dtype=torch.float16, device=mel.device)
    _lib.check(_lib.lib().dsb_mel_pack_f16(mel.data_ptr(), out.data_ptr(), B, Cm, T, pad, Kp, _stream()), "dsb_mel_pack_f16")
    return out


def edge_pad_f16(state, T, P, d, col0, ncols, reflect=True):
    """state (B, T + 2P, ld) fp16: fill pad rows P-j / P+T-1+j (j = 1..d) of columns [col0, col0+ncols) by reflection (or zeros)."""
    _need_cuda(state)
    B, Tp, ld = state.shape
    _lib.check(_lib.lib().dsb_edge_pad_f16(state.data_ptr(), ld, Tp * ld, B, T, P, d, col0, ncols, 1 if reflect else 0, _stream()), "dsb_edge_pad_f16")


def conv_out_pair(state, T, row0, col0, w, bias, scale, out=None):
    """state (B, rows, ld) fp16 with the activated (hi | lo) pair at columns [col0, col0 + 2 cs); w (kt, cs) fp32 -> tanh(scale * conv + bias) (B, T) fp32."""
    _need_cuda(state, w, bias)
    B, rows, ld = state.shape
    kt, cs = w.shape
    out = torch.empty(B, T, dtype=torch.float32, device=state.device) if out is None else out
    _lib.check(_lib.lib().dsb_conv_out_pair(state.data_ptr(), ld, rows * ld, B, T, row0, col0, cs, kt, w.data_ptr(), _ptr(bias), float(scale), out.data_ptr(),
                                            _stream()), "dsb_conv_out_pair")
    return out


def gemm_f32(a, w, bias=None, residual=None, out=None, *, gelu=False, round_out=False):
    """Exact fp32 FFMA GEMM (set-up tables, fp32-exact mode)."""
    _need_cuda(a, w, bias, residual, out)
    M, K = a.shape
    N = w.shape[0]
    out = torch.empty((M, N), dtype=torch.float32, device=a.device) if out is None else out
    flags = (GELU2 if gelu else 0) | (ROUND_TF32 if round_out else 0)
    _lib.check(_lib.lib().dsb_gemm_f32(a.data_ptr(), w.data_ptr(), _ptr(bias), _ptr(residual), out.data_ptr(), M, N, K, a.stride(0), w.stride(0),
                                       out.stride(0), residual.stride(0) if residual is not None else 0, flags, _stream()), "dsb_gemm_f32")
    return out


def embed_tokens(ids, emb, height_emb, width_emb, out=None, err_flag=None):
    _need_cuda(ids, emb, height_emb, width_emb)
    B, L = ids.shape
    D = emb.shape[1]
    H, W = height_emb.shape[0], width_emb.shape[0]
    out = torch.empty((B, L, D), dtype=torch.float32, device=ids.device) if out is None else out
    _lib.check(_lib.lib().dsb_embed_tokens(ids.data_ptr(), emb.data_ptr(), height_emb.data_ptr(), width_emb.data_ptr(), out.data_ptr(), B, L, D, H, W,
                                           emb.shape[0], _ptr(err_flag), _stream()), "dsb_embed_tokens")
    return out


def _out_flags(out, round_out, split=False):
    if split:
        return OUT_F16_SPLIT
    if out.dtype == torch.float16:
        return OUT_F16
    if out.dtype == torch.bfloat16:
        return OUT_BF16
    return ROUND_TF32 if round_out else 0


def layernorm(x, gamma, beta, out=None, *, eps=1e-5, round_out=False, out_bf16=False, split=False):
    """split: out is the fp16 (hi | lo) pair (..., 2D) of the fp32 result (the A operand of gemm_f16x3)."""
    _need_cuda(x, gamma, beta)
    D = x.shape[-1]
    rows = x.numel() // D
    if out is None:
        out = torch.empty(*x.shape[:-1], 2 * D, dtype=torch.float16, device=x.device) if split else \
            torch.empty(x.shape, dtype=torch.bfloat16 if out_bf16 else torch.float32, device=x.device)
    if split and (out.dtype != torch.float16 or out.shape[-1] != 2 * D):
        raise RuntimeError("layernorm(split=True) writes an fp16 (..., 2D) tensor")
    flags = _out_flags(out, round_out, split)
    _lib.check(_lib.lib().dsb_layernorm(x.data_ptr(), out.data_ptr(), gamma.data_ptr(), beta.data_ptr(), rows, D, eps, flags, _stream()), "dsb_layernorm")
    return out


def ada_layernorm(x, table, t, out=None, *, eps=1e-5, round_out=False, out_bf16=False, split=False):
    """x (B,L,D), table (T,2D) = Linear(SiLU(emb)) rows, t (B,) int64.  split: as layernorm()."""
    _need_cuda(x, table, t)
    B, L, D = x.shape
    if out is None:
        out = torch.empty(B, L, 2 * D, dtype=torch.float16, device=x.device) if split else \
            torch.empty(x.shape, dtype=torch.bfloat16 if out_bf16 else torch.float32, device=x.device)
    if split and (out.dtype != torch.float16 or out.shape[-1] != 2 * D):
        raise RuntimeError("ada_layernorm(split=True) writes an fp16 (..., 2D) tensor")
    flags = _out_flags(out, round_out, split)
    _lib.check(_lib.lib().dsb_ada_layernorm(x.data_ptr(), out.data_ptr(), table.data_ptr(), t.data_ptr(), B, L, D, table.shape[0], eps, flags, _stream()),
               "dsb_ada_layernorm")
    return out


def l2_normalize_rows_(x):
    """x (..., D) contiguous fp32: every row divided by its L2 norm, in place."""
    _need_cuda(x)
    D = x.shape[-1]
    _lib.check(_lib.lib().dsb_l2_normalize_rows(x.data_ptr(), x.numel() // D, D, _stream()), "dsb_l2_normalize_rows")
    return x


ATTN_CAUSAL = 1024


def attention(q, k, v, out, *, B, H, Lq, Lk, scale, round_out=False, causal=False):
    """q/out: row-strided views with (B*Lq) rows; k/v: (B*Lk) rows; head h = columns [64h, 64h+64).  causal (fp16 path): key j visible to query i iff j <= i."""
    _need_cuda(q, k, v, out)
    for t_ in (q, k, v, out):
        if t_.stride(-1) != 1:
            raise RuntimeError("attention operands must be contiguous in the head dimension")
    if q.dtype == torch.float16:
        if k.dtype != torch.float16 or v.dtype != torch.float16:
            raise RuntimeError("attention: q, k, v must share a dtype")
        _lib.check(_lib.lib().dsb_attention_f16(q.data_ptr(), q.stride(0), k.data_ptr(), k.stride(0), v.data_ptr(), v.stride(0), out.data_ptr(),
                                                out.stride(0), B, H, Lq, Lk, scale, _out_flags(out, False) | (ATTN_CAUSAL if causal else 0), _stream()),
                   "dsb_attention_f16")
        return out
    if causal:
        raise RuntimeError("causal attention is implemented for fp16 operands")
    _lib.check(_lib.lib().dsb_attention(q.data_ptr(), q.stride(0), k.data_ptr(), k.stride(0), v.data_ptr(), v.stride(0), out.data_ptr(), out.stride(0),
                                        B, H, Lq, Lk, scale, _out_flags(out, round_out), _stream()), "dsb_attention")
    return out


STAGE_INPUT_LOGPROB, STAGE_SKIP_POSTERIOR, STAGE_SKIP_SAMPLE = 1, 2, 4


def attention_tc(q, k, v, out, *, B, H, Lq, Lk, scale, pipelined=True):
    """tcgen05/TMEM attention core (fp16 in/out); same argument conventions as attention()."""
    _need_cuda(q, k, v, out)
    if not all(t_.dtype == torch.float16 and t_.stride(-1) == 1 for t_ in (q, k, v, out)):
        raise RuntimeError("attention_tc needs fp16 tensors contiguous in the head dimension")
    fn = _lib.lib().dsb_attention_tc2 if pipelined else _lib.lib().dsb_attention_tc
    _lib.check(fn(q.data_ptr(), q.stride(0), k.data_ptr(), k.stride(0), v.data_ptr(), v.stride(0), out.data_ptr(), out.stride(0),
                  B, H, Lq, Lk, scale, _stream()), "dsb_attention_tc")
    return out


def attention_tc_split(q, k, v, out, *, q_lo, k_lo, v_lo, o_lo, B, H, Lq, Lk, scale):
    """Split-fp16 tcgen05 attention: q/k/v/out are the hi halves (row-strided fp16 views, head h = columns [64h, 64h+64)); the matching lo half
    of every row lies *_lo elements further along the row."""
    _need_cuda(q, k, v, out)
    if not all(t_.dtype == torch.float16 and t_.stride(-1) == 1 for t_ in (q, k, v, out)):
        raise RuntimeError("attention_tc_split needs fp16 tensors contiguous in the head dimension")
    _lib.check(_lib.lib().dsb_attention_tc_split(q.data_ptr(), q.stride(0), q_lo, k.data_ptr(), k.stride(0), k_lo, v.data_ptr(), v.stride(0), v_lo,
                                                 out.data_ptr(), out.stride(0), o_lo, B, H, Lq, Lk, scale, _stream()), "dsb_attention_tc_split")
    return out


def posterior_sample(inp, x_t, t, uniform, sched, *, T, trunc_mode=1, trunc_r=0.85, trunc_k=0, t_post=None, x_next=None, log_prob_out=None,
                     stage=0):
    """Fused p_sample tail (see dsb_posterior_sample).  inp: raw logits (B,L,K) fp32, or (B,K+1,L) log-probs with STAGE_INPUT_LOGPROB;
    x_t (B,L) int64; uniform (B,K+1,L); sched (8,T+1) -> x_next (B,L) int64 (None when sampling is skipped)."""
    _need_cuda(inp, x_t, t, uniform, sched, log_prob_out)
    if stage & STAGE_INPUT_LOGPROB:
        B, C_, L = inp.shape
        K = C_ - 1
    else:
        B, L, K = inp.shape
    for t_ in (inp, x_t, uniform, sched, log_prob_out, t, t_post):
        if t_ is not None and not t_.is_contiguous():
            raise RuntimeError("posterior_sample needs contiguous tensors")
    if uniform is not None and tuple(uniform.shape) != (B, K + 1, L):
        raise RuntimeError(f"uniform must be (B,K+1,L)={(B, K + 1, L)}, got {tuple(uniform.shape)}")
    if sched is not None and tuple(sched.shape) != (8, T + 1):
        raise RuntimeError("sched must be (8, T+1)")
    if not (stage & STAGE_SKIP_SAMPLE) and x_next is None:
        x_next = torch.empty((B, L), dtype=torch.int64, device=inp.device)
    _lib.check(_lib.lib().dsb_posterior_sample(inp.data_ptr(), _ptr(x_t), _ptr(t), _ptr(t_post), _ptr(uniform), _ptr(sched), _ptr(x_next),
                                               _ptr(log_prob_out), B, K, L, T, trunc_mode, trunc_r, trunc_k, stage, _stream()), "dsb_posterior_sample")
    return x_next


def aten_rand_geometry(numel: int, device=None):
    """(nthreads, counter_offset) of the kernel ATen launches for torch.rand / rand_like on a contiguous float tensor of `numel` elements
    (ATen/native/cuda/DistributionTemplates.h calc_execution_policy: block 256, grid = min(SMs * (maxThreadsPerSM // 256), ceil(numel / 256)),
    four values per curand call)."""
    pr = torch.cuda.get_device_properties(device if device is not None else torch.cuda.current_device())
    grid = min(pr.multi_processor_count * (pr.max_threads_per_multi_processor // 256), (numel + 255) // 256)
    return 256 * grid, ((numel - 1) // (256 * grid * 4) + 1) * 4


def aten_uniform(numel: int, seed: int, offset: int, device=None) -> torch.Tensor:
    """The tensor torch.rand(numel, device='cuda') would return for generator state (seed, philox offset), computed by this library's Philox."""
    out = torch.empty(numel, dtype=torch.float32, device=device if device is not None else "cuda")
    nthreads, _ = aten_rand_geometry(numel, out.device)
    _lib.check(_lib.lib().dsb_aten_uniform(out.data_ptr(), numel, seed & (2 ** 64 - 1), offset, nthreads, _stream()), "dsb_aten_uniform")
    return out


def posterior_sample_loop(logits, x, t, t_post, sched, ctrl, t_sched, t_post_sched, *, T, trunc_mode=1, trunc_r=0.85, trunc_k=0):
    """One step of the fused sampling loop (see dsb_posterior_sample_loop): in-kernel uniforms, x updated in place, t / t_post / RNG offset advanced on
    the device by the kernel itself."""
    _need_cuda(logits, x, t, t_post, sched, ctrl, t_sched, t_post_sched)
    B, L, K = logits.shape
    _lib.check(_lib.lib().dsb_posterior_sample_loop(logits.data_ptr(), x.data_ptr(), t.data_ptr(), t_post.data_ptr(), sched.data_ptr(), ctrl.data_ptr(),
                                                    t_sched.data_ptr(), t_post_sched.data_ptr(), B, K, L, T, trunc_mode, trunc_r, trunc_k, _stream()),
               "dsb_posterior_sample_loop")
    return x


# ---------------------------------------------------------------------------------------------- decoder / vocoder support
def codebook_gather_padded(ids, codebook, H, W, *, round_out=True, split=False, split_f16=False, err_flag=None):
    _need_cuda(ids, codebook)
    B = ids.shape[0]
    E = codebook.shape[1]
    out = torch.empty(B, H + 2, W + 2, 2 * E if (split or split_f16) else E, dtype=torch.float16 if split_f16 else torch.float32, device=ids.device)
    _lib.check(_lib.lib().dsb_codebook_gather_padded(ids.contiguous().data_ptr(), codebook.data_ptr(), out.data_ptr(), B, H, W, E, codebook.shape[0],
                                                     SPLIT_OUT_F16 if split_f16 else (SPLIT_OUT if split else (ROUND_TF32 if round_out else 0)), _ptr(err_flag), _stream()),
               "dsb_codebook_gather_padded")
    return out


def groupnorm_stats(x_pad, stats=None, groups=32):
    """x_pad (B, Hp, Wp, C) zero-bordered -> stats (B, groups, 2) fp64 (sum, sumsq)."""
    _need_cuda(x_pad)
    B, Hp, Wp, C = x_pad.shape
    stats = torch.empty(B, groups, 2, dtype=torch.float64, device=x_pad.device) if stats is None else stats
    _lib.check(_lib.lib().dsb_groupnorm_stats(x_pad.data_ptr(), stats.data_ptr(), B, Hp * Wp, C, groups, _stream()), "dsb_groupnorm_stats")
    return stats


def groupnorm_apply(x_pad, stats, gamma, beta, *, eps=1e-6, swish=True, round_out=True, compact_len=0, out=None, groups=32, split=False, split_f16=False):
    _need_cuda(x_pad, stats, gamma, beta)
    B, Hp, Wp, C = x_pad.shape
    H, W = Hp - 2, Wp - 2
    flags = (GN_SWISH if swish else 0) | (ROUND_TF32 if round_out and not (split or split_f16) else 0) | (GN_COMPACT if compact_len else 0) | \
        (SPLIT_OUT_F16 if split_f16 else (SPLIT_OUT if split else 0))
    if out is None:
        Co = 2 * C if (split or split_f16) else C
        out = torch.empty((B, compact_len, Co) if compact_len else (B, Hp, Wp, Co), dtype=torch.float16 if split_f16 else torch.float32, device=x_pad.device)
    _lib.check(_lib.lib().dsb_groupnorm_apply(x_pad.data_ptr(), stats.data_ptr(), gamma.data_ptr(), beta.data_ptr(), out.data_ptr(), B, H, W, C, groups,
                                              eps, flags, compact_len, _stream()), "dsb_groupnorm_apply")
    return out


def upsample2x_padded(x_pad, *, round_out=True, split=False, split_f16=False):
    _need_cuda(x_pad)
    B, Hp, Wp, C = x_pad.shape
    H, W = Hp - 2, Wp - 2
    out = torch.empty(B, 2 * H + 2, 2 * W + 2, 2 * C if (split or split_f16) else C, dtype=torch.float16 if split_f16 else torch.float32, device=x_pad.device)
    _lib.check(_lib.lib().dsb_upsample2x_padded(x_pad.data_ptr(), out.data_ptr(), B, H, W, C,
                                                SPLIT_OUT_F16 if split_f16 else (SPLIT_OUT if split else (ROUND_TF32 if round_out else 0)), _stream()),
               "dsb_upsample2x_padded")
    return out


def space_to_depth_padded(x_pad, *, split=False, round_out=False):
    """(B, H+2, W+2, C) zero-bordered image -> its four stride-2 phases on the half-resolution padded grid (B, H/2+2, W/2+2, 4C [8C if split])."""
    _need_cuda(x_pad)
    B, Hp, Wp, C = x_pad.shape
    H, W = Hp - 2, Wp - 2
    out = torch.empty(B, H // 2 + 2, W // 2 + 2, (8 if split else 4) * C, dtype=torch.float32, device=x_pad.device)
    _lib.check(_lib.lib().dsb_space_to_depth_padded(x_pad.data_ptr(), out.data_ptr(), B, H, W, C, SPLIT_OUT if split else (ROUND_TF32 if round_out else 0),
                                                    _stream()), "dsb_space_to_depth_padded")
    return out


def row_argmin(x, n: int):
    """x: (rows, ld) fp32 -> int64 (rows,) index of the smallest of the first n columns (first on ties)."""
    _need_cuda(x)
    out = torch.empty(x.shape[0], dtype=torch.int64, device=x.device)
    _lib.check(_lib.lib().dsb_row_argmin(x.data_ptr(), x.stride(0), x.shape[0], n, out.data_ptr(), _stream()), "dsb_row_argmin")
    return out


def softmax_rows_(x, n_valid, *, round_out=True):
    _need_cuda(x)
    assert x.is_contiguous()
    ld = x.shape[-1]
    _lib.check(_lib.lib().dsb_softmax_rows(x.data_ptr(), x.numel() // ld, n_valid, ld, ROUND_TF32 if round_out else 0, _stream()), "dsb_softmax_rows")
    return x


def tokens_add_to_padded_(tok, x_pad):
    _need_cuda(tok, x_pad)
    B, Hp, Wp, C = x_pad.shape
    _lib.check(_lib.lib().dsb_tokens_add_to_padded(tok.data_ptr(), x_pad.data_ptr(), B, Hp - 2, Wp - 2, C, tok.shape[1], _stream()),
               "dsb_tokens_add_to_padded")
    return x_pad


def lrelu_pad(x, pad, *, slope=0.2, reflect=True, channel_major=False, round_out=True, split=False):
    """x (B,T,C) channels-last, or (B,C,T) with channel_major -> (B, T+2*pad, C), or the split-TF32 operand (B, T+2*pad, 2*Cp)."""
    _need_cuda(x)
    x = x.contiguous()
    if channel_major:
        B, Cc, T = x.shape
    else:
        B, T, Cc = x.shape
    Co = 2 * ((Cc + 31) // 32 * 32) if split else Cc
    out = torch.empty(B, T + 2 * pad, Co, dtype=torch.float32, device=x.device)
    _lib.check(_lib.lib().dsb_lrelu_pad(x.data_ptr(), out.data_ptr(), B, T, Cc, pad, slope, 1 if reflect else 0, 1 if channel_major else 0,
                                        SPLIT_OUT if split else (ROUND_TF32 if round_out else 0), _stream()), "dsb_lrelu_pad")
    return out
