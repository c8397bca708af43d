"""CPU stand-ins for dsb_gemm_ex's descriptor form (ops.gemm_desc) and the split-fp16 support kernels, used ONLY by tests/test_cpu_codec_host.py to
check the HOST LOGIC of the MelGAN / SpecVQGAN engines (buffer layouts, byte offsets, tap lists, column groups, in-place updates) without a GPU.
Each function restates the documented contract of include/diffsound_b200.h in plain torch (fp64 accumulation; fp16 storage is honoured, so the
(hi | lo) arithmetic is the real one).  TEST INFRASTRUCTURE -- never imported by the product package."""
import torch

F16 = 2
GELU2, ROUND_TF32, OUT_BF16, LRELU, TANH, RES_BEFORE_ACT, OUT_F16, OUT_F16_SPLIT, DUAL_LRELU, SPLIT_OUT_F16, NO_STORE = 1, 2, 4, 8, 16, 128, 256, 2048, 4096, 8192, 16384
_LIVE = []  # tensors whose storage may be addressed by raw pointers


def track(t):
    _LIVE.append(t)
    return t


def _flat(addr, dtype):
    """Flat view of the registered buffer that contains byte address `addr`, starting at that address."""
    es = torch.tensor([], dtype=dtype).element_size()
    for t in reversed(_LIVE):
        if t.dtype != dtype:
            continue
        lo = t.data_ptr()
        hi = lo + t.numel() * es
        if lo <= addr < hi:
            assert (addr - lo) % es == 0
            return t.view(-1)[(addr - lo) // es:]
    raise AssertionError(f"address {addr:#x} ({dtype}) is not inside any tracked buffer")


def split_f16(x, scale=1.0, out=None):
    v = x.double() * scale
    h = v.to(torch.float16)
    l = (v - h.double()).to(torch.float16)
    r = torch.cat([h, l], dim=-1)
    return track(r if out is None else out.copy_(r))


def mel_pack_f16(mel, pad, Kp):
    B, Cm, T = mel.shape
    x = torch.nn.functional.pad(mel.double(), (pad, pad), mode="reflect").transpose(1, 2)  # (B, T+2p, Cm)
    h = x.to(torch.float16)
    l = (x - h.double()).to(torch.float16)
    out = torch.zeros(B, T + 2 * pad, 2 * Kp, dtype=torch.float16)
    out[..., :Cm], out[..., Kp:Kp + Cm] = h, l
    return track(out)


def edge_pad_f16(state, T, P, d, col0, ncols, reflect=True):
    for j in range(1, d + 1):
        state[:, P - j, col0:col0 + ncols] = state[:, P + j, col0:col0 + ncols] if reflect else 0
        state[:, P + T - 1 + j, col0:col0 + ncols] = state[:, P + T - 1 - j, col0:col0 + ncols] if reflect else 0


def conv_out_pair(state, T, row0, col0, w, bias, scale, out=None):
    """dsb_conv_out_pair's contract: tanh(scale * sum_j x[row0 + t + j] . w[j] + bias), x = hi + lo of the pair columns."""
    B = state.shape[0]
    kt, cs = w.shape
    x = state[:, :, col0:col0 + cs].double() + state[:, :, col0 + cs:col0 + 2 * cs].double()
    acc = sum(x[:, row0 + j:row0 + j + T] @ w[j].double() for j in range(kt))
    y = torch.tanh(acc * scale + bias.double()[0]).float()
    if out is None:
        return y
    out.view(B, T).copy_(y)
    return out


def gemm_desc(*, A, W, out, M, N, K, taps, lda, ldw, ldo, dtype=F16, batch=1, a_rows=0, a_cols=0, a_batch_stride=0, w_cols=0, out_batch_stride=0,
              bias=None, flags=0, alpha=1.0, split_off=0, dual_off=0, out_col_group=0, out_col_group_stride=0, A2=None, lda2=0, a2_rows=0, a2_cols=0,
              a2_batch_stride=0, block_n=0, cta_pair=0, residual=None, ld_res=0, geo=None, amax_out=None, resident_w=0, w_batch_stride=0,
              res_batch_stride=0, max_ctas=0, a_mn=False, w_mn=False, use_tap_wcol=1):
    assert use_tap_wcol and not (w_batch_stride or res_batch_stride or a_mn or w_mn), "batched W / residual, MN-major operands and default W columns are not emulated"
    assert not resident_w or (K == 64 and N <= 128 and len(taps) <= 32 and len(taps) * ((N + 15) // 16 * 16) * 128 <= 96 * 1024), "resident_w contract"
    assert dtype == F16
    a_rows, a_cols = a_rows or M, a_cols or K
    Wm = _flat(W, torch.float16)
    Wm = torch.as_strided(Wm, (N, w_cols or ldw), (ldw, 1)).double()
    split = bool(flags & OUT_F16_SPLIT)
    out_flat = _flat(out, torch.float16 if split else torch.float32)
    res_flat = None if residual is None else _flat(residual, torch.float32)
    sp = split_off or N
    if block_n and N > block_n and split and A is not None:
        pass  # (the real kernel would tile N; an in-place update is only safe with one N tile -- asserted by the caller's test below)

    def operand(addr, ld, rows, cols, bstride, b):
        f = _flat(addr, torch.float16)[b * bstride:]
        return torch.as_strided(f, (rows, cols), (ld, 1)).double()

    cols_idx = torch.arange(N)
    ocol = (cols_idx // out_col_group) * out_col_group_stride + cols_idx % out_col_group if out_col_group else cols_idx
    for b in range(batch):
        acc = torch.zeros(M, N, dtype=torch.float64)
        Amat = operand(A, lda, a_rows, a_cols, a_batch_stride, b)
        A2mat = operand(A2, lda2, a2_rows or M, a2_cols or K, a2_batch_stride, b) if A2 is not None else None
        for (sh, ac, wc, use2) in taps:
            src = A2mat if use2 else Amat
            blk = torch.zeros(M, K, dtype=torch.float64)
            r0, r1 = max(0, -sh), min(M, src.shape[0] - sh)       # rows of the tile whose shifted source row exists (TMA zero-fills the rest)
            c1 = min(K, src.shape[1] - ac)                         # columns beyond the tensor are zero-filled too
            if r1 > r0 and c1 > 0:
                blk[r0:r1, :c1] = src[r0 + sh:r1 + sh, ac:ac + c1]
            wb = torch.zeros(N, K, dtype=torch.float64)
            wc1 = min(K, Wm.shape[1] - wc)
            wb[:, :wc1] = Wm[:, wc:wc + wc1]
            acc += blk @ wb.T
        y = acc * alpha
        if bias is not None:
            y = y + bias.double()
        rows = torch.arange(M)
        if res_flat is not None and (flags & RES_BEFORE_ACT):
            y = y + torch.as_strided(res_flat[b * 0:], (M, N), (ld_res, 1)).double()
        if flags & GELU2:
            y = y * torch.sigmoid(1.702 * y)
        elif flags & LRELU:
            y = torch.where(y > 0, y, 0.2 * y)
        elif flags & TANH:
            y = torch.tanh(y)
        if res_flat is not None and not (flags & RES_BEFORE_ACT):
            y = y + torch.as_strided(res_flat, (M, N), (ld_res, 1)).double()
        if geo is not None:
            gP, gW, y0, y1, x0, x1 = geo
            pp = rows % gP
            yy, xx = pp // gW, pp % gW
            inside = (yy >= y0) & (yy < y1) & (xx >= x0) & (xx < x1)
            y = y * inside[:, None]
        if amax_out is not None:
            amax_out.fill_(max(float(amax_out), float(y.float().abs().max())))
        if flags & NO_STORE:
            continue
        base = b * out_batch_stride
        idx = base + rows[:, None] * ldo + ocol[None, :]
        if split:
            copies = [(0, y)] + ([(dual_off, torch.where(y > 0, y, 0.2 * y))] if flags & DUAL_LRELU else [])
            for off, v in copies:
                h = v.float().to(torch.float16)               # the kernel rounds the fp32 accumulator
                l = (v.float() - h.float()).to(torch.float16)
                out_flat[idx + off] = h
                out_flat[idx + off + sp] = l
        else:
            out_flat[idx] = y.float()
