"""dsb_gemm_ex's kernel choice on the CPU: csrc/gemm_plan.cuh (descriptor checks, tile width, kernel, launch geometry) compiled by g++ into a
small host library (tests/native/gemm_plan_host.cpp) and fed the descriptors the engines build, for a 148-SM B200.  Every expected value is
derived by hand from the selection rules, as the comments show; the B=16 rows agree with the kernel names and grid sizes of the launch lists
profiles/r2_e_launches_{denoiser,decoder,vocoder}.csv."""
import ctypes
import os
import subprocess

import pytest

from tests.helpers import ROOT

import _pkg

_pkg.load()
from diffsound_b200 import _lib, packing  # noqa: E402  (the package loads through _pkg)

SMS = 148
GEMM_1CTA, GEMM_PAIR, GEMM_F16X3_PAIR, CONV_RESIDENT = 0, 1, 2, 3
TF32, BF16, F16 = 0, 1, 2
OUT_F16_SPLIT, DUAL_LRELU = 2048, 4096
# every kernel with a fixed ring: 192 KB of stages + 1 KB alignment slack + 256 B of barriers + 32 KB of epilogue transpose tiles
SMEM_RING = 192 * 1024 + 1024 + 256 + 32 * 1024


class PlanOut(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int) for n in ("kernel", "block_n", "grid", "smem_bytes", "w_box_rows", "l2_promo_128", "tiles_m", "tiles_n", "n_pad",
                                            "a_stages", "f3_nsp", "lo_a", "lo_w")] + \
               [("tap_share_mask", ctypes.c_uint), ("tap_shift", ctypes.c_int * 32), ("tap_acol", ctypes.c_int * 32), ("tap_wcol", ctypes.c_int * 32)]


@pytest.fixture(scope="module")
def plan_lib(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("gemmplan") / "gemm_plan_host.so")
    src = os.path.join(ROOT, "tests", "native", "gemm_plan_host.cpp")
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "text-to-sound-synthesis_b200", "csrc"),
                           src, "-o", out])
    lib = ctypes.CDLL(out)
    lib.plan_gemm_host.argtypes = [ctypes.POINTER(_lib.GemmDesc), ctypes.c_int, ctypes.POINTER(PlanOut)]
    lib.plan_gemm_host.restype = ctypes.c_int
    lib.plan_gemm_error.restype = ctypes.c_char_p
    return lib


def run(lib, d):
    o = PlanOut()
    rc = lib.plan_gemm_host(ctypes.byref(d), SMS, ctypes.byref(o))
    return rc, o, lib.plan_gemm_error().decode()


def plan(lib, d):
    rc, o, err = run(lib, d)
    assert rc == 0, err
    return o


def desc(M, N, K, taps, dtype=F16, use_tap_wcol=1, **fields):
    """taps [(row_shift, a_col, w_col, use_a2)] as ops.gemm_desc takes them.  The pointers are fake: the plan never dereferences them."""
    d = _lib.GemmDesc()
    d.A, d.W, d.out = 0x100000, 0x200000, 0x300000
    d.M, d.N, d.K, d.batch, d.dtype = M, N, K, 1, dtype
    d.num_taps, d.use_tap_wcol = len(taps), use_tap_wcol
    for i, (sh, ac, wc, a2) in enumerate(taps):
        d.tap_shift[i], d.tap_acol[i], d.tap_wcol[i], d.tap_a2[i] = sh, ac, wc, a2
    for k, v in fields.items():
        setattr(d, k, v)
    return d


def linear_f16x3(M, N, K, **fields):
    """ops.gemm_f16x3's descriptor: A (M, 2K) = [hi | lo], W (N, 2K) = [hi | lo]; passes lo*hi, hi*lo, hi*hi."""
    return desc(M, N, K, [(0, K, 0, 0), (0, 0, K, 0), (0, 0, 0, 0)], **fields)


def packed(Kp, fold=False):
    """A PackedConv without weights: its tap lists depend only on the K-block width and the packing form."""
    cv = packing.PackedConv.__new__(packing.PackedConv)
    cv.Kp, cv.fold = Kp, fold
    return cv


def shape(o):
    return {"kernel": o.kernel, "block_n": o.block_n, "grid": o.grid}


# ---------------------------------------------------------------- denoiser, B=16: M = 16 x 265 = 4240 rows = 34 tiles of 128
# K x 3 taps >= 2048, so the pair form is possible and 128-wide tiles need a fifth fewer waves than 256-wide ones (cost256 = 2 x waves):
#   N=3072: 204 vs 408 tiles -> cost256 = 6, cost128 = 6;  N=4096: 8 vs 8;  N=1024: 2 vs 2  ->  256 -> pair -> fused pair kernel.
# 256-row pair tiles: 17 x N/256 tiles on 74 pairs: 204 and 272 tiles fill every SM; 68 tiles leave 6 pairs idle (grid 136).
@pytest.mark.parametrize("N,K,grid", [(3072, 1024, 148), (4096, 1024, 148), (1024, 1024, 136), (1024, 4096, 136)], ids=["qkv", "mlp1", "proj", "mlp2"])
def test_denoiser_linears_run_the_fused_pair_kernel(plan_lib, N, K, grid):
    o = plan(plan_lib, linear_f16x3(4240, N, K))
    assert shape(o) == {"kernel": GEMM_F16X3_PAIR, "block_n": 256, "grid": grid}
    assert (o.tiles_m, o.tiles_n, o.smem_bytes, o.w_box_rows, o.l2_promo_128) == (17, N // 256, SMEM_RING, 128, 0)
    # the triple folded into one spatial tap: hi columns at 0, lo halves K columns further right
    assert (o.f3_nsp, o.lo_a, o.lo_w, o.tap_shift[0], o.tap_acol[0], o.tap_wcol[0]) == (1, K, K, 0, 0, 0)


def test_to_logits_runs_the_single_cta_kernel(plan_lib):
    # N = 256 codes: cost256 = 2 x ceil(34 / 148) = 2, cost128 = ceil(68 / 148) = 1, 5 < 8 -> 128-wide: no pair, so no fused form either
    o = plan(plan_lib, linear_f16x3(4240, 256, 1024))
    assert shape(o) == {"kernel": GEMM_1CTA, "block_n": 128, "grid": 68}
    assert (o.tiles_m, o.tiles_n, o.smem_bytes, o.w_box_rows, o.f3_nsp) == (34, 2, SMEM_RING, 128, 0)
    assert list(o.tap_acol[:3]) == [1024, 0, 0] and list(o.tap_wcol[:3]) == [0, 1024, 0]


# M = 256 clips x 265 = 67 840 rows = 530 tiles.  N=1024: cost256 = 2 x ceil(2120 / 148) = 30, cost128 = ceil(4240 / 148) = 29;
# N=4096: 2 x 58 = 116 vs 115.  A bare "fewer waves" rule takes 128 (the 1-CTA kernel); a fifth fewer is required, so 256 and the fused pair kernel.
@pytest.mark.parametrize("N,K", [(1024, 1024), (1024, 4096), (4096, 1024)])
def test_large_batch_keeps_the_fused_pair_kernel(plan_lib, N, K):
    o = plan(plan_lib, linear_f16x3(67840, N, K))
    assert shape(o) == {"kernel": GEMM_F16X3_PAIR, "block_n": 256, "grid": 148}
    assert (o.tiles_m, o.tiles_n) == (265, N // 256)


def test_cross_attention_kv_of_all_layers(plan_lib):
    # 16 x 77 condition rows = 10 tiles, N = 19 layers x 2 x 1024, K = 512: K x 3 = 1536 < 2048 rules out pairs, so fewer waves decides:
    # cost256 = 2 x ceil(1520 / 148) = 22, cost128 = ceil(3040 / 148) = 21 -> 128-wide on the 1-CTA kernel, three taps
    o = plan(plan_lib, linear_f16x3(1232, 38912, 512, flags=OUT_F16_SPLIT, split_off=38912))
    assert shape(o) == {"kernel": GEMM_1CTA, "block_n": 128, "grid": 148}
    assert (o.tiles_m, o.tiles_n, o.w_box_rows, o.f3_nsp) == (10, 304, 128, 0)


# ---------------------------------------------------------------- MelGAN narrow stages, B=16 (vocoder_engine: 9 pad rows, state rows [raw | act] pairs)
# resident weights: w_bytes = taps x n_pad x 128; A ring depth = (227 KB - 1 KB - 33.5 KB fixed - w_bytes) // 16 KB, at most 12.
# A tap with the previous tap's (shift, A column, operand) reuses its staged A box: bit i of tap_share_mask.
@pytest.mark.parametrize("T,C,fold,spatial,extra,mask,n_pad,a_stages,smem", [
    # ResnetBlock 3-tap conv, dilation 3, 64 channels: taps (lo.Wh, hi.Wl, hi.Wh) per spatial tap, the last two share hi -> bits 2, 5, 8;
    # 9 x 64 x 128 = 72 KB of weights -> 7 stages
    pytest.param(108544, 64, False, [(9 + (j - 1) * 3, 128, 192, 0) for j in range(3)], {}, 0b100100100, 64, 7, 34304 + 73728 + 7 * 16384, id="g1_64"),
    # the same conv at 32 channels, folded: one A box [hi | lo] per spatial tap feeds both taps -> bits 1, 3, 5; 24 KB of weights -> 10 stages
    pytest.param(217088, 32, True, [(9 + (j - 1) * 3, 64, 96, 0) for j in range(3)], {}, 0b101010, 32, 10, 34304 + 24576 + 10 * 16384, id="g1_32_folded"),
    # ResnetBlock tail: shortcut(x) over the state (A) + 1x1 conv over Y (A2), in place -> bits 2 and 5 (tap 3 reads the other operand); 9 stages
    pytest.param(108544, 64, False, [(9, 0, 64, 0), (0, 0, 64, 1)], {"A2": 0x400000, "block_n": 128}, 0b100100, 64, 9, 34304 + 49152 + 9 * 16384, id="tail_64"),
])
def test_vocoder_narrow_stages_run_the_resident_kernel(plan_lib, T, C, fold, spatial, extra, mask, n_pad, a_stages, smem):
    taps = packed(64, fold).taps64(spatial)
    o = plan(plan_lib, desc(T, C, 64, taps, batch=16, resident_w=1, flags=OUT_F16_SPLIT | DUAL_LRELU, split_off=C, dual_off=2 * C, **extra))
    # T / 128 x 16 clips tiles, far more than one per SM
    assert shape(o) == {"kernel": CONV_RESIDENT, "block_n": n_pad, "grid": 148}
    assert (o.tap_share_mask, o.n_pad, o.a_stages, o.smem_bytes, o.w_box_rows, o.l2_promo_128) == (mask, n_pad, a_stages, smem, n_pad, 1)
    assert (o.tiles_m, o.tiles_n) == (T // 128, 1)


# ---------------------------------------------------------------- SpecVQGAN decoder, B=16: a 3x3 conv over 128 channels at 80 x 848 (padded 82 x 850)
def decoder_conv(**fields):
    Wp = 850
    shifts = [dy * Wp + dx for dy in (-1, 0, 1) for dx in (-1, 0, 1)]
    return shifts, desc(16 * 82 * Wp, 128, 128, packed(128).taps([(sh, 0, 128, 0) for sh in shifts]), **fields)


def test_decoder_conv_runs_the_fused_conv_form(plan_lib):
    # 9 triples with constant hi -> lo distances, tile shape left to the library: fused conv form; N = 128 -> the 128-wide pair tile;
    # 1 115 200 rows = 4357 pair tiles
    shifts, d = decoder_conv()
    o = plan(plan_lib, d)
    assert shape(o) == {"kernel": GEMM_F16X3_PAIR, "block_n": 128, "grid": 148}
    assert (o.tiles_m, o.tiles_n, o.smem_bytes, o.w_box_rows) == (4357, 1, SMEM_RING, 64)
    assert (o.f3_nsp, o.lo_a, o.lo_w) == (9, 128, 128)
    assert list(o.tap_shift[:9]) == shifts and list(o.tap_acol[:9]) == [0] * 9 and list(o.tap_wcol[:9]) == [256 * j for j in range(9)]


def test_decoder_conv_with_a_fixed_tile_width_is_not_fused(plan_lib):
    shifts, d = decoder_conv(block_n=128)
    o = plan(plan_lib, d)
    assert shape(o) == {"kernel": GEMM_1CTA, "block_n": 128, "grid": 148}
    assert (o.tiles_m, o.f3_nsp, o.w_box_rows) == (8713, 0, 128)
    assert list(o.tap_shift[:27]) == [sh for sh in shifts for _ in range(3)]


# ---------------------------------------------------------------- training (bf16, ops.gemm: no tap_wcol)
@pytest.mark.parametrize("M,N,K,a_mn,block_n,grid", [
    (1024, 1024, 4240, 1, 128, 64),   # dW = dY^T X: 8 x 8 tiles of 128 (cost128 = 1 < cost256 = 2)
    (4240, 1024, 3072, 0, 256, 136),  # dX = dY W with W as stored: cost 2 vs 2 -> 256-wide, 34 x 4 tiles
])
def test_mn_major_training_gemms_run_the_single_cta_kernel(plan_lib, M, N, K, a_mn, block_n, grid):
    # MN-major operands rule out CTA pairs
    o = plan(plan_lib, desc(M, N, K, [(0, 0, 0, 0)], dtype=BF16, use_tap_wcol=0, a_mn_major=a_mn, b_mn_major=1))
    assert shape(o) == {"kernel": GEMM_1CTA, "block_n": block_n, "grid": grid}


# ---------------------------------------------------------------- caller overrides
def test_cta_pair_override(plan_lib):
    linear = lambda **f: desc(4240, 1024, 1024, [(0, 0, 0, 0)], use_tap_wcol=0, **f)
    # one tap, K = 1024 < 2048: no pairs by default; cost 2 vs 2 -> 256-wide, 136 tiles
    assert shape(plan(plan_lib, linear())) == {"kernel": GEMM_1CTA, "block_n": 256, "grid": 136}
    # forced pairs: 17 x 4 pair tiles on 68 pairs
    o = plan(plan_lib, linear(cta_pair=1))
    assert shape(o) == {"kernel": GEMM_PAIR, "block_n": 256, "grid": 136}
    assert (o.tiles_m, o.w_box_rows, o.smem_bytes) == (17, 128, SMEM_RING)
    # a split triple with pairs forbidden: no fused form (it is a pair kernel); 128-wide saves no waves (2 vs 2)
    o = plan(plan_lib, linear_f16x3(4240, 1024, 1024, cta_pair=-1))
    assert shape(o) == {"kernel": GEMM_1CTA, "block_n": 256, "grid": 136}
    assert o.f3_nsp == 0
    # a split triple with pairs forced: the fused pair kernel
    assert shape(plan(plan_lib, linear_f16x3(4240, 1024, 1024, cta_pair=1))) == {"kernel": GEMM_F16X3_PAIR, "block_n": 256, "grid": 136}


# ---------------------------------------------------------------- malformed descriptors
@pytest.mark.parametrize("d,msg", [
    (linear_f16x3(4240, 1024, 1024, flags=DUAL_LRELU, dual_off=2048), "dsb_gemm_ex: DSB_GEMM_DUAL_LRELU needs DSB_GEMM_OUT_F16_SPLIT and dual_off > 0"),
    (desc(108544, 256, 64, packed(64).taps64([(9, 128, 192, 0)]), resident_w=1),
     "dsb_gemm_ex: resident_w needs a 2-byte dtype, K-major operands, K == 64 per tap, N <= 128, explicit tap_wcol and an unbatched W"),
    (desc(1024, 1024, 4240, [(1, 0, 0, 0)], dtype=BF16, use_tap_wcol=0, a_mn_major=1),
     "dsb_gemm_ex: MN-major operands need a 2-byte dtype and a single unshifted tap"),
], ids=["dual_lrelu_without_split", "resident_wide_n", "mn_major_shifted_tap"])
def test_malformed_descriptors_are_rejected(plan_lib, d, msg):
    rc, _, err = run(plan_lib, d)
    assert rc == 2 and err == msg
