"""GPU: every softmax kernel against float64 at sharp, shifted, masked and tile-boundary logits (tests/softmax_cases.py).

The other op-level tests feed randn logits, whose rows span at most ~20 nats: a kernel that subtracts the wrong
maximum (one taken over lanes past C, over three of four warps, or a stale one) passes them.  Here the logits are
prescribed exactly, so such a kernel writes inf / NaN or wrong weights.  Everything goes through the C ABI.

Checkers: float64 softmax (and P V) of the SAME rounded inputs, with masked_fill(-10000) after the scale, computed per
column on the device.  Gates are those of tests/test_gpu_ops.py and tests/test_gpu_col_attn_probs.py -- ctx 2e-5 (fp32),
2e-3 (fp16), 1e-2 (bf16); fp32 probability maps 2e-5 (rows) and 1e-5 (column probabilities); 16-bit P 5e-3 -- plus
softmax_cases.large_logit_term(|s|max) for the fp32 rounding of large logits (derived there).  Every output must be
finite in every case.
"""
import math

import numpy as np
import pytest
import torch

import softmax_cases as SC
from oracle import msa_ref as O

pytestmark = pytest.mark.gpu

CTX_TOL = {0: 2e-5, 1: 1e-2, 2: 2e-3}
ROW_MAP_TOL, COL_PROBS_TOL, LP_TOL = 2e-5, 1e-5, 5e-3
UMMA_R = [2, 63, 64, 65, 127, 128]
FA_R = [129, 255, 256, 257, 383, 384, 385, 513, 1025]
ROW_C = [1, 31, 32, 33, 128, 129, 256, 257, 512, 513, 1024, 1025]


@pytest.fixture(scope="module")
def L():
    from rnamsm_b200 import _lib
    _lib.device_check(torch.device("cuda:0"))
    return _lib


def rel(a, b):
    return O.rel_err(a.detach().double().cpu(), b.detach().double().cpu())


def finite(t):
    return bool(torch.isfinite(t.float()).all())


# ------------------------------------------------------------------------------------------ column attention
def col_inputs(L, regimes, R, C, H, code, seed, blk=None):
    """Device q|k|v in the operand dtype, its float64 copy (the rounded values), pad, and |s|max over real keys."""
    qkv, pad = SC.col_case(regimes, R, C, H, seed, blk)
    dt = L.torch_dtype(code)
    x = torch.from_numpy(qkv).to(dt).cuda()
    return x, x.double(), torch.from_numpy(pad).cuda()


def col_reference(q64, pad, R, C, H):
    """Per column on the device: float64 P [H, R, R] -> yields (c, P); also returns |s|max over real keys."""
    D = H * 64
    for c in range(C):
        q = q64[:, c, :D].view(R, H, 64)
        k = q64[:, c, D:2 * D].view(R, H, 64)
        s = torch.einsum("ihd,jhd->hij", q, k)
        keep = ~pad[:, c].bool()
        smax = float(s[:, :, keep].abs().max()) if bool(keep.any()) else 0.0
        yield c, s.masked_fill(~keep[None, None, :], SC.MASK_VALUE).softmax(-1), smax


def col_ctx_reference(q64, pad, R, C, H):
    D = H * 64
    ctx = torch.empty(R, C, D, dtype=torch.float64, device=q64.device)
    smax = 0.0
    for c, p, sm in col_reference(q64, pad, R, C, H):
        v = q64[:, c, 2 * D:].view(R, H, 64)
        ctx[:, c] = torch.einsum("hij,jhd->ihd", p, v).reshape(R, D)
        smax = max(smax, sm)
    return ctx.view(R * C, D), smax


def run_col_attn(L, qkv, R, C, H, code, col_major, pad):
    ctx = torch.full((R * C, H * 64), float("nan"), dtype=L.torch_dtype(code), device="cuda")
    arg = qkv.transpose(0, 1).contiguous() if col_major else qkv
    L.check(L.lib.rnamsm_col_attn(L.ptr(arg), R, C, H, code, col_major, L.ptr(pad), L.ptr(ctx), L.stream_ptr()),
            "col_attn")
    return ctx


def check_col_attn(L, regimes, R, C, H, code, seed):
    qkv, q64, pad = col_inputs(L, regimes, R, C, H, code, seed, 64 if code == 0 else None)
    ctx_ref, smax = col_ctx_reference(q64, pad, R, C, H)
    ctx = run_col_attn(L, qkv, R, C, H, code, 0, pad)
    torch.cuda.synchronize()
    assert finite(ctx), "non-finite ctx"
    e = rel(ctx, ctx_ref)
    gate = CTX_TOL[code] + SC.large_logit_term(smax)
    assert e < gate, f"ctx err {e:.2e} > {gate:.2e}"
    if code != 0:          # the column-major q|k|v layout: same problem, bit-identical result
        ctx_t = run_col_attn(L, qkv, R, C, H, code, 1, pad)
        assert torch.equal(ctx_t, ctx)


@pytest.mark.parametrize("R", [63, 64, 65, 128, 129])
@pytest.mark.parametrize("regime", SC.REGIMES)
def test_col_attn_f32(L, regime, R):
    check_col_attn(L, regime, R, 3, 2, 0, seed=11)


@pytest.mark.parametrize("R", UMMA_R + FA_R)
@pytest.mark.parametrize("regime", SC.REGIMES)
@pytest.mark.parametrize("code", [1, 2], ids=["bf16", "f16"])
def test_col_attn_16(L, regime, R, code):
    check_col_attn(L, regime, R, 3, 2, code, seed=13)


@pytest.mark.parametrize("code", [1, 2], ids=["bf16", "f16"])
def test_col_attn_fa_many_items_mixed_regimes(L, code):
    """More work items than four per SM, a different regime per column: each CTA carries rescales across items, behind
    the deferred read-out of the item before."""
    R, C, H = SC.fa_depth_shape()
    regimes = [SC.REGIMES[c % len(SC.REGIMES)] for c in range(C)]
    check_col_attn(L, regimes, R, C, H, code, seed=17)


# ------------------------------------------------------------------------------------------ column probabilities
@pytest.mark.parametrize("R,code,col_major", [(R, 0, 0) for R in (2, 63, 64, 65, 128, 129)]
                         + [(R, code, cm) for R in (2, 127, 128, 129, 255, 256, 257) for code, cm in ((1, 0), (2, 0), (2, 1))])
@pytest.mark.parametrize("regime", SC.REGIMES)
def test_col_attn_probs(L, regime, R, code, col_major):
    C, H = 3, 2
    qkv, q64, pad = col_inputs(L, regime, R, C, H, code, seed=19, blk=64 if code == 0 else 128)
    probs = torch.full((H, C, R, R), float("nan"), device="cuda")
    mean = torch.full((H, R, R), float("nan"), device="cuda")
    scratch = torch.empty(max(1, L.lib.rnamsm_col_probs_scratch_bytes(R, C, H)), dtype=torch.uint8, device="cuda")
    arg = qkv.transpose(0, 1).contiguous() if col_major else qkv
    L.check(L.lib.rnamsm_col_attn_probs(L.ptr(arg), R, C, H, code, col_major, L.ptr(pad), L.ptr(probs), L.ptr(mean),
                                        L.ptr(scratch), L.stream_ptr()), "col_attn_probs")
    torch.cuda.synchronize()
    assert finite(probs) and finite(mean)
    mean_ref = torch.zeros(H, R, R, dtype=torch.float64, device="cuda")
    e_full, smax = 0.0, 0.0
    for c, p, sm in col_reference(q64, pad, R, C, H):
        e_full = max(e_full, rel(probs[:, c], p))
        mean_ref += p / C
        smax = max(smax, sm)
    gate = COL_PROBS_TOL + SC.large_logit_term(smax)
    e_mean = rel(mean, mean_ref)
    assert e_full <= gate and e_mean <= gate, f"full {e_full:.2e} mean {e_mean:.2e} gate {gate:.2e}"
    assert float((probs.double().sum(-1) - 1).abs().max()) <= gate


# ------------------------------------------------------------------------------------------ row softmax (K5)
LOGIT_SCALE = 0.5          # the partials carry 2 s, so the scaled logits are exactly the constructed s


def row_inputs(regime, Cn, H, n_splits, seed):
    s, keypad = SC.row_logits(regime, Cn, H, seed)
    parts = torch.from_numpy(SC.split_partials(2.0 * s, n_splits, seed)).cuda()
    return parts, torch.from_numpy(keypad.astype(np.uint8)).cuda()


def row_reference(parts, keypad):
    s = parts.double().sum(0) * LOGIT_SCALE
    keep = ~keypad.bool()
    smax = float(s[:, :, keep].abs().max()) if bool(keep.any()) else 0.0
    return s.masked_fill(~keep[None, None, :], SC.MASK_VALUE).softmax(-1), smax


def run_row_softmax(L, parts, keypad, H, Cn, code, ld_lp):
    n_splits = parts.shape[0]
    pmap = torch.full((H, Cn, Cn), float("nan"), device="cuda")
    plp = torch.full((H, Cn, ld_lp), 7.0, dtype=L.torch_dtype(code), device="cuda")
    L.check(L.lib.rnamsm_row_softmax(L.ptr(parts), n_splits, H, Cn, L.ptr(keypad), LOGIT_SCALE, L.ptr(pmap), L.ptr(plp),
                                     ld_lp, code, L.stream_ptr()), "row_softmax")
    return pmap, plp


def check_row_maps(pmap, plp, ref, smax, Cn, code, lp_base=LP_TOL):
    assert finite(pmap) and finite(plp)
    term = SC.large_logit_term(smax)
    e = rel(pmap, ref)
    assert e < ROW_MAP_TOL + term, f"map err {e:.2e}"
    e_lp = rel(plp[..., :Cn], ref)
    assert e_lp < (ROW_MAP_TOL if code == 0 else lp_base) + term, f"16-bit P err {e_lp:.2e}"
    assert float(plp[..., Cn:].float().abs().sum()) == 0.0          # zero-filled padding columns


@pytest.mark.parametrize("n_splits", [1, 5])
@pytest.mark.parametrize("Cn", ROW_C)
@pytest.mark.parametrize("regime", SC.REGIMES)
def test_row_softmax(L, regime, Cn, n_splits):
    """Every kQ variant (4 / 8 / 16 / 32 and the looping kQ = 0 past C = 1024) and its tail lanes, the four-split load
    group partly full, all three dtypes, ld_lp > C."""
    H = 2
    parts, keypad = row_inputs(regime, Cn, H, n_splits, seed=23)
    ref, smax = row_reference(parts, keypad)
    ld_lp = (Cn + 7) // 8 * 8 + 8
    for code in (0, 1, 2):
        pmap, plp = run_row_softmax(L, parts, keypad, H, Cn, code, ld_lp)
        torch.cuda.synchronize()
        check_row_maps(pmap, plp, ref, smax, Cn, code)


# ------------------------------------------------------------------------------------------ one-launch short row attention
@pytest.mark.parametrize("code", [1, 2], ids=["bf16", "f16"])
@pytest.mark.parametrize("Cn", [1, 31, 32, 33, 127, 128])
@pytest.mark.parametrize("regime", SC.REGIMES)
def test_row_attn_short(L, regime, Cn, code):
    """Tied logits made sharp through the kernel's own phase 1: q and k constant over the R rows, so the tied logit
    is R (q_i . k_j), times logit_scale = 1 / sqrt(R)."""
    R, H = 4, 2
    chunks = L.lib.rnamsm_row_attn_short_chunks(R, Cn, H)
    if chunks == 0:
        pytest.skip("one-launch row attention disabled (RNAMSM_ROW_SHORT=0)")
    D = H * 64
    qkv = np.zeros((R, Cn, 3 * D))
    keypad = None
    for h in range(H):
        q, k, kp = SC.head_qk(regime, Cn, h, 29, 64)
        qkv[:, :, h * 64:(h + 1) * 64] = q[None]
        qkv[:, :, D + h * 64:D + (h + 1) * 64] = k[None]
        keypad = kp if keypad is None else keypad
    qkv[:, :, 2 * D:] = np.random.default_rng([29, Cn]).standard_normal((R, Cn, D))
    dt = L.torch_dtype(code)
    x = torch.from_numpy(qkv).to(dt).cuda()
    x64 = x.double().view(R, Cn, 3, H, 64)
    kp = torch.from_numpy(keypad.astype(np.uint8)).cuda()
    scale = 1.0 / math.sqrt(R)
    s = torch.einsum("rihd,rjhd->hij", x64[:, :, 0], x64[:, :, 1]) * scale
    keep = ~kp.bool()
    smax = float(s[:, :, keep].abs().max()) if bool(keep.any()) else 0.0
    ref = s.masked_fill(~keep[None, None, :], SC.MASK_VALUE).softmax(-1)
    ctx_ref = torch.einsum("hij,rjhd->rihd", ref, x64[:, :, 2]).reshape(R * Cn, D)
    ldp = (Cn + 7) // 8 * 8
    partial = torch.full((chunks, H, Cn, Cn), float("nan"), device="cuda")
    pmap = torch.full((H, Cn, Cn), float("nan"), device="cuda")
    plp = torch.full((H, Cn, ldp), 7.0, dtype=dt, device="cuda")
    ctx = torch.full((R * Cn, D), float("nan"), dtype=dt, device="cuda")
    L.check(L.lib.rnamsm_row_attn_short(L.ptr(x), R, Cn, H, code, L.ptr(kp), scale, L.ptr(partial), chunks, L.ptr(pmap),
                                        L.ptr(plp), ldp, L.ptr(ctx), L.stream_ptr()), "row_attn_short")
    torch.cuda.synchronize()
    check_row_maps(pmap, plp, ref, smax, Cn, code)
    assert finite(ctx)
    e = rel(ctx, ctx_ref)
    assert e < CTX_TOL[code] + SC.large_logit_term(smax), f"ctx err {e:.2e}"


# ------------------------------------------------------------------------------------------ sharded row softmax, one rank
def p2p_warp3_logits(Cn, H):
    """Each row's maximum, 104 nats above the rest, in columns 384-511 of a 512-column group: the fourth warp of the
    vec kernel's block."""
    s = np.random.default_rng(31).integers(-64, 65, size=(H, Cn, Cn)) / 16.0
    for h in range(H):
        for i in range(Cn):
            g = (i % 2) * 512 if Cn >= 1024 else 0
            s[h, i, min(g + 384 + (i * 7 + h * 3) % 128, Cn - 1)] = 104.0
    return s, np.zeros(Cn, dtype=bool)


@pytest.mark.parametrize("case", ["max_in_warp3", "onehot", "shifted", "masked_prefix", "fully_masked", "below_mask"])
@pytest.mark.parametrize("Cn", [512, 1024, 1023, 1025], ids=["vec512", "vec1024", "scalar_cached", "scalar_uncached"])
def test_row_softmax_p2p_one_rank(L, Cn, case):
    """rnamsm_row_softmax_p2p with n_ranks = 1 and local pointers: the vec kernel (C % 4 == 0) and the scalar kernel,
    with the summed row cached in registers (C <= 1024) and not.  Its fp32 map must match K5's on the same partials."""
    H, n_splits = 2, 5
    if case == "max_in_warp3":
        s, keypad = p2p_warp3_logits(Cn, H)
    else:
        s, keypad = SC.row_logits(case, Cn, H, seed=37)
    parts = torch.from_numpy(SC.split_partials(2.0 * s, n_splits, seed=37)).cuda()
    kp = torch.from_numpy(keypad.astype(np.uint8)).cuda()
    ref, smax = row_reference(parts, kp)
    ld_lp = (Cn + 7) // 8 * 8 + 8
    for code in (1, 2):
        pmap = torch.full((H, Cn, Cn), float("nan"), device="cuda")
        plp = torch.full((H, Cn, ld_lp), 7.0, dtype=L.torch_dtype(code), device="cuda")
        peer_partial = (L.C.c_void_p * 1)(parts.data_ptr())
        peer_probs = (L.C.c_void_p * 1)(plp.data_ptr())
        L.check(L.lib.rnamsm_row_softmax_p2p(peer_partial, 1, 0, n_splits, H, Cn, L.ptr(kp), LOGIT_SCALE, L.ptr(pmap),
                                             peer_probs, ld_lp, code, L.stream_ptr()), "row_softmax_p2p")
        k5_map, _ = run_row_softmax(L, parts, kp, H, Cn, code, ld_lp)
        torch.cuda.synchronize()
        check_row_maps(pmap, plp, ref, smax, Cn, code)
        assert rel(pmap, k5_map) < 1e-6
