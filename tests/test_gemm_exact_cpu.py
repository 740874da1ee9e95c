"""CPU: the operands and references of tests/test_gpu_gemm_exact.py (tests/gemm_exact.py).

Every case the GPU file runs must stay below 2^24 grid steps, every operand must survive the trip to fp16, bf16 and
(for the tf32 cases) tf32 unchanged, the per-split and A V references must equal the einsum forms of
tests/test_gpu_ops.py, the multi-wave shapes must produce the tile counts they are named for, and the GELU gate must
hold a float32 emulation of the 16-bit epilogue's gelu_fast2 while rejecting it without its highest-order term.
"""
import math
import os
import re

import numpy as np
import pytest
import torch

import gemm_exact as GE
import softmax_cases as SC


def test_every_listed_case_is_exact():
    assert GE.cases_bounds_ok()
    # the largest cases, spelled out: K = 3072 with the q scale, the tied sum over 513 rows x 64, A V over 1024 keys
    assert GE.dense_bound_steps(3072, 0) < 2 ** 24 and GE.dense_bound_steps(3072, 2) < 2 ** 24
    assert GE.tied_bound_steps(513) < 2 ** 24 and GE.av_bound_steps(1024) < 2 ** 24
    assert GE.tied_bound_steps(4096) >= 2 ** 24            # the bound is not vacuous: 4096 rows would not be exact


def test_every_axis_value_is_covered():
    cases = GE.linear_cases()
    for code in GE.CODES:
        for epi in GE.EPIS:
            sub = [c for c in cases if c["code"] == code and c["epi"] == epi]
            assert {c["M"] for c in sub} == set(GE.LINEAR_MS)
            assert {c["N"] for c in sub} == set(GE.LINEAR_NS), (code, epi)
            assert {c["K"] for c in sub} == set(GE.LINEAR_KS), (code, epi)
            if epi == 0:
                kinds = {("0" if c["q_cols"] == 0 else "64" if c["q_cols"] == 64 else "N" if c["q_cols"] == c["N"] else
                          "768") for c in sub}
                assert kinds == {"0", "64", "768", "N"}, (code, sub)
                assert any(c["q_cols"] == 768 and c["N"] > 768 for c in sub)
    assert {c for c, _, _ in GE.TIED_CASES} == {1, 63, 64, 65, 127, 128, 129, 255, 256, 257, 513, 1024, 100}
    assert {h for _, h, _ in GE.TIED_CASES} == {1, 12} and {r for _, _, r in GE.TIED_CASES} == {1, 2, 7, 64, 513}
    assert {GE.tied_tile_n(c) for c, _, _ in GE.TIED_CASES} == {64, 128, 256}
    av = GE.av_cases()
    assert {c["R"] for c in av} == set(GE.AV_RS) and {c["C"] for c in av} == set(GE.AV_CS)
    assert {c["ldp"] - GE.roundup8(c["C"]) for c in av} == set(GE.LDP_PADS)
    assert {c for c, _, _ in GE.SHORT_CASES} == {1, 31, 64, 65, 127, 128}


@pytest.mark.parametrize("P", [2, 3, 5, 37, 64, 70, 72, 74, 148])
def test_multiwave_shapes_have_the_named_tile_counts(P):
    for epi in GE.EPIS:
        for t in GE.WAVE_TARGETS:
            M, N, K, tiles, w = GE.multiwave_case(P, epi, t)
            assert (N, K) in GE.PRODUCTION_NK[epi] and N % 64 == 0 and K % 64 == 0
            assert GE.dense_tiles(M, N) == tiles
            GE.check_wave_counts(GE.tiles_per_pair(tiles, P), t, w, P)
    # the first (production) shape is taken whenever its n-tile count allows the exact count
    assert GE.multiwave_case(P, 0, "3P+")[1:3] == (2304, 768)


def test_tiles_per_pair_walks_tile_at():
    assert GE.tiles_per_pair(5, 74) == [1] * 5                  # fewer tiles than pairs: one launch pair per tile
    assert GE.tiles_per_pair(75, 74) == [2] + [1] * 73
    assert GE.tiles_per_pair(147, 74) == [2] * 73 + [1]
    assert sum(GE.tiles_per_pair(1000, 3)) == 1000 and GE.tiles_per_pair(1000, 3) == [334, 333, 333]
    assert GE.tied_tiles(128, 12, 3) == 12 * 1 * 1 * 3 and GE.tied_tile_n(129) == 256
    assert GE.av_tiles(7, 257, 2) == 2 * 2 * 2


@pytest.mark.parametrize("K", [64, 768, 3072])
def test_dense_operands_round_trip(K):
    x, W, bias = GE.exact_gemm_operands(70, 320, K, seed=3)
    resid = GE.exact_affine((70, 320), 4)
    for t in (x, W):
        for dt in ("fp16", "bf16"):
            assert SC.exact_in(t.double().numpy(), dt)
        assert GE.exact_in_tf32(t)
    for t in (bias, resid):
        assert torch.equal(torch.round(t.double() / GE.GRID) * GE.GRID, t.double()) and float(t.abs().max()) <= 4
    # fp32 in two orders equals float64 for every epilogue that is exact, and so does the 16-bit rounding
    mask = GE.row_mask_for(70, 5, device="cpu")
    for epi in (0, 2):
        ref = GE.dense_ref(x, W, bias, epi, GE.Q_SCALE, 64, mask, resid)
        seq = torch.zeros(70, 320)
        for k in reversed(range(K)):
            seq = seq + x[:, k:k + 1] * W[:, k][None]
        a32 = seq + bias
        got = a32 + resid if epi == 2 else torch.cat([a32[:, :64] * GE.Q_SCALE, a32[:, 64:]], 1)
        if epi == 0:
            got[mask.bool(), :64] = 0
        assert torch.equal(got.double(), ref)
        assert torch.equal((x @ W.T + bias).double(), GE.dense_preact(x, W, bias))
        for dt in (torch.float16, torch.bfloat16):
            assert torch.equal(got.to(dt), ref.to(dt))


def test_tied_operands_round_trip_and_refs_match_einsum():
    R, C, H = 9, 37, 2
    qkv = GE.exact_qkv(R, C, H, seed=8)
    P = GE.exact_probs(H, C, 48, seed=9)
    for t in (qkv, P[..., :C]):
        for dt in ("fp16", "bf16"):
            assert SC.exact_in(t.double().numpy(), dt)
    assert torch.isnan(P[..., C:]).all()
    D = H * 64
    q, k = qkv[..., :D].abs().max(), qkv[..., D:2 * D].abs().max()
    assert float(q) == 1.0 and float(k) == 0.125                   # q and k on different grids
    # the einsum forms of tests/test_gpu_ops.py
    q64 = qkv.double()
    qh, kh, vh = (q64[..., i * D:(i + 1) * D].view(R, C, H, 64) for i in range(3))
    logits_ref = torch.einsum("rihd,rjhd->hij", qh, kh)
    for ns in (1, 2, 3, 5, 9):
        parts = GE.tied_split_refs(qkv, R, C, H, ns)
        assert parts.shape == (ns, H, C, C) and torch.equal(parts.sum(0), logits_ref)
        for s, (r0, r1) in enumerate(GE.split_rows(R, ns)):
            assert r0 < r1 and torch.equal(parts[s], torch.einsum("rihd,rjhd->hij", qh[r0:r1], kh[r0:r1]))
            assert torch.equal(parts[s].float().double(), parts[s])        # exact in fp32
    # 9 rows in 4 splits of 3 leave the last one empty: rejected by the ABI, skipped by the tests
    assert not GE.valid_splits(9, 4) and GE.valid_splits(9, 5) and GE.valid_splits(9, 9) and not GE.valid_splits(9, 10)
    ctx_ref = torch.einsum("hij,rjhd->rihd", P[..., :C].double(), vh).reshape(R * C, D)
    got = GE.av_ref(P, qkv, R, C, H)
    assert torch.equal(got, ctx_ref) and torch.isfinite(got).all()
    assert torch.equal(got.float().double(), got)


def test_tf32_operands_have_no_lo_half():
    M, N, K, _, _ = GE.multiwave_case(74, 0, "Pw+1")
    x, W, _ = GE.exact_gemm_operands(64, N, K, seed=11)
    assert GE.exact_in_tf32(x) and GE.exact_in_tf32(W)
    assert not GE.exact_in_tf32(torch.tensor([1.0 + 2.0 ** -20]))


@pytest.mark.parametrize("code", [0, 1, 2], ids=["f32", "bf16", "f16"])
def test_ulp_is_the_spacing_of_the_output_type(code):
    dt = GE.torch_dtype(code)
    assert float(GE.ulp(torch.tensor([0.0]), code)) == 2.0 ** (GE.EMIN[code] - GE.MANT[code])
    # x + ulp(x) is the next representable value and x + ulp(x) / 4 rounds back to x, normal and subnormal x alike
    rng = np.random.default_rng(code)
    for e in list(range(GE.EMIN[code] - GE.MANT[code] + 2, 15)):
        x = torch.tensor(float(rng.integers(1, 2 ** min(GE.MANT[code], 7)) * 2.0 ** e), dtype=torch.float64)
        x = x.to(dt).double()
        if x == 0 or not torch.isfinite(x):
            continue
        u = GE.ulp(x, code)
        assert torch.equal((x + u).to(dt).double(), x + u), (code, float(x), float(u))
        assert torch.equal((x + u / 4).to(dt).double(), x), (code, float(x), float(u))
    assert float(GE.ulp(torch.tensor([6e-8]), 2)) == 2.0 ** -24             # fp16 subnormal spacing
    assert float(GE.ulp(torch.tensor([3e4]), 2)) == 16.0


# ------------------------------------------------------------------------------------------ GELU gate
A_AND_S = [0.0705230784, 0.0422820123, 0.0092705272, 0.0001520143, 0.0002765672, 0.0000430638]   # a1 .. a6 (7.1.28)


def gelu_fast2_f32(x: np.ndarray, coeffs=A_AND_S) -> np.ndarray:
    """float32 emulation of umma_gemm.cu gelu_fast2: Horner from a6 with fused multiply-adds (float64 product and sum
    rounded once), the reciprocal rounded to float32, erfc = r^16 by four squarings, 0.5 (x + |x| (1 - erfc))."""
    f = np.float32
    x = x.astype(f)

    def fma(a, b, c):
        return (a.astype(np.float64) * np.float64(b) + np.float64(c)).astype(f)

    ax = np.abs(x)
    z = (ax * f(0.70710678118654752440)).astype(f)
    a = [f(c) for c in coeffs]
    if len(a) == 6:
        p = fma(z, a[5], a[4])
    else:                                   # highest-order term dropped
        p = np.full_like(z, a[4])
    for c in (a[3], a[2], a[1], a[0], f(1.0)):
        p = fma(p, z, c)
    r = (1.0 / p.astype(np.float64)).astype(f)
    for _ in range(4):
        r = (r * r).astype(f)
    t = fma(r, f(-1.0), f(1.0))
    u = fma(ax, t, x)
    return (u * f(0.5)).astype(f)


def test_gelu_fast2_coefficients_are_those_emulated():
    src = open(os.path.join(os.path.dirname(SC.__file__), "..", "rna-msm_b200", "csrc", "umma_gemm.cu")).read()
    body = src[src.index("void gelu_fast2("):]
    body = body[:body.index("\n}\n")]
    nums = [float(v) for v in re.findall(r"f32x2_pack\(([0-9.]+)f, \1f\)", body)]
    assert nums[:8] == [0.70710678118654752440, A_AND_S[5], A_AND_S[4], A_AND_S[3], A_AND_S[2], A_AND_S[1], A_AND_S[0], 1.0]


@pytest.mark.parametrize("code", [1, 2], ids=["bf16", "f16"])
def test_gelu_gate_covers_the_epilogue_and_rejects_a_dropped_term(code):
    a = np.concatenate([np.arange(-10.0, 10.0 + 2 ** -11, 2 ** -11), np.linspace(-1e-3, 1e-3, 4001)]).astype(np.float32)
    at = torch.from_numpy(a).double()
    dt = GE.torch_dtype(code)
    y = torch.from_numpy(gelu_fast2_f32(a)).to(dt)                 # the epilogue rounds the fp32 value once (cvt.rn)
    worst = GE.gelu_excess(y, at, code)
    print(f"[gelu gate {dt}] worst {worst:.3f} of the gate")
    assert worst <= 1.0
    # without a6 z^6 the erfc of negative pre-activations is off by up to ~20 % relative: far outside the gate
    y_bad = torch.from_numpy(gelu_fast2_f32(a, A_AND_S[:5])).to(dt)
    assert GE.gelu_excess(y_bad, at, code) > 4.0
    # a NaN output never passes
    y_nan = y.clone()
    y_nan[17] = float("nan")
    assert not GE.gelu_excess(y_nan, at, code) <= 1.0


def test_gelu_gate_covers_erff_in_fp32():
    """The fp32 paths compute 0.5 x (1 + erff(x / sqrt 2)): emulated with the correctly rounded erf in float32."""
    from scipy.special import erf
    a = np.arange(-10.0, 10.0 + 2 ** -11, 2 ** -11).astype(np.float32)
    f = np.float32
    e = erf((a * f(0.70710678118654752440)).astype(np.float64)).astype(f)
    y = ((f(0.5) * a).astype(f) * (f(1.0) + e).astype(f)).astype(f)
    assert GE.gelu_excess(torch.from_numpy(y), torch.from_numpy(a).double(), 0) <= 1.0
    assert math.isclose(float(GE.gelu64(torch.tensor([1.0]))), 0.8413447460685429)
