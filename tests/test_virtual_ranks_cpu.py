"""CPU: the references of tests/test_gpu_virtual_ranks.py (tests/virtual_ranks.py) and the argument checks of the
sharded forward's peer-memory entry points.

The index maps must agree with the shard plan the sharded forward uses and with a brute-force walk over the contract
of include/rnamsm_b200.h; the exact GEMM operands must really be exact; the partial logits must sum exactly in the
order every rank's softmax kernel pulls them in.  The argument checks reject a call before anything is launched.
"""
import numpy as np
import pytest
import torch

import softmax_cases as SC
import virtual_ranks as VR
from test_gpu_softmax_edges import p2p_warp3_logits

NS = [1, 2, 3, 4, 8]


# ------------------------------------------------------------------------------------------ index maps
@pytest.mark.parametrize("n", NS)
def test_index_maps_match_shard_plan_and_brute_force(n):
    from rnamsm_b200.sharded import ShardPlan
    R, C = 3 * n, 16 * n
    Rn, Cn = VR.shard(R, C, n)
    plans = [ShardPlan(R, C, n, g) for g in range(n)]
    for g, p in enumerate(plans):
        assert (p.Rn, p.Cn, p.r0, p.c0) == (Rn, Cn, g * Rn, g * Cn)
        rows = p.rows()
        assert VR.owned_rows(g, C, n) == range(p.cols().start, p.cols().stop)   # owned query rows = the column shard
        assert rows == slice(g * Rn, (g + 1) * Rn)

    # push: token (r, c) goes to the owner of column c, at row (c - c0(owner)) * R + r; every row hit once
    owner, row = VR.push_index(R, C, n)
    hits = np.zeros((n, Cn * R), dtype=int)
    for r in range(R):
        for c in range(C):
            d = next(g for g, p in enumerate(plans) if p.cols().start <= c < p.cols().stop)
            want = (d, (c - plans[d].c0) * R + r)
            assert VR.push_dest(r, c, R, C, n) == want
            assert (owner[r * C + c], row[r * C + c]) == want
            hits[want] += 1
    assert (hits == 1).all()

    # scatter: output row m = r * Cn + cl of rank g goes to the owner of MSA row r, at row (r - r0(owner)) * C + c0(g) + cl
    hits = np.zeros((n, Rn * C), dtype=int)
    for g in range(n):
        owner, row = VR.scatter_index(g, R, C, n)
        for m in range(R * Cn):
            r, cl = m // Cn, m % Cn
            d = next(k for k, p in enumerate(plans) if p.rows().start <= r < p.rows().stop)
            want = (d, (r - plans[d].r0) * C + plans[g].c0 + cl)
            assert VR.scatter_dest(g, m, R, C, n) == want
            assert (owner[m], row[m]) == want
            hits[want] += 1
    assert (hits == 1).all()

    # owned query rows partition [0, C)
    rows = sorted(i for g in range(n) for i in VR.owned_rows(g, C, n))
    assert rows == list(range(C))


# ------------------------------------------------------------------------------------------ exact GEMM operands
@pytest.mark.parametrize("K", [128, 768])
def test_exact_operands_are_exact(K):
    ctx, W, bias = VR.exact_gemm_operands(96, 320, K, seed=3)
    x = VR.exact_affine((96, 320), 4)
    for t in (ctx, W):                       # the GEMM operands go to the kernel in 16 bits, bias and x in fp32
        for dt in ("fp16", "bf16"):
            assert SC.exact_in(t.double().numpy(), dt)
    assert float(ctx.abs().max()) <= 1 and float(W.abs().max()) <= 1 / 8
    assert float(bias.abs().max()) <= 4 and float(x.abs().max()) <= 4
    assert VR.exact_sum_bound_ulps(K) < 2 ** 24
    assert VR.exact_sum_bound_ulps(768) < 2 ** 16
    # every term sits on the 2^-9 grid
    for t in (ctx[:, :, None] * W.T[None], bias, x):
        assert torch.equal(torch.round(t.double() / VR.GRID) * VR.GRID, t.double())
    # fp32 in any order equals float64: torch's blocked float32 matmul, then a sequential fp32 sum
    ref = x.double() + ctx.double() @ W.double().T + bias.double()
    got = x + (ctx @ W.T + bias)
    assert torch.equal(got.double(), ref)
    seq = torch.zeros(96, 320)
    for k in reversed(range(K)):
        seq = seq + ctx[:, k:k + 1] * W[:, k][None]
    assert torch.equal((x + (seq + bias)).double(), ref)
    # 16-bit rounding of the exact fp32 value is the rounding of the float64 value
    for dt in (torch.float16, torch.bfloat16):
        assert torch.equal(got.to(dt), ref.to(dt))


# ------------------------------------------------------------------------------------------ softmax partials
@pytest.mark.parametrize("n_splits", [1, 3])
@pytest.mark.parametrize("regime", ["onehot", "shifted", "masked_prefix", "fully_masked", "below_mask", "max_in_warp3"])
def test_rotated_partial_sum_is_exact(regime, n_splits):
    """For every rank count and rank, the fp32 sum in the kernels' rotated order is float32(logits)."""
    C, H = 384, 2                           # divisible by every n in NS
    if regime == "max_in_warp3":
        s, _ = p2p_warp3_logits(C, H)
    else:
        s, _ = SC.row_logits(regime, C, H, seed=41)
    want = (2.0 * s).astype(np.float32)
    for n in NS:
        parts = VR.p2p_partials(s, n, n_splits, seed=41 + n)
        assert parts.shape == (n * n_splits, H, C, C)
        for g in range(n):
            order = VR.rotated_order(g, n, n_splits)
            assert sorted(order) == list(range(n * n_splits)) and order[0] == ((g + 1) % n) * n_splits
            assert np.array_equal(VR.rotated_sum(parts, g, n, n_splits), want), (n, g)


# ------------------------------------------------------------------------------------------ argument checks
@pytest.fixture(scope="module")
def L():
    from rnamsm_b200 import _lib
    return _lib


def ptrs(L, n, base=0x1000):
    return (L.C.c_void_p * max(n, 1))(*[base + 0x100000 * g for g in range(max(n, 1))])


def expect_error(L, rc, pattern):
    assert rc != 0
    msg = L.lib.rnamsm_last_error().decode()
    assert pattern in msg, msg


def test_layernorm_push_rejects_bad_arguments(L):
    """Checked before anything is launched (the pointers are never touched)."""
    f = L.lib.rnamsm_layernorm_push
    x = 0x2000

    def call(n, Rn, C, R, r0, D=256, code=L.F16):
        return f(x, x, x, ptrs(L, n), n, Rn, C, R, r0, D, 1e-5, code, None)

    expect_error(L, call(9, 1, 72, 9, 0), "ranks")                      # n > RNAMSM_MAX_PEERS
    expect_error(L, call(0, 1, 72, 9, 0), "ranks")
    expect_error(L, call(3, 2, 64, 6, 0), "must divide")                # C % n
    expect_error(L, call(2, 2, 64, 4, 0, D=200), "D=200")
    expect_error(L, call(2, 2, 64, 4, 0, code=L.F32), "16-bit")
    expect_error(L, call(4, 3, 64, 12, 10), "outside")                  # r0 + Rn > R
    expect_error(L, call(4, 3, 64, 12, -3), "outside")                  # r0 < 0
    expect_error(L, call(4, -1, 64, 12, 0), "outside")
    expect_error(L, call(1, 2, 64, 1, 0), "outside")                    # Rn > R


def test_row_softmax_p2p_rejects_bad_arguments(L):
    f = L.lib.rnamsm_row_softmax_p2p

    def call(n, rank, C, code=L.F16):
        return f(ptrs(L, n), n, rank, 1, 2, C, None, 0.5, None, ptrs(L, n, 0x9000), C + 8, code, None)

    expect_error(L, call(2, 2, 64), "bad rank")
    expect_error(L, call(2, -1, 64), "bad rank")
    expect_error(L, call(9, 0, 72), "bad rank")
    expect_error(L, call(3, 0, 64), "must divide")
    expect_error(L, call(2, 0, 64, code=L.F32), "16-bit")


def test_linear_residual_scatter_rejects_bad_arguments(L):
    f = L.lib.rnamsm_linear_residual_scatter
    x = 0x2000

    def call(n, R, Cn, Rn, C, c0, N=768, K=768, code=L.F16):
        return f(x, x, x, R, Cn, N, K, code, ptrs(L, n), n, Rn, C, c0, 1, None)

    expect_error(L, call(4, 12, 48, 3, 192, 0, code=L.F32), "16-bit")
    expect_error(L, call(4, 12, 48, 3, 192, 0, N=96), "multiples of 64")
    expect_error(L, call(9, 9, 16, 1, 144, 0), "ranks")                 # n > RNAMSM_MAX_PEERS
    expect_error(L, call(4, 12, 48, 2, 192, 0), "ranks")                # Rn * n != R
    expect_error(L, call(4, 12, 40, 3, 160, 0), "multiple of 16")       # Cn % 16
    expect_error(L, call(4, 12, 48, 3, 192, -48), "column shard")       # c0 < 0
    expect_error(L, call(4, 12, 48, 3, 192, 24), "column shard")        # c0 % Cn
    expect_error(L, call(4, 12, 48, 3, 192, 192), "column shard")       # c0 + Cn > C
    expect_error(L, call(2, 12, 48, 6, 192, 96), "column shard")        # c0 / Cn >= n (C > n Cn)
