"""CPU checks of tests/softmax_cases.py: the constructed q|k give the intended logits exactly after the 16-bit round
trip, and a replay of col_attn_fa_kernel's max bookkeeping shows each depth case does in that kernel what its name
says.  (The GPU side is tests/test_gpu_softmax_edges.py.)"""
import inspect
import re

import numpy as np
import pytest
import torch

import softmax_cases as SC

FA_R = [129, 255, 256, 257, 383, 384, 385, 513, 1025]
ALL_R = [1, 2, 31, 33, 63, 64, 65, 127, 128] + FA_R


def problem(regime, n, variant, seed=3):
    q, k, keypad = SC.head_qk(regime, n, variant, seed, SC.key_block(n))
    return q, k, keypad, SC.masked_logits(q @ k.T, keypad)


@pytest.mark.parametrize("regime", SC.REGIMES)
def test_constructors_are_exact_in_16_bits(regime):
    for n in ALL_R:
        for variant in (0, 1, 5):
            q, k, keypad, s = problem(regime, n, variant)
            for dt in ("fp16", "bf16"):
                assert SC.exact_in(q, dt) and SC.exact_in(k, dt), (regime, n, variant, dt)
            # the products lie on the 2^-12 grid: below 2^12 every fp32 sum of them is exact, in any order
            t = torch.from_numpy(q).to(torch.bfloat16).double() @ torch.from_numpy(k).to(torch.float16).double().T
            assert torch.equal(t, torch.from_numpy(q @ k.T))
            if regime != "below_mask":
                assert np.abs(q @ k.T).max() < 2 ** 12
                assert SC.exact_in(q @ k.T, "fp32")
            assert np.isfinite(s).all()


@pytest.mark.parametrize("n", ALL_R)
def test_regimes_have_their_shape(n):
    """Each regime's logits are what its name says, on every depth the GPU file runs."""
    for variant in range(4):
        # uniform: k = 0, so every real logit is exactly 0
        q, k, keypad, s = problem("uniform", n, variant)
        assert not k.any() and (s[:, ~keypad] == 0).all() and (~keypad).any()
        # onehot: each row's largest logit beats every other by more than 100 nats
        _, _, keypad, s = problem("onehot", n, variant)
        if n > 1:
            top2 = np.sort(s, 1)[:, -2:]
            assert (top2[:, 1] - top2[:, 0] > 100).all()
        # shifted: every real logit within a few nats of +-300
        _, _, keypad, s = problem("shifted", n, variant)
        real = s[:, ~keypad]
        assert (np.abs(np.abs(real) - 300) <= 5).all()
        # staircase_cross: block b's max is 12 b nats (+ up to 1 nat of per-problem step, + noise)
        blk = SC.key_block(n)
        _, _, _, s = problem("staircase_cross", n, variant)
        for b in range((n + blk - 1) // blk):
            mb = s[:, b * blk:(b + 1) * blk].max(1)
            assert (np.abs(mb - (12 + 0.5 * (variant % 3)) * b) < 0.2).all()
        # masked_prefix: a padded prefix and at least one real key after it
        _, _, keypad, _ = problem("masked_prefix", n, variant)
        if n > 1:
            p = int(keypad.sum())
            assert p >= 1 and keypad[:p].all() and not keypad[p:].any()
            if n > 128:
                assert p in (128, 256)
        # fully_masked: every key padded
        _, _, keypad, _ = problem("fully_masked", n, variant)
        assert keypad.all()
        # below_mask: padded keys exist and every real logit sits > 2000 nats below the mask value
        q, k, keypad, _ = problem("below_mask", n, variant)
        assert keypad.any()
        assert ((q @ k.T)[:, ~keypad] < SC.MASK_VALUE - 2000).all()


def test_split_partials_sum_exactly():
    """K5 sums the split partials in split order in fp32: the constructed splits add up to the logits exactly."""
    for regime in SC.REGIMES:
        if regime == "below_mask":
            continue
        for C in (33, 257):
            s, _ = SC.row_logits(regime, C, 2, seed=5)
            for n_splits in (1, 5):
                parts = SC.split_partials(2.0 * s, n_splits, seed=9)
                acc = np.zeros(parts.shape[1:], dtype=np.float32)
                for p in parts:
                    acc = acc + p
                assert np.array_equal(acc.astype(np.float64), 2.0 * s), (regime, C, n_splits)


def test_replay_threshold_is_the_kernels():
    """The replay runs with col_attn_fa.cu's own kRescaleThreshold and key block, so the cases below follow a change of
    either constant (and this file then says whether they still provoke what they are named for)."""
    with open(f"{SC._CSRC}/col_attn_fa.cu") as f:
        src = f.read()
    m = re.search(r"kRescaleThreshold\s*=\s*([^;]+?)f?;", src)
    assert m and float(m.group(1)) == SC.FA_RESCALE_THRESHOLD
    assert 0 < SC.FA_RESCALE_THRESHOLD < 64
    sig = inspect.signature(SC.fa_replay)
    assert sig.parameters["threshold"].default == SC.FA_RESCALE_THRESHOLD
    assert sig.parameters["blk"].default == SC.FA_KEY_BLOCK == 128


def fa_problems(regime, R, n_variants=4):
    for variant in range(n_variants):
        _, _, _, s = problem(regime, R, variant)
        yield variant, SC.fa_replay(s)


@pytest.mark.parametrize("R", FA_R)
def test_replay_staircase_cross_rescales_every_warp(R):
    for variant, r in fa_problems("staircase_cross", R):
        assert r["warp_rescale"][:, 1:].all(), (R, variant)      # every 32-row warp, every block after the first
        assert r["growth_log2"] > 16                             # fp16 P would overflow without the rescale
        if R >= 1025:
            nblk = r["grow"].shape[1]
            assert (12 * (nblk - 1)) * SC.LOG2E > 128            # bf16 P and the fp32 row sum would overflow too


@pytest.mark.parametrize("R", FA_R)
def test_replay_staircase_under_never_rescales(R):
    for variant, r in fa_problems("staircase_under", R):
        assert not r["grow"][:, 1:].any(), (R, variant)
        assert r["max_p_log2"] >= 7 and r["max_p_log2"] < SC.FA_RESCALE_THRESHOLD


@pytest.mark.parametrize("R", FA_R)
def test_replay_mixed_splits_warps(R):
    for variant, r in fa_problems("mixed", R):
        g = r["grow"][:, 1:]
        assert g.any(), (R, variant)
        n_warps = r["warp_rescale"].shape[0]
        split = [w for w in range(n_warps) if g[w * 32:(w + 1) * 32].any(0).any()
                 and (~g[w * 32:(w + 1) * 32]).any(0)[g[w * 32:(w + 1) * 32].any(0)].any()]
        assert split, (R, variant)                               # some lanes grow while others of the warp do not
        assert r["growth_log2"] > 16


@pytest.mark.parametrize("R", FA_R)
def test_replay_masked_prefix_rescales_from_the_mask(R):
    for variant, r in fa_problems("masked_prefix", R):
        _, _, keypad, _ = problem("masked_prefix", R, variant)
        first_real_block = int(np.argmin(keypad)) // SC.FA_KEY_BLOCK
        if first_real_block > 0:
            assert r["grow"][:, first_real_block].all()          # m_ref moves up from -10000 log2(e)
            assert r["growth_log2"] > 10000 * SC.LOG2E - 100


@pytest.mark.parametrize("R", FA_R)
def test_replay_onehot_and_shifted_stay_finite(R):
    """The kernel's P never exceeds 2^threshold, whatever the logits, as long as it rescales."""
    for regime in ("onehot", "shifted", "uniform", "fully_masked", "below_mask"):
        for variant, r in fa_problems(regime, R, 2):
            assert r["max_p_log2"] <= SC.FA_RESCALE_THRESHOLD, (regime, R, variant)


def test_fa_depth_shape_spans_several_items_per_cta():
    R, C, H = SC.fa_depth_shape()
    assert C * H * -(-R // 256) > 4 * 148
