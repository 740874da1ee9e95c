"""CPU: iterative masked sampling -- the Philox4x32-10 restatement against Random123's known answers, the mask draw and
the inverse-CDF sampler of ``tests/sampling_ref.py``, argument validation of ``sample_msa``, the sampling workspace
layout, and the group planning of the chains."""
import ctypes as C

import numpy as np
import pytest
import torch

import sampling_ref as S


@pytest.fixture(scope="module")
def pkg():
    import rnamsm_b200
    return rnamsm_b200


# ------------------------------------------------------------------------------------------------ Philox4x32-10
@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
])
def test_philox_known_answers(ctr, key, want):
    """Random123's kat_vectors for philox4x32 with 10 rounds."""
    assert tuple(int(w) for w in S.philox4x32_10(ctr, key)) == want


def test_uniform_layout():
    """Key = (seed low, seed high), counter = (k, s, r*C + c, purpose), u = (word0 >> 8) * 2^-24."""
    seed = 0x0123456789ABCDEF
    w0 = int(S.philox4x32_10((3, 7, 40, 1), (0x89ABCDEF, 0x01234567))[0])
    u = S.uniform(seed, 3, 7, 40, 1)
    assert u == (w0 >> 8) / 2 ** 24 and np.float32(u) == u and 0 <= u < 1
    # vectorised over tokens = the scalar calls
    t = np.arange(50, dtype=np.uint64)
    assert np.array_equal(S.uniform(5, 1, 2, t, 0), [S.uniform(5, 1, 2, int(i), 0) for i in range(50)])
    # every coordinate moves the stream
    base = S.uniform(5, 1, 2, 3, 0)
    assert len({base, S.uniform(6, 1, 2, 3, 0), S.uniform(5, 2, 2, 3, 0), S.uniform(5, 1, 3, 3, 0),
                S.uniform(5, 1, 2, 4, 0), S.uniform(5, 1, 2, 3, 1), S.uniform(5 + (1 << 32), 1, 2, 3, 0)}) == 7


def test_uniform_is_uniform():
    u = S.uniform(11, 0, 0, np.arange(200000, dtype=np.uint64), 0)
    hist = np.histogram(u, bins=20, range=(0, 1))[0]
    from scipy.stats import chisquare
    assert chisquare(hist).pvalue > 1e-3 and u.min() >= 0 and u.max() < 1


# ------------------------------------------------------------------------------------------------ mask draw
def test_mask_set_eligibility():
    R, Cc, PAD = 6, 40, 1
    state = np.full((R, Cc), 4, dtype=np.int64)
    state[:, 0] = 0
    state[2, 30:] = PAD
    rows = [0, 2, 5]
    m = S.mask_set(state, rows, PAD, 1.0, 9, 0, 0)
    assert not m[:, 0].any() and not m[[1, 3, 4]].any() and not m[2, 30:].any()
    assert m[0, 1:].all() and m[2, 1:30].all() and m[5, 1:].all()
    assert not S.mask_set(state, rows, PAD, 0.0, 9, 0, 0).any()
    # fraction near p over many tokens and steps; chains and steps draw different sets
    big = np.full((64, 257), 4, dtype=np.int64)
    frac = np.mean([S.mask_set(big, range(64), PAD, 0.15, 3, 0, s)[:, 1:].mean() for s in range(4)])
    assert abs(frac - 0.15) < 0.005
    assert not np.array_equal(S.mask_set(big, range(64), PAD, 0.15, 3, 0, 0), S.mask_set(big, range(64), PAD, 0.15, 3, 1, 0))


def test_mask_set_compares_float32_p():
    """u is a multiple of 2^-24, so u < p and u < float32(p) agree for every p."""
    u = S.uniform(1, 0, 0, np.arange(100000, dtype=np.uint64), 0)
    for p in (0.1, 1 / 3, 0.7, 1e-6):
        assert np.array_equal(u < p, u < np.float32(p))


# ------------------------------------------------------------------------------------------------ sampler
def test_draw_inverse_cdf():
    allowed = [4, 5, 6, 7, 10]
    logits = np.zeros(12, dtype=np.float32)
    # uniform over five tokens: boundaries at 0.2, 0.4, ...
    assert [S.draw(logits, allowed, 1.0, u)[0] for u in (0.0, 0.19, 0.21, 0.5, 0.79, 0.81, 1 - 2 ** -24)] == \
        [4, 4, 5, 6, 7, 10, 10]
    assert S.draw(logits, allowed, 1.0, 0.2 + 5e-6)[1] and not S.draw(logits, allowed, 1.0, 0.3)[1]
    # temperature scales the logits: T -> large flattens, small sharpens
    lg = np.array([0, 0, 0, 0, 2.0, 1.0, 0, 0, 0, 0, 0, 0], dtype=np.float32)
    a = [4, 5]
    p_hot = np.exp(2.0 / 2) / (np.exp(2.0 / 2) + np.exp(1.0 / 2))
    assert S.draw(lg, a, 2.0, p_hot - 1e-3)[0] == 4 and S.draw(lg, a, 2.0, p_hot + 1e-3)[0] == 5
    # T = 0: argmax over the allowed tokens, ties to the lowest index
    assert S.draw(lg, a, 0.0, 0.99) == (4, False)
    assert S.draw(lg, [5, 6, 7], 0.0, 0.0)[0] == 5
    tie = np.zeros(12, dtype=np.float32)
    tie[[6, 10]] = 3.0
    assert S.draw(tie, allowed, 0.0, 0.5)[0] == 6


def test_draw_frequencies_follow_softmax():
    rng = np.random.default_rng(0)
    lg = rng.normal(size=12).astype(np.float32)
    allowed = [4, 5, 6, 7, 10]
    u = S.uniform(2, 0, 0, np.arange(40000, dtype=np.uint64), S.DRAW)
    for T in (0.5, 1.0, 2.0):
        got = np.bincount([S.draw(lg, allowed, T, x)[0] for x in u[:8000]], minlength=12)[allowed]
        p = np.exp(lg[allowed].astype(np.float64) / T)
        p /= p.sum()
        from scipy.stats import chisquare
        assert chisquare(got, p * got.sum()).pvalue > 1e-3


def test_step_writes_only_masked():
    R, Cc = 3, 9
    state = np.full((R, Cc), 7, dtype=np.int64)
    state[:, 0] = 0
    state[1, 7:] = 1
    logits = np.zeros((R, Cc, 12), dtype=np.float32)
    logits[..., 5] = 50.0                         # every draw is G
    new, m, near = S.step(state, logits, [1, 2], 1, [4, 5, 6, 7, 10], 0.5, 1.0, 4, 0, 3)
    assert m.any() and not near.any()
    assert np.array_equal(new[m], np.full(int(m.sum()), 5)) and np.array_equal(new[~m], state[~m])


# ------------------------------------------------------------------------------------------------ arguments
@pytest.fixture(scope="module")
def cpu_model(pkg):
    return pkg.MSATransformer(pkg.Vocab(pkg.Alphabet()), num_layers=1, embed_dim=64, num_attention_heads=1).eval()


@pytest.mark.parametrize("kw,match", [
    (dict(mask_prob=-0.1), "mask_prob"),
    (dict(mask_prob=1.5), "mask_prob"),
    (dict(mask_prob=float("nan")), "mask_prob"),
    (dict(temperature=-1.0), "temperature"),
    (dict(temperature=float("nan")), "temperature"),
    (dict(steps=-1), "steps"),
    (dict(start_step=-2), "start_step"),
    (dict(n_chains=0), "n_chains"),
    (dict(seed=-1), "seed"),
    (dict(seed=1 << 64), "seed"),
    (dict(allowed=""), "allowed is empty"),
    (dict(allowed="AGZ"), "residue or gap"),
    (dict(allowed=["A", "<mask>"]), "residue or gap"),
    (dict(allowed="AG<pad>"), "residue or gap"),
    (dict(rows=[0, 6]), "outside"),
    (dict(rows=[-1]), "outside"),
    (dict(rows=[]), "empty"),
])
def test_sample_msa_rejects(cpu_model, kw, match):
    """Checked before anything touches a device."""
    args = dict(steps=2)
    args.update(kw)
    with pytest.raises(ValueError, match=match):
        cpu_model.sample_msa(torch.zeros((6, 10), dtype=torch.int64), **args)


def test_allowed_bitmask(cpu_model):
    idx = cpu_model.vocab.tokens_to_idx
    assert cpu_model._allowed_bitmask("AGCU-") == sum(1 << idx[a] for a in "AGCU-") == 0b10011110000
    assert cpu_model._allowed_bitmask(["N", "X"]) == (1 << 8) | (1 << 9)
    assert cpu_model._allowed_bitmask("GG") == 1 << 5


def test_sample_msa_needs_cuda_tokens(cpu_model):
    with pytest.raises(RuntimeError, match="CUDA"):
        cpu_model.sample_msa(torch.zeros((6, 10), dtype=torch.int64), 1)
    with pytest.raises(ValueError, match="n_chains"):
        cpu_model.sample_msa(torch.zeros((3, 6, 10), dtype=torch.int64), 1, n_chains=2)


# ------------------------------------------------------------------------------------------------ workspace
def _layout(lib, R, Cc, code, g, n_rows, D=768, H=12, F=3072):
    """The regions rnamsm_sample_workspace_bytes documents, rebuilt from the library's other size functions."""
    a = lambda x: (x + 255) // 256 * 256
    dt, tensor = code & 0xFF, bool(code & 0x100)
    T, M = R * Cc, g * n_rows * Cc
    if dt in (1, 2) and R >= 2:
        Rs, Cs = (C.c_int * g)(*[R] * g), (C.c_int * g)(*[Cc] * g)
        fwd = lib.rnamsm_batch_workspace_bytes(g, Rs, Cs, D, H, F, dt)
    else:
        fwd = lib.rnamsm_workspace_bytes(R, Cc, D, H, F, code) + a(T)
    total = a(g * T * 8) + a(g * T * D * 4) + a(fwd)
    total += a(M * D * 4) if n_rows < R else 0
    total += a(M * D * 2) if dt in (1, 2) else 0
    total += 2 * a(M * D * 4)
    total += lib.rnamsm_linear_tf32_scratch_bytes(M, D, D) if tensor else 0
    return total


@pytest.mark.parametrize("R,Cc", [(512, 36), (256, 101), (8, 14), (1, 21)])
@pytest.mark.parametrize("precision", ["fp16", "bf16", "fp32", "tf32x3"])
def test_sample_workspace_bytes_matches_layout(R, Cc, precision):
    from rnamsm_b200 import _lib
    code = _lib.forward_code(precision)
    for g in (1, 3, 14):
        for n_rows in sorted({1, R}):
            got = _lib.lib.rnamsm_sample_workspace_bytes(R, Cc, 768, 12, 3072, code, g, n_rows)
            assert got == _layout(_lib.lib, R, Cc, code, g, n_rows) and got % 256 == 0


def test_sample_workspace_bytes_invalid_is_zero():
    from rnamsm_b200 import _lib
    f = _lib.lib.rnamsm_sample_workspace_bytes
    assert f(0, 36, 768, 12, 3072, _lib.F16, 1, 1) == 0
    assert f(512, 36, 768, 12, 3072, _lib.F16, 0, 1) == 0
    assert f(512, 36, 768, 12, 3072, _lib.F16, 1, 0) == 0
    assert f(512, 36, 768, 12, 3072, _lib.F16, 1, 513) == 0
    assert b"n_rows" in _lib.lib.rnamsm_last_error()
    assert f(512, 36, 768, 12, 3072, 7, 1, 1) == 0
    assert b"dtype" in _lib.lib.rnamsm_last_error()


# ------------------------------------------------------------------------------------------------ group planning
def test_plan_chain_groups():
    """sample_msa runs its chains in passes of plan_score_group(R, C, n_chains, token_budget)[0]."""
    from rnamsm_b200 import plan_score_group
    assert plan_score_group(512, 36, 4) == (4, 1)
    assert plan_score_group(512, 36, 100) == (14, 8)
    assert plan_score_group(256, 101, 100) == (10, 10)
    assert plan_score_group(8, 14, 4000) == (2340, 2)
    assert plan_score_group(8, 14, 5, token_budget=2 * 112) == (2, 3)
