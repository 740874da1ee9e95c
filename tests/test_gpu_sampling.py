"""GPU: iterative masked sampling with the LM head (``MSATransformer.sample_msa``, ``rnamsm_msa_gibbs_sample``,
``python -m rnamsm_b200.generate``).

One step equals the CPU restatement of the algorithm (``tests/sampling_ref.py``) applied to ``forward``'s logits of the
masked grid, in every precision and on both routes; results do not depend on how chains are grouped or steps are split
into calls; the draws follow ``softmax(logits / T)``."""
import os

import numpy as np
import pytest
import torch

from oracle import msa_ref as O
import sampling_ref as S

pytestmark = pytest.mark.gpu

PAD = O.PAD_IDX
MASK = O.TOK_TO_IDX["<mask>"]
ACGU_GAP = [4, 5, 6, 7, 10]


@pytest.fixture(scope="module")
def pkg():
    import rnamsm_b200
    return rnamsm_b200


def build(pkg, seed, layers=10, sharpen=1.0, precision="fp32"):
    model = pkg.MSATransformer(pkg.Vocab(pkg.Alphabet()), num_layers=layers, precision=precision)
    model.load_state_dict(O.make_weights(int(seed), num_layers=layers, sharpen=float(sharpen)), strict=True)
    return model.eval().cuda()


def golden(golden_dir, name):
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    return g, torch.from_numpy(g["tokens"].astype(np.int64))[0]


def reference_step(model, state, rows, allowed, p, T, seed, k, s):
    """-> (state after step s of chain k, masked, near) from forward's logits of the masked grid."""
    m = S.mask_set(state, rows, PAD, p, seed, k, s)
    grid = state.copy()
    grid[m] = MASK
    logits = model(torch.from_numpy(grid).cuda().unsqueeze(0), want_logits=True)["logits"][0].cpu().numpy()
    return S.step(state, logits, rows, PAD, allowed, p, T, seed, k, s)


# ------------------------------------------------------------------------------------------------ one step is exact
# (shape, rows): single_row runs one forward per grid in every precision; tiny_pad has pads and samples a subset of
# rows (the row gather); 2DRB_1 samples all rows (the head reads the layer output directly) and a subset.
CASES = [("single_row", None), ("tiny_pad", [0, 3, 5]), ("2DRB_1", None), ("2DRB_1", [0, 100, 511])]


@pytest.mark.parametrize("case", range(len(CASES)), ids=[f"{n}-{'all' if r is None else 'subset'}" for n, r in CASES])
@pytest.mark.parametrize("precision", ["fp16", "bf16", "fp32", "tf32x3"])
def test_one_step_matches_cpu_sampler(pkg, golden_dir, case, precision):
    name, rows = CASES[case]
    g, t = golden(golden_dir, name)
    model = build(pkg, g["wseed"], int(g["layers"]), float(g["sharpen"]), precision)
    R = t.shape[0]
    rows_l = list(range(R)) if rows is None else rows
    p, seed, s0, n_chains = 0.3, 0x5EED0000F00D + case, 5, 2
    draws = mism = 0
    for T in (1.0, 0.0):
        out = model.sample_msa(t.cuda(), 1, mask_prob=p, temperature=T, rows=rows, n_chains=n_chains, seed=seed,
                               start_step=s0).cpu().numpy()
        assert out.shape == (n_chains, *t.shape) and out.dtype == np.int64
        for k in range(n_chains):
            new, m, near = reference_step(model, t.numpy(), rows_l, ACGU_GAP, p, T, seed, k, s0)
            assert m.sum() > 0
            bad = out[k] != new
            assert not (bad & ~near).any(), (k, T, np.argwhere(bad & ~near)[:5])
            assert not (bad & ~m).any()
            draws += int(m.sum())
            mism += int(bad.sum())
    assert mism <= 1e-4 * draws, (mism, draws)


# ------------------------------------------------------------------------------------------------ resumable, grouping
@pytest.mark.parametrize("precision", ["fp16", "fp32"])
def test_steps_split_across_calls(pkg, golden_dir, precision):
    g, t = golden(golden_dir, "tiny_pad")
    model = build(pkg, g["wseed"], 10, 1.0, precision)
    kw = dict(mask_prob=0.25, rows=[0, 1, 4, 7], n_chains=3, seed=77)
    t = t.cuda()
    whole = model.sample_msa(t, 3, **kw)
    x = t
    for s in range(3):
        x = model.sample_msa(x, 1, start_step=s, **kw)
    assert torch.equal(whole, x)
    a = model.sample_msa(model.sample_msa(t, 2, **kw), 1, start_step=2, **kw)
    assert torch.equal(whole, a)
    assert not torch.equal(whole[0], whole[1])          # chains draw independently
    assert torch.equal(model.sample_msa(t, 0, **kw), t.expand(3, -1, -1))


@pytest.mark.parametrize("precision", ["fp16", "fp32"])
def test_group_does_not_change_results(pkg, golden_dir, precision):
    g, t = golden(golden_dir, "tiny_pad")
    model = build(pkg, g["wseed"], 10, 1.0, precision)
    t = t.cuda()
    T = t.numel()
    kw = dict(mask_prob=0.2, n_chains=5, seed=3, start_step=11)
    ref = model.sample_msa(t, 2, token_budget=T, **kw)                       # one chain per pass
    assert torch.equal(model.sample_msa(t, 2, token_budget=5 * T, **kw), ref)   # all chains in one pass
    assert torch.equal(model.sample_msa(t, 2, token_budget=2 * T, **kw), ref)   # 2 + 2 + 1
    assert torch.equal(model.sample_msa(t, 2, **kw), ref)


def test_invariants(pkg, golden_dir):
    g, t = golden(golden_dir, "tiny_pad")
    model = build(pkg, g["wseed"], 10, 1.0, "fp16")
    t = t.cuda()
    R, Cc = t.shape
    rows = [1, 2, 6]
    out = model.sample_msa(t, 6, mask_prob=0.5, rows=rows, n_chains=4, seed=1, allowed="GC")
    same = out == t
    assert same[:, :, 0].all()                                         # BOS column
    assert same[:, [r for r in range(R) if r not in rows]].all()       # rows outside `rows`
    pad = (t == PAD).expand_as(out)
    assert pad.any() and (out[pad] == PAD).all() and not (out[~pad] == PAD).any()
    changed = out[~same]
    assert changed.numel() > 0 and torch.isin(changed, torch.tensor([5, 6], device="cuda")).all()
    assert not (out == MASK).any()
    assert torch.equal(model.sample_msa(t, 3, mask_prob=0.0, n_chains=2, seed=1), t.expand(2, -1, -1))


# ------------------------------------------------------------------------------------------------ distribution
def test_draws_follow_softmax(pkg):
    """p = 1 on the query row: every chain masks the same tokens, so every draw at a column comes from the same
    logits.  The frequencies over 4000 chains match softmax(logits / T) over the allowed tokens at every column."""
    from scipy.stats import chisquare
    t = O.make_tokens(8, 20, 5)[0].cuda()
    model = build(pkg, 5, 4, 1.0, "fp16")
    grid = t.clone()
    grid[0, 1:] = MASK
    logits = model(grid.unsqueeze(0), want_logits=True)["logits"][0, 0].double().cpu()
    n = 4000
    for T in (0.5, 1.0, 2.0):
        out = model.sample_msa(t, 1, mask_prob=1.0, temperature=T, rows=[0], n_chains=n, seed=int(T * 10)).cpu()
        assert torch.equal(out[:, 1:], t[1:].cpu().expand(n, -1, -1))
        for c in range(1, t.shape[1]):
            p = torch.softmax(logits[c, ACGU_GAP] / T, -1).numpy()
            got = np.bincount(out[:, 0, c].numpy(), minlength=12)
            assert got[ACGU_GAP].sum() == n
            pv = chisquare(got[ACGU_GAP], p * n).pvalue
            assert pv > 1e-3, (T, c, pv, got[ACGU_GAP], p * n)


# ------------------------------------------------------------------------------------------------ routing
def launches(pkg):
    return pkg._lib.lib.rnamsm_launch_count()


def test_launch_counts(pkg):
    """16-bit: one step of a pass of g chains = rnamsm_msa_forward_batch on g grids minus its final LayerNorm, plus 6
    launches (mask, final LayerNorm, LM-head dense, LM-head LayerNorm, vocab projection, draw) and the row gather when
    `rows` is a subset.  fp32: one forward per grid without its final LayerNorm, plus the same 6 per pass."""
    t = O.make_tokens(24, 30, 3, pad_cols=2)[0].cuda()
    m16 = build(pkg, 4, 3, 1.0, "fp16")
    T = t.numel()
    m16.sample_msa(t, 1, n_chains=3, token_budget=3 * T)
    torch.cuda.synchronize()
    c0 = launches(pkg)
    m16.forward_batch([t, t, t])
    c1 = launches(pkg)
    m16.sample_msa(t, 1, n_chains=3, token_budget=3 * T)
    c2 = launches(pkg)
    m16.sample_msa(t, 2, n_chains=3, token_budget=3 * T, rows=[0, 5])
    c3 = launches(pkg)
    m16.sample_msa(t, 1, n_chains=6, token_budget=3 * T)          # two passes
    c4 = launches(pkg)
    fb = c1 - c0
    assert c2 - c1 == fb - 1 + 6
    assert c3 - c2 == 2 * (fb - 1 + 7)
    assert c4 - c3 == 2 * (fb - 1 + 6)
    m32 = build(pkg, 4, 3, 1.0, "fp32")
    m32(t.unsqueeze(0), want_logits=False)
    c0 = launches(pkg)
    m32(t.unsqueeze(0), want_logits=False)
    c1 = launches(pkg)
    m32.sample_msa(t, 1, n_chains=3, token_budget=3 * T)
    c2 = launches(pkg)
    assert c2 - c1 == 3 * ((c1 - c0) - 1) + 6


# ------------------------------------------------------------------------------------------------ CLI
def test_generate_cli(pkg, tmp_path):
    from rnamsm_b200 import generate
    from rnamsm_b200.inference import build_model
    rng = np.random.default_rng(4)
    L_, N_ = 23, 12
    seqs = ["".join(rng.choice(list("AGCU-"), L_)) for _ in range(N_)]
    a2m = tmp_path / "toy.a2m_msa2"
    a2m.write_text("".join(f">s{i}\n{s}\n" for i, s in enumerate(seqs)))
    for rows, n_rows in (("query", 1), ("all", N_)):
        out = tmp_path / f"gen_{rows}.fasta"
        generate.main(["--MSA_file", str(a2m), "--steps", "3", "--n_chains", "2", "--out", str(out), "--rows", rows,
                       "--mask_prob", "0.3", "--seed", "9"])
        names, got = pkg.read_msa(str(out), max_seqs=10 ** 6)
        assert len(got) == 2 * n_rows and all(len(s) == L_ for s in got)
        assert names[0] == "chain0_row0 source=0" and names[-1] == f"chain1_row{n_rows - 1} source={n_rows - 1}"
        model, vocab = build_model(None)
        tokens, _ = pkg.ingest_msa(str(a2m), vocab)
        ref = model.sample_msa(tokens, 3, mask_prob=0.3, rows=range(n_rows), n_chains=2, seed=9).cpu()
        want = ["".join(vocab.tokens[v] for v in ref[k, r, 1:].tolist()) for k in range(2) for r in range(n_rows)]
        assert got == want
        assert got[:n_rows] != [seqs[r] for r in range(n_rows)]
