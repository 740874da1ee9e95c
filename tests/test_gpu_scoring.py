"""GPU: LM-head scoring (``MSATransformer.masked_marginals`` / ``pseudo_log_likelihood`` / ``score_mutations``,
``rnamsm_msa_masked_marginals``, ``python -m rnamsm_b200.score``).

The logits are bit-identical to ``forward``'s logits of each masked grid at the scored token, in every precision and
on every route (the batch layer path in groups of grids, one forward per grid); log-probabilities match
``torch.log_softmax`` of them; and the marginals follow the float64 oracle within the model-level parity bounds."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from oracle import msa_ref as O
import scoring_ref as S

pytestmark = pytest.mark.gpu

# the model-level bounds of the forward's parity tests, applied as there: (precision, deep sharpened stack) -> bound
FP32_TOL = 1e-4
BF16_TOL = 2e-2
BF16_TOL_DEEP_SHARP = 8e-2
MASK = O.TOK_TO_IDX["<mask>"]


def tol(precision, sharp_deep):
    if precision == "fp32":
        return FP32_TOL
    return BF16_TOL_DEEP_SHARP if sharp_deep else BF16_TOL


@pytest.fixture(scope="module")
def pkg():
    import rnamsm_b200
    return rnamsm_b200


def build(pkg, seed, layers=10, sharpen=1.0, precision="fp32"):
    model = pkg.MSATransformer(pkg.Vocab(pkg.Alphabet()), num_layers=layers, precision=precision)
    sd = O.make_weights(int(seed), num_layers=layers, sharpen=float(sharpen))
    model.load_state_dict(sd, strict=True)
    return model.eval().cuda(), sd


def golden(golden_dir, name):
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    return g, torch.from_numpy(g["tokens"].astype(np.int64))[0]


def masked_logits(model, t, row, col):
    m = t.clone()
    m[row, col] = MASK
    return model(m.unsqueeze(0), want_logits=True)["logits"][0, row, col]


# ------------------------------------------------------------------------------------------------ bit identity
SHAPES = ["tiny", "tiny_pad", "single_row", "2DRB_1", "seeded_160x140"]


def shape_case(golden_dir, name):
    """-> (weight seed, sharpen, tokens [R, C], [(row, positions)])"""
    if name == "seeded_160x140":
        t = O.make_tokens(160, 140, 11, gap_p=0.1)[0]
        return 11, 1.0, t, [(0, [1, 2, 70, 139]), (97, [5, 64])]
    g, t = golden(golden_dir, name)
    R, Cc = t.shape
    if name == "2DRB_1":
        return int(g["wseed"]), float(g["sharpen"]), t, [(0, [1, 2, 17, 35]), (300, [9, 30])]
    cases = [(0, S.default_positions(t, 0))]
    if R > 2:
        cases.append((R // 2, S.default_positions(t, R // 2)[:5]))
    return int(g["wseed"]), float(g["sharpen"]), t, cases


@pytest.mark.parametrize("name", SHAPES)
@pytest.mark.parametrize("precision", ["fp16", "bf16", "fp32", "tf32x3"])
def test_logits_bit_identical_to_forward(pkg, golden_dir, name, precision):
    seed, sharpen, t, cases = shape_case(golden_dir, name)
    model, _ = build(pkg, seed, 10, sharpen, precision)
    t = t.cuda()
    T = t.numel()
    for row, pos in cases:
        ref = torch.stack([masked_logits(model, t, row, c) for c in pos])
        for group in (1, 3, len(pos)):                      # the last one runs every position in one pass
            lp, lg = model.masked_marginals(t, pos, row=row, token_budget=group * T, return_logits=True)
            assert lp.shape == lg.shape == (len(pos), 12) and lp.dtype == torch.float32
            assert torch.equal(lg, ref), (row, group, (lg - ref).abs().max().item())
            assert (lp - torch.log_softmax(ref, -1)).abs().max().item() <= 1e-6
        # wt-marginals: one forward, every position read from it
        wt = model(t.unsqueeze(0), want_logits=True)["logits"][0, row, pos]
        lp, lg = model.masked_marginals(t, pos, row=row, masked=False, token_budget=2 * T, return_logits=True)
        assert torch.equal(lg, wt)
        assert (lp - torch.log_softmax(wt, -1)).abs().max().item() <= 1e-6


def test_default_positions_and_3d_tokens(pkg, golden_dir):
    g, t = golden(golden_dir, "tiny_pad")
    model, _ = build(pkg, g["wseed"], 10, g["sharpen"], "fp16")
    t = t.cuda()
    for row in range(t.shape[0]):
        pos = S.default_positions(t.cpu(), row)
        a = model.masked_marginals(t, row=row)
        b = model.masked_marginals(t.unsqueeze(0), pos, row=row)
        assert a.shape == (len(pos), 12) and torch.equal(a, b)
    with pytest.raises(ValueError, match="padding"):
        model.masked_marginals(t, [t.shape[1] - 1], row=int((t.cpu() == O.PAD_IDX).any(1).nonzero()[0]))
    with pytest.raises(ValueError, match="outside"):
        model.masked_marginals(t, [t.shape[1]])
    with pytest.raises(ValueError, match="row"):
        model.masked_marginals(t, row=t.shape[0])
    with pytest.raises(RuntimeError, match="CUDA"):
        model.masked_marginals(t.cpu())


# ------------------------------------------------------------------------------------------------ float64 oracle
_ORACLE = {}


def oracle_marginals(name, sd, t, pos):
    key = (name, tuple(pos))
    if key not in _ORACLE:
        _ORACLE[key] = S.marginals(O.to_dtype(sd, torch.float64), t, pos)
    return _ORACLE[key]


@pytest.mark.parametrize("name", ["ragged_sharp", "mid_sharp"])
@pytest.mark.parametrize("precision", ["fp32", "fp16", "bf16"])
def test_marginals_vs_float64_oracle(pkg, golden_dir, name, precision):
    """Centred log-probabilities (each position minus its mean over V: random-init marginals sit near -log 12) against
    the float64 oracle; in 16-bit modes the argmax must agree wherever the oracle's top two are > 5e-3 apart."""
    g, t = golden(golden_dir, name)
    layers, sharpen = int(g["layers"]), float(g["sharpen"])
    model, sd = build(pkg, g["wseed"], layers, sharpen, precision)
    pos = S.default_positions(t)[::9][:4]
    ref = oracle_marginals(name, sd, t, pos)
    lp = model.masked_marginals(t.cuda(), pos).cpu().double()
    centred = lambda x: x - x.mean(-1, keepdim=True)
    err = O.rel_err(centred(lp), centred(ref))
    print(f"[{name}/{precision}] centred log-prob rel err {err:.3e}")
    assert err <= tol(precision, sharpen >= 3 and layers >= 10)
    if precision != "fp32":
        top2 = ref.topk(2, -1).values
        clear = (top2[:, 0] - top2[:, 1]) > 5e-3
        assert bool((lp.argmax(-1) == ref.argmax(-1))[clear].all())


# ------------------------------------------------------------------------------------------------ routing
def launches(pkg):
    return pkg._lib.lib.rnamsm_launch_count()


def test_routing_launch_counts(pkg):
    """16-bit: a pass of g grids = rnamsm_msa_forward_batch on those g grids minus its final LayerNorm, plus 7 launches
    (variant grids, gather, final LayerNorm, LM-head dense, LM-head LayerNorm, vocab projection, log-softmax).
    fp32: one forward per variant (without its final LayerNorm) plus a gather each, and 6 launches per pass."""
    t = O.make_tokens(24, 30, 3, pad_cols=2)[0].cuda()
    T = t.numel()
    m16, _ = build(pkg, 4, 3, 1.0, "fp16")
    grids = []
    for c in (1, 2, 3):
        g_ = t.clone()
        g_[0, c] = MASK
        grids.append(g_)
    m16.masked_marginals(t, [1, 2, 3], token_budget=3 * T)      # warm: weights staged, modules loaded
    torch.cuda.synchronize()
    c0 = launches(pkg)
    m16.forward_batch(grids)
    c1 = launches(pkg)
    m16.masked_marginals(t, [1, 2, 3], token_budget=3 * T)
    c2 = launches(pkg)
    m16.masked_marginals(t, [1, 2, 3, 1, 2, 3], token_budget=3 * T)     # two full passes
    c3 = launches(pkg)
    assert c2 - c1 == (c1 - c0) - 1 + 7
    assert c3 - c2 == 2 * (c2 - c1)
    m32, _ = build(pkg, 4, 3, 1.0, "fp32")
    m32(t.unsqueeze(0), want_logits=False)
    c0 = launches(pkg)
    m32(grids[0].unsqueeze(0), want_logits=False)
    c1 = launches(pkg)
    m32.masked_marginals(t, [1, 2, 3], token_budget=3 * T)
    c2 = launches(pkg)
    assert c2 - c1 == 3 * ((c1 - c0) - 1 + 1) + 6


def test_repeat_calls_are_bitwise_equal(pkg):
    t = O.make_tokens(40, 50, 8, pad_cols=3)[0].cuda()
    model, _ = build(pkg, 8, 4, 2.0, "fp16")
    a = model.masked_marginals(t, return_logits=True, token_budget=5 * t.numel())
    b = model.masked_marginals(t, return_logits=True, token_budget=5 * t.numel())
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.parametrize("precision", ["fp16", "fp32"])
def test_invalid_columns_give_nan_rows(pkg, precision):
    """The C entry called directly: an out-of-range column and a pad column come back as NaN rows; the valid entries
    around them are unaffected."""
    L = pkg._lib
    t = O.make_tokens(6, 12, 2, pad_cols=3)[0].cuda()
    R, Cc = t.shape
    model, _ = build(pkg, 2, 2, 1.0, precision)
    cols_l = [2, -1, Cc + 5, Cc - 1, 5, 1 << 20]
    cols = torch.tensor(cols_l, dtype=torch.int32, device="cuda")
    n, V, D, H = len(cols_l), 12, model.embed_dim, model.num_attention_heads
    lp = torch.zeros((n, V), device="cuda")
    lg = torch.zeros((n, V), device="cuda")
    group = 2
    code = model._fwd_code
    nbytes = L.lib.rnamsm_score_workspace_bytes(R, Cc, D, H, 4 * D, code, group)
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    m = model.c_weights(model._code)
    L.check(L.lib.rnamsm_msa_masked_marginals(C.byref(m), t.data_ptr(), R, Cc, 1, code, 0, cols.data_ptr(), n, MASK, group,
                                              lg.data_ptr(), lp.data_ptr(), ws.data_ptr(), nbytes, L.stream_ptr()))
    torch.cuda.synchronize()
    bad = [1, 2, 3, 5]
    assert bool(torch.isnan(lp[bad]).all()) and bool(torch.isnan(lg[bad]).all())
    good_lp, good_lg = model.masked_marginals(t, [2, 5], return_logits=True)
    assert torch.equal(lp[[0, 4]], good_lp) and torch.equal(lg[[0, 4]], good_lg)


# ------------------------------------------------------------------------------------------------ scores and PLL
@pytest.mark.parametrize("method", ["masked-marginals", "wt-marginals"])
def test_scores_and_pll_vs_reference(pkg, method):
    t = O.make_tokens(6, 14, 9, pad_cols=2)[0]
    model, sd = build(pkg, 9, 2, 1.0, "fp32")
    vocab = model.vocab
    q = t[0].tolist()
    letter = {v: k for k, v in vocab.tokens_to_idx.items()}
    alt = lambda c: "A" if letter[q[c]] != "A" else "G"
    muts = [f"{letter[q[3]]}3{alt(3)}", f"{letter[q[5]]}5{alt(5)}:{letter[q[11]]}11{alt(11)}",
            f"{letter[q[3]]}3U:{letter[q[1]]}1{alt(1)}", f"{letter[q[7]]}7{letter[q[7]]}"]
    got = model.score_mutations(t.cuda(), muts, method=method)
    assert got.dtype == torch.float64 and got.device.type == "cpu" and got.shape == (4,)
    parsed = [pkg.parse_mutant(s, q, vocab) for s in muts]
    pos = sorted({c for p in parsed for c, _, _ in p})
    ref_lp = S.marginals(O.to_dtype(sd, torch.float64), t, pos, masked=method == "masked-marginals")
    ref = torch.tensor(S.mutant_scores(ref_lp, pos, parsed), dtype=torch.float64)
    assert (got - ref).abs().max().item() <= 5e-4
    assert got[3].item() == 0.0
    # the scores are the stated sums of the library's own marginals
    lp = model.masked_marginals(t.cuda(), pos, masked=method == "masked-marginals").cpu().double()
    assert torch.equal(got, torch.tensor(S.mutant_scores(lp, pos, parsed), dtype=torch.float64))
    if method == "masked-marginals":
        pll, per = model.pseudo_log_likelihood(t.cuda())
        dpos = S.default_positions(t)
        ref_pll, ref_per = S.pll(S.marginals(O.to_dtype(sd, torch.float64), t, dpos), t, dpos)
        assert per.shape == (len(dpos),) and (per.cpu().double() - ref_per).abs().max().item() <= 5e-4
        assert abs(pll - ref_pll) <= 5e-4 * len(dpos)
        assert pll == float(per.double().sum())
    with pytest.raises(ValueError, match="wild type"):
        model.score_mutations(t.cuda(), [f"{'A' if letter[q[2]] != 'A' else 'G'}2C"], method=method)
    with pytest.raises(ValueError, match="padding"):
        model.score_mutations(t.cuda(), ["A13G"], method=method)


def test_score_cli(pkg, tmp_path):
    """python -m rnamsm_b200.score: TSV in input order, scores equal to score_mutations on the ingested tokens."""
    from rnamsm_b200 import score
    from rnamsm_b200.inference import build_model
    rng = np.random.default_rng(3)
    L_, N_ = 19, 24
    seqs = ["".join(rng.choice(list("AGCU-"), L_)) for _ in range(N_)]
    seqs[0] = seqs[0].replace("-", "A")
    a2m = tmp_path / "toy.a2m_msa2"
    a2m.write_text("".join(f">s{i}\n{s}\n" for i, s in enumerate(seqs)))
    q = seqs[0]
    alt = lambda c: "G" if c != "G" else "C"
    muts = [f"{q[9]}10{alt(q[9])}", f"{q[0]}1{alt(q[0])}:{q[18]}19T", f"{q[4]}5{alt(q[4])}"]
    (tmp_path / "muts.txt").write_text("\n".join(muts) + "\n")
    out, marg = tmp_path / "scores.tsv", tmp_path / "marg.npy"
    score.main(["--MSA_file", str(a2m), "--mutations", str(tmp_path / "muts.txt"), "--out", str(out),
                "--max_seqs_per_msa", "16", "--marginals_out", str(marg)])
    lines = out.read_text().splitlines()
    assert lines[0] == "mutant\tscore" and [ln.split("\t")[0] for ln in lines[1:]] == muts
    model, vocab = build_model(None)
    tokens, _ = pkg.ingest_msa(str(a2m), vocab, 16)
    ref = model.score_mutations(tokens, muts)
    assert [float(ln.split("\t")[1]) for ln in lines[1:]] == ref.tolist()
    lp = np.load(marg)
    assert lp.shape == (L_, 12) and lp.dtype == np.float32
    assert np.array_equal(lp, model.masked_marginals(tokens).cpu().numpy())
