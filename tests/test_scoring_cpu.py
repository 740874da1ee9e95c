"""CPU: LM-head scoring -- mutant parsing, pass planning, the scoring workspace layout, and the float64 reference
(masked / wt marginals, mutant scores, pseudo-log-likelihood) against the reference's own committed logits."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from oracle import msa_ref as O
import scoring_ref as S


@pytest.fixture(scope="module")
def vocab():
    import rnamsm_b200
    return rnamsm_b200.Vocab(rnamsm_b200.Alphabet())


def _query(vocab, seq, pad=0):
    """Token ids of one row: <cls> + seq + pad x <pad>."""
    return [vocab.bos_idx] + [vocab.tokens_to_idx[c] for c in seq] + [vocab.pad_idx] * pad


# ------------------------------------------------------------------------------------------------ mutant parsing
def test_parse_single_and_multi_site(vocab):
    from rnamsm_b200.mutations import parse_mutant
    q = _query(vocab, "GACU-N")
    idx = vocab.tokens_to_idx
    assert parse_mutant("G1A", q, vocab) == [(1, idx["G"], idx["A"])]
    assert parse_mutant("G1A:C3U", q, vocab) == [(1, idx["G"], idx["A"]), (3, idx["C"], idx["U"])]
    assert parse_mutant(" C3G : U4- ", q, vocab) == [(3, idx["C"], idx["G"]), (4, idx["U"], idx["-"])]
    assert parse_mutant("-5A", q, vocab) == [(5, idx["-"], idx["A"])]
    assert parse_mutant("A2A", q, vocab) == [(2, idx["A"], idx["A"])]     # a synonymous entry scores 0


def test_parse_reads_t_as_u(vocab):
    from rnamsm_b200.mutations import parse_mutant
    q = _query(vocab, "GACU")
    u = vocab.tokens_to_idx["U"]
    assert parse_mutant("G1T", q, vocab) == [(1, vocab.tokens_to_idx["G"], u)]
    assert parse_mutant("T4A", q, vocab) == [(4, u, vocab.tokens_to_idx["A"])]


@pytest.mark.parametrize("spec,match", [
    ("A1G", "wild type"),                 # the query has G at 1
    ("G0A", "outside"),                   # column 0 is <cls>
    ("G9A", "outside"),                   # past the last column
    ("A6G", "padding"),                   # a pad column of the query
    ("G1Z", "unknown residue"),
    ("B1A", "unknown residue"),
    ("G1A:G1C", "twice"),
    ("G1A:A2G:G1U", "twice"),
    ("G1", "not <wt><index><mt>"),
    ("1A", "not <wt><index><mt>"),
    ("G1A;C3U", "not <wt><index><mt>"),
    ("", "empty"),
])
def test_parse_errors(vocab, spec, match):
    from rnamsm_b200.mutations import parse_mutant
    q = _query(vocab, "GACUU", pad=3)     # columns 0..8, 6..8 pad
    with pytest.raises(ValueError, match=match):
        parse_mutant(spec, q, vocab)


def test_read_mutants(tmp_path):
    from rnamsm_b200.mutations import read_mutants
    p = tmp_path / "m.txt"
    p.write_text("G1A\n\n# comment\n  C3U:G1A  \n")
    assert read_mutants(str(p)) == ["G1A", "C3U:G1A"]


# ------------------------------------------------------------------------------------------------ pass planning
def test_plan_score_group():
    from rnamsm_b200 import plan_score_group
    assert plan_score_group(512, 36, 35) == (14, 3)           # 262144 // 18432 = 14 grids; 14 + 14 + 7
    assert plan_score_group(512, 256, 255) == (2, 128)        # 127 full passes and a last one of 1
    assert plan_score_group(512, 36, 35, token_budget=1) == (1, 35)
    assert plan_score_group(6, 9, 8) == (8, 1)                # capped at the position count: one pass
    assert plan_score_group(6, 9, 8, token_budget=54 * 3) == (3, 3)   # 3 + 3 + 2
    assert plan_score_group(4096, 128, 10) == (1, 10)         # one grid above the budget still runs, alone
    assert plan_score_group(6, 9, 0)[1] == 0


# ------------------------------------------------------------------------------------------------ workspace
def _layout(lib, R, Cc, code, g, D=768, H=12, F=3072):
    """The regions rnamsm_score_workspace_bytes documents, rebuilt from the library's other size functions."""
    a = lambda x: (x + 255) // 256 * 256
    dt, tensor = code & 0xFF, bool(code & 0x100)
    T = R * Cc
    batch = dt in (1, 2) and R >= 2
    if batch:
        Rs, Cs = (C.c_int * g)(*[R] * g), (C.c_int * g)(*[Cc] * g)
        fwd = lib.rnamsm_batch_workspace_bytes(g, Rs, Cs, D, H, F, dt)
    else:
        fwd = lib.rnamsm_workspace_bytes(R, Cc, D, H, F, code) + a(T)
    total = a(g * T * 8) + a((g if batch else 1) * T * D * 4) + a(fwd) + a(g * D * 4)
    total += a(g * D * 2) if dt in (1, 2) else 0
    total += 2 * a(g * D * 4)
    total += lib.rnamsm_linear_tf32_scratch_bytes(g, D, D) if tensor else 0
    return total


@pytest.mark.parametrize("R,Cc", [(512, 36), (512, 256), (6, 9), (1, 21), (160, 140)])
@pytest.mark.parametrize("precision", ["fp16", "bf16", "fp32", "tf32x3"])
def test_score_workspace_bytes_matches_layout(R, Cc, precision):
    from rnamsm_b200 import _lib
    code = _lib.forward_code(precision)
    for g in (1, 3, 14):
        got = _lib.lib.rnamsm_score_workspace_bytes(R, Cc, 768, 12, 3072, code, g)
        assert got == _layout(_lib.lib, R, Cc, code, g) and got % 256 == 0
    assert _lib.lib.rnamsm_score_workspace_bytes(R, Cc, 768, 12, 3072, code, 3) > \
        _lib.lib.rnamsm_score_workspace_bytes(R, Cc, 768, 12, 3072, code, 1)


def test_score_workspace_bytes_invalid_is_zero():
    from rnamsm_b200 import _lib
    f = _lib.lib.rnamsm_score_workspace_bytes
    assert f(0, 36, 768, 12, 3072, _lib.F16, 1) == 0
    assert f(512, 0, 768, 12, 3072, _lib.F16, 1) == 0
    assert f(512, 36, 768, 12, 3072, _lib.F16, 0) == 0
    assert f(512, 36, 768, 12, 3072, 7, 1) == 0
    assert f(512, 36, 768, 12, 3072, _lib.F16 | _lib.F32_TENSOR, 1) == 0
    assert b"dtype" in _lib.lib.rnamsm_last_error()


# ------------------------------------------------------------------------------------------------ reference
@pytest.fixture(scope="module")
def sd64():
    return O.to_dtype(O.make_weights(42, num_layers=10), torch.float64)


@pytest.mark.parametrize("name", ["tiny", "tiny_pad"])
def test_reference_wt_marginals_match_golden_logits(golden_dir, sd64, name):
    """The reference's own logits (golden, fp32) through log_softmax equal the float64 wt-marginals."""
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    assert int(g["wseed"]) == 42 and int(g["layers"]) == 10 and float(g["sharpen"]) == 1.0
    tokens = torch.from_numpy(g["tokens"].astype(np.int64))[0]
    rows = g["rep_rows"].tolist()
    for i, row in enumerate(rows[:3]):
        pos = S.default_positions(tokens, row)
        lp = S.marginals(sd64, tokens, pos, row=row, masked=False)
        ref = torch.log_softmax(torch.from_numpy(g["logits"][0, i, pos]).double(), -1)
        assert lp.shape == (len(pos), 12)
        assert (lp - ref).abs().max() < 1e-5


def test_reference_masked_marginals_mask_the_scored_token():
    """Entry k of the masked marginals is the wt forward of the grid with that one token masked."""
    sd = O.to_dtype(O.make_weights(3, num_layers=2), torch.float64)
    tokens = O.make_tokens(4, 8, 1, pad_cols=2)[0]
    pos = S.default_positions(tokens, 1)
    assert pos == [1, 2, 3, 4, 5]
    lp = S.marginals(sd, tokens, pos, row=1)
    for k, c in enumerate(pos):
        t = tokens.clone()
        t[1, c] = O.TOK_TO_IDX["<mask>"]
        assert torch.equal(lp[k], S.marginals(sd, t, [c], row=1, masked=False)[0])
    assert torch.allclose(lp.exp().sum(-1), torch.ones((), dtype=torch.float64))


def test_reference_scores_and_pll_are_the_stated_sums(vocab):
    from rnamsm_b200.mutations import parse_mutant
    sd = O.to_dtype(O.make_weights(5, num_layers=2), torch.float64)
    tokens = O.make_tokens(3, 7, 2)[0]
    pos = S.default_positions(tokens)
    lp = S.marginals(sd, tokens, pos)
    q = tokens[0].tolist()
    letter = {v: k for k, v in vocab.tokens_to_idx.items()}
    w1, w3 = letter[q[1]], letter[q[3]]
    m1 = "A" if w1 != "A" else "G"
    m3 = "C" if w3 != "C" else "U"
    muts = [f"{w1}1{m1}", f"{w1}1{m1}:{w3}3{m3}", f"{w3}3{w3}"]
    parsed = [parse_mutant(s, q, vocab) for s in muts]
    sc = S.mutant_scores(lp, pos, parsed)
    a = float(lp[0, vocab.tokens_to_idx[m1]] - lp[0, q[1]])
    b = float(lp[2, vocab.tokens_to_idx[m3]] - lp[2, q[3]])
    assert sc[0] == pytest.approx(a, abs=1e-12) and sc[1] == pytest.approx(a + b, abs=1e-12) and sc[2] == 0.0
    total, per = S.pll(lp, tokens, pos)
    assert per.shape == (len(pos),) and total == pytest.approx(sum(float(lp[i, q[c]]) for i, c in enumerate(pos)), abs=1e-12)
    assert total < 0
