"""CPU: pin the oracle (oracle/msa_ref.py) against the committed golden vectors, which are outputs
of the reference's own modules (oracle/gen_golden.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import msa_ref as O

CASES = ["tiny", "tiny_pad", "ragged_sharp", "single_row", "batch2_pad", "mid_sharp"]


def load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name + ".npz"))


def run_oracle(g, dtype=torch.float32, **kw):
    layers = int(g["layers"])
    sd = O.make_weights(int(g["wseed"]), num_layers=layers, sharpen=float(g["sharpen"]))
    if dtype != torch.float32:
        sd = O.to_dtype(sd, dtype)
    tokens = torch.from_numpy(g["tokens"].astype(np.int64))
    return O.forward(sd, tokens, repr_layers=[0, 1, layers], need_head_weights=True, num_layers=layers, **kw), layers


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_reference_golden(golden_dir, name):
    g = load(golden_dir, name)
    out, layers = run_oracle(g)
    rows = g["rep_rows"]
    # un-chunked reference path: the restatement is the same op sequence => fp32 noise only
    assert O.rel_err(out["representations"][0][:, rows], g["rep0"]) < 1e-6
    assert O.rel_err(out["representations"][1][:, rows], g["rep1"]) < 1e-5
    assert O.rel_err(out["representations"][layers][:, rows], g["rep_last"]) < 1e-5
    assert O.rel_err(out["logits"][:, rows], g["logits"]) < 1e-5
    ra = out["row_attentions"]
    if "row_attentions" in g:
        assert O.rel_err(ra, g["row_attentions"]) < 1e-5
    else:
        flat = ra.reshape(ra.shape[0], -1, ra.shape[-2], ra.shape[-1])
        assert O.rel_err(flat[:, g["row_attentions_sel_idx"]], g["row_attentions_sel"]) < 1e-5
        assert O.rel_err(flat.mean(1), g["row_attentions_mean"]) < 1e-5
    if "emb" in g:
        emb, atp = O.extract_features(out, layers)
        assert emb.dtype == np.float32 and emb.shape == g["emb"].shape
        assert O.rel_err(emb, g["emb"]) < 1e-5
        if "atp" in g:
            assert atp.dtype == np.float32 and atp.shape == g["atp"].shape
            assert O.rel_err(atp, g["atp"]) < 1e-5


def test_oracle_chunked_reference_path(golden_dir):
    """R*C > 16384: the reference takes its chunked path (different fp32 summation order)."""
    g = load(golden_dir, "chunked")
    out, layers = run_oracle(g)
    rows = g["rep_rows"]
    assert O.rel_err(out["representations"][layers][:, rows], g["rep_last"]) < 2e-4
    ra = out["row_attentions"]
    flat = ra.reshape(ra.shape[0], -1, ra.shape[-2], ra.shape[-1])
    assert O.rel_err(flat[:, g["row_attentions_sel_idx"]], g["row_attentions_sel"]) < 2e-3


def test_oracle_layer_matches_reference_layer(golden_dir):
    g = load(golden_dir, "layer")
    sd = O.make_weights(int(g["wseed"]), num_layers=1, sharpen=float(g["sharpen"]))
    x = torch.from_numpy(g["x"])
    pad = torch.from_numpy(g["pad"])
    for tag, pm in (("nopad", None), ("pad", pad)):
        y, col, row = O.axial_layer(sd, 0, x, pm, return_col_probs=True)
        assert O.rel_err(y, g[f"y_{tag}"]) < 1e-6
        assert O.rel_err(row, g[f"row_{tag}"]) < 1e-6
        assert O.rel_err(col, g[f"col_{tag}"]) < 1e-6


def test_oracle_2drb_config1(golden_dir):
    """BASELINE config 1 (results/2DRB_1.a2m_msa2, first 512 rows): emb (35,768) + atp (120,35,35)."""
    g = load(golden_dir, "2DRB_1")
    sd = O.make_weights(int(g["wseed"]), sharpen=float(g["sharpen"]))
    tokens = torch.from_numpy(g["tokens"].astype(np.int64))
    assert tuple(tokens.shape) == (1, 512, 36)
    out = O.forward(sd, tokens, repr_layers=[10], need_head_weights=True, want_logits=False)
    emb, atp = O.extract_features(out)
    assert tuple(g["shipped_atp_shape"]) == atp.shape == (120, 35, 35)
    assert tuple(g["shipped_emb_shape"]) == emb.shape == (35, 768)
    assert O.rel_err(emb, g["emb"]) < 5e-5      # reference used its chunked path here
    assert O.rel_err(atp, g["atp"]) < 1e-4
    # invariants of the shipped fixtures: non-negative, rows sum to <= 1 (BOS column removed)
    assert atp.min() >= 0 and atp.sum(-1).max() <= 1 + 1e-5


def test_oracle_fp64_close_to_fp32(golden_dir):
    g = load(golden_dir, "tiny_pad")
    o32, layers = run_oracle(g)
    o64, _ = run_oracle(g, torch.float64)
    assert O.rel_err(o32["representations"][layers], o64["representations"][layers]) < 1e-5
    assert O.rel_err(o32["row_attentions"], o64["row_attentions"]) < 1e-5


def test_positions_rule():
    tok = torch.tensor([[0, 4, 1, 5, 1, 1], [0, 1, 1, 4, 5, 6]])
    assert O.positions_from_tokens(tok).tolist() == [[2, 3, 1, 4, 1, 1], [2, 1, 1, 3, 4, 5]]


def test_row_limit_error():
    sd = O.make_weights(0, num_layers=1)
    with pytest.raises(RuntimeError):
        O.embed(sd, torch.zeros(1, 1025, 3, dtype=torch.int64))


def test_read_a2m_matches_shipped_msa(golden_dir, msa_2drb_file):
    _, tok = O.read_a2m(msa_2drb_file, 512)
    g = load(golden_dir, "2DRB_1")
    assert np.array_equal(tok.numpy(), g["tokens"][0].astype(np.int64))


def test_oracle_rsa_input_matches_reference(golden_dir):
    """oracle rsa_input vs the tensor produced by executing the reference's own packing statements
    (oracle/gen_golden_rsa.py): bit-exact, including the float64 -> f32 one-hot z-scores."""
    g = load(golden_dir, "rsa_pack")
    x = O.rsa_input(g["emb"], str(g["seq"]), g["mu_emb"], g["std_emb"], g["mu_oh"], g["std_oh"])
    assert x.shape == g["x"].shape == (1, 773, len(str(g["seq"]))) and x.dtype == np.float32
    assert np.array_equal(x, g["x"])
    x0 = O.rsa_input(g["emb"], str(g["seq"]), g["mu_emb"], g["std_emb"])
    assert np.array_equal(x0[0], g["x"][0, 4:])

