"""CPU: the references the column-attention probability export is checked against, and its scratch-size math."""
import os

import numpy as np
import torch

from oracle import msa_ref as O
from col_probs_ref import forward_col_probs


def test_oracle_col_probs_match_reference_layer(golden_dir):
    """oracle axial_layer's column probabilities vs the reference layer's own (layer.npz col_nopad / col_pad,
    [H, C, B, R, R] at sharpen 8, padded rows and columns) at the bound oracle/gen_golden.py asserted."""
    g = np.load(os.path.join(golden_dir, "layer.npz"))
    sd = O.make_weights(int(g["wseed"]), num_layers=1, sharpen=float(g["sharpen"]))
    x = torch.from_numpy(g["x"])
    for tag, pm in (("nopad", None), ("pad", torch.from_numpy(g["pad"]))):
        _, col, _ = O.axial_layer(sd, 0, x, pm, return_col_probs=True)
        assert tuple(col.shape) == g[f"col_{tag}"].shape == (12, 19, 1, 7, 7)
        assert O.rel_err(col, g[f"col_{tag}"]) <= 2e-5


def test_model_level_reference_is_consistent_with_the_layer():
    """forward_col_probs: layer l's slab is axial_layer's probabilities on that layer's input, the mean is
    full.mean over the columns, rows sum to one, and padded keys get (almost) nothing."""
    sd = O.make_weights(3, num_layers=2, sharpen=2.0)
    tokens = O.make_tokens(5, 9, 1, batch=2, pad_cols=2)
    full, mean = forward_col_probs(sd, tokens)
    B, R, C = tokens.shape
    assert tuple(full.shape) == (B, 2, O.NUM_HEADS, C, R, R) and tuple(mean.shape) == (B, 2, O.NUM_HEADS, R, R)
    assert torch.allclose(mean, full.mean(3), rtol=0, atol=1e-7)
    assert torch.allclose(full.sum(-1), torch.ones(()), atol=1e-5)
    _, mean_only = forward_col_probs(sd, tokens, full=False)
    assert torch.equal(mean_only, mean)
    x, pm = O.embed(sd, tokens)
    x = x.permute(1, 2, 0, 3)
    x1, cp0, _ = O.axial_layer(sd, 0, x, pm, return_col_probs=True)
    assert torch.equal(full[:, 0], cp0.permute(2, 0, 1, 3, 4))
    _, cp1, _ = O.axial_layer(sd, 1, x1, pm, return_col_probs=True)
    assert torch.equal(full[:, 1], cp1.permute(2, 0, 1, 3, 4))
    # the model-level pass leaves the representations alone
    ref = O.forward(sd, tokens, repr_layers=[2], num_layers=2, want_logits=False)
    xr = O.layer_norm(O.axial_layer(sd, 1, x1, pm)[0], sd["emb_layer_norm_after.weight"], sd["emb_layer_norm_after.bias"])
    assert torch.equal(ref["representations"][2], xr.permute(2, 0, 1, 3))


def test_single_row_reference_is_all_ones():
    sd = O.make_weights(4, num_layers=1)
    full, mean = forward_col_probs(sd, O.make_tokens(1, 6, 2))
    assert tuple(full.shape) == (1, 1, O.NUM_HEADS, 6, 1, 1) and bool((full == 1).all()) and bool((mean == 1).all())


def test_col_probs_scratch_bytes_is_pure_host_math():
    """Two fp32 [H, C, R] arrays (per-row max and log-sum), 256 B aligned."""
    from rnamsm_b200 import _lib
    f = _lib.lib.rnamsm_col_probs_scratch_bytes
    assert f(512, 256, 12) == 2 * 12 * 256 * 512 * 4
    assert f(7, 19, 12) == (2 * 12 * 19 * 7 * 4 + 255) // 256 * 256
    assert f(4096, 128, 12) > f(512, 256, 12) and f(4096, 128, 12) % 256 == 0
    assert f(0, 64, 12) == 0 and f(64, 0, 12) == 0
