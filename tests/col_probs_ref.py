"""Model-level CPU reference for the column-attention probabilities: the oracle's layer-streaming forward
(oracle/msa_ref.forward) with each layer's column probabilities kept (oracle/msa_ref.axial_layer,
return_col_probs=True, pinned to the reference's own vectors by tests/test_oracle.py)."""
from typing import Optional

import torch

from oracle import msa_ref as O


@torch.no_grad()
def forward_col_probs(sd, tokens: torch.Tensor, num_layers: Optional[int] = None, full: bool = True):
    """-> (col_attentions [B, N, H, C, R, R] or None when full=False, col_attentions_mean [B, N, H, R, R]), in the
    dtype of ``sd`` -- the layout of the reference's msm/ model and of MSATransformer.forward(need_col_weights=True)."""
    if num_layers is None:
        num_layers = 1 + max(int(k.split(".")[1]) for k in sd if k.startswith("layers."))
    x, padding_mask = O.embed(sd, tokens)
    x = x.permute(1, 2, 0, 3)                                       # B,R,C,D -> R,C,B,D
    cols, means = [], []
    for l in range(num_layers):
        x, cp, _ = O.axial_layer(sd, l, x, padding_mask, return_col_probs=True)   # cp: H,C,B,R,R
        if full:
            cols.append(cp.permute(2, 0, 1, 3, 4))
        means.append(cp.mean(1).permute(1, 0, 2, 3))
    return (torch.stack(cols, 1) if full else None), torch.stack(means, 1)
