"""CPU reference for LM-head scoring: masked / wt marginals from the oracle's forward (oracle/msa_ref.forward), and the
mutant scores and pseudo-log-likelihood as the plain sums of those marginals."""
from typing import List, Optional, Sequence, Tuple

import torch

from oracle import msa_ref as O


def default_positions(tokens2d: torch.Tensor, row: int = 0) -> List[int]:
    """Every non-pad column of ``row`` except the BOS column 0."""
    return [c for c in range(1, tokens2d.shape[1]) if int(tokens2d[row, c]) != O.PAD_IDX]


@torch.no_grad()
def marginals(sd, tokens2d: torch.Tensor, positions: Optional[Sequence[int]] = None, row: int = 0, masked: bool = True,
              num_layers: Optional[int] = None) -> torch.Tensor:
    """-> log-probabilities ``[P, V]`` in the dtype of ``sd``: entry k from the grid with ``(row, positions[k])``
    replaced by ``<mask>`` (``masked=False``: all from one forward of ``tokens2d``)."""
    if positions is None:
        positions = default_positions(tokens2d, row)
    out = []
    if not masked:
        logits = O.forward(sd, tokens2d.unsqueeze(0), num_layers=num_layers)["logits"][0]
        return torch.log_softmax(logits[row, list(positions)], -1)
    for c in positions:
        t = tokens2d.clone()
        t[row, c] = O.TOK_TO_IDX["<mask>"]
        logits = O.forward(sd, t.unsqueeze(0), num_layers=num_layers)["logits"][0]
        out.append(torch.log_softmax(logits[row, c], -1))
    return torch.stack(out)


def mutant_scores(lp: torch.Tensor, positions: Sequence[int], parsed: Sequence[Sequence[Tuple[int, int, int]]]) -> List[float]:
    """``sum over (col, wt, mt) of lp[col, mt] - lp[col, wt]`` per mutant; ``lp`` rows follow ``positions``."""
    at = {c: i for i, c in enumerate(positions)}
    return [sum(float(lp[at[c], mt]) - float(lp[at[c], wt]) for c, wt, mt in subs) for subs in parsed]


def pll(lp: torch.Tensor, tokens2d: torch.Tensor, positions: Sequence[int], row: int = 0) -> Tuple[float, torch.Tensor]:
    """-> (float64 sum, per-position ``log p(wt | wt masked)``) over ``positions`` (the rows of ``lp``)."""
    per = torch.stack([lp[i, int(tokens2d[row, c])] for i, c in enumerate(positions)])
    return float(per.double().sum()), per
