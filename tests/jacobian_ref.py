"""CPU reference for the categorical Jacobian of the LM head (csrc/jacobian.cu): J from the oracle's forward
(oracle/msa_ref.forward), and the contact map from J, restated in float64 numpy."""
from typing import Sequence

import numpy as np
import torch

from oracle import msa_ref as O


@torch.no_grad()
def jacobian(sd, tokens2d: torch.Tensor, positions: Sequence[int], alphabet: Sequence[int], row: int = 0) -> np.ndarray:
    """``J[i, a, j, b] = f(G(i, a))[j, b] - f(tokens)[j, b]`` in the dtype of ``sd``; ``alphabet`` holds token indices.
    A wild-type substitution is not run: its slab is 0."""
    pos, alph = list(positions), list(alphabet)
    f = lambda t: O.forward(sd, t.unsqueeze(0))["logits"][0, row][pos][:, alph].numpy()
    wt = f(tokens2d)
    J = np.zeros((len(pos), len(alph), len(pos), len(alph)), dtype=wt.dtype)
    for i, c in enumerate(pos):
        for a, v in enumerate(alph):
            if int(tokens2d[row, c]) == v:
                continue
            t = tokens2d.clone()
            t[row, c] = v
            J[i, a] = f(t) - wt
    return J


def apc(F: np.ndarray) -> np.ndarray:
    """oracle/msa_ref.py::apc, with a correction of 0 when the total is 0."""
    total = F.sum()
    if total == 0:
        return F.copy()
    return F - F.sum(-1, keepdims=True) * F.sum(-2, keepdims=True) / total


def contacts(J: np.ndarray) -> np.ndarray:
    """[P, A, P, A] -> float64 [P, P]: centre over i, a, j, b in turn; Frobenius norm of each A x A block with a zero
    diagonal; APC with the diagonal zeroed again; (F + F^T) / 2."""
    Jc = np.asarray(J, dtype=np.float64)
    for axis in range(4):
        Jc = Jc - Jc.mean(axis=axis, keepdims=True)
    F = np.sqrt((Jc ** 2).sum(axis=(1, 3)))
    np.fill_diagonal(F, 0.0)
    F = apc(F)
    np.fill_diagonal(F, 0.0)
    return (F + F.T) / 2
