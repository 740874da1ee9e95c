"""Statistics of an alignment itself, with no model: sequence weights, the effective number of sequences (Neff) and
mean-field DCA contacts (Morcos et al., PNAS 2011), on the device over every row of the alignment
(``rnamsm_msa_seq_weights``, ``rnamsm_msa_dca``; DESIGN.md section 4.14).

Neff at 80 % identity says how deep an alignment really is; the DCA contacts are the classical coevolution baseline
that language-model contacts are compared against.  Read every record and column of a file with
``ingest_msa(path, vocab, sys.maxsize, sys.maxsize, "first")``."""
from __future__ import annotations

from typing import Dict, Tuple

import torch

from . import _lib as L


def _grid(tokens) -> torch.Tensor:
    if not isinstance(tokens, torch.Tensor):
        raise ValueError("tokens must be a torch.Tensor")
    t = tokens
    if t.dim() == 3:
        if t.shape[0] != 1:
            raise ValueError(f"tokens of shape {tuple(t.shape)}: expected [N, C] or [1, N, C]")
        t = t[0]
    if t.dim() != 2:
        raise ValueError(f"tokens of shape {tuple(tokens.shape)}: expected [N, C] or [1, N, C]")
    if t.dtype != torch.int64:
        raise ValueError(f"tokens must be int64, got {t.dtype}")
    N, C = t.shape
    if N < 1 or C < 2:
        raise ValueError(f"need at least one row and one residue column besides BOS, got [{N}, {C}]")
    if N > 2**31 - 1 or C > 2**31 - 1:
        raise ValueError(f"tokens [{N}, {C}] exceed the int32 sizes of the C entries")
    L.require_cuda(t, "tokens")
    return t.contiguous()


def _check_theta(theta: float) -> float:
    theta = float(theta)
    if not (0.0 < theta <= 1.0):
        raise ValueError(f"theta {theta} outside (0, 1]")
    return theta


def _check_pseudocount(pseudocount: float) -> float:
    pseudocount = float(pseudocount)
    if not (0.0 < pseudocount < 1.0):
        raise ValueError(f"pseudocount {pseudocount} outside (0, 1)")
    return pseudocount


def _workspace(nbytes: int, what: str, dev) -> torch.Tensor:
    if nbytes == 0:
        raise RuntimeError(f"{what}: " + L.lib.rnamsm_last_error().decode(errors="replace"))
    return torch.empty(nbytes, dtype=torch.uint8, device=dev)


@torch.no_grad()
def sequence_weights(tokens: torch.Tensor, theta: float = 0.8) -> Tuple[torch.Tensor, float]:
    """Sequence weights of an alignment and its effective number of sequences.

    ``tokens``: int64 ``[N, C]`` or ``[1, N, C]`` on the device, column 0 BOS (as ``ingest_msa`` returns them).  Row k
    is a neighbour of row n when at least ``theta * L`` of the ``L = C - 1`` residue columns hold the same state (A, G,
    C, U, or the gap state for every other token; gap matching gap counts); every row is its own neighbour.  Returns
    ``(weights, neff)``: float64 ``[N]`` on the device with ``w[n] = 1 / (neighbours of n)``, and ``neff = sum(w)``
    as a Python float (one host sync).  ``ValueError`` on a bad shape or theta, ``RuntimeError`` on CPU tensors."""
    theta = _check_theta(theta)
    t = _grid(tokens)
    N, C = t.shape
    dev = t.device
    L.device_check(dev)
    with torch.cuda.device(dev):
        weights = torch.empty(N, dtype=torch.float64, device=dev)
        neff = torch.empty(1, dtype=torch.float64, device=dev)
        nbytes = L.lib.rnamsm_seq_weights_workspace_bytes(N, C - 1)
        ws = _workspace(nbytes, "rnamsm_seq_weights_workspace_bytes", dev)
        L.check(L.lib.rnamsm_msa_seq_weights(L.ptr(t), N, C, theta, L.ptr(weights), L.ptr(neff), L.ptr(ws), nbytes,
                                             L.stream_ptr()), "msa_seq_weights")
        return weights, float(neff.item())


@torch.no_grad()
def dca_contacts(tokens: torch.Tensor, theta: float = 0.8, pseudocount: float = 0.5) -> Dict[str, object]:
    """Mean-field DCA contacts of an alignment, from every row of it.

    Sequence weights as :func:`sequence_weights`; weighted single-site and pair frequencies with pseudocount
    ``pseudocount``; the couplings ``e = -Cov^-1`` of the covariance over the states A, G, C, U (the gap state dropped);
    the Frobenius norm of each 4 x 4 coupling block in the zero-sum gauge; then the average product correction and
    symmetrisation of ``categorical_jacobian``'s contacts.  Returns ``{"contacts": fp32 [L, L], "weights": float64
    [N], "neff": float}`` (tensors on the device; one host sync).  The outputs and the workspace (two float64 matrices
    of side about 4L) are allocated before the first launch, so a size that does not fit fails before any kernel runs.
    ``ValueError`` on a bad shape, theta or pseudocount, ``RuntimeError`` on CPU tensors or a covariance matrix whose
    factorisation meets a non-positive pivot."""
    theta = _check_theta(theta)
    pseudocount = _check_pseudocount(pseudocount)
    t = _grid(tokens)
    N, C = t.shape
    Lr = C - 1
    dev = t.device
    L.device_check(dev)
    with torch.cuda.device(dev):
        weights = torch.empty(N, dtype=torch.float64, device=dev)
        neff = torch.empty(1, dtype=torch.float64, device=dev)
        contacts = torch.empty((Lr, Lr), dtype=torch.float32, device=dev)
        nbytes = L.lib.rnamsm_dca_workspace_bytes(N, Lr)
        ws = _workspace(nbytes, "rnamsm_dca_workspace_bytes", dev)
        L.check(L.lib.rnamsm_msa_dca(L.ptr(t), N, C, theta, pseudocount, L.ptr(weights), L.ptr(neff), L.ptr(contacts),
                                     L.ptr(ws), nbytes, L.stream_ptr()), "msa_dca")
        status = ws[:4].view(torch.int32).to(torch.float64)           # 0, or 1 + the first non-positive pivot
        neff_v, pivot = torch.cat([neff, status]).tolist()
    if pivot != 0:
        raise RuntimeError(f"rnamsm_b200 msa_dca: the covariance matrix is not positive definite: pivot "
                           f"{int(pivot) - 1} of {4 * Lr} is not positive")
    return {"contacts": contacts, "weights": weights, "neff": neff_v}
