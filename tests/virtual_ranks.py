"""Virtual ranks: the sharded forward's peer-memory kernels run for n ranks in one process on one GPU (CPU helpers).

The exchange kernels of rna-msm_b200/sharded.py (csrc/peer.cu, the scatter epilogue of csrc/umma_gemm.cu) take an array
of per-rank device pointers and never ask whether those point into another GPU.  One process can therefore stand in for
n ranks: it allocates n local buffers per exchange, calls the kernel once per virtual rank with that rank's rank / r0 /
c0, and checks every buffer afterwards.  Stream order replaces the barriers between phases.

This module holds what those tests compare against, written from the contract in include/rnamsm_b200.h rather than from
the kernels:
  - the index maps of the exchanges (push destination, scatter destination, owned query rows);
  - GEMM operands on which the tensor-core result is exact, so the scatter checks need no tolerance;
  - partial logits whose sum in the rotated order the softmax kernels pull them in is exact.
"""
from __future__ import annotations

import numpy as np

import softmax_cases as SC


# ------------------------------------------------------------------------------------------ index maps
def shard(R: int, C: int, n: int):
    """Rows and columns per rank (Rn, Cn) of an R x C grid over n ranks."""
    assert R % n == 0 and C % n == 0, (R, C, n)
    return R // n, C // n


def push_dest(r: int, c: int, R: int, C: int, n: int):
    """rnamsm_layernorm_push: token (r, c) of the MSA -> (owner, row) in the column owner's [C/n * R, D] buffer."""
    _, Cn = shard(R, C, n)
    d = c // Cn
    return d, (c - d * Cn) * R + r


def scatter_dest(g: int, m: int, R: int, C: int, n: int):
    """rnamsm_linear_residual_scatter of rank g (columns [g Cn, (g+1) Cn)): output row m = r * Cn + cl of its GEMM ->
    (owner, row) in the row owner's [Rn * C, N] buffer."""
    Rn, Cn = shard(R, C, n)
    r, cl = divmod(m, Cn)
    owner = r // Rn
    return owner, (r - owner * Rn) * C + g * Cn + cl


def owned_rows(g: int, C: int, n: int) -> range:
    """rnamsm_row_softmax_p2p: the query rows rank g owns."""
    Cq = C // n
    return range(g * Cq, (g + 1) * Cq)


def push_index(R: int, C: int, n: int):
    """push_dest for every token in token-major order (r * C + c) -> owner [R*C], row [R*C] (int64 arrays)."""
    _, Cn = shard(R, C, n)
    r, c = np.divmod(np.arange(R * C), C)
    d = c // Cn
    return d, (c - d * Cn) * R + r


def scatter_index(g: int, R: int, C: int, n: int):
    """scatter_dest for every output row m of rank g's GEMM -> owner [R*Cn], row [R*Cn] (int64 arrays)."""
    Rn, Cn = shard(R, C, n)
    r, cl = np.divmod(np.arange(R * Cn), Cn)
    owner = r // Rn
    return owner, (r - owner * Rn) * C + g * Cn + cl


# ------------------------------------------------------------------------------------------ exact GEMM operands
# ctx = i / 8 and W = j / 64, bias and the residual stream on the 2^-9 grid: tests/gemm_exact.py.
from gemm_exact import (AFFINE_MAX, CTX_DEN, GRID, W_DEN, exact_affine, exact_gemm_operands,  # noqa: E402,F401
                        exact_sum_bound_ulps)


# ------------------------------------------------------------------------------------------ softmax partials
def p2p_partials(s: np.ndarray, n: int, n_splits: int, seed: int) -> np.ndarray:
    """[n * n_splits, H, C, C] float32 partial logits of 2 s (LOGIT_SCALE 0.5 gives back s): rank g holds slabs
    [g n_splits, (g+1) n_splits).  softmax_cases.split_partials: all slabs but the last are multiples of 1/8 in
    [-4, 4], the last is the remainder, so every partial sum in any order stays on the logits' grid."""
    return SC.split_partials(2.0 * s, n * n_splits, seed)


def rotated_order(rank: int, n: int, n_splits: int):
    """Slab indices in the order the p2p softmax kernels of `rank` add them: t = 1..n, source (rank + t) % n, splits
    in order."""
    return [((rank + t) % n) * n_splits + s for t in range(1, n + 1) for s in range(n_splits)]


def rotated_sum(parts: np.ndarray, rank: int, n: int, n_splits: int) -> np.ndarray:
    """The fp32 sum the kernels of `rank` form, starting from 0 and adding one slab at a time."""
    acc = np.zeros(parts.shape[1:], dtype=np.float32)
    for k in rotated_order(rank, n, n_splits):
        acc = acc + parts[k]
    return acc
