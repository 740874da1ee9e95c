"""Nested secondary structure from a pair map, folded on the device (``rnamsm_fold``; DESIGN.md section 4.15), and the
files an RNA user reads it in: dot-bracket, ``.ct`` and ``.bpseq``.

Any of the library's pair maps folds: the contact head's probabilities (``predict_contacts``, ``forward_windows(...,
return_contacts=True)``) with ``mode="mea"``, and the APC scores of ``categorical_jacobian`` and ``dca_contacts`` with
``mode="score"``.  ``tests/fold_ref.py`` restates the folding in float32 numpy, and the device result is bit-identical
to it."""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional

import numpy as np
import torch

from . import _lib as L

MODES = {"mea": 0, "score": 1}
# sequence codes of the C entry: A G C U pair, every other letter never does
_LETTERS = "AGCUXN-"
_LUT = np.full(256, 255, dtype=np.uint8)
for _n, _c in enumerate(_LETTERS):
    _LUT[ord(_c)] = _n


def _codes(seq: str, Lm: int, m: int) -> np.ndarray:
    if not isinstance(seq, str):
        raise ValueError(f"sequence {m} must be a str, got {type(seq).__name__}")
    if len(seq) != Lm:
        raise ValueError(f"sequence {m} has {len(seq)} letters but its map is {Lm} x {Lm}")
    c = _LUT[np.frombuffer(seq.encode("latin-1", errors="replace"), dtype=np.uint8)]
    if (c == 255).any():
        bad = sorted({ch for ch in seq if ch not in _LETTERS})
        raise ValueError(f"sequence {m} has letters {bad} outside {' '.join(_LETTERS)}")
    return c


@torch.no_grad()
def fold_pairs(maps, sequences=None, mode: str = "mea", gamma: float = 1.0, threshold: float = 0.0,
               min_loop: int = 3, canonical: Optional[bool] = None):
    """Fold pair maps into nested secondary structures.

    ``maps``: one fp32 ``[L, L]`` CUDA tensor, or a list of them (lengths may differ; all on one device).  Only the
    upper triangle ``S[i, j]``, ``i < j``, is read.  A pair ``(i, j)`` is allowed when ``j - i > min_loop``,
    ``S[i, j] > threshold`` (compared in fp32) and, with ``canonical``, the letters pair as AU, GC or GU in either
    order (``X``, ``N`` and ``-`` never pair).  ``canonical`` defaults to on when ``sequences`` are given: one str per
    map (a str for a single map), letters of ``A G C U X N -``.

    ``mode="mea"`` (maps of pair probabilities; maximum expected accuracy): maximises ``sum_pairs 2 gamma S[i, j] +
    sum_unpaired (1 - sum_{j != i} S[i, j])``.  ``mode="score"`` (any score, e.g. APC contacts): maximises the sum of
    ``S`` over the pairs (``gamma`` ignored).  Ties break towards "unpaired", then towards the nearest partner.

    Returns ``(pairs, score)`` for one map and ``(list of pairs, list of scores)`` for a list: ``pairs`` int32 ``[L]``
    on the device, the partner of each position or -1; ``score`` the optimum as a Python float (an fp32 value).  One
    host sync.  Outputs and the workspace (two fp32 tables of about ``L x L`` per map) are allocated before the first
    launch, so a size that does not fit fails before any kernel runs.  ``ValueError`` on bad arguments or a
    non-finite map entry, ``RuntimeError`` on CPU tensors."""
    single = isinstance(maps, torch.Tensor)
    mlist = [maps] if single else list(maps)
    if not mlist:
        raise ValueError("no maps")
    if mode not in MODES:
        raise ValueError(f"mode {mode!r}: expected 'mea' or 'score'")
    gamma, threshold = float(gamma), float(threshold)
    with np.errstate(over="ignore"):
        g32, t32 = np.float32(2.0 * gamma), np.float32(threshold)
    if mode == "mea" and not (gamma > 0.0 and math.isfinite(gamma) and math.isfinite(g32)):
        raise ValueError(f"gamma {gamma} must be positive and finite")
    if not math.isfinite(threshold) or not math.isfinite(t32):
        raise ValueError(f"threshold {threshold} must be finite in fp32")
    if isinstance(min_loop, bool) or not isinstance(min_loop, (int, np.integer)) or min_loop < 0:
        raise ValueError(f"min_loop {min_loop!r} must be an int >= 0")
    for m, t in enumerate(mlist):
        if not isinstance(t, torch.Tensor):
            raise ValueError(f"map {m} must be a torch.Tensor")
        if t.dim() != 2 or t.shape[0] != t.shape[1] or t.shape[0] < 1:
            raise ValueError(f"map {m} of shape {tuple(t.shape)}: expected [L, L], L >= 1")
        if t.dtype != torch.float32:
            raise ValueError(f"map {m} must be float32, got {t.dtype}")
    Ls = [int(t.shape[0]) for t in mlist]
    if sequences is not None:
        seqs = [sequences] if single and isinstance(sequences, str) else sequences
        if isinstance(seqs, str) or len(seqs) != len(mlist):
            raise ValueError(f"need one sequence per map ({len(mlist)})")
        codes = [_codes(s, Lm, m) for m, (s, Lm) in enumerate(zip(seqs, Ls))]
    if canonical is None:
        canonical = sequences is not None
    canonical = bool(canonical)
    if canonical and sequences is None:
        raise ValueError("canonical pairing needs the sequences")
    for m, t in enumerate(mlist):
        L.require_cuda(t, f"map {m}")
    dev = mlist[0].device
    if any(t.device != dev for t in mlist):
        raise ValueError("all maps must be on one device")
    n = len(mlist)
    L.device_check(dev)
    Larr = (C.c_int * n)(*Ls)
    with torch.cuda.device(dev):
        nbytes = L.lib.rnamsm_fold_workspace_bytes(n, Larr)
        if nbytes == 0:
            raise ValueError("rnamsm_fold_workspace_bytes: " + L.lib.rnamsm_last_error().decode(errors="replace"))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        pairs = [torch.empty(Lm, dtype=torch.int32, device=dev) for Lm in Ls]
        scores = torch.empty(n, dtype=torch.float32, device=dev)
        S = [t.contiguous() for t in mlist]
        seq_dev = [torch.from_numpy(c).to(dev) for c in codes] if canonical else None
        maps_arr = (C.c_void_p * n)(*[t.data_ptr() for t in S])
        pairs_arr = (C.c_void_p * n)(*[p.data_ptr() for p in pairs])
        seq_arr = (C.c_void_p * n)(*[c.data_ptr() for c in seq_dev]) if canonical else None
        L.check(L.lib.rnamsm_fold(n, maps_arr, Larr, seq_arr, MODES[mode], gamma, threshold, int(min_loop),
                                  int(canonical), pairs_arr, L.ptr(scores), L.ptr(ws), nbytes, L.stream_ptr()), "fold")
        flag = ws[:4].view(torch.int32).to(torch.float32)
        *score_list, status = torch.cat([scores, flag]).tolist()       # the one host sync
    if int(status) & 1:
        raise ValueError("fold_pairs: a map has a non-finite value in its upper triangle")
    if int(status) & 2:
        raise ValueError(f"fold_pairs: a pair weight 2 gamma S or an unpaired weight 1 - sum S overflows float32 "
                         f"(gamma {gamma})")
    return (pairs[0], score_list[0]) if single else (pairs, score_list)


def _host_pairs(pairs) -> np.ndarray:
    p = pairs.cpu().numpy() if isinstance(pairs, torch.Tensor) else np.asarray(pairs)
    p = p.astype(np.int64).reshape(-1)
    n = p.shape[0]
    for i, k in enumerate(p):
        if k != -1 and not (0 <= k < n and k != i and p[k] == i):
            raise ValueError(f"pairs[{i}] = {k} is not a partner index (-1 for unpaired, symmetric)")
    return p


def dot_bracket(pairs) -> str:
    """'(' and ')' for the pairs of a nested structure, '.' for unpaired positions."""
    p = _host_pairs(pairs)
    out = ["."] * p.shape[0]
    for i, k in enumerate(p):
        if k > i:
            out[i], out[k] = "(", ")"
    return "".join(out)


def _check_seq(seq: str, p: np.ndarray) -> None:
    if len(seq) != p.shape[0]:
        raise ValueError(f"sequence of {len(seq)} letters for {p.shape[0]} positions")


def write_ct(path: str, name: str, seq: str, pairs) -> None:
    """Connectivity table: a header ``L name``, then per position: index, base, index - 1, index + 1 (0 past the end),
    partner, index; indices 1-based, partner 0 when unpaired."""
    p = _host_pairs(pairs)
    _check_seq(seq, p)
    n = p.shape[0]
    with open(path, "w") as f:
        f.write(f"{n}\t{name}\n")
        for i in range(n):
            f.write(f"{i + 1}\t{seq[i]}\t{i}\t{i + 2 if i + 1 < n else 0}\t{p[i] + 1}\t{i + 1}\n")


def write_bpseq(path: str, seq: str, pairs) -> None:
    """BPSEQ: per position the 1-based index, the base and the 1-based partner (0 when unpaired)."""
    p = _host_pairs(pairs)
    _check_seq(seq, p)
    with open(path, "w") as f:
        for i in range(p.shape[0]):
            f.write(f"{i + 1} {seq[i]} {p[i] + 1}\n")
