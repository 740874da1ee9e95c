"""Float64 numpy restatement of the window plan and the stitching of rnamsm_msa_forward_windows (csrc/windows.cu), from
per-window outputs."""
import numpy as np


def window_starts(L, window, stride):
    """-> the residue offsets s_k of the windows, or None for invalid arguments."""
    if L < 1 or not 1 <= stride <= window:
        return None
    W = min(window, L)
    K = 1 + -(-(L - W) // stride)
    return [min(k * stride, L - W) for k in range(K)]


def tent(p, s, W):
    """w_k(p) for residues p (array) of the window starting at s; 0 outside it."""
    p = np.asarray(p)
    inside = (p >= s) & (p < s + W)
    return np.where(inside, np.minimum(p - s + 1, s + W - p), 0).astype(np.int64)


def coefficients(L, W, starts):
    """-> (c1 [K, L], c2 [K, L, L]) float64: the residue and pair coefficients of each window; 0 where the window does
    not hold the residue (pair) or no window does."""
    p = np.arange(L)
    w = np.stack([tent(p, s, W) for s in starts])                       # [K, L] integers
    pair = w[:, :, None] * w[:, None, :]                                  # [K, L, L] integers
    with np.errstate(invalid="ignore", divide="ignore"):
        c1 = w / w.sum(0, keepdims=True)
        den = pair.sum(0, keepdims=True)
        c2 = np.where(den > 0, pair / np.where(den > 0, den, 1), 0.0)
    return c1, c2


def stitch(embs, maps, starts, L, contacts=None):
    """embs [K, W, D], maps [K, NH, W, W] (BOS stripped), contacts [K, W, W] or None -> float64 (emb [L, D],
    atp [NH, L, L], contacts [L, L] or None)."""
    embs = np.asarray(embs, dtype=np.float64)
    maps = np.asarray(maps, dtype=np.float64)
    K, W, D = embs.shape
    NH = maps.shape[1]
    c1, c2 = coefficients(L, W, starts)
    emb = np.zeros((L, D))
    atp = np.zeros((NH, L, L))
    con = np.zeros((L, L)) if contacts is not None else None
    for k, s in enumerate(starts):
        sl = slice(s, s + W)
        emb[sl] += c1[k, sl, None] * embs[k]
        atp[:, sl, sl] += c2[k, sl, sl][None] * maps[k]
        if con is not None:
            con[sl, sl] += c2[k, sl, sl] * np.asarray(contacts[k], dtype=np.float64)
    return emb, atp, con


def covered(L, W, starts):
    """[L, L] bool: the pairs some window holds."""
    m = np.zeros((L, L), dtype=bool)
    for s in starts:
        m[s:s + W, s:s + W] = True
    return m


def single(L, W, starts):
    """[L, L] int: the index of the one window holding each pair, -1 where none or several do."""
    n = np.zeros((L, L), dtype=np.int64)
    idx = np.full((L, L), -1, dtype=np.int64)
    for k, s in enumerate(starts):
        n[s:s + W, s:s + W] += 1
        idx[s:s + W, s:s + W] = k
    return np.where(n == 1, idx, -1)
