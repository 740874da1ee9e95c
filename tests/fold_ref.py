"""float32 numpy restatement of the folding of ``rnamsm_b200.fold_pairs`` (csrc/fold.cu, DESIGN.md section 4.15).

Every table entry is one float32 add of two stored values and ``max`` is exact, so this restatement, which fills one
row ``i`` at a time as a vector-matrix max-plus product over the finished rows below it, gives the same bits as the
tiled device fill.  Also: the float64 score of a given structure and a brute-force maximum over every nested
structure, for small ``L``."""
import numpy as np

CODES = {"A": 0, "G": 1, "C": 2, "U": 3, "X": 4, "N": 5, "-": 6}
_CANON = np.zeros((8, 8), dtype=bool)
for _a, _b in ("AU", "GC", "GU"):
    _CANON[CODES[_a], CODES[_b]] = _CANON[CODES[_b], CODES[_a]] = True


def codes(seq):
    return np.array([CODES[c] for c in seq], dtype=np.uint8)


def allowed(S, seq=None, threshold=0.0, min_loop=3, canonical=None):
    """bool [L, L]: (i, j), i < j, with j - i > min_loop, S[i, j] > fp32(threshold) and, with canonical (default: a
    sequence is given), {s_i, s_j} in {AU, GC, GU}."""
    S = np.asarray(S, dtype=np.float32)
    L = S.shape[0]
    i, j = np.indices((L, L))
    ok = (j - i > min_loop) & (S > np.float32(threshold))
    if canonical is None:
        canonical = seq is not None
    if canonical:
        c = codes(seq)
        ok &= _CANON[c[:, None], c[None, :]]
    return ok


def weights(S, seq=None, mode="mea", gamma=1.0, threshold=0.0, min_loop=3, canonical=None):
    """-> (w float32 [L, L], -inf where not allowed; u float32 [L])."""
    S = np.asarray(S, dtype=np.float32)
    L = S.shape[0]
    up = np.triu(np.ones((L, L), dtype=bool), 1)
    if not np.isfinite(S[up]).all():
        raise ValueError("non-finite value in the upper triangle")
    ok = allowed(S, seq, threshold, min_loop, canonical)
    if mode == "mea":
        w = np.float32(2.0 * gamma) * S
        sym = np.triu(S.astype(np.float64), 1)
        sym = sym + sym.T                                    # exact: one of the two terms is 0
        acc = np.zeros(L, dtype=np.float64)
        for j in range(L):                                   # ascending j, one rounding per add
            acc += sym[:, j]
        u = (1.0 - acc).astype(np.float32)
    elif mode == "score":
        w = S.copy()
        u = np.zeros(L, dtype=np.float32)
    else:
        raise ValueError(mode)
    if not np.isfinite(w[ok]).all():
        raise ValueError("a weight overflows float32")
    return np.where(ok, w, np.float32(-np.inf)).astype(np.float32), u


def fill(w, u):
    """-> (M float32 [L + 1, L + 1] with M[i, j] for i <= j, 0 on the subdiagonal (the empty interval) and -inf below
    it; P float32 [L, L], P[i, k] = w[i, k] + M[i + 1, k - 1])."""
    L = w.shape[0]
    M = np.full((L + 1, L + 1), -np.inf, dtype=np.float32)
    M[np.arange(1, L + 1), np.arange(L)] = 0.0
    P = np.full((L, L), -np.inf, dtype=np.float32)
    for i in range(L - 1, -1, -1):
        P[i, i + 1:] = w[i, i + 1:] + M[i + 1, i:L - 1]
        row = M[i + 1, i:L] + u[i]
        if i + 1 < L:
            pair = (P[i, i + 1:, None] + M[i + 2:L + 1, i:L]).max(axis=0)    # k > j meets -inf below the subdiagonal
            row = np.maximum(row, pair)
        M[i, i:L] = row
    return M, P


def traceback(M, P, u):
    L = P.shape[0]
    pairs = np.full(L, -1, dtype=np.int32)
    stack = [(0, L - 1)]
    while stack:
        i, j = stack.pop()
        while i <= j:
            if M[i, j] == M[i + 1, j] + u[i]:
                i += 1
                continue
            k = i + 1 + int(np.flatnonzero(P[i, i + 1:j + 1] + M[i + 2:j + 2, j] == M[i, j])[0])
            pairs[i], pairs[k] = k, i
            if k + 1 <= j:
                stack.append((k + 1, j))
            i, j = i + 1, k - 1
    return pairs


def fold(S, seq=None, mode="mea", gamma=1.0, threshold=0.0, min_loop=3, canonical=None):
    """-> (pairs int32 [L], score float32)"""
    w, u = weights(S, seq, mode, gamma, threshold, min_loop, canonical)
    M, P = fill(w, u)
    return traceback(M, P, u), M[0, w.shape[0] - 1]


def structure_score(w, u, pairs):
    """float64 sum of w over the pairs and u over the unpaired positions."""
    s = 0.0
    for i, k in enumerate(pairs):
        if k < 0:
            s += float(u[i])
        elif i < k:
            s += float(w[i, k])
    return s


def nested_structures(ok):
    """Every nested structure (a list of pairs) whose pairs are allowed by the bool matrix ok."""
    L = ok.shape[0]
    memo = {}

    def rec(i, j):
        if i > j:
            return [[]]
        if (i, j) in memo:
            return memo[(i, j)]
        out = [s for s in rec(i + 1, j)]
        for k in range(i + 1, j + 1):
            if ok[i, k]:
                for a in rec(i + 1, k - 1):
                    for b in rec(k + 1, j):
                        out.append([(i, k)] + a + b)
        memo[(i, j)] = out
        return out

    return rec(0, L - 1)


def brute_force(w, u):
    """float64 maximum over every nested structure of allowed pairs (finite w)."""
    L = w.shape[0]
    best = -np.inf
    for s in nested_structures(np.isfinite(w)):
        pairs = np.full(L, -1)
        for i, k in s:
            pairs[i], pairs[k] = k, i
        best = max(best, structure_score(w, u, pairs))
    return best
