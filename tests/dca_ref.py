"""Float64 numpy restatement of the alignment statistics of csrc/coevolution.cu (rnamsm_b200.coevolution): sequence
weights, Neff and mean-field DCA contacts (Morcos et al., PNAS 2011), from their definitions."""
import numpy as np

Q = 5


def states(tokens) -> np.ndarray:
    """int64 [N, C] (or [1, N, C]) tokens, column 0 BOS -> int [N, L] states: A G C U (4 .. 7) -> 0 .. 3, else 4."""
    t = np.asarray(tokens)
    if t.ndim == 3:
        t = t[0]
    r = t[:, 1:]
    return np.where((r >= 4) & (r <= 7), r - 4, 4).astype(np.int64)


def one_hot(s: np.ndarray) -> np.ndarray:
    """[N, L] states -> float64 [N, L * Q]"""
    N, L = s.shape
    X = np.zeros((N, L, Q))
    X[np.arange(N)[:, None], np.arange(L)[None, :], s] = 1.0
    return X.reshape(N, L * Q)


def weights(tokens, theta: float = 0.8):
    """-> (float64 [N] weights, Neff): row k is a neighbour of n iff (double) m(n, k) >= theta * (double) L, with
    m(n, k) the number of columns of equal states, exact integers from one-hot products in row blocks."""
    s = states(tokens)
    N, L = s.shape
    X = one_hot(s)
    count = np.zeros(N, dtype=np.int64)
    thr = theta * float(L)
    for a in range(0, N, 2048):
        m = np.rint(X[a:a + 2048] @ X.T)
        count[a:a + 2048] = (m >= thr).sum(1)
    w = 1.0 / count.astype(np.float64)
    return w, float(w.sum())


def covariance(tokens, theta: float = 0.8, lam: float = 0.5):
    """-> (Cov float64 [4L, 4L], w, Neff): f_i, f_ij with pseudocount lam; Cov[(i, a), (j, b)] = f_ij(a, b) - f_i(a)
    f_j(b) for a, b < 4, f_ii(a, b) = f_i(a) d_ab."""
    s = states(tokens)
    N, L = s.shape
    w, neff = weights(tokens, theta)
    X = one_hot(s)
    fi = (1 - lam) / neff * (w @ X) + lam / Q                                  # [L * Q]
    fij = (1 - lam) / neff * ((X * w[:, None]).T @ X) + lam / Q ** 2           # [L * Q, L * Q]
    fi2, fij4 = fi.reshape(L, Q), fij.reshape(L, Q, L, Q)
    for i in range(L):
        fij4[i, :, i, :] = np.diag(fi2[i])
    C = fij4 - fi2[:, :, None, None] * fi2[None, None, :, :]
    return C[:, :4, :, :4].reshape(4 * L, 4 * L), w, neff


def apc(F: np.ndarray) -> np.ndarray:
    total = F.sum()
    if total == 0:
        return F.copy()
    return F - F.sum(-1, keepdims=True) * F.sum(-2, keepdims=True) / total


def scores(e: np.ndarray, L: int) -> np.ndarray:
    """e [4L, 4L] -> float64 [L, L]: Frobenius norms of the zero-sum-gauge 5 x 5 blocks (zero gap row and column),
    zero diagonal; APC with the diagonal zeroed again; (F + F^T) / 2."""
    E = np.zeros((L, Q, L, Q))
    E[:, :4, :, :4] = e.reshape(L, 4, L, 4)
    E = E - E.mean(axis=3, keepdims=True) - E.mean(axis=1, keepdims=True) + E.mean(axis=(1, 3), keepdims=True)
    F = np.sqrt((E ** 2).sum(axis=(1, 3)))
    np.fill_diagonal(F, 0.0)
    F = apc(F)
    np.fill_diagonal(F, 0.0)
    return (F + F.T) / 2


def dca(tokens, theta: float = 0.8, lam: float = 0.5):
    """-> {"contacts": float64 [L, L], "weights", "neff", "cov"}"""
    C, w, neff = covariance(tokens, theta, lam)
    L = C.shape[0] // 4
    e = -np.linalg.inv(C)
    return {"contacts": scores(e, L), "weights": w, "neff": neff, "cov": C}


def planted_alignment(N: int, L: int, i: int, j: int, seed: int, gap_p: float = 0.0) -> np.ndarray:
    """int64 tokens [N, L + 1] with BOS: random residues, except columns i < j (1-based residue indices) which hold a
    Watson-Crick pair (AU, UA, GC, CG) in every row."""
    rng = np.random.default_rng(seed)
    t = np.empty((N, L + 1), dtype=np.int64)
    t[:, 0] = 0
    t[:, 1:] = rng.integers(4, 8, size=(N, L))
    if gap_p:
        t[:, 1:][rng.random((N, L)) < gap_p] = 10                             # '-'
    A, G, Cc, U = 4, 5, 6, 7
    pairs = np.array([(A, U), (U, A), (G, Cc), (Cc, G)])
    k = rng.integers(0, 4, size=N)
    t[:, i] = pairs[k, 0]
    t[:, j] = pairs[k, 1]
    return t
