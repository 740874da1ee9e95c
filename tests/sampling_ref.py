"""CPU restatement of iterative masked sampling (``MSATransformer.sample_msa``, csrc/sample.cu): Philox4x32-10, the
mask draw and the float64 inverse-CDF sampler, vectorised with numpy."""
import numpy as np

M0, M1 = 0xD2511F53, 0xCD9E8D57
W0, W1 = 0x9E3779B9, 0xBB67AE85
U32 = np.uint64(0xFFFFFFFF)
MASK, DRAW = 0, 1
BOUNDARY = 1e-5


def philox4x32_10(ctr, key):
    """ctr: four uint32 arrays (broadcastable), key: two -> the four output words (uint64 arrays holding uint32)."""
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) for c in ctr)
    k0, k1 = (np.asarray(k, dtype=np.uint64) for k in key)
    for _ in range(10):
        p0, p1 = np.uint64(M0) * c0, np.uint64(M1) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & U32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & U32
        k0, k1 = (k0 + np.uint64(W0)) & U32, (k1 + np.uint64(W1)) & U32
    return c0, c1, c2, c3


def uniform(seed, k, s, t, purpose):
    """u(seed, chain k, step s, token t = r * C + c, purpose) = (word0 >> 8) * 2^-24, float64 (exact in fp32)."""
    w0 = philox4x32_10((k, s, t, purpose), (seed & 0xFFFFFFFF, seed >> 32))[0]
    return (w0 >> np.uint64(8)).astype(np.float64) * 2.0 ** -24


def mask_set(state, rows, pad_idx, mask_prob, seed, k, s):
    """bool [R, C]: the tokens of chain k's state [R, C] masked at step s."""
    R, C = state.shape
    t = np.arange(R * C, dtype=np.uint64).reshape(R, C)
    elig = np.zeros((R, C), dtype=bool)
    elig[sorted(rows), 1:] = True
    elig &= state != pad_idx
    return elig & (uniform(seed, k, s, t, MASK) < np.float32(mask_prob))


def draw(logits, allowed, temperature, u):
    """One masked token: logits [V] (fp32), allowed: ascending vocabulary indices -> (token, near) where ``near`` says
    u lies within BOUNDARY of an inner CDF boundary (where fp32 and float64 may pick neighbours)."""
    z = np.asarray(logits, dtype=np.float64)[allowed]
    if temperature == 0:
        return allowed[int(np.argmax(z))], False
    w = np.exp((z - z.max()) / np.float64(np.float32(temperature)))
    cdf = np.cumsum(w) / w.sum()
    i = min(int(np.searchsorted(cdf, u, side="right")), len(allowed) - 1)
    return allowed[i], bool((np.abs(cdf[:-1] - u) < BOUNDARY).any())


def step(state, logits, rows, pad_idx, allowed, mask_prob, temperature, seed, k, s):
    """One step of chain k from ``state`` [R, C] with the logits [R, C, V] of its masked grid -> (new state, masked,
    near) where ``near`` [R, C] marks draws within BOUNDARY of a CDF boundary."""
    m = mask_set(state, rows, pad_idx, mask_prob, seed, k, s)
    new, near = state.copy(), np.zeros(state.shape, dtype=bool)
    C = state.shape[1]
    for r, c in zip(*np.nonzero(m)):
        u = float(uniform(seed, k, s, np.uint64(r * C + c), DRAW))
        new[r, c], near[r, c] = draw(logits[r, c], allowed, temperature, u)
    return new, m, near
