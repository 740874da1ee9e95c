"""Softmax edge cases for the attention kernels (CPU helpers, no GPU).

The op-level tests elsewhere feed randn logits: near-uniform rows whose range stays far below the ~88 nats where fp32
exp over- or underflows, so a kernel that subtracts the wrong maximum still gives the right answer there.  The cases
here prescribe the logits instead -- sharp, shifted, staircased and masked rows -- so such a kernel writes inf / NaN.

Logit construction.  For one (column, head) problem of n query rows and n keys, q and k are [n, 64] with the structure
in the first few head dimensions and seeded noise in the rest:
    s_ij = sum_{t < T} A[i, t] B[j, t]  +  sum_{t >= T} qn[i, t] kn[j, t]
A and B hold small integers and short dyadic values; the noise values are multiples of 2^-6 with |x| <= 2^-4.  All of
them are exact in fp16 and bf16, and every product lies on the 2^-12 grid.  A logit of magnitude below 2^12 is then a
sum of terms that are exact in fp32 in any order and any rounding mode (24 bits span 2^-12 .. 2^12): the kernels'
fp32 logits equal the float64 logits of the rounded tensors bit for bit, and a test measures the softmax alone.  (The
one exception is `below_mask`, whose real logits sit near -12288; there the padded keys carry all the weight.)

Regimes, and what each is meant to provoke:
    uniform          k = 0: every unpadded key weighs the same; the answer is the mean of V over them.
    onehot           one key per row above the rest by 104 nats, its position walking across lanes, warps and blocks.
    shifted          every logit near +300 or -300 with a few nats of spread: a wrong max gives inf / NaN or 0 / 0.
    staircase_cross  the max of key block b is ~12 b nats: growth beyond 16 log2 units per block (fp16 P overflows
                     without a rescale), beyond 128 log2 units in total at 1025 keys (bf16 P and the fp32 sum too).
    staircase_under  block maxima 5 - 7.6 log2 units above block 0's: P approaches 2^8 without a lazy rescale.
    mixed            even query rows see a rising staircase, odd rows a falling one: only some lanes of a warp grow.
    masked_prefix    the first 128 or 256 keys padded (half the keys when fewer exist): rescale from m = -10000 log2e.
    fully_masked     every key padded: uniform rows.
    below_mask       real logits near -12288 and some padded keys: the padded keys (-10000) win, which is
                     masked_fill(-10000) semantics, not -inf.

`fa_replay` restates col_attn_fa_kernel's per-row max bookkeeping (csrc/col_attn_fa.cu) so a CPU test can show each
case does in that kernel what its name says.
"""
from __future__ import annotations

import math
import os
import re

import numpy as np

HD = 64
MASK_VALUE = -10000.0
LOG2E = 1.4426950408889634

REGIMES = ["uniform", "onehot", "shifted", "staircase_cross", "staircase_under", "mixed", "masked_prefix",
           "fully_masked", "below_mask"]

_CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "rna-msm_b200", "csrc")


def _fa_constant(pattern: str) -> float:
    with open(os.path.join(_CSRC, "col_attn_fa.cu")) as f:
        m = re.search(pattern, f.read())
    assert m, f"col_attn_fa.cu: {pattern!r} not found"
    return float(m.group(1))


# The fa kernel's lazy-rescale threshold (log2 units) and key-block size, read from its source so the cases follow them.
FA_RESCALE_THRESHOLD = _fa_constant(r"constexpr\s+float\s+kRescaleThreshold\s*=\s*([0-9.eE+-]+)f")
FA_KEY_BLOCK = int(_fa_constant(r"constexpr\s+int\s+NT\s*=\s*\d+\s*,\s*BQ\s*=\s*\d+\s*,\s*BKV\s*=\s*(\d+)"))

# Gate term for large logits.  The kernels get the logits exactly (module docstring), but the 16-bit probability
# kernels round s * log2(e) to fp32 once per key (col_attn_probs.cu), and the row softmax kernels round s * logit_scale
# once per key: an exponent error of up to |s| 2^-24 log2(e) log2 units = |s| 2^-24 nats, i.e. a relative error of
# |s| 2^-24 on that key's probability.  The fp32 constant log2(e) carries its own relative error of up to 2^-24, which
# adds the same bound again.  Normalising by a sum of such probabilities at most doubles it (the sum's error is a
# weighted mean of the keys' errors): c = 2 * (1 + 1) = 4.  Padded keys all carry the same -10000, so their rounding is
# common to them and cancels in the normalisation; |s|max is taken over the real keys.
LARGE_LOGIT_C = 4.0


def large_logit_term(s_absmax: float) -> float:
    return LARGE_LOGIT_C * float(s_absmax) * 2.0 ** -24


def key_block(R: int) -> int:
    """Key-block size of the 16-bit column kernel that runs at depth R: col_attn_fa (128) above 128 rows,
    col_attn_umma (64) up to 128.  The fp32 kernels (simt_f32.cu, col_attn_probs.cu) use 64."""
    return FA_KEY_BLOCK if R > 128 else 64


def _noise(rng, shape):
    return rng.integers(-4, 5, size=shape).astype(np.float64) / 64.0


def _spread(n_rows, n_keys, variant):
    """A few nats of exact structure: a in 1..4, b in [-1, 1] on the 1/8 grid."""
    a = (np.arange(n_rows) % 4 + 1).astype(np.float64)
    b = (((np.arange(n_keys) * 5 + variant) % 17) - 8) / 8.0
    return a, b


def _stairs(n, blk, step, variant):
    """Block b's keys at step * b minus 0 .. 3.5 nats (zero at every 8th key from the block start, so a block of one
    key still reaches its step)."""
    j = np.arange(n)
    return step * (j // blk) - 0.5 * (((j % blk) * 3) % 8)


def pattern(regime: str, n: int, variant: int = 0, blk: int = 128):
    """Structure of one (column, head) problem with n queries and n keys.
    -> A [n, T], B [n, T] (float64, exact in fp16 / bf16), keypad [n] bool, k_noise (False: k is zero outside B)."""
    j = np.arange(n)
    i = np.arange(n)
    keypad = np.zeros(n, dtype=bool)
    k_noise = True
    if regime == "uniform":
        A, B = np.zeros((n, 0)), np.zeros((n, 0))
        keypad = (j % 5) == 3
        k_noise = False
    elif regime == "onehot":
        G = min(48, n)                                             # rows i = g mod G share hot key hot[g]
        hot = (np.arange(G) * 97 + 13 + 29 * variant) % n          # 97 = 3 * 32 + 1: lanes, warps and blocks all walk
        A = (i[:, None] % G == np.arange(G)[None, :]).astype(np.float64)
        B = np.where(j[:, None] == hot[None, :], 104.0, 0.0)
    elif regime == "shifted":
        sign = 1.0 if variant % 2 == 0 else -1.0
        a, b = _spread(n, n, variant)
        A = np.stack([np.ones(n), a], 1)
        B = np.stack([np.full(n, 300.0 * sign), b], 1)
        keypad = (j % 13) == 7
    elif regime == "staircase_cross":
        A = np.ones((n, 1))
        B = _stairs(n, blk, 12.0 + 0.5 * (variant % 3), variant)[:, None]
    elif regime == "staircase_under":
        # block 1 at 5.25 nats = 7.57 log2 units above block 0, later blocks 5.05 .. 7.21 log2 units above it
        lift = np.array([3.5, 4.0, 4.5, 5.0])
        b_idx = j // blk
        g = np.where(b_idx == 0, 0.0, np.where(b_idx == 1, 5.25, lift[(b_idx + variant) % 4]))
        A = np.ones((n, 1))
        B = (g - 0.5 * (((j % blk) * 3) % 8))[:, None]
    elif regime == "mixed":
        nb = (n + blk - 1) // blk
        rise = _stairs(n, blk, 12.0, variant)
        fall = 12.0 * (nb - 1 - j // blk) - 0.5 * (((j % blk) * 3) % 8)
        A = np.stack([(i % 2 == 0), (i % 2 == 1)], 1).astype(np.float64)
        B = np.stack([rise, fall], 1)
    elif regime == "masked_prefix":
        want = 128 if variant % 2 == 0 else 256
        prefix = want if want < n else (128 if 128 < n else max(n // 2, 1) if n > 1 else 0)
        a, b = _spread(n, n, variant)
        A, B = a[:, None], b[:, None]
        keypad = j < prefix
    elif regime == "fully_masked":
        a, b = _spread(n, n, variant)
        A, B = a[:, None] * 8.0, b[:, None]                        # a +-32 nat spread that the mask must hide
        keypad = np.ones(n, dtype=bool)
    elif regime == "below_mask":
        a, b = _spread(n, n, variant)
        A = np.stack([np.ones(n), a], 1)
        B = np.stack([np.full(n, -12288.0), b], 1)
        keypad = ((j % 5) == 2) | (j == n - 1)
    else:
        raise ValueError(regime)
    return A.astype(np.float64), B.astype(np.float64), keypad, k_noise


def head_qk(regime: str, n: int, variant: int, seed: int, blk: int = 128):
    """q, k [n, 64] float64 (exact in fp16 and bf16) and keypad [n] of one (column, head) problem."""
    A, B, keypad, k_noise = pattern(regime, n, variant, blk)
    T = A.shape[1]
    rng = np.random.default_rng([seed, variant, n])
    q = _noise(rng, (n, HD))
    k = _noise(rng, (n, HD)) if k_noise else np.zeros((n, HD))
    q[:, :T] = A
    k[:, :T] = B
    return q, k, keypad


def col_case(regimes, R: int, C: int, H: int, seed: int, blk: int | None = None):
    """Column-attention inputs: q|k|v float64 [R, C, 3 H 64] (q|k exact in 16 bits; v is seeded randn, rounded by the
    caller) and pad uint8 [R, C].  regimes: one name for every column, or a list with one name per column.  Column c,
    head h is variant c * H + h, so hot positions, signs and prefixes differ between problems."""
    if isinstance(regimes, str):
        regimes = [regimes] * C
    blk = key_block(R) if blk is None else blk
    D = H * HD
    qkv = np.zeros((R, C, 3 * D))
    pad = np.zeros((R, C), dtype=np.uint8)
    for c in range(C):
        for h in range(H):
            q, k, keypad = head_qk(regimes[c], R, c * H + h, seed, blk)
            qkv[:, c, h * HD:(h + 1) * HD] = q
            qkv[:, c, D + h * HD:D + (h + 1) * HD] = k
            if h == 0:
                pad[:, c] = keypad
    rng = np.random.default_rng([seed, R, C, 7])
    qkv[:, :, 2 * D:] = rng.standard_normal((R, C, D))
    return qkv, pad


def row_logits(regime: str, C: int, H: int, seed: int, blk: int = 128):
    """Row-attention logits [H, C, C] float64 (head h = variant h; exact in fp32 except `below_mask`) and the key
    mask [C] (variant 0's: one mask serves every head, as in the row block)."""
    out = np.empty((H, C, C))
    keypad = None
    for h in range(H):
        q, k, kp = head_qk(regime, C, h, seed, blk)
        out[h] = q @ k.T
        if h == 0:
            keypad = kp
    return out, keypad


def split_partials(logits: np.ndarray, n_splits: int, seed: int) -> np.ndarray:
    """[n_splits, *logits.shape] float32 whose split-order fp32 sum is exactly float32(logits) where logits are exact
    in fp32 and below 2^11: all splits but the last are multiples of 1/8 in [-4, 4], the last is the remainder."""
    rng = np.random.default_rng([seed, n_splits])
    parts = np.empty((n_splits,) + logits.shape, dtype=np.float32)
    acc = np.zeros(logits.shape)
    for s in range(n_splits - 1):
        parts[s] = rng.integers(-32, 33, size=logits.shape) / 8.0
        acc += parts[s]
    parts[-1] = (logits - acc).astype(np.float32)
    return parts


def masked_logits(s: np.ndarray, keypad: np.ndarray) -> np.ndarray:
    """masked_fill(-10000) along the last (key) axis."""
    return np.where(keypad, MASK_VALUE, s)


def fa_replay(s: np.ndarray, threshold: float = FA_RESCALE_THRESHOLD, blk: int = FA_KEY_BLOCK):
    """col_attn_fa_kernel's max bookkeeping for one problem.  s: [n_queries, n_keys] logits after masking, as the
    kernel holds them in fp32.  Per query row and key block b: mx = (block max) * log2e; grow = mx > m_ref + threshold
    (always on block 0, where m_ref = -inf); on grow m_ref = mx.  A warp of 32 query rows rescales O at block b > 0 when
    any of its rows grows there.  The P written for a key is 2^(s log2e - m_ref).
    -> dict(grow [n, nblk] bool, warp_rescale [n_warps, nblk] bool, growth_log2 (largest mx - m_ref before the update,
    over rows and blocks b > 0; -inf with one block), max_p_log2 (largest log2 P after the update))."""
    s32 = s.astype(np.float32)
    n, nk = s32.shape
    nblk = (nk + blk - 1) // blk
    l2e = np.float32(LOG2E)
    m_ref = np.full(n, -np.inf, dtype=np.float32)
    grow = np.zeros((n, nblk), dtype=bool)
    growth = -np.inf
    max_p = -np.inf
    with np.errstate(invalid="ignore"):
        for b in range(nblk):
            mx = s32[:, b * blk:(b + 1) * blk].max(1) * l2e
            g = mx > m_ref + np.float32(threshold)
            if b > 0:
                growth = max(growth, float((mx - m_ref).max()))
            grow[:, b] = g
            m_ref = np.where(g, mx, m_ref)
            max_p = max(max_p, float((mx - m_ref).max()))
    n_warps = (n + 31) // 32
    warp_rescale = np.zeros((n_warps, nblk), dtype=bool)
    for w in range(n_warps):
        warp_rescale[w] = grow[w * 32:(w + 1) * 32].any(0)
    warp_rescale[:, 0] = False                                     # block 0 sets the reference; nothing to rescale
    return dict(grow=grow, warp_rescale=warp_rescale, growth_log2=growth, max_p_log2=max_p)


def exact_in(x: np.ndarray, dtype: str) -> bool:
    """Is every value of x exactly representable in fp16 / bf16 / fp32?"""
    import torch
    t = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64))
    tdt = {"fp16": torch.float16, "bf16": torch.bfloat16, "fp32": torch.float32}[dtype]
    return bool(torch.equal(t.to(tdt).double(), t))


def real_absmax(s: np.ndarray, keypad: np.ndarray) -> float:
    """max |s| over unpadded keys (0 when every key is padded)."""
    real = np.broadcast_to(~keypad, s.shape)
    return float(np.abs(s[real]).max()) if real.any() else 0.0


def fa_depth_shape(n_sms: int = 148):
    """R, C, H of a column-attention case whose fa work items (C H ceil(R / 256)) exceed four per SM: a CTA then carries
    items of different regimes, and their rescales, through the deferred read-out of the item before."""
    R, H = 257, 2
    C = 4 * n_sms // (H * math.ceil(R / 256)) + 12
    return R, C, H
