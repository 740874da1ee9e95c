"""Cases, float64 references and derived gates for the one-warp-per-row kernels (CPU helpers, device-agnostic).

Kernels covered: the embedding + LayerNorm (rnamsm_embed_layernorm, K1), the LayerNorm (rnamsm_layernorm, K2 / K9, and
rnamsm_add_layernorm), the tied vocabulary projection (rnamsm_vocab_proj, K9b), the contact head (rnamsm_contact_head)
and the 16-bit range scan (rnamsm_range_scan).  The references are torch float64 and run on whatever device their
inputs live on; the emulation of warp_layernorm is numpy float32.

LayerNorm row regimes (fp32 rows; what each is meant to provoke):
    randn          N(0, 1): the rows of the existing tests.
    offset         mean 1e4, spread 1 (|mu| / sigma = 1e4): a one-pass variance E[x^2] - mu^2 cancels catastrophically.
    outlier        N(0, 1) plus +-1e3 on features 0, 127, 128 and D - 1 (lane and vector boundaries): a trained residual
                   stream's outlier channels; |z| up to ~30 exercises the |z|-proportional part of the gate.
    constant_grid  one value k / 8 per row: every fp32 sum is exact, var = 0 and the output is exactly b.
    constant_any   one arbitrary value per row: var is the rounding residue of the mean; the output is b within the gate.
    zero           all zero: var = 0, output exactly b.
    near_eps       0.5 + 1e-3 N(0, 1): var ~ 1e-6 next to eps = 1e-5.
The eighth regime, `saturating`, is a property of the affine weight (|w| ~ 3e4, so fp16 outputs pass 65504) rather
than of the rows: SATURATING_W builds that weight.

The LayerNorm gate (ln_reference).  warp_layernorm (csrc/common.cuh) holds a row as nv = D / 128 float4 per lane and
computes, in fp32:
    S    = butterfly-sum over lanes of  sum_i ((x0 + x1) + (x2 + x3))      every input passes <= nv + 7 additions
    mu_f = S / D                                                           one more rounding
    d_k  = x_k - mu_f                                                      one rounding
    Q    = butterfly-sum of  sum_i ((d0 d0 + d1 d1) + (d2 d2 + d3 d3))     fma / mul / add: <= nv + 8 roundings
    rstd = rsqrtf(Q / D + eps)                                             2 roundings, then rsqrtf: <= 2 ulp = 4u
    y_k  = fma(d_k * rstd, w_k, b_k)                                       2 roundings
with u = 2^-24 and g(n) = n u / (1 - n u) (Higham's gamma).  Against float64 mu, sigma = sqrt(var + eps) and
z_k = (x_k - mu) / sigma of the same fp32 inputs:
    |mu_f - mu|  <= dmu = g(nv + 8) mean|x|                      (summation + division)
    r = dmu / sigma
    sum d_k^2 = (sum (x_k - mu)^2 + D (mu_f - mu)^2) (1 + 2u): the mean's error enters the variance squared, so
    rel. error of Q / D + eps  <= g(nv + 12) + r^2,  and of rstd  <= eps_r = (g(nv + 12) + r^2) / 2 + 4u
    |d_k rstd - z_k|  <= t_k = (r + |z_k| (eps_r + 2u)) (1 + 4u)
    |y_f - y|  <= g32_k = |w_k| t_k + u (|y_k| + |w_k| t_k)          (the fma's rounding)
A 16-bit output adds its own rounding of y_f: half an ulp, <= (|y| + g32) 2^-(p + 1) with p = 10 (fp16) or 7 (bf16),
and at least the fp16 subnormal half-step 2^-25.  fp16 outputs saturate (cvt.rn.satfinite), so the fp16 reference is
clamp(y, +-65504): clamping is 1-Lipschitz and the bound carries over.  The gate is proportional to |mu| / sigma
through r and to |w| |z|, so it is tight on randn rows and loose exactly where the arithmetic is.

A one-pass variance (E[x^2] - mu^2) has error ~ (nv + 8) u E[x^2] instead, ~ (mu / sigma)^2 times the bound above:
emulate_layernorm(..., one_pass=True) shows the gate rejects it on `offset` rows.  (On `outlier` rows the mean is
small next to the spread, so a one-pass variance stays inside the gate there too; those rows have teeth against wrong
lane or vector indexing instead.)

Exact-operand builders: embedding tables on a 2^-10 grid (token + position + row scalar is exact in fp32, so K1's
LayerNorm input equals the float64 sum) and vocabulary-projection operands h = a / 16, E = b / 64 (|a| <= 16,
|b| <= 64), whose products lie on the 2^-10 grid: a 1024-term dot product stays below 2^10, so every partial sum and
the bias add are exact in fp32 in any order, and the kernel's output must equal float64 bit for bit.
"""
from __future__ import annotations

import math

import numpy as np
import torch

U = 2.0 ** -24
LN_EPS = 1e-5
EPS32 = float(np.float32(LN_EPS))              # the eps the kernels add: rnamsm_layernorm takes it as a float
F16_MAX = 65504.0
OUT_BITS = {1: 7, 2: 10}                       # explicit mantissa bits of bf16 / fp16
ROW_REGIMES = ["randn", "offset", "outlier", "constant_grid", "constant_any", "zero", "near_eps"]
EXACT_B_REGIMES = ("constant_grid", "zero")
SATURATING_W = 3e4


def gamma(n: float) -> float:
    return n * U / (1.0 - n * U)


def outlier_features(D: int):
    return sorted({0, 127, min(128, D - 1), D - 1})


# ------------------------------------------------------------------------------------------ LayerNorm inputs
def ln_rows(regime: str, n: int, D: int, seed: int) -> np.ndarray:
    """n fp32 rows of one regime."""
    g = np.random.default_rng([seed, D, n, ROW_REGIMES.index(regime)])
    if regime == "randn":
        x = g.standard_normal((n, D))
    elif regime == "offset":
        x = 1e4 + g.standard_normal((n, D))
    elif regime == "outlier":
        x = g.standard_normal((n, D))
        f = outlier_features(D)
        x[:, f] = 1e3 * np.where(g.random((n, len(f))) < 0.5, -1.0, 1.0)
    elif regime == "constant_grid":
        x = np.repeat(g.integers(-64, 65, size=(n, 1)) / 8.0, D, axis=1)
    elif regime == "constant_any":
        x = np.repeat(0.3 + g.standard_normal((n, 1)), D, axis=1)
    elif regime == "zero":
        x = np.zeros((n, D))
    elif regime == "near_eps":
        x = 0.5 + 1e-3 * g.standard_normal((n, D))
    else:
        raise ValueError(regime)
    return x.astype(np.float32)


def ln_mixed_rows(n: int, D: int, seed: int, rotate: int = 0):
    """n rows, row r in regime ROW_REGIMES[(r + rotate) % 7]: every regime on every lane of a block and every grid
    position.  Returns the fp32 rows and the regime index of each row."""
    reg = (np.arange(n) + rotate) % len(ROW_REGIMES)
    x = np.empty((n, D), dtype=np.float32)
    for k, name in enumerate(ROW_REGIMES):
        idx = np.nonzero(reg == k)[0]
        if idx.size:
            x[idx] = ln_rows(name, idx.size, D, seed)
    return x, reg


def ln_affine(D: int, seed: int, saturating: bool = False):
    """fp32 w, b.  b on a coarse grid is not needed: exactness of b comes from the kernel's fma(0, w, b)."""
    g = np.random.default_rng([seed, D, 99])
    w = 1.0 + 0.1 * g.standard_normal(D)
    if saturating:
        w = SATURATING_W * w * np.where(g.random(D) < 0.5, -1.0, 1.0)
    b = 0.1 * g.standard_normal(D)
    return w.astype(np.float32), b.astype(np.float32)


# ------------------------------------------------------------------------------------------ LayerNorm reference + gate
def ln_reference(x: torch.Tensor, w: torch.Tensor, b: torch.Tensor, out_code: int, eps: float = EPS32):
    """float64 LayerNorm of the fp32 values in x ([N, D], any float dtype; w, b [D]) and the per-element gate of the
    module docstring for output type out_code (0 fp32, 1 bf16, 2 fp16).  Returns (ref, gate): ref is clamped to
    +-65504 for fp16."""
    x = x.double()
    w = w.double()
    b = b.double()
    D = x.shape[-1]
    nv = D // 128
    mu = x.mean(-1, keepdim=True)
    xc = x - mu
    var = (xc * xc).mean(-1, keepdim=True)
    sigma = torch.sqrt(var + eps)
    z = xc / sigma
    y = z * w + b
    r = gamma(nv + 8) * x.abs().mean(-1, keepdim=True) / sigma
    eps_r = 0.5 * (gamma(nv + 12) + r * r) + 4 * U
    t = (r + z.abs() * (eps_r + 2 * U)) * (1 + 4 * U)
    g32 = w.abs() * t
    g32 = g32 + U * (y.abs() + g32)
    if out_code == 0:
        return y, g32
    p = OUT_BITS[out_code]
    gate = g32 + (y.abs() + g32) * 2.0 ** -(p + 1)
    if out_code == 2:
        gate = gate + 2.0 ** -25
        y = y.clamp(-F16_MAX, F16_MAX)
    return y, gate


def ln_expected_b(b: torch.Tensor, out_code: int) -> torch.Tensor:
    """What a var = 0 row must be: b, rounded once to the output type."""
    return b.float().to({0: torch.float32, 1: torch.bfloat16, 2: torch.float16}[out_code])


# ------------------------------------------------------------------------------------------ warp_layernorm in fp32
def _fma32(a, b, c):
    """fp32 fma: the product is exact in float64, the add rounds once there and once more to fp32 (a double rounding
    that can differ from a true fma by one ulp in rare ties; the emulation is only held against the gate)."""
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)


def _butterfly(v):
    """warp_sum: v[lane] += v[lane ^ o] for o = 16 .. 1 (every lane ends with the same value; lane 0 is returned)."""
    lanes = np.arange(32)
    for o in (16, 8, 4, 2, 1):
        v = (v + v[:, lanes ^ o]).astype(np.float32)
    return v[:, 0]


def _rsqrt32(a, ulps: int):
    with np.errstate(invalid="ignore"):         # a one-pass variance can go negative: NaN, as rsqrtf gives
        r = (1.0 / np.sqrt(a.astype(np.float64))).astype(np.float32)
    step = np.float32(np.inf) if ulps > 0 else np.float32(0)
    for _ in range(abs(ulps)):
        r = np.nextafter(r, step)
    return r


def emulate_layernorm(x: np.ndarray, w: np.ndarray, b: np.ndarray, eps: float = EPS32, rsqrt_ulps: int = 0,
                      one_pass: bool = False) -> np.ndarray:
    """warp_layernorm in its own operation order, fp32 throughout; rsqrtf modelled as the correctly rounded value
    moved by rsqrt_ulps ulp (rsqrtf's documented bound is 2).  one_pass=True: the mutant E[x^2] - mu^2."""
    x = np.asarray(x, dtype=np.float32)
    n, D = x.shape
    nv = D // 128
    f32 = np.float32
    v = x.reshape(n, nv, 32, 4)                                  # feature i * 128 + lane * 4 + c
    s = np.zeros((n, 32), dtype=f32)
    for i in range(nv):
        t = (v[:, i, :, 0] + v[:, i, :, 1]) + (v[:, i, :, 2] + v[:, i, :, 3])
        s = (s + t).astype(f32)
    mean = (_butterfly(s) / f32(D)).astype(f32)[:, None, None, None]
    dv = v if one_pass else (v - mean).astype(f32)
    q = np.zeros((n, 32), dtype=f32)
    for i in range(nv):
        d = dv[:, i]
        p01 = _fma32(d[..., 0], d[..., 0], (d[..., 1] * d[..., 1]).astype(f32))
        p23 = _fma32(d[..., 2], d[..., 2], (d[..., 3] * d[..., 3]).astype(f32))
        q = (q + (p01 + p23).astype(f32)).astype(f32)
    var = (_butterfly(q) / f32(D)).astype(f32)
    if one_pass:
        m = mean[:, 0, 0, 0]
        var = (var - (m * m).astype(f32)).astype(f32)
        dv = (v - mean).astype(f32)
    rstd = _rsqrt32((var + f32(eps)).astype(f32), rsqrt_ulps)[:, None, None, None]
    t = (dv * rstd).astype(f32)
    y = _fma32(t, w.astype(f32).reshape(1, nv, 32, 4), b.astype(f32).reshape(1, nv, 32, 4))
    return y.reshape(n, D)


def round_out(y32: torch.Tensor, out_code: int) -> torch.Tensor:
    """The kernels' 16-bit stores: round to nearest even; fp16 saturates at +-65504 (cvt.rn.satfinite)."""
    if out_code == 0:
        return y32.float()
    if out_code == 2:
        return y32.float().clamp(-F16_MAX, F16_MAX).to(torch.float16)
    return y32.float().to(torch.bfloat16)


def gate_ratio(got: torch.Tensor, ref: torch.Tensor, gate: torch.Tensor) -> float:
    """max |got - ref| / gate (NaN anywhere in got counts as infinitely far)."""
    d = (got.double() - ref).abs()
    if bool(torch.isnan(d).any()):
        return math.inf
    return float((d / gate).max())


# ------------------------------------------------------------------------------------------ embedding (K1)
def embed_tables(vocab: int, n_pos: int, R: int, D: int, seed: int, pad_idx: int):
    """fp32 tables on a 2^-10 grid: token [-1, 1] step 2^-6, position [-1/4, 1/4] step 2^-8, row scalar
    [-1/16, 1/16] step 2^-10.  Any sum of one of each is exact in fp32.  The pad row of the token table is zero, as
    nn.Embedding(padding_idx) keeps it."""
    g = np.random.default_rng([seed, vocab, n_pos, R, D])
    tok = (g.integers(-64, 65, size=(vocab, D)) / 64.0).astype(np.float32)
    tok[pad_idx] = 0.0
    pos = (g.integers(-64, 65, size=(n_pos, D)) / 256.0).astype(np.float32)
    row = (g.integers(-64, 65, size=R) / 1024.0).astype(np.float32)
    return tok, pos, row


def positions(tokens: torch.Tensor, pad_idx: int) -> torch.Tensor:
    """LearnedPositionalEmbedding's index rule (modules.py:286-291), per row: cumsum(tok != pad) * (tok != pad) + pad."""
    keep = tokens.ne(pad_idx).long()
    return torch.cumsum(keep, dim=-1) * keep + pad_idx


def embed_input(tokens: torch.Tensor, tok_emb: torch.Tensor, pos_emb: torch.Tensor, row_pos, pad_idx: int):
    """float64 [R, C, D] LayerNorm input of K1: E_tok[tok] + E_pos[pos] + p_row[r] (row_pos None: no row term)."""
    x = tok_emb.double()[tokens] + pos_emb.double()[positions(tokens, pad_idx)]
    if row_pos is not None:
        x = x + row_pos.double()[: tokens.shape[0], None, None]
    return x


def embed_reference(tokens, tok_emb, pos_emb, row_pos, ln_w, ln_b, pad_idx: int, eps: float = EPS32):
    """float64 K1: (x [R, C, D] with pad tokens zeroed, gate, pad mask [R, C])."""
    R, C = tokens.shape
    x = embed_input(tokens, tok_emb, pos_emb, row_pos, pad_idx)
    y, gate = ln_reference(x.reshape(R * C, -1), ln_w, ln_b, 0, eps)
    pad = tokens.eq(pad_idx)
    y = y.view(R, C, -1).masked_fill(pad[..., None], 0.0)
    return y, gate.view(R, C, -1), pad


def embed_tokens(R: int, C: int, vocab: int, pad_idx: int, seed: int, mid_pads=(31, 32, 63, 64, 127)):
    """int64 [R, C]: column 0 BOS (token 0), the rest uniform over every non-pad token 0 .. vocab - 1.
    Row 0 has no pad (its last position is C + pad_idx, the largest of the grid); row 1 has pads at the mid_pads
    columns below C with real tokens after each; row 2 (R > 2) is BOS and pads only; rows 3.. get random pads."""
    g = np.random.default_rng([seed, R, C])
    choices = np.array([t for t in range(vocab) if t != pad_idx])
    t = choices[g.integers(0, len(choices), size=(R, C))]
    t[:, 0] = 0
    t[0, :] = np.where(np.arange(C) == 0, 0, t[0, :])
    if C > 1:
        t[0, -1] = vocab - 1
    if R > 1:
        for c in mid_pads:
            if c < C - 1:
                t[1, c] = pad_idx
    if R > 2:
        t[2, 1:] = pad_idx
    if R > 3:
        t[3:][g.random((R - 3, C)) < 0.2] = pad_idx
        t[3:, 0] = 0
    return torch.from_numpy(t.astype(np.int64))


# ------------------------------------------------------------------------------------------ vocabulary projection
def vocab_exact_operands(M: int, V: int, D: int, seed: int):
    """h [M, D], E [V, D], bias [V] fp32 on which every dot product is exact in fp32 (module docstring)."""
    g = np.random.default_rng([seed, M, V, D])
    h = (g.integers(-16, 17, size=(M, D)) / 16.0).astype(np.float32)
    E = (g.integers(-64, 65, size=(V, D)) / 64.0).astype(np.float32)
    bias = (g.integers(-1024, 1025, size=V) / 1024.0).astype(np.float32)
    return h, E, bias


def vocab_reference(h: torch.Tensor, E: torch.Tensor, bias: torch.Tensor):
    """float64 logits and the fp32 dot-product gate: each lane accumulates its 4 nv products in order, the warp adds 32
    lane sums in a 5-level butterfly and the bias is added once, so every product passes <= 4 nv + 6 roundings:
    |out_f - out| <= g(4 nv + 6) (sum |h_k E_k| + |bias|)."""
    D = h.shape[-1]
    h64, E64, b64 = h.double(), E.double(), bias.double()
    ref = h64 @ E64.T + b64
    gate = gamma(4 * (D // 128) + 6) * (h64.abs() @ E64.abs().T + b64.abs())
    return ref, gate


# ------------------------------------------------------------------------------------------ contact head
CONTACT_MAPS = ["softmax", "onehot", "column", "asymmetric", "sink", "all_bos"]


def contact_maps(kind: str, K: int, C: int, seed: int) -> np.ndarray:
    """fp32 [K, C, C] non-negative attention-like maps, rows summing to ~1 over all C keys (column 0 = BOS).
        softmax     rand().softmax(-1): what the existing tests use; row and column sums nearly constant.
        onehot      each query attends one key: row sums 1, column sums 0 .. many.
        column      most of every row on 3 shared keys: column sums concentrated, a1 far from constant.
        asymmetric  strictly lower-triangular mass: A and A^T disjoint.
        sink        99.9 % on the BOS column: the stripped block carries 1e-3 of the mass, a12 tiny.
        all_bos     every row entirely on BOS: the stripped block (start = 1) is zero and a12 = 0, so the reference
                    itself is 0 / 0 = NaN (with start = 0 the BOS column is in the block and nothing is NaN)."""
    g = np.random.default_rng([seed, K, C, CONTACT_MAPS.index(kind)])
    if kind == "softmax":
        a = g.random((K, C, C))
        a = np.exp(a) / np.exp(a).sum(-1, keepdims=True)
    elif kind == "onehot":
        a = np.zeros((K, C, C))
        j = g.integers(0, C, size=(K, C))
        np.put_along_axis(a, j[..., None], 1.0, axis=-1)
    elif kind == "column":
        a = 0.05 * g.random((K, C, C)) / C
        cols = g.integers(0, C, size=(K, 3))
        for k in range(K):
            a[k][:, cols[k]] += np.array([0.6, 0.25, 0.1])
        a = a / a.sum(-1, keepdims=True)
    elif kind == "asymmetric":
        a = np.tril(g.random((K, C, C)) + 0.01, -1)
        a[:, 0, 0] = 1.0
        a = a / a.sum(-1, keepdims=True)
    elif kind == "sink":
        a = g.random((K, C, C))
        a = 1e-3 * a / a.sum(-1, keepdims=True)
        a[:, :, 0] += 0.999
    elif kind == "all_bos":
        a = np.zeros((K, C, C))
        a[:, :, 0] = 1.0
    else:
        raise ValueError(kind)
    return a.astype(np.float32)


def contact_reference(maps: torch.Tensor, start: int, L: int, w: torch.Tensor, bias: torch.Tensor):
    """float64 contact head over the block [start, start + L)^2 of maps [K, C, C], written from the reference's
    formula (symmetrize, APC, logistic regression; NaN where it is NaN).  Returns (out, logit, logit_gate) with the
    gate of the fp32 kernel (csrc/contact.cu) on the logit, for non-negative maps:
      margins: a1_i = row sum + column sum of S = A + A^T takes <= L / 8 + 10 roundings (column sums run over L / 8
      rows per thread and 8 partials; row sums over L / 32 per lane and a 5-level butterfly); a12 adds <= L / 32 + 6,
      so both are within eta = g(L / 8 + 16) relative (all terms non-negative).  The APC term p = a1_i a1_j / a12 is
      within 3 eta + 3u, S_ij within u, S - p within u |S - p|, and the K-term fma chain adds g(K + 1) sum |w apc|:
        |logit_f - logit| <= sum_k |w_k| (u S + (3 eta + 3u) p + u |S - p|) + g(K + 1) (sum_k |w_k apc_k| + |b|)."""
    K = maps.shape[0]
    A = maps.double()[:, start:start + L, start:start + L]
    S = A + A.transpose(-1, -2)
    a1 = S.sum(-1)
    a12 = a1.sum(-1)
    p = a1[:, :, None] * a1[:, None, :] / a12[:, None, None]
    apc = S - p
    w64 = w.double().reshape(K, 1, 1)
    b64 = bias.double().reshape(())
    logit = (w64 * apc).sum(0) + b64
    eta = gamma(L / 8 + 16)
    gate = (w64.abs() * (U * S + (3 * eta + 3 * U) * p + U * apc.abs())).sum(0) \
        + gamma(K + 1) * ((w64 * apc).abs().sum(0) + b64.abs())
    return torch.sigmoid(logit), logit, gate


def contact_out_gate(logit: torch.Tensor, logit_gate: torch.Tensor) -> torch.Tensor:
    """Gate on the sigmoid output 1 / (1 + __expf(-l)): the logit's error times the sigmoid's largest slope within
    that error of l, plus __expf's documented 2 + floor(1.173 |l|) ulp (relative 2^-23 each) on e^-l, which moves the
    output by sigma (1 - sigma) times that, plus two fp32 roundings (add, divide).  Below a logit of about -83 the
    output nears fp32's subnormal range, where e^-l overflows or the result flushes: there it may be anything in
    [0, sigmoid(l + gate)]."""
    s = torch.sigmoid(logit)
    near = torch.sign(logit) * (logit.abs() - logit_gate).clamp(min=0)
    sn = torch.sigmoid(near)
    e_exp = (2 + 1.173 * (logit.abs() + logit_gate)) * 2.0 ** -23
    hi = logit + logit_gate
    tiny = torch.where(hi < -83, torch.sigmoid(hi), torch.zeros_like(hi))
    return sn * (1 - sn) * (logit_gate + e_exp) + 2 * U * s + tiny + 2.0 ** -149


def contact_logit_gate(out: torch.Tensor, logit: torch.Tensor, logit_gate: torch.Tensor) -> torch.Tensor:
    """Gate on the logit recovered from the kernel's output, log(o) - log(1 - o): the logit's own error, __expf's
    relative error, and the output's two roundings seen through d logit / d o = 1 / (o (1 - o)), i.e. 2u / (1 - o)."""
    o = out.double()
    e_exp = (2 + 1.173 * (logit.abs() + logit_gate)) * 2.0 ** -23
    return logit_gate + e_exp + 2 * U / (1 - o)


def logit_of(out: torch.Tensor) -> torch.Tensor:
    o = out.double()
    return torch.log(o) - torch.log1p(-o)


# ------------------------------------------------------------------------------------------ range scan
F16_EDGE, BF16_EDGE = 0x7BFF, 0x7F7F           # largest finite magnitude of each type: at or above it is "edge"


def range_patterns(code: int) -> np.ndarray:
    """uint16 bit patterns every buffer mixes in: the largest finite value, the one below it, inf, NaN, of both signs;
    the smallest and largest subnormals; +-0; 1.0."""
    if code == 2:
        mags = [0x7BFF, 0x7BFE, 0x7C00, 0x7E00, 0x7C01, 0x7FFF, 0x0001, 0x03FF, 0x0000, 0x3C00]
    else:
        mags = [0x7F7F, 0x7F7E, 0x7F80, 0x7FC0, 0x7F81, 0x7FFF, 0x0001, 0x007F, 0x0000, 0x3F80]
    m = np.array(mags, dtype=np.uint16)
    return np.concatenate([m, m | np.uint16(0x8000)])


def range_buffer(code: int, n: int, seed: int, patterns: bool = True) -> np.ndarray:
    """uint16 [n]: random finite magnitudes below 1.0 with random signs; patterns=True also places every
    range_patterns word at the start, at the end and at a random position (as far as n allows)."""
    g = np.random.default_rng([seed, code, n])
    one = 0x3C00 if code == 2 else 0x3F80
    buf = g.integers(0, one, size=n).astype(np.uint16) | (g.integers(0, 2, size=n).astype(np.uint16) << 15)
    if n == 0 or not patterns:
        return buf
    for j, p in enumerate(range_patterns(code)):
        for pos in (j, n - 1 - j, int(g.integers(0, n))):
            if 0 <= pos < n:
                buf[pos] = p
    return buf


def range_reference(buf: np.ndarray, code: int):
    """(count of edge elements, fp32 bit pattern of the largest non-edge |v|, 0 when there is none)."""
    a = buf.astype(np.uint32) & 0x7FFF
    edge = a >= (F16_EDGE if code == 2 else BF16_EDGE)
    rest = a[~edge]
    if rest.size == 0:
        return int(edge.sum()), 0
    m = int(rest.max())                         # non-negative floats order as their bit patterns
    if code == 2:
        bits = int(np.array([m], dtype=np.uint16).view(np.float16).astype(np.float32).view(np.uint32)[0])
    else:
        bits = m << 16
    return int(edge.sum()), bits
