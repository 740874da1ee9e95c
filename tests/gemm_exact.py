"""Exact operands and float64 references for the tensor-core GEMM (csrc/umma_gemm.cu) and its FFMA and one-launch
siblings (csrc/simt_f32.cu, phase 1 of csrc/row_attn_short.cu).

Exactness.  Every operand is a small integer on a power-of-two grid: x = i / 8 and W = j / 64 with integers |i|, |j| <= 8,
so every product is a multiple of 2^-9 of magnitude <= 1/8 (64 grid steps).  Bias and the residual stream are multiples of
2^-9 with magnitude <= 4.  Every partial sum, in any order, is then a multiple of 2^-9; while its magnitude stays below
2^24 grid steps it is exact in fp32 (24-bit significand), so the tensor core's truncating fp32 accumulator, the FFMA
kernel and float64 all give the same number.  Each case's worst-case sum is bounded by `*_bound_steps` below.  A 16-bit
output is then float64_ref.to(dtype): the fp32 value is exact and the kernel rounds it once (cvt.rn).

The tied row-attention operands follow the same rule with q = i / 8, k = j / 64 (different grids, so a kernel that mixed
q and k up would not get the same sums) and v = i / 8; the A V probabilities are P = j / 64.

The erf-GELU epilogues are not exact (A&S 7.1.28 polynomial and rcp.approx in the 16-bit path, erff in the fp32 path).
They are checked on the exact pre-activation a with |y - gelu64(a)| <= ulp_out(|gelu64(a)|) + 2^-20 |a|.

The module also holds the ABI-level runners the GPU tests share, and runs as a script in a child process with a
different environment (RNAMSM_GEMM_PAIRS, RNAMSM_GELU_WIDE, RNAMSM_AV_WIDE, RNAMSM_PDL are read once per process):

    python tests/gemm_exact.py OUT.pt

runs `child_cases`, checks the exact ones against float64, and saves every output for the parent to compare bit for bit.
"""
from __future__ import annotations

import math
import os
import sys

import numpy as np
import torch

# ------------------------------------------------------------------------------------------ exact operands
CTX_DEN, W_DEN, GRID = 8, 64, 2.0 ** -9
AFFINE_MAX = 4.0
PROD_STEPS = 8 * 8                       # |i j| / 512 <= 64 / 512: 64 grid steps per product
AFFINE_STEPS = int(AFFINE_MAX / GRID)    # 2048 grid steps per bias / residual term
Q_SCALE = 3.0 / 8.0                      # exact, and it moves the grid to 2^-12 (3 times the steps)
FP32_STEPS = 2 ** 24


def _rng(seed):
    return seed if isinstance(seed, np.random.Generator) else np.random.default_rng(seed)


def _ints(rng, shape, lim=8):
    return torch.from_numpy(rng.integers(-lim, lim + 1, size=shape, dtype=np.int8))


def exact_affine(shape, rng_or_seed, device="cpu") -> torch.Tensor:
    """float32 multiples of 2^-9 with magnitude <= 4 (bias, the residual stream)."""
    rng = _rng(rng_or_seed)
    return torch.from_numpy(rng.integers(-AFFINE_STEPS, AFFINE_STEPS + 1, size=shape, dtype=np.int32)).to(device).float() * GRID


def exact_gemm_operands(M: int, N: int, K: int, seed: int, device="cpu"):
    """x [M, K] = i / 8, W [N, K] = j / 64, bias [N] as float32 tensors on `device` (exact in fp16, bf16 and tf32)."""
    rng = np.random.default_rng([seed, M, N, K])
    x = _ints(rng, (M, K)).to(device).float() / CTX_DEN
    W = _ints(rng, (N, K)).to(device).float() / W_DEN
    bias = exact_affine((N,), rng, device)
    return x, W, bias


def exact_qkv(R: int, C: int, H: int, seed: int, device="cpu") -> torch.Tensor:
    """q|k|v [R, C, 3 H 64] float32, token-major: q = i / 8, k = j / 64, v = i / 8."""
    rng = np.random.default_rng([seed, R, C, H])
    D = H * 64
    t = _ints(rng, (R, C, 3 * D)).to(device).float()
    t[..., :D] /= CTX_DEN
    t[..., D:2 * D] /= W_DEN
    t[..., 2 * D:] /= CTX_DEN
    return t


def exact_probs(H: int, C: int, ldp: int, seed: int, device="cpu") -> torch.Tensor:
    """P [H, C, ldp] float32 = j / 64 in columns [0, C) and NaN in the padding columns [C, ldp)."""
    rng = np.random.default_rng([seed, H, C, ldp])
    P = torch.full((H, C, ldp), float("nan"), device=device)
    P[..., :C] = _ints(rng, (H, C, C)).to(device).float() / W_DEN
    return P


def exact_sum_bound_ulps(K: int) -> int:
    """Largest |x + sum_k ctx_k W_k + b| of the dense operands, in 2^-9 grid steps (residual epilogue)."""
    return dense_bound_steps(K, 2)


def dense_bound_steps(K: int, epi: int) -> int:
    """Worst |output| of the dense GEMM in steps of its output grid: 2^-9, or 2^-12 after the q scale (epilogue 0)."""
    pre = K * PROD_STEPS + AFFINE_STEPS                   # sum_k x W + b
    if epi == 0:
        return 3 * pre                                    # (3 / 8) a = 3 a / 2^3: three times the steps of 2^-12
    if epi == 2:
        return pre + AFFINE_STEPS                         # + the residual stream
    return pre                                            # GELU: the pre-activation is what must be exact


def tied_bound_steps(R: int) -> int:
    """Worst |sum_{r, d} q k| over all R rows (every split is a subset of them)."""
    return R * 64 * PROD_STEPS


def av_bound_steps(C: int) -> int:
    return C * PROD_STEPS


def exact_in_tf32(t: torch.Tensor) -> bool:
    """Does t equal its tf32 part (low 13 mantissa bits zero), i.e. is the lo half of the split 0?"""
    b = t.float().contiguous().view(torch.int32)
    return bool((b & 0x1FFF).eq(0).all())


# ------------------------------------------------------------------------------------------ float64 references
def dense_preact(x, W, bias):
    return x.double() @ W.double().T + bias.double()


def dense_ref(x, W, bias, epi, q_scale=1.0, q_cols=0, row_mask=None, resid=None):
    """float64 out of rnamsm_linear: epilogue 0 with q scale and row mask on columns [0, q_cols), 1 GELU, 2 residual."""
    a = dense_preact(x, W, bias)
    if epi == 0:
        if q_cols:
            a[:, :q_cols] *= q_scale
            if row_mask is not None:
                a[row_mask.to(a.device).bool(), :q_cols] = 0.0
        return a
    if epi == 1:
        return gelu64(a)
    return resid.double() + a


def gelu64(a: torch.Tensor) -> torch.Tensor:
    """nn.GELU() (erf form) in float64."""
    a = a.double()
    return 0.5 * a * (1.0 + torch.special.erf(a / math.sqrt(2.0)))


MANT = {0: 23, 1: 7, 2: 10}          # fp32, bf16, fp16
EMIN = {0: -126, 1: -126, 2: -14}


def ulp(x: torch.Tensor, code: int) -> torch.Tensor:
    """Spacing of the output type (0 fp32, 1 bf16, 2 fp16) at |x| >= 0, subnormal range included (float64)."""
    x = x.double().abs()
    _, e = torch.frexp(x)                                  # x = m 2^e, m in [0.5, 1)
    e = torch.where(x > 0, e - 1, torch.full_like(e, EMIN[code]))
    e = torch.clamp(e, min=EMIN[code])
    return torch.pow(2.0, (e - MANT[code]).double())


def gelu_gate(a: torch.Tensor, code: int) -> torch.Tensor:
    """Allowed |y - gelu64(a)|: one output ulp plus 2^-20 |a| (the A&S error and the cancellation in
    x + |x| (1 - erfc) for negative a)."""
    return ulp(gelu64(a), code) + 2.0 ** -20 * a.double().abs()


def gelu_excess(y: torch.Tensor, a: torch.Tensor, code: int) -> float:
    """max |y - gelu64(a)| / gelu_gate(a): <= 1 passes; NaN when y holds a NaN."""
    err = (y.double() - gelu64(a)).abs() / gelu_gate(a, code)
    if torch.isnan(err).any():
        return float("nan")
    return float(err.max()) if err.numel() else 0.0


def split_rows(R: int, n_splits: int):
    """Row ranges of the tied logits' splits (and of row_attn_short's chunks): [s rps, min(R, (s + 1) rps))."""
    rps = -(-R // n_splits)
    return [(s * rps, min(R, (s + 1) * rps)) for s in range(n_splits)]


def valid_splits(R: int, n_splits: int) -> bool:
    """The ABI rejects a split count that leaves an empty split."""
    return 1 <= n_splits <= R and (n_splits - 1) * -(-R // n_splits) < R


def tied_split_refs(qkv: torch.Tensor, R: int, C: int, H: int, n_splits: int) -> torch.Tensor:
    """float64 [n_splits, H, C, C]: slab s = sum over rows r of split s of q[r, i, h, :] . k[r, j, h, :]."""
    D = H * 64
    q = qkv.view(R, C, 3 * D)[..., :D].double().view(R, C, H, 64)
    k = qkv.view(R, C, 3 * D)[..., D:2 * D].double().view(R, C, H, 64)
    out = torch.empty(n_splits, H, C, C, dtype=torch.float64, device=qkv.device)
    for s, (r0, r1) in enumerate(split_rows(R, n_splits)):
        out[s] = torch.einsum("rihd,rjhd->hij", q[r0:r1], k[r0:r1])
    return out


def av_ref(P: torch.Tensor, qkv: torch.Tensor, R: int, C: int, H: int) -> torch.Tensor:
    """float64 ctx [R C, H 64]: ctx[r, i, h, :] = sum_{j < C} P[h, i, j] v[r, j, h, :] (padding columns not read)."""
    D = H * 64
    v = qkv.view(R, C, 3 * D)[..., 2 * D:].double().view(R, C, H, 64)
    return torch.einsum("hij,rjhd->rihd", P[..., :C].double(), v).reshape(R * C, D)


# ------------------------------------------------------------------------------------------ persistent tile schedule
PAIR_M, BLOCK_N = 256, 256


def tied_tile_n(C: int) -> int:
    """kBN of the tied-logit instance (umma_gemm.cu tied_tile_n)."""
    return 64 if C <= 64 else (128 if C <= 128 else BLOCK_N)


def dense_tiles(M: int, N: int) -> int:
    return -(-M // PAIR_M) * -(-N // BLOCK_N)


def tied_tiles(C: int, H: int, n_splits: int) -> int:
    return H * -(-C // PAIR_M) * -(-C // tied_tile_n(C)) * n_splits


def av_tiles(R: int, C: int, H: int) -> int:
    return H * -(-C // PAIR_M) * -(-R // 4)


def tiles_per_pair(total: int, P: int):
    """Tiles each launched pair runs: the launch has min(total, P) pairs, and pair p walks tile = p + lt n_pairs while
    that is below total (umma_gemm.cu tile_at)."""
    n_pairs = min(total, P)
    counts = []
    for pair in range(n_pairs):
        lt = 0
        while pair + lt * n_pairs < total:
            lt += 1
        counts.append(lt)
    return counts


# Production (N, K) of each epilogue, first choice first: q|k|v, out_proj / LM dense; fc1, LM dense; fc2, out_proj.  The
# last entry (one n-tile) always has a solution for the exact tile counts.
PRODUCTION_NK = {0: [(2304, 768), (768, 768), (192, 768)],
                 1: [(3072, 768), (768, 768), (192, 768)],
                 2: [(768, 3072), (768, 768), (192, 768)]}
WAVE_TARGETS = ["Pw-1", "Pw+1", "3P+"]


def multiwave_case(P: int, epi: int, target: str):
    """(M, N, K, tiles, w) whose dense tile count is P w - 1 (w >= 2: the last wave leaves one pair idle), P w + 1 (one
    pair runs a tile more than the others) or >= 3 P (every pair loops at least three times, both accumulator buffers
    twice).  M leaves a tail in the last m-tile: 1 row, none, 179 rows."""
    for N, K in PRODUCTION_NK[epi]:
        nt = -(-N // BLOCK_N)
        if target == "3P+":
            m_tiles = -(-3 * P // nt) + 1
            return m_tiles * PAIR_M - 77, N, K, m_tiles * nt, None
        for w in range(2 if target == "Pw-1" else 1, 2 + nt):
            tiles = P * w - 1 if target == "Pw-1" else P * w + 1
            if tiles % nt == 0 and tiles // nt >= 1:
                m_tiles = tiles // nt
                return m_tiles * PAIR_M - (255 if target == "Pw-1" else 0), N, K, tiles, w
    raise AssertionError("unreachable: the one-n-tile shape always has a solution")


def check_wave_counts(counts, target: str, w, P: int):
    """The schedule the multi-wave case was built for."""
    total = sum(counts)
    assert len(counts) == min(total, P)
    if target == "Pw-1":
        assert total == P * w - 1 and max(counts) == w and counts.count(w - 1) == 1, counts
    elif target == "Pw+1":
        assert total == P * w + 1 and max(counts) == w + 1 and counts.count(w + 1) == 1, counts
    else:
        assert total >= 3 * P and min(counts) >= 3, counts


# ------------------------------------------------------------------------------------------ case lists
LINEAR_MS = [1, 31, 32, 33, 127, 128, 129, 255, 256, 257, 513]
LINEAR_NS = [64, 192, 320, 768, 832, 2304, 3072]
LINEAR_KS = [64, 128, 384, 448, 768, 3072]
CODES = [0, 1, 2]
EPIS = [0, 1, 2]


def q_cols_for(i: int, N: int) -> int:
    """q_cols in {0, 64, 768, N}, cycling with the case index (768 only where N allows it)."""
    q = [0, 64, 768, N][i % 4]
    return q if q <= N else N


def linear_cases():
    """Every value of each axis for every dtype x epilogue: M walks LINEAR_MS; N and K cycle with different strides."""
    cases = []
    for code in CODES:
        for epi in EPIS:
            for i, M in enumerate(LINEAR_MS):
                N = LINEAR_NS[(3 * i + epi) % len(LINEAR_NS)]
                K = LINEAR_KS[(i + code + epi) % len(LINEAR_KS)]
                q_cols = q_cols_for(i, N) if epi == 0 else 0
                cases.append(dict(M=M, N=N, K=K, code=code, epi=epi, q_cols=q_cols))
    return cases


# (C, H, R): every C of the three kBN instances and their m- and n-tile tails, H in {1, 12}, R in {1, 2, 7, 64, 513}
TIED_CASES = [(1, 12, 7), (63, 1, 513), (64, 12, 64), (65, 1, 2), (127, 12, 1), (128, 12, 64), (128, 1, 513),
              (129, 12, 7), (255, 1, 64), (256, 12, 2), (257, 1, 513), (513, 12, 2), (1024, 1, 7), (100, 12, 1)]
AV_RS = [1, 2, 3, 4, 5, 7, 64]
AV_CS = [1, 8, 63, 64, 65, 129, 256, 257, 513, 1024]
LDP_PADS = [0, 8, 64]


def roundup8(c: int) -> int:
    return (c + 7) // 8 * 8


def av_cases():
    cases = []
    for ci, C in enumerate(AV_CS):
        for li, pad in enumerate(LDP_PADS):
            R = AV_RS[(3 * ci + li) % len(AV_RS)]
            H = 12 if C <= 65 else 2
            cases.append(dict(R=R, C=C, H=H, ldp=roundup8(C) + pad))
    return cases


# (C, H, R) of row_attn_short's phase 1
SHORT_CASES = [(1, 12, 7), (31, 1, 130), (64, 12, 64), (65, 1, 9), (127, 12, 5), (128, 1, 64), (128, 12, 12)]


def short_chunk_options(R: int, H: int, default: int, n_sms: int):
    return sorted({n for n in (1, default, 5, R) if valid_splits(R, n) and H * n <= n_sms})


def cases_bounds_ok(P_values=range(1, 149)) -> bool:
    """Every case the GPU file lists stays below 2^24 grid steps (for every pair count P the device may report)."""
    ok = all(dense_bound_steps(c["K"], c["epi"]) < FP32_STEPS for c in linear_cases())
    for P in P_values:
        for epi in EPIS:
            for t in WAVE_TARGETS:
                ok &= dense_bound_steps(multiwave_case(P, epi, t)[2], epi) < FP32_STEPS
    ok &= all(tied_bound_steps(R) < FP32_STEPS for _, _, R in TIED_CASES + SHORT_CASES)
    ok &= all(av_bound_steps(c["C"]) < FP32_STEPS for c in av_cases())
    for c in child_linear_cases():
        ok &= dense_bound_steps(c["K"], c["epi"]) < FP32_STEPS
    return ok


# ------------------------------------------------------------------------------------------ ABI runners (GPU)
def torch_dtype(code: int) -> torch.dtype:
    return {0: torch.float32, 1: torch.bfloat16, 2: torch.float16}[code]


def bits(t: torch.Tensor) -> torch.Tensor:
    return t.contiguous().view({2: torch.int16, 4: torch.int32}[t.element_size()])


def same_bits(a: torch.Tensor, b: torch.Tensor) -> bool:
    return a.dtype == b.dtype and a.shape == b.shape and torch.equal(bits(a), bits(b))


class Guarded:
    """A flat NaN-filled buffer: `guard` elements, the body of `shape`, `guard` elements.  Kernels get the body's
    address; `intact()` says whether both guards still hold the NaN they were filled with."""

    def __init__(self, shape, dtype, guard, init=None):
        n = math.prod(shape)
        self.g = max(128, -(-guard // 128) * 128)          # keeps the body 256 B aligned for TMA
        self.buf = torch.full((n + 2 * self.g,), float("nan"), dtype=dtype, device="cuda")
        self.body = self.buf[self.g:self.g + n].view(shape)
        if init is not None:
            self.body.copy_(init)

    def intact(self) -> bool:
        nan = torch.full((self.g,), float("nan"), dtype=self.buf.dtype, device=self.buf.device)
        return same_bits(self.buf[:self.g], nan) and same_bits(self.buf[-self.g:], nan)


def run_linear(L, x, W, bias, code, epi, q_scale=1.0, q_cols=0, row_mask=None, resid=None, tf32=False, stream=None):
    """One rnamsm_linear (or rnamsm_linear_tf32) call on float32 operands (cast to the dtype) -> Guarded output."""
    M, K = x.shape
    N = W.shape[0]
    dt = torch.float32 if tf32 else torch_dtype(code)
    xd, Wd = x.to(dt).contiguous(), W.to(dt).contiguous()
    st = L.stream_ptr() if stream is None else stream
    out = Guarded((M, N), torch.float32 if (epi == 2 or tf32) else dt, 16 * N, init=resid if epi == 2 else None)
    if tf32:
        nb = L.lib.rnamsm_linear_tf32_scratch_bytes(M, N, K)
        scratch = torch.empty(nb, dtype=torch.uint8, device="cuda")
        L.check(L.lib.rnamsm_linear_tf32(L.ptr(xd), L.ptr(Wd), L.ptr(bias), M, N, K, epi, q_scale, q_cols, L.ptr(row_mask),
                                         L.ptr(out.body), L.ptr(scratch), nb, st), "linear_tf32")
        out.keep = (xd, Wd, scratch)
    else:
        L.check(L.lib.rnamsm_linear(L.ptr(xd), L.ptr(Wd), L.ptr(bias), M, N, K, code, epi, q_scale, q_cols, L.ptr(row_mask),
                                    L.ptr(out.body), st), "linear")
        out.keep = (xd, Wd)                                 # alive until the stream has run
    return out


def run_logits(L, qkv, R, C, H, code, n_splits, stream=None):
    q = qkv.to(torch_dtype(code)).contiguous()
    out = Guarded((n_splits, H, C, C), torch.float32, H * C * C)
    L.check(L.lib.rnamsm_row_attn_logits(L.ptr(q), R, C, H, code, L.ptr(out.body), n_splits,
                                         L.stream_ptr() if stream is None else stream), "row_attn_logits")
    out.keep = (q,)
    return out


def run_av(L, P, ldp, qkv, R, C, H, code, stream=None):
    dt = torch_dtype(code)
    Pd, q = P.to(dt).contiguous(), qkv.to(dt).contiguous()
    out = Guarded((R * C, H * 64), dt, 16 * H * 64)
    L.check(L.lib.rnamsm_row_attn_av(L.ptr(Pd), ldp, L.ptr(q), R, C, H, code, L.ptr(out.body),
                                     L.stream_ptr() if stream is None else stream), "row_attn_av")
    out.keep = (Pd, q)
    return out


def run_short(L, qkv, R, C, H, code, n_chunks):
    """rnamsm_row_attn_short -> the Guarded phase-1 partials (its softmax and context are not exact and not returned)."""
    dt = torch_dtype(code)
    q = qkv.to(dt).contiguous()
    ldp = roundup8(C)
    part = Guarded((n_chunks, H, C, C), torch.float32, H * C * C)
    pmap = torch.empty(H, C, C, device="cuda")
    plp = torch.empty(H, C, ldp, dtype=dt, device="cuda")
    ctx = torch.empty(R * C, H * 64, dtype=dt, device="cuda")
    L.check(L.lib.rnamsm_row_attn_short(L.ptr(q), R, C, H, code, None, 1.0, L.ptr(part.body), n_chunks, L.ptr(pmap),
                                        L.ptr(plp), ldp, L.ptr(ctx), L.stream_ptr()), "row_attn_short")
    part.keep = (q, pmap, plp, ctx)
    return part


def row_mask_for(M: int, seed: int, device="cuda") -> torch.Tensor:
    """About a fifth of the rows, always the first and the last."""
    m = (np.random.default_rng([seed, M]).random(M) < 0.2).astype(np.uint8)
    m[0] = m[-1] = 1
    return torch.from_numpy(m).to(device)


# ------------------------------------------------------------------------------------------ child-process cases
def child_linear_cases():
    """Multi-wave at 1 and 3 pairs, every epilogue (GELU on the 8-warp instance with RNAMSM_GELU_WIDE=0)."""
    return [dict(M=1000, N=2304, K=768, epi=0, q_cols=768), dict(M=700, N=3072, K=768, epi=1, q_cols=0),
            dict(M=600, N=768, K=3072, epi=2, q_cols=0)]


CHILD_TIED = [(64, 12, 64, 2), (128, 12, 64, 3), (257, 2, 7, 7)]        # (C, H, R, n_splits): the three kBN instances
CHILD_AV = [(7, 257, 2, 264), (64, 64, 12, 128)]                          # (R, C, H, ldp)
CHILD_SHORT = (65, 12, 64, 5)                                             # (C, H, R, n_chunks)


def child_cases(L):
    """Runs the reduced case list on the current device -> {name: output tensor (cpu)}; asserts that every exact case
    equals float64.  Split and chunk counts are explicit: the defaults depend on the pair count."""
    outs = {}
    for code in (1, 2):
        dt = torch_dtype(code)
        for c in child_linear_cases():
            x, W, bias = exact_gemm_operands(c["M"], c["N"], c["K"], seed=61, device="cuda")
            mask = row_mask_for(c["M"], 62) if c["q_cols"] else None
            resid = exact_affine((c["M"], c["N"]), 63, device="cuda") if c["epi"] == 2 else None
            out = run_linear(L, x, W, bias, code, c["epi"], Q_SCALE, c["q_cols"], mask, resid)
            torch.cuda.synchronize()
            assert out.intact(), f"linear {c}: write outside the output"
            if c["epi"] == 1:
                assert gelu_excess(out.body, dense_preact(x, W, bias), code) <= 1.0, f"linear {c}"
            else:
                want = dense_ref(x, W, bias, c["epi"], Q_SCALE, c["q_cols"], mask, resid).to(out.body.dtype)
                assert torch.equal(out.body, want), f"linear {c}"
            outs[f"linear_{code}_{c['epi']}"] = out.body.cpu()
        for C, H, R, ns in CHILD_TIED:
            qkv = exact_qkv(R, C, H, seed=64, device="cuda")
            out = run_logits(L, qkv, R, C, H, code, ns)
            torch.cuda.synchronize()
            assert out.intact() and torch.equal(out.body.double(), tied_split_refs(qkv, R, C, H, ns)), f"logits {C} {H} {R} {ns}"
            outs[f"logits_{code}_{C}_{H}_{R}_{ns}"] = out.body.cpu()
        for R, C, H, ldp in CHILD_AV:
            qkv = exact_qkv(R, C, H, seed=65, device="cuda")
            P = exact_probs(H, C, ldp, seed=66, device="cuda")
            out = run_av(L, P, ldp, qkv, R, C, H, code)
            torch.cuda.synchronize()
            assert out.intact() and torch.equal(out.body, av_ref(P, qkv, R, C, H).to(dt)), f"av {R} {C} {H} {ldp}"
            outs[f"av_{code}_{R}_{C}_{H}"] = out.body.cpu()
        C, H, R, nc = CHILD_SHORT
        qkv = exact_qkv(R, C, H, seed=67, device="cuda")
        out = run_short(L, qkv, R, C, H, code, nc)
        torch.cuda.synchronize()
        assert out.intact() and torch.equal(out.body.double(), tied_split_refs(qkv, R, C, H, nc)), "short"
        outs[f"short_{code}"] = out.body.cpu()
    outs.update(chains(L))
    return outs


def chains(L, code=2):
    """Dependent launches on one stream with no synchronisation between them; only the first GEMM of each branch has
    exact inputs.  FFN: x -> fc1 + GELU -> fc2 residual.  Row attention: x -> q|k|v -> tied logits -> softmax -> A V."""
    dt = torch_dtype(code)
    st = L.stream_ptr()
    M, D, F = 600, 768, 3072
    x, W1, b1 = exact_gemm_operands(M, F, D, seed=71, device="cuda")
    _, W2, b2 = exact_gemm_operands(1, D, F, seed=72, device="cuda")
    resid = exact_affine((M, D), 73, device="cuda")
    h = run_linear(L, x, W1, b1, code, 1, stream=st)
    y = run_linear(L, h.body, W2, b2, code, 2, resid=resid, stream=st)

    R, C, H = 16, 100, 12
    D = H * 64
    xa, Wq, bq = exact_gemm_operands(R * C, 3 * D, D, seed=74, device="cuda")
    mask = row_mask_for(R * C, 75)
    qkv = run_linear(L, xa, Wq, bq, code, 0, 0.125, D, mask, stream=st)
    ns = 3
    part = Guarded((ns, H, C, C), torch.float32, H * C * C)
    L.check(L.lib.rnamsm_row_attn_logits(L.ptr(qkv.body), R, C, H, code, L.ptr(part.body), ns, st), "row_attn_logits")
    ldp = roundup8(C)
    key_pad = torch.zeros(C, dtype=torch.uint8, device="cuda")
    key_pad[-3:] = 1
    pmap = torch.full((H, C, C), float("nan"), device="cuda")
    plp = torch.full((H, C, ldp), float("nan"), dtype=dt, device="cuda")
    L.check(L.lib.rnamsm_row_softmax(L.ptr(part.body), ns, H, C, L.ptr(key_pad), 1.0 / math.sqrt(R), L.ptr(pmap), L.ptr(plp),
                                     ldp, code, st), "row_softmax")
    ctx = Guarded((R * C, D), dt, 16 * D)
    L.check(L.lib.rnamsm_row_attn_av(L.ptr(plp), ldp, L.ptr(qkv.body), R, C, H, code, L.ptr(ctx.body), st), "row_attn_av")
    torch.cuda.synchronize()
    for g in (h, y, qkv, part, ctx):
        assert g.intact(), "chain: write outside an output"
    for t in (h.body, y.body, qkv.body, part.body, pmap, plp, ctx.body):
        assert torch.isfinite(t.float()).all(), "chain: non-finite output"
    want_qkv = dense_ref(xa, Wq, bq, 0, 0.125, D, mask).to(dt)
    assert torch.equal(qkv.body, want_qkv), "chain: q|k|v (exact inputs)"
    return {"chain_fc1": h.body.cpu(), "chain_fc2": y.body.cpu(), "chain_qkv": qkv.body.cpu(), "chain_logits": part.body.cpu(),
            "chain_map": pmap.cpu(), "chain_probs": plp.cpu(), "chain_ctx": ctx.body.cpu()}


def _main(out_path: str) -> None:
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if root not in sys.path:
        sys.path.insert(0, root)
    from rnamsm_b200 import _lib as L
    torch.cuda.set_device(0)
    L.device_check(torch.device("cuda:0"))
    want = int(os.environ["RNAMSM_GEMM_PAIRS"])
    got = L.lib.rnamsm_gemm_pairs()
    assert got == want, f"rnamsm_gemm_pairs() = {got}, RNAMSM_GEMM_PAIRS = {want}"
    outs = child_cases(L)
    outs["pairs"] = torch.tensor([got])
    torch.save(outs, out_path)
    print(f"gemm_exact child: {len(outs) - 1} outputs at {got} pairs")


if __name__ == "__main__":
    _main(sys.argv[1])
