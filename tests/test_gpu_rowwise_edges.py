"""GPU: the one-warp-per-row kernels against float64 at hostile rows, every width and every grid-stride edge
(tests/rowwise_cases.py), through the C ABI only.

Kernels: rnamsm_layernorm (fp32 / bf16 / fp16 out, plain, token-transposed and in place), rnamsm_add_layernorm,
rnamsm_embed_layernorm (K1), rnamsm_vocab_proj (K9b), rnamsm_contact_head and rnamsm_range_scan.  The LayerNorm and
contact-head gates are derived per element in rowwise_cases; the vocabulary projection is bit-exact on exact operands
and within the fp32 dot-product bound on randn ones; the range scan's counters are exact.

Every output goes into a buffer filled with a signalling-NaN sentinel, with GUARD sentinel elements before and after
it: the guards must come back untouched and no element of the output may still hold the sentinel (a kernel-made NaN
has another bit pattern).  Each entry point is called twice on the same inputs and must give the same bits.

Row counts straddle the grid-stride sweeps: the LayerNorm kernels run at most 148 * 32 blocks of 8 warps
(37 888 rows per sweep), the vocabulary projection 148 * 16 blocks of 8 warps (18 944 tokens) and the range scan
148 * 8 blocks of 256 threads (303 104 elements).  The float64 references run on the device.
"""
import numpy as np
import pytest
import torch

import rowwise_cases as RC

pytestmark = pytest.mark.gpu

GUARD = 256                                                  # elements; keeps every view 16-byte aligned
SENTINEL = {torch.float32: (torch.int32, 0x7FA5A5A5), torch.bfloat16: (torch.int16, 0x7FA5),
            torch.float16: (torch.int16, 0x7E5A), torch.uint8: (torch.uint8, 0xA5)}
WIDTHS = [128 * k for k in range(1, 9)]
LN_ROWS = [1, 7, 8, 9, 37887, 37888, 37889, 75777]
POOL = 4099          # distinct rows per large case (prime: no row repeats at a grid-stride or transpose period)
CODES = [0, 1, 2]
VOCAB, PAD = 12, 1


@pytest.fixture(scope="module")
def L():
    from rnamsm_b200 import _lib
    _lib.device_check(torch.device("cuda:0"))
    return _lib


class Guarded:
    """n elements of dtype between two GUARD-long sentinel regions."""

    def __init__(self, n, dtype):
        idt, word = SENTINEL[dtype]
        self.bits = torch.full((GUARD + n + GUARD,), word, dtype=idt, device="cuda")
        self.buf = self.bits.view(dtype)
        self.out = self.buf[GUARD:GUARD + n]
        self.word, self.n = word, n

    def check(self, what=""):
        g = torch.cat([self.bits[:GUARD], self.bits[GUARD + self.n:]])
        assert bool((g == self.word).all()), f"{what}: guard region written"
        assert not bool((self.bits[GUARD:GUARD + self.n] == self.word).any()), f"{what}: element(s) never written"
        return self.out


def bits(t):
    return t.contiguous().view({4: torch.int32, 2: torch.int16, 1: torch.uint8}[t.element_size()])


def same_bits(a, b):
    return torch.equal(bits(a), bits(b))


def mixed_rows(rows, D, seed, rotate=0):
    """ln_mixed_rows, with large row counts tiled from a POOL-row pool (regime of each row returned alongside)."""
    n = min(rows, POOL)
    x, reg = RC.ln_mixed_rows(n, D, seed, rotate)
    xt, rt = torch.from_numpy(x).cuda(), torch.from_numpy(reg).cuda()
    if rows > n:
        idx = torch.arange(rows, device="cuda") % n
        xt, rt = xt[idx].contiguous(), rt[idx]
    return xt, rt


def affine(D, seed, saturating=False):
    w, b = RC.ln_affine(D, seed, saturating)
    return torch.from_numpy(w).cuda(), torch.from_numpy(b).cuda()


def run_layernorm(L, x, w, b, code, tr=(0, 0), y=None):
    rows, D = x.shape
    g = None
    if y is None:
        g = Guarded(rows * D, L.torch_dtype(code))
        y = g.out
    L.check(L.lib.rnamsm_layernorm(L.ptr(x), L.ptr(w), L.ptr(b), L.ptr(y), code, rows, D, RC.LN_EPS, tr[0], tr[1],
                                   L.stream_ptr()), "layernorm")
    if g is None:
        return y.view(rows, D)
    torch.cuda.synchronize()
    return g.check("layernorm").view(rows, D)


def transpose_shape(rows):
    d = max([k for k in range(1, int(rows ** 0.5) + 1) if rows % k == 0])
    return rows // d, d                                      # (tr_R, tr_C); a prime count permutes nothing


WORST = {}


def record(kernel, ratio):
    WORST[kernel] = max(WORST.get(kernel, 0.0), ratio)


@pytest.fixture(scope="module", autouse=True)
def report_worst():
    yield
    for k, v in sorted(WORST.items()):
        print(f"[rowwise] {k}: worst error / gate {v:.3f}")


# ------------------------------------------------------------------------------------------ rnamsm_layernorm
@pytest.mark.parametrize("rows", LN_ROWS)
@pytest.mark.parametrize("D", WIDTHS)
def test_layernorm(L, D, rows):
    """Every regime (row r in regime (r + rotation) % 7), every output type: within the derived gate; constant_grid
    and zero rows exactly b; the transposed form equal to the permuted plain form; in-place fp32 equal to
    out-of-place; a second call bit-identical."""
    w, b = affine(D, 5)
    for rotate in (range(len(RC.ROW_REGIMES)) if rows < len(RC.ROW_REGIMES) else [0]):
        x, reg = mixed_rows(rows, D, 11, rotate)
        exact_b = torch.zeros_like(reg, dtype=torch.bool)
        for name in RC.EXACT_B_REGIMES:
            exact_b |= reg == RC.ROW_REGIMES.index(name)
        for code in CODES:
            ref, gate = RC.ln_reference(x, w, b, code)
            y = run_layernorm(L, x, w, b, code)
            assert bool(torch.isfinite(y.float()).all())
            ratio = RC.gate_ratio(y, ref, gate)
            record(f"layernorm out{code}", ratio)
            assert ratio <= 1.0, f"code {code} rotate {rotate}: error / gate {ratio:.3f}"
            if bool(exact_b.any()):
                assert same_bits(y[exact_b], RC.ln_expected_b(b, code).expand(int(exact_b.sum()), D))
            assert same_bits(run_layernorm(L, x, w, b, code), y), "second call differs"
            R_, C_ = transpose_shape(rows)
            yt = run_layernorm(L, x, w, b, code, tr=(R_, C_))
            assert same_bits(yt.view(C_, R_, D), y.view(R_, C_, D).transpose(0, 1)), "transposed form differs"
            del ref, gate
        x_in = x.clone()
        y_in = run_layernorm(L, x_in, w, b, 0, y=x_in)
        torch.cuda.synchronize()
        assert same_bits(y_in, run_layernorm(L, x, w, b, 0)), "in-place form differs"


@pytest.mark.parametrize("rows", [9, 37889])
@pytest.mark.parametrize("D", WIDTHS)
def test_layernorm_saturating(L, D, rows):
    """|w| ~ 3e4: fp16 outputs past 65504 are exactly +-65504 (cvt.rn.satfinite), never inf; bf16 is round to nearest
    within the gate; fp32 within the gate."""
    w, b = affine(D, 5, saturating=True)
    x, _ = mixed_rows(rows, D, 13)
    y32ref, g32 = RC.ln_reference(x, w, b, 0)
    assert float(y32ref.abs().max()) > RC.F16_MAX
    for code in CODES:
        ref, gate = RC.ln_reference(x, w, b, code)
        y = run_layernorm(L, x, w, b, code)
        assert bool(torch.isfinite(y.float()).all())
        ratio = RC.gate_ratio(y, ref, gate)
        record(f"layernorm saturating out{code}", ratio)
        assert ratio <= 1.0, f"code {code}: error / gate {ratio:.3f}"
        if code == 2:
            over = (y32ref.abs() - g32) > RC.F16_MAX + 16    # beyond the rounding midpoint to the next fp16 step
            assert bool(over.any())
            assert torch.equal(y.double()[over], torch.sign(y32ref[over]) * RC.F16_MAX)


# ------------------------------------------------------------------------------------------ rnamsm_add_layernorm
@pytest.mark.parametrize("rows", [9, 37889])
@pytest.mark.parametrize("ycode", [1, 2], ids=["y_bf16", "y_f16"])
@pytest.mark.parametrize("dcode", [1, 2], ids=["d_bf16", "d_f16"])
@pytest.mark.parametrize("D", WIDTHS)
def test_add_layernorm(L, D, dcode, ycode, rows):
    """x += float(delta) exactly as fp32 adds it; y = LayerNorm(x) in 16 bits within the derived gate; rows of every
    regime."""
    w, b = affine(D, 7)
    x, _ = mixed_rows(rows, D, 17)
    g = torch.Generator(device="cuda").manual_seed(D + rows)
    delta = (0.5 * torch.randn(rows, D, generator=g, device="cuda")).to(L.torch_dtype(dcode))
    want_x = x + delta.float()
    ref, gate = RC.ln_reference(want_x, w, b, ycode)
    outs = []
    for _ in range(2):
        xx = x.clone()
        gy = Guarded(rows * D, L.torch_dtype(ycode))
        L.check(L.lib.rnamsm_add_layernorm(L.ptr(xx), L.ptr(delta), dcode, L.ptr(w), L.ptr(b), L.ptr(gy.out), ycode,
                                           rows, D, RC.LN_EPS, L.stream_ptr()), "add_layernorm")
        torch.cuda.synchronize()
        outs.append((xx, gy.check("add_layernorm").view(rows, D)))
    (xx, y), (xx2, y2) = outs
    assert same_bits(xx, want_x), "updated x differs from x + float(delta)"
    assert same_bits(xx2, xx) and same_bits(y2, y), "second call differs"
    ratio = RC.gate_ratio(y, ref, gate)
    record(f"add_layernorm d{dcode} y{ycode}", ratio)
    assert ratio <= 1.0, f"error / gate {ratio:.3f}"


# ------------------------------------------------------------------------------------------ rnamsm_embed_layernorm
def run_embed(L, tokens, tok, pos, row, w, b, D):
    R, C = tokens.shape
    gx, gp = Guarded(R * C * D, torch.float32), Guarded(R * C, torch.uint8)
    L.check(L.lib.rnamsm_embed_layernorm(L.ptr(tokens), R, C, L.ptr(tok), VOCAB, L.ptr(pos), pos.shape[0], L.ptr(row),
                                         L.ptr(w), L.ptr(b), D, PAD, RC.LN_EPS, L.ptr(gx.out), L.ptr(gp.out),
                                         L.stream_ptr()), "embed_layernorm")
    torch.cuda.synchronize()
    return gx.check("embed x").view(R, C, D), gp.check("embed pad").view(R, C)


@pytest.mark.parametrize("R,C,D", [(4, c, 768) for c in (1, 31, 32, 33, 63, 64, 65, 127, 128, 129, 1000)]
                         + [(1024, 33, 128), (1024, 130, 1024), (3, 1000, 1024)])
@pytest.mark.parametrize("with_row_pos", [True, False], ids=["row_pos", "no_row_pos"])
def test_embed_layernorm(L, R, C, D, with_row_pos):
    """Pads mid-row at columns 31, 32, 63, 64 and 127 with real tokens after them (their count carries across 32-column
    scan steps and 64-column blocks), a BOS-only row, tokens 0 and vocab - 1, and a positional table whose last row is
    exactly the largest position used.  Exact-grid tables: the LayerNorm input is exact, so the LayerNorm gate applies
    as is; pad rows exactly 0; pad_out exact."""
    tokens = RC.embed_tokens(R, C, VOCAB, PAD, seed=C)
    n_pos = int(RC.positions(tokens, PAD).max()) + 1
    tok, pos, row = (torch.from_numpy(a).cuda() for a in RC.embed_tables(VOCAB, n_pos, R, D, seed=3, pad_idx=PAD))
    row = row if with_row_pos else None
    w, b = affine(D, 9)
    tokens = tokens.cuda()
    ref, gate, pad = RC.embed_reference(tokens, tok, pos, row, w, b, PAD)
    x, pad_out = run_embed(L, tokens, tok, pos, row, w, b, D)
    x2, pad_out2 = run_embed(L, tokens, tok, pos, row, w, b, D)
    assert same_bits(x2, x) and torch.equal(pad_out2, pad_out), "second call differs"
    assert torch.equal(pad_out, pad.to(torch.uint8))
    assert bool((bits(x[pad]) == 0).all()), "pad rows must be exactly +0"
    keep = ~pad
    ratio = RC.gate_ratio(x[keep], ref[keep], gate[keep])
    record("embed_layernorm", ratio)
    assert ratio <= 1.0, f"error / gate {ratio:.3f}"


# ------------------------------------------------------------------------------------------ rnamsm_vocab_proj
def run_vocab(L, h, E, bias):
    M, D = h.shape
    V = E.shape[0]
    outs = []
    for _ in range(2):
        g = Guarded(M * V, torch.float32)
        L.check(L.lib.rnamsm_vocab_proj(L.ptr(h), L.ptr(E), L.ptr(bias), M, V, D, L.ptr(g.out), L.stream_ptr()),
                "vocab_proj")
        torch.cuda.synchronize()
        outs.append(g.check("vocab_proj").view(M, V))
    assert same_bits(outs[0], outs[1]), "second call differs"
    return outs[0]


@pytest.mark.parametrize("M", [1, 18943, 18944, 18945])
@pytest.mark.parametrize("D", [128, 768, 1024])
@pytest.mark.parametrize("V", [1, 12, 31, 32])
def test_vocab_proj(L, V, D, M):
    h, E, bias = (torch.from_numpy(a).cuda() for a in RC.vocab_exact_operands(M, V, D, seed=5))
    ref, _ = RC.vocab_reference(h, E, bias)
    assert torch.equal(run_vocab(L, h, E, bias).double(), ref), "exact operands: not bit-exact"
    g = torch.Generator(device="cuda").manual_seed(M * 7 + V)
    h, E, bias = (torch.randn(s, generator=g, device="cuda") for s in ((M, D), (V, D), (V,)))
    ref, gate = RC.vocab_reference(h, E, bias)
    ratio = RC.gate_ratio(run_vocab(L, h, E, bias), ref, gate)
    record("vocab_proj", ratio)
    assert ratio <= 1.0, f"error / gate {ratio:.3f}"


# ------------------------------------------------------------------------------------------ rnamsm_contact_head
CONTACT_CASES = ([(kind, Ls, K, start) for kind in RC.CONTACT_MAPS for Ls in (1, 2, 31, 32, 33, 64, 65)
                  for K in (1, 24, 120) for start in (0, 1)]
                 + [(kind, 1023, 24, 1) for kind in RC.CONTACT_MAPS])


def run_contact(L, maps, start, Ls, w, bias):
    K, C, _ = maps.shape
    ws = torch.empty(K * Ls + K, device="cuda")
    g = Guarded(Ls * Ls, torch.float32)
    L.check(L.lib.rnamsm_contact_head(L.ptr(maps), K, C, start, Ls, L.ptr(w), L.ptr(bias), L.ptr(g.out), L.ptr(ws),
                                      L.stream_ptr()), "contact_head")
    torch.cuda.synchronize()
    return g.check("contact_head").view(Ls, Ls)


@pytest.mark.parametrize("kind,Ls,K,start", CONTACT_CASES)
def test_contact_head(L, kind, Ls, K, start):
    """Structured maps over the block [start, start + L) of C = L + 1 columns: output within the derived gate, its
    logit too where the sigmoid is not saturated, NaN exactly where the float64 formula is NaN, exact symmetry."""
    C = Ls + 1
    maps = torch.from_numpy(RC.contact_maps(kind, K, C, seed=Ls)).cuda()
    g = torch.Generator(device="cuda").manual_seed(K * 1000 + Ls)
    w = torch.randn(K, generator=g, device="cuda")
    bias = torch.randn(1, generator=g, device="cuda")
    out = run_contact(L, maps, start, Ls, w, bias)
    assert same_bits(run_contact(L, maps, start, Ls, w, bias), out), "second call differs"
    assert same_bits(out, out.T), "not exactly symmetric"
    ref, logit, lgate = RC.contact_reference(maps, start, Ls, w, bias)
    nan = torch.isnan(ref)
    assert torch.equal(torch.isnan(out), nan)
    if kind == "all_bos":
        assert bool(nan.all()) == (start == 1)
    ok = ~nan
    if not bool(ok.any()):
        return
    assert bool(torch.isfinite(out[ok]).all())
    ratio = RC.gate_ratio(out[ok], ref[ok], RC.contact_out_gate(logit[ok], lgate[ok]))
    record("contact_head out", ratio)
    assert ratio <= 1.0, f"output error / gate {ratio:.3f}"
    o = out.double()
    live = ok & (o > 2.0 ** -60) & (o < 1 - 2.0 ** -10)
    if bool(live.any()):
        lr = RC.gate_ratio(RC.logit_of(out[live]), logit[live], RC.contact_logit_gate(out[live], logit[live], lgate[live]))
        record("contact_head logit", lr)
        assert lr <= 1.0, f"logit error / gate {lr:.3f}"


# ------------------------------------------------------------------------------------------ rnamsm_range_scan
def scan(L, buf, n, code, counters):
    L.check(L.lib.rnamsm_range_scan(L.ptr(buf), n, code, L.ptr(counters), L.stream_ptr()), "range_scan")
    torch.cuda.synchronize()
    return int(counters[0]), int(counters[1])


@pytest.mark.parametrize("n", [0, 1, 255, 256, 303103, 303104, 303105, 1000003])
@pytest.mark.parametrize("code", [1, 2], ids=["bf16", "f16"])
def test_range_scan(L, code, n):
    """Exact edge counts (largest finite value, inf and NaN of both signs; subnormals and zeros are not edges) and
    the bit pattern of the largest non-edge magnitude; a second call accumulates the count and keeps the maximum; a
    call on smaller values leaves both; n = 0 touches nothing."""
    big = RC.range_buffer(code, n, seed=1)
    small = RC.range_buffer(code, n, seed=2, patterns=False)
    cb, mb = RC.range_reference(big, code)
    cs, ms = RC.range_reference(small, code)
    assert cs == 0
    dev = {k: torch.from_numpy(a.view(np.int16)).cuda() for k, a in (("big", big), ("small", small))}
    counters = torch.zeros(2, dtype=torch.int64, device="cuda")
    assert scan(L, dev["small"], n, code, counters) == (0, ms)
    assert scan(L, dev["big"], n, code, counters) == (cb, max(mb, ms))
    assert scan(L, dev["big"], n, code, counters) == (2 * cb, max(mb, ms))
    assert scan(L, dev["small"], n, code, counters) == (2 * cb, max(mb, ms))
    counters.copy_(torch.tensor([5, 123]))
    assert scan(L, dev["big"], 0, code, counters) == (5, 123)
