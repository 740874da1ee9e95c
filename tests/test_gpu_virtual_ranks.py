"""GPU: the sharded forward's peer-memory kernels at 2 to 8 ranks on one GPU (tests/virtual_ranks.py).

One process stands in for n ranks: every exchange gets n local buffers, the kernel runs once per virtual rank with that
rank's rank / r0 / c0, and then every buffer is checked -- the rows a rank owns, the rows it must leave alone, the
guard rows around each buffer.  Each case runs twice: the n ranks one after another on the current stream (the
correctness check), then each rank on its own stream after the destinations are reset (event-ordered against the
current stream).  The second pass must be bit-identical to the first: no rank's writes land in another's region while
the others are in flight.

References: float64 and the single-GPU kernels.  LayerNorm push and add_layernorm are bit-identical to
rnamsm_layernorm and within test_layernorm's 16-bit gates of float64; the p2p softmax within the float64 gates of
tests/test_gpu_softmax_edges.py and 1e-6 of rnamsm_row_softmax on the same partials; the residual scatter runs on
operands on which the tensor-core GEMM is exact, so it equals float64 bit for bit, as does the map copy.
"""
import numpy as np
import pytest
import torch

import softmax_cases as SC
import virtual_ranks as VR
from oracle import msa_ref as O
from test_gpu_softmax_edges import LOGIT_SCALE, check_row_maps, p2p_warp3_logits, row_reference, run_row_softmax

pytestmark = pytest.mark.gpu

GUARD = 16                                   # rows before and after every destination buffer
LN_TOL = {1: 5e-3, 2: 6e-4}                  # tests/test_gpu_ops.py::test_layernorm, 16-bit outputs
CODES = pytest.mark.parametrize("code", [1, 2], ids=["bf16", "f16"])


@pytest.fixture(scope="module")
def L():
    from rnamsm_b200 import _lib
    _lib.device_check(torch.device("cuda:0"))
    return _lib


def bits(t):
    return t.view({2: torch.int16, 4: torch.int32}[t.element_size()])


def same_bits(a, b):
    return torch.equal(bits(a), bits(b))


def rel(a, b):
    return O.rel_err(a.detach().double().cpu(), b.detach().double().cpu())


def guarded(rows, cols, dtype):
    """NaN-filled [GUARD + rows + GUARD, cols] -> (whole buffer, its body of `rows` rows)."""
    buf = torch.full((rows + 2 * GUARD, cols), float("nan"), dtype=dtype, device="cuda")
    return buf, buf[GUARD:GUARD + rows]


def guards_intact(buf):
    sentinel = torch.full_like(buf[:GUARD], float("nan"))
    return same_bits(buf[:GUARD], sentinel) and same_bits(buf[-GUARD:], sentinel)


def ptr_array(L, tensors):
    return (L.C.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])


def run_ranks(n, launch, concurrent):
    """launch(g, stream_handle) for every virtual rank g: one after another on the current stream, or each on its
    own stream that waits for the current one (and that the current one waits for afterwards)."""
    main = torch.cuda.current_stream()
    if not concurrent:
        for g in range(n):
            launch(g, main.cuda_stream)
    else:
        streams = [torch.cuda.Stream() for _ in range(n)]
        for s in streams:
            s.wait_stream(main)
        for g, s in enumerate(streams):
            launch(g, s.cuda_stream)
        for s in streams:
            main.wait_stream(s)
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------ a) rnamsm_layernorm_push
LN_SHAPES = [(2, 8, 32, 768), (3, 9, 48, 768), (4, 12, 64, 256), (8, 24, 128, 768), (8, 8, 128, 128)]


@CODES
@pytest.mark.parametrize("shape,x_kind", [(s, "plain") for s in LN_SHAPES] + [((3, 9, 48, 768), "shifted")],
                         ids=[f"n{s[0]}_R{s[1]}_C{s[2]}_D{s[3]}" for s in LN_SHAPES] + ["n3_R9_C48_D768_shifted"])
def test_layernorm_push(L, shape, x_kind, code):
    """Token (r, c) of rank r // Rn's row shard lands in the column owner's buffer at row (c % Cn) * R + r."""
    n, R, C, D = shape
    Rn, Cn = VR.shard(R, C, n)
    gen = torch.Generator().manual_seed(1000 * n + D)
    if x_kind == "shifted":        # rows at +-64 with unit spread: a one-pass variance would cancel catastrophically
        x = torch.randn(R * C, D, generator=gen) + 64.0 * (1 - 2 * (torch.arange(R * C) % 2))[:, None]
    else:
        x = 2.0 * torch.randn(R * C, D, generator=gen) + 0.5
    w, b = (1 + 0.1 * torch.randn(D, generator=gen)).cuda(), (0.1 * torch.randn(D, generator=gen)).cuda()
    x_alloc = torch.zeros(R * C + C, D, device="cuda")        # C spare rows behind the last shard
    x_alloc[:R * C] = x.cuda()
    xd = x_alloc[:R * C]
    dt = L.torch_dtype(code)

    # single-GPU LayerNorm, token-major and transposed to column-major (c * R + r)
    y_tok = torch.empty(R * C, D, dtype=dt, device="cuda")
    y_cm = torch.empty(R * C, D, dtype=dt, device="cuda")
    L.check(L.lib.rnamsm_layernorm(L.ptr(xd), L.ptr(w), L.ptr(b), L.ptr(y_tok), code, R * C, D, O.LN_EPS, 0, 0,
                                   L.stream_ptr()), "layernorm")
    L.check(L.lib.rnamsm_layernorm(L.ptr(xd), L.ptr(w), L.ptr(b), L.ptr(y_cm), code, R * C, D, O.LN_EPS, R, C,
                                   L.stream_ptr()), "layernorm")
    owner, row = VR.push_index(R, C, n)
    owner, row = torch.from_numpy(owner).cuda(), torch.from_numpy(row).cuda()

    bufs = [guarded(Cn * R, D, dt) for _ in range(n)]
    dst = ptr_array(L, [body for _, body in bufs])

    def launch(g, st):
        L.check(L.lib.rnamsm_layernorm_push(L.ptr(xd[g * Rn * C:(g + 1) * Rn * C]), L.ptr(w), L.ptr(b), dst, n, Rn, C, R,
                                            g * Rn, D, O.LN_EPS, code, st), "layernorm_push")

    run_ranks(n, launch, concurrent=False)
    for buf, body in bufs:
        assert guards_intact(buf), "a write outside [0, Cn R)"
        assert not bool(torch.isnan(body.float()).any()), "a destination row was not written"
    first = [body.clone() for _, body in bufs]
    got = torch.cat(first)                                   # owner d's rows at [d Cn R, (d+1) Cn R)
    assert same_bits(got, y_cm), "differs from rnamsm_layernorm (tr_R = R, tr_C = C)"
    assert same_bits(got[owner * Cn * R + row], y_tok), "differs from the index map"
    ref = O.layer_norm(x.double(), w.double().cpu(), b.double().cpu())
    assert rel(got[owner * Cn * R + row], ref) < LN_TOL[code]

    for _, body in bufs:
        body.fill_(float("nan"))
    run_ranks(n, launch, concurrent=True)
    for (buf, body), f in zip(bufs, first):
        assert guards_intact(buf) and same_bits(body, f), "concurrent ranks differ from sequential ranks"


# ------------------------------------------------------------------------------------------ b) rnamsm_row_softmax_p2p
P2P_SHAPES = [(2, 1024, 2), (4, 256, 2), (8, 128, 2), (2, 4096, 1), (3, 1023, 2), (3, 1029, 2)]
P2P_IDS = ["vec_n2_C1024", "vec_n4_C256", "vec_n8_C128", "vec_n2_C4096", "scalar_cached_n3_C1023",
           "scalar_uncached_n3_C1029"]


@pytest.mark.parametrize("n_splits", [1, 3])
@pytest.mark.parametrize("regime", ["max_in_warp3", "onehot", "shifted", "masked_prefix", "fully_masked", "below_mask"])
@pytest.mark.parametrize("shape", P2P_SHAPES, ids=P2P_IDS)
def test_row_softmax_p2p(L, shape, regime, n_splits):
    """Rank g pulls rows [g C/n, (g+1) C/n) of every rank's partials, writes those map rows into its own map_out and
    the 16-bit rows into every rank's probs buffer."""
    n, C, H = shape
    if regime == "max_in_warp3":     # the maximum in the fourth warp of the vec kernel's block, on every rank's rows
        s, keypad = p2p_warp3_logits(C, H)
    else:
        s, keypad = SC.row_logits(regime, C, H, seed=43)
    parts = torch.from_numpy(VR.p2p_partials(s, n, n_splits, seed=43 + n)).cuda()
    kp = torch.from_numpy(keypad.astype(np.uint8)).cuda()
    ref, smax = row_reference(parts, kp)
    ld_lp = (C + 7) // 8 * 8 + 8
    slabs = [parts[g * n_splits:(g + 1) * n_splits] for g in range(n)]
    partial = ptr_array(L, slabs)
    Cq = C // n
    for code in (1, 2):
        dt = L.torch_dtype(code)
        maps = [torch.full((H, C, C), float("nan"), device="cuda") for _ in range(n)]
        probs = [torch.full((H, C, ld_lp), float("nan"), dtype=dt, device="cuda") for _ in range(n)]
        probs_arr = ptr_array(L, probs)

        def launch(g, st):
            L.check(L.lib.rnamsm_row_softmax_p2p(partial, n, g, n_splits, H, C, L.ptr(kp), LOGIT_SCALE, L.ptr(maps[g]),
                                                 probs_arr, ld_lp, code, st), "row_softmax_p2p")

        run_ranks(n, launch, concurrent=False)
        k5_map, _ = run_row_softmax(L, parts, kp, H, C, code, ld_lp)       # K5 on all n * n_splits slabs
        torch.cuda.synchronize()
        full = torch.full((H, C, C), float("nan"), device="cuda")
        for g in range(n):
            rows = slice(g * Cq, (g + 1) * Cq)
            assert list(VR.owned_rows(g, C, n)) == list(range(C))[rows]
            full[:, rows] = maps[g][:, rows]
            assert rel(maps[g][:, rows], k5_map[:, rows]) < 1e-6, f"rank {g} differs from K5"
            others = torch.ones(C, dtype=torch.bool, device="cuda")
            others[rows] = False
            assert bool(torch.isnan(maps[g][:, others]).all()), f"rank {g} wrote map rows it does not own"
        for g in range(1, n):
            assert same_bits(probs[g], probs[0]), f"rank {g}'s probs differ from rank 0's"
        check_row_maps(full, probs[0], ref, smax, C, code)              # finite, float64 gates, zero padding

        first_maps, first_probs = [m.clone() for m in maps], [p.clone() for p in probs]
        for m, p in zip(maps, probs):
            m.fill_(float("nan"))
            p.fill_(float("nan"))
        run_ranks(n, launch, concurrent=True)
        for m, p, fm, fp in zip(maps, probs, first_maps, first_probs):
            assert same_bits(m, fm) and same_bits(p, fp), "concurrent ranks differ from sequential ranks"


# ------------------------------------------------------------------------------------------ c) rnamsm_linear_residual_scatter
SCATTER_SHAPES = [(8, 8, 128, 768, 768), (4, 12, 192, 768, 768), (8, 256, 512, 768, 768), (2, 6, 32, 320, 128)]
SCATTER_IDS = ["n8_Cn16_Rn1", "n4_Cn48_odd_offsets", "n8_Cn64_wrapped_tiles", "n2_N320_partial_ntile"]


@pytest.mark.parametrize("delta16", [0, 1], ids=["reduce32", "delta16"])
@CODES
@pytest.mark.parametrize("shape", SCATTER_SHAPES, ids=SCATTER_IDS)
def test_linear_residual_scatter(L, shape, code, delta16):
    """Output row m = r Cn + cl of rank g lands in rank (r // Rn)'s buffer at row (r % Rn) C + g Cn + cl; on exact
    operands the result equals float64 bit for bit."""
    n, R, C, N, K = shape
    Rn, Cn = VR.shard(R, C, n)
    dt = L.torch_dtype(code)
    ctx, W, bias = VR.exact_gemm_operands(R * C, N, K, seed=7, device="cuda")      # ctx rows token-major (r, c)
    y64 = ctx.double() @ W.double().T + bias.double()                              # exact: see virtual_ranks.py
    ctx_g = [ctx.view(R, C, K)[:, g * Cn:(g + 1) * Cn].reshape(R * Cn, K).to(dt).contiguous() for g in range(n)]
    Wd = W.to(dt)
    del ctx
    if delta16:
        init = None
        want = y64.to(dt)
        bufs = [guarded(Rn * C, N, dt) for _ in range(n)]
    else:
        init = VR.exact_affine((R * C, N), 8, device="cuda")                       # the owners' residual streams
        want = (init.double() + y64).float()
        assert torch.equal(want.double(), init.double() + y64)
        bufs = [guarded(Rn * C, N, torch.float32) for _ in range(n)]
    del y64

    def reset():
        for d, (_, body) in enumerate(bufs):
            if delta16:
                body.fill_(float("nan"))
            else:
                body.copy_(init[d * Rn * C:(d + 1) * Rn * C])

    reset()
    dst = ptr_array(L, [body for _, body in bufs])

    def launch(g, st):
        L.check(L.lib.rnamsm_linear_residual_scatter(L.ptr(ctx_g[g]), L.ptr(Wd), L.ptr(bias), R, Cn, N, K, code, dst, n,
                                                     Rn, C, g * Cn, delta16, st), "linear_residual_scatter")

    run_ranks(n, launch, concurrent=False)
    for buf, _ in bufs:
        assert guards_intact(buf), "a write outside [0, Rn C)"
    first = [body.clone() for _, body in bufs]
    got = torch.cat(first)                      # owner d's rows (r - d Rn) C + c at d Rn C + ...: token-major (r, c)
    assert same_bits(got, want), f"max |err| {float((got.double() - want.double()).abs().max()):.3e}"

    # each rank's contribution equals rnamsm_linear on its ctx, rearranged by the index map
    for g in range(n):
        owner, row = VR.scatter_index(g, R, C, n)
        idx = torch.from_numpy(owner * Rn * C + row).cuda()
        if delta16:
            plain = torch.empty(R * Cn, N, dtype=dt, device="cuda")
            L.check(L.lib.rnamsm_linear(L.ptr(ctx_g[g]), L.ptr(Wd), L.ptr(bias), R * Cn, N, K, code, L.EPI_BIAS, 1.0, 0,
                                        None, L.ptr(plain), L.stream_ptr()), "linear")
        else:
            plain = init[idx].contiguous()
            L.check(L.lib.rnamsm_linear(L.ptr(ctx_g[g]), L.ptr(Wd), L.ptr(bias), R * Cn, N, K, code,
                                        L.EPI_BIAS_RESIDUAL, 1.0, 0, None, L.ptr(plain), L.stream_ptr()), "linear")
        torch.cuda.synchronize()
        assert same_bits(got[idx], plain), f"rank {g} differs from rnamsm_linear"

    reset()
    run_ranks(n, launch, concurrent=True)
    for (buf, body), f in zip(bufs, first):
        assert guards_intact(buf) and same_bits(body, f), "concurrent ranks differ from sequential ranks"


# ------------------------------------------------------------------------------------------ d) rnamsm_add_layernorm
@pytest.mark.parametrize("D", [128, 768, 1024])
@pytest.mark.parametrize("rows", [1, 7, 1001])
@pytest.mark.parametrize("ycode", [1, 2], ids=["y_bf16", "y_f16"])
@pytest.mark.parametrize("dcode", [1, 2], ids=["delta_bf16", "delta_f16"])
def test_add_layernorm(L, dcode, ycode, rows, D):
    """The receiving end of the 16-bit scatter payload: x += delta in fp32, then the LayerNorm of rnamsm_layernorm."""
    gen = torch.Generator().manual_seed(rows * D + 10 * dcode + ycode)
    x0 = (2.0 * torch.randn(rows, D, generator=gen) + 0.5).cuda()
    delta = (0.5 * torch.randn(rows, D, generator=gen)).to(L.torch_dtype(dcode)).cuda()
    w, b = (1 + 0.1 * torch.randn(D, generator=gen)).cuda(), (0.1 * torch.randn(D, generator=gen)).cuda()
    ydt = L.torch_dtype(ycode)
    x = x0.clone()
    y = torch.full((rows, D), float("nan"), dtype=ydt, device="cuda")
    L.check(L.lib.rnamsm_add_layernorm(L.ptr(x), L.ptr(delta), dcode, L.ptr(w), L.ptr(b), L.ptr(y), ycode, rows, D,
                                       O.LN_EPS, L.stream_ptr()), "add_layernorm")
    y_plain = torch.empty(rows, D, dtype=ydt, device="cuda")
    L.check(L.lib.rnamsm_layernorm(L.ptr(x), L.ptr(w), L.ptr(b), L.ptr(y_plain), ycode, rows, D, O.LN_EPS, 0, 0,
                                   L.stream_ptr()), "layernorm")
    torch.cuda.synchronize()
    assert same_bits(x, x0 + delta.float())
    assert same_bits(y, y_plain)
    assert rel(y, O.layer_norm(x.double(), w.double(), b.double())) < LN_TOL[ycode]


# ------------------------------------------------------------------------------------------ e) rnamsm_copy_map_rows_d2h
def test_copy_map_rows_d2h(L):
    """Eight owners of a 128-column layer copy their query rows of the stripped block [1, 127)^2 into one pinned host
    buffer.  Each owner's map holds only its own rows (NaN elsewhere), as the p2p softmax leaves it."""
    n, C, H, start = 8, 128, 2, 1
    Ls, Cq = C - 2, C // n
    vals = torch.randn(H, C, C, generator=torch.Generator().manual_seed(5)).cuda()
    maps = []
    for g in range(n):
        m = torch.full((H, C, C), float("nan"), device="cuda")
        m[:, g * Cq:(g + 1) * Cq] = vals[:, g * Cq:(g + 1) * Cq]
        maps.append(m)
    empty_map = torch.full((H, C, C), float("nan"), device="cuda")
    host = torch.full((H, Ls, Ls), float("nan")).pin_memory()
    want = vals[:, start:start + Ls, start:start + Ls].cpu()

    def launch(g, st):
        L.check(L.lib.rnamsm_copy_map_rows_d2h(L.ptr(maps[g]), H, C, g * Cq, (g + 1) * Cq, start, Ls, host.data_ptr(),
                                               st), "copy_map_rows_d2h")

    for concurrent in (False, True):
        host.fill_(float("nan"))
        run_ranks(n, launch, concurrent)
        # [0, 1) lies inside the stripped prefix: nothing to copy (from a map that is all NaN)
        L.check(L.lib.rnamsm_copy_map_rows_d2h(L.ptr(empty_map), H, C, 0, 1, start, Ls, host.data_ptr(), L.stream_ptr()),
                "copy_map_rows_d2h")
        torch.cuda.synchronize()
        assert not bool(torch.isnan(host).any())
        assert same_bits(host, want)
