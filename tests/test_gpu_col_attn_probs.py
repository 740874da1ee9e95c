"""GPU: column-attention probabilities on request (rnamsm_col_attn_probs and the *_col_probs drivers, the
need_weights / need_col_weights / need_col_weights_mean keywords).

Per op the checker is a float64 softmax of the SAME (already rounded) q|k, so what remains is the kernels' own
arithmetic: fp32 logits (tensor-core or FFMA accumulation, ~1e-7 relative), one fp32 rounding of s * log2(e) and
ex2.approx.ftz (2 ulp) in the 16-bit path, expf / logf in the fp32 path, and the fp32 running sum of the log-sum-exp
over <= 1024 keys.  Together a few 1e-7 of the largest probability; the gate is 1e-5.
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from col_probs_ref import forward_col_probs
from oracle import msa_ref as O

pytestmark = pytest.mark.gpu

PROBS_TOL = 1e-5
PRECISIONS = ["fp32", "fp16", "bf16"]


@pytest.fixture(scope="module")
def L():
    from rnamsm_b200 import _lib
    _lib.device_check(torch.device("cuda:0"))
    return _lib


@pytest.fixture(scope="module")
def pkg():
    import rnamsm_b200
    return rnamsm_b200


# "bf16" runs the column block on bf16 operands (only the tied row block stays fp16).  On layer.npz's sharpen-8 weights
# the column logits span tens of nats, and one bf16 rounding of q and k (2^-9 relative) moves a logit of 40 by ~0.1:
# the column maps measured 1.0e-1 against the reference there, and 3.0e-2 between the fused layer and the blocks called
# one by one (fp16: within 2e-2 and 1e-2).  That mode is gated at its own envelope, as tests/test_gpu_model.py does for
# its row maps.
BF16_COL_LAYER_TOL = 0.15


def tols(precision, sharp_deep=False):
    """The map tolerances of tests/test_gpu_model.py (test_model_vs_reference_golden)."""
    if precision == "fp32":
        return 1e-4
    if precision == "fp16":
        return 8e-2 if sharp_deep else 2e-2
    return max(6e-2, 8e-2 if sharp_deep else 0)


def rel(a, b):
    return O.rel_err(a.detach().double().cpu(), b.detach().double().cpu())


def make_qkv(R, Cc, H, code, L, seed, scale=0.6):
    """Token-major q|k|v [R, C, 3D] in the operand dtype (q scaled as the QKV epilogue does) + its float64 copy."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    D = H * 64
    x = torch.randn(R, Cc, 3 * D, generator=g, device="cuda") * scale
    x[..., :D] *= 64 ** -0.5 * 8
    qkv = x.to(L.torch_dtype(code))
    return qkv, qkv.double()


def ref_probs(q64, R, Cc, H, pad):
    """float64 [H, C, R, R] softmax of q k^T with padded keys replaced by -10000."""
    D = H * 64
    q = q64[..., :D].reshape(R, Cc, H, 64)
    k = q64[..., D:2 * D].reshape(R, Cc, H, 64)
    s = torch.einsum("ichd,jchd->hcij", q, k)
    if pad is not None:
        s = s.masked_fill(pad.T.bool()[None, :, None, :], -10000)
    return s.softmax(-1)


def col_probs(L, qkv, R, Cc, H, code, col_major, pad, full=True, mean=True):
    dev = qkv.device
    probs = torch.full((H, Cc, R, R), float("nan"), device=dev) if full else None
    mp = torch.full((H, R, R), float("nan"), device=dev) if mean else None
    scratch = torch.empty(max(1, L.lib.rnamsm_col_probs_scratch_bytes(R, Cc, H)), dtype=torch.uint8, device=dev)
    L.check(L.lib.rnamsm_col_attn_probs(L.ptr(qkv), R, Cc, H, code, col_major, L.ptr(pad), L.ptr(probs), L.ptr(mp),
                                        L.ptr(scratch), L.stream_ptr()), "col_attn_probs")
    return probs, mp


# ------------------------------------------------------------------------------------------ per op
@pytest.mark.parametrize("R,Cc", [(2, 5), (7, 19), (64, 3), (127, 4), (128, 3), (129, 5), (300, 3), (1024, 2)])
@pytest.mark.parametrize("code,col_major", [(0, 0), (1, 0), (2, 0), (1, 1), (2, 1)],
                         ids=["f32", "bf16", "f16", "bf16-colmajor", "f16-colmajor"])
def test_col_attn_probs_vs_float64(L, R, Cc, code, col_major):
    H = 2
    qkv, q64 = make_qkv(R, Cc, H, code, L, 7 * R + Cc)
    pad = torch.zeros(R, Cc, dtype=torch.uint8)
    pad[-1, :] = 1
    pad[R // 2, 0] = 1
    pad[:, Cc - 1] = 1                                        # a fully padded column -> uniform rows
    ref = ref_probs(q64.cpu(), R, Cc, H, pad)
    pad_d = pad.cuda()
    arg = qkv.transpose(0, 1).contiguous() if col_major else qkv
    probs, mean = col_probs(L, arg, R, Cc, H, code, col_major, pad_d)
    torch.cuda.synchronize()
    e_full, e_mean = rel(probs, ref), rel(mean, ref.mean(1))
    print(f"[R={R} C={Cc} code={code} cm={col_major}] full {e_full:.2e} mean {e_mean:.2e}")
    assert e_full <= PROBS_TOL and e_mean <= PROBS_TOL
    assert (probs.sum(-1) - 1).abs().max().item() <= 1e-5
    # the two outputs from one launch, and each alone, are the same numbers; repeated calls are bitwise equal
    p2, m2 = col_probs(L, arg, R, Cc, H, code, col_major, pad_d)
    p_only, _ = col_probs(L, arg, R, Cc, H, code, col_major, pad_d, mean=False)
    _, m_only = col_probs(L, arg, R, Cc, H, code, col_major, pad_d, full=False)
    assert torch.equal(p2, probs) and torch.equal(m2, mean) and torch.equal(p_only, probs) and torch.equal(m_only, mean)
    # P V in float64 reproduces the flash kernel's ctx within that kernel's own tolerance (tests/test_gpu_ops.py)
    D = H * 64
    v = q64[..., 2 * D:].reshape(R, Cc, H, 64)
    ctx_ref = torch.einsum("hcij,jchd->ichd", probs.double(), v).reshape(R * Cc, D)
    ctx = torch.empty(R * Cc, D, dtype=L.torch_dtype(code), device="cuda")
    L.check(L.lib.rnamsm_col_attn(L.ptr(qkv), R, Cc, H, code, 0, L.ptr(pad_d), L.ptr(ctx), L.stream_ptr()), "col_attn")
    assert rel(ctx, ctx_ref) < {0: 2e-5, 1: 1e-2, 2: 2e-3}[code]


def test_col_attn_probs_single_row_and_errors(L):
    """R == 1: all ones without reading q|k or scratch; a missing scratch is an error, not a fault."""
    probs = torch.zeros(3, 5, 1, 1, device="cuda")
    mean = torch.zeros(3, 1, 1, device="cuda")
    L.check(L.lib.rnamsm_col_attn_probs(None, 1, 5, 3, L.F16, 0, None, L.ptr(probs), L.ptr(mean), None, L.stream_ptr()))
    torch.cuda.synchronize()
    assert bool((probs == 1).all()) and bool((mean == 1).all())
    qkv, _ = make_qkv(4, 3, 1, L.F16, L, 1)
    out = torch.empty(1, 3, 4, 4, device="cuda")
    assert L.lib.rnamsm_col_attn_probs(L.ptr(qkv), 4, 3, 1, L.F16, 0, None, L.ptr(out), None, None, L.stream_ptr()) != 0
    assert b"scratch" in L.lib.rnamsm_last_error()
    assert L.lib.rnamsm_col_attn_probs(L.ptr(qkv.float()), 4, 3, 1, L.F32, 1, None, L.ptr(out), None,
                                       L.ptr(out), L.stream_ptr()) != 0


# ------------------------------------------------------------------------------------------ layer level
@pytest.mark.parametrize("precision", PRECISIONS)
def test_layer_col_weights_vs_reference_layer(pkg, golden_dir, precision):
    """need_col_weights=True against the reference layer's own column probabilities (layer.npz col_nopad / col_pad,
    sharpen 8); y and the row maps are exactly those of the call without the keyword."""
    g = np.load(os.path.join(golden_dir, "layer.npz"))
    sd = O.make_weights(int(g["wseed"]), num_layers=1, sharpen=float(g["sharpen"]))
    layer = pkg.AxialTransformerLayer(768, 3072, 12).set_precision(precision)
    layer.load_state_dict({k[len("layers.0."):]: v for k, v in sd.items() if k.startswith("layers.0.")}, strict=True)
    layer = layer.eval().cuda()
    x = torch.from_numpy(g["x"]).cuda()
    pad = torch.from_numpy(g["pad"]).cuda()
    for tag, pm in (("nopad", None), ("pad", pad)):
        y, col, row = layer(x, self_attn_padding_mask=pm, need_col_weights=True)
        y0, col0, row0 = layer(x, self_attn_padding_mask=pm, need_head_weights=True)
        assert col0 is None and tuple(col.shape) == g[f"col_{tag}"].shape == (12, 19, 1, 7, 7)
        assert torch.equal(y, y0) and torch.equal(row, row0)
        e = rel(col, torch.from_numpy(g[f"col_{tag}"]))
        print(f"[layer col/{tag}/{precision}] {e:.3e}")
        assert e < (BF16_COL_LAYER_TOL if precision == "bf16" else tols(precision))
        # the blocks called one by one: the column block returns the same layout (from its own un-fused input -- rounded
        # to 16 bits in the 16-bit path -- so close rather than equal; the sharpened logits amplify the difference)
        h, _ = layer.row_self_attention(x, self_attn_padding_mask=pm)
        _, col_sub = layer.column_self_attention(h, self_attn_padding_mask=pm, need_weights=True)
        assert tuple(col_sub.shape) == tuple(col.shape)
        assert rel(col_sub, col) < {"fp32": 1e-4, "fp16": 1e-2, "bf16": BF16_COL_LAYER_TOL}[precision]


def test_layer_col_weights_batch2(pkg):
    """B = 2: each batch entry's slab equals that entry run alone."""
    sd = O.make_weights(2, num_layers=1)
    layer = pkg.AxialTransformerLayer(768, 3072, 12).set_precision("fp16")
    layer.load_state_dict({k[len("layers.0."):]: v for k, v in sd.items() if k.startswith("layers.0.")}, strict=True)
    layer = layer.eval().cuda()
    x = torch.randn(9, 11, 2, 768, generator=torch.Generator().manual_seed(3)).cuda()
    _, col, _ = layer(x, need_col_weights=True)
    for b in range(2):
        _, cb, _ = layer(x[:, :, b:b + 1].contiguous(), need_col_weights=True)
        assert torch.equal(col[:, :, b], cb[:, :, 0])


# ------------------------------------------------------------------------------------------ model level
_REF = {}


def model_ref(golden_dir, name):
    if name not in _REF:
        g = np.load(os.path.join(golden_dir, name + ".npz"))
        layers = int(g["layers"])
        sd = O.to_dtype(O.make_weights(int(g["wseed"]), num_layers=layers, sharpen=float(g["sharpen"])), torch.float64)
        tokens = torch.from_numpy(g["tokens"].astype(np.int64))
        _REF[name] = (g, forward_col_probs(sd, tokens, layers))
    return _REF[name]


@pytest.mark.parametrize("name", ["tiny", "tiny_pad", "batch2_pad", "ragged_sharp", "single_row"])
@pytest.mark.parametrize("precision", PRECISIONS)
def test_model_col_weights_vs_oracle(pkg, golden_dir, name, precision):
    g, (ref_full, ref_mean) = model_ref(golden_dir, name)
    layers = int(g["layers"])
    vocab = pkg.Vocab(pkg.Alphabet())
    model = pkg.MSATransformer(vocab, num_layers=layers, precision=precision)
    model.load_state_dict(O.make_weights(int(g["wseed"]), num_layers=layers, sharpen=float(g["sharpen"])), strict=True)
    model = model.eval().cuda()
    tokens = torch.from_numpy(g["tokens"].astype(np.int64)).cuda()
    base = model(tokens, repr_layers=[0, 1, layers], need_head_weights=True)
    out = model(tokens, repr_layers=[0, 1, layers], need_head_weights=True, need_col_weights=True,
                need_col_weights_mean=True)
    B, R, Cc = tokens.shape
    assert tuple(out["col_attentions"].shape) == (B, layers, 12, Cc, R, R)
    assert tuple(out["col_attentions_mean"].shape) == (B, layers, 12, R, R)
    if R == 1:
        assert bool((out["col_attentions"] == 1).all()) and bool((out["col_attentions_mean"] == 1).all())
    tol = tols(precision, sharp_deep=float(g["sharpen"]) >= 3 and layers >= 10)
    e = (rel(out["col_attentions"], ref_full), rel(out["col_attentions_mean"], ref_mean))
    print(f"[{name}/{precision}] col {e[0]:.3e} mean {e[1]:.3e}")
    assert max(e) < tol
    # every other output is bit-identical to the call without the keywords
    assert torch.equal(out["logits"], base["logits"]) and torch.equal(out["row_attentions"], base["row_attentions"])
    for l in (0, 1, layers):
        assert torch.equal(out["representations"][l], base["representations"][l])
    # either keyword alone, without need_head_weights, gives the same numbers
    only = model(tokens, need_col_weights_mean=True, want_logits=False)
    assert "row_attentions" not in only and "col_attentions" not in only
    assert torch.equal(only["col_attentions_mean"], out["col_attentions_mean"])


# ------------------------------------------------------------------------------------------ at size
def _one_layer(pkg, R, Cc, seed, embed_positions_msa=True):
    vocab = pkg.Vocab(pkg.Alphabet())
    model = pkg.MSATransformer(vocab, num_layers=1, embed_positions_msa=embed_positions_msa, precision="fp16")
    model.load_state_dict(O.make_weights(seed, num_layers=1, embed_positions_msa=embed_positions_msa), strict=True)
    return model.eval().cuda(), O.make_tokens(R, Cc, seed, pad_cols=3).cuda()


def test_mean_equals_full_mean_cfg1(pkg):
    """512 x 36 (BASELINE config 1's shape): the mean output is the column mean of the full output."""
    model, tokens = _one_layer(pkg, 512, 36, 5)
    out = model(tokens, need_col_weights=True, need_col_weights_mean=True, want_logits=False)
    full, mean = out["col_attentions"], out["col_attentions_mean"]
    assert rel(mean, full.double().mean(3)) < 1e-6
    assert (full.sum(-1) - 1).abs().max().item() < 1e-5


@pytest.mark.parametrize("R,Cc", [(512, 256), (4096, 128)])
def test_mean_alone_at_size(pkg, L, R, Cc):
    """The mean without the full tensor (which would take 3 GB per layer at 512 x 256 and 64 GB at 4096 x 128):
    per op against float64 references on sampled (h, i) rows, in the column-major layout the layer uses; at model
    level, one layer's mean rows sum to one and x is bit-identical to the forward without the keyword."""
    H = 12
    qkv, q64 = make_qkv(R, Cc, H, L.F16, L, R + Cc)
    pad = torch.zeros(R, Cc, dtype=torch.uint8, device="cuda")
    pad[-3:, :] = 1
    pad[:, -2:] = 1
    _, mean = col_probs(L, qkv.transpose(0, 1).contiguous(), R, Cc, H, L.F16, 1, pad, full=False)
    del qkv
    D = H * 64
    g = torch.Generator().manual_seed(1)
    for h, i in zip(torch.randint(0, H, (6,), generator=g).tolist(), torch.randint(0, R, (6,), generator=g).tolist()):
        q = q64[i, :, h * 64:(h + 1) * 64]                                  # [C, 64]
        k = q64[:, :, D + h * 64:D + (h + 1) * 64]                          # [R, C, 64]
        s = torch.einsum("cd,jcd->cj", q, k).masked_fill(pad.T.bool(), -10000)
        ref = s.softmax(-1).mean(0)
        assert rel(mean[h, i], ref) <= PROBS_TOL
    del q64
    model, tokens = _one_layer(pkg, R, Cc, 9, embed_positions_msa=False)
    base = model(tokens, repr_layers=[1], want_logits=False)
    out = model(tokens, repr_layers=[1], want_logits=False, need_col_weights_mean=True)
    assert torch.equal(out["representations"][1], base["representations"][1])
    m = out["col_attentions_mean"]
    assert tuple(m.shape) == (1, 1, H, R, R) and (m.sum(-1) - 1).abs().max().item() < 1e-5


# ------------------------------------------------------------------------------------------ no regression
@pytest.mark.parametrize("precision", ["fp32", "fp16"])
def test_col_probs_entry_with_null_outputs_is_the_plain_forward(pkg, L, precision):
    """rnamsm_msa_forward_col_probs with both outputs NULL: bit-identical x / maps and the same launch count."""
    model, tokens = _one_layer(pkg, 24, 40, 4)
    model.set_precision(precision)
    code = L.forward_code(precision)
    m = model.c_weights(L.dtype_code(precision))
    R, Cc, D, H, N = 24, 40, 768, 12, 1
    nbytes = L.lib.rnamsm_workspace_bytes(R, Cc, D, H, 4 * D, code) + ((R * Cc + 255) // 256) * 256
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    tok = tokens[0].contiguous()
    res = []
    for fn in ("rnamsm_msa_forward", "rnamsm_msa_forward_col_probs"):
        x = torch.empty(R * Cc, D, device="cuda")
        maps = torch.empty(N, H, Cc, Cc, device="cuda")
        reps = (C.c_void_p * (N + 1))()
        extra = (None, None) if fn.endswith("col_probs") else ()
        before = L.lib.rnamsm_launch_count()
        L.check(getattr(L.lib, fn)(C.byref(m), L.ptr(tok), R, Cc, 1, code, L.ptr(x), L.ptr(maps), *extra, reps, None,
                                   L.ptr(ws), nbytes, L.stream_ptr()), fn)
        torch.cuda.synchronize()
        res.append((x, maps, L.lib.rnamsm_launch_count() - before))
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1]) and res[0][2] == res[1][2]
