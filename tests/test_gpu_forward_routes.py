"""Every route of the whole forward at its dispatch boundaries, against float64, and the process-level switches against
the default, bit for bit (tests/forward_routes.py has the route mirror, the shapes and the child runner).

Gates are the project's (tests/test_gpu_model.py): fp32 1e-4, tf32x3 1e-3, the 16-bit gate 2e-2 on representations,
logits and maps, and for bf16 the maps envelope 6e-2; both 16-bit modes keep the row-argmax of >= 99 % of the maps'
rows (the seeded weights are sharpened, so the maps are not near-uniform).  Routes measured far below those gates are
held to tighter ones (ROUTE_GATES, with the measured values).  Errors are norm-relative (max |d| / max |ref|)
against O.forward of the same weights in float64, run on the device.
"""
import os
import subprocess
import sys

import pytest
import torch

import forward_routes as FR
from oracle import msa_ref as O

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-4
TF32X3_TOL = 1e-3
F16_TOL = 2e-2
BF16_MAP_TOL = 6e-2
ARGMAX_MIN = 0.99
GATES = {"fp32": (FP32_TOL, FP32_TOL), "tf32x3": (TF32X3_TOL, TF32X3_TOL), "fp16": (F16_TOL, F16_TOL),
         "bf16": (F16_TOL, BF16_MAP_TOL)}          # (representations and logits, maps)
# Routes that measure far below their precision's gate get a tighter one: (precision, row, col) -> (representations and
# logits, maps), about three times the worst value over the cases of that route, measured on an NVIDIA B200 at a
# 1000 W power limit (the kernels are deterministic, so the values repeat).  Measured worst in the comments.
ROUTE_GATES = {
    ("fp32", "f32", "f32"): (1e-5, 4e-5),          # 1.9e-6, 1.1e-5 (64 x 257)
    ("fp32", "f32", "r1"): (1e-5, 1e-5),           # 1.2e-6, 1.9e-6
    ("tf32x3", "f32", "f32"): (1e-4, 5e-4),        # 2.9e-5, 1.5e-4 (300 x 33)
    ("tf32x3", "f32", "r1"): (1e-4, 1e-4),         # 1.5e-5, 3.1e-5
    ("fp16", "short", "umma"): (3e-3, 1.2e-2),     # 9.4e-4, 3.8e-3 (128 x 128)
    ("fp16", "short", "fa"): (3e-3, 2e-2),         # 1.0e-3, 7.9e-3 (300 x 33)
    ("fp16", "chain", "umma"): (3e-3, 1e-2),       # 6.9e-4, 2.9e-3 (64 x 257)
    ("fp16", "chain", "fa"): (3e-3, 1.5e-2),       # 9.0e-4, 4.4e-3 (129 x 129)
    ("fp16", "chain", "r1"): (3e-3, 5e-3),         # 5.9e-4, 1.3e-3
    ("bf16", "short", "umma"): (2e-2, 3.5e-2),     # 5.4e-3, 1.1e-2 (128 x 9)
    ("bf16", "short", "fa"): (2e-2, 6e-2),         # 4.7e-3, 1.7e-2 (300 x 33)
    ("bf16", "chain", "umma"): (2e-2, 3e-2),       # 4.3e-3, 8.1e-3 (64 x 257)
    ("bf16", "chain", "fa"): (2e-2, 4e-2),         # 4.9e-3, 1.3e-2 (129 x 129)
    ("bf16", "chain", "r1"): (2e-2, 1e-2),         # 5.1e-3, 3.2e-3
}
assert all(t <= GATES[p][0] and m <= GATES[p][1] for (p, _, _), (t, m) in ROUTE_GATES.items())
ROW_SUM_TOL = 1e-5
# RNAMSM_ROW_SHORT=0 against the default.  Both row attentions evaluate the same maps from the same first-layer q|k|v, but
# they split the sum over the R rows differently (row chunks of row_attn_short.cu, split-K count of the tied-logit GEMM),
# so their fp32 partial sums round differently.  Each route keeps its maps within the per-op float64 bound 2e-5
# (tests/test_gpu_ops.py test_row_attention_short), so the two agree within twice that, not within the 1e-6 that holds
# when both softmaxes read the same partial sums (measured 1.8e-5 at 300 x 33).  Every output after them inherits the
# context difference and is held to the per-op context bound of the activation type (the same test's tol(): fp16 2e-3,
# bf16 1e-2; the tied row block itself is fp16 in both modes).  Measured on the B200 above: 1.2e-3 (fp16, column
# probabilities at 129 x 9), 4.2e-3 (bf16, logits at 128 x 128).
SHORT_MAP_TOL = 4e-5
SHORT_OUT_TOL = {"fp16": 2e-3, "bf16": 1e-2}

REPORT = []


@pytest.fixture(scope="module")
def pkg():
    import rnamsm_b200
    return rnamsm_b200


@pytest.fixture(scope="module")
def model_for(pkg):
    cache = {}

    def get(precision):
        if precision not in cache:
            cache[precision] = FR.build_model(pkg, precision)
        return cache[precision]
    return get


@pytest.fixture(scope="module")
def ref_for():
    """float64 reference per case, computed once on the device and shared by every precision (one case kept at a time)."""
    sd64 = FR.weights(torch.float64)
    sd64 = {k: v.cuda() for k, v in sd64.items()}
    cache = {}

    def get(case):
        if case.name not in cache:
            cache.clear()
            cache[case.name] = FR.reference(case.tokens(), sd64, device="cuda")
        return cache[case.name]
    return get


def same_bits(a, b):
    if a.dtype != b.dtype or a.shape != b.shape:
        return False
    view = {1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}[a.element_size()]
    return torch.equal(a.contiguous().view(view), b.contiguous().view(view))


def max_diff(a, b):
    return float((a.double() - b.double()).abs().max()) if a.numel() else 0.0


def argmax_agreement(maps, ref_maps, skip_queries):
    """Share of map rows whose argmax key agrees, over the query columns not in skip_queries (columns padded in every
    row: their logits are exactly 0 and the row is uniform, a tie in any precision)."""
    keep = ~skip_queries
    a = maps[..., keep, :].reshape(-1, maps.shape[-1])
    b = ref_maps[..., keep, :].reshape(-1, maps.shape[-1])
    return float((a.argmax(-1) == b.argmax(-1)).double().mean()) if a.shape[0] else 1.0


def structural_checks(case, tokens, got, ref, tol):
    """Finite outputs, map rows summing to 1, masked keys at exactly 0, pad tokens' representations as the oracle's."""
    for k, v in got.items():
        assert torch.isfinite(v).all(), f"{case}: non-finite {k}"
    maps = got["maps"]
    assert float((maps.double().sum(-1) - 1).abs().max()) <= ROW_SUM_TOL, f"{case}: a map row does not sum to 1"
    key_pad = tokens[0, 0].eq(O.PAD_IDX).cuda()              # the key mask comes from MSA row 0
    if key_pad.any():
        assert float(maps[..., key_pad].abs().max()) == 0.0, f"{case}: probability on a masked key column"
    pad = tokens[0].eq(O.PAD_IDX).cuda()
    if pad.any():
        assert float(got["rep0"][0][pad].abs().max()) == 0.0, f"{case}: embedding of a pad token is not 0"
        for k in ("rep1", "rep2", "logits"):
            e = O.rel_err(got[k][0][pad], ref[k][0][pad])
            assert e < tol, f"{case}: {k} of the pad tokens {e:.3e} >= {tol:g}"


def ref_outputs(ref):
    reps = ref["representations"]
    return {"rep0": reps[0], "rep1": reps[1], "rep2": reps[FR.LAYERS], "logits": ref["logits"], "maps": ref["row_attentions"]}


def errors_vs_reference(tokens, got, ref):
    want = ref_outputs(ref)
    errs = {k: O.rel_err(got[k], want[k]) for k in ("rep0", "rep1", "rep2", "logits", "maps")}
    all_pad = tokens[0].eq(O.PAD_IDX).all(0).cuda()
    agree = argmax_agreement(got["maps"], want["maps"], all_pad)
    return errs, agree


def check_gates(tag, errs, agree, precision, tol, map_tol):
    assert errs["rep0"] < 1e-5, f"{tag}: embedding {errs['rep0']:.3e}"          # fp32 in every mode
    for k in ("rep1", "rep2", "logits"):
        assert errs[k] < tol, f"{tag}: {k} {errs[k]:.3e} >= {tol:g}"
    assert errs["maps"] < map_tol, f"{tag}: maps {errs['maps']:.3e} >= {map_tol:g}"
    if precision in FR.SIXTEEN:
        assert agree >= ARGMAX_MIN, f"{tag}: row-argmax agreement {agree:.4f}"


# ------------------------------------------------------------------------------------------ switches, in child processes
def run_child(name, out_dir):
    path = os.path.join(str(out_dir), f"{name}.pt")
    r = subprocess.run(FR.child_command(path), env=FR.child_env(name), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, f"child {name} failed:\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}"
    out = torch.load(path)
    os.remove(path)
    switches = out.pop("switches")
    assert switches == {k: FR.CHILD_ENVS[name].get(k, "") for k in FR.SWITCHES}, switches
    return out


@pytest.fixture(scope="module")
def default_outputs(pkg, tmp_path_factory):
    """The child list under the default switches: in this process unless a switch is set in its environment."""
    if any(os.environ.get(k) for k in FR.SWITCHES):
        return run_child("default", tmp_path_factory.mktemp("default"))
    return FR.child_outputs(pkg)


def differing(child, parent):
    assert child.keys() == parent.keys(), sorted(set(child) ^ set(parent))
    return {k: max_diff(child[k], parent[k]) for k in parent if not same_bits(child[k], parent[k])}


@pytest.mark.parametrize("name", ["fuse_ln", "pdl"])
def test_switch_is_bit_identical(default_outputs, name, tmp_path):
    """RNAMSM_FUSE_LN=1 (every LayerNorm behind a residual GEMM computed in that GEMM's epilogue, the next layer's first
    LayerNorm in fc2's, xn_ready chaining in forward, forward_batch and the layer-by-layer streamed extraction) and
    RNAMSM_PDL=1 (programmatic dependent launch) change no bit of any output."""
    bad = differing(run_child(name, tmp_path), default_outputs)
    print(f"[{name}] {len(default_outputs)} outputs compared, {len(bad)} differ")
    assert not bad, f"{name}: outputs differ from the default run (max |d|): {bad}"


def test_row_short_off_matches_default_and_float64(default_outputs, ref_for, tmp_path):
    """RNAMSM_ROW_SHORT=0 runs the three-kernel chain where the one-launch row attention would run (C <= 128).  Shapes
    above 128 columns take the chain either way and must not change at all; the others must keep the first layer's maps
    within SHORT_MAP_TOL of the default, every output within the context bound SHORT_OUT_TOL, and the forward within
    the float64 gates of its precision."""
    child = run_child("row_short0", tmp_path)
    assert child.keys() == default_outputs.keys()
    changed, first, rest = [], {}, {}
    for key, want in default_outputs.items():
        precision, _, name, out = key.split("/")
        C = int(name.split("-")[0].split("x")[1])
        got = child[key]
        if C > FR.SHORT_MAX_C:
            if not same_bits(got, want):
                changed.append(key)
            continue
        if out in ("maps", "atp"):
            first[key] = O.rel_err(got[:, 0], want[:, 0]) if out == "maps" else O.rel_err(got[:FR.H], want[:FR.H])
        rest.setdefault(precision, {})[key] = O.rel_err(got, want)
    k0 = max(first, key=first.get)
    print(f"[row_short0] worst vs default: first-layer maps {first[k0]:.3e} ({k0})")
    for precision, errs in rest.items():
        k1 = max(errs, key=errs.get)
        print(f"[row_short0] worst vs default, {precision}: {errs[k1]:.3e} ({k1})")
    assert not changed, f"changed although the chain runs in both configurations: {changed}"
    assert first[k0] < SHORT_MAP_TOL
    for precision, errs in rest.items():
        assert max(errs.values()) < SHORT_OUT_TOL[precision], precision
    for name in FR.CHILD_CASES:
        case = FR.CASE[name]
        tokens = case.tokens()
        ref = ref_for(case)
        for precision in FR.SIXTEEN:
            got = {k: child[f"{precision}/forward/{name}/{k}"].cuda() for k in ("rep0", "rep1", "rep2", "logits", "maps")}
            errs, agree = errors_vs_reference(tokens, got, ref)
            print(f"[row_short0 {name}/{precision}] " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()) +
                  f" argmax {agree:.4f}")
            check_gates(f"row_short0 {name}/{precision}", errs, agree, precision, *GATES[precision])


# ------------------------------------------------------------------------------------------ forward_batch across boundaries
@pytest.mark.parametrize("precision", FR.SIXTEEN)
def test_forward_batch_across_boundaries(pkg, model_for, precision):
    """One forward_batch list with chain and one-launch row attention, umma and flash column attention, R = 128 and
    padded rows: every member bit-identical to its own forward."""
    model = model_for(precision)
    L = pkg._lib
    toks = [c.tokens().cuda() for c in FR.BATCH_MEMBERS]
    kinds = {(r["row"], r["col"]) for r in (FR.routes(c.R, c.C, precision, L.lib) for c in FR.BATCH_MEMBERS)}
    assert {"short", "chain"} <= {k[0] for k in kinds} and {"umma", "fa"} <= {k[1] for k in kinds}
    outs = model.forward_batch(toks, need_head_weights=True)
    for c, t, o in zip(FR.BATCH_MEMBERS, toks, outs):
        one = model(t, repr_layers=[FR.LAYERS], need_head_weights=True, want_logits=False)
        assert same_bits(o["representations"][FR.LAYERS], one["representations"][FR.LAYERS]), f"{c}: representations"
        assert same_bits(o["row_attentions"], one["row_attentions"]), f"{c}: maps"


# ------------------------------------------------------------------------------------------ every route against float64
ROUTE_CASES = [(c, p) for c in FR.CASES for p in FR.PRECISIONS]


@pytest.mark.parametrize("case,precision", ROUTE_CASES, ids=[f"{c.name}-{p}" for c, p in ROUTE_CASES])
def test_route_vs_float64(pkg, model_for, ref_for, case, precision):
    L = pkg._lib
    route = FR.routes(case.R, case.C, precision, L.lib)
    assert route == FR.routes(case.R, case.C, precision), "the Python dispatch mirror disagrees with the library"
    tokens = case.tokens()
    got = FR.forward_outputs(model_for(precision), tokens)
    ref = ref_for(case)
    errs, agree = errors_vs_reference(tokens, got, ref)
    tol, map_tol = ROUTE_GATES.get((precision, route["row"], route["col"]), GATES[precision])
    REPORT.append((case.name, precision, route, errs, agree, (tol, map_tol)))
    print(f"[{case.name}/{precision}] {route} " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()) + f" argmax {agree:.4f}")
    structural_checks(f"{case.name}/{precision}", tokens, got, ref_outputs(ref), GATES[precision][0])
    check_gates(f"{case.name}/{precision}", errs, agree, precision, tol, map_tol)


def test_zz_report():
    """The measured error of every route, with the shape that exercised it and the card it ran on."""
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    print(f"\nforward routes on {name}, power limit {power}")
    print("| shape | pad | precision | row | col | q/k/v | dense | rep1 | rep2 | logits | maps | argmax | gates |")
    print("|---|---|---|---|---|---|---|---|---|---|---|---|---|")
    for cname, precision, r, e, agree, (tol, map_tol) in REPORT:
        shape, pad = cname.split("-")
        print(f"| {shape} | {pad} | {precision} | {r['row']} | {r['col']} | {r['qkv']} | {r['dense']} | {e['rep1']:.1e} | "
              f"{e['rep2']:.1e} | {e['logits']:.1e} | {e['maps']:.1e} | {agree:.4f} | {tol:g} / {map_tol:g} |")
    worst = {}
    for _, precision, r, e, _, _ in REPORT:
        k = (precision, r["row"], r["col"])
        worst[k] = max(worst.get(k, 0.0), max(e[x] for x in ("rep1", "rep2", "logits", "maps")))
    for k, v in sorted(worst.items()):
        print(f"worst {k}: {v:.2e}")
