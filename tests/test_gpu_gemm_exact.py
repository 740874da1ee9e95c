"""GPU: the tensor-core GEMM (csrc/umma_gemm.cu), the FFMA kernels of the fp32 path (csrc/simt_f32.cu) and phase 1 of
the one-launch short row attention (csrc/row_attn_short.cu) on exact operands, compared with float64 over the whole
output and with no tolerance (tests/gemm_exact.py).

Every call goes through the C ABI into a NaN-filled output with NaN guards before and after it; the guards must come back
untouched and every output element must equal the float64 value rounded once to the output type (zeros compare by
value).  The 16-bit and fp32 erf-GELU epilogues are not exact and are held to ulp_out(|gelu64(a)|) + 2^-20 |a| on the
exact pre-activation a.

  - rnamsm_linear: every dtype x epilogue over M, N, K and q_cols tails, plus shapes whose persistent tile count is
    P w - 1, P w + 1 and >= 3 P for the device's pair count P (second tiles per pair, both accumulator buffers, operand
    rings that wrap across tiles, q scale and row mask on later waves); rnamsm_linear_tf32 at the same shapes.
  - rnamsm_row_attn_logits: each split's slab against its own row range, for the three kBN instances and their tails.
  - rnamsm_row_attn_av: 4-row N tiles, 2 rows per CTA, padding columns of P holding NaN.
  - rnamsm_row_attn_short phase 1: each chunk's slab.
  - Two child processes with RNAMSM_GEMM_PAIRS=1, RNAMSM_GELU_WIDE=0, RNAMSM_AV_WIDE=0 and RNAMSM_GEMM_PAIRS=3,
    RNAMSM_PDL=1 (read once per process): their outputs must be bit-identical to this process's.

284 cases; 15 s on a B200 at a 1000 W power limit, of which the two child processes take about 4 s each.
"""
import os
import subprocess
import sys

import pytest
import torch

import gemm_exact as GE

pytestmark = pytest.mark.gpu

GELU_WORST = {}


@pytest.fixture(scope="module")
def L():
    from rnamsm_b200 import _lib
    _lib.device_check(torch.device("cuda:0"))
    return _lib


@pytest.fixture(scope="module")
def P(L):
    return L.lib.rnamsm_gemm_pairs()


def n_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def mismatches(got, want):
    bad = got != want
    return f"{int(bad.sum())} of {bad.numel()} elements differ"


def check_linear(out, x, W, bias, code, epi, q_cols, mask, resid, what):
    torch.cuda.synchronize()
    assert out.intact(), f"{what}: a write outside the output"
    if epi == 1:
        worst = GE.gelu_excess(out.body, GE.dense_preact(x, W, bias), code)
        GELU_WORST[code] = max(GELU_WORST.get(code, 0.0), worst)
        print(f"[{what}] GELU worst {worst:.3f} of the gate")
        assert worst <= 1.0, f"{what}: GELU outside the gate ({worst:.3f})"
    else:
        want = GE.dense_ref(x, W, bias, epi, GE.Q_SCALE, q_cols, mask, resid).to(out.body.dtype)
        assert torch.equal(out.body, want), f"{what}: {mismatches(out.body, want)}"


def linear_once(L, M, N, K, code, epi, q_cols, seed, tf32=False):
    x, W, bias = GE.exact_gemm_operands(M, N, K, seed=seed, device="cuda")
    mask = GE.row_mask_for(M, seed) if q_cols else None
    resid = GE.exact_affine((M, N), seed + 1, device="cuda") if epi == 2 else None
    out = GE.run_linear(L, x, W, bias, code, epi, GE.Q_SCALE, q_cols, mask, resid, tf32=tf32)
    check_linear(out, x, W, bias, code, epi, q_cols, mask, resid, f"{'tf32 ' if tf32 else ''}{M}x{N}x{K} code {code} epi {epi} "
                 f"q_cols {q_cols}")


# ------------------------------------------------------------------------------------------ rnamsm_linear
LINEAR = GE.linear_cases()


@pytest.mark.parametrize("c", LINEAR, ids=[f"{c['M']}x{c['N']}x{c['K']}-c{c['code']}-e{c['epi']}-q{c['q_cols']}" for c in LINEAR])
def test_linear_exact(L, c):
    linear_once(L, c["M"], c["N"], c["K"], c["code"], c["epi"], c["q_cols"], seed=c["M"] + c["N"])


@pytest.mark.parametrize("target", GE.WAVE_TARGETS)
@pytest.mark.parametrize("epi", GE.EPIS, ids=["bias", "gelu", "resid"])
@pytest.mark.parametrize("code", GE.CODES, ids=["f32", "bf16", "f16"])
def test_linear_multiwave(L, P, code, epi, target):
    M, N, K, tiles, w = GE.multiwave_case(P, epi, target)
    GE.check_wave_counts(GE.tiles_per_pair(tiles, P), target, w, P)
    linear_once(L, M, N, K, code, epi, N // 3 if epi == 0 else 0, seed=17)


@pytest.mark.parametrize("target", GE.WAVE_TARGETS)
@pytest.mark.parametrize("epi", GE.EPIS, ids=["bias", "gelu", "resid"])
def test_linear_tf32_multiwave(L, P, epi, target):
    """tf32-representable operands: the lo halves are 0 and the three MMAs per k-step add exact terms."""
    M, N, K, tiles, w = GE.multiwave_case(P, epi, target)
    GE.check_wave_counts(GE.tiles_per_pair(tiles, P), target, w, P)
    linear_once(L, M, N, K, 0, epi, N // 3 if epi == 0 else 0, seed=19, tf32=True)


# ------------------------------------------------------------------------------------------ tied logits
@pytest.mark.parametrize("code", GE.CODES, ids=["f32", "bf16", "f16"])
@pytest.mark.parametrize("C,H,R", GE.TIED_CASES, ids=[f"C{c}-H{h}-R{r}" for c, h, r in GE.TIED_CASES])
def test_row_attn_logits_each_split(L, C, H, R, code):
    qkv = GE.exact_qkv(R, C, H, seed=23, device="cuda")
    default = L.lib.rnamsm_row_attn_splits(R, C, H, code)
    for ns in sorted({1, default, 3, R}):
        if not GE.valid_splits(R, ns):
            continue
        out = GE.run_logits(L, qkv, R, C, H, code, ns)
        want = GE.tied_split_refs(qkv, R, C, H, ns)
        torch.cuda.synchronize()
        assert out.intact(), f"splits={ns}: a write outside the slabs"
        for s in range(ns):
            assert torch.equal(out.body[s].double(), want[s]), f"splits={ns} slab {s}: {mismatches(out.body[s].double(), want[s])}"


# ------------------------------------------------------------------------------------------ tied A V
AV = GE.av_cases()


@pytest.mark.parametrize("code", GE.CODES, ids=["f32", "bf16", "f16"])
@pytest.mark.parametrize("c", AV, ids=[f"R{c['R']}-C{c['C']}-H{c['H']}-ldp{c['ldp']}" for c in AV])
def test_row_attn_av(L, c, code):
    R, C, H, ldp = c["R"], c["C"], c["H"], c["ldp"]
    qkv = GE.exact_qkv(R, C, H, seed=29, device="cuda")
    P = GE.exact_probs(H, C, ldp, seed=31, device="cuda")            # columns [C, ldp) are NaN: never read
    out = GE.run_av(L, P, ldp, qkv, R, C, H, code)
    want = GE.av_ref(P, qkv, R, C, H).to(out.body.dtype)
    torch.cuda.synchronize()
    assert out.intact(), "a write outside ctx"
    assert torch.equal(out.body, want), mismatches(out.body, want)


# ------------------------------------------------------------------------------------------ row_attn_short, phase 1
@pytest.mark.parametrize("code", [1, 2], ids=["bf16", "f16"])
@pytest.mark.parametrize("C,H,R", GE.SHORT_CASES, ids=[f"C{c}-H{h}-R{r}" for c, h, r in GE.SHORT_CASES])
def test_row_attn_short_each_chunk(L, C, H, R, code):
    qkv = GE.exact_qkv(R, C, H, seed=37, device="cuda")
    default = L.lib.rnamsm_row_attn_short_chunks(R, C, H)
    assert default >= 1
    for nc in GE.short_chunk_options(R, H, default, n_sms()):
        out = GE.run_short(L, qkv, R, C, H, code, nc)
        want = GE.tied_split_refs(qkv, R, C, H, nc)
        torch.cuda.synchronize()
        assert out.intact(), f"chunks={nc}: a write outside the partials"
        for s in range(nc):
            assert torch.equal(out.body[s].double(), want[s]), f"chunks={nc} chunk {s}: {mismatches(out.body[s].double(), want[s])}"


# ------------------------------------------------------------------------------------------ other configurations
CHILD_ENVS = {"pairs1_narrow": {"RNAMSM_GEMM_PAIRS": "1", "RNAMSM_GELU_WIDE": "0", "RNAMSM_AV_WIDE": "0"},
              "pairs3_pdl": {"RNAMSM_GEMM_PAIRS": "3", "RNAMSM_PDL": "1"}}


@pytest.fixture(scope="module")
def parent_outputs(L):
    return GE.child_cases(L)


@pytest.mark.parametrize("name", list(CHILD_ENVS))
def test_other_configuration_is_bit_identical(L, parent_outputs, name, tmp_path):
    """The switches are read once per process, so each configuration runs in a child process of its own (killed if it
    outlives the timeout).  Each output element is computed by one tile in a fixed k order with the same epilogue
    arithmetic, whatever the pair count, the epilogue width or PDL: the outputs must match this process's bit for bit."""
    env = dict(os.environ)
    for k in ("RNAMSM_GEMM_PAIRS", "RNAMSM_GELU_WIDE", "RNAMSM_AV_WIDE", "RNAMSM_PDL"):
        env.pop(k, None)
    env.update(CHILD_ENVS[name])
    path = tmp_path / "outputs.pt"
    script = os.path.join(os.path.dirname(os.path.abspath(GE.__file__)), "gemm_exact.py")
    r = subprocess.run([sys.executable, script, str(path)], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, f"child {name} failed:\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}"
    child = torch.load(path)
    assert int(child.pop("pairs")[0]) == int(CHILD_ENVS[name]["RNAMSM_GEMM_PAIRS"])
    assert child.keys() == parent_outputs.keys()
    for k, want in parent_outputs.items():
        assert GE.same_bits(child[k], want), f"{name}: {k} differs from the default configuration"


def test_zz_report_gelu_worst():
    """The worst GELU error observed in this run, in units of the gate."""
    print(f"GELU worst of the gate per output dtype: {GELU_WORST}")
    assert all(v <= 1.0 for v in GELU_WORST.values())
