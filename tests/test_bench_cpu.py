"""CPU: bench.py's host-side pieces -- FLOP model, cfg3 task-farm assignment, and the reference arm's JSON
contract (``--impl reference`` runs the oracle port on the host cores; no GPU needed)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402
from oracle import msa_ref as O  # noqa: E402


def test_flop_model_matches_survey_totals():
    # SURVEY.md 8d: cfg2 27.99 TF, cfg4 167.6 TF, cfg5 265.1 TF (the LM head's 0.6 % is not in the per-class split)
    for (R, C), want in (((512, 256), 27.99e12), ((4096, 128), 167.6e12), ((1024, 1024), 265.1e12)):
        assert abs(O.flops(R, C) - want) / want < 2e-3
        assert abs(bench.total_flops(R, C) - O.flops(R, C)) / want < 1e-12
        by_class = sum(bench.flops_breakdown(R, C).values())
        assert 0.99 < by_class / O.flops(R, C) <= 1.0


def test_cfg3_farm_assignment_is_balanced_and_complete():
    lens = bench.cfg3_lengths()
    assert len(lens) == 64 and all(51 <= c <= 501 for c in lens) and lens == bench.cfg3_lengths()
    costs = [O.flops(256, c) for c in lens]
    for world in (1, 2, 4, 8):
        jobs = bench.lpt_assign(costs, world)
        assert sorted(i for j in jobs for i in j) == list(range(64))
        loads = [sum(costs[i] for i in j) for j in jobs]
        assert max(loads) / (sum(loads) / world) < 1.05          # LPT keeps the slowest rank within 5 % of the mean


def test_measured_arm_does_not_import_the_oracle():
    """Only the CPU-baseline leg may touch oracle/ (the product path must not route through it)."""
    src = open(os.path.join(ROOT, "bench.py")).read()
    body = src[src.index("def run_ours("):src.index("def main(")]
    assert "from oracle" not in body and "import oracle" not in body and "msa_ref" not in body
    t = bench.synthetic_tokens(5, 7, 1)
    assert t.shape == (1, 5, 7) and int(t[0, :, 0].abs().sum()) == 0 and int(t[0, :, 1:].min()) >= 4 and int(t.max()) <= 10


def test_product_tree_never_imports_the_oracle():
    """The package, the kernels' build script and tools/ must not import, link or execute anything under oracle/
    (only tests/, __graft_entry__.smoke() and bench's CPU legs may)."""
    import glob
    import re
    files = (glob.glob(os.path.join(ROOT, "rna-msm_b200", "**", "*.py"), recursive=True)
             + glob.glob(os.path.join(ROOT, "rna-msm_b200", "csrc", "*"))
             + glob.glob(os.path.join(ROOT, "tools", "**", "*.py"), recursive=True)
             + glob.glob(os.path.join(ROOT, "include", "*.h")))
    assert len(files) > 20
    pat = re.compile(r"^\s*(from\s+oracle|import\s+oracle)|oracle[./]msa|msa_ref|msa_ingest_ref", re.M)
    bad = [f for f in files if os.path.isfile(f) and pat.search(open(f, errors="replace").read())]
    assert not bad, bad


def test_reference_arm_json_contract():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup",
                        "0", "--workload", "cfg1"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "tokens/s" and line["higher_is_better"] is True
    assert line["metric"] == bench.METRIC and line["value"] > 0 and line["n_gpus"] == 1
    from oracle import build_ref
    assert line["cpu_baseline"]["kind"] == ("reference" if build_ref.available() else "port")
    assert line["cpu_baseline"]["cores"] >= 1
    # the sample time is what ms_per_step reports; the x10 extrapolation has its own fields
    assert line["extrapolated_from_layers"] == 1 and line["ms_per_forward_extrapolated"] > line["ms_per_step"]
    assert abs(line["value"] - line["config"]["tokens_per_step"] / (line["ms_per_forward_extrapolated"] * 1e-3)) < 1e-6 * line["value"]
    assert {"workload", "R", "C", "tokens_per_step", "layers"} <= set(line["config"])
    assert line["e2e"] == {"value": line["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"]


def test_both_arms_print_the_same_config_keys():
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert src.count("_config(desc, R, C, tokens") >= 2     # run_reference and run_ours build `config` the same way
    a = bench._config("w", 1, 2, 3, batch_tokens=None, tokens_per_step_scope="x", precision="p", parallelism="q", l2="r")
    assert list(a)[:5] == ["workload", "R", "C", "tokens_per_step", "layers"]
