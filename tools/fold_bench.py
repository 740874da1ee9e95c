"""Cost of folding pair maps (rnamsm_b200.fold_pairs): per-stage device times, the max-plus rate, and the float32 numpy
restatement's host time.

    python tools/fold_bench.py [--out DIR] [--reps 5]

Workloads: one map at L = 512, 2048 and 8192, and a batch of 64 maps with L drawn from [50, 500] (the alignment
lengths of a many-short-MSA run), all seeded probability maps folded with mode "mea".  Per workload:
  - the whole call, timed with CUDA events after a warm-up call, median of --reps (it includes the allocation of the
    tables and the one host sync);
  - per-stage kernel times from one torch.profiler run of the call (CUDA activities), summed by kernel name: prep
    (fold_prep_kernel), fill (fold_fill_kernel, one launch per tile diagonal) and traceback (fold_traceback_kernel);
  - (i, j, k) triples of the recurrence, sum over maps of L^3 / 6, over the fill time.
The restatement (tests/fold_ref.py) is timed on the host at L = 512 and 1024 and its result compared with the device.
The GPU's name and power limit are read in the same run.  Prints one JSON line per workload; with --out, also writes
them to DIR/fold_bench.jsonl.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

STAGES = {"prep": "fold_prep_kernel", "fill": "fold_fill_kernel", "traceback": "fold_traceback_kernel"}


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True)
    f = [x.strip() for x in (r.stdout.strip().splitlines() or [",,,"])[0].split(",")] + ["", "", "", ""]
    return {"gpu": f[0] or torch.cuda.get_device_name(0), "power_limit": f[1], "sm_clock": f[2], "sm_clock_max": f[3]}


def prob_map(L, seed):
    """Symmetric pair probabilities, rows summing to at most 0.8 (tests/test_gpu_fold.py's generator)."""
    rng = np.random.default_rng(seed)
    S = rng.random((L, L)) ** 4
    S = S + S.T
    return (S / S.sum(axis=1).max() * 0.8).astype(np.float32)


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def stage_ms(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {k: 0.0 for k in STAGES}
    launches = {k: 0 for k in STAGES}
    for e in prof.key_averages():
        for k, name in STAGES.items():
            if name in e.key:
                out[k] += e.device_time_total / 1000.0
                launches[k] += e.count
    return out, launches


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args(argv)
    assert torch.cuda.is_available(), "fold_bench needs a CUDA device"
    import rnamsm_b200 as pkg
    import fold_ref as F

    info = gpu_info()
    rng = np.random.default_rng(0)
    workloads = [("L512", [512]), ("L2048", [2048]), ("L8192", [8192]),
                 ("batch64_L50-500", [int(x) for x in rng.integers(50, 501, size=64)])]
    rows = []
    for name, Ls in workloads:
        maps = [torch.from_numpy(prob_map(L, L)).cuda() for L in Ls]
        call = lambda: pkg.fold_pairs(maps)                                   # noqa: E731
        call()
        times = [event_ms(call) for _ in range(a.reps)]
        stages, launches = stage_ms(call)
        triples = sum(L ** 3 / 6 for L in Ls)
        row = {"workload": name, "maps": len(Ls), "L_max": max(Ls), "L_sum": sum(Ls), "call_ms": statistics.median(times),
               "call_ms_all": [round(t, 3) for t in times], **{f"{k}_ms": round(v, 4) for k, v in stages.items()},
               "fill_launches": launches["fill"], "triples": triples,
               "triples_per_s_fill": triples / (stages["fill"] / 1e3) if stages["fill"] > 0 else None, **info}
        rows.append(row)
        print(json.dumps(row), flush=True)
    for L in (512, 1024):
        S = prob_map(L, L)
        t = time.perf_counter()
        ref_pairs, ref_score = F.fold(S)
        host_s = time.perf_counter() - t
        pairs, score = pkg.fold_pairs(torch.from_numpy(S).cuda())
        row = {"workload": f"numpy_restatement_L{L}", "host_s": host_s,
               "device_equal": bool(np.array_equal(pairs.cpu().numpy(), ref_pairs) and np.float32(score) == ref_score),
               **info}
        rows.append(row)
        print(json.dumps(row), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "fold_bench.jsonl"), "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
