"""Cost of the alignment statistics (rnamsm_b200.dca_contacts): per-stage device times, achieved rates, the two
designs of the neighbour count, and the float64 numpy restatement's host time.

    python tools/dca_bench.py [--out DIR] [--reps 3] [--ref_limit 2e12]

Shapes N x L: 1176 x 35 (the size of the 2DRB_1 alignment), 10^4 x 200, 10^5 x 200 and 5000 x 1000, seeded alignments
of mutated copies of N / 4 ancestors (tests/test_gpu_dca.py's generator).  Per shape:
  - the whole call, timed with CUDA events after a warm-up call, median of --reps;
  - per-stage kernel times from one torch.profiler run of the call (CUDA activities), summed by kernel name:
      neighbour counts  dca_states, dca_neighbour_count, dca_weights        N^2 L state comparisons
      pair counts       dca_sites, dca_pairs                                N L (L - 1) / 2 weighted pair updates
      inverse           dca_potrf_*, dca_trtri, dca_lauum                    M^3 flops, M = 4L (M^3/3 each for the
                                                                            factorisation, L^-1 and L^-T L^-1)
      scores            dca_scores, jacobian_margins / total / contacts      L^2 blocks
  - the other design of the neighbour count, in the same run: the 16-bit tcgen05 GEMM (rnamsm_linear, fp16 in, fp16
    out: exact for counts up to 2048) of the one-hot rows [N, 5L] against themselves, row block by row block, timed
    with CUDA events; its threshold pass is not included (a lower bound for that design), and its counts are checked
    against the SIMT kernel's on the first block;
  - the float64 numpy restatement (tests/dca_ref.py), host time, where N^2 * 5L <= --ref_limit, and the contacts'
    error against it.
The GPU's name and power limit are read in the same run.  Prints one JSON line per shape; with --out, also writes
them to DIR/dca_bench.jsonl.
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

SHAPES = [(1176, 35), (10_000, 200), (100_000, 200), (5000, 1000)]
STAGES = {"neighbour counts": ("dca_states", "dca_neighbour_count", "dca_weights"),
          "pair counts": ("dca_sites", "dca_pairs"),
          "inverse": ("dca_potrf", "dca_trtri", "dca_lauum"),
          "scores": ("dca_scores", "jacobian_margins", "jacobian_total", "jacobian_contacts")}


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True)
    f = [x.strip() for x in (r.stdout.strip().splitlines() or [",,,"])[0].split(",")] + ["", "", "", ""]
    return {"gpu": f[0] or torch.cuda.get_device_name(0), "power_limit": f[1], "sm_clock": f[2], "sm_clock_max": f[3]}


def family(N, L, seed, mut=0.15, gap_p=0.05):
    from test_gpu_dca import family as fam
    return fam(N, L, seed, mut, gap_p)


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def stage_times(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {k: 0.0 for k in STAGES}
    other = 0.0
    for e in prof.key_averages():
        us = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
        for stage, keys in STAGES.items():
            if any(k in e.key for k in keys):
                out[stage] += us / 1000.0
                break
        else:
            other += us / 1000.0
    out["other"] = other
    return out


def gemm_design(tokens, w_ref, reps):
    """Neighbour counts as one-hot products on the tensor cores: per row block, C = X_blk X^T in fp16."""
    from rnamsm_b200 import _lib as L
    import dca_ref as D
    N, C = tokens.shape
    Lr = C - 1
    s = torch.from_numpy(D.states(tokens.cpu().numpy())).cuda()
    K = -(-5 * Lr // 64) * 64
    Np = -(-N // 64) * 64
    X = torch.zeros((Np, K), dtype=torch.float16, device="cuda")
    X[:N, :5 * Lr] = torch.nn.functional.one_hot(s, 5).reshape(N, 5 * Lr).half()
    bias = torch.zeros(Np, dtype=torch.float32, device="cuda")
    B = min(Np, 8192)
    out = torch.empty((B, Np), dtype=torch.float16, device="cuda")
    st = L.stream_ptr()

    def run():
        for r0 in range(0, N, B):
            m = min(B, N - r0)
            L.check(L.lib.rnamsm_linear(X[r0].data_ptr(), X.data_ptr(), bias.data_ptr(), m, Np, K, L.F16, L.EPI_BIAS,
                                        1.0, 0, None, out.data_ptr(), st), "linear")

    run()
    m = min(B, N)
    counts = (out[:m, :N].float() >= 0.8 * Lr).sum(1).double()
    exact = bool(torch.equal(1.0 / counts, w_ref[:m]))
    ms = statistics.median(event_ms(run) for _ in range(reps))
    return ms, exact


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=None, help="directory for dca_bench.jsonl (none: print only)")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--ref_limit", type=float, default=2e12, help="run the numpy restatement where N^2 * 5L <= this")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "dca_bench needs a CUDA device"
    import rnamsm_b200 as pkg
    import dca_ref as D
    info = gpu_info()
    print(json.dumps(info), flush=True)
    lines = []
    for N, Lr in SHAPES:
        t_np = family(N, Lr, N + Lr)
        t = torch.from_numpy(t_np).cuda()
        call = lambda: pkg.dca_contacts(t)
        res = call()                                                             # warm-up
        total = statistics.median(event_ms(call) for _ in range(a.reps))
        wt = statistics.median(event_ms(lambda: pkg.sequence_weights(t)) for _ in range(a.reps))
        st = stage_times(call)
        M = 4 * Lr
        work = {"neighbour counts": (float(N) * N * Lr, "state comparisons"),
                "pair counts": (float(N) * Lr * (Lr - 1) / 2, "pair updates"),
                "inverse": (float(M) ** 3, "flop"),
                "scores": (float(Lr) * Lr, "blocks")}
        rates = {k: (work[k][0] / (st[k] * 1e-3) if st[k] > 0 else None, work[k][1] + "/s") for k in work}
        gemm_ms, gemm_exact = gemm_design(t, res["weights"], a.reps)
        rec = {"N": N, "L": Lr, "neff": res["neff"], "call_ms": total, "seq_weights_call_ms": wt,
               "stage_ms": st, "work": work, "rate": rates,
               "neighbour_simt_ms": st["neighbour counts"], "neighbour_gemm_fp16_ms": gemm_ms,
               "gemm_counts_exact_first_block": gemm_exact, **info}
        if float(N) * N * 5 * Lr <= a.ref_limit:
            h0 = time.perf_counter()
            ref = D.dca(t_np)
            rec["numpy_ref_s"] = time.perf_counter() - h0
            got = res["contacts"].cpu().double().numpy()
            rec["contacts_err_rel_max"] = float(np.abs(got - ref["contacts"]).max() / np.abs(ref["contacts"]).max())
            rec["weights_bit_identical"] = bool(np.array_equal(res["weights"].cpu().numpy(), ref["weights"]))
        else:
            rec["numpy_ref_s"] = None
        print(json.dumps(rec), flush=True)
        lines.append(rec)
        del res
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "dca_bench.jsonl"), "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")
    print(json.dumps(gpu_info()), flush=True)


if __name__ == "__main__":
    main()
