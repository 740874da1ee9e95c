"""Cost of LM-head scoring: masked marginals of every residue of the query row, three ways.

    python tools/score_bench.py [--reps 3] [--warmup 1] [--out DIR]

Shapes, fp16, 10 layers, seeded random-init weights: 512 x 36 (the 2DRB_1 tokens, all 35 positions) and 512 x 256
(seeded tokens, all 255 positions).  Per shape, after warm-up, the three ways run alternately, ``--reps`` times each:
  (a) the user loop: forward(masked grid, want_logits=True) per position, then torch.log_softmax at that token;
  (b) MSATransformer.masked_marginals with group = 1 (token_budget = R * C);
  (c) MSATransformer.masked_marginals with the default token budget (group = plan_score_group(...)).
Each is timed with a host clock around work that ends in a device synchronise.  Reports ms per position and
positions/s (median over the repeats), with the GPU's name, power limit and SM clock read in the same run.  Asserts
that (b) and (c) are bit-identical, that their logits are bit-identical to (a)'s, and that all three log-probabilities
agree to 1e-6.  Prints one JSON line per shape between two lines of GPU state (before and after); with --out, also
writes them to DIR/score_bench.jsonl.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True)
    f = [x.strip() for x in (r.stdout.strip().splitlines() or [",,,"])[0].split(",")] + ["", "", "", ""]
    return {"gpu": f[0] or torch.cuda.get_device_name(0), "power_limit": f[1], "sm_clock": f[2], "sm_clock_max": f[3]}


def user_loop(model, t, pos, mask_idx):
    out_lp, out_lg = [], []
    for c in pos:
        m = t.clone()
        m[0, c] = mask_idx
        lg = model(m.unsqueeze(0), want_logits=True)["logits"][0, 0, c]
        out_lg.append(lg)
        out_lp.append(torch.log_softmax(lg, -1))
    return torch.stack(out_lp), torch.stack(out_lg)


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, r


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args(argv)
    import rnamsm_b200 as pkg
    torch.manual_seed(42)
    model = pkg.MSATransformer(pkg.Vocab(pkg.Alphabet()), num_layers=10, precision="fp16").eval().cuda()
    mask_idx = model.vocab.mask_idx
    g = np.load(os.path.join(ROOT, "tests", "golden", "2DRB_1.npz"))
    gen = torch.Generator().manual_seed(7)                         # uniform over A G C U X N - (4..10), BOS column
    seeded = torch.randint(4, 11, (512, 256), generator=gen, dtype=torch.int64)
    seeded[:, 0] = model.vocab.bos_idx
    shapes = [("512x36", torch.from_numpy(g["tokens"].astype(np.int64))[0]), ("512x256", seeded)]
    lines = [dict(gpu_info(), what="device")]
    print(json.dumps(lines[0]), flush=True)
    for name, t in shapes:
        t = t.cuda()
        R, Cc = t.shape
        pos = list(range(1, Cc))
        group, passes = pkg.plan_score_group(R, Cc, len(pos))
        ways = {
            "a_user_loop": lambda: user_loop(model, t, pos, mask_idx),
            "b_group1": lambda: model.masked_marginals(t, pos, token_budget=R * Cc, return_logits=True),
            "c_default": lambda: model.masked_marginals(t, pos, return_logits=True),
        }
        for _ in range(a.warmup):
            for fn in ways.values():
                fn()
        ms = {k: [] for k in ways}
        res = {}
        for _ in range(a.reps):
            for k, fn in ways.items():
                dt, res[k] = timed(fn)
                ms[k].append(dt)
        (lpa, lga), (lpb, lgb), (lpc, lgc) = res["a_user_loop"], res["b_group1"], res["c_default"]
        assert torch.equal(lpb, lpc) and torch.equal(lgb, lgc), "group 1 and the default group differ"
        assert torch.equal(lgb, lga), "masked_marginals logits differ from forward's"
        assert (lpb - lpa).abs().max().item() <= 1e-6
        row = {"what": "shape", "shape": name, "precision": "fp16", "positions": len(pos), "default_group": group,
               "default_passes": passes, "reps": a.reps}
        for k, v in ms.items():
            med = sorted(v)[len(v) // 2]
            row[k] = {"ms_total": round(med, 2), "ms_per_position": round(med / len(pos), 3),
                      "positions_per_s": round(len(pos) / med * 1e3, 1), "ms_all": [round(x, 2) for x in v]}
        row["speedup_c_vs_a"] = round(row["a_user_loop"]["ms_total"] / row["c_default"]["ms_total"], 2)
        row["speedup_c_vs_b"] = round(row["b_group1"]["ms_total"] / row["c_default"]["ms_total"], 3)
        lines.append(row)
        print(json.dumps(row), flush=True)
    lines.append(dict(gpu_info(), what="device_after"))
    print(json.dumps(lines[-1]), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "score_bench.jsonl"), "w") as f:
            f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
