"""Cost of generation by iterative masked sampling, per step per chain, against the Python loop a user would write.

    python tools/sample_bench.py [--steps 4] [--n_chains 4] [--reps 3] [--out DIR]

Shapes, fp16, 10 layers, seeded random-init weights: 512 x 36 (the 2DRB_1 tokens) and 256 x 101 (seeded tokens).
mask_prob 0.1, temperature 1, allowed A G C U -.  Per shape, after one warm-up of each, the ways run alternately,
``--reps`` times each, in reversed order every other repeat:
  (a) the user loop: per step and chain, a torch mask over the eligible tokens, forward(masked grid, want_logits=True),
      torch.softmax over the allowed logits at the masked tokens and torch.multinomial;
  (b) MSATransformer.sample_msa over all rows;
  (c) MSATransformer.sample_msa over the query row only (the LM head runs on that row alone).
Each is timed with a host clock around work that ends in a device synchronise, and reported as ms per step per chain
(median over the repeats), with the GPU's name, power limit and SM clock read in the same run.  Prints one JSON line
per shape between two lines of GPU state (before and after); with --out, also writes them to DIR/sample_bench.jsonl.
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


def user_loop(model, t, steps, n_chains, p, temperature, allowed, gen):
    vocab = model.vocab
    states = t.expand(n_chains, -1, -1).clone()
    elig = t.ne(vocab.pad_idx)
    elig[:, 0] = False
    for _ in range(steps):
        for k in range(n_chains):
            m = (torch.rand(t.shape, device=t.device, generator=gen) < p) & elig
            grid = states[k].masked_fill(m, vocab.mask_idx)
            lg = model(grid.unsqueeze(0), want_logits=True)["logits"][0]
            probs = torch.softmax(lg[m][:, allowed] / temperature, -1)
            states[k][m] = allowed[torch.multinomial(probs, 1).squeeze(1)]
    return states


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, r


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--n_chains", type=int, default=4)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args(argv)
    import rnamsm_b200 as pkg
    torch.manual_seed(42)
    model = pkg.MSATransformer(pkg.Vocab(pkg.Alphabet()), num_layers=10, precision="fp16").eval().cuda()
    g = np.load(os.path.join(ROOT, "tests", "golden", "2DRB_1.npz"))
    gen = torch.Generator().manual_seed(7)                         # uniform over A G C U X N - (4..10), BOS column
    seeded = torch.randint(4, 11, (256, 101), generator=gen, dtype=torch.int64)
    seeded[:, 0] = model.vocab.bos_idx
    shapes = [("512x36", torch.from_numpy(g["tokens"].astype(np.int64))[0]), ("256x101", seeded)]
    allowed = torch.tensor([4, 5, 6, 7, 10], device="cuda")
    p, T, S, K = 0.1, 1.0, a.steps, a.n_chains
    lines = [dict(gpu_info(), what="device")]
    print(json.dumps(lines[0]), flush=True)
    for name, t in shapes:
        t = t.cuda()
        R, Cc = t.shape
        tgen = torch.Generator(device="cuda").manual_seed(1)
        ways = {
            "a_user_loop": lambda: user_loop(model, t, S, K, p, T, allowed, tgen),
            "b_sample_all_rows": lambda: model.sample_msa(t, S, mask_prob=p, temperature=T, n_chains=K, seed=1),
            "c_sample_query_row": lambda: model.sample_msa(t, S, mask_prob=p, temperature=T, rows=[0], n_chains=K, seed=1),
        }
        for fn in ways.values():
            fn()
        ms = {k: [] for k in ways}
        for i in range(a.reps):      # the order reverses every repeat, so clock drift under the power cap evens out
            for k in (list(ways) if i % 2 == 0 else list(ways)[::-1]):
                ms[k].append(timed(ways[k])[0])
        group, passes = pkg.plan_score_group(R, Cc, K)
        row = {"what": "shape", "shape": name, "precision": "fp16", "steps": S, "n_chains": K, "mask_prob": p,
               "group": group, "passes": passes, "reps": a.reps}
        for k, v in ms.items():
            med = sorted(v)[len(v) // 2]
            row[k] = {"ms_per_step_per_chain": round(med / (S * K), 3), "ms_all": [round(x, 2) for x in v]}
        for k in ("b_sample_all_rows", "c_sample_query_row"):
            row[f"speedup_{k[0]}_vs_a"] = round(row["a_user_loop"]["ms_per_step_per_chain"] /
                                                row[k]["ms_per_step_per_chain"], 2)
        lines.append(row)
        print(json.dumps(row), flush=True)
    lines.append(dict(gpu_info(), what="device_after"))
    print(json.dumps(lines[-1]), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "sample_bench.jsonl"), "w") as f:
            f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
