"""Cost of the categorical Jacobian of the query row, two ways, and its contacts across precisions.

    python tools/jacobian_bench.py [--reps 3] [--warmup 1] [--out DIR]

Shapes, fp16, 10 layers, seeded random-init weights: 512 x 36 (the 2DRB_1 tokens, all 35 positions: 106 forwards) and
256 x 101 (seeded tokens, all 100 positions: about 300 forwards).  Alphabet AGCU.  Per shape, after warm-up, the two ways
run alternately, ``--reps`` times each, the order reversed every other repeat:
  (a) the user loop: clone + substitute, forward(grid, want_logits=True), slice the query row and subtract, per grid;
  (b) MSATransformer.categorical_jacobian(..., return_jacobian=True) with the default token budget.
Each is timed with a host clock around work that ends in a device synchronise; the median over the repeats is
reported, with the GPU's name, power limit and SM clock read in the same run.  Asserts that J from (a) and (b) are
bit-identical.  Then, on 2DRB_1, the fp16 and bf16 contacts against the fp32 contacts: norm-relative difference and
the overlap of the top-L pairs (i < j).  Prints one JSON line per measurement between two lines of GPU state (before
and after); with --out, also writes them to DIR/jacobian_bench.jsonl.
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


def user_loop(model, t, pos, alph):
    P, A = len(pos), len(alph)
    pos_d = torch.tensor(pos, device=t.device)
    alph_d = torch.tensor(alph, device=t.device)
    f = lambda g: model(g.unsqueeze(0), want_logits=True)["logits"][0, 0].index_select(0, pos_d).index_select(1, alph_d)
    wt = f(t)
    q = t[0].tolist()
    J = torch.zeros((P, A, P, A), dtype=torch.float32, device=t.device)
    for i, c in enumerate(pos):
        for a, v in enumerate(alph):
            if q[c] != v:
                g = t.clone()
                g[0, c] = v
                J[i, a] = f(g) - wt
    return J


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, r


def top_pairs(c, k):
    iu = np.triu_indices(c.shape[0], 1)
    order = np.argsort(-c[iu], kind="stable")[:k]
    return set(zip(iu[0][order].tolist(), iu[1][order].tolist()))


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args(argv)
    import rnamsm_b200 as pkg
    vocab = pkg.Vocab(pkg.Alphabet())
    torch.manual_seed(42)
    sd = pkg.MSATransformer(vocab, num_layers=10, precision="fp32").state_dict()

    def make(precision):
        m = pkg.MSATransformer(vocab, num_layers=10, precision=precision)
        m.load_state_dict(sd, strict=True)
        return m.eval().cuda()

    model = make("fp16")
    alph = [vocab.tokens_to_idx[c] for c in "AGCU"]
    g = np.load(os.path.join(ROOT, "tests", "golden", "2DRB_1.npz"))
    drb = torch.from_numpy(g["tokens"].astype(np.int64))[0]
    gen = torch.Generator().manual_seed(7)                         # uniform over A G C U X N - (4..10), BOS column
    seeded = torch.randint(4, 11, (256, 101), generator=gen, dtype=torch.int64)
    seeded[:, 0] = vocab.bos_idx
    lines = [dict(gpu_info(), what="device")]
    print(json.dumps(lines[0]), flush=True)
    for name, t in (("512x36", drb), ("256x101", seeded)):
        t = t.cuda()
        R, Cc = t.shape
        pos = [c for c in range(1, Cc) if int(t[0, c]) != vocab.pad_idx]
        n = len(pkg.jacobian_entries([int(t[0, c]) for c in pos], alph))
        group, passes = pkg.plan_score_group(R, Cc, n)
        ways = {
            "a_user_loop": lambda: user_loop(model, t, pos, alph),
            "b_categorical_jacobian": lambda: model.categorical_jacobian(t, positions=pos, return_jacobian=True)[1],
        }
        for _ in range(a.warmup):
            for fn in ways.values():
                fn()
        ms = {k: [] for k in ways}
        res = {}
        for rep in range(a.reps):
            for k in (list(ways) if rep % 2 == 0 else list(ways)[::-1]):
                dt, res[k] = timed(ways[k])
                ms[k].append(dt)
        assert torch.equal(res["a_user_loop"], res["b_categorical_jacobian"]), "J of the user loop and the call differ"
        row = {"what": "shape", "shape": name, "precision": "fp16", "layers": 10, "positions": len(pos),
               "forwards": n + 1, "default_group": group, "default_passes": passes, "reps": a.reps,
               "J_bit_identical": True}
        for k, v in ms.items():
            med = sorted(v)[len(v) // 2]
            row[k] = {"ms_total": round(med, 1), "ms_per_forward": round(med / (n + 1), 3),
                      "ms_all": [round(x, 1) for x in v]}
        row["speedup_b_vs_a"] = round(row["a_user_loop"]["ms_total"] / row["b_categorical_jacobian"]["ms_total"], 3)
        lines.append(row)
        print(json.dumps(row), flush=True)
    # contacts of the 16-bit precisions against fp32 on 2DRB_1 (a measurement, not a bound)
    t = drb.cuda()
    contacts = {p: make(p).categorical_jacobian(t).cpu().double().numpy() for p in ("fp32", "fp16", "bf16")}
    L_ = contacts["fp32"].shape[0]
    ref = contacts["fp32"]
    for p in ("fp16", "bf16"):
        c = contacts[p]
        row = {"what": "contacts_vs_fp32", "shape": "512x36", "precision": p, "L": L_,
               "norm_rel_diff": float(np.linalg.norm(c - ref) / np.linalg.norm(ref)),
               "top_L_overlap": len(top_pairs(c, L_) & top_pairs(ref, L_)) / L_}
        lines.append(row)
        print(json.dumps(row), flush=True)
    lines.append(dict(gpu_info(), what="device_after"))
    print(json.dumps(lines[-1]), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "jacobian_bench.jsonl"), "w") as f:
            f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
