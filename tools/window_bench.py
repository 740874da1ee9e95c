"""Full-length features of alignments longer than the learned positions, two ways, and the stitch kernel alone.

    python tools/window_bench.py [--reps 3] [--warmup 1] [--out DIR]

Shapes, fp16, 10 layers, seeded random-init weights, seeded tokens: 128 x 1501 and 512 x 2001 residues, default window
1023 and stride 511 (2 and 3 windows).  Per shape, after warm-up, the two ways run alternately, ``--reps`` times each,
the order reversed every other repeat:
  (a) the user loop: one forward(window grid, need_head_weights=True) per window, then the stitch in torch: the same
      coefficients (float64 quotients of the integer tent-weight sums, rounded to fp32) and fp32 addcmul in window order;
  (b) MSATransformer.forward_windows with the default token budget.
Each is timed with a host clock around work that ends in a device synchronise; the median over the repeats is reported,
with the GPU's name, power limit and SM clock read in the same run.  The outputs of (a) and (b) are compared bitwise
(and their largest difference reported if they are not identical).  Then the stitch kernel alone: its device time from
CUDA events around each of its launches (rnamsm_profile_collect, a separate run of (b)), and the bytes it has to move,
counted from the shapes and the window plan by stitch_bytes(): every window map and embedding read once, every output
element written once per pass that covers it (the first pass also writes the zeros), and read back when an earlier pass
covered it too.  Achieved bytes/s are set against the 7.7 TB/s of the B200 data sheet.  Prints one JSON line per
measurement between two lines of GPU state; with --out, also writes them to DIR/window_bench.jsonl.
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

HBM_BYTES_PER_S = 7.7e12


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True)
    f = [x.strip() for x in (r.stdout.strip().splitlines() or [",,,"])[0].split(",")] + ["", "", "", ""]
    return {"gpu": f[0] or torch.cuda.get_device_name(0), "power_limit": f[1], "sm_clock": f[2], "sm_clock_max": f[3]}


def tent_rows(L, W, starts, device):
    """[K, L] int64 tent weights, 0 outside each window."""
    p = torch.arange(L, device=device)
    rows = []
    for s in starts:
        w = torch.minimum(p - s + 1, s + W - p)
        rows.append(torch.where((p >= s) & (p < s + W), w, torch.zeros_like(w)))
    return torch.stack(rows)


def user_loop(model, t, window, stride):
    import rnamsm_b200 as pkg
    N, H, D = model.num_layers, model.num_attention_heads, model.embed_dim
    R, Cc = t.shape
    L = Cc - 1
    K = pkg._lib.lib.rnamsm_window_starts(L, window, stride, None)
    starts = [min(k * stride, L - min(window, L)) for k in range(K)]
    W = min(window, L)
    w = tent_rows(L, W, starts, t.device)
    den1 = w.sum(0).double()
    den2 = (w[:, :, None] * w[:, None, :]).sum(0).double()
    emb = torch.zeros((L, D), dtype=torch.float32, device=t.device)
    atp = torch.zeros((N * H, L, L), dtype=torch.float32, device=t.device)
    for k, s in enumerate(starts):
        g = torch.cat([t[:, :1], t[:, 1 + s:1 + s + W]], dim=1)
        r = model(g.unsqueeze(0), repr_layers=[N], need_head_weights=True, want_logits=False)
        sl = slice(s, s + W)
        wk = w[k, sl].double()
        c1 = (wk / den1[sl]).float()
        c2 = (wk[:, None] * wk[None, :] / den2[sl, sl]).float()
        emb[sl].addcmul_(r["representations"][N][0, 0, 1:], c1[:, None])
        atp[:, sl, sl].addcmul_(r["row_attentions"][0].reshape(N * H, W + 1, W + 1)[:, 1:, 1:], c2[None])
        del r
    return emb, atp


def stitch_bytes(L, W, starts, group, NH, D):
    """Bytes the stitch kernels of one call move (emb and atp; no contacts), from the shapes and the window plan."""
    K = len(starts)
    s = np.asarray(starts)
    p = np.arange(L)
    lo, hi = np.minimum.outer(p, p), np.maximum.outer(p, p)
    ka = np.searchsorted(s, hi - W + 1, side="left")                  # first window holding the pair
    kb = np.searchsorted(s, lo, side="right") - 1                     # last window holding the pair
    covered = ka <= kb
    pa = np.searchsorted(s, p - W + 1, side="left")
    total = 4 * K * (NH * W * W + W * D)                              # every window value read once
    total += 4 * NH * int((~covered).sum())                           # zeros, written by the first pass
    for k0 in range(0, K, group):
        k1 = min(k0 + group, K) - 1
        touched = covered & (ka <= k1) & (kb >= k0)
        total += 4 * NH * int(touched.sum())                          # written
        total += 4 * NH * int((touched & (ka < k0)).sum())            # read back: an earlier pass covered it
        res = (pa <= k1) & (np.minimum(np.searchsorted(s, p, side="right") - 1, K - 1) >= k0)
        total += 4 * D * int(res.sum()) + 4 * D * int((res & (pa < k0)).sum())
    return total


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
    L_ = pkg._lib
    vocab = pkg.Vocab(pkg.Alphabet())
    torch.manual_seed(42)
    model = pkg.MSATransformer(vocab, num_layers=10, precision="fp16").eval().cuda()
    NH, D = model.num_layers * model.num_attention_heads, model.embed_dim
    window = model.embed_positions.max_positions - 1
    stride = window // 2
    lines = [dict(gpu_info(), what="device")]
    print(json.dumps(lines[0]), flush=True)
    for R, L in ((128, 1501), (512, 2001)):
        gen = torch.Generator().manual_seed(R + L)                 # uniform over A G C U X N - (4..10), BOS column
        t = torch.randint(4, 11, (R, L + 1), generator=gen, dtype=torch.int64)
        t[:, 0] = vocab.bos_idx
        t = t.cuda()
        K = L_.lib.rnamsm_window_starts(L, window, stride, None)
        group, passes = pkg.plan_score_group(R, window + 1, K)
        ways = {
            "a_user_loop": lambda: user_loop(model, t, window, stride),
            "b_forward_windows": lambda: (lambda o: (o["emb"], o["atp"]))(model.forward_windows(t)),
        }
        for _ in range(a.warmup):
            for fn in ways.values():
                fn()
        ms = {k: [] for k in ways}
        res = {}
        for rep in range(a.reps):
            for k in (list(ways) if rep % 2 == 0 else list(ways)[::-1]):
                res[k] = None
                torch.cuda.empty_cache()
                dt, res[k] = timed(ways[k])
                ms[k].append(dt)
        (ea, aa), (eb, ab) = res["a_user_loop"], res["b_forward_windows"]
        same = torch.equal(ea, eb) and torch.equal(aa, ab)
        row = {"what": "shape", "shape": f"{R}x{L}", "precision": "fp16", "layers": 10, "window": window,
               "stride": stride, "windows": K, "default_group": group, "default_passes": passes, "reps": a.reps,
               "outputs_bit_identical": same}
        if not same:
            row["max_abs_diff"] = {"emb": float((ea - eb).abs().max()), "atp": float((aa - ab).abs().max())}
        for k, v in ms.items():
            row[k] = {"ms_median": round(sorted(v)[len(v) // 2], 1), "ms_all": [round(x, 1) for x in v]}
        row["speedup_b_vs_a"] = round(row["a_user_loop"]["ms_median"] / row["b_forward_windows"]["ms_median"], 3)
        del ea, aa, eb, ab, res
        # the stitch kernel alone: CUDA events around its launches in a run of its own
        L_.profile_enable(True)
        model.forward_windows(t)
        torch.cuda.synchronize()
        prof = L_.profile_collect()
        L_.profile_enable(False)
        st_ms, st_n = prof["window_stitch"]
        starts = [min(k * stride, L - window) for k in range(K)]
        nbytes = stitch_bytes(L, window, starts, group, NH, D)
        row["stitch"] = {"launches": st_n, "ms": round(st_ms, 3), "bytes": nbytes,
                         "bytes_per_s": round(nbytes / (st_ms * 1e-3), 1),
                         "frac_of_7p7_TBps": round(nbytes / (st_ms * 1e-3) / HBM_BYTES_PER_S, 3),
                         "build_ms": round(prof["window_build"][0], 3)}
        lines.append(row)
        print(json.dumps(row), flush=True)
        torch.cuda.empty_cache()
    lines.append(dict(gpu_info(), what="device_after"))
    print(json.dumps(lines[-1]), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "window_bench.jsonl"), "w") as f:
            f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
