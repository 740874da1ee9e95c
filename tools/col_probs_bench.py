"""Cost of exporting the column-attention probabilities (need_col_weights / need_col_weights_mean).

    python tools/col_probs_bench.py [--steps 3] [--warmup 2] [--layers 10]

Prints ONE JSON line: the GPU's name and power limit (read in the same run), then per workload (cfg1 512x36,
cfg2 512x256, cfg5 1024x1024, cfg4 4096x128 without row positions) the 10-layer fp16 forward time with no export,
with the column mean and with the full [N, H, C, R, R] tensor where it fits in memory (CUDA events after warm-up,
median of the steps), and the probability kernels alone (rnamsm_col_attn_probs on a q|k of that shape, 12 heads,
column-major as the layer hands it over): time, exponentials/s and, for the full form, bytes written/s.  Each pass
makes R*R*C*H exponentials (the log-sum-exp pass and the probability pass); the full form writes 4*R*R*C*H bytes.
Parity at the timed sizes: the mean kernel against float64 on sampled (h, i) rows, and the forward's mean output
against the mean of its full output where both exist.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = [("cfg1", 512, 36, True), ("cfg2", 512, 256, True), ("cfg5", 1024, 1024, True), ("cfg4", 4096, 128, False)]
H = 12


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    name, power = (r.stdout.strip().splitlines() or [","])[0].split(",")[:2]
    return {"gpu": name.strip() or torch.cuda.get_device_name(0), "power_limit": power.strip()}


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return sorted(ms)[len(ms) // 2]


def kernel_bench(L, R, Cc, steps, warmup, full_fits):
    g = torch.Generator(device="cuda").manual_seed(R + Cc)
    D = H * 64
    qkv = (torch.randn(Cc, R, 3 * D, generator=g, device="cuda") * 0.6)
    qkv = qkv.half()
    scratch = torch.empty(L.lib.rnamsm_col_probs_scratch_bytes(R, Cc, H), dtype=torch.uint8, device="cuda")
    mean = torch.empty(H, R, R, device="cuda")
    st = L.stream_ptr()

    def run(probs, m):
        L.check(L.lib.rnamsm_col_attn_probs(L.ptr(qkv), R, Cc, H, L.F16, 1, None, L.ptr(probs), L.ptr(m), L.ptr(scratch),
                                            st), "col_attn_probs")

    n_exp = 2.0 * R * R * Cc * H
    out = {}
    t = timed(lambda: run(None, mean), steps * 3, warmup)
    out["mean_kernel_ms"] = round(t, 4)
    out["mean_kernel_exp_per_s"] = float(f"{n_exp / (t * 1e-3):.4g}")
    # parity of the timed mean on sampled (h, i) rows
    q64 = qkv.double()
    gs = torch.Generator().manual_seed(0)
    err = 0.0
    for h, i in zip(torch.randint(0, H, (4,), generator=gs).tolist(), torch.randint(0, R, (4,), generator=gs).tolist()):
        s = torch.einsum("cd,cjd->cj", q64[:, i, h * 64:(h + 1) * 64], q64[:, :, D + h * 64:D + (h + 1) * 64])
        ref = s.softmax(-1).mean(0)
        err = max(err, float((mean[h, i].double() - ref).abs().max() / ref.abs().max()))
    out["mean_kernel_rel_err_vs_fp64"] = float(f"{err:.3g}")
    del q64
    if full_fits:
        probs = torch.empty(H, Cc, R, R, device="cuda")
        t = timed(lambda: run(probs, None), steps * 3, warmup)
        nbytes = 4.0 * R * R * Cc * H
        out["full_kernel_ms"] = round(t, 4)
        out["full_kernel_exp_per_s"] = float(f"{n_exp / (t * 1e-3):.4g}")
        out["full_kernel_bytes_per_s"] = float(f"{nbytes / (t * 1e-3):.4g}")
        del probs
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--layers", type=int, default=10)
    ap.add_argument("--only", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("col_probs_bench.py needs a CUDA device")
    import rnamsm_b200 as pkg
    from rnamsm_b200 import _lib as L

    torch.cuda.set_device(0)
    res = {"tool": "col_probs_bench", **gpu_info(), "precision": "fp16", "layers": a.layers, "heads": H,
           "bounds": "exponentials: ex2 on the MUFU unit, 16 / clk / SM; full form: HBM writes (7.7 TB/s data sheet)",
           "workloads": {}}
    free = torch.cuda.mem_get_info()[0]
    for name, R, Cc, epm in WORKLOADS:
        if a.only and name not in a.only.split(","):
            continue
        vocab = pkg.Vocab(pkg.Alphabet())
        torch.manual_seed(1)                                     # the model's own random init (init_weights)
        model = pkg.MSATransformer(vocab, num_layers=a.layers, embed_positions_msa=epm, precision="fp16").eval().cuda()
        tokens = torch.randint(4, 8, (1, R, Cc), generator=torch.Generator().manual_seed(1))   # A G C U
        tokens[..., 0] = vocab.bos_idx                           # BOS column
        tokens = tokens.cuda()
        full_bytes = 4 * a.layers * H * Cc * R * R
        full_fits = full_bytes < 0.5 * free
        w = {"R": R, "C": Cc, "full_bytes": full_bytes}
        fwd = lambda **kw: model(tokens, want_logits=False, **kw)                     # noqa: E731
        w["forward_ms"] = round(timed(fwd, a.steps, a.warmup), 3)
        w["forward_mean_ms"] = round(timed(lambda: fwd(need_col_weights_mean=True), a.steps, a.warmup), 3)
        if full_fits:
            w["forward_full_ms"] = round(timed(lambda: fwd(need_col_weights=True), a.steps, a.warmup), 3)
            out = fwd(need_col_weights=True, need_col_weights_mean=True)
            full, mean = out["col_attentions"], out["col_attentions_mean"]
            ref = full[0, -1].double().mean(1)
            err = float((mean[0, -1].double() - ref).abs().max() / ref.abs().max())
            w["forward_mean_vs_full_mean_rel_err"] = float(f"{err:.3g}")
            del out, full, mean, ref
        else:
            w["forward_full_ms"] = None
        w["mean_cost_ms_per_layer"] = round((w["forward_mean_ms"] - w["forward_ms"]) / a.layers, 4)
        if w["forward_full_ms"] is not None:
            w["full_cost_ms_per_layer"] = round((w["forward_full_ms"] - w["forward_ms"]) / a.layers, 4)
        del model
        torch.cuda.empty_cache()
        w.update(kernel_bench(L, R, Cc, a.steps, a.warmup, 4 * H * Cc * R * R < 0.5 * free))
        torch.cuda.empty_cache()
        res["workloads"][name] = w
        print(f"# {name}: {w}", file=sys.stderr, flush=True)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
