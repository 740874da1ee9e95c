#!/usr/bin/env python
"""bench.py -- RNA-MSM MSA-transformer forward throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload cfg2|cfg1|cfg4|cfg5] [--precision fp16|bf16|fp32] [--dump-outputs DIR]

A "step" is one full forward of the hot path over one synthetic MSA: int64 token grid ->
emb (L,768) + 120 tied-row attention maps, with random-init weights of the real architecture
(10 layers, D=768, 12 heads; the trained checkpoint is not available offline).  At N=1 the
workload is BASELINE config[1]: depth 512 x L 256 (token grid R x C = 512 x 256, 131 072 tokens).
N > 1 (torchrun, one rank per GPU): independent MSAs are data-parallel with NO collective
(SURVEY.md 8e, row 1) -- every rank runs its own MSA of the same shape, weak scaling;
value = all ranks' tokens / max-over-ranks device time.

Printed JSON (rank 0, one line):
  value        tokens/s with the tokens already resident in HBM (device-timed, CUDA events)
  e2e          same metric through the public API `MSATransformer.forward` + `extract_features`
               with pinned HOST tokens in and emb/atp copied back to the host every step
  roofline     dominant kernel class (the tcgen05 dense GEMM): algorithmic FLOPs / live
               CUDA-event time per launch vs the measured bf16 peak in MEASURED_PEAKS.json
  cpu_baseline the oracle (port of the reference's fp32 CPU forward) timed on this box's cores on
               a bounded sample: ONE of the 10 AxialTransformerLayers at the full shape, x10
  --impl reference : the CPU arm alone, same metric/config, one sample per step.

--dump-outputs DIR writes what the last device-timed step returned (see dump_outputs) as DIR/<name>.npy.  Weights
(torch seed 42) and tokens (seeded per rank) are the same in every run, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "MSA tokens/sec (depth x L) full forward incl. emb+atp"
WORKLOADS = {
    # name: (R, C, embed_positions_msa, description)
    "cfg1": (512, 36, True, "cfg1 2DRB_1-shaped MSA depth 512 x L 35 (+BOS)"),
    "cfg2": (512, 256, True, "cfg2 synthetic MSA depth 512 x L 256 (token grid 512x256), batch 1"),
    "cfg4": (4096, 128, False, "cfg4 synthetic deep MSA depth 4096 x L 128, embed_positions_msa=False"),
    "cfg5": (1024, 1024, True, "cfg5 synthetic long MSA depth 1024 x L 1024 token grid"),
    # cfg3: 64 independent MSAs, depth 256, L ~ U{50..500} (seeded), farmed over the ranks longest-first
    "cfg3": (256, None, True, "cfg3 batch of 64 synthetic MSAs, depth 256, L 50-500 (RNAcmap3-like), one B=1 forward each, "
                              "longest-processing-time-first assignment over the ranks, no collective"),
}


def measured_traffic(workload, precision):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel class, from the committed
    ncu --set full capture of the same workload (profiles/r01e_traffic.json); None for other workloads."""
    p = os.path.join(ROOT, "profiles", "r01e_traffic.json")
    try:
        d = json.load(open(p))
        if d.get("workload") == workload and d.get("precision") == precision:
            return d["dense_gemm"]["dram_bytes_per_launch"], d["dense_gemm"]["algorithmic_bytes_per_launch"]
    except Exception:
        pass
    return None, None


def total_flops(R, C):
    """Algorithmic FLOPs of one forward (SURVEY.md 8d): N [32 T D^2 + 4 T D (R + C)] + 2 T (D^2 + V D)."""
    T = R * C
    return NL * (32.0 * T * D * D + 4.0 * T * D * (R + C)) + 2.0 * T * (D * D + V * D)


def synthetic_tokens(R, C, seed):
    """Synthetic MSA (SURVEY.md 8d): uniform over A,G,C,U,X,N,- (indices 4..10), column 0 = <cls>, no <pad>."""
    import torch
    g = torch.Generator().manual_seed(seed)
    t = torch.randint(4, 11, (1, R, C), generator=g, dtype=torch.int64)
    t[:, :, 0] = 0
    return t


def cfg3_lengths(n=64, seed=3):
    import random
    rng = random.Random(seed)
    return [rng.randint(50, 500) + 1 for _ in range(n)]          # token columns C = L + 1 (BOS)


def lpt_assign(costs, world):
    """Longest-processing-time-first: job indices per rank (SURVEY.md 8e row 1)."""
    loads, jobs = [0.0] * world, [[] for _ in range(world)]
    for i in sorted(range(len(costs)), key=lambda i: -costs[i]):
        g = min(range(world), key=lambda r: loads[r])
        loads[g] += costs[i]
        jobs[g].append(i)
    return jobs
D, H, F, NL, V = 768, 12, 3072, 10, 12


def flops_breakdown(R, C):
    """Algorithmic FLOPs per forward by kernel class (SURVEY.md 8d; multiply-add = 2)."""
    T = R * C
    return {
        "linear_qkv": NL * 2 * (2.0 * T * D * 3 * D),
        "linear_out_resid": NL * 2 * (2.0 * T * D * D),
        "linear_fc1_gelu": NL * (2.0 * T * D * F),
        "linear_fc2_resid": NL * (2.0 * T * D * F),
        "row_logits": NL * (2.0 * R * C * C * D),
        "row_av": NL * (2.0 * R * C * C * D),
        "col_attn": NL * (4.0 * R * R * C * D),
    }


def class_flops(R, C):
    """flops_breakdown keyed by the library's timing classes: short alignments (C <= 128) run tied logits + softmax + AV
    as ONE launch (row_attn_short.cu), whose class carries both terms."""
    fl = flops_breakdown(R, C)
    if C <= 128:            # the one-launch path takes these shapes (16-bit precisions)
        fl["row_attn_short"] = fl["row_logits"] + fl["row_av"]
        fl["row_logits"] = fl["row_av"] = 0.0
    else:
        fl["row_attn_short"] = 0.0
    return fl


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.stop_flag = threading.Event()
        self.proc = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
                if self.stop_flag.is_set():
                    break
        except Exception:
            pass

    def finish(self):
        self.stop_flag.set()
        if self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 3), ("hw_thermal_slowdown", 4), ("sw_thermal_slowdown", 5),
                              ("sw_power_cap", 6)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        busy = sorted(sm)[len(sm) // 2:]          # upper half ~ samples taken under load
        return {"sm_mhz": busy[len(busy) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return {"bf16_burst": d["bf16_tflops"], "bf16_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    "hbm": d["hbm_gbs"], "source": "measured"}
        except Exception:
            pass
    return {"bf16_burst": 1590.0, "bf16_sustained": 1400.0, "hbm": 6650.0, "source": "fallback"}


# ------------------------------------------------------------------------------------------------
def _config(desc, R, C, tokens_per_step, **extra):
    """The `config` object both arms print: identical keys and values for the same workload."""
    cfg = {"workload": desc, "R": R, "C": C, "tokens_per_step": tokens_per_step, "layers": NL, "embed_dim": D, "heads": H,
           "weights": "random-init (reference recipe model.py:89-101, seed 42)"}
    cfg.update(extra)
    return cfg


class CpuReference:
    """The CPU arm: the reference's OWN ``modules.AxialTransformerLayer`` (staged unmodified in oracle/_ref by
    oracle/build_ref.py; shipped chunking ``max_tokens_per_msa=16384``, i.e. its real ``_batched_forward`` path,
    modules.py:717-750 / 849-873) on all host cores; the oracle port only if the staged files are missing.
    One sample = embedding (oracle restatement of model.py:346-367; < 1 % of the time) + ONE layer at the full shape
    with ``need_head_weights=True`` as model.py:379-383 calls it; the column probabilities are dropped per layer
    (the unmodified model keeps 10 x [12,C,1,R,R] fp32 alive: 32 GiB at cfg2)."""

    def __init__(self, R, C, embed_positions_msa, threads=None):
        import torch
        from oracle import msa_ref as O
        from oracle import build_ref
        self.torch, self.O = torch, O
        # torchrun exports OMP_NUM_THREADS=1; the CPU arm uses every host core (count reported in the JSON)
        torch.set_num_threads(threads or os.cpu_count() or 1)
        self.threads = torch.get_num_threads()
        self.R, self.C = R, C
        self.sd = O.make_weights(42, num_layers=1, embed_positions_msa=embed_positions_msa)
        self.tokens = O.make_tokens(R, C, 0)
        self.kind = "port"
        self.layer = None
        if build_ref.available():
            ref_modules, _ = build_ref.import_reference()
            layer = ref_modules.AxialTransformerLayer(D, F, H, 0.1, 0.1, 0.1, max_tokens_per_msa=2 ** 14)
            own = {k[len("layers.0."):]: v for k, v in self.sd.items() if k.startswith("layers.0.")}
            layer.load_state_dict(own, strict=True)
            self.layer = layer.eval()
            self.kind = "reference"

    def describe(self):
        what = ("the reference's own modules.AxialTransformerLayer (oracle/_ref, unmodified, max_tokens_per_msa=16384: "
                "its chunked _batched_forward path)" if self.kind == "reference"
                else "oracle port of the reference fp32 CPU forward (oracle/_ref not staged)")
        return f"embedding + ONE of {NL} AxialTransformerLayers at the full {self.R}x{self.C} shape per step: {what}"

    def one_layer(self, x, pm):
        if self.layer is not None:
            y, col_attn, row_attn = self.layer(x, self_attn_padding_mask=pm, need_head_weights=True)
            del col_attn
            return y, row_attn
        y, _, rp = self.O.axial_layer(self.sd, 0, x, pm)
        return y, rp

    def sample(self):
        """-> (seconds embedding, seconds one layer)."""
        torch = self.torch
        with torch.no_grad():
            t0 = time.perf_counter()
            x, pm = self.O.embed(self.sd, self.tokens)
            x = x.permute(1, 2, 0, 3).contiguous()
            t1 = time.perf_counter()
            self.one_layer(x, pm)
            t2 = time.perf_counter()
        return t1 - t0, t2 - t1

    def full_forward(self):
        """One REAL forward: embedding + all 10 layers (same layer object: every layer of the random-init model has
        the same shapes and cost) + final LayerNorm, streaming the maps.  -> seconds."""
        torch = self.torch
        with torch.no_grad():
            t0 = time.perf_counter()
            x, pm = self.O.embed(self.sd, self.tokens)
            x = x.permute(1, 2, 0, 3).contiguous()
            maps = []
            for _ in range(NL):
                x, rp = self.one_layer(x, pm)
                maps.append(rp)
            x = self.O.layer_norm(x, self.sd["emb_layer_norm_after.weight"], self.sd["emb_layer_norm_after.bias"])
            return time.perf_counter() - t0


def cpu_reference_sample(R, C, embed_positions_msa, threads=None):
    """(seconds embedding, seconds one layer, threads, kind, description) of one CPU sample."""
    ref = CpuReference(R, C, embed_positions_msa, threads)
    t_emb, t_layer = ref.sample()
    return t_emb, t_layer, ref.threads, ref.kind, ref.describe()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    R, C, epm, desc = WORKLOADS[args.workload]
    if C is None:                                        # cfg3: bounded sample = the median-length MSA of the batch
        lens = cfg3_lengths()
        C = sorted(lens)[len(lens) // 2]
    tokens = R * C
    ref = CpuReference(R, C, epm)
    samples, fwd = [], []
    for i in range(args.warmup + args.steps):
        t_emb, t_layer = ref.sample()
        if i >= args.warmup:
            samples.append(t_emb + t_layer)
            fwd.append(t_emb + NL * t_layer)            # one layer timed; the other nine are identical in shape and cost
    per_sample = sum(samples) / len(samples)
    per_fwd = sum(fwd) / len(fwd)
    value = tokens / per_fwd
    full = None
    if per_fwd < float(os.environ.get("RNAMSM_REF_FULL_FORWARD_MAX_S", "150")):
        t_full = ref.full_forward()                     # one real 10-layer forward, to check the extrapolation
        full = {"ms": t_full * 1e3, "tokens_per_s": tokens / t_full, "layers": NL}
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "tokens/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_sample * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": _config(desc, R, C, tokens, batch_tokens=None, tokens_per_step_scope="one MSA per step",
                          precision="fp32 torch CPU (the reference's own arithmetic)",
                          parallelism=f"{ref.threads} host threads, one process", l2="n/a (CPU)"),
        "extrapolated_from_layers": 1,
        "ms_per_forward_extrapolated": per_fwd * 1e3,
        "full_forward_measured": full,
        "cpu_baseline": {"value": value, "unit": "tokens/s", "cores": ref.threads, "kind": ref.kind,
                         "sample": ref.describe() + f"; value = tokens / (t_emb + {NL} x t_layer)"},
        "e2e": {"value": value, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------
DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, out):
    """Write the arrays ``MSATransformer.forward`` returned to its caller as float32 ``out_dir/<name>.npy``:
    ``row_attentions`` [1, layers, heads, C, C] and ``representations_<layers>`` [1, R, C, D].  Each array gets half of
    DUMP_BYTES; a larger one is cut to a fixed, seeded sample of its query positions (maps) or MSA rows
    (representations), always including index 0 and kept in ascending order."""
    import numpy as np
    import torch
    arrays = {"row_attentions": (out["row_attentions"], 3), f"representations_{NL}": (out["representations"][NL], 1)}
    os.makedirs(out_dir, exist_ok=True)
    for name, (t, axis) in arrays.items():
        n = t.shape[axis]
        keep = max(1, (DUMP_BYTES // len(arrays) - 1024) // (t.numel() // n * 4))    # 1 KB: room for the .npy header
        if keep < n:
            g = torch.Generator().manual_seed(0)
            idx = torch.cat([torch.zeros(1, dtype=torch.int64), 1 + torch.randperm(n - 1, generator=g)[:keep - 1]])
            t = t.index_select(axis, idx.sort().values.to(t.device))
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def _rel_err(a, b):
    """max|a - b| / max|b| (the norm-relative gate of SURVEY.md 8d)."""
    return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))


def run_secondary(args, pkg, _lib, world, rank, peaks):
    """The other BASELINE configs in the same run, so that the driver's records carry them (rank 0 returns the dict).

    N = 1 : cfg5 (1024x1024), cfg4 (4096x128), cfg1 (512x36) single-GPU forwards, a few steps each: ms, tokens/s, e2e,
            per-class TF/s incl. the tied row attention's fraction of the measured bf16 peak; cfg2 in the fp32 path.
    N > 1 : cfg5 and cfg4 as ONE MSA sharded over the N ranks (fused peer-memory schedule): device ms (max over
            ranks), e2e ms (host tokens in, every rank's map rows + rank 0's emb back in host memory), against the
            single-GPU forward of the same MSA timed on rank 0 in the same run -> speed-up; plus `parity`: the sharded
            result against the single-GPU forward on a small padded MSA (max over ranks of the norm-relative error).
    All ranks must call this together."""
    import torch
    import torch.distributed as dist
    from rnamsm_b200.sharded import ShardedHostOutput, sharded_forward

    vocab = pkg.Vocab(pkg.Alphabet())
    steps = 3
    out = {}

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def make_model(epm, precision="fp16"):
        torch.manual_seed(42)
        return pkg.MSATransformer(vocab, num_layers=NL, embed_positions_msa=epm, precision=precision).eval().cuda()

    def time_events(fn, n, warm):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    def time_wall(fn, n, warm):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(n):
            fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3 / n

    def single_gpu(model, R, C, n_steps, with_classes):
        """device ms, e2e ms (+ per-class TF/s) of the one-GPU forward of a synthetic R x C MSA."""
        tok_host = synthetic_tokens(R, C, seed=100).pin_memory()
        tok_dev = tok_host.cuda()
        emb_host = torch.empty((C - 1, D), dtype=torch.float32).pin_memory()
        atp_host = torch.empty((NL * H, C - 1, C - 1), dtype=torch.float32).pin_memory()
        fwd = lambda: model(tok_dev, repr_layers=[NL], need_head_weights=True, want_logits=False)
        ms = time_events(fwd, n_steps, 2 if R * C > 100000 else 5)
        res = {"ms_per_step": round(ms, 3), "tokens_per_s": round(R * C / (ms * 1e-3), 1),
               "whole_forward_tflops": round(total_flops(R, C) / (ms * 1e-3) / 1e12, 1)}
        e2e = time_wall(lambda: pkg.extract_features_streamed(model, tok_host, atp_host, emb_host), n_steps, 1)
        res["e2e_ms_per_step"] = round(e2e, 3)
        res["e2e_tokens_per_s"] = round(R * C / (e2e * 1e-3), 1)
        if with_classes:
            _lib.profile_enable(True)
            for _ in range(n_steps):
                fwd()
            torch.cuda.synchronize()
            prof = _lib.profile_collect()
            _lib.profile_enable(False)
            fl = class_flops(R, C)
            res["class_tflops"] = {k: round(fl[k] * n_steps / (prof[k][0] * 1e-3) / 1e12, 1) for k in fl if prof[k][0] > 0}
            tot = sum(v[0] for v in prof.values())
            res["class_time_share"] = {k: round(v[0] / tot, 4) for k, v in prof.items() if v[1]}
            t_short = prof.get("row_attn_short", (0.0, 0))[0]   # one launch does logits + softmax + AV when C <= 128
            t_tied = prof["row_logits"][0] + prof["row_av"][0] + t_short
            fl_tied = fl["row_logits"] + fl["row_av"] + fl["row_attn_short"]
            tied = fl_tied * n_steps / (t_tied * 1e-3) / 1e12
            tied_sm = fl_tied * n_steps / ((t_tied + prof["row_softmax"][0]) * 1e-3) / 1e12
            res["tied_row_attention"] = {
                "tflops": round(tied, 1), "frac_of_bf16_sustained": round(tied / peaks["bf16_sustained"], 4),
                "frac_of_bf16_burst": round(tied / peaks["bf16_burst"], 4),
                "tflops_incl_softmax_pass": round(tied_sm, 1),
                "what": ("row_attn_short_kernel (logits + softmax + AV in one launch, C <= 128)" if t_short > 0 else
                         "tied logits (umma_gemm_kernel<TIED>) + AV (umma_gemm_kernel<AV>)") +
                        ": 4 R C^2 D flops per layer over their live CUDA-event time inside the forward"}
        del tok_dev, atp_host, emb_host
        return res

    def farm_cfg3(model):
        """BASELINE configs[2]: the batch of 64 MSAs (depth 256, L 50-500), LPT-assigned to the ranks, no collective on
        the data path.  One pass = every rank runs its MSAs; time = max over ranks; tokens/s = whole batch / time."""
        Rf = WORKLOADS["cfg3"][0]
        lens = cfg3_lengths()
        mine = lpt_assign([total_flops(Rf, c) for c in lens], world)[rank]
        toks = [synthetic_tokens(Rf, lens[i], seed=200 + i).cuda() for i in mine]
        bt = 131072
        groups = pkg.plan_batches([(Rf, lens[i]) for i in mine], bt)

        def one_by_one():
            for t in toks:
                model(t, repr_layers=[NL], need_head_weights=True, want_logits=False)

        def batched():
            for g in groups:
                model.forward_batch([toks[i] for i in g], need_head_weights=True)

        res = {"workload": WORKLOADS["cfg3"][3], "n_msa": len(lens), "R": Rf, "n_gpus": world,
               "tokens_per_pass": Rf * sum(lens), "parallelism": f"dp{world} independent MSAs (LPT by flops), no collective"}
        for key, fn in (("one_forward_per_msa", one_by_one), ("forward_batch", batched)):
            sync_all()
            ms = time_events(fn, 2, 1)
            if world > 1:
                t = torch.tensor([ms], dtype=torch.float64, device="cuda")
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t[0])
            res[key] = {"ms_per_pass": round(ms, 3), "tokens_per_s": round(Rf * sum(lens) / (ms * 1e-3), 1)}
        res["forward_batch"]["batch_tokens"] = bt
        res["forward_batch"]["passes_on_rank0"] = len(groups)
        del toks
        torch.cuda.empty_cache()
        return res

    big = (("cfg5", 1024, 1024, True), ("cfg4", 4096, 128, False))
    if world == 1:
        models = {}
        for name, R, C, epm in (("cfg1", 512, 36, True),) + big:   # (the 5 ms forward first: it is the one a hot, power-capped GPU distorts most)
            if epm not in models:
                models[epm] = make_model(epm)
            out[name] = {"workload": WORKLOADS[name][3], "R": R, "C": C,
                         **single_gpu(models[epm], R, C, steps if name != "cfg1" else 10, True)}
            torch.cuda.empty_cache()
        try:
            out["cfg3"] = farm_cfg3(models[True])
        except Exception as e:                          # never lose the main line to a secondary measurement
            out["cfg3"] = {"error": repr(e)[:300]}
        models.clear()
        torch.cuda.empty_cache()
        for key, prec, what in (("cfg2_fp32", "fp32", "fp32 path (FFMA, the <= 1e-4 parity path)"),
                                ("cfg2_tf32x3", "tf32x3", "fp32 storage, nn.Linear layers as tf32 x 3 on tcgen05")):
            try:                                        # BASELINE configs[1] also names the fp32 path
                m32 = make_model(True, prec)
                R, C = 512, 256
                tok = synthetic_tokens(R, C, seed=100).cuda()
                ms = time_events(lambda: m32(tok, repr_layers=[NL], need_head_weights=True, want_logits=False), 2, 1)
                out[key] = {"workload": WORKLOADS["cfg2"][3] + ", " + what, "ms_per_step": round(ms, 2),
                            "tokens_per_s": round(R * C / (ms * 1e-3), 1),
                            "whole_forward_tflops": round(total_flops(R, C) / (ms * 1e-3) / 1e12, 1)}
                del m32
                torch.cuda.empty_cache()
            except Exception as e:                      # never lose the main line to a secondary measurement
                out[key] = {"error": repr(e)[:200]}
        return out

    # ---------------- N > 1: one MSA sharded over the ranks -----------------------------------------
    def max_over_ranks(v):
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    models = {}
    for name, R, C, epm in big:
        entry = {"workload": WORKLOADS[name][3], "R": R, "C": C, "n_gpus": world,
                 "parallelism": "rows (tied row attention, P2P logit reduce-scatter + softmax + all-gather) <-> columns "
                                "(column attention, LayerNorm push / out-projection scatter), peer-memory kernels over "
                                "NVLink, flag barriers in peer memory"}
        try:
            if R % world or C % world or (C // world) % 16:
                raise ValueError(f"{R}x{C} does not split over {world} ranks")
            if epm not in models:
                models[epm] = make_model(epm)
            model = models[epm]
            single = single_gpu(model, R, C, 2, False) if rank == 0 else None      # same box, same run, rank 0 alone
            torch.cuda.empty_cache()
            sync_all()
            tok_host = synthetic_tokens(R, C, seed=100).pin_memory()
            tok_dev = tok_host.cuda()
            host = ShardedHostOutput(NL, H, C, D, start=1)
            dev_fn = lambda: sharded_forward(model, tok_dev, fused=True, gather_maps=False)
            for _ in range(2):
                dev_fn()
            sync_all()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                dev_fn()
            e1.record()
            sync_all()
            ms = max_over_ranks(e0.elapsed_time(e1) / steps)
            e2e_fn = lambda: sharded_forward(model, tok_host.cuda(non_blocking=True), fused=True, host_out=host,
                                             gather_maps=False)
            e2e_fn()
            sync_all()
            t0 = time.perf_counter()
            for _ in range(steps):
                e2e_fn()
            sync_all()
            e2e = max_over_ranks((time.perf_counter() - t0) * 1e3 / steps)
            host.close()
            if rank == 0:
                entry.update({
                    "single_gpu_ms": single["ms_per_step"], "single_gpu_e2e_ms": single["e2e_ms_per_step"],
                    "sharded_ms": round(ms, 3), "sharded_e2e_ms": round(e2e, 3),
                    "speedup": round(single["ms_per_step"] / ms, 3), "e2e_speedup": round(single["e2e_ms_per_step"] / e2e, 3),
                    "tokens_per_s": round(R * C / (ms * 1e-3), 1), "e2e_tokens_per_s": round(R * C / (e2e * 1e-3), 1),
                    "whole_forward_tflops_per_gpu": round(total_flops(R, C) / world / (ms * 1e-3) / 1e12, 1),
                    "steps": steps, "d2h_bytes_per_step_all_ranks": (NL * H * (C - 1) ** 2 + (C - 1) * D) * 4})
            del tok_dev, host
            torch.cuda.empty_cache()
        except Exception as e:
            entry["error"] = repr(e)[:300]
        out[name] = entry
    try:
        if True not in models:
            models[True] = make_model(True)
        res3 = farm_cfg3(models[True])
        out["cfg3"] = res3
    except Exception as e:
        out["cfg3"] = {"error": repr(e)[:300]}
    # ---- multi-rank parity: the sharded forward against the one-GPU forward of the same model, small padded MSA ----
    try:
        Rp, Cp = 64, 128
        model = models.get(True) or make_model(True)
        tok = synthetic_tokens(Rp, Cp, seed=7)
        tok[:, -2:, 1:] = vocab.pad_idx                 # two all-pad rows
        tok[:, :, -3:] = vocab.pad_idx                  # three pad columns (masked keys, zeroed queries)
        tok = tok.cuda()
        ref = model(tok, repr_layers=[NL], need_head_weights=True, want_logits=False)
        got = sharded_forward(model, tok, fused=True, gather_maps=True)
        r0, r1 = got["row_shard"]
        e_rep = _rel_err(got["representations"][NL], ref["representations"][NL][:, r0:r1])
        e_map = _rel_err(got["row_attentions"], ref["row_attentions"])
        got_n = sharded_forward(model, tok, fused=False, gather_rows=True)
        e_rep_n = _rel_err(got_n["representations"][NL], ref["representations"][NL])
        e_map_n = _rel_err(got_n["row_attentions"], ref["row_attentions"])
        errs = [max_over_ranks(v) for v in (e_rep, e_map, e_rep_n, e_map_n)]
        out["parity"] = {"shape": [Rp, Cp], "pad_rows": 2, "pad_cols": 3, "layers": NL, "n_gpus": world,
                         "fused_emb_err": errs[0], "fused_map_err": errs[1], "nccl_emb_err": errs[2], "nccl_map_err": errs[3],
                         "parity_err": max(errs), "gate": 3e-3, "ok": max(errs) < 3e-3,
                         "what": "max over ranks of max|sharded - single GPU| / max|single GPU| on representations[10] "
                                 "(each rank's row shard) and on the 120 maps; fp16 path (the re-laid-out tensors are "
                                 "rounded to 16 bits once more, hence not bit-equal)"}
    except Exception as e:
        out["parity"] = {"error": repr(e)[:300]}
    sync_all()
    return out if rank == 0 else None


# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    import rnamsm_b200 as pkg
    from rnamsm_b200 import _lib
    # NB: the measured arm never touches oracle/: weights are the model's own random init (the reference
    # recipe, model.py:89-101), tokens are generated here.  Only cpu_reference_sample() imports the oracle.

    R, C, epm, desc = WORKLOADS[args.workload]
    farm = C is None                                   # cfg3: a list of MSAs per rank instead of one shape
    if farm:
        lens = cfg3_lengths()
        mine = lpt_assign([total_flops(R, c) for c in lens], world)[rank]
        my_C = [lens[i] for i in mine]
        C = max(lens)
        tokens_per_step = R * sum(lens)                # whole job (all ranks)
    else:
        tokens_per_step = R * C
    vocab = pkg.Vocab(pkg.Alphabet())
    torch.manual_seed(42)                              # seed_everything(42), RNA_MSM_Inference.py:17
    model = pkg.MSATransformer(vocab, num_layers=NL, embed_positions_msa=epm, precision=args.precision)
    model = model.eval().cuda()
    tok_host = synthetic_tokens(R, C, seed=100 + rank).pin_memory()
    tok_dev = tok_host.cuda()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    shard = bool(args.shard) and world > 1
    # the other BASELINE configs, measured in the same run (cfg5 / cfg4: single GPU at N = 1, ONE MSA sharded over the
    # ranks at N > 1, with a multi-rank parity number) -- see run_secondary
    want_secondary = args.workload == "cfg2" and not args.shard and not args.no_secondary and args.precision == "fp16"
    shard_host = None
    if shard:
        from rnamsm_b200.sharded import ShardedHostOutput, sharded_forward
        tok_host = synthetic_tokens(R, C, seed=100).pin_memory()   # the SAME MSA on every rank
        tok_dev = tok_host.cuda()
        if args.fused:                                             # host results: shared atp buffer + rank 0's emb
            shard_host = ShardedHostOutput(NL, H, C, D, start=1)

    if farm:
        farm_host = [synthetic_tokens(R, c, seed=200 + i).pin_memory() for i, c in zip(mine, my_C)]
        farm_dev = [t.cuda() for t in farm_host]
        # --batch-tokens > 0: short MSAs grouped into forward_batch passes (SURVEY.md 8f row 4); results per MSA
        # are bit-identical to the one-forward-per-MSA farm (tests/test_gpu_model.py)
        groups = pkg.plan_batches([(R, c) for c in my_C], args.batch_tokens) if args.batch_tokens > 0 else None

    def step_device():
        if shard:
            return sharded_forward(model, tok_dev, fused=args.fused, gather_maps=not args.fused)
        if farm:
            out = None
            if groups is not None:
                for g in groups:
                    out = model.forward_batch([farm_dev[i] for i in g], need_head_weights=True)
                return out
            for t in farm_dev:
                out = model(t, repr_layers=[NL], need_head_weights=True, want_logits=False)
            return out
        return model(tok_dev, repr_layers=[NL], need_head_weights=True, want_logits=False)

    emb_host = torch.empty((C - 1, D), dtype=torch.float32).pin_memory()
    atp_host = torch.empty((NL * H, C - 1, C - 1), dtype=torch.float32).pin_memory()

    if farm:                                           # per-MSA views of the pinned result buffers
        farm_atp = [atp_host.view(-1)[:NL * H * (c - 1) ** 2].view(NL * H, c - 1, c - 1) for c in my_C]
        farm_emb = [emb_host.view(-1)[:(c - 1) * D].view(c - 1, D) for c in my_C]

    def step_e2e():
        if farm and groups is not None:                # pinned host tokens in, every MSA's emb + atp back in pinned memory
            pkg.extract_features_batch_streamed(model, farm_host, farm_atp, farm_emb, args.batch_tokens)
            return
        if farm:
            for th in farm_host:                       # contiguous pinned views sized for this MSA
                c = th.shape[-1]
                pkg.extract_features_streamed(model, th, atp_host.view(-1)[:NL * H * (c - 1) ** 2].view(NL * H, c - 1, c - 1),
                                              emb_host.view(-1)[:(c - 1) * D].view(c - 1, D))
            return
        if shard and args.fused:
            # every rank DMAs the map rows it owns into the shared host buffer over its own PCIe link, rank 0 its emb
            sharded_forward(model, tok_host.cuda(non_blocking=True), fused=True, host_out=shard_host, gather_maps=False)
            return
        if shard:
            out = sharded_forward(model, tok_host.cuda(non_blocking=True), fused=False)
            if rank == 0:                                           # rank 0 owns MSA row 0 and writes the files
                att = out["row_attentions"][..., 1:, 1:].reshape(-1, C - 1, C - 1)
                atp_host.copy_(att, non_blocking=True)
                emb_host.copy_(out["representations"][NL][0, 0, 1:, :], non_blocking=True)
            torch.cuda.synchronize()
            return
        # public API: forward + the reference's slicing, D2H of every layer's maps overlapped with the next layer
        pkg.extract_features_streamed(model, tok_host, atp_host, emb_host)

    # ---- warm-up, then the device-timed region with per-kernel-class events recording -----------
    for _ in range(max(args.warmup, 3)):
        step_device()
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    launches0 = _lib.lib.rnamsm_launch_count()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps - 1):
        step_device()
    last = step_device()
    ev1.record()
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    del last
    launches = _lib.lib.rnamsm_launch_count() - launches0
    # per-kernel-class CUDA events over a second, identical region of K steps: two event records around each of the
    # ~132 launches per forward cost ~0.5 ms, which would be charged to `value` if they sat in the region above
    _lib.profile_enable(True)
    barrier()
    for _ in range(args.steps):
        step_device()
    barrier()
    prof = _lib.profile_collect()
    _lib.profile_enable(False)

    # ---- end-to-end region (host tokens in, emb + atp back on the host, every step) --------------
    for _ in range(2):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    barrier()
    e2e_s = time.perf_counter() - t0
    clocks = sampler.finish() if sampler else None

    if world > 1:
        tt = torch.tensor([ms_total, e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_total, e2e_s = float(tt[0]), float(tt[1])

    if rank == 0:
        ms_per_step = ms_total / args.steps
        jobs = 1 if (shard or farm) else world   # sharded / cfg3: tokens_per_step already is the whole job
        value = jobs * tokens_per_step / (ms_per_step * 1e-3)
        e2e_value = jobs * tokens_per_step / (e2e_s / args.steps)
        peaks = measured_peaks()
        if farm:                                        # this rank's MSAs
            fl = {}
            for c in my_C:
                for k, v in class_flops(R, c).items():
                    fl[k] = fl.get(k, 0.0) + v
        else:
            fl = class_flops(R, C)
        if shard:                                       # per-rank share of the one sharded MSA
            fl = {k: v / world for k, v in fl.items()}
        gemm_classes = ["linear_qkv", "linear_out_resid", "linear_fc1_gelu", "linear_fc2_resid"]
        gemm_ms = sum(prof[k][0] for k in gemm_classes)
        gemm_launches = sum(prof[k][1] for k in gemm_classes)
        gemm_flops_per_step = sum(fl[k] for k in gemm_classes)
        kernel_ms_total = sum(v[0] for v in prof.values())
        shares = {k: round(v[0] / kernel_ms_total, 4) for k, v in prof.items() if v[1]}
        tflops = {k: round(fl[k] * args.steps / (prof[k][0] * 1e-3) / 1e12, 1) for k in fl if prof.get(k, (0, 0))[0] > 0}
        achieved = gemm_flops_per_step * args.steps / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
        peak = peaks["bf16_sustained"] if args.precision not in ("fp32", "tf32x3") else None
        roofline = {
            "kernel": "umma_gemm_kernel<DENSE> (2-CTA tcgen05 dense linear: QKV / out-proj / fc1+GELU / fc2)"
                      if args.precision not in ("fp32", "tf32x3") else
                      ("umma_gemm_kernel<DENSE, tf32> (three kind::tf32 MMAs on hi / lo operand halves)" if args.precision == "tf32x3"
                       else "sgemm_kernel<LinearProb> (fp32 FFMA)"),
            "bound": "tensor", "achieved": round(achieved, 2), "peak": peak, "unit": "TFLOP/s",
            "frac": round(achieved / peak, 4) if peak else None,
            "peak_source": f"{peaks['source']} bf16_tflops_sustained (cuBLAS bf16; kind::f16 runs fp16 and bf16 at the same "
                           "rate; kernel timed inside a long step)",
            "flops_per_launch": gemm_flops_per_step / max(1, gemm_launches / args.steps),
            "avg_launch_ms": gemm_ms / max(1, gemm_launches), "launches": gemm_launches,
            "share_of_kernel_time": round(gemm_ms / kernel_ms_total, 4) if kernel_ms_total else None,
            "traffic": measured_traffic(args.workload, args.precision)[0] if not (shard or farm) else None,
            "traffic_unit": "bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum, profiles/r01e_traffic.json)",
            "algorithmic_bytes_per_launch": measured_traffic(args.workload, args.precision)[1] if not (shard or farm) else None,
            "class_time_share": shares, "class_tflops": tflops,
            "whole_forward_tflops_per_gpu": round((sum(total_flops(R, c) for c in my_C) if farm else total_flops(R, C) / (world if shard else 1))
                                                  * args.steps / (ms_total * 1e-3) / 1e12, 2),
        }
        cpu = None
        if world == 1 and not args.no_cpu_baseline:     # contract: the CPU baseline is timed at N=1 only
            c_cpu = sorted(lens)[len(lens) // 2] if farm else C   # cfg3: bounded sample = the median-length MSA
            t_emb, t_layer, threads, kind, what = cpu_reference_sample(R, c_cpu, epm)
            per_fwd = t_emb + NL * t_layer
            cpu = {"value": R * c_cpu / per_fwd, "unit": "tokens/s", "cores": threads, "kind": kind,
                   "sample": f"{what} = {t_emb + t_layer:.1f} s measured; value = tokens / (t_emb + {NL} x t_layer)"}
        secondary = run_secondary(args, pkg, _lib, world, rank, peaks) if want_secondary else None
        line = {
            "metric": METRIC, "value": value, "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong" if shard else "weak",
            "vs_baseline": None, "dtype": {"fp16": "fp16", "bf16": "bf16", "bf16_pure": "bf16", "fp32": "f32", "tf32x3": "tf32x3"}[args.precision],
            "data": "synthetic",
            "config": _config(desc, R, C, tokens_per_step, batch_tokens=(args.batch_tokens if farm else None),
                              tokens_per_step_scope="whole job" if (shard or farm) else "per GPU (x n_gpus independent MSAs)",
                              precision=f"{args.precision}: 16-bit operands on tcgen05 (kind::f16), fp32 accumulate / residual "
                                        "stream / LayerNorm / softmax / exported maps" if args.precision not in ("fp32", "tf32x3")
                                        else ("fp32 FFMA parity path" if args.precision == "fp32" else
                                              "fp32 storage / attention, nn.Linear layers as tf32 x 3 on tcgen05"),
                              parallelism=(f"one MSA sharded over {world} GPUs: rows (tied row attention, fp32 logit exchange) "
                                           f"<-> columns (column attention, 16-bit re-layout), "
                                           + ("fused peer-memory kernels over NVLink" if args.fused else "NCCL over NVLink")) if shard
                                          else f"dp{world} independent MSAs, no collective",
                              l2="no explicit flush: per-step working set (>= 1.4 GB activations + 183 MB weights at "
                                 "cfg2) exceeds the 126 MB L2"),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "tokens/s", "h2d_bytes_per_step": (sum(t.numel() for t in farm_host) if farm else tok_host.numel()) * 8,
                    "d2h_bytes_per_step": (sum(NL * H * (c - 1) ** 2 + (c - 1) * D for c in my_C) if farm
                                           else atp_host.numel() + emb_host.numel()) * 4,
                    "ms_per_step": e2e_s / args.steps * 1e3},
            "gpu_launches": int(launches),
            "roofline": roofline,
            "cpu_baseline": cpu,
            "secondary": secondary,
        }
        print(json.dumps(line), flush=True)
    elif want_secondary:
        run_secondary(args, pkg, _lib, world, rank, measured_peaks())
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="fp16", choices=["fp16", "bf16", "bf16_pure", "tf32x3", "fp32"])
    ap.add_argument("--batch-tokens", type=int, default=0,
                    help="cfg3 only: group the MSAs into forward_batch passes of at most this many tokens "
                         "(0 = one forward per MSA, the reference's B=1 loop)")
    ap.add_argument("--no-secondary", action="store_true",
                    help="skip the `secondary` block (cfg5 / cfg4 / cfg1 / fp32 at N = 1; the sharded single-MSA forward "
                         "with its parity check at N > 1)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU baseline sample (development runs)")
    ap.add_argument("--shard", action="store_true",
                    help="N > 1: ONE deep MSA sharded over the ranks (rows for tied row attention, columns for column "
                         "attention; NCCL all-reduce + all-to-all) -> strong scaling.  Default: independent MSAs, weak.")
    ap.add_argument("--fused", action="store_true",
                    help="with --shard: the peer-memory schedule (softmax pulling/pushing logits over NVLink, LayerNorm "
                         "pushing rows to the column owners, out-projection reducing into the row owners' residual)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32, at most 64 MB in all; "
                         "single-MSA workloads, rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload == "cfg3" or args.shard):
        ap.error("--dump-outputs needs --impl ours, a single-MSA workload (not cfg3) and no --shard")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
