"""Routes of the whole forward, their boundary shapes, float64 references and the child-process runner.

`layer_forward` (rna-msm_b200/csrc/api.cu) chains different kernels depending on R (rows), C (columns, BOS included) and
the precision.  `routes()` restates its predicates in plain Python:

  row    16-bit tied row attention: "short" (row_attn_short.cu, one cooperative launch) when
         rnamsm_row_attn_short_chunks(R, C, 12) > 0, otherwise "chain" (logits -> softmax -> A V); "f32" on the fp32 path
  col    column attention: "r1" (R == 1: out_proj(v_proj(x))), 16-bit "umma" (col_attn_umma.cu, R <= 128) or "fa"
         (col_attn_fa.cu, R > 128), "f32" on the fp32 path
  qkv    layout of the column block's q|k|v: "col_major" for 16-bit with R > 1, else "token_major"
  dense  nn.Linear layers: "tf32x3" when the fp32 path runs with RNAMSM_F32_TENSOR and N % 32 == 0 and K % 32 == 0,
         "ffma" on the plain fp32 path, "umma16" in 16 bits

On a machine without a device the short row attention is assumed to apply for C <= 128 (its only shape condition; the
device adds the residency check, 12 heads always fit a B200).  Every shape case lists the routes it is expected to hit.

The module also runs as a script in a child process with a different environment (RNAMSM_FUSE_LN, RNAMSM_PDL and
RNAMSM_ROW_SHORT are read once per process):

    python tests/forward_routes.py OUT.pt

runs `child_outputs` -- forward with head weights, forward_batch, extract_features_streamed and the column-probabilities
entry, in fp16 and bf16, at the boundary shapes -- and saves every output for the parent to compare.
"""
from __future__ import annotations

import argparse
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import msa_ref as O  # noqa: E402

H = O.NUM_HEADS
D = O.EMBED_DIM
LAYERS = 2
WSEED, SHARPEN = 11, 2.0
SHORT_MAX_C = 128          # row_attn_short.cu kMaxC
UMMA_MAX_R = 128           # col_attn_umma.cu launch_col_attn_16: R <= 128 keeps the small-depth kernel
PRECISIONS = ["fp32", "tf32x3", "fp16", "bf16"]
SIXTEEN = ("fp16", "bf16")
SWITCHES = ("RNAMSM_FUSE_LN", "RNAMSM_PDL", "RNAMSM_ROW_SHORT")
CHILD_ENVS = {"default": {}, "fuse_ln": {"RNAMSM_FUSE_LN": "1"}, "pdl": {"RNAMSM_PDL": "1"},
              "row_short0": {"RNAMSM_ROW_SHORT": "0"}}


# ------------------------------------------------------------------------------------------ dispatch mirror
def short_chunks(R: int, C: int, lib=None) -> int:
    """Row chunks of the one-launch row attention, 0 when the three-kernel chain runs (lib: the loaded library)."""
    if lib is not None:
        return int(lib.rnamsm_row_attn_short_chunks(R, C, H))
    return 1 if 1 <= C <= SHORT_MAX_C else 0


def dense_route(precision: str, N: int, K: int) -> str:
    if precision in SIXTEEN:
        return "umma16"
    if precision == "tf32x3" and N % 32 == 0 and K % 32 == 0:
        return "tf32x3"
    return "ffma"


# (N, K) of every nn.Linear the forward runs: q|k|v, out_proj / LM dense / the R == 1 v projection, fc1, fc2
MODEL_GEMMS = [(3 * D, D), (D, D), (4 * D, D), (D, 4 * D)]


def routes(R: int, C: int, precision: str, lib=None) -> dict:
    sixteen = precision in SIXTEEN
    if sixteen:
        row = "short" if short_chunks(R, C, lib) > 0 else "chain"
        col = "r1" if R == 1 else ("umma" if R <= UMMA_MAX_R else "fa")
    else:
        row, col = "f32", ("r1" if R == 1 else "f32")
    dense = sorted({dense_route(precision, N, K) for N, K in MODEL_GEMMS})
    return {"row": row, "col": col, "qkv": "col_major" if sixteen and R > 1 else "token_major", "dense": "+".join(dense)}


# ------------------------------------------------------------------------------------------ boundary shapes
class Case:
    """One alignment: R rows, C columns (BOS included) and a pad layout:
      none   no padding
      cols   trailing pad columns in every row
      mid    one pad in the middle of row 0 (the row attention's key mask comes from row 0)
      rows   fully padded trailing rows (BOS column included)"""

    def __init__(self, R: int, C: int, pad: str, seed: int):
        self.R, self.C, self.pad, self.seed = R, C, pad, seed
        self.name = f"{R}x{C}-{pad}"

    def tokens(self) -> torch.Tensor:
        t = O.make_tokens(self.R, self.C, self.seed)
        if self.pad == "cols":
            t[:, :, self.C - self.pad_cols():] = O.PAD_IDX
        elif self.pad == "mid":
            t[0, 0, self.C // 2] = O.PAD_IDX
        elif self.pad == "rows":
            t[0, self.R - self.pad_rows():, :] = O.PAD_IDX
        return t

    def pad_cols(self) -> int:
        return max(1, min(5, (self.C - 1) // 4))

    def pad_rows(self) -> int:
        return max(1, self.R // 8)

    def valid(self) -> bool:
        """Row 0 keeps its BOS and a residue, so no key column and no alignment column is fully masked."""
        if self.pad == "cols":
            return self.C - self.pad_cols() >= 2
        if self.pad == "mid":
            return self.C >= 3
        if self.pad == "rows":
            return self.R >= 2
        return True

    def __repr__(self):
        return self.name


# Ordered by size: the largest shapes run last.  Each threshold (C <= 128, R <= 128, R == 1) has a case on each side.
CASES = [Case(3, 1, "none", 1), Case(2, 2, "none", 2), Case(2, 128, "mid", 3), Case(2, 129, "cols", 4),
         Case(1, 129, "cols", 5), Case(1, 300, "mid", 6), Case(127, 9, "rows", 7), Case(128, 9, "cols", 8),
         Case(129, 9, "mid", 9), Case(300, 33, "cols", 10), Case(128, 128, "rows", 11), Case(257, 64, "rows", 12),
         Case(64, 257, "mid", 13), Case(129, 129, "rows", 14)]
CASE = {c.name: c for c in CASES}

# The dispatch thresholds of `routes`: tests/test_forward_routes_cpu.py checks that CASES sit on both sides of each.
THRESHOLDS = {"C<=128": lambda c: c.C <= SHORT_MAX_C, "R<=128": lambda c: c.R <= UMMA_MAX_R, "R==1": lambda c: c.R == 1}

# forward_batch members across the boundaries (R, C, pad layout): chain / short rows, umma / fa columns, padded rows
BATCH_MEMBERS = [Case(2, 129, "none", 21), Case(129, 9, "none", 22), Case(128, 128, "none", 23), Case(64, 257, "none", 24),
                 Case(40, 17, "rows", 25)]

# the child's list: every route, kept small enough that its outputs fit one file comfortably
CHILD_CASES = ["3x1-none", "2x2-none", "2x128-mid", "2x129-cols", "1x129-cols", "1x300-mid", "127x9-rows", "128x9-cols",
               "129x9-mid", "300x33-cols", "128x128-rows"]
CHILD_BATCH = [Case(2, 129, "none", 31), Case(129, 9, "mid", 32), Case(40, 17, "rows", 33), Case(7, 140, "cols", 34)]
CHILD_COL_PROBS = ["2x129-cols", "129x9-mid", "128x9-cols"]


# ------------------------------------------------------------------------------------------ float64 reference
def weights(dtype=torch.float32):
    sd = O.make_weights(WSEED, num_layers=LAYERS, sharpen=SHARPEN)
    return sd if dtype == torch.float32 else O.to_dtype(sd, dtype)


def reference(tokens: torch.Tensor, sd=None, device="cpu", dtype=torch.float64) -> dict:
    """O.forward of the 2-layer seeded weights in `dtype` on `device` (the oracle is plain torch and device-agnostic):
    representations of layers 0, 1, 2, logits and row attentions."""
    if sd is None:
        sd = weights(dtype)
    sd = {k: v.to(device) for k, v in sd.items()}
    return O.forward(sd, tokens.to(device), repr_layers=[0, 1, LAYERS], need_head_weights=True, num_layers=LAYERS)


# ------------------------------------------------------------------------------------------ runs on the device
def build_model(pkg, precision: str):
    model = pkg.MSATransformer(pkg.Vocab(pkg.Alphabet()), num_layers=LAYERS, precision=precision)
    model.load_state_dict(weights(), strict=True)
    return model.eval().cuda()


def forward_outputs(model, tokens: torch.Tensor) -> dict:
    """{rep0, rep1, rep2, logits, maps} of model.forward with head weights."""
    out = model(tokens.cuda(), repr_layers=[0, 1, LAYERS], need_head_weights=True)
    reps = out["representations"]
    return {"rep0": reps[0], "rep1": reps[1], "rep2": reps[LAYERS], "logits": out["logits"], "maps": out["row_attentions"]}


def batch_outputs(model, cases) -> dict:
    outs = model.forward_batch([c.tokens().cuda() for c in cases], need_head_weights=True)
    res = {}
    for c, o in zip(cases, outs):
        res[f"{c.name}/rep2"] = o["representations"][LAYERS]
        res[f"{c.name}/maps"] = o["row_attentions"]
    return res


def streamed_outputs(pkg, model, tokens: torch.Tensor) -> dict:
    C = tokens.shape[-1]
    atp = torch.empty((LAYERS * H, C - 1, C - 1), dtype=torch.float32).pin_memory()
    emb = torch.empty((C - 1, D), dtype=torch.float32).pin_memory()
    pkg.extract_features_streamed(model, tokens.pin_memory(), atp, emb)
    return {"atp": atp, "emb": emb}


def col_probs_outputs(model, tokens: torch.Tensor) -> dict:
    out = model(tokens.cuda(), repr_layers=[LAYERS], need_head_weights=True, want_logits=False, need_col_weights=True,
                need_col_weights_mean=True)
    return {"col": out["col_attentions"], "col_mean": out["col_attentions_mean"], "rep2": out["representations"][LAYERS],
            "maps": out["row_attentions"]}


def child_outputs(pkg) -> dict:
    """Every output of the child's fixed list, as CPU tensors keyed '<precision>/<entry>/<case>/<output>'."""
    res = {}

    def put(prefix, d):
        for k, v in d.items():
            res[f"{prefix}/{k}"] = v.detach().cpu()

    for precision in SIXTEEN:
        model = build_model(pkg, precision)
        for name in CHILD_CASES:
            t = CASE[name].tokens()
            put(f"{precision}/forward/{name}", forward_outputs(model, t))
            if CASE[name].C >= 2:
                put(f"{precision}/streamed/{name}", streamed_outputs(pkg, model, t))
        put(f"{precision}/batch", batch_outputs(model, CHILD_BATCH))
        for name in CHILD_COL_PROBS:
            put(f"{precision}/col_probs/{name}", col_probs_outputs(model, CASE[name].tokens()))
        torch.cuda.synchronize()
        del model
    return res


def child_env(name: str, base=None) -> dict:
    """The environment of child `name`: `base` (default os.environ) without any forward switch, plus that child's."""
    env = dict(os.environ if base is None else base)
    for k in SWITCHES:
        env.pop(k, None)
    env.update(CHILD_ENVS[name])
    return env


def child_command(out_path: str) -> list:
    return [sys.executable, os.path.abspath(__file__), str(out_path)]


def parse_args(argv):
    p = argparse.ArgumentParser(description="Run the forward-route list and save every output.")
    p.add_argument("out", help="output .pt file (a dict of CPU tensors)")
    return p.parse_args(argv)


def main(argv=None) -> None:
    args = parse_args(sys.argv[1:] if argv is None else argv)
    if not torch.cuda.is_available():
        raise SystemExit("forward_routes: no CUDA device; the route list runs on the GPU only")
    import rnamsm_b200 as pkg
    from rnamsm_b200 import _lib as L
    torch.cuda.set_device(0)
    L.device_check(torch.device("cuda:0"))
    outs = child_outputs(pkg)
    outs["switches"] = {k: os.environ.get(k, "") for k in SWITCHES}
    torch.save(outs, args.out)
    print(f"forward_routes child: {len(outs) - 1} outputs, switches {outs['switches']}")


if __name__ == "__main__":
    main()
