"""Feature extraction, the B200 counterpart of ``RNA_MSM_Inference.py`` (reference lines 90-168):
for every RNA id, MSA -> tokens -> ``MSATransformer`` -> ``<id>_atp.npy`` ``(120, L, L)`` f32 and
``<id>_emb.npy`` ``(L, 768)`` f32, byte-compatible with what the ``_downstream_tasks`` SS / RSA
predictors read.  Same knob names as the reference's hydra config (``data.*`` / ``model.*``),
exposed through argparse because hydra is not a dependency here::

    python -m rnamsm_b200.inference --root_path . --MSA_path results --MSA_list rna_id.txt \
        --model_path pretrained/RNA_MSM_pretrained.ckpt
"""
from __future__ import annotations

import argparse
import os
import sys
from typing import Dict, Optional, Tuple

import numpy as np
import torch

from .alphabet import Alphabet, Vocab, tokenize_msa
from .model import MSATransformer


def extract_features(results: Dict[str, object], vocab: Vocab, num_layers: int) -> Tuple[np.ndarray, np.ndarray]:
    """RNA_MSM_Inference.py:150-166: strip BOS row/column, flatten (layer, head) -> 120 maps, and
    take MSA row 0 of the final representation.  One D2H copy per output."""
    attentions = results["row_attentions"]
    start_idx = int(vocab.prepend_bos)
    end_idx = attentions.size(-1) - int(vocab.append_eos)
    attentions = attentions[..., start_idx:end_idx, start_idx:end_idx]
    seqlen = attentions.size(-1)
    atp = attentions.reshape(-1, seqlen, seqlen).cpu().numpy()
    embedding = results["representations"][num_layers]
    end_idx = embedding.size(-2) - int(vocab.append_eos)
    emb = embedding[:, 0, start_idx:end_idx, :].squeeze(0).cpu().numpy()
    return emb, atp


@torch.no_grad()
def extract_features_windowed(model: MSATransformer, tokens: torch.Tensor, window: Optional[int] = None,
                              stride: Optional[int] = None) -> Tuple[np.ndarray, np.ndarray]:
    """``extract_features`` for an alignment of any length: ``MSATransformer.forward_windows`` (overlapping windows of
    at most the learned positions, stitched with tent weights) -> ``(emb (L, D), atp (N*H, L, L))`` as numpy, the
    ``*_emb.npy`` / ``*_atp.npy`` layout.  Pairs further apart than the windows reach are 0 in ``atp``.  For
    ``L <= window`` this is exactly ``extract_features(model(tokens, ...))``."""
    out = model.forward_windows(tokens.to(model.device), window=window, stride=stride)
    return out["emb"].cpu().numpy(), out["atp"].cpu().numpy()


@torch.no_grad()
def extract_features_streamed(model: MSATransformer, tokens: torch.Tensor, atp_host: torch.Tensor,
                              emb_host: torch.Tensor) -> None:
    """``RNA_MSM_Inference.py:147-166`` for one MSA with the device->host copies overlapped with compute:
    the forward runs layer by layer (``rnamsm_layer_forward``) and every layer's 12 maps start their copy into
    the pinned ``atp_host [(N*H), L, L]`` on a side stream while the next layer computes; ``emb_host [L, D]``
    follows the final LayerNorm.  ``tokens``: ``[1, R, C]`` int64, pinned host or device.  Returns when both
    host buffers are complete."""
    import ctypes as C
    from . import _lib as L
    dev = model.device
    vocab = model.vocab
    assert tokens.ndim == 3 and tokens.shape[0] == 1
    _, R, Cc = tokens.shape
    D, H, N = model.embed_dim, model.num_attention_heads, model.num_layers
    start = int(vocab.prepend_bos)
    Ls = Cc - start - int(vocab.append_eos)
    with torch.cuda.device(dev):
        code = model._code
        main = torch.cuda.current_stream()
        side = getattr(model, "_copy_stream", None)
        if side is None:
            side = model._copy_stream = torch.cuda.Stream()
        tok = tokens.to(dev, non_blocking=True).long().contiguous()
        # same limits and exceptions as forward(); host tokens are checked on the host, so the first kernel does not
        # wait for a device -> host round trip of the "any padding?" flag (model.py:347)
        has_pad, _ = model.check_tokens(tokens if tokens.device.type == "cpu" else tok)
        x = torch.empty((R * Cc, D), dtype=torch.float32, device=dev)
        pad = torch.empty(R * Cc, dtype=torch.uint8, device=dev)
        maps = torch.empty((N, H, Cc, Cc), dtype=torch.float32, device=dev)
        m = model.c_weights(code)
        fcode = model._fwd_code
        nbytes = L.lib.rnamsm_workspace_bytes(R, Cc, D, H, 4 * D, fcode)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        st = L.stream_ptr()
        L.check(L.lib.rnamsm_embed_layernorm(L.ptr(tok[0]), R, Cc, m.tok_emb, m.vocab, m.pos_emb, m.n_pos, m.row_pos,
                                             m.ln_before_w, m.ln_before_b, D, m.pad_idx, m.ln_eps, L.ptr(x), L.ptr(pad), st),
                "embed_layernorm")
        chain = bool(L.lib.rnamsm_fused_layernorm(code))   # layer l's fc2 epilogue writes layer l+1's first LayerNorm
        for l in range(N):
            nxt = m.layers[l + 1].row if (chain and l + 1 < N) else None
            L.check(L.lib.rnamsm_layer_forward(C.byref(m.layers[l]), D, H, 4 * D, m.ln_eps, L.ptr(x), R, Cc,
                                               L.ptr(pad) if has_pad else None, fcode, L.ptr(maps[l]), L.ptr(ws), nbytes,
                                               int(chain and l > 0), nxt.ln_w if nxt is not None else None,
                                               nxt.ln_b if nxt is not None else None, nxt.dtype if nxt is not None else 0, st),
                    "layer_forward")
            ev = torch.cuda.Event()
            ev.record(main)
            side.wait_event(ev)
            if atp_host.is_contiguous() and atp_host.dtype == torch.float32 and tuple(atp_host.shape[-2:]) == (Ls, Ls):
                # one pitched DMA per layer straight into the *_atp.npy layout: no staging kernel on the GPU
                L.check(L.lib.rnamsm_copy_map_rows_d2h(L.ptr(maps[l]), H, Cc, 0, Cc, start, Ls, atp_host[l * H].data_ptr(),
                                                       side.cuda_stream), "copy_map_rows_d2h")
            else:
                with torch.cuda.stream(side):
                    atp_host[l * H:(l + 1) * H].copy_(maps[l, :, start:start + Ls, start:start + Ls], non_blocking=True)
        # *_emb.npy is MSA row 0 of the final representation (RNA_MSM_Inference.py:159-166): the final LayerNorm is
        # token-local, so only that row's C tokens are normalised here (forward() returns all rows and normalises all)
        L.check(L.lib.rnamsm_layernorm(L.ptr(x), m.ln_after_w, m.ln_after_b, L.ptr(x), L.F32, Cc, D, m.ln_eps, 0, 0, st),
                "layernorm")
        emb_host.copy_(x.view(R, Cc, D)[0, start:start + Ls], non_blocking=True)
        maps.record_stream(side)
        side.synchronize()
        main.synchronize()


@torch.no_grad()
def pack_ss_input(row_attentions: torch.Tensor, sequence: str, prepend_bos: bool = True) -> torch.Tensor:
    """The ``[1, 128, L, L]`` input of the downstream SS predictor (``_downstream_tasks/SS``:
    ``DataProcess.feature_load`` + ``format_input_shape``) built on the device from ``row_attentions
    [1, N, H, C, C]`` -- no ``*_atp.npy`` round trip, no O(L^2) Python loop (``outer_concatenation``)."""
    from . import _lib as L
    L.require_cuda(row_attentions, "row_attentions")
    _, N, H, Cc, _ = row_attentions.shape
    start = int(prepend_bos)
    Ls = Cc - start
    if len(sequence) != Ls:
        raise ValueError(f"sequence length {len(sequence)} != map size {Ls}")
    codes = torch.tensor([_SEQ_CODES.get(ch, 255) for ch in sequence], dtype=torch.uint8, device=row_attentions.device)
    maps = row_attentions[0].float().contiguous()
    out = torch.empty((1, 8 + N * H, Ls, Ls), dtype=torch.float32, device=maps.device)
    with torch.cuda.device(maps.device):
        L.check(L.lib.rnamsm_ss_pack(L.ptr(maps), N * H, Cc, start, Ls, L.ptr(codes), L.ptr(out), L.stream_ptr()), "ss_pack")
    return out


@torch.no_grad()
def extract_features_batch_streamed(model: MSATransformer, tokens_list, atp_hosts, emb_hosts,
                                    token_budget: int = 262144) -> None:
    """``extract_features_batch`` with host buffers on both sides: ``tokens_list[i]`` ``[1, R_i, C_i]`` (pinned host
    or device), ``atp_hosts[i]`` ``[(N*H), L_i, L_i]`` and ``emb_hosts[i]`` ``[L_i, D]`` pinned fp32.  Each group's
    device->host copies run on a side stream while the next group computes.  Returns when every buffer is complete."""
    vocab, N, H = model.vocab, model.num_layers, model.num_attention_heads
    start = int(vocab.prepend_bos)
    shapes = [tuple(t.shape[-2:]) for t in tokens_list]
    with torch.cuda.device(model.device):
        main = torch.cuda.current_stream()
        side = getattr(model, "_copy_stream", None)
        if side is None:
            side = model._copy_stream = torch.cuda.Stream()
        for batch in plan_batches(shapes, token_budget):
            res = model.forward_batch([tokens_list[i].to(model.device, non_blocking=True) for i in batch],
                                      need_head_weights=True)
            ev = torch.cuda.Event()
            ev.record(main)
            with torch.cuda.stream(side):
                side.wait_event(ev)
                for i, r in zip(batch, res):
                    Ls = shapes[i][1] - start - int(vocab.append_eos)
                    att, rep = r["row_attentions"], r["representations"][N]
                    atp_hosts[i].copy_(att[0, :, :, start:start + Ls, start:start + Ls].reshape(N * H, Ls, Ls),
                                       non_blocking=True)
                    emb_hosts[i].copy_(rep[0, 0, start:start + Ls], non_blocking=True)
                    att.record_stream(side)
                    rep.record_stream(side)
        side.synchronize()
        main.synchronize()


_SEQ_CODES = {"A": 0, "C": 1, "G": 2, "U": 3}


@torch.no_grad()
def pack_rsa_input(representation: torch.Tensor, sequence: str, mu_emb, std_emb, mu_oh=None, std_oh=None,
                   prepend_bos: bool = True) -> torch.Tensor:
    """The ``[1, 4 + D + 1, L]`` input of the downstream RSA predictor (``_downstream_tasks/RSA/predict.py:131-141``:
    z-scored one-hot | z-scored embedding | ones, channels first) built on the device from
    ``representations[num_layers]`` ``[1, R, C, D]`` -- no ``*_emb.npy`` round trip.  ``mu_*`` / ``std_*`` are the
    arrays of the predictor's ``statistic_dict_{oh,emb}.pickle``; without ``mu_oh`` the one-hot channels are left
    out (the embedding-only predictor, ``models/RNA-MSM_Emb``).  Bit-identical to the reference's expression."""
    import ctypes as C
    from . import _lib as L
    L.require_cuda(representation, "representation")
    assert representation.ndim == 4 and representation.shape[0] == 1
    _, R, Cc, D = representation.shape
    start = int(prepend_bos)
    Ls = Cc - start
    if len(sequence) != Ls:
        raise ValueError(f"sequence length {len(sequence)} != embedding length {Ls}")
    if (mu_oh is None) != (std_oh is None):
        raise ValueError("mu_oh and std_oh go together")
    dev = representation.device
    x = representation.float().contiguous()
    codes = torch.tensor([_SEQ_CODES.get(ch, 255) for ch in sequence], dtype=torch.uint8, device=dev)
    mu = torch.as_tensor(np.asarray(mu_emb, dtype=np.float32)).to(dev)
    sd = torch.as_tensor(np.asarray(std_emb, dtype=np.float32)).to(dev)
    if mu.numel() != D or sd.numel() != D:
        raise ValueError(f"mu_emb / std_emb must have {D} entries")
    n_oh = 4 if mu_oh is not None else 0
    oh_mu = (C.c_double * 4)(*np.asarray(mu_oh, dtype=np.float64).tolist()) if n_oh else None
    oh_sd = (C.c_double * 4)(*np.asarray(std_oh, dtype=np.float64).tolist()) if n_oh else None
    out = torch.empty((1, n_oh + D + 1, Ls), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        L.check(L.lib.rnamsm_rsa_pack(x[0, 0, start:].data_ptr(), D, Ls, D, L.ptr(codes), oh_mu, oh_sd, L.ptr(mu), L.ptr(sd),
                                      L.ptr(out), L.stream_ptr()), "rsa_pack")
    return out


def plan_batches(shapes, token_budget: int = 262144):
    """Group MSAs ``[(R, C), ...]`` for ``MSATransformer.forward_batch``: largest first, each batch filled with
    the largest remaining alignments that still fit ``token_budget`` tokens (an alignment above the budget
    runs alone).  Returns lists of indices into ``shapes``; every index appears exactly once."""
    order = sorted(range(len(shapes)), key=lambda i: -shapes[i][0] * shapes[i][1])
    batches, used = [], [False] * len(shapes)
    for i in order:
        if used[i]:
            continue
        used[i] = True
        batch, room = [i], token_budget - shapes[i][0] * shapes[i][1]
        for j in order:
            t = shapes[j][0] * shapes[j][1]
            if not used[j] and t <= room:
                used[j] = True
                batch.append(j)
                room -= t
        batches.append(batch)
    return batches


@torch.no_grad()
def extract_features_batch(model: MSATransformer, tokens_list, token_budget: int = 262144):
    """``RNA_MSM_Inference.py:147-166`` for many MSAs: grouped by ``plan_batches`` and run through
    ``forward_batch``; returns ``[(emb (L_i, D), atp (N*H, L_i, L_i)), ...]`` as numpy arrays in input order,
    identical to calling ``extract_features(model(tokens_i, ...))`` one MSA at a time."""
    vocab, N = model.vocab, model.num_layers
    shapes = [tuple(t.shape[-2:]) for t in tokens_list]
    out = [None] * len(tokens_list)
    for batch in plan_batches(shapes, token_budget):
        res = model.forward_batch([tokens_list[i].to(model.device) for i in batch], need_head_weights=True)
        for i, r in zip(batch, res):
            out[i] = extract_features(r, vocab, N)
    return out


def build_model(model_path: Optional[str], device: str = "cuda", precision: str = "fp16", embed_dim: int = 768,
                num_attention_heads: int = 12, num_layers: int = 10, embed_positions_msa: bool = True,
                max_tokens: int = 16384, max_seqlen: int = 1024, seed: int = 42) -> Tuple[MSATransformer, Vocab]:
    alphabet = Alphabet.from_architecture("rna language")
    vocab = Vocab.from_esm_alphabet(alphabet)
    torch.manual_seed(seed)                                   # seed_everything(42), RNA_MSM_Inference.py:17
    model = MSATransformer(vocab, embed_dim=embed_dim, num_attention_heads=num_attention_heads,
                           num_layers=num_layers, embed_positions_msa=embed_positions_msa,
                           max_tokens_per_msa=max_tokens, max_seqlen=max_seqlen, precision=precision)
    if model_path:
        ckpt = torch.load(model_path, map_location="cpu")
        model.load_state_dict(ckpt["state_dict"] if "state_dict" in ckpt else ckpt, strict=True)
    model = model.eval().to(device)
    return model, vocab


@torch.no_grad()
def run_inference(model: MSATransformer, vocab: Vocab, root_path: str, MSA_path: str, rna_ids, max_seqs_per_msa=512,
                  max_seqlen=1024, verbose=True, sample_method: str = "first", long_mode: str = "crop",
                  window: Optional[int] = None, stride: Optional[int] = None) -> str:
    """``long_mode``: what happens to an alignment longer than ``max_seqlen - 1`` columns.  ``"crop"`` (the reference's
    behaviour) keeps its first ``max_seqlen - 1`` columns; ``"window"`` keeps every column and writes full-length
    features from overlapping windows (``extract_features_windowed`` with ``window`` / ``stride``)."""
    if long_mode not in ("crop", "window"):
        raise ValueError(f"long_mode {long_mode!r}: expected 'crop' or 'window'")
    if long_mode == "crop" and (window is not None or stride is not None):
        raise ValueError("window and stride apply to long_mode='window' only")
    save_feat_path = os.path.join(root_path, MSA_path)
    os.makedirs(save_feat_path, exist_ok=True)
    for rna_id in sorted(rna_ids):
        msa_file = os.path.join(root_path, MSA_path, rna_id + ".a2m_msa2")
        # MSA ingest on the device (csrc/ingest.cu): cleaning, optional diversity sub-sampling, tokenisation
        from .ingest import ingest_msa
        if long_mode == "window":
            tokens, _ = ingest_msa(msa_file, vocab, max_seqs_per_msa, sys.maxsize, sample_method, device=str(model.device))
            emb, atp = extract_features_windowed(model, tokens, window, stride)
        else:
            tokens, _ = ingest_msa(msa_file, vocab, max_seqs_per_msa, max_seqlen, sample_method, device=str(model.device))
            results = model(tokens.unsqueeze(0), repr_layers=[model.num_layers], need_head_weights=True, want_logits=False)
            emb, atp = extract_features(results, vocab, model.num_layers)
        np.save(os.path.join(save_feat_path, rna_id + "_atp.npy"), atp)
        np.save(os.path.join(save_feat_path, rna_id + "_emb.npy"), emb)
        if verbose:
            print(f"{rna_id}: tokens {tuple(tokens.shape)} -> atp {atp.shape}, emb {emb.shape}")
    if verbose:
        print(f"Done! Generated files are saved at {save_feat_path}")
    return save_feat_path


def parse_args(argv=None) -> argparse.Namespace:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--device", default="cuda")
    ap.add_argument("--root_path", default=".")
    ap.add_argument("--MSA_path", default="results")
    ap.add_argument("--MSA_list", default="rna_id.txt")
    ap.add_argument("--model_path", default=None, help="Lightning checkpoint ('state_dict'); random init if omitted")
    ap.add_argument("--max_seqlen", type=int, default=1024)
    ap.add_argument("--max_tokens", type=int, default=16384)
    ap.add_argument("--max_seqs_per_msa", type=int, default=512)
    ap.add_argument("--sample_method", default="first", choices=["first", "diversity-max", "diversity-min"],
                    help="the reference's default 'hhfilter' needs an external binary; 'first' keeps the first rows "
                         "(what it does with hhfilter's surplus), 'diversity-*' is MSA.greedy_select on the GPU")
    ap.add_argument("--embed_dim", type=int, default=768)
    ap.add_argument("--num_attention_heads", type=int, default=12)
    ap.add_argument("--num_layers", type=int, default=10)
    ap.add_argument("--no_embed_positions_msa", action="store_true")
    ap.add_argument("--precision", default="fp16", choices=["fp16", "bf16", "bf16_pure", "tf32x3", "fp32"])
    ap.add_argument("--long", default="crop", choices=["crop", "window"],
                    help="alignments longer than max_seqlen - 1 columns: 'crop' keeps the first max_seqlen - 1 columns "
                         "(the reference's behaviour); 'window' writes full-length features from overlapping windows")
    ap.add_argument("--window", type=int, default=None,
                    help="--long window: window width in residues (default: the learned positions, max_seqlen - 1)")
    ap.add_argument("--stride", type=int, default=None, help="--long window: window stride (default: window // 2)")
    a = ap.parse_args(argv)
    if a.long == "crop" and (a.window is not None or a.stride is not None):
        ap.error("--window and --stride need --long window")
    for name in ("window", "stride"):
        v = getattr(a, name)
        if v is not None and v < 1:
            ap.error(f"--{name} must be >= 1 (got {v})")
    return a


def main(argv=None):
    a = parse_args(argv)
    model, vocab = build_model(a.model_path, a.device, a.precision, a.embed_dim, a.num_attention_heads, a.num_layers,
                               not a.no_embed_positions_msa, a.max_tokens, a.max_seqlen)
    print(f"Maximum Number of MSA Seqs:{a.max_seqs_per_msa}")
    print(f"Inference on: {model.device}")
    with open(os.path.join(a.root_path, a.MSA_list)) as f:
        ids = f.read().splitlines()
    run_inference(model, vocab, a.root_path, a.MSA_path, ids, a.max_seqs_per_msa, a.max_seqlen,
                  sample_method=a.sample_method, long_mode=a.long, window=a.window, stride=a.stride)


if __name__ == "__main__":
    main()
