"""``MSATransformer`` -- drop-in for the reference's top-level ``model.MSATransformer``
(model.py:258-433; ``msm/model.py:206-423`` is the same network): same constructor arguments,
same 275 state-dict keys (so the published checkpoint loads with ``strict=True``), same
``forward(tokens, repr_layers, need_head_weights, return_contacts)`` result dict.

The forward body is one call into ``rnamsm_msa_forward`` per MSA: K1 (embedding + LayerNorm) ->
10 x [LN -> QKV GEMM -> tied logits -> softmax/map export -> AV -> out-proj+residual ->
LN -> QKV GEMM -> flash column attention -> out-proj+residual -> LN -> fc1+GELU -> fc2+residual]
-> final LN (-> LM head).  The Lightning training shell of the reference (model.py:29-255) is out
of scope (SURVEY.md section 2.1).
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Iterable, List, Optional, Sequence

import torch
import torch.nn as nn

from . import _lib as L
from .alphabet import Vocab
from .modules import (AxialTransformerLayer, ColumnSelfAttention, ContactPredictionHead, LearnedPositionalEmbedding,
                      RobertaLMHead, RowSelfAttention, _PrecisionMixin, _infer_only)


class MSATransformer(nn.Module, _PrecisionMixin):
    def __init__(
        self,
        vocab: Vocab,
        optimizer_config=None,          # accepted and ignored: training shell is out of scope
        contact_train_data=None,        # accepted and ignored
        embed_dim: int = 768,
        num_attention_heads: int = 12,
        num_layers: int = 12,
        embed_positions_msa: bool = True,
        dropout: float = 0.1,
        attention_dropout: float = 0.1,
        activation_dropout: float = 0.1,
        max_tokens_per_msa: int = 2 ** 14,
        max_seqlen: int = 1024,
        precision: Optional[str] = None,
    ):
        super().__init__()
        self.vocab = vocab
        self.embed_dim = embed_dim
        self.num_attention_heads = num_attention_heads
        self.num_layers = num_layers
        self.embed_positions_msa = embed_positions_msa
        self.dropout = dropout
        self.attention_dropout = attention_dropout
        self.activation_dropout = activation_dropout
        self.max_tokens_per_msa = max_tokens_per_msa

        self.embed_tokens = nn.Embedding(len(vocab), embed_dim, padding_idx=vocab.pad_idx)
        if embed_positions_msa:
            # one SCALAR per MSA row, as in the shipped model/checkpoint (model.py:293-296)
            self.msa_position_embedding = nn.Parameter(0.01 * torch.randn(1, 1024, 1, 1), requires_grad=True)
        else:
            self.register_parameter("msa_position_embedding", None)
        self.dropout_module = nn.Dropout(dropout)
        self.layers = nn.ModuleList([
            AxialTransformerLayer(embedding_dim=embed_dim, ffn_embedding_dim=4 * embed_dim,
                                  num_attention_heads=num_attention_heads, dropout=dropout,
                                  attention_dropout=attention_dropout, activation_dropout=activation_dropout,
                                  max_tokens_per_msa=max_tokens_per_msa)
            for _ in range(num_layers)
        ])
        self.contact_head = ContactPredictionHead(num_layers * num_attention_heads, vocab.prepend_bos,
                                                  vocab.append_eos, eos_idx=vocab.eos_idx)
        self.contact_head.requires_grad_(False)
        self.embed_positions = LearnedPositionalEmbedding(max_seqlen, embed_dim, vocab.pad_idx)
        self.emb_layer_norm_before = nn.LayerNorm(embed_dim)
        self.emb_layer_norm_after = nn.LayerNorm(embed_dim)
        self.lm_head = RobertaLMHead(embed_dim=embed_dim, output_dim=len(self.vocab), weight=self.embed_tokens.weight)
        self.init_weights()
        if precision is not None:
            self.set_precision(precision)
        self._wstruct = None

    # -- reference API -------------------------------------------------------------------------
    def init_weights(self):
        """model.py:89-101."""
        for module in self.modules():
            if isinstance(module, nn.Linear):
                nn.init.normal_(module.weight, std=0.02)
                if module.bias is not None:
                    nn.init.zeros_(module.bias)
            elif isinstance(module, nn.Embedding):
                nn.init.normal_(module.weight, std=0.02)
                if module.padding_idx is not None:
                    module.weight.data[module.padding_idx].zero_()
            elif isinstance(module, nn.LayerNorm) and module.elementwise_affine:
                nn.init.ones_(module.weight)
                nn.init.zeros_(module.bias)

    @property
    def device(self) -> torch.device:
        return self.embed_tokens.weight.device

    def max_tokens_per_msa_(self, value: int) -> None:
        """Kept callable for API parity (model.py:418-428).  The reference uses it to chunk
        attention so that activations fit in memory; these kernels never materialise those
        activations, so the value is recorded and has no effect on results or memory."""
        self.max_tokens_per_msa = value
        for module in self.modules():
            if isinstance(module, (RowSelfAttention, ColumnSelfAttention)):
                module.max_tokens_per_msa = value

    @torch.no_grad()
    def check_fp16_range(self, tokens, fallback: Optional[str] = "bf16") -> Dict[str, object]:
        """Guard for weights never validated in fp16 (the trained RNA-MSM checkpoint is not available offline,
        RNA_MSM_Inference.py:133-135): runs ONE forward of ``tokens`` under the library's range watch, which scans every
        16-bit activation the forward writes (LayerNorm outputs, q|k|v, attention contexts, the post-GELU hidden) for the
        type's largest finite value -- where the fp16 kernels clamp (``cvt.rn.satfinite``).  Returns
        ``{"saturated": n, "max_abs": m, "precision": p}`` (n, m of the fp16 pass); if anything saturated and ``fallback``
        is given, the model is switched to that precision (default ``'bf16'``: fp32's exponent range; its tied row block
        is still fp16, so the watch runs once more and ``'bf16_pure'`` is selected if that block is what overflowed).
        A debugging pass: it adds one scan per activation tensor, so call it once per checkpoint / input family."""
        if self.precision not in ("fp16",):
            return {"saturated": 0, "max_abs": float("nan"), "precision": self.precision}

        def watched():
            with L.RangeWatch() as w:
                self(tokens, repr_layers=[self.num_layers], need_head_weights=True, want_logits=False)
            return w

        w = watched()
        if w.saturated and fallback is not None:
            self.set_precision(fallback)
            if fallback == "bf16" and watched().saturated:
                self.set_precision("bf16_pure")
        return {"saturated": w.saturated, "max_abs": w.max_abs, "precision": self.precision}

    def get_sequence_attention(self, tokens):
        return self(tokens.to(device=self.device), need_head_weights=True)["row_attentions"]

    def predict_contacts(self, tokens):
        return self(tokens, return_contacts=True)["contacts"]

    def check_msa_shape(self, R: int, Cc: int, n_nonpad_max: int) -> None:
        """The reference's input limits, raised identically by every entry point (forward, forward_batch, the streamed
        and the sharded paths): depth <= 1024 with the learned row positions (model.py:354-359) and non-pad length
        within the learned column positions (F.embedding raises IndexError, modules.py:292)."""
        if self.msa_position_embedding is not None and R > 1024:
            raise RuntimeError(
                "Using model with MSA position embedding trained on maximum MSA "
                f"depth of 1024, but received {R} alignments.")
        if n_nonpad_max + self.vocab.pad_idx >= self.embed_positions.weight.shape[0]:
            raise IndexError(
                f"sequence length {Cc} exceeds the {self.embed_positions.max_positions} learned positions")

    def check_tokens(self, tokens: torch.Tensor):
        """-> (has_pad, padding_mask) after check_msa_shape; one host sync, as model.py:347."""
        R, Cc = tokens.shape[-2:]
        padding_mask = tokens.eq(self.vocab.pad_idx)
        has_pad = bool(padding_mask.any())
        n_nonpad_max = int((~padding_mask).sum(-1).max()) if has_pad else Cc
        self.check_msa_shape(R, Cc, n_nonpad_max)
        return has_pad, padding_mask

    # -- C-ABI plumbing ------------------------------------------------------------------------
    def c_weights(self, code: int) -> L.ModelWeights:
        key = (code, self._row_code) + tuple((p.data_ptr(), p._version) for p in self.parameters())
        if self._wstruct is not None and self._wstruct[0] == key:
            return self._wstruct[1]
        keep = []

        def f32(t):
            if t is None:
                return None
            t = t.detach().float().contiguous()
            keep.append(t)
            return t.data_ptr()

        layer_array = (L.LayerWeights * self.num_layers)(*[layer.c_weights(code) for layer in self.layers])
        keep.append(layer_array)
        m = L.ModelWeights()
        m.num_layers, m.embed_dim, m.num_heads = self.num_layers, self.embed_dim, self.num_attention_heads
        m.ffn_dim, m.vocab = 4 * self.embed_dim, len(self.vocab)
        m.n_pos, m.pad_idx = self.embed_positions.weight.shape[0], self.vocab.pad_idx
        m.ln_eps = float(self.emb_layer_norm_before.eps)
        m.tok_emb = f32(self.embed_tokens.weight)
        m.pos_emb = f32(self.embed_positions.weight)
        m.row_pos = f32(self.msa_position_embedding.reshape(-1)) if self.msa_position_embedding is not None else None
        m.ln_before_w, m.ln_before_b = f32(self.emb_layer_norm_before.weight), f32(self.emb_layer_norm_before.bias)
        m.ln_after_w, m.ln_after_b = f32(self.emb_layer_norm_after.weight), f32(self.emb_layer_norm_after.bias)
        m.lm_dense_w, m.lm_dense_b = f32(self.lm_head.dense.weight), f32(self.lm_head.dense.bias)
        m.lm_ln_w, m.lm_ln_b = f32(self.lm_head.layer_norm.weight), f32(self.lm_head.layer_norm.bias)
        m.lm_bias = f32(self.lm_head.bias)
        m.layers = C.cast(layer_array, C.POINTER(L.LayerWeights))
        if code != L.F32:                                              # LM-head dense GEMM on the tensor cores
            w16 = self.lm_head.dense.weight.detach().to(L.torch_dtype(code)).contiguous()
            keep.append(w16)
            m.lm_dense_w16 = w16.data_ptr()
        self._wstruct = (key, m, keep)
        return m

    # -- forward -------------------------------------------------------------------------------
    @torch.no_grad()
    def forward(self, tokens, repr_layers: Iterable[int] = (), need_head_weights: bool = False,
                return_contacts: bool = False, want_logits: bool = True, need_col_weights: bool = False,
                need_col_weights_mean: bool = False) -> Dict[str, object]:
        """model.py:338-416.  ``want_logits=False`` (extension) skips the LM head, which the
        inference script never reads.

        Column-attention probabilities (extensions, off by default; either works with or without
        ``need_head_weights``): ``need_col_weights`` adds ``col_attentions`` ``[B, N, H, C, R, R]`` fp32
        (the key and layout of the reference's ``msm/`` model); ``need_col_weights_mean`` adds
        ``col_attentions_mean`` ``[B, N, H, R, R]``, their mean over the C columns, computed without
        the full tensor (which outgrows the GPU at R x C = 1024 x 1024)."""
        if return_contacts:
            need_head_weights = True
        _infer_only(self)
        assert tokens.ndim == 3                                            # model.py:344
        L.require_cuda(tokens, "tokens")
        if tokens.device != self.device:
            raise RuntimeError(f"tokens on {tokens.device} but model on {self.device}")
        L.device_check(tokens.device)
        B, R, Cc = tokens.shape
        D, H, N = self.embed_dim, self.num_attention_heads, self.num_layers
        tokens = tokens.long().contiguous()
        has_pad, _ = self.check_tokens(tokens)                             # model.py:347, 354-359; modules.py:292
        repr_layers = set(repr_layers)
        code = self._code
        dev = tokens.device
        x = torch.empty((B, R, Cc, D), dtype=torch.float32, device=dev)
        row_att = torch.empty((B, N, H, Cc, Cc), dtype=torch.float32, device=dev) if need_head_weights else None
        logits = torch.empty((B, R, Cc, len(self.vocab)), dtype=torch.float32, device=dev) if want_logits else None
        # allocated before the first launch, so a size that does not fit fails before any kernel runs
        col_att = torch.empty((B, N, H, Cc, R, R), dtype=torch.float32, device=dev) if need_col_weights else None
        col_mean = torch.empty((B, N, H, R, R), dtype=torch.float32, device=dev) if need_col_weights_mean else None
        want_col = need_col_weights or need_col_weights_mean
        reps: Dict[int, torch.Tensor] = {
            l: torch.empty((B, R, Cc, D), dtype=torch.float32, device=dev) for l in sorted(repr_layers) if 0 <= l < N}
        with torch.cuda.device(dev):
            m = self.c_weights(code)
            fcode = self._fwd_code
            nbytes = L.lib.rnamsm_workspace_bytes(R, Cc, D, H, 4 * D, fcode) + ((R * Cc + 255) // 256) * 256
            if want_col:
                nbytes += L.lib.rnamsm_col_probs_scratch_bytes(R, Cc, H)
            ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            st = L.stream_ptr()
            for b in range(B):
                rep_ptrs = (C.c_void_p * (N + 1))(*[reps[l][b].data_ptr() if l in reps else None for l in range(N + 1)])
                if want_col:
                    L.check(L.lib.rnamsm_msa_forward_col_probs(
                        C.byref(m), L.ptr(tokens[b]), R, Cc, int(has_pad), fcode, L.ptr(x[b]),
                        L.ptr(row_att[b]) if row_att is not None else None,
                        L.ptr(col_att[b]) if col_att is not None else None,
                        L.ptr(col_mean[b]) if col_mean is not None else None, rep_ptrs,
                        L.ptr(logits[b]) if logits is not None else None, L.ptr(ws), nbytes, st), "msa_forward_col_probs")
                    continue
                L.check(L.lib.rnamsm_msa_forward(
                    C.byref(m), L.ptr(tokens[b]), R, Cc, int(has_pad), fcode, L.ptr(x[b]),
                    L.ptr(row_att[b]) if row_att is not None else None, rep_ptrs,
                    L.ptr(logits[b]) if logits is not None else None, L.ptr(ws), nbytes, st), "msa_forward")
        if N in repr_layers:
            reps[N] = x                                                    # post-LN, model.py:400-401
        result: Dict[str, object] = {"logits": logits, "representations": reps}
        if need_head_weights:
            result["row_attentions"] = row_att                             # B x N x H x C x C
            if return_contacts:
                result["contacts"] = self.contact_head(tokens, row_att)
        if need_col_weights:
            result["col_attentions"] = col_att                             # B x N x H x C x R x R
        if need_col_weights_mean:
            result["col_attentions_mean"] = col_mean                       # B x N x H x R x R
        return result

    @torch.no_grad()
    def forward_batch(self, tokens_list, need_head_weights: bool = False):
        """Several MSAs of different shapes in ONE pass (``rnamsm_msa_forward_batch``, SURVEY.md 8f row 4).

        ``tokens_list``: ``[1, R_i, C_i]`` (or ``[R_i, C_i]``) int64 grids.  Returns one dict per MSA with
        ``representations[num_layers]`` ``[1, R_i, C_i, D]`` and (optionally) ``row_attentions``
        ``[1, N, H, C_i, C_i]`` -- bit-identical to ``forward`` called on each MSA alone (each MSA keeps its own
        ``1/sqrt(R_i)`` in the tied attention, modules.py:713-715), unlike the reference's padded ``[B, R, C]``
        batch.  The token-local kernels run once over all MSAs' tokens, which is what makes short alignments
        (256 x 51) fill the GPU.  16-bit precisions; the fp32 parity path and single-row inputs go one by one."""
        _infer_only(self)
        grids = []
        for t in tokens_list:
            t = t[0] if t.ndim == 3 and t.shape[0] == 1 else t
            assert t.ndim == 2, "forward_batch takes one MSA per entry ([1,R,C] or [R,C])"
            L.require_cuda(t, "tokens")
            if t.device != self.device:
                raise RuntimeError(f"tokens on {t.device} but model on {self.device}")
            grids.append(t.long().contiguous())
        if not grids:
            return []
        N, D, H = self.num_layers, self.embed_dim, self.num_attention_heads
        code = self._code
        if code == L.dtype_code("fp32") or any(g.shape[0] < 2 for g in grids):
            outs = []
            for g in grids:
                r = self.forward(g.unsqueeze(0), repr_layers=[N], need_head_weights=need_head_weights, want_logits=False)
                outs.append({"representations": {N: r["representations"][N]}, **(
                    {"row_attentions": r["row_attentions"]} if need_head_weights else {})})
            return outs
        dev = self.device
        L.device_check(dev)
        n = len(grids)
        Rs, Cs = [g.shape[0] for g in grids], [g.shape[1] for g in grids]
        flat = torch.cat([g.reshape(-1) for g in grids])
        is_pad = flat.eq(self.vocab.pad_idx)
        sizes = [R * Cc for R, Cc in zip(Rs, Cs)]
        pad_counts = torch.stack([c.sum() for c in is_pad.split(sizes)]).tolist()      # one host sync for the batch
        for g, cnt, R, Cc in zip(grids, pad_counts, Rs, Cs):
            self.check_msa_shape(R, Cc, int((~g.eq(self.vocab.pad_idx)).sum(-1).max()) if cnt else Cc)
        has_pad = bytes(1 if c else 0 for c in pad_counts)
        T = sum(sizes)
        x = torch.empty((T, D), dtype=torch.float32, device=dev)
        maps = [torch.empty((1, N, H, Cc, Cc), dtype=torch.float32, device=dev) for Cc in Cs] if need_head_weights else None
        with torch.cuda.device(dev):
            m = self.c_weights(code)
            Ra, Ca = (C.c_int * n)(*Rs), (C.c_int * n)(*Cs)
            nbytes = L.lib.rnamsm_batch_workspace_bytes(n, Ra, Ca, D, H, 4 * D, code)
            if nbytes == 0:
                raise RuntimeError("rnamsm_batch_workspace_bytes: " + L.lib.rnamsm_last_error().decode(errors="replace"))
            ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            map_ptrs = (C.c_void_p * n)(*[t.data_ptr() for t in maps]) if maps is not None else None
            L.check(L.lib.rnamsm_msa_forward_batch(C.byref(m), n, L.ptr(flat), Ra, Ca, has_pad, code, L.ptr(x), map_ptrs,
                                                   L.ptr(ws), nbytes, L.stream_ptr()), "msa_forward_batch")
        outs = []
        for i, xi in enumerate(x.split(sizes)):
            o = {"representations": {N: xi.view(1, Rs[i], Cs[i], D)}}
            if maps is not None:
                o["row_attentions"] = maps[i]
            outs.append(o)
        return outs

    # -- full-length features from overlapping windows ---------------------------------------------
    @torch.no_grad()
    def forward_windows(self, tokens, window: Optional[int] = None, stride: Optional[int] = None,
                        return_contacts: bool = False, token_budget: int = 262144) -> Dict[str, object]:
        """Features of an alignment of any length, past the learned column positions (``rnamsm_msa_forward_windows``).

        ``tokens``: ``[1, R, C]`` or ``[R, C]`` on the model's device, BOS at column 0, ``L = C - 1`` residues.  The
        residues are covered by ``K`` windows of width ``W = min(window, L)`` starting at ``s_k = min(k * stride, L - W)``;
        window ``k`` is the grid of column 0 and columns ``1 + s_k .. W + s_k`` and runs as an MSA of its own.  Its row 0
        of the final representation and its ``N*H`` maps (BOS stripped) are blended with tent weights ``w_k(p) =
        min(p - s_k + 1, s_k + W - p)``: a residue counts most in the windows where it sits centrally.  A pair of
        residues that no window holds together (further apart than the windows reach) is exactly 0 in the maps and
        contacts: this method does not see such pairs.  ``window`` defaults to ``embed_positions.max_positions - 1``
        (1023) and ``stride`` to ``window // 2``; ``1 <= stride <= window <= max_positions - 1``.  When ``L <= window``
        the outputs are bit-identical to ``extract_features(forward(tokens, ...))``.  The windows run
        ``plan_score_group(R, W + 1, K, token_budget)[0]`` at a time; the result does not depend on that grouping.

        Returns fp32 device tensors ``{"emb": [L, D], "atp": [N*H, L, L], "window_starts": [s_0, ...]}`` plus
        ``"contacts": [L, L]`` with ``return_contacts``.  One host sync.  ``ValueError`` on bad arguments."""
        _infer_only(self)
        if self.vocab.append_eos or not self.vocab.prepend_bos:
            raise ValueError("forward_windows needs a vocabulary that prepends BOS and appends no EOS")
        t = tokens[0] if tokens.ndim == 3 and tokens.shape[0] == 1 else tokens
        if t.ndim != 2:
            raise ValueError(f"forward_windows takes one MSA, [1, R, C] or [R, C]; got shape {tuple(tokens.shape)}")
        L.require_cuda(t, "tokens")
        if t.device != self.device:
            raise RuntimeError(f"tokens on {t.device} but model on {self.device}")
        R, Cc = t.shape
        Ls = Cc - 1
        if Ls < 1:
            raise ValueError(f"the alignment has no residues after the BOS column (C = {Cc})")
        max_window = self.embed_positions.max_positions - 1
        window = max_window if window is None else int(window)
        stride = max(1, window // 2) if stride is None else int(stride)
        if not 1 <= stride <= window <= max_window:
            raise ValueError(f"need 1 <= stride <= window <= {max_window} (the learned positions); "
                             f"got stride {stride}, window {window}")
        if int(token_budget) < 1:
            raise ValueError(f"token_budget {token_budget} must be >= 1")
        K = L.lib.rnamsm_window_starts(Ls, window, stride, None)
        if K == 0:
            raise ValueError("rnamsm_window_starts: " + L.lib.rnamsm_last_error().decode(errors="replace"))
        starts = (C.c_int * K)()
        L.lib.rnamsm_window_starts(Ls, window, stride, starts)
        W = min(window, Ls)
        L.device_check(t.device)
        t = t.long().contiguous()
        has_pad = bool(t.eq(self.vocab.pad_idx).any())                     # the one host sync
        self.check_msa_shape(R, W + 1, W + 1)                              # depth; a window grid fits the positions
        group, _ = plan_score_group(R, W + 1, K, token_budget)
        D, H, N = self.embed_dim, self.num_attention_heads, self.num_layers
        dev = t.device
        # allocated before the first launch, so a size that does not fit fails before any kernel runs
        emb = torch.empty((Ls, D), dtype=torch.float32, device=dev)
        atp = torch.empty((N * H, Ls, Ls), dtype=torch.float32, device=dev)
        contacts = torch.empty((Ls, Ls), dtype=torch.float32, device=dev) if return_contacts else None
        cw = cb = None
        if return_contacts:
            reg = self.contact_head.regression
            cw = reg.weight.detach().float().reshape(-1).contiguous()
            cb = reg.bias.detach().float().contiguous() if reg.bias is not None else None
        with torch.cuda.device(dev):
            m = self.c_weights(self._code)
            fcode = self._fwd_code
            nbytes = L.lib.rnamsm_windows_workspace_bytes(R, Cc, D, H, 4 * D, N, fcode, group, window, stride,
                                                          int(return_contacts))
            if nbytes == 0:
                raise RuntimeError("rnamsm_windows_workspace_bytes: " + L.lib.rnamsm_last_error().decode(errors="replace"))
            ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            L.check(L.lib.rnamsm_msa_forward_windows(
                C.byref(m), L.ptr(t), R, Cc, int(has_pad), fcode, window, stride, group, L.ptr(emb), L.ptr(atp),
                L.ptr(contacts), L.ptr(cw), L.ptr(cb), L.ptr(ws), nbytes, L.stream_ptr()), "msa_forward_windows")
        out: Dict[str, object] = {"emb": emb, "atp": atp, "window_starts": list(starts)}
        if return_contacts:
            out["contacts"] = contacts
        return out

    # -- LM-head scoring ---------------------------------------------------------------------------
    def _score_grid(self, tokens, row: int):
        """[1, R, C] or [R, C] CUDA tokens -> (int64 [R, C] grid, has_pad, host pad flags of ``row``, host tokens of
        ``row``) after the input limits of ``forward``.  One host sync."""
        _infer_only(self)
        t = tokens[0] if tokens.ndim == 3 and tokens.shape[0] == 1 else tokens
        if t.ndim != 2:
            raise ValueError(f"scoring takes one MSA, [1, R, C] or [R, C]; got shape {tuple(tokens.shape)}")
        L.require_cuda(t, "tokens")
        if t.device != self.device:
            raise RuntimeError(f"tokens on {t.device} but model on {self.device}")
        L.device_check(t.device)
        t = t.long().contiguous()
        R, Cc = t.shape
        if not 0 <= row < R:
            raise ValueError(f"row {row} outside the {R} MSA rows")
        pad = t.eq(self.vocab.pad_idx)
        host = torch.cat([(~pad).sum(-1), pad[row].long(), t[row]]).cpu()   # non-pad count per row | pad flags | tokens of `row`
        n_nonpad_max = int(host[:R].max())
        self.check_msa_shape(R, Cc, n_nonpad_max)
        return t, bool(int(host[:R].min()) < Cc), host[R:R + Cc].bool().tolist(), host[R + Cc:].tolist()

    def _marginals(self, t, has_pad, row_pad, positions, row, masked, token_budget, return_logits):
        R, Cc = t.shape
        start = int(self.vocab.prepend_bos)
        if positions is None:
            positions = [c for c in range(start, Cc) if not row_pad[c]]
        positions = [int(c) for c in positions]
        for c in positions:
            if not 0 <= c < Cc:
                raise ValueError(f"position {c} outside the {Cc} grid columns")
            if row_pad[c]:
                raise ValueError(f"position {c} is a padding token of row {row}")
        P, V = len(positions), len(self.vocab)
        dev = t.device
        lp = torch.empty((P, V), dtype=torch.float32, device=dev)
        logits = torch.empty((P, V), dtype=torch.float32, device=dev) if return_logits else None
        if P:
            group, _ = plan_score_group(R, Cc, P, token_budget)
            D, H = self.embed_dim, self.num_attention_heads
            cols = torch.tensor(positions, dtype=torch.int32).to(dev)
            with torch.cuda.device(dev):
                m = self.c_weights(self._code)
                fcode = self._fwd_code
                nbytes = L.lib.rnamsm_score_workspace_bytes(R, Cc, D, H, 4 * D, fcode, group)
                if nbytes == 0:
                    raise RuntimeError("rnamsm_score_workspace_bytes: " + L.lib.rnamsm_last_error().decode(errors="replace"))
                ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
                L.check(L.lib.rnamsm_msa_masked_marginals(
                    C.byref(m), L.ptr(t), R, Cc, int(has_pad), fcode, row, L.ptr(cols), P,
                    self.vocab.mask_idx if masked else -1, group, L.ptr(logits), L.ptr(lp), L.ptr(ws), nbytes,
                    L.stream_ptr()), "msa_masked_marginals")
        return positions, lp, logits

    @torch.no_grad()
    def masked_marginals(self, tokens, positions: Optional[Iterable[int]] = None, row: int = 0, masked: bool = True,
                         token_budget: int = 262144, return_logits: bool = False):
        """LM-head log-probabilities of ``row`` under masking (``rnamsm_msa_masked_marginals``).

        Row ``k`` of the result is ``log_softmax`` of the logits at ``(row, positions[k])`` of the grid with that token
        replaced by ``<mask>``; ``masked=False`` reads every position from one forward of ``tokens`` itself
        ("wt-marginals").  ``tokens``: ``[1, R, C]`` or ``[R, C]`` on the model's device.  ``positions``: grid columns;
        by default every non-pad column of ``row`` except the BOS column 0.  The masked grids run ``group =
        max(1, token_budget // (R * C))`` at a time (``plan_score_group``).  Returns fp32 ``[P, V]`` on the device, and
        the logits ``[P, V]`` too with ``return_logits=True``; the logits are bit-identical to
        ``forward(masked grid)["logits"][0, row, col]``.  One host sync per call."""
        t, has_pad, row_pad, _ = self._score_grid(tokens, row)
        _, lp, logits = self._marginals(t, has_pad, row_pad, positions, row, masked, token_budget, return_logits)
        return (lp, logits) if return_logits else lp

    @torch.no_grad()
    def pseudo_log_likelihood(self, tokens, row: int = 0, token_budget: int = 262144):
        """-> ``(pll, per_position)``: ``per_position[i] = log p(wt_i | wt_i masked)`` (fp32, device) over the default
        positions of ``masked_marginals`` (the non-pad residues of ``row``), ``pll`` their float64 sum.  The
        pseudo-perplexity is ``exp(-pll / L)`` with ``L = len(per_position)``."""
        t, has_pad, row_pad, _ = self._score_grid(tokens, row)
        positions, lp, _ = self._marginals(t, has_pad, row_pad, None, row, True, token_budget, False)
        wt = t[row, positions].view(-1, 1)
        per_position = lp.gather(1, wt).view(-1)
        return float(per_position.double().sum()), per_position

    @torch.no_grad()
    def score_mutations(self, tokens, mutations, row: int = 0, method: str = "masked-marginals",
                        token_budget: int = 262144) -> torch.Tensor:
        """Zero-shot mutant scores: float64 ``[len(mutations)]`` on the CPU, mutant ``i`` scoring
        ``sum over its substitutions of logp[pos, mt] - logp[pos, wt]``.  Mutants are strings such as ``"G12A"`` or
        ``"G12A:C30U"`` (``rnamsm_b200.mutations``): 1-based residues of query ``row``, so residue ``k`` is grid column
        ``k``.  ``method``: ``"masked-marginals"`` (logp at a position from the grid with that position masked) or
        ``"wt-marginals"`` (all from one unmasked forward).  Marginals are computed once for the union of mutated
        positions: one forward per distinct position, not per mutant.  ``ValueError`` on a malformed mutant, a wild
        type that does not match the query, an index out of range or on a pad / BOS column, or a repeated position."""
        from .mutations import parse_mutant
        if method not in ("masked-marginals", "wt-marginals"):
            raise ValueError(f"method {method!r}: expected 'masked-marginals' or 'wt-marginals'")
        t, has_pad, row_pad, query = self._score_grid(tokens, row)
        parsed = [parse_mutant(s, query, self.vocab) for s in mutations]
        positions = sorted({c for subs in parsed for c, _, _ in subs})
        _, lp, _ = self._marginals(t, has_pad, row_pad, positions, row, method == "masked-marginals", token_budget, False)
        lp = lp.cpu().double()
        at = {c: i for i, c in enumerate(positions)}
        scores = torch.zeros(len(parsed), dtype=torch.float64)
        for i, subs in enumerate(parsed):
            scores[i] = sum(float(lp[at[c], mt] - lp[at[c], wt]) for c, wt, mt in subs)
        return scores

    # -- categorical Jacobian of the LM head ------------------------------------------------------------
    @torch.no_grad()
    def categorical_jacobian(self, tokens, row: int = 0, positions: Optional[Iterable[int]] = None,
                             alphabet: str = "AGCU", token_budget: int = 262144, return_jacobian: bool = False):
        """Contacts of query ``row`` read from the LM head alone (Zhang et al., PNAS 2024), with no contact regression
        (``rnamsm_msa_categorical_jacobian``, ``rnamsm_jacobian_contacts``).

        ``J[i, a, j, b] = f(G(i, a))[j, b] - f(tokens)[j, b]``, fp32 ``[P, A, P, A]``: ``G(i, a)`` is ``tokens`` with
        ``(row, positions[i])`` replaced by ``alphabet[a]``, ``f(G)[j, b]`` the LM-head logit of ``G`` at
        ``(row, positions[j])`` for ``alphabet[b]``.  A substitution by the wild type is not run and its slab is exactly
        0, so a call runs ``sum_i (A - [wt_i in alphabet]) + 1`` forwards: ``3P + 1`` for ``"AGCU"`` over a gap-free
        query, in passes of ``plan_score_group(R, C, n_substitutions, token_budget)[0]`` grids.  The cost grows as
        ``P`` forwards of the whole ``R x C`` alignment: about ``3C`` forwards, so ~106 at 512 x 36 and ~766 at
        512 x 256.  Each slab is bit-identical to the difference of ``forward(G(i, a))["logits"]`` and
        ``forward(tokens)["logits"]`` at those entries.

        Contacts ``[P, P]`` fp32: ``J`` centred over each of its axes in turn (i, a, j, b), the Frobenius norm of each
        ``A x A`` block with a zero diagonal, average product correction, then ``(F + F^T) / 2``.

        ``tokens``: ``[1, R, C]`` or ``[R, C]`` on the model's device.  ``positions``: grid columns of ``row``; by
        default every non-pad column except the BOS column 0.  ``alphabet``: distinct letters of ``A G C U X N -``.
        Returns the contacts on the device, and ``(contacts, J)`` with ``return_jacobian=True``.  One host sync.
        ``ValueError`` on a bad alphabet, a row or position out of range, a position on a pad token or on the BOS
        column, or fewer than two positions."""
        alph = self._alphabet_indices(alphabet)
        t, has_pad, row_pad, query = self._score_grid(tokens, row)
        R, Cc = t.shape
        start = int(self.vocab.prepend_bos)
        if positions is None:
            positions = [c for c in range(start, Cc) if not row_pad[c]]
        positions = [int(c) for c in positions]
        for c in positions:
            if not 0 <= c < Cc:
                raise ValueError(f"position {c} outside the {Cc} grid columns")
            if c < start:
                raise ValueError(f"position {c} is the BOS column")
            if row_pad[c]:
                raise ValueError(f"position {c} is a padding token of row {row}")
        P, A = len(positions), len(alph)
        if P < 2:
            raise ValueError(f"a Jacobian needs at least two positions, got {P}")
        entries = jacobian_entries([query[c] for c in positions], alph)
        n = len(entries)
        dev = t.device
        J = torch.empty((P, A, P, A), dtype=torch.float32, device=dev)
        contacts = torch.empty((P, P), dtype=torch.float32, device=dev)
        group, _ = plan_score_group(R, Cc, max(n, 1), token_budget)
        D, H = self.embed_dim, self.num_attention_heads
        IntP = lambda v: (C.c_int * len(v))(*v)
        with torch.cuda.device(dev):
            m = self.c_weights(self._code)
            fcode = self._fwd_code
            nbytes = L.lib.rnamsm_jacobian_workspace_bytes(R, Cc, D, H, 4 * D, fcode, group, P, A, n)
            if nbytes == 0:
                raise RuntimeError("rnamsm_jacobian_workspace_bytes: " + L.lib.rnamsm_last_error().decode(errors="replace"))
            ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            st = L.stream_ptr()
            L.check(L.lib.rnamsm_msa_categorical_jacobian(
                C.byref(m), L.ptr(t), R, Cc, int(has_pad), fcode, row, IntP(positions), P, IntP(alph), A,
                IntP(entries), n, group, L.ptr(J), L.ptr(ws), nbytes, st), "msa_categorical_jacobian")
            del ws
            sbytes = L.lib.rnamsm_jacobian_contacts_scratch_bytes(P, A)
            scratch = torch.empty(sbytes, dtype=torch.uint8, device=dev)
            L.check(L.lib.rnamsm_jacobian_contacts(L.ptr(J), P, A, L.ptr(contacts), L.ptr(scratch), sbytes, st),
                    "jacobian_contacts")
        return (contacts, J) if return_jacobian else contacts

    def _alphabet_indices(self, alphabet) -> List[int]:
        """``alphabet`` (a string of distinct letters of ``A G C U X N -``) -> their vocabulary indices, in order."""
        from .alphabet import RNA_TOKS
        letters = list(alphabet)
        if not letters:
            raise ValueError("alphabet is empty")
        for a in letters:
            if a not in RNA_TOKS:
                raise ValueError(f"alphabet letter {a!r} is not a residue or gap ({' '.join(RNA_TOKS)})")
        if len(set(letters)) != len(letters):
            raise ValueError(f"alphabet {alphabet!r} repeats a letter")
        return [self.vocab.tokens_to_idx[a] for a in letters]

    # -- generation with the LM head ---------------------------------------------------------------
    @torch.no_grad()
    def sample_msa(self, tokens, steps: int, mask_prob: float = 0.1, temperature: float = 1.0,
                   rows: Optional[Iterable[int]] = None, n_chains: int = 1, seed: int = 0, start_step: int = 0,
                   allowed: str = "AGCU-", token_budget: int = 262144) -> torch.Tensor:
        """New sequences from one alignment by iterative masked sampling (``rnamsm_msa_gibbs_sample``).

        Each of ``n_chains`` chains starts from ``tokens`` and takes steps ``start_step .. start_step + steps - 1``.  A
        step masks every non-pad token of ``rows`` (default: all rows) outside the BOS column with probability
        ``mask_prob``, runs the model on the masked grid and replaces each masked token by a draw from
        ``softmax(logits / temperature)`` over the ``allowed`` tokens (``temperature=0``: the argmax).  The random
        numbers are a stateless function of ``(seed, chain, step, row, column)`` (DESIGN.md §4.11), so the result does
        not depend on ``token_budget`` and ``steps=a+b`` equals ``steps=a`` followed by ``steps=b, start_step=a`` on its
        output.  ``tokens``: ``[R, C]`` or ``[1, R, C]`` (every chain starts there) or ``[n_chains, R, C]`` (chain ``k``
        starts from ``tokens[k]``; the grids share one pad layout) on the model's device.  Chains run
        ``plan_score_group(R, C, n_chains, token_budget)[0]`` at a time.  Returns int64 ``[n_chains, R, C]`` on the
        device; the steps are enqueued without a host sync."""
        if not 0.0 <= mask_prob <= 1.0:
            raise ValueError(f"mask_prob {mask_prob} outside [0, 1]")
        if not temperature >= 0.0:
            raise ValueError(f"temperature {temperature} must be >= 0")
        if steps < 0 or start_step < 0:
            raise ValueError(f"steps {steps} and start_step {start_step} must be >= 0")
        if n_chains < 1:
            raise ValueError(f"n_chains {n_chains} must be >= 1")
        if not 0 <= seed < 1 << 64:
            raise ValueError(f"seed {seed} outside [0, 2**64)")
        bitmask = self._allowed_bitmask(allowed)
        R = tokens.shape[-2]
        rows = list(range(R)) if rows is None else sorted({int(r) for r in rows})
        if not rows:
            raise ValueError("rows is empty")
        if rows[0] < 0 or rows[-1] >= R:
            raise ValueError(f"rows {rows[0]} .. {rows[-1]} outside the {R} MSA rows")
        t, has_pad = self._sample_grid(tokens, n_chains)
        Cc = t.shape[2]
        dev = t.device
        out = torch.empty((n_chains, R, Cc), dtype=torch.int64, device=dev)
        if t.shape[0] > 1:
            out.copy_(t)
        group, _ = plan_score_group(R, Cc, n_chains, token_budget)
        D, H = self.embed_dim, self.num_attention_heads
        rows_d = torch.tensor(rows, dtype=torch.int32).to(dev)
        with torch.cuda.device(dev):
            m = self.c_weights(self._code)
            fcode = self._fwd_code
            nbytes = L.lib.rnamsm_sample_workspace_bytes(R, Cc, D, H, 4 * D, fcode, group, len(rows))
            if nbytes == 0:
                raise RuntimeError("rnamsm_sample_workspace_bytes: " + L.lib.rnamsm_last_error().decode(errors="replace"))
            ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            L.check(L.lib.rnamsm_msa_gibbs_sample(
                C.byref(m), L.ptr(t[0]) if t.shape[0] == 1 else None, R, Cc, int(has_pad), fcode, L.ptr(rows_d),
                len(rows), n_chains, steps, start_step, mask_prob, temperature, bitmask, seed, group, L.ptr(out),
                L.ptr(ws), nbytes, L.stream_ptr()), "msa_gibbs_sample")
        return out

    def _allowed_bitmask(self, allowed) -> int:
        """``allowed`` (a string of residue / gap letters such as ``"AGCU-"``, or an iterable of them) -> the bit set
        of their vocabulary indices.  ``ValueError`` when empty or when an entry is not one of ``A G C U X N -``."""
        from .alphabet import RNA_TOKS
        letters = list(allowed)
        if not letters:
            raise ValueError("allowed is empty")
        bits = 0
        for a in letters:
            if a not in RNA_TOKS:
                raise ValueError(f"allowed token {a!r} is not a residue or gap ({' '.join(RNA_TOKS)})")
            bits |= 1 << self.vocab.tokens_to_idx[a]
        return bits

    def _sample_grid(self, tokens, n_chains: int):
        """[R, C], [1, R, C] or [n_chains, R, C] CUDA tokens -> (int64 [1 or n_chains, R, C], has_pad) after the input
        limits of ``forward``.  One host sync."""
        _infer_only(self)
        t = tokens.unsqueeze(0) if tokens.ndim == 2 else tokens
        if t.ndim != 3 or t.shape[0] not in (1, n_chains):
            raise ValueError(f"sampling takes one MSA, [R, C], [1, R, C] or [n_chains={n_chains}, R, C]; "
                             f"got shape {tuple(tokens.shape)}")
        L.require_cuda(t, "tokens")
        if t.device != self.device:
            raise RuntimeError(f"tokens on {t.device} but model on {self.device}")
        L.device_check(t.device)
        t = t.long().contiguous()
        R, Cc = t.shape[1:]
        pad = t.eq(self.vocab.pad_idx)
        host = torch.cat([(~pad[0]).sum(-1), (pad != pad[:1]).any().view(1).long()]).cpu()   # non-pad counts | layouts differ
        if int(host[R]):
            raise ValueError("the chains' starting grids must share one pad layout")
        self.check_msa_shape(R, Cc, int(host[:R].max()))
        return t, bool(int(host[:R].min()) < Cc)


def plan_score_group(R: int, C: int, n_positions: int, token_budget: int = 262144):
    """-> ``(group, passes)`` of ``masked_marginals`` (and of ``sample_msa``, with its chains as the positions):
    ``group = max(1, token_budget // (R * C))`` grids per pass (the token budget of ``plan_batches``), at most
    ``n_positions``, and ``passes = ceil(n_positions / group)``; the last pass may be partial."""
    group = max(1, min(int(token_budget) // (R * C), n_positions))
    return group, -(-n_positions // group)


def jacobian_entries(wild_type: Sequence[int], alphabet: Sequence[int]) -> List[int]:
    """The substitutions ``categorical_jacobian`` runs, as slabs ``i * A + a`` of ``J`` in ascending order: every
    ``(i, a)`` with ``alphabet[a] != wild_type[i]`` (token indices).  A wild type outside the alphabet (``N``, ``X``,
    ``-``) gets all ``A`` substitutions."""
    A = len(alphabet)
    return [i * A + a for i, w in enumerate(wild_type) for a, v in enumerate(alphabet) if v != w]
