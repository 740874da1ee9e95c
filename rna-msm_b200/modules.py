"""Host-side mirror of the reference's building blocks (top-level ``modules.py`` ==
``msm/modules.py`` + ``msm/axial_attention.py``), same class names, constructor arguments,
parameter names and ``forward`` signatures, with every forward body dispatching to the
hand-written sm_100a kernels in ``librnamsm_b200.so`` through the C ABI.

Inference only (eval mode, no autograd), CUDA only, no fallback.  Tensors follow the reference:
``x`` is ``[R, C, B, D]`` (rows, columns, batch, features), padding masks are bool ``[B, R, C]``.
B > 1 is handled by looping over the batch entries (the kernels process one MSA at a time; the
tied-attention scale uses that call's row count exactly like modules.py:713-715).
"""
from __future__ import annotations

import ctypes as C
import math
import os
from typing import Optional

import torch
import torch.nn as nn

from . import _lib as L

_DEFAULT_PRECISION = os.environ.get("RNAMSM_PRECISION", "fp16")


def _infer_only(module: nn.Module) -> None:
    if module.training:
        raise RuntimeError(
            f"{type(module).__name__}: rnamsm_b200 implements the inference forward only "
            "(dropout is the identity); call .eval() first, as RNA_MSM_Inference.py:136 does")


def _pad_u8(self_attn_padding_mask: Optional[torch.Tensor], b: int) -> Optional[torch.Tensor]:
    """bool [B,R,C] -> contiguous uint8 [R*C] of batch entry b (or None)."""
    if self_attn_padding_mask is None:
        return None
    return self_attn_padding_mask[b].to(torch.uint8).contiguous()


class _PrecisionMixin:
    """``precision``: 'fp16' (default: fp16 operands on the tcgen05 tensor cores, fp32 accumulate /
    residual stream / LayerNorm / softmax), 'bf16' (bf16 operands except the tied row-attention
    block, which stays fp16), 'bf16_pure' (bf16 everywhere), 'fp32' (FFMA parity path, <= 1e-4) or 'tf32x3' (fp32
    storage and attention, the nn.Linear layers as three-term tf32 products on the tensor cores: 3x faster than 'fp32',
    ~1e-4-grade rather than 1e-5-grade because the tensor core truncates when it accumulates)."""

    precision: str = _DEFAULT_PRECISION

    def set_precision(self, precision: str):
        L.dtype_code(precision)
        for m in self.modules():
            if isinstance(m, _PrecisionMixin):
                m.precision = precision
        return self

    @property
    def _code(self) -> int:
        return L.dtype_code(self.precision)

    @property
    def _row_code(self) -> int:
        return L.row_dtype_code(self.precision)

    @property
    def _fwd_code(self) -> int:
        """dtype for the whole-layer / whole-model C entry points (carries the tf32x3 flag)."""
        return L.forward_code(self.precision)


def _linear(x2d: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, code: int, epilogue: int = L.EPI_BIAS,
            q_scale: float = 1.0, q_cols: int = 0, row_mask: Optional[torch.Tensor] = None,
            out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """rnamsm_linear on 2-D operands already in the compute dtype (weight [N,K], x [M,K])."""
    M, K = x2d.shape
    N = weight.shape[0]
    if out is None:
        out = torch.empty((M, N), dtype=x2d.dtype, device=x2d.device)
    L.check(L.lib.rnamsm_linear(L.ptr(x2d), L.ptr(weight), L.ptr(bias), M, N, K, code, epilogue, float(q_scale),
                                int(q_cols), L.ptr(row_mask), L.ptr(out), L.stream_ptr()), "linear")
    return out


class _AxialAttentionBase(nn.Module, _PrecisionMixin):
    def __init__(self, embed_dim, num_heads, dropout=0.0, max_tokens_per_msa: int = 2 ** 16):
        super().__init__()
        self.num_heads = num_heads
        self.dropout = dropout
        self.head_dim = embed_dim // num_heads
        if self.head_dim != 64 or self.head_dim * num_heads != embed_dim:
            raise ValueError("rnamsm_b200 kernels are specialised for head_dim == 64 (RNA-MSM: 768 / 12)")
        self.scaling = self.head_dim ** -0.5
        # kept for API parity (model.py:418-428); the kernels never materialise what it bounded
        self.max_tokens_per_msa = max_tokens_per_msa
        self.k_proj = nn.Linear(embed_dim, embed_dim)
        self.v_proj = nn.Linear(embed_dim, embed_dim)
        self.q_proj = nn.Linear(embed_dim, embed_dim)
        self.out_proj = nn.Linear(embed_dim, embed_dim)
        self.dropout_module = nn.Dropout(dropout)
        self._packed = None

    def _pack(self, code: int):
        """q|k|v rows concatenated, in the compute dtype; cached until a parameter changes."""
        key = (code,) + tuple((p.data_ptr(), p._version) for p in self.parameters())
        if self._packed is None or self._packed[0] != key:
            dt = L.torch_dtype(code)
            w_qkv = torch.cat([self.q_proj.weight, self.k_proj.weight, self.v_proj.weight], 0).detach().to(dt).contiguous()
            b_qkv = torch.cat([self.q_proj.bias, self.k_proj.bias, self.v_proj.bias], 0).detach().float().contiguous()
            w_out = self.out_proj.weight.detach().to(dt).contiguous()
            b_out = self.out_proj.bias.detach().float().contiguous()
            self._packed = (key, w_qkv, b_qkv, w_out, b_out)
        return self._packed[1:]

    def _check_input(self, x, self_attn_mask):
        _infer_only(self)
        if self_attn_mask is not None:
            raise NotImplementedError  # modules.py:776-777, 909-910
        L.require_cuda(x, "x")
        L.device_check(x.device)
        if x.dim() != 4:
            raise ValueError(f"expected x of shape [R, C, B, D], got {tuple(x.shape)}")


class RowSelfAttention(_AxialAttentionBase):
    """Tied row attention (modules.py:688-821): K3 -> K4 -> K5 -> K6."""

    def __init__(self, embed_dim, num_heads, dropout=0.0, max_tokens_per_msa: int = 2 ** 16):
        super().__init__(embed_dim, num_heads, dropout, max_tokens_per_msa)
        self.attn_shape = "hnij"

    def align_scaling(self, q):
        num_rows = q.size(0)
        return self.scaling / math.sqrt(num_rows)

    @torch.no_grad()
    def forward(self, x, self_attn_mask=None, self_attn_padding_mask=None):
        self._check_input(x, self_attn_mask)
        R, Cc, B, D = x.shape
        H = self.num_heads
        code = self._row_code
        dt = L.torch_dtype(code)
        w_qkv, b_qkv, w_out, b_out = self._pack(code)
        out = torch.empty((R, Cc, B, D), dtype=torch.float32, device=x.device)
        probs = torch.empty((H, B, Cc, Cc), dtype=torch.float32, device=x.device)
        scaling = self.align_scaling(x)
        # 16-bit path: q carries 64^-1/2 (exact), the 1/sqrt(R) goes on the fp32 logit sums (K5)
        q_scale, logit_scale = (self.scaling, scaling / self.scaling) if code != L.F32 else (scaling, 1.0)
        with torch.cuda.device(x.device):
            st = L.stream_ptr()
            for b in range(B):
                xb = x[:, :, b, :].to(dt).contiguous().view(R * Cc, D)
                pad = _pad_u8(self_attn_padding_mask, b)
                qkv = _linear(xb, w_qkv, b_qkv, code, L.EPI_BIAS, q_scale, D, pad)
                pmap = torch.empty((H, Cc, Cc), dtype=torch.float32, device=x.device)
                ctx = torch.empty((R * Cc, D), dtype=dt, device=x.device)
                if code != L.F32:
                    ldp = (Cc + 7) // 8 * 8
                    plp = torch.empty((H, Cc, ldp), dtype=dt, device=x.device)
                else:
                    ldp, plp = Cc, None
                chunks = L.lib.rnamsm_row_attn_short_chunks(R, Cc, H) if code != L.F32 else 0
                if chunks > 0:
                    # short alignment (C <= 128): K4 + K5 + K6 in one cooperative launch, as the fused layer does
                    partial = torch.empty((chunks, H, Cc, Cc), dtype=torch.float32, device=x.device)
                    L.check(L.lib.rnamsm_row_attn_short(L.ptr(qkv), R, Cc, H, code, L.ptr(pad), float(logit_scale),
                                                        L.ptr(partial), chunks, L.ptr(pmap), L.ptr(plp), ldp, L.ptr(ctx), st),
                            "row_attn_short")
                else:
                    splits = L.lib.rnamsm_row_attn_splits(R, Cc, H, code)
                    partial = torch.empty((splits, H, Cc, Cc), dtype=torch.float32, device=x.device)
                    L.check(L.lib.rnamsm_row_attn_logits(L.ptr(qkv), R, Cc, H, code, L.ptr(partial), splits, st), "row_attn_logits")
                    L.check(L.lib.rnamsm_row_softmax(L.ptr(partial), splits, H, Cc, L.ptr(pad), float(logit_scale),
                                                     L.ptr(pmap), L.ptr(plp), ldp, code, st), "row_softmax")
                    L.check(L.lib.rnamsm_row_attn_av(L.ptr(plp if plp is not None else pmap), ldp, L.ptr(qkv), R, Cc, H,
                                                     code, L.ptr(ctx), st), "row_attn_av")
                ob = _linear(ctx, w_out, b_out, code)
                out[:, :, b, :] = ob.view(R, Cc, D).float()
                probs[:, b] = pmap
        return out, probs


class ColumnSelfAttention(_AxialAttentionBase):
    """Column attention over the MSA depth (modules.py:824-945): K3 -> K7 (flash) -> out_proj.

    The flash kernel never materialises the probabilities, so by default the second return value is
    ``None`` (except R == 1, where the reference's all-ones tensor is cheap).  ``need_weights=True``
    returns the reference's ``[H, C, B, R, R]`` fp32 probabilities, computed by a separate pair of
    kernels from the same q|k (``rnamsm_col_attn_probs``); ``out`` is the same either way.
    """

    @torch.no_grad()
    def forward(self, x, self_attn_mask=None, self_attn_padding_mask=None, need_weights: bool = False):
        self._check_input(x, self_attn_mask)
        R, Cc, B, D = x.shape
        H = self.num_heads
        code = self._code
        dt = L.torch_dtype(code)
        w_qkv, b_qkv, w_out, b_out = self._pack(code)
        out = torch.empty((R, Cc, B, D), dtype=torch.float32, device=x.device)
        want = need_weights and R > 1
        if want:
            attn = torch.empty((H, Cc, B, R, R), dtype=torch.float32, device=x.device)
            probs = attn[:, :, 0] if B == 1 else torch.empty((H, Cc, R, R), dtype=torch.float32, device=x.device)
            scratch = torch.empty(L.lib.rnamsm_col_probs_scratch_bytes(R, Cc, H), dtype=torch.uint8, device=x.device)
        with torch.cuda.device(x.device):
            st = L.stream_ptr()
            for b in range(B):
                xb = x[:, :, b, :].to(dt).contiguous().view(R * Cc, D)
                if R == 1:  # modules.py:882-894
                    v = _linear(xb, w_qkv[2 * D:], b_qkv[2 * D:], code)
                    ob = _linear(v, w_out, b_out, code)
                else:
                    pad = _pad_u8(self_attn_padding_mask, b)
                    qkv = _linear(xb, w_qkv, b_qkv, code, L.EPI_BIAS, self.scaling, D, None)
                    ctx = torch.empty((R * Cc, D), dtype=dt, device=x.device)
                    L.check(L.lib.rnamsm_col_attn(L.ptr(qkv), R, Cc, H, code, 0, L.ptr(pad), L.ptr(ctx), st), "col_attn")
                    if want:
                        L.check(L.lib.rnamsm_col_attn_probs(L.ptr(qkv), R, Cc, H, code, 0, L.ptr(pad), L.ptr(probs), None,
                                                            L.ptr(scratch), st), "col_attn_probs")
                        if B > 1:
                            attn[:, :, b] = probs
                    ob = _linear(ctx, w_out, b_out, code)
                out[:, :, b, :] = ob.view(R, Cc, D).float()
        if not want:
            attn = torch.ones(H, Cc, B, 1, 1, device=x.device, dtype=x.dtype) if R == 1 else None
        return out, attn


class FeedForwardNetwork(nn.Module, _PrecisionMixin):
    """fc2(gelu_erf(fc1(x))) (modules.py:404-427): two GEMMs, GELU fused in the first epilogue."""

    def __init__(self, embedding_dim: int, ffn_embedding_dim: int, activation_dropout: float = 0.1,
                 max_tokens_per_msa: int = 2 ** 14):
        super().__init__()
        self.embedding_dim = embedding_dim
        self.ffn_embedding_dim = ffn_embedding_dim
        self.max_tokens_per_msa = max_tokens_per_msa
        self.activation_fn = nn.GELU()
        self.activation_dropout_module = nn.Dropout(activation_dropout)
        self.fc1 = nn.Linear(embedding_dim, ffn_embedding_dim)
        self.fc2 = nn.Linear(ffn_embedding_dim, embedding_dim)
        self._packed = None

    def _pack(self, code: int):
        key = (code,) + tuple((p.data_ptr(), p._version) for p in self.parameters())
        if self._packed is None or self._packed[0] != key:
            dt = L.torch_dtype(code)
            self._packed = (key, self.fc1.weight.detach().to(dt).contiguous(), self.fc1.bias.detach().float().contiguous(),
                            self.fc2.weight.detach().to(dt).contiguous(), self.fc2.bias.detach().float().contiguous())
        return self._packed[1:]

    @torch.no_grad()
    def forward(self, x):
        _infer_only(self)
        L.require_cuda(x, "x")
        L.device_check(x.device)
        code = self._code
        dt = L.torch_dtype(code)
        w1, b1, w2, b2 = self._pack(code)
        shape = x.shape
        with torch.cuda.device(x.device):
            x2 = x.reshape(-1, shape[-1]).to(dt).contiguous()
            h = _linear(x2, w1, b1, code, L.EPI_BIAS_GELU)
            y = _linear(h, w2, b2, code)
        return y.float().view(shape)


class NormalizedResidualBlock(nn.Module, _PrecisionMixin):
    """x + layer(LayerNorm(x)) (modules.py:369-401); LayerNorm runs on the K2 kernel."""

    def __init__(self, layer: nn.Module, embedding_dim: int, dropout: float = 0.1):
        super().__init__()
        self.embedding_dim = embedding_dim
        self.layer = layer
        self.dropout_module = nn.Dropout(dropout)
        self.layer_norm = nn.LayerNorm(self.embedding_dim)

    @torch.no_grad()
    def forward(self, x, *args, **kwargs):
        _infer_only(self)
        L.require_cuda(x, "x")
        residual = x
        xc = x.float().contiguous()
        xn = torch.empty_like(xc)
        with torch.cuda.device(x.device):
            L.check(L.lib.rnamsm_layernorm(L.ptr(xc), L.ptr(self.layer_norm.weight), L.ptr(self.layer_norm.bias),
                                           L.ptr(xn), L.F32, xc.numel() // xc.shape[-1], xc.shape[-1],
                                           float(self.layer_norm.eps), 0, 0, L.stream_ptr()), "layernorm")
        outputs = self.layer(xn, *args, **kwargs)
        if isinstance(outputs, tuple):
            y, *out = outputs
        else:
            y, out = outputs, None
        y = residual + y
        if out is not None:
            return (y,) + tuple(out)
        return y


class AxialTransformerLayer(nn.Module, _PrecisionMixin):
    """One axial block (modules.py:191-267).  ``forward`` runs the whole layer through
    ``rnamsm_layer_forward`` (13 kernels, one C call); the sub-modules keep the reference's
    parameter names and remain individually callable."""

    def __init__(self, embedding_dim: int = 768, ffn_embedding_dim: int = 3072, num_attention_heads: int = 8,
                 dropout: float = 0.1, attention_dropout: float = 0.1, activation_dropout: float = 0.1,
                 max_tokens_per_msa: int = 2 ** 14) -> None:
        super().__init__()
        self.embedding_dim = embedding_dim
        self.ffn_embedding_dim = ffn_embedding_dim
        self.num_attention_heads = num_attention_heads
        self.dropout_prob = dropout
        row_self_attention = RowSelfAttention(embedding_dim, num_attention_heads, dropout=dropout,
                                              max_tokens_per_msa=max_tokens_per_msa)
        column_self_attention = ColumnSelfAttention(embedding_dim, num_attention_heads, dropout=dropout,
                                                    max_tokens_per_msa=max_tokens_per_msa)
        feed_forward_layer = FeedForwardNetwork(embedding_dim, ffn_embedding_dim,
                                                activation_dropout=activation_dropout,
                                                max_tokens_per_msa=max_tokens_per_msa)
        self.row_self_attention = self.build_residual(row_self_attention)
        self.column_self_attention = self.build_residual(column_self_attention)
        self.feed_forward_layer = self.build_residual(feed_forward_layer)
        self._wstruct = None

    def build_residual(self, layer: nn.Module):
        return NormalizedResidualBlock(layer, self.embedding_dim, self.dropout_prob)

    def c_weights(self, code: int) -> L.LayerWeights:
        """The rnamsm_layer_weights struct for this layer (device pointers into the packed
        weights; the struct keeps the tensors alive through ``_wstruct``)."""
        key = (code, self._row_code) + tuple((p.data_ptr(), p._version) for p in self.parameters())
        if self._wstruct is not None and self._wstruct[0] == key:
            return self._wstruct[1]
        keep = []

        def f32(t):
            t = t.detach().float().contiguous()
            keep.append(t)
            return t.data_ptr()

        def attn(block: NormalizedResidualBlock, blk_code: int) -> L.AttnWeights:
            w_qkv, b_qkv, w_out, b_out = block.layer._pack(blk_code)
            keep.extend([w_qkv, b_qkv, w_out, b_out])
            return L.AttnWeights(f32(block.layer_norm.weight), f32(block.layer_norm.bias), w_qkv.data_ptr(),
                                 b_qkv.data_ptr(), w_out.data_ptr(), b_out.data_ptr(), blk_code)

        ffn = self.feed_forward_layer
        w1, b1, w2, b2 = ffn.layer._pack(code)
        keep.extend([w1, b1, w2, b2])
        s = L.LayerWeights(attn(self.row_self_attention, self._row_code), attn(self.column_self_attention, code),
                           f32(ffn.layer_norm.weight),
                           f32(ffn.layer_norm.bias), w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr())
        self._wstruct = (key, s, keep)
        return s

    @torch.no_grad()
    def forward(self, x: torch.Tensor, self_attn_mask: Optional[torch.Tensor] = None,
                self_attn_padding_mask: Optional[torch.Tensor] = None, need_head_weights: bool = False,
                need_col_weights: bool = False):
        """``need_col_weights=True`` (implies ``need_head_weights``) also returns the column attention's
        probabilities ``[H, C, B, R, R]`` as the middle element, where it is ``None`` otherwise."""
        if need_col_weights:
            need_head_weights = True
        _infer_only(self)
        if self_attn_mask is not None:
            raise NotImplementedError
        L.require_cuda(x, "x")
        L.device_check(x.device)
        R, Cc, B, D = x.shape
        H, F = self.num_attention_heads, self.ffn_embedding_dim
        code = self._code
        eps = float(self.row_self_attention.layer_norm.eps)
        y = torch.empty((R, Cc, B, D), dtype=torch.float32, device=x.device)
        row_attn = torch.empty((H, B, Cc, Cc), dtype=torch.float32, device=x.device) if need_head_weights else None
        col_attn = torch.empty((H, Cc, B, R, R), dtype=torch.float32, device=x.device) if need_col_weights else None
        with torch.cuda.device(x.device):
            w = self.c_weights(code)
            fcode = self._fwd_code
            nbytes = L.lib.rnamsm_workspace_bytes(R, Cc, D, H, F, fcode)
            if need_col_weights:
                nbytes += L.lib.rnamsm_col_probs_scratch_bytes(R, Cc, H)
                cp = col_attn[:, :, 0] if B == 1 else torch.empty((H, Cc, R, R), dtype=torch.float32, device=x.device)
            ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
            for b in range(B):
                # fresh fp32 copy (never a view of the caller's x): the kernels update it in place
                xb = torch.empty((R, Cc, D), dtype=torch.float32, device=x.device)
                xb.copy_(x[:, :, b, :])
                pad = _pad_u8(self_attn_padding_mask, b)
                pm = torch.empty((H, Cc, Cc), dtype=torch.float32, device=x.device) if need_head_weights else None
                if need_col_weights:
                    L.check(L.lib.rnamsm_layer_forward_col_probs(C.byref(w), D, H, F, eps, L.ptr(xb), R, Cc, L.ptr(pad),
                                                                 fcode, L.ptr(pm), L.ptr(cp), None, L.ptr(ws), nbytes, 0,
                                                                 None, None, 0, L.stream_ptr()), "layer_forward_col_probs")
                    if B > 1:
                        col_attn[:, :, b] = cp
                else:
                    L.check(L.lib.rnamsm_layer_forward(C.byref(w), D, H, F, eps, L.ptr(xb), R, Cc, L.ptr(pad), fcode,
                                                       L.ptr(pm), L.ptr(ws), nbytes, 0, None, None, 0, L.stream_ptr()),
                            "layer_forward")
                y[:, :, b, :] = xb
                if need_head_weights:
                    row_attn[:, b] = pm
        if need_head_weights:
            # without need_col_weights the column probabilities are not computed (see ColumnSelfAttention)
            return y, col_attn, row_attn
        return y


class LearnedPositionalEmbedding(nn.Embedding):
    """Parameter container with the reference's shape rule (modules.py:270-284): the lookup itself
    is fused into K1 (rnamsm_embed_layernorm)."""

    def __init__(self, num_embeddings: int, embedding_dim: int, padding_idx: int):
        if padding_idx is not None:
            num_embeddings_ = num_embeddings + padding_idx + 1
        else:
            num_embeddings_ = num_embeddings
        super().__init__(num_embeddings_, embedding_dim, padding_idx)
        self.max_positions = num_embeddings


class RobertaLMHead(nn.Module):
    """Masked-LM head parameters (modules.py:303-319); evaluated inside rnamsm_msa_forward."""

    def __init__(self, embed_dim, output_dim, weight):
        super().__init__()
        self.dense = nn.Linear(embed_dim, embed_dim)
        self.layer_norm = nn.LayerNorm(embed_dim)
        self.weight = weight
        self.bias = nn.Parameter(torch.zeros(output_dim))


class ContactPredictionHead(nn.Module):
    """Symmetrize + APC + logistic regression over the 120 maps (modules.py:322-366), on the device in
    three small HBM-bound kernels (``rnamsm_contact_head``; SURVEY.md section 8f row 2).  Keeps the
    reference's parameter (``regression.{weight,bias}``) so the state dict loads strictly."""

    def __init__(self, in_features: int, prepend_bos: bool, append_eos: bool, bias=True, eos_idx: Optional[int] = None):
        super().__init__()
        self.in_features = in_features
        self.prepend_bos = prepend_bos
        self.append_eos = append_eos
        if append_eos and eos_idx is None:
            raise ValueError("Using an alphabet with eos token, but no eos token was passed in.")
        self.eos_idx = eos_idx
        self.regression = nn.Linear(in_features, 1, bias)
        self.activation = nn.Sigmoid()

    @torch.no_grad()
    def forward(self, tokens, attentions):
        L.require_cuda(attentions, "attentions")
        if self.append_eos:
            # modules.py:349-353 zeroes the EOS row/column and drops the last position; the RNA alphabet
            # never appends EOS (msm/data.py:166-172), so this branch only keeps other vocabularies working
            eos_mask = tokens.ne(self.eos_idx).to(attentions)
            eos_mask = eos_mask.unsqueeze(1) * eos_mask.unsqueeze(2)
            attentions = attentions * eos_mask[:, None, None, :, :]
        batch_size, layers, heads, Cc, _ = attentions.size()
        start = 1 if self.prepend_bos else 0
        seqlen = Cc - start - (1 if self.append_eos else 0)
        K = layers * heads
        maps = attentions.float().contiguous()
        w = self.regression.weight.detach().float().reshape(-1).contiguous()
        b = self.regression.bias.detach().float().contiguous() if self.regression.bias is not None else None
        out = torch.empty((batch_size, seqlen, seqlen), dtype=torch.float32, device=maps.device)
        ws = torch.empty(K * seqlen + K, dtype=torch.float32, device=maps.device)
        with torch.cuda.device(maps.device):
            for bi in range(batch_size):
                L.check(L.lib.rnamsm_contact_head(L.ptr(maps[bi]), K, Cc, start, seqlen, L.ptr(w), L.ptr(b), L.ptr(out[bi]),
                                                  L.ptr(ws), L.stream_ptr()), "contact_head")
        return out
