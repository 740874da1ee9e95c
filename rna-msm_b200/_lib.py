"""ctypes binding of librnamsm_b200.so (C ABI: include/rnamsm_b200.h).

The product path has NO fallback: if the shared library is missing or fails to load, importing
this module raises, and every op raises ``RuntimeError`` carrying ``rnamsm_last_error()`` when a
call returns non-zero.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "librnamsm_b200.so")

F32, BF16, F16 = 0, 1, 2
EPI_BIAS, EPI_BIAS_GELU, EPI_BIAS_RESIDUAL = 0, 1, 2

_vp, _i, _f, _ll, _sz = C.c_void_p, C.c_int, C.c_float, C.c_longlong, C.c_size_t


class AttnWeights(C.Structure):
    _fields_ = [("ln_w", _vp), ("ln_b", _vp), ("w_qkv", _vp), ("b_qkv", _vp), ("w_out", _vp), ("b_out", _vp),
                ("dtype", _i)]


class LayerWeights(C.Structure):
    _fields_ = [("row", AttnWeights), ("col", AttnWeights), ("ffn_ln_w", _vp), ("ffn_ln_b", _vp),
                ("fc1_w", _vp), ("fc1_b", _vp), ("fc2_w", _vp), ("fc2_b", _vp)]


class ModelWeights(C.Structure):
    _fields_ = [("num_layers", _i), ("embed_dim", _i), ("num_heads", _i), ("ffn_dim", _i), ("vocab", _i),
                ("n_pos", _i), ("pad_idx", _i), ("ln_eps", _f),
                ("tok_emb", _vp), ("pos_emb", _vp), ("row_pos", _vp),
                ("ln_before_w", _vp), ("ln_before_b", _vp), ("ln_after_w", _vp), ("ln_after_b", _vp),
                ("lm_dense_w", _vp), ("lm_dense_b", _vp), ("lm_ln_w", _vp), ("lm_ln_b", _vp), ("lm_bias", _vp),
                ("layers", C.POINTER(LayerWeights)), ("lm_dense_w16", _vp)]


# name -> (restype, argtypes); every symbol include/rnamsm_b200.h declares
SIGNATURES = {
    "rnamsm_version": (_i, []),
    "rnamsm_last_error": (C.c_char_p, []),
    "rnamsm_device_check": (_i, []),
    "rnamsm_launch_count": (_ll, []),
    "rnamsm_gemm_pairs": (_i, []),
    "rnamsm_profile_enable": (_i, [_i]),
    "rnamsm_profile_num_classes": (_i, []),
    "rnamsm_profile_class_name": (C.c_char_p, [_i]),
    "rnamsm_profile_collect": (_i, [C.POINTER(C.c_double), C.POINTER(_ll), _i]),
    "rnamsm_embed_layernorm": (_i, [_vp, _i, _i, _vp, _i, _vp, _i, _vp, _vp, _vp, _i, _i, _f, _vp, _vp, _vp]),
    "rnamsm_layernorm": (_i, [_vp, _vp, _vp, _vp, _i, _ll, _i, _f, _i, _i, _vp]),
    "rnamsm_linear": (_i, [_vp, _vp, _vp, _ll, _i, _i, _i, _i, _f, _i, _vp, _vp, _vp]),
    "rnamsm_linear_tf32_scratch_bytes": (_sz, [_ll, _i, _i]),
    "rnamsm_linear_tf32": (_i, [_vp, _vp, _vp, _ll, _i, _i, _i, _f, _i, _vp, _vp, _vp, _sz, _vp]),
    "rnamsm_linear_residual_layernorm": (_i, [_vp, _vp, _vp, _ll, _i, _i, _i, _vp, _vp, _vp, _f, _vp, _i, _i, _i, _vp, _vp]),
    "rnamsm_row_attn_logits": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _vp]),
    "rnamsm_row_attn_splits": (_i, [_i, _i, _i, _i]),
    "rnamsm_row_attn_short_chunks": (_i, [_i, _i, _i]),
    "rnamsm_row_attn_short": (_i, [_vp, _i, _i, _i, _i, _vp, _f, _vp, _i, _vp, _vp, _i, _vp, _vp]),
    "rnamsm_row_softmax": (_i, [_vp, _i, _i, _i, _vp, _f, _vp, _vp, _i, _i, _vp]),
    "rnamsm_row_attn_av": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _vp, _vp]),
    "rnamsm_col_attn": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "rnamsm_col_attn_probs": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "rnamsm_col_probs_scratch_bytes": (_sz, [_i, _i, _i]),
    "rnamsm_vocab_proj": (_i, [_vp, _vp, _vp, _ll, _i, _i, _vp, _vp]),
    "rnamsm_msa_clean": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp]),
    "rnamsm_msa_greedy_workspace": (_sz, [_i, _i]),
    "rnamsm_msa_greedy_select": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "rnamsm_msa_tokenize": (_i, [_vp, _i, _vp, _i, _vp, _i, _vp, _vp]),
    "rnamsm_ss_pack": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "rnamsm_contact_head": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "rnamsm_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i]),
    "rnamsm_fused_layernorm": (_i, [_i]),
    "rnamsm_range_scan": (_i, [_vp, _ll, _i, _vp, _vp]),
    "rnamsm_debug_range_watch": (_i, [_vp]),
    "rnamsm_layer_forward": (_i, [C.POINTER(LayerWeights), _i, _i, _i, _f, _vp, _i, _i, _vp, _i, _vp, _vp, _sz,
                                  _i, _vp, _vp, _i, _vp]),
    "rnamsm_layer_forward_col_probs": (_i, [C.POINTER(LayerWeights), _i, _i, _i, _f, _vp, _i, _i, _vp, _i, _vp, _vp, _vp,
                                            _vp, _sz, _i, _vp, _vp, _i, _vp]),
    "rnamsm_peer_alloc": (_i, [_sz, C.POINTER(_vp)]),
    "rnamsm_peer_free": (_i, [_vp]),
    "rnamsm_ipc_export": (_i, [_vp, _vp]),
    "rnamsm_ipc_import": (_i, [_vp, C.POINTER(_vp)]),
    "rnamsm_ipc_close": (_i, [_vp]),
    "rnamsm_layernorm_push": (_i, [_vp, _vp, _vp, C.POINTER(_vp), _i, _i, _i, _i, _i, _i, _f, _i, _vp]),
    "rnamsm_row_softmax_p2p": (_i, [C.POINTER(_vp), _i, _i, _i, _i, _i, _vp, _f, _vp, C.POINTER(_vp), _i, _i, _vp]),
    "rnamsm_peer_barrier": (_i, [C.POINTER(_vp), _i, _i, C.c_uint, _vp]),
    "rnamsm_copy_map_rows_d2h": (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "rnamsm_host_register": (_i, [_vp, _sz]),
    "rnamsm_host_unregister": (_i, [_vp]),
    "rnamsm_linear_residual_scatter": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, C.POINTER(_vp), _i, _i, _i, _i, _i, _vp]),
    "rnamsm_add_layernorm": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _i, _ll, _i, _f, _vp]),
    "rnamsm_msa_forward": (_i, [C.POINTER(ModelWeights), _vp, _i, _i, _i, _i, _vp, _vp, C.POINTER(_vp), _vp, _vp,
                                _sz, _vp]),
    "rnamsm_msa_forward_col_probs": (_i, [C.POINTER(ModelWeights), _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp,
                                          C.POINTER(_vp), _vp, _vp, _sz, _vp]),
    "rnamsm_batch_workspace_bytes": (_sz, [_i, C.POINTER(_i), C.POINTER(_i), _i, _i, _i, _i]),
    "rnamsm_msa_forward_batch": (_i, [C.POINTER(ModelWeights), _i, _vp, C.POINTER(_i), C.POINTER(_i), C.c_char_p, _i, _vp,
                                      C.POINTER(_vp), _vp, _sz, _vp]),
    "rnamsm_score_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i, _i]),
    "rnamsm_msa_masked_marginals": (_i, [C.POINTER(ModelWeights), _vp, _i, _i, _i, _i, _i, _vp, _i, _i, _i, _vp, _vp,
                                         _vp, _sz, _vp]),
    "rnamsm_sample_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i, _i, _i]),
    "rnamsm_msa_gibbs_sample": (_i, [C.POINTER(ModelWeights), _vp, _i, _i, _i, _i, _vp, _i, _i, _i, _i, C.c_float,
                                     C.c_float, C.c_uint, C.c_ulonglong, _i, _vp, _vp, _sz, _vp]),
    "rnamsm_jacobian_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i, _i, _i, _i, _i]),
    "rnamsm_msa_categorical_jacobian": (_i, [C.POINTER(ModelWeights), _vp, _i, _i, _i, _i, _i, C.POINTER(_i), _i,
                                             C.POINTER(_i), _i, C.POINTER(_i), _i, _i, _vp, _vp, _sz, _vp]),
    "rnamsm_jacobian_contacts_scratch_bytes": (_sz, [_i, _i]),
    "rnamsm_jacobian_contacts": (_i, [_vp, _i, _i, _vp, _vp, _sz, _vp]),
    "rnamsm_window_starts": (_i, [_i, _i, _i, C.POINTER(_i)]),
    "rnamsm_windows_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i]),
    "rnamsm_msa_forward_windows": (_i, [C.POINTER(ModelWeights), _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp,
                                        _vp, _sz, _vp]),
    "rnamsm_seq_weights_workspace_bytes": (_sz, [_i, _i]),
    "rnamsm_msa_seq_weights": (_i, [_vp, _i, _i, C.c_double, _vp, _vp, _vp, _sz, _vp]),
    "rnamsm_dca_workspace_bytes": (_sz, [_i, _i]),
    "rnamsm_msa_dca": (_i, [_vp, _i, _i, C.c_double, C.c_double, _vp, _vp, _vp, _vp, _sz, _vp]),
    "rnamsm_fold_workspace_bytes": (_sz, [_i, C.POINTER(_i)]),
    "rnamsm_fold": (_i, [_i, C.POINTER(_vp), C.POINTER(_i), C.POINTER(_vp), _i, C.c_double, _f, _i, _i, C.POINTER(_vp),
                         _vp, _vp, _sz, _vp]),
    "rnamsm_rsa_pack":(_i, [_vp, _i, _i, _i, _vp, C.POINTER(C.c_double), C.POINTER(C.c_double), _vp, _vp, _vp, _vp]),
}

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} not found: build it with `python rna-msm_b200/build.py` "
        "(nvcc, sm_100a).  rnamsm_b200 has no CPU / PyTorch fallback.")

lib = C.CDLL(LIB_PATH)
for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)  # AttributeError here = ABI mismatch, fail loudly
    _fn.restype = _res
    _fn.argtypes = _args

ABI_VERSION = 3
assert lib.rnamsm_version() == ABI_VERSION, "librnamsm_b200.so ABI version mismatch"


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib.rnamsm_last_error().decode(errors="replace")
        raise RuntimeError(f"rnamsm_b200 {what} failed (status {rc}): {msg}")


def ptr(t):
    """Device pointer of a tensor (or None)."""
    return None if t is None else t.data_ptr()


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(
            f"rnamsm_b200: {what} must be a CUDA tensor (got {t.device}); this package is the B200 "
            "CUDA path and has no CPU fallback")


_checked_devices = set()


def device_check(device: torch.device) -> None:
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx in _checked_devices:
        return
    with torch.cuda.device(idx):
        check(lib.rnamsm_device_check(), "device_check")
    _checked_devices.add(idx)


def dtype_code(precision: str) -> int:
    if precision in ("bf16", "bfloat16", "bf16_pure"):
        return BF16
    if precision in ("fp16", "float16", "f16"):
        return F16
    if precision in ("fp32", "float32", "f32", "tf32x3"):
        return F32
    raise ValueError(f"unknown precision {precision!r} (expected 'fp16', 'bf16', 'bf16_pure', 'tf32x3' or 'fp32')")


F32_TENSOR = 0x100


def forward_code(precision: str) -> int:
    """dtype argument of rnamsm_workspace_bytes / rnamsm_layer_forward / rnamsm_msa_forward: 'tf32x3' is the fp32 path
    with RNAMSM_F32_TENSOR (nn.Linear layers as three-term tf32 products on the tensor cores)."""
    return dtype_code(precision) | (F32_TENSOR if precision == "tf32x3" else 0)


def row_dtype_code(precision: str) -> int:
    """Operand type of the tied row-attention block.  The production 'bf16' path runs it in fp16
    (same tensor-core rate, 3 more mantissa bits: the tied logits are sums of R*64 products and
    feed the exported maps); 'bf16_pure' keeps bf16 there too (RNAMSM_ROW_ATTN_FP16=0 does the same)."""
    code = dtype_code(precision)
    if code == BF16 and precision != "bf16_pure" and os.environ.get("RNAMSM_ROW_ATTN_FP16", "1") != "0":
        return F16
    return code


def torch_dtype(code: int) -> torch.dtype:
    return {BF16: torch.bfloat16, F16: torch.float16}.get(code, torch.float32)


def profile_enable(on: bool) -> None:
    check(lib.rnamsm_profile_enable(int(on)), "profile_enable")


def profile_collect():
    """-> {class_name: (milliseconds, launches)} accumulated since profile_enable(True)."""
    n = lib.rnamsm_profile_num_classes()
    ms = (C.c_double * n)()
    cnt = (_ll * n)()
    check(lib.rnamsm_profile_collect(ms, cnt, n), "profile_collect")
    return {lib.rnamsm_profile_class_name(i).decode(): (ms[i], cnt[i]) for i in range(n)}


class RangeWatch:
    """``with RangeWatch() as w: model(tokens)`` then ``w.saturated`` / ``w.max_abs``: did any 16-bit activation of the
    forward reach the edge of its type's range (fp16: 65504, where the kernels clamp with satfinite)?  Debugging aid."""

    def __enter__(self):
        self.counters = torch.zeros(2, dtype=torch.int64, device="cuda")
        check(lib.rnamsm_debug_range_watch(self.counters.data_ptr()), "debug_range_watch")
        return self

    def __exit__(self, *exc):
        check(lib.rnamsm_debug_range_watch(None), "debug_range_watch")
        torch.cuda.synchronize()
        c = self.counters.cpu()
        self.saturated = int(c[0])
        self.max_abs = float(torch.tensor([int(c[1])], dtype=torch.int64).to(torch.int32).view(torch.float32)[0])
        return False
