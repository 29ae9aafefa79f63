"""ctypes binding of libcogview_b200.so (the C ABI declared in include/cogview_b200.h).

There is no CPU or PyTorch fallback: if the library is missing or a call fails, this raises.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libcogview_b200.so")

_lib = None

c_void_p = ctypes.c_void_p
c_int = ctypes.c_int
c_int64 = ctypes.c_int64
c_float = ctypes.c_float


class CogViewB200Error(RuntimeError):
    pass


class DecodeStepArgs(ctypes.Structure):
    """cv_decode_step_args of include/cogview_b200.h (host struct)."""
    _fields_ = [("layers", c_void_p),
                ("num_layers", c_int), ("hidden", c_int), ("heads", c_int), ("vocab", c_int), ("batch", c_int),
                ("max_len", c_int),
                ("eps", c_float), ("eps_final", c_float),
                ("wte", c_void_p), ("wpe", c_void_p), ("lnf_g", c_void_p), ("lnf_b", c_void_p),
                ("ids", c_void_p), ("pos", c_void_p), ("cur_len", c_void_p),
                ("cache", c_void_p), ("cache_layer_stride", c_int64), ("cache_batch_stride", c_int64),
                ("logits", c_void_p), ("ld_logits", c_int64),
                ("workspace", c_void_p), ("prof", c_void_p)]


def _declare(lib):
    lib.cv_version.restype = c_int
    lib.cv_last_error.restype = ctypes.c_char_p
    sigs = {
        "cv_gemm_bf16": [c_void_p, c_int, c_int64, c_void_p, c_int, c_int64, c_void_p, c_int, c_int64, c_void_p,
                         c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p],
    }
    P, I, L, F = c_void_p, c_int, c_int64, c_float
    U64, U32 = ctypes.c_uint64, ctypes.c_uint32
    sigs.update({
        "cv_layernorm_absmax_fwd": [P, I, P, P, P, F, P, P, I, P, P, P, I, I, P],
        "cv_layernorm_absmax_bwd": [P, I, P, I, P, P, P, P, P, I, P, P, P, I, I, F, U64, U32, P, P],
        "cv_absmax": [P, I, L, P, P],
        "cv_attn_fwd": [P, L, L, P, L, L, P, L, L, P, L, L, P, I, I, I, I, I, I, F, U64, U32, P, P],
        "cv_attn_bwd": [P, L, L, P, L, L, P, L, L, P, P, P, P, P, I, I, I, I, I, F, P, P],
        "cv_linear_small_m": [P, L, P, L, P, P, L, I, I, P, I, I, I, P],
        "cv_ln_pair_small_m": [P, P, P, P, P, P, P, F, P, P, I, I, P],
        "cv_attn_gather": [P, L, L, P, L, P, P, I, I, I, I, I, P],
        "cv_attn_decode": [P, P, L, P, I, P, P, I, I, I, I, I, P],
        "cv_sparse_plan": [P, L, P, I, I, I, I, I, P, P, I, P, P, P],
        "cv_attn_decode_gather": [P, P, L, P, P, L, P, P, P, I, I, I, I, I, P],
        "cv_adamw_step": [P, P, P, P, P, L, F, F, F, F, F, I, P, F, P],
        "cv_sumsq_bf16": [P, L, P, P],
        "cv_adamw_step_multi": [P, I, F, F, F, P, F, P, P],
        "cv_sumsq_bf16_multi": [P, I, P, P],
        "cv_clip_coef": [P, F, P, P, P, P],
        "cv_conv2d_k4s2": [P, P, P, P, I, I, I, I, I, I, P],
        "cv_conv_transpose2d_k4s2": [P, P, P, P, I, I, I, I, I, I, P],
        "cv_im2col_k4s2_c3": [P, P, I, I, I, P],
        "cv_vq_split3": [P, P, L, I, P],
        "cv_vq_argmin": [P, L, P, P, P, P, L, I, I, F, P],
        "cv_vq_lookup": [P, P, P, P, L, I, P],
        "cv_conv1x1_out3": [P, P, P, P, P, P, I, I, I, I, P],
        "cv_embed_fwd": [P, P, P, P, P, P, I, I, F, U64, U32, P],
        "cv_embed_bwd": [P, P, P, P, P, I, I, F, U64, U32, P],
        "cv_dropout_mask": [P, L, F, U64, U32, P],
        "cv_gemm_bf16_dropout": [P, I, L, P, I, L, P, I, L, P, P, I, P, I, I, I, I, F, U64, U32, P],
        "cv_cross_entropy_fwd": [P, L, P, P, P, P, I, I, P],
        "cv_cross_entropy_bwd": [P, L, P, P, P, P, P, L, I, I, P],
        "cv_gelu_bwd": [P, P, P, L, P],
        "cv_colsum_bf16": [P, L, P, P, I, I, P],
        "cv_attn_sparse_fwd": [P, L, L, P, L, L, P, L, L, P, P, L, L, P, P, I, I, I, I, I, I, I, P],
        "cv_attn_sparse_bwd": [P, L, L, P, L, L, P, L, L, P, P, P, P, P, P, I, I, I, I, I, I, I, P],
        "cv_attn_sparse_dropout_fwd": [P, L, L, P, L, L, P, L, L, P, P, L, L, P, P, I, I, I, I, I, I, I, F, U64, U32, P,
                                       P],
        "cv_attn_sparse_dropout_bwd": [P, L, L, P, L, L, P, L, L, P, P, P, P, P, P, I, I, I, I, I, I, I, F, P, P],
        "cv_decode_step": [ctypes.POINTER(DecodeStepArgs), P],
        "cv_sample_topk": [P, L, I, I, F, I, ctypes.POINTER(c_int), I, U64, P, P, P, P, L, P, P, P, P, P, P],
    })
    lib.cv_attn_sparse_workspace_bytes.argtypes = [I, I, I, I]
    lib.cv_attn_sparse_workspace_bytes.restype = L
    lib.cv_attn_sparse_bwd_workspace_bytes.argtypes = [I, I, I, I, I]
    lib.cv_attn_sparse_bwd_workspace_bytes.restype = L
    lib.cv_attn_sparse_drop_mask_words.argtypes = [I, I, I, I, I, I]
    lib.cv_attn_sparse_drop_mask_words.restype = L
    lib.cv_decode_step_workspace_bytes.argtypes = [I, I]
    lib.cv_decode_step_workspace_bytes.restype = L
    lib.cv_layernorm_bwd_workspace_bytes.argtypes = [I, I]
    lib.cv_layernorm_bwd_workspace_bytes.restype = L
    lib.cv_attn_bwd_workspace_bytes.argtypes = [I, I, I, I]
    lib.cv_attn_bwd_workspace_bytes.restype = L
    lib.cv_attn_decode_workspace_bytes.argtypes = [I, I, I]
    lib.cv_attn_decode_workspace_bytes.restype = L
    lib.cv_launch_count.restype = ctypes.c_longlong
    lib.cv_set_reserved_sms.argtypes = [I]
    lib.cv_set_reserved_sms.restype = I
    lib.cv_colsum_workspace_bytes.argtypes = [I]
    lib.cv_colsum_workspace_bytes.restype = L
    for name, args in sigs.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = c_int
    return sigs


def lib():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CogViewB200Error(
                "libcogview_b200.so not found at %s — build it with `python -m cogview_b200.csrc.build` "
                "(there is no fallback path)" % LIB_PATH)
        _lib = ctypes.CDLL(LIB_PATH)
        _declare(_lib)
    return _lib


def check(rc, name="call"):
    if rc != 0:
        msg = lib().cv_last_error()
        raise CogViewB200Error("%s failed (rc=%d): %s" % (name, rc, msg.decode() if msg else "?"))


def stream_ptr():
    return torch.cuda.current_stream().cuda_stream


def ptr(t):
    return 0 if t is None else t.data_ptr()


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise CogViewB200Error("cogview_b200 kernels need CUDA tensors; got a %s tensor (no CPU fallback)"
                                   % t.device)
