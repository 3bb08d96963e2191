"""ctypes binding of libmobgt.so — the thin C-ABI custom-op layer (include/mobgt.h).

There is NO fallback: if the shared library is missing or a call fails, a MobgtError is raised.
Tensors cross the boundary as raw device pointers (`tensor.data_ptr()`), the current torch CUDA
stream as a `void*`.
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libmobgt.so")

c_i32, c_i64, c_p, c_f32 = ctypes.c_int32, ctypes.c_int64, ctypes.c_void_p, ctypes.c_float

# include/mobgt.h limits
MAX_NODES = 512          # MOBGT_MAX_NODES: the collator's default cap
MAX_MODEL_NODES = 1024   # MOBGT_MAX_MODEL_NODES: the model's kernels (K2 / K3), T <= 1025 (collator large_graphs=True)
MAX_APSP_NODES = 1024    # MOBGT_MAX_APSP_NODES: K1 (mobgt_apsp_edge_input, mobgt_gen_edge_input)


class MobgtError(RuntimeError):
    pass


# name -> argtypes ; every function returns int32 status (include/mobgt.h)
SIGNATURES = {
    "mobgt_version": [],
    "mobgt_last_error": [ctypes.c_char_p, ctypes.c_size_t],
    "mobgt_device_check": [],
    "mobgt_launch_count": [c_p],
    "mobgt_apsp_edge_input": [c_p, c_p, c_p, c_p, c_i32, c_i32, c_i32, c_i32, c_i32, c_p, c_p, c_p, c_p, c_p],
    "mobgt_gen_edge_input": [c_p, c_p, c_p, c_p, c_i32, c_i32, c_i32, c_i32, c_p, c_p],
    "mobgt_degrees": [c_p, c_p, c_p, c_p, c_i32, c_i32, c_p, c_p, c_p],
    "mobgt_poi_pos": [c_p, c_p, c_p, c_p, c_p, c_f32, c_i32, c_i32, c_i32, c_p, c_p],
    "mobgt_bias_fwd": [c_p, c_p, c_p, c_p, c_p, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_p, c_p, c_p, c_p, c_p, c_p,
                       c_p, c_i32, c_p],
    "mobgt_bias_fwd_workspace_bytes": [c_i32, c_i32],
    "mobgt_bias_bwd_workspace_bytes": [c_i32, c_i32, c_i32],
    "mobgt_bias_bwd_heads_workspace_bytes": [c_i32, c_i32, c_i32, c_i32],
    "mobgt_bias_bwd": [c_p, c_p, c_p, c_p, c_p, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_p, c_i32, c_i32, c_i64, c_p,
                       c_p, c_p, c_i64, c_p, c_p, c_p, c_p, c_p, c_p],
    "mobgt_bias_direct_fwd": [c_p, c_p, c_p, c_p, c_p, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_p, c_p, c_p, c_p, c_p, c_i32, c_p],
    "mobgt_bias_direct_bwd_workspace_bytes": [c_i32, c_i32, c_i32],
    "mobgt_bias_direct_bwd": [c_p, c_p, c_p, c_p, c_p, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_p, c_i32, c_i32, c_i64, c_p, c_i64,
                              c_p, c_p, c_p, c_p, c_p],
    "mobgt_attn_fwd": [c_p, c_p, c_p, c_i64, c_p, c_p, c_p, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_f32, c_f32, ctypes.c_uint64,
                       c_p, c_p, c_p, c_p],
    "mobgt_attn_bwd": [c_p, c_p, c_p, c_i64, c_p, c_p, c_p, c_p, c_p, c_p, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_f32, c_p,
                       c_p, c_p, c_i64, c_p, c_i32, c_f32, ctypes.c_uint64, c_p, c_p],
    "mobgt_attn_f32_fwd": [c_p, c_p, c_p, c_i64, c_p, c_p, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_f32, c_f32, ctypes.c_uint64, c_p,
                           c_p, c_p, c_p],
    "mobgt_attn_f32_bwd": [c_p, c_p, c_p, c_i64, c_p, c_p, c_p, c_p, c_p, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_f32, c_p, c_p, c_p,
                           c_i64, c_p, c_i32, c_f32, ctypes.c_uint64, c_p, c_p],
    # the same four with an int32 head_dim before the stream (built: 16, 24)
    "mobgt_attn_fwd_hd": [c_p, c_p, c_p, c_i64, c_p, c_p, c_p, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_f32, c_f32,
                          ctypes.c_uint64, c_p, c_p, c_p, c_i32, c_p],
    "mobgt_attn_bwd_hd": [c_p, c_p, c_p, c_i64, c_p, c_p, c_p, c_p, c_p, c_p, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_f32, c_p,
                          c_p, c_p, c_i64, c_p, c_i32, c_f32, ctypes.c_uint64, c_p, c_i32, c_p],
    "mobgt_attn_f32_fwd_hd": [c_p, c_p, c_p, c_i64, c_p, c_p, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_f32, c_f32, ctypes.c_uint64,
                              c_p, c_p, c_p, c_i32, c_p],
    "mobgt_attn_f32_bwd_hd": [c_p, c_p, c_p, c_i64, c_p, c_p, c_p, c_p, c_p, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_f32, c_p, c_p,
                              c_p, c_i64, c_p, c_i32, c_f32, ctypes.c_uint64, c_p, c_i32, c_p],
    "mobgt_embed_gather_fwd": [c_p, c_p, c_p, c_p, c_p, c_p, c_i32, c_i32, c_i32, c_i32, c_p, c_i32, c_p],
    "mobgt_embed_sum_fwd": [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i32, c_i32, c_p, c_i32, c_p],
    "mobgt_segment_sum": [c_p, c_i32, c_i64, c_i32, c_i32, c_p, c_p, c_i32, c_p, c_i32, c_p, c_i64, c_p],
    "mobgt_head_topk": [c_p, c_p, c_p, c_p, c_i32, c_i32, c_i32, c_i64, c_i32, c_i32, c_i32, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p],
    "mobgt_head_topk_f32": [c_p, c_p, c_p, c_p, c_i32, c_i32, c_i32, c_i64, c_i32, c_i32, c_i32, c_p, c_p, c_p, c_p, c_p, c_p, c_p,
                            c_p],
    "mobgt_topk_merge": [c_p, c_p, c_p, c_p, c_i32, c_i32, c_i32, c_p, c_p, c_p, c_p],
    "mobgt_layernorm_fwd": [c_p, c_p, c_p, c_f32, c_i32, c_i32, c_p, c_p, c_p, c_p, c_p],
    "mobgt_layernorm_bwd_workspace_bytes": [c_i32],
    "mobgt_layernorm_bwd": [c_p, c_p, c_p, c_p, c_p, c_p, c_i32, c_i32, c_p, c_p, c_p, c_p, c_i64, c_p],
    "mobgt_add_dropout_layernorm_fwd": [c_p, c_p, c_f32, ctypes.c_uint64, c_p, c_p, c_f32, c_i32, c_i32, c_p, c_p, c_p, c_p, c_p, c_p, c_p],
    "mobgt_add_dropout_layernorm_bwd": [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i32, c_i32, c_f32, ctypes.c_uint64, c_p, c_p, c_p, c_p,
                                        c_p, c_p, c_i64, c_p, c_p],
    "mobgt_colsum_workspace_bytes": [c_i32, c_i32],
    "mobgt_colsum": [c_p, c_i32, c_i64, c_i32, c_i32, c_p, c_p, c_i64, c_p],
    "mobgt_gelu_bwd_colsum": [c_p, c_p, c_i32, c_i32, c_p, c_p, c_p, c_i64, c_p],
    "mobgt_loss_workspace_bytes": [c_i32, c_i32],
    "mobgt_lsm_nll_fwd": [c_p, c_i32, c_i64, c_p, c_i64, c_i32, c_i32, c_p, c_i64, c_p, c_p, c_p],
    "mobgt_lsm_nll_bwd": [c_p, c_i32, c_i64, c_p, c_i64, c_i32, c_i32, c_p, c_p, c_p, c_p, c_i64, c_p],
    "mobgt_gtl_fwd": [c_p, c_i32, c_i64, c_p, c_f32, c_i32, c_i32, c_p, c_i64, c_p, c_p],
    "mobgt_gtl_bwd": [c_p, c_i32, c_i64, c_p, c_f32, c_i32, c_i32, c_p, c_p, c_i64, c_p],
    "mobgt_spmm_csr": [c_p, c_p, c_p, c_i32, c_p, c_i32, c_p, c_f32, c_i32, c_p, c_p],
    "mobgt_adamw_step": [c_p, c_p, c_p, c_p, c_i64, c_f32, c_f32, c_f32, c_f32, c_f32, c_i64, c_p],
    "mobgt_gemm_workspace_bytes": [c_i32, c_i32, c_i32],
    "mobgt_gemm_bf16": [c_p, c_i64, c_p, c_i64, c_p, c_p, c_i64, c_i32, c_i32, c_i32, c_i32, c_p, c_i64, c_p, c_i64, c_i32, c_p, c_p,
                        c_i64, c_p],
    "mobgt_debug_set_timeline": [c_p],
    "mobgt_debug_head_cluster": [c_i32],
    "mobgt_gemm_exact_gelu": [c_i32],
    "mobgt_selftest_umma": [c_p, c_p, c_i32, c_i32, c_i32, c_i32, c_p, c_p],
}

_lib = None


def lib():
    """Load libmobgt.so (once).  Raises MobgtError if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MobgtError(
                f"{LIB_PATH} not found: build it with `python -m mobgt_b200.build` "
                "(there is no CPU / PyTorch fallback for the MobGT hot path)")
        L = ctypes.CDLL(LIB_PATH)
        for name, argt in SIGNATURES.items():
            fn = getattr(L, name)
            fn.argtypes = argt
            fn.restype = c_i64 if name.endswith("_bytes") else c_i32
        _lib = L
    return _lib


def last_error():
    buf = ctypes.create_string_buffer(512)
    lib().mobgt_last_error(buf, 512)
    return buf.value.decode("utf-8", "replace")


def call(name, *args):
    """Call an entry point; raise MobgtError(status, message) on a non-zero status."""
    rc = getattr(lib(), name)(*args)
    if rc != 0:
        raise MobgtError(f"{name} failed with status {rc}: {last_error()}")
    return rc


def ptr(t):
    """Device (or host) pointer of a torch tensor / None -> NULL."""
    if t is None:
        return None
    assert t.is_contiguous(), "libmobgt expects contiguous tensors"
    return t.data_ptr()


def stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream


_cuda_ok = False


def require_cuda():
    global _cuda_ok
    if _cuda_ok:
        return
    import torch
    if not torch.cuda.is_available():
        raise MobgtError("the MobGT hot path runs on a B200 (sm_100a) only: no CUDA device is available "
                         "and there is no CPU fallback")
    call("mobgt_device_check")
    _cuda_ok = True


def launch_count():
    """libmobgt kernels launched by this process so far."""
    v = ctypes.c_int64(0)
    call("mobgt_launch_count", ctypes.byref(v))
    return int(v.value)
