"""ctypes binding of libb200llama.so (include/b2l.h).  Fails loudly: there is no CPU
or PyTorch fallback behind these calls."""
import ctypes as C
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200llama.so")

B2L_BF16, B2L_F32 = 0, 1
PRO_NONE, PRO_RMSNORM = 0, 1
EPI_STORE, EPI_RESIDUAL, EPI_SWIGLU = 0, 1, 2
F_PDL, F_NO_ALIAS_N, F_ROPE_ROWS = 1, 2, 4

c_void_p, c_int, c_float, c_size_t = C.c_void_p, C.c_int, C.c_float, C.c_size_t


class Q4LinearArgs(C.Structure):
    _fields_ = [
        ("x", c_void_p), ("ldx", c_int),
        ("qw_tiled", c_void_p), ("scales", c_void_p), ("zeros", c_void_p), ("sz_dtype", c_int),
        ("y", c_void_p), ("ldy", c_int),
        ("M", c_int), ("N", c_int), ("K", c_int),
        ("prologue", c_int), ("norm_scale", c_void_p), ("eps", c_float),
        ("epilogue", c_int), ("res", c_void_p), ("ldres", c_int),
        ("split_k", c_int), ("flags", c_int), ("trace", c_void_p), ("workspace", c_void_p),
        ("pf_ptr", c_void_p * 4), ("pf_bytes", C.c_ulonglong * 4),
        ("pf_kv", c_void_p * 2), ("pf_rows", c_void_p), ("pf_rows_max", c_int), ("pf_nseg", c_int), ("pf_row_bytes", c_int),
        ("pf_seg_stride", C.c_ulonglong),
    ]


class Q4Weight(C.Structure):
    _fields_ = [("qw_tiled", c_void_p), ("qw_mma", c_void_p), ("scales", c_void_p), ("zeros", c_void_p), ("N", c_int), ("K", c_int)]


class Layer(C.Structure):
    _fields_ = [
        ("rms_1", c_void_p), ("rms_2", c_void_p),
        ("c_attn", Q4Weight), ("c_proj", Q4Weight), ("c_fc12", Q4Weight), ("mlp_proj", Q4Weight),
        ("k_cache", c_void_p), ("v_cache", c_void_p),
    ]


class DecodeArgs(C.Structure):
    _fields_ = [
        ("n_layer", c_int), ("n_head", c_int), ("n_embd", c_int), ("n_hidden", c_int), ("vocab", c_int),
        ("B", c_int), ("S", c_int), ("sz_dtype", c_int), ("eps", c_float),
        ("layers", C.POINTER(Layer)),
        ("wte", c_void_p), ("ln_f", c_void_p), ("lm_head", Q4Weight), ("rope", c_void_p),
        ("idx", c_void_p), ("idx_is_i64", c_int),
        ("input_pos", c_void_p), ("ring_start", c_void_p), ("block_size", c_int),
        ("x", c_void_p), ("qkv", c_void_p), ("att", c_void_p), ("hid", c_void_p), ("attn_work", c_void_p),
        ("logits", c_void_p), ("flags", c_int), ("timeline", c_void_p), ("batch_work", c_void_p),
    ]


class TPComm(C.Structure):
    _fields_ = [("peer_buf", c_void_p * 8), ("rank", c_int), ("world", c_int), ("max_elems", c_int), ("epoch", c_void_p), ("status", c_void_p)]


_SIGS = {
    "b2l_version": (c_int, []),
    "b2l_last_error": (C.c_char_p, []),
    "b2l_device_info": (c_int, [C.POINTER(c_int)] * 3),
    "b2l_q_dequant": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "b2l_q_linear": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int,
                             c_int, c_int, c_int, c_int, c_void_p]),
    "b2l_q4_tiled_bytes": (c_size_t, [c_int, c_int]),
    "b2l_q4_tile": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "b2l_q4_untile": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "b2l_q4_linear_tc": (c_int, [C.POINTER(Q4LinearArgs), c_void_p]),
    "b2l_q4_gemm": (c_int, [C.POINTER(Q4LinearArgs), c_void_p]),
    "b2l_q4_tiled_mma_bytes": (c_size_t, [c_int, c_int]),
    "b2l_q4_tile_mma": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "b2l_q4_untile_mma": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "b2l_q4_tiled_i8_bytes": (c_size_t, [c_int, c_int]),
    "b2l_q4_tile_i8": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "b2l_q4_untile_i8": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "b2l_q4_gemv": (c_int, [C.POINTER(Q4LinearArgs), c_void_p]),
    "b2l_q4_gemv_batch": (c_int, [C.POINTER(Q4LinearArgs), c_void_p]),
    "b2l_q4_gemv_batch_workspace_bytes": (c_size_t, [c_int]),
    "b2l_rmsnorm": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, c_void_p]),
    "b2l_embedding": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "b2l_silu_mul": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "b2l_add": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "b2l_topk_softmax": (c_int, [c_void_p, c_float, c_int, c_void_p, c_int, c_void_p]),
    "b2l_topk_softmax_sample": (c_int, [c_void_p, c_float, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "b2l_q8_tiled_bytes": (c_size_t, [c_int, c_int]),
    "b2l_q8_tile": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "b2l_q8_gemv": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, c_int, c_void_p]),
    "b2l_q8_outlier_mask": (c_int, [c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_void_p]),
    "b2l_attn_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int]),
    "b2l_attention": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                              c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "b2l_tp_buffer_bytes": (c_size_t, [c_int, c_int]),
    "b2l_tp_allreduce": (c_int, [C.POINTER(TPComm), c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "b2l_ring_advance": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p]),
    "b2l_attention_nocache": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "b2l_kv_unroll": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "b2l_decode_step": (c_int, [C.POINTER(DecodeArgs), c_void_p]),
    "b2l_decode_step_launches": (c_int, [C.POINTER(DecodeArgs)]),
}

EXPORTS = tuple(_SIGS)

_lib = None
_lock = threading.Lock()


def lib():
    """The loaded library.  Raises if it has not been built (`python -c 'import
    __graft_entry__ as g; g.build()'`)."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
                        "lit_llama_b200 has no CPU or PyTorch fallback.")
                handle = C.CDLL(LIB_PATH)
                for name, (res, args) in _SIGS.items():
                    fn = getattr(handle, name)
                    fn.restype = res
                    fn.argtypes = args
                _lib = handle
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().b2l_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed (rc={rc}): {msg}")


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def require_cuda_bf16(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"{what}: tensor is on {t.device}; lit_llama_b200 runs on CUDA only (no CPU fallback)")
    if t.dtype != torch.bfloat16:
        raise RuntimeError(f"{what}: dtype {t.dtype} unsupported; activations must be torch.bfloat16")


def sz_dtype_of(t: torch.Tensor) -> int:
    if t.dtype == torch.bfloat16:
        return B2L_BF16
    if t.dtype == torch.float32:
        return B2L_F32
    raise RuntimeError(f"scales/zeros dtype {t.dtype} unsupported (bf16 or fp32)")
