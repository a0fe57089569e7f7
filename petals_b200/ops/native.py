"""ctypes bindings for the native libraries.

``lib()`` returns the sm_100a kernel library (needs a CUDA device at call time, not at load time);
``rt()`` returns the host-only runtime library (scheduler queue, KV page allocator, safetensors reader).
Both are built in-tree by :mod:`petals_b200._build`. On a GPU host a missing/stale CUDA library is a hard
error — the engine never silently falls back to PyTorch eager for its hot ops.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from typing import Optional

import torch

from petals_b200 import _build

PB_MAX_PEERS = 8
_ERRORS = {1: "bad shape/arguments", 2: "CUDA launch error", 3: "unsupported configuration", 4: "driver entry point unavailable"}

_lock = threading.Lock()
_lib: Optional[C.CDLL] = None
_rt: Optional[C.CDLL] = None


class NativeError(RuntimeError):
    pass


class LinearDecodeArgs(C.Structure):
    _fields_ = [
        ("x", C.c_void_p), ("w", C.c_void_p), ("w2", C.c_void_p), ("bias", C.c_void_p), ("bias2", C.c_void_p),
        ("residual", C.c_void_p), ("out", C.c_void_p), ("norm_w", C.c_void_p), ("norm_b", C.c_void_p),
        ("x_out", C.c_void_p),
        ("eps", C.c_float), ("norm_kind", C.c_int), ("act", C.c_int), ("M", C.c_int), ("N", C.c_int), ("K", C.c_int),
        ("n_parts", C.c_int), ("parts", C.c_void_p * PB_MAX_PEERS),
        ("wait_flag", C.c_void_p), ("wait_per_epoch", C.c_uint64), ("epoch", C.c_void_p),
        ("n_push", C.c_int), ("push_out", C.c_void_p * PB_MAX_PEERS), ("push_flag", C.c_void_p * PB_MAX_PEERS),
        ("error_flag", C.c_void_p),
        ("num_sms", C.c_int), ("fixed_grid", C.c_int), ("out_grid", C.POINTER(C.c_int)),
        ("done_counter", C.c_void_p),
        ("rope_q_out", C.c_void_p), ("rope_k_pool", C.c_void_p), ("rope_v_pool", C.c_void_p), ("rope_block_table", C.c_void_p),
        ("rope_pos_ptr", C.c_void_p), ("rope_cos", C.c_void_p), ("rope_sin", C.c_void_p),
        ("rope_T", C.c_int), ("rope_Hq", C.c_int), ("rope_Hkv", C.c_int), ("rope_D", C.c_int), ("rope_max_pages", C.c_int), ("rope_max_pos", C.c_int),
        ("n_ll_parts", C.c_int), ("ll_parts", C.c_void_p * PB_MAX_PEERS), ("n_ll_push", C.c_int), ("ll_push", C.c_void_p * PB_MAX_PEERS),
        ("ll_tag_mul", C.c_uint32), ("ll_tag_add", C.c_uint32), ("rope_num_pages", C.c_int),
    ]


class LinearFp8Args(C.Structure):
    _fields_ = [
        ("x", C.c_void_p), ("w", C.c_void_p), ("w_scale", C.c_void_p), ("w2", C.c_void_p), ("w2_scale", C.c_void_p),
        ("bias", C.c_void_p), ("bias2", C.c_void_p), ("residual", C.c_void_p), ("out", C.c_void_p), ("norm_w", C.c_void_p),
        ("norm_b", C.c_void_p), ("eps", C.c_float), ("norm_kind", C.c_int), ("act", C.c_int), ("M", C.c_int), ("N", C.c_int),
        ("K", C.c_int), ("num_sms", C.c_int),
    ]


class GemmFp8Args(C.Structure):
    _fields_ = [
        ("a_q", C.c_void_p), ("a_sf", C.c_void_p), ("b_q", C.c_void_p), ("b_sf", C.c_void_p), ("b2_q", C.c_void_p), ("b2_sf", C.c_void_p),
        ("residual", C.c_void_p), ("out", C.c_void_p),
        ("M", C.c_int), ("N", C.c_int), ("K", C.c_int), ("ldo", C.c_int), ("ldres", C.c_int), ("act", C.c_int), ("num_sms", C.c_int),
    ]


class GemmArgs(C.Structure):
    _fields_ = [
        ("a", C.c_void_p), ("b", C.c_void_p), ("b2", C.c_void_p),
        ("bias", C.c_void_p), ("bias2", C.c_void_p), ("residual", C.c_void_p), ("out", C.c_void_p),
        ("M", C.c_int), ("N", C.c_int), ("K", C.c_int),
        ("lda", C.c_int), ("ldb", C.c_int), ("ldo", C.c_int), ("ldres", C.c_int),
        ("b_mn_major", C.c_int), ("act", C.c_int), ("out_fp32", C.c_int), ("accumulate", C.c_int),
        ("n_push", C.c_int), ("push_out", C.c_void_p * PB_MAX_PEERS), ("push_flag", C.c_void_p * PB_MAX_PEERS),
        ("wait_flag", C.c_void_p), ("wait_per_epoch", C.c_uint64), ("epoch", C.c_void_p), ("error_flag", C.c_void_p),
        ("num_sms", C.c_int), ("block_n", C.c_int),
        ("push_done_flag", C.c_void_p * PB_MAX_PEERS), ("done_counter", C.c_void_p), ("push_rows_per_owner", C.c_int),
        ("grp", C.c_void_p), ("grp_cap", C.c_int), ("grp_experts", C.c_int),
    ]


class RopeKvArgs(C.Structure):
    _fields_ = [
        ("qkv", C.c_void_p), ("q_out", C.c_void_p), ("k_pool", C.c_void_p), ("v_pool", C.c_void_p),
        ("block_table", C.c_void_p), ("pos_ptr", C.c_void_p), ("cos", C.c_void_p), ("sin", C.c_void_p),
        ("qkv_bias", C.c_void_p),
        ("B", C.c_int), ("T", C.c_int), ("Hq", C.c_int), ("Hkv", C.c_int), ("D", C.c_int), ("page", C.c_int),
        ("max_pages", C.c_int), ("max_pos", C.c_int), ("interleaved_qkv", C.c_int),
        ("error_flag", C.c_void_p), ("num_pages", C.c_int),
    ]


class DecodeSpanArgs(C.Structure):
    _fields_ = [
        ("layers", C.c_void_p), ("n_layers", C.c_int),
        ("H", C.c_int), ("Hq", C.c_int), ("Hkv", C.c_int), ("D", C.c_int), ("I", C.c_int),
        ("eps", C.c_float), ("attn_scale", C.c_float),
        ("x_in", C.c_void_p), ("x_out", C.c_void_p), ("in_flag", C.c_void_p), ("in_per_epoch", C.c_uint64),
        ("block_table", C.c_void_p), ("max_pages", C.c_int), ("num_pages", C.c_int), ("pos_ptr", C.c_void_p),
        ("cos", C.c_void_p), ("sin", C.c_void_p), ("max_pos", C.c_int),
        ("qkv_ll", C.c_void_p), ("attp_ll", C.c_void_p), ("attn_ll", C.c_void_p), ("x_ll", C.c_void_p), ("act_ll", C.c_void_p),
        ("max_chunks", C.c_int),
        ("R", C.c_int), ("rank", C.c_int),
        ("oproj_push", C.c_void_p * PB_MAX_PEERS), ("mlp_push", C.c_void_p * PB_MAX_PEERS),
        ("oproj_in", C.c_void_p), ("mlp_in", C.c_void_p),
        ("epoch", C.c_void_p), ("error_flag", C.c_void_p), ("num_sms", C.c_int), ("prepare_only", C.c_int), ("timing", C.c_void_p),
        ("oproj_mc_push", C.c_void_p), ("mlp_mc_push", C.c_void_p), ("oproj_mc_sum", C.c_void_p), ("mlp_mc_sum", C.c_void_p), ("nvls_reduce", C.c_int),
    ]


class NormReduceGatherArgs(C.Structure):
    _fields_ = [
        ("x_res_in", C.c_void_p), ("x_res_out", C.c_void_p),
        ("n_parts", C.c_int), ("parts", C.c_void_p * PB_MAX_PEERS),
        ("norm_w", C.c_void_p), ("norm_b", C.c_void_p), ("eps", C.c_float), ("norm_kind", C.c_int),
        ("n_gather", C.c_int), ("gather_out", C.c_void_p * PB_MAX_PEERS), ("gather_flag", C.c_void_p * PB_MAX_PEERS),
        ("wait_flag", C.c_void_p), ("wait_per_epoch", C.c_uint64), ("epoch", C.c_void_p),
        ("done_counter", C.c_void_p), ("error_flag", C.c_void_p),
        ("rows", C.c_int), ("H", C.c_int), ("num_sms", C.c_int),
    ]


class AttnArgs(C.Structure):
    _fields_ = [
        ("q", C.c_void_p), ("k_pool", C.c_void_p), ("v_pool", C.c_void_p), ("block_table", C.c_void_p),
        ("pos_ptr", C.c_void_p), ("out", C.c_void_p), ("partial_o", C.c_void_p), ("partial_lse", C.c_void_p),
        ("alibi_slopes", C.c_void_p), ("scale", C.c_float),
        ("B", C.c_int), ("T", C.c_int), ("Hq", C.c_int), ("Hkv", C.c_int), ("D", C.c_int), ("page", C.c_int),
        ("max_pages", C.c_int), ("window", C.c_int), ("splits", C.c_int), ("pos_static", C.c_int), ("num_pages", C.c_int), ("impl", C.c_int), ("split_counter", C.c_void_p), ("lse_out", C.c_void_p),
    ]


class AttnBwdArgs(C.Structure):
    _fields_ = [
        ("q", C.c_void_p), ("k_pool", C.c_void_p), ("v_pool", C.c_void_p), ("block_table", C.c_void_p),
        ("out", C.c_void_p), ("d_out", C.c_void_p), ("lse", C.c_void_p), ("delta", C.c_void_p),
        ("dq", C.c_void_p), ("dk", C.c_void_p), ("dv", C.c_void_p), ("scale", C.c_float),
        ("B", C.c_int), ("T", C.c_int), ("Hq", C.c_int), ("Hkv", C.c_int), ("D", C.c_int), ("max_pages", C.c_int), ("num_pages", C.c_int),
    ]


def _declare(lib: C.CDLL) -> None:
    vp, ci, cl, cf = C.c_void_p, C.c_int, C.c_long, C.c_float
    lib.pb_attention_bwd.argtypes = [C.POINTER(AttnBwdArgs), vp]
    lib.pb_rmsnorm_bwd.argtypes = [vp, vp, vp, vp, vp, ci, ci, cf, vp]
    lib.pb_swiglu_bwd.argtypes = [vp, vp, vp, cl, vp]
    lib.pb_qkv_grad_merge.argtypes = [vp, vp, vp, vp, vp, vp, ci, ci, ci, ci, ci, ci, vp]
    for name in ("pb_attention_bwd", "pb_rmsnorm_bwd", "pb_swiglu_bwd", "pb_qkv_grad_merge"):
        getattr(lib, name).restype = ci
    lib.pb_linear_decode.argtypes = [C.POINTER(LinearDecodeArgs), vp]
    lib.pb_gemm_bf16.argtypes = [C.POINTER(GemmArgs), vp]
    lib.pb_linear_decode_mma.argtypes = [C.POINTER(LinearDecodeArgs), vp, vp, vp]
    lib.pb_linear_decode_mma.restype = ci
    lib.pb_linear_decode_fp8.argtypes = [C.POINTER(LinearFp8Args), vp]
    lib.pb_linear_decode_fp8.restype = ci
    lib.pb_dequant_mxfp8.argtypes = [vp, vp, vp, cl, vp]
    lib.pb_dequant_mxfp8.restype = ci
    lib.pb_gemm_tiles.argtypes = [ci, ci, ci, ci]
    lib.pb_norm.argtypes = [vp, vp, vp, vp, vp, vp, ci, ci, cf, ci, vp]
    lib.pb_swiglu.argtypes = [vp, vp, vp, cl, vp]
    lib.pb_add.argtypes = [vp, vp, vp, cl, vp]
    lib.pb_gelu.argtypes = [vp, vp, cl, ci, vp]
    lib.pb_gelu.restype = ci
    lib.pb_embedding.argtypes = [vp, vp, vp, ci, ci, vp]
    lib.pb_argmax.argtypes = [vp, ci, vp, ci, ci, vp]
    lib.pb_add_prompts.argtypes = [vp, vp, ci, ci, ci, ci, ci, vp, vp]
    lib.pb_bump_epoch.argtypes = [vp, vp]
    lib.pb_advance_pos.argtypes = [vp, ci, vp]
    lib.pb_rope_kv.argtypes = [C.POINTER(RopeKvArgs), vp]
    lib.pb_attention.argtypes = [C.POINTER(AttnArgs), vp]
    lib.pb_decode_span.argtypes = [C.POINTER(DecodeSpanArgs), vp]
    lib.pb_decode_span.restype = ci
    lib.pb_decode_span_smem.argtypes = [C.POINTER(DecodeSpanArgs), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.pb_decode_span_smem.restype = ci
    lib.pb_norm_reduce_gather.argtypes = [C.POINTER(NormReduceGatherArgs), vp]
    lib.pb_norm_reduce_gather.restype = ci
    lib.pb_kv_copy_pages.argtypes = [vp, vp, vp, ci, cl, cl, ci, vp]
    lib.pb_device_sm_count.argtypes = [ci]
    vpp = C.POINTER(C.c_void_p)
    u64 = C.c_uint64
    lib.pb_ipc_malloc.argtypes = [vpp, cl]
    lib.pb_ipc_free.argtypes = [vp]
    lib.pb_ipc_get_handle.argtypes = [vp, C.c_char_p]
    lib.pb_ipc_open_handle.argtypes = [C.c_char_p, vpp]
    lib.pb_ipc_close_handle.argtypes = [vp]
    lib.pb_ipc_handle_size.argtypes = []
    lib.pb_push_rows.argtypes = [vp, vpp, vpp, ci, cl, vp]
    lib.pb_wait_flag.argtypes = [vp, vp, u64, u64, vp, vp]
    lib.pb_argmax_val.argtypes = [vp, vp, vp, ci, ci, vp]
    lib.pb_argmax_exchange.argtypes = [vp, vp, cl, ci, ci, ci, vpp, vpp, ci, vp, vp, vp, vp, vp, vp]
    lib.pb_reduce_parts.argtypes = [vp, vpp, ci, vp, u64, vp, vp, cl, vp, vp]
    lib.pb_peer_copy.argtypes = [vp, vp, cl, ci, vp]
    lib.pb_pingpong.argtypes = [vp, vp, ci, ci, vp, vp, vp]
    for name in ("pb_ipc_malloc", "pb_ipc_free", "pb_ipc_get_handle", "pb_ipc_open_handle", "pb_ipc_close_handle", "pb_ipc_handle_size",
                 "pb_push_rows", "pb_wait_flag", "pb_argmax_val", "pb_argmax_exchange", "pb_reduce_parts", "pb_peer_copy", "pb_pingpong"):
        getattr(lib, name).restype = ci
    lib.pb_moe_router.argtypes = [vp, vp, vp, vp, vp, vp, ci, ci, ci, ci, cf, vp]
    lib.pb_moe_gemv.argtypes = [vp, vp, vp, vp, vp, ci, ci, ci, cl, ci, ci, vp]
    lib.pb_moe_combine.argtypes = [vp, vp, vp, vp, ci, ci, ci, vp]
    lib.pb_moe_plan.argtypes = [vp, ci, ci, vp, vp, ci, vp]
    lib.pb_moe_gather.argtypes = [vp, vp, vp, ci, ci, ci, vp]
    lib.pb_moe_combine_pos.argtypes = [vp, vp, vp, vp, vp, ci, ci, ci, vp]
    for name in ("pb_moe_router", "pb_moe_gemv", "pb_moe_combine", "pb_moe_plan", "pb_moe_gather", "pb_moe_combine_pos"):
        getattr(lib, name).restype = ci
    lib.pb_gemm_bf16_2cta.argtypes = [C.POINTER(GemmArgs), vp]
    lib.pb_gemm_bf16_2cta.restype = ci
    lib.pb_ll_reduce.argtypes = [vp, vpp, ci, vp, C.c_uint, C.c_uint, vp, cl, vp, vp]
    lib.pb_ll_push.argtypes = [vp, vpp, ci, vp, C.c_uint, C.c_uint, cl, vp]
    lib.pb_ll_reduce.restype = lib.pb_ll_push.restype = ci
    lib.pb_gemm_mxfp8.argtypes = [C.POINTER(GemmFp8Args), vp]
    lib.pb_quant_mxfp8.argtypes = [vp, vp, C.c_float, vp, vp, ci, ci, vp]
    lib.pb_gemm_mxfp8_2cta.argtypes = [C.POINTER(GemmFp8Args), vp]
    lib.pb_gemm_mxfp8.restype = lib.pb_quant_mxfp8.restype = lib.pb_gemm_mxfp8_2cta.restype = ci
    lib.pb_last_error.argtypes = []
    lib.pb_last_error.restype = C.c_char_p
    for name in ("pb_linear_decode", "pb_gemm_bf16", "pb_gemm_tiles", "pb_norm", "pb_swiglu", "pb_add", "pb_embedding",
                 "pb_argmax", "pb_add_prompts", "pb_bump_epoch", "pb_advance_pos", "pb_rope_kv", "pb_attention",
                 "pb_kv_copy_pages", "pb_device_sm_count", "pb_version"):
        getattr(lib, name).restype = ci


def _declare_rt(rt: C.CDLL) -> None:
    vp, ci, cl, cd = C.c_void_p, C.c_int, C.c_long, C.c_double
    ip = C.POINTER(C.c_int)
    rt.pb_kv_create.argtypes = [ci]; rt.pb_kv_create.restype = vp
    rt.pb_kv_destroy.argtypes = [vp]; rt.pb_kv_destroy.restype = None
    rt.pb_kv_alloc.argtypes = [vp, ci, ip]; rt.pb_kv_alloc.restype = ci
    rt.pb_kv_incref.argtypes = [vp, ip, ci]; rt.pb_kv_incref.restype = None
    rt.pb_kv_free.argtypes = [vp, ip, ci]; rt.pb_kv_free.restype = None
    rt.pb_kv_num_free.argtypes = [vp]; rt.pb_kv_num_free.restype = ci
    rt.pb_kv_refcount.argtypes = [vp, ci]; rt.pb_kv_refcount.restype = ci
    rt.pb_kv_reserve.argtypes = [vp, cl, cd]; rt.pb_kv_reserve.restype = ci
    rt.pb_kv_unreserve.argtypes = [vp, cl]; rt.pb_kv_unreserve.restype = None
    rt.pb_kv_reserved.argtypes = [vp]; rt.pb_kv_reserved.restype = cl
    rt.pb_tq_create.argtypes = []; rt.pb_tq_create.restype = vp
    rt.pb_tq_destroy.argtypes = [vp]; rt.pb_tq_destroy.restype = None
    rt.pb_tq_push.argtypes = [vp, cd, C.c_int64]; rt.pb_tq_push.restype = None
    rt.pb_tq_pop.argtypes = [vp, cd, C.POINTER(C.c_int64), C.POINTER(cd)]; rt.pb_tq_pop.restype = ci
    rt.pb_tq_size.argtypes = [vp]; rt.pb_tq_size.restype = ci
    rt.pb_tq_close.argtypes = [vp]; rt.pb_tq_close.restype = None
    rt.pb_st_open.argtypes = [C.c_char_p]; rt.pb_st_open.restype = vp
    rt.pb_st_close.argtypes = [vp]; rt.pb_st_close.restype = None
    rt.pb_st_num_tensors.argtypes = [vp]; rt.pb_st_num_tensors.restype = ci
    rt.pb_st_tensor_info.argtypes = [vp, ci, C.c_char_p, ci, C.c_char_p, ci, C.POINTER(C.c_int64),
                                     C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    rt.pb_st_tensor_info.restype = ci
    rt.pb_st_find.argtypes = [vp, C.c_char_p]; rt.pb_st_find.restype = ci
    rt.pb_st_data.argtypes = [vp]; rt.pb_st_data.restype = vp
    rt.pb_st_read.argtypes = [vp, ci, vp, C.c_int64, ci]; rt.pb_st_read.restype = ci
    rt.pb_st_error.argtypes = []; rt.pb_st_error.restype = C.c_char_p
    rt.pb_sock_send_frames.argtypes = [ci, C.POINTER(vp), C.POINTER(C.c_int64), ci, cd]; rt.pb_sock_send_frames.restype = ci
    rt.pb_sock_recv_exact.argtypes = [ci, vp, C.c_int64, cd]; rt.pb_sock_recv_exact.restype = ci


def _ensure_built() -> None:
    if not _build.is_current():
        if os.environ.get("PB_NO_BUILD") == "1" and _build.LIB_PATH.exists():
            return
        _build.build()


def lib() -> C.CDLL:
    """The CUDA kernel library. Raises if it cannot be built/loaded (never falls back silently)."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                _ensure_built()
                l = C.CDLL(str(_build.LIB_PATH))
                _declare(l)
                _lib = l
    return _lib


def rt() -> C.CDLL:
    """The host-only runtime library."""
    global _rt
    if _rt is None:
        with _lock:
            if _rt is None:
                _ensure_built()
                r = C.CDLL(str(_build.RT_LIB_PATH))
                _declare_rt(r)
                _rt = r
    return _rt


def available() -> bool:
    """True when the CUDA kernels can run here (a CUDA device is visible and the library loads)."""
    if not torch.cuda.is_available():
        return False
    lib()
    return True


launch_count = 0  # kernels of this library launched (directly) by this process; graph replays add their captured count


def check(code: int, what: str, launches: int = 1) -> None:
    global launch_count
    if code != 0:
        detail = ""
        try:
            detail = lib().pb_last_error().decode()
        except Exception:  # noqa: BLE001
            pass
        raise NativeError(f"{what} failed: {_ERRORS.get(code, code)}" + (f" [{detail}]" if detail else ""))
    launch_count += launches


def add_launches(n: int) -> None:
    global launch_count
    launch_count += n


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


_sm_count: dict[int, int] = {}


def sm_count(device: Optional[int] = None) -> int:
    d = torch.cuda.current_device() if device is None else device
    if d not in _sm_count:
        _sm_count[d] = torch.cuda.get_device_properties(d).multi_processor_count
    return _sm_count[d]
