"""Python entry points of the sm_100a kernels + their plain-PyTorch fp32 oracles.

Each ``op(...)`` launches the hand-written CUDA kernel on the current stream (CUDA tensors only; raises
if the native library is unavailable). Each ``op_ref(...)`` is the straightforward PyTorch definition of
the same math — used on CPU (plumbing tests, BASELINE config #1) and as the numerics oracle in
``tests/test_kernels_gpu.py``.
"""
from __future__ import annotations

import os

import ctypes as C
import math
from typing import Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

from petals_b200.ops import native
from petals_b200.ops.native import AttnArgs, GemmArgs, LinearDecodeArgs, RopeKvArgs, check, ptr, stream_ptr

PAGE = 64  # tokens per KV-cache page (== attention KV tile)

ACT_NONE, ACT_SWIGLU, ACT_GELU_TANH, ACT_GELU_ERF = 0, 1, 2, 3
NORM_NONE, NORM_RMS, NORM_LAYER = 0, 1, 2


def _bf16c(t: Optional[torch.Tensor], name: str) -> Optional[torch.Tensor]:
    if t is None:
        return None
    if t.dtype != torch.bfloat16 or not t.is_cuda:
        raise TypeError(f"{name}: expected a CUDA bfloat16 tensor, got {t.dtype} on {t.device}")
    if not t.is_contiguous():
        raise ValueError(f"{name}: tensor must be contiguous")
    return t


# ----------------------------------------------------------------------------------------------------
# decode-shape linear
# ----------------------------------------------------------------------------------------------------
def _linear_decode_args(
    x: torch.Tensor, w: torch.Tensor, *, w2: Optional[torch.Tensor] = None, bias: Optional[torch.Tensor] = None,
    bias2: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None,
    norm_weight: Optional[torch.Tensor] = None, norm_bias: Optional[torch.Tensor] = None, norm_kind: int = NORM_NONE,
    eps: float = 1e-6, act: int = ACT_NONE, out: Optional[torch.Tensor] = None, x_out: Optional[torch.Tensor] = None,
    parts: Sequence[torch.Tensor] = (), wait_flag: Optional[int] = None, wait_per_epoch: int = 0,
    epoch: Optional[int] = None, push_out: Sequence[int] = (), push_flag: Sequence[int] = (),
    error_flag: Optional[int] = None, fixed_grid: int = 0, store_local: bool = True, done_counter: Optional[int] = None,
    rope: Optional[dict] = None, ll_parts: Sequence[int] = (), ll_push: Sequence[int] = (), ll_tag: Tuple[int, int] = (1, 0),
):
    """Build the C argument block of one decode linear. Returns (args, result tensor, tensors that must outlive the launch)."""
    x = _bf16c(x, "x"); w = _bf16c(w, "w")
    M, K = x.reshape(-1, x.shape[-1]).shape
    N = w.shape[0]
    if w.shape[1] != K:
        raise ValueError(f"weight shape {tuple(w.shape)} incompatible with K={K}")
    if rope is not None:
        store_local = False
    if out is None and store_local:
        out = torch.empty(*x.shape[:-1], N, dtype=torch.bfloat16, device=x.device)
    keep = [x, w, _bf16c(w2, "w2"), _bf16c(bias, "bias"), _bf16c(bias2, "bias2"), _bf16c(residual, "residual"), _bf16c(norm_weight, "norm_weight"),
            _bf16c(norm_bias, "norm_bias")]
    a = LinearDecodeArgs()
    a.x, a.w, a.w2 = ptr(x), ptr(w), ptr(keep[2])
    a.bias, a.bias2 = ptr(keep[3]), ptr(keep[4])
    a.residual = ptr(keep[5])
    a.out = ptr(out) if store_local else None
    a.norm_w, a.norm_b = ptr(keep[6]), ptr(keep[7])
    a.x_out = ptr(x_out)
    a.eps, a.norm_kind, a.act = eps, norm_kind, act
    a.M, a.N, a.K = M, N, K
    a.n_parts = len(parts)
    for i, p in enumerate(parts):
        a.parts[i] = p if isinstance(p, int) else ptr(p)
    a.wait_flag, a.wait_per_epoch, a.epoch = wait_flag, wait_per_epoch, epoch
    a.n_push = len(push_out)
    for i, p in enumerate(push_out):
        a.push_out[i] = p
        a.push_flag[i] = push_flag[i] if i < len(push_flag) else None
    a.error_flag = error_flag
    a.num_sms = native.sm_count(x.device.index)
    a.fixed_grid = fixed_grid
    a.done_counter = done_counter
    a.n_ll_parts, a.n_ll_push = len(ll_parts), len(ll_push)
    for i, p in enumerate(ll_parts):
        a.ll_parts[i] = p
    for i, p in enumerate(ll_push):
        a.ll_push[i] = p
    a.ll_tag_mul, a.ll_tag_add = ll_tag
    if rope is not None:
        cos, sin, table = rope.get("cos"), rope.get("sin"), rope["block_table"]
        a.rope_q_out, a.rope_k_pool, a.rope_v_pool = ptr(rope["q_out"]), ptr(rope["k_pool"]), ptr(rope["v_pool"])
        a.rope_block_table, a.rope_pos_ptr = ptr(table), rope["pos_ptr"]
        a.rope_cos, a.rope_sin = ptr(cos), ptr(sin)
        a.rope_T, a.rope_Hq, a.rope_Hkv, a.rope_D = rope["T"], rope["Hq"], rope["Hkv"], rope["D"]
        a.rope_max_pages, a.rope_max_pos = table.shape[1], (cos.shape[0] if cos is not None else 0)
        a.rope_num_pages = rope["k_pool"].shape[0]
    return a, (rope["q_out"] if rope is not None else out), keep


def linear_decode(x: torch.Tensor, w: torch.Tensor, **kw) -> torch.Tensor:
    """``out[M,N] = epilogue(prologue(x)[M,K] @ w[N,K]^T)`` for M <= 8 tokens. See csrc/linear_decode.cu.

    Keyword arguments: ``w2`` (SwiGLU up projection, with ``act=ACT_SWIGLU``), ``bias``/``bias2``, ``residual``, ``norm_weight`` /
    ``norm_bias`` / ``norm_kind`` / ``eps`` (fused norm prologue), ``act``, ``out``, ``x_out``, ``parts`` (+ ``wait_flag`` /
    ``wait_per_epoch`` / ``epoch``: flag-protocol all-reduce tail), ``push_out`` / ``push_flag`` / ``done_counter`` (peer pushes),
    ``ll_parts`` / ``ll_push`` / ``ll_tag`` (LL-protocol all-reduce), ``error_flag``, ``fixed_grid``, ``store_local``.
    ``push_out`` / ``push_flag`` / ``wait_flag`` / ``epoch`` / ``ll_*`` are raw device addresses (peer-mapped buffers from
    :mod:`petals_b200.parallel.symmetric`).

    ``rope`` (QKV projection of Llama-style blocks) fuses RoPE + the paged KV append into the epilogue: a dict with ``q_out``
    [M, Hq*D], ``k_pool``/``v_pool`` (this block's page pools), ``block_table`` [B, max_pages] int32, ``pos_ptr`` (device address),
    ``cos``/``sin`` (fp32 tables or None), ``T``, ``Hq``, ``Hkv``, ``D``. Nothing is stored to ``out`` then; ``q_out`` is returned.
    """
    a, result, _keep = _linear_decode_args(x, w, **kw)
    if _SKINNY["on"] and _skinny_ok(a):
        scratch, counters = _skinny_buffers(x.device, a.N)
        check(native.lib().pb_linear_decode_mma(C.byref(a), ptr(scratch), ptr(counters), stream_ptr()), "linear_decode_mma")
        return result
    check(native.lib().pb_linear_decode(C.byref(a), stream_ptr()), "linear_decode")
    return result


# ---- 4..8 rows on the tensor cores (csrc/linear_decode_mma.cu) -------------------------------------------------------------------
# Measured on B200 at Llama-3-70B shapes (profiles/r1_kernel_bench_skinny.txt): the mma.sync kernel wins for every shape at
# M >= 5 (the FMA kernel drops to 34-52 % of HBM there) and for the large MLP matrices at M = 4 (86 vs 52 %); the FMA kernel
# keeps M <= 3 and the small matrices at M = 4 (its prologue is cheaper). PETALS_B200_SKINNY=0 disables the routing,
# =2 forces the tensor-core kernel wherever it is applicable.
_SKINNY = {"on": os.environ.get("PETALS_B200_SKINNY", "1") not in ("", "0"), "force": os.environ.get("PETALS_B200_SKINNY", "1") == "2", "bufs": {}}


def set_skinny_gemm(on: bool, force: bool = True) -> None:
    """Route plain decode linears with 2..8 rows (no peer traffic, no RoPE epilogue) to the mma.sync skinny-GEMM kernel.
    ``force`` bypasses the size heuristic (tests, benchmarks)."""
    _SKINNY["on"], _SKINNY["force"] = bool(on), bool(on and force)


def _skinny_ok(a) -> bool:
    if not _SKINNY["force"]:
        big = a.N * a.K * (2 if a.act == ACT_SWIGLU else 1) >= (128 << 20)
        if a.M < 4 or (a.M == 4 and not big):
            return False
    return (2 <= a.M <= 8 and a.N % 16 == 0 and a.K % 128 == 0 and a.n_parts == 0 and a.n_push == 0 and a.n_ll_parts == 0 and a.n_ll_push == 0
            and not a.wait_flag and not a.rope_q_out and not a.x_out and a.out and (a.norm_kind == 0 or 8 * (a.K * 2 + 8) <= 160 * 1024))


def _skinny_buffers(device: torch.device, N: int):
    """Zero-initialised reduction scratch [2, N, 8] fp32 and per-row-block arrival counters; every launch leaves them zero."""
    key = (device.type, device.index)
    have = _SKINNY["bufs"].get(key)
    if have is None or have[2] < N:
        cap = max(N, 32768)
        with torch.inference_mode(False):
            have = (torch.zeros(2 * cap * 8, dtype=torch.float32, device=device), torch.zeros(cap // 16, dtype=torch.int32, device=device), cap)
        _SKINNY.setdefault("keep", []).append(have)  # captured CUDA graphs may still hold the previous (smaller) buffers
        _SKINNY["bufs"][key] = have
    return have[0], have[1]


def linear_decode_fp8(x: torch.Tensor, w_q: torch.Tensor, w_scale: torch.Tensor, *, w2_q: Optional[torch.Tensor] = None,
                      w2_scale: Optional[torch.Tensor] = None, bias=None, bias2=None, residual=None, norm_weight=None, norm_bias=None,
                      norm_kind: int = NORM_NONE, eps: float = 1e-6, act: int = ACT_NONE, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Decode linear over MXFP8 weights (``ops.quant.quantize_mxfp8``): payload [N,K] float8_e4m3fn, scales [N,K/32] uint8."""
    from petals_b200.ops.native import LinearFp8Args

    x = _bf16c(x, "x")
    M, K = x.reshape(-1, x.shape[-1]).shape
    N = w_q.shape[0]
    if out is None:
        out = torch.empty(*x.shape[:-1], N, dtype=torch.bfloat16, device=x.device)
    a = LinearFp8Args()
    a.x, a.w, a.w_scale = ptr(x), ptr(w_q.contiguous()), ptr(w_scale.contiguous())
    a.w2, a.w2_scale = ptr(w2_q), ptr(w2_scale)
    a.bias, a.bias2, a.residual = ptr(_bf16c(bias, "bias")), ptr(_bf16c(bias2, "bias2")), ptr(_bf16c(residual, "residual"))
    a.out, a.norm_w, a.norm_b = ptr(out), ptr(_bf16c(norm_weight, "norm_weight")), ptr(_bf16c(norm_bias, "norm_bias"))
    a.eps, a.norm_kind, a.act, a.M, a.N, a.K = eps, norm_kind, act, M, N, K
    a.num_sms = native.sm_count(x.device.index)
    check(native.lib().pb_linear_decode_fp8(C.byref(a), stream_ptr()), "linear_decode_fp8")
    return out


def dequant_mxfp8(w_q: torch.Tensor, w_scale: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """MXFP8 -> bf16 on the device (feeds the tcgen05 GEMM at prefill time)."""
    if out is None:
        out = torch.empty(w_q.shape, dtype=torch.bfloat16, device=w_q.device)
    check(native.lib().pb_dequant_mxfp8(ptr(w_q), ptr(w_scale), ptr(out), w_q.numel(), stream_ptr()), "dequant_mxfp8")
    return out


def _act_ref(v: torch.Tensor, act: int) -> torch.Tensor:
    if act == ACT_GELU_TANH:
        return F.gelu(v, approximate="tanh")
    if act == ACT_GELU_ERF:
        return F.gelu(v)
    return v


def norm_ref(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor], kind: int, eps: float) -> torch.Tensor:
    xf = x.float()
    if kind == NORM_RMS:
        y = xf * torch.rsqrt(xf.pow(2).mean(-1, keepdim=True) + eps)
        return (y.to(x.dtype).float() * weight.float()).to(x.dtype)
    y = F.layer_norm(xf, (x.shape[-1],), weight.float(), None if bias is None else bias.float(), eps)
    return y.to(x.dtype)


def linear_ref(
    x: torch.Tensor, w: torch.Tensor, *, w2=None, bias=None, bias2=None, residual=None, norm_weight=None,
    norm_bias=None, norm_kind: int = NORM_NONE, eps: float = 1e-6, act: int = ACT_NONE,
) -> torch.Tensor:
    """Oracle for both linear_decode and gemm (same math, HF rounding points)."""
    dt = x.dtype
    if norm_kind != NORM_NONE:
        x = norm_ref(x, norm_weight, norm_bias, norm_kind, eps)
    y = F.linear(x.float(), w.float(), None if bias is None else bias.float())
    if act == ACT_SWIGLU:
        u = F.linear(x.float(), w2.float(), None if bias2 is None else bias2.float())
        y = (F.silu(y.to(dt).float()).to(dt).float() * u.to(dt).float())
    else:
        y = _act_ref(y, act)
    if residual is not None:
        y = y.to(dt).float() + residual.float()
    return y.to(dt)


# ----------------------------------------------------------------------------------------------------
# tcgen05 GEMM
# ----------------------------------------------------------------------------------------------------
def gemm(
    a_: torch.Tensor, b: torch.Tensor, *, b2: Optional[torch.Tensor] = None, bias: Optional[torch.Tensor] = None,
    bias2: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None, act: int = ACT_NONE,
    b_mn_major: bool = False, out: Optional[torch.Tensor] = None, out_fp32: bool = False, block_n: int = 0,
    wait_flag: Optional[int] = None, wait_per_epoch: int = 0, epoch: Optional[int] = None,
    push_out: Sequence[int] = (), push_flag: Sequence[int] = (), error_flag: Optional[int] = None,
    store_local: bool = True, push_done_flag: Sequence[int] = (), done_counter: Optional[int] = None,
    push_rows_per_owner: int = 0, grp: Optional[torch.Tensor] = None, grp_cap: int = 0, grp_experts: int = 0,
) -> torch.Tensor:
    """``out[M,N] = epilogue(a[M,K] @ op(b))`` on the tcgen05 tensor cores. See csrc/gemm_tcgen05.cu.

    ``b`` is ``[N,K]`` (nn.Linear weight) or, with ``b_mn_major=True``, ``[K,N]`` (weight used transposed).
    """
    a2 = _bf16c(a_, "a").reshape(-1, a_.shape[-1])
    b = _bf16c(b, "b")
    M, K = a2.shape
    if grp is not None:  # grouped: b is [E, N, K] (experts stacked along N), rows of `a` are grouped by expert (see moe_prefill)
        if b.dim() != 3 or b_mn_major or b.shape[0] != grp_experts or b.shape[2] != K:
            raise ValueError(f"grouped GEMM needs b [E, N, K]; got {tuple(b.shape)} for E={grp_experts}, K={K}")
        N = b.shape[1]
    else:
        N = b.shape[1] if b_mn_major else b.shape[0]
        if (b.shape[0] if b_mn_major else b.shape[1]) != K:
            raise ValueError(f"b shape {tuple(b.shape)} incompatible with K={K}")
    if out is None and store_local:
        out = torch.empty(*a_.shape[:-1], N, dtype=torch.float32 if out_fp32 else torch.bfloat16, device=a_.device)
    g = GemmArgs()
    g.a, g.b, g.b2 = ptr(a2), ptr(b), ptr(_bf16c(b2, "b2"))
    g.bias, g.bias2, g.residual = ptr(_bf16c(bias, "bias")), ptr(_bf16c(bias2, "bias2")), ptr(_bf16c(residual, "residual"))
    g.out = ptr(out) if store_local else None
    g.M, g.N, g.K = M, N, K
    g.lda = g.ldb = g.ldo = g.ldres = 0
    g.b_mn_major, g.act, g.out_fp32, g.accumulate = int(b_mn_major), act, int(out_fp32), 0
    g.n_push = len(push_out)
    for i, p in enumerate(push_out):
        g.push_out[i] = p
        g.push_flag[i] = push_flag[i] if i < len(push_flag) else None
        g.push_done_flag[i] = push_done_flag[i] if i < len(push_done_flag) else None
    g.done_counter = done_counter
    g.push_rows_per_owner = push_rows_per_owner
    g.wait_flag, g.wait_per_epoch, g.epoch, g.error_flag = wait_flag, wait_per_epoch, epoch, error_flag
    g.num_sms = native.sm_count(a_.device.index)
    g.block_n = block_n
    g.grp, g.grp_cap, g.grp_experts = ptr(grp), grp_cap, grp_experts
    if (_GEMM_2CTA and M >= 1024 and N >= 1024 and block_n == 0 and not push_out and grp is None and bias is None and bias2 is None and not out_fp32
            and (act == ACT_NONE or (act == ACT_SWIGLU and not b_mn_major)) and (not b_mn_major or (_GEMM_2CTA_MN and N % 64 == 0))):
        # large plain GEMMs: one 256 x 256 tile per SM pair (csrc/gemm_tcgen05_2cta.cu): each SM stages only half of the weight tile
        check(native.lib().pb_gemm_bf16_2cta(C.byref(g), stream_ptr()), "gemm_bf16_2cta")
        return out
    check(native.lib().pb_gemm_bf16(C.byref(g), stream_ptr()), "gemm_bf16")
    return out


# Measured on B200 (profiles/r2_gemm_2cta.txt): the bf16 pair kernel is 4-8 % faster on the 70B shapes and 12-19 % on smaller ones (default on);
# the block-scaled FP8 pair kernel is not faster than its 1-CTA twin (that kernel is bound by per-stage issue overhead, not operand traffic),
# so it stays opt-in (PETALS_B200_FP8_2CTA=1).
_GEMM_2CTA = os.environ.get("PETALS_B200_GEMM_2CTA", "1") != "0"
_FP8_2CTA = os.environ.get("PETALS_B200_FP8_2CTA", "0") != "0"
_GEMM_2CTA_MN = os.environ.get("PETALS_B200_GEMM_2CTA_MN", "1") != "0"  # MN-major B (the dgrad of rpc_backward) on the pair kernel


def set_gemm_2cta(on: bool, fp8: Optional[bool] = None, mn: Optional[bool] = None) -> None:
    """Route large plain GEMMs to the 2-CTA (cta_group::2) kernels (tests and tools/kernel_bench.py flip it). ``fp8``: the block-scaled
    FP8 pair kernel, ``mn``: MN-major B (dgrad) on the pair kernel — both have their own switches (default: follow ``on``)."""
    global _GEMM_2CTA, _FP8_2CTA, _GEMM_2CTA_MN
    _GEMM_2CTA = bool(on)
    _FP8_2CTA = bool(on if fp8 is None else fp8)
    _GEMM_2CTA_MN = bool(on if mn is None else mn)


# ----------------------------------------------------------------------------------------------------
# norms / elementwise
# ----------------------------------------------------------------------------------------------------
def norm(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor] = None, *, kind: int = NORM_RMS,
         eps: float = 1e-6, residual: Optional[torch.Tensor] = None, sum_out: Optional[torch.Tensor] = None,
         out: Optional[torch.Tensor] = None) -> torch.Tensor:
    x = _bf16c(x, "x")
    if out is None:
        out = torch.empty_like(x)
    rows, cols = x.numel() // x.shape[-1], x.shape[-1]
    check(native.lib().pb_norm(ptr(x), ptr(_bf16c(residual, "residual")), ptr(_bf16c(weight, "weight")),
                               ptr(_bf16c(bias, "bias")), ptr(out), ptr(sum_out), rows, cols, eps, kind, stream_ptr()),
          "norm")
    return out


def norm_reduce_gather(x_res_in: Optional[torch.Tensor], x_res_out: Optional[torch.Tensor], *, rows: int, H: int, parts: Sequence[int] = (),
                       norm_weight: Optional[torch.Tensor] = None, norm_bias: Optional[torch.Tensor] = None, norm_kind: int = NORM_NONE,
                       eps: float = 1e-6, gather_out: Sequence[int] = (), gather_flag: Sequence[int] = (), wait_flag: Optional[int] = None,
                       wait_per_epoch: int = 0, epoch: Optional[int] = None, done_counter: Optional[int] = None,
                       error_flag: Optional[int] = None, device_index: Optional[int] = None) -> None:
    """Owner-side tail of the fused reduce-scatter (sum of the peers' GEMM-epilogue partial rows + residual slice), norm, and
    all-gather of the normalised rows into every peer's activation buffer. ``parts``/``gather_out``/``gather_flag`` are raw
    (symmetric-heap) addresses. See csrc/seq_parallel.cu."""
    a = native.NormReduceGatherArgs()
    a.x_res_in, a.x_res_out = ptr(x_res_in), ptr(x_res_out)
    a.n_parts = len(parts)
    for i, p_ in enumerate(parts):
        a.parts[i] = p_
    a.norm_w, a.norm_b, a.eps, a.norm_kind = ptr(_bf16c(norm_weight, "norm_weight")), ptr(_bf16c(norm_bias, "norm_bias")), eps, norm_kind
    a.n_gather = len(gather_out)
    for i, p_ in enumerate(gather_out):
        a.gather_out[i] = p_
        a.gather_flag[i] = gather_flag[i] if i < len(gather_flag) else None
    a.wait_flag, a.wait_per_epoch, a.epoch = wait_flag, wait_per_epoch, epoch
    a.done_counter, a.error_flag = done_counter, error_flag
    a.rows, a.H = rows, H
    a.num_sms = native.sm_count(device_index if device_index is not None else torch.cuda.current_device())
    check(native.lib().pb_norm_reduce_gather(C.byref(a), stream_ptr()), "norm_reduce_gather")


def swiglu(gate: torch.Tensor, up: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    if out is None:
        out = torch.empty_like(gate)
    check(native.lib().pb_swiglu(ptr(_bf16c(gate, "gate")), ptr(_bf16c(up, "up")), ptr(out), gate.numel(), stream_ptr()), "swiglu")
    return out


def activation(x: torch.Tensor, act: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """The stand-alone form of a fused epilogue activation (``ACT_GELU_TANH`` / ``ACT_GELU_ERF``; ``ACT_NONE`` copies)."""
    out = torch.empty_like(x) if out is None else out
    if act == ACT_NONE:
        return out.copy_(x)
    if act not in (ACT_GELU_TANH, ACT_GELU_ERF):
        raise ValueError(f"activation {act} has no stand-alone kernel")
    check(native.lib().pb_gelu(ptr(_bf16c(x, "x")), ptr(out), x.numel(), int(act == ACT_GELU_ERF), stream_ptr()), "gelu")
    return out


def add(a: torch.Tensor, b: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    if out is None:
        out = torch.empty_like(a)
    check(native.lib().pb_add(ptr(_bf16c(a, "a")), ptr(_bf16c(b, "b")), ptr(out), a.numel(), stream_ptr()), "add")
    return out


def embedding(table: torch.Tensor, ids: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    ids = ids.contiguous()
    if ids.dtype != torch.int64:
        ids = ids.long()
    if out is None:
        out = torch.empty(*ids.shape, table.shape[1], dtype=torch.bfloat16, device=table.device)
    check(native.lib().pb_embedding(ptr(_bf16c(table, "table")), ptr(ids), ptr(out), ids.numel(), table.shape[1], stream_ptr()), "embedding")
    return out


def argmax(logits: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    rows, vocab = logits.numel() // logits.shape[-1], logits.shape[-1]
    if out is None:
        out = torch.empty(logits.shape[:-1], dtype=torch.int64, device=logits.device)
    check(native.lib().pb_argmax(ptr(logits.contiguous()), int(logits.dtype == torch.float32), ptr(out), rows, vocab, stream_ptr()), "argmax")
    return out


def add_prompts(hidden: torch.Tensor, prompts: torch.Tensor, pos_ptr: Optional[int] = None) -> torch.Tensor:
    """In place: hidden[:, :P] += prompts (deep-prompt injection, reference backend.py:231-233)."""
    B, T, H = hidden.shape
    Bp, P, _ = prompts.shape
    check(native.lib().pb_add_prompts(ptr(_bf16c(hidden, "hidden")), ptr(_bf16c(prompts, "prompts")), B, T, H, Bp, P, pos_ptr, stream_ptr()), "add_prompts")
    return hidden


# ----------------------------------------------------------------------------------------------------
# RoPE + paged KV, attention
# ----------------------------------------------------------------------------------------------------
def rope_tables(head_dim: int, max_pos: int, theta: float = 10000.0, scaling: Optional[dict] = None,
                device="cpu") -> tuple[torch.Tensor, torch.Tensor]:
    """fp32 cos/sin tables [max_pos, D/2] for the position-independent ``rope_scaling`` types: ``linear``, ``llama3`` and ``yarn``
    (YaRN, arXiv:2309.00071: per-frequency blend of interpolation and extrapolation + an attention temperature folded into the
    tables). Types that change with the running sequence length (``dynamic``, ``longrope``) are rejected instead of ignored."""
    inv = 1.0 / (theta ** (torch.arange(0, head_dim, 2, dtype=torch.float32) / head_dim))
    amplitude = 1.0
    if scaling:
        kind = scaling.get("rope_type", scaling.get("type"))
        factor = float(scaling.get("factor", 1.0))
        if kind in (None, "default"):
            pass
        elif kind == "yarn":
            orig = float(scaling.get("original_max_position_embeddings") or max(1, round(max_pos / factor)))
            beta_fast, beta_slow = float(scaling.get("beta_fast") or 32.0), float(scaling.get("beta_slow") or 1.0)

            def temperature(scale: float, m: float = 1.0) -> float:
                return 1.0 if scale <= 1 else 0.1 * m * math.log(scale) + 1.0

            amplitude = scaling.get("attention_factor")
            if amplitude is None:
                m, m_all = scaling.get("mscale"), scaling.get("mscale_all_dim")
                amplitude = temperature(factor, m) / temperature(factor, m_all) if m and m_all else temperature(factor)

            def dim_of_rotations(n_rot: float) -> float:  # the dimension whose wavelength makes n_rot turns over the original context
                return head_dim * math.log(orig / (n_rot * 2 * math.pi)) / (2 * math.log(theta))

            low, high = dim_of_rotations(beta_fast), dim_of_rotations(beta_slow)
            if scaling.get("truncate", True):
                low, high = math.floor(low), math.ceil(high)
            low, high = max(low, 0), min(high, head_dim - 1)
            if low == high:
                high += 0.001
            ramp = ((torch.arange(head_dim // 2, dtype=torch.float32) - low) / (high - low)).clamp_(0, 1)
            inv = (inv / factor) * ramp + inv * (1 - ramp)  # high frequencies extrapolate, low frequencies interpolate
        elif kind == "llama3":
            lo, hi = float(scaling.get("low_freq_factor", 1.0)), float(scaling.get("high_freq_factor", 4.0))
            old = float(scaling.get("original_max_position_embeddings", 8192))
            wavelen = 2 * math.pi / inv
            smooth = ((old / wavelen) - lo) / (hi - lo)
            scaled = torch.where(wavelen > old / lo, inv / factor, inv)
            mid = (wavelen <= old / lo) & (wavelen >= old / hi)
            inv = torch.where(mid, (1 - smooth) * inv / factor + smooth * inv, scaled)
        elif kind == "linear":
            inv = inv / factor
        else:
            raise NotImplementedError(f"rope_scaling type {kind!r} is not supported (supported: default, linear, llama3, yarn)")
    ang = torch.arange(max_pos, dtype=torch.float32)[:, None] * inv[None, :]
    return (ang.cos() * float(amplitude)).to(device).contiguous(), (ang.sin() * float(amplitude)).to(device).contiguous()


def rope_kv_append(qkv: torch.Tensor, q_out: torch.Tensor, k_pool: torch.Tensor, v_pool: torch.Tensor,
                   block_table: torch.Tensor, pos_ptr: int, cos: Optional[torch.Tensor], sin: Optional[torch.Tensor],
                   *, B: int, T: int, Hq: int, Hkv: int, D: int, qkv_bias: Optional[torch.Tensor] = None,
                   interleaved: bool = False, error_flag: Optional[int] = None) -> None:
    a = RopeKvArgs()
    a.qkv, a.q_out, a.k_pool, a.v_pool = ptr(qkv), ptr(q_out), ptr(k_pool), ptr(v_pool)
    a.block_table, a.pos_ptr = ptr(block_table), pos_ptr
    a.cos, a.sin, a.qkv_bias = ptr(cos), ptr(sin), ptr(qkv_bias)
    a.B, a.T, a.Hq, a.Hkv, a.D, a.page = B, T, Hq, Hkv, D, PAGE
    a.max_pages, a.num_pages = block_table.shape[1], k_pool.shape[0]
    a.max_pos = cos.shape[0] if cos is not None else 0
    a.interleaved_qkv = int(interleaved)
    a.error_flag = error_flag
    check(native.lib().pb_rope_kv(C.byref(a), stream_ptr()), "rope_kv")


def paged_attention(q: torch.Tensor, k_pool: torch.Tensor, v_pool: torch.Tensor, block_table: torch.Tensor,
                    pos_ptr: Optional[int], out: torch.Tensor, *, B: int, T: int, Hq: int, Hkv: int, D: int,
                    scale: float, splits: int = 1, partial_o: Optional[torch.Tensor] = None,
                    partial_lse: Optional[torch.Tensor] = None, alibi_slopes: Optional[torch.Tensor] = None,
                    window: int = 0, pos_static: int = 0, impl: int = 0, split_counter: Optional[torch.Tensor] = None,
                    lse_out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Flash attention over the paged cache. ``impl``: 0 = auto (tcgen05 kernel for prefill-sized tiles, split-KV mma.sync kernel for
    decode), 1 / 2 force the mma.sync / tcgen05 kernel. ``lse_out`` (fp32 [B*T*Hq], training forward): the log2-domain
    log-sum-exp of every query row, written by the mma.sync kernel (forces ``impl = 1``, needs ``splits == 1``)."""
    if lse_out is not None:
        if splits != 1:
            raise ValueError("lse_out needs splits == 1")
        impl = 1
    a = AttnArgs()
    a.q, a.k_pool, a.v_pool, a.block_table, a.pos_ptr = ptr(q), ptr(k_pool), ptr(v_pool), ptr(block_table), pos_ptr
    a.out, a.partial_o, a.partial_lse, a.alibi_slopes = ptr(out), ptr(partial_o), ptr(partial_lse), ptr(alibi_slopes)
    a.scale = scale
    a.B, a.T, a.Hq, a.Hkv, a.D, a.page = B, T, Hq, Hkv, D, PAGE
    a.max_pages, a.window, a.splits, a.pos_static = block_table.shape[1], window, splits, pos_static
    a.num_pages, a.impl, a.split_counter, a.lse_out = k_pool.shape[0], impl, ptr(split_counter), ptr(lse_out)
    check(native.lib().pb_attention(C.byref(a), stream_ptr()), "attention", 2 if (splits > 1 and split_counter is None) else 1)
    return out


def attention_bwd(q: torch.Tensor, k_pool: torch.Tensor, v_pool: torch.Tensor, block_table: torch.Tensor, out: torch.Tensor, d_out: torch.Tensor,
                  lse: torch.Tensor, *, B: int, T: int, Hq: int, Hkv: int, D: int, scale: float, dq: Optional[torch.Tensor] = None,
                  dk: Optional[torch.Tensor] = None, dv: Optional[torch.Tensor] = None, delta: Optional[torch.Tensor] = None):
    """Backward of the causal attention of a cache-less forward (positions 0..T-1 per sequence): returns (dq [M, Hq*D],
    dk [M, Hkv*D], dv [M, Hkv*D]) given the rotated queries, the paged keys/values, the forward output and its ``lse_out``."""
    from petals_b200.ops.native import AttnBwdArgs

    M = B * T
    dev = q.device
    dq = torch.empty(M, Hq * D, dtype=torch.bfloat16, device=dev) if dq is None else dq
    dk = torch.empty(M, Hkv * D, dtype=torch.bfloat16, device=dev) if dk is None else dk
    dv = torch.empty(M, Hkv * D, dtype=torch.bfloat16, device=dev) if dv is None else dv
    delta = torch.empty(M * Hq, dtype=torch.float32, device=dev) if delta is None else delta
    a = AttnBwdArgs()
    a.q, a.k_pool, a.v_pool, a.block_table = ptr(_bf16c(q, "q")), ptr(k_pool), ptr(v_pool), ptr(block_table)
    a.out, a.d_out, a.lse, a.delta = ptr(_bf16c(out, "out")), ptr(_bf16c(d_out, "d_out")), ptr(lse), ptr(delta)
    a.dq, a.dk, a.dv, a.scale = ptr(dq), ptr(dk), ptr(dv), scale
    a.B, a.T, a.Hq, a.Hkv, a.D, a.max_pages, a.num_pages = B, T, Hq, Hkv, D, block_table.shape[1], k_pool.shape[0]
    check(native.lib().pb_attention_bwd(C.byref(a), stream_ptr()), "attention_bwd", 3)
    return dq, dk, dv


def rmsnorm_bwd(dy: torch.Tensor, x: torch.Tensor, weight: torch.Tensor, eps: float, d_res: Optional[torch.Tensor] = None,
                out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``d_res + d/dx [rmsnorm(x) * weight] . dy`` for rows [M, H] (``d_res``: gradient arriving over the residual connection)."""
    M, H = x.shape
    out = torch.empty_like(x) if out is None else out
    check(native.lib().pb_rmsnorm_bwd(ptr(_bf16c(dy, "dy")), ptr(_bf16c(x, "x")), ptr(_bf16c(weight, "weight")), ptr(_bf16c(d_res, "d_res")),
                                      ptr(out), M, H, eps, stream_ptr()), "rmsnorm_bwd")
    return out


def swiglu_bwd_(d_act: torch.Tensor, g: torch.Tensor, u: torch.Tensor) -> None:
    """In place: ``g <- d(act)/d(g) * d_act``, ``u <- d(act)/d(u) * d_act`` for ``act = silu(g) * u``."""
    check(native.lib().pb_swiglu_bwd(ptr(_bf16c(d_act, "d_act")), ptr(_bf16c(g, "g")), ptr(_bf16c(u, "u")), g.numel(), stream_ptr()), "swiglu_bwd")


def qkv_grad_merge(dq: torch.Tensor, dk: torch.Tensor, dv: torch.Tensor, cos, sin, *, T: int, Hq: int, Hkv: int, D: int,
                   out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """[R^T dq | R^T dk | dv] in the fused QKV projection's column layout (the backward of RoPE + the q/k/v split)."""
    M = dq.shape[0]
    out = torch.empty(M, (Hq + 2 * Hkv) * D, dtype=torch.bfloat16, device=dq.device) if out is None else out
    check(native.lib().pb_qkv_grad_merge(ptr(dq), ptr(dk), ptr(dv), ptr(cos), ptr(sin), ptr(out), M, T, Hq, Hkv, D,
                                         cos.shape[0] if cos is not None else 0, stream_ptr()), "qkv_grad_merge")
    return out


def rope_ref(x: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor) -> torch.Tensor:
    """HF rotate_half RoPE with HF's rounding (cos/sin cast to x.dtype). x: [..., T, H, D]; cos/sin: [T, D/2]."""
    dt = x.dtype
    c = torch.cat([cos, cos], -1).to(dt)[:, None, :]
    s = torch.cat([sin, sin], -1).to(dt)[:, None, :]
    half = x.shape[-1] // 2
    rot = torch.cat([-x[..., half:], x[..., :half]], -1)
    return (x * c) + (rot * s)


def attention_ref(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, *, pos0: int, scale: float,
                  alibi_slopes: Optional[torch.Tensor] = None, window: int = 0) -> torch.Tensor:
    """fp32 oracle. q: [B,T,Hq,D]; k,v: [B,L,Hkv,D] with L = pos0 + T. Returns [B,T,Hq,D] in q.dtype."""
    B, T, Hq, D = q.shape
    L, Hkv = k.shape[1], k.shape[2]
    G = Hq // Hkv
    kf = k.float().repeat_interleave(G, dim=2)
    vf = v.float().repeat_interleave(G, dim=2)
    s = torch.einsum("bthd,blhd->bhtl", q.float(), kf) * scale
    qpos = pos0 + torch.arange(T, device=q.device)[:, None]
    kpos = torch.arange(L, device=q.device)[None, :]
    if alibi_slopes is not None:
        s = s + alibi_slopes.float().view(1, Hq, 1, 1) * (kpos - qpos).float()[None, None]
    ok = kpos <= qpos
    if window > 0:
        ok = ok & (kpos > qpos - window)
    s = s.masked_fill(~ok[None, None], float("-inf"))
    p = torch.softmax(s, dim=-1)
    return torch.einsum("bhtl,blhd->bthd", p, vf).to(q.dtype)


# ----------------------------------------------------------------------------------------------------
# sparse MoE (decode)
# ----------------------------------------------------------------------------------------------------
def moe_decode(h: torch.Tensor, norm_w: torch.Tensor, router: torch.Tensor, we_gate: torch.Tensor, we_up: torch.Tensor, we_down: torch.Tensor,
               *, top_k: int, eps: float, out: torch.Tensor, bufs: Optional[dict] = None, add_residual: bool = True) -> torch.Tensor:
    """out = h + MoE(RMSNorm(h)) for M <= 8 rows without any host synchronisation (csrc/moe.cu). ``add_residual=False``: out = MoE(...)
    alone — a tensor-parallel rank's partial sum over its slice of every expert's FFN columns (the residual joins in the all-reduce)."""
    M, H = h.shape
    E, I, _ = we_gate.shape
    bufs = bufs if bufs is not None else {}

    def buf(name, shape, dtype):  # keyed by shape, never replaced: captured CUDA graphs hold these addresses
        key = (name, tuple(shape))
        t = bufs.get(key)
        if t is None:
            with torch.inference_mode(False):
                t = torch.empty(shape, dtype=dtype, device=h.device)
            bufs[key] = t
        return t

    xn = buf("moe_xn", (M, H), torch.bfloat16)
    topi = buf("moe_topi", (M * top_k,), torch.int32)
    topw = buf("moe_topw", (M * top_k,), torch.float32)
    act = buf("moe_act", (M * top_k, I), torch.bfloat16)
    y = buf("moe_y", (M * top_k, H), torch.bfloat16)
    lib, st = native.lib(), stream_ptr()
    sms = native.sm_count(h.device.index)
    check(lib.pb_moe_router(ptr(h), ptr(norm_w), ptr(router), ptr(xn), ptr(topi), ptr(topw), M, H, E, top_k, eps, st), "moe_router")
    check(lib.pb_moe_gemv(ptr(xn), ptr(we_gate), ptr(we_up), ptr(topi), ptr(act), M * top_k, I, H, I * H, top_k, sms, st), "moe_gemv(gate/up)")
    check(lib.pb_moe_gemv(ptr(act), ptr(we_down), None, ptr(topi), ptr(y), M * top_k, H, I, H * I, 1, sms, st), "moe_gemv(down)")
    check(lib.pb_moe_combine(ptr(y), ptr(topw), ptr(h) if add_residual else None, ptr(out), M, H, top_k, st), "moe_combine")
    return out


def ll_reduce(x: torch.Tensor, parts: Sequence[int], tag: Tuple[int, int], epoch: int, out: torch.Tensor, error_flag: int = 0) -> torch.Tensor:
    """``out = x + sum_r parts[r]`` where every part is a buffer of LL {2 x bf16, tag} units (addresses) written by ``ll_push`` /
    a GEMV epilogue of source rank r; tag = epoch * tag[0] + tag[1] (csrc/ll_collectives.cu)."""
    arr = (C.c_void_p * len(parts))(*parts)
    check(native.lib().pb_ll_reduce(ptr(x), arr, len(parts), epoch, tag[0], tag[1], ptr(out), x.numel(), error_flag or None, stream_ptr()), "ll_reduce")
    return out


def ll_push(x: torch.Tensor, dst: Sequence[int], tag: Tuple[int, int], epoch: int) -> None:
    """Store ``x`` as LL units into ``dst`` (one address per destination rank: this rank's slot over there)."""
    arr = (C.c_void_p * len(dst))(*dst)
    check(native.lib().pb_ll_push(ptr(x), arr, len(dst), epoch, tag[0], tag[1], x.numel(), stream_ptr()), "ll_push")


def quant_mxfp8(x: torch.Tensor, norm_weight: Optional[torch.Tensor] = None, eps: float = 0.0, *, q: Optional[torch.Tensor] = None,
                sf: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Rows of ``x`` [M, K] (bf16; with ``norm_weight``: RMSNorm(x) * weight first) -> MXFP8: E4M3 payload [M, K] (uint8 storage) and the
    UE8M0 scales in the tensor cores' block layout (ops/quant.py:pack_scales)."""
    x = _bf16c(x, "x")
    M, K = x.shape
    if q is None:
        q = torch.empty(M, K, dtype=torch.uint8, device=x.device)
    if sf is None:
        sf = torch.zeros((K // 128) * ((M + 127) // 128) * 512, dtype=torch.uint8, device=x.device)
    check(native.lib().pb_quant_mxfp8(ptr(x), ptr(_bf16c(norm_weight, "norm_weight")), eps, ptr(q), ptr(sf), M, K, stream_ptr()), "quant_mxfp8")
    return q, sf


def gemm_mxfp8(a_q: torch.Tensor, a_sf: torch.Tensor, b_q: torch.Tensor, b_sf: torch.Tensor, *, b2_q: Optional[torch.Tensor] = None,
               b2_sf: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``out = [residual +] A B^T`` with both operands MXFP8 and packed scales (``tcgen05.mma.kind::mxf8f6f4.block_scale``); with ``b2``
    the epilogue emits ``silu(A B^T) * (A B2^T)``. A [M, K], B [N, K] (nn.Linear layout), out bf16 [M, N]."""
    M, K = a_q.shape
    N = b_q.shape[0]
    if b_q.shape[1] != K or K % 128:
        raise ValueError(f"gemm_mxfp8: A {tuple(a_q.shape)} x B {tuple(b_q.shape)} (K must match and be a multiple of 128)")
    if out is None:
        out = torch.empty(M, N, dtype=torch.bfloat16, device=a_q.device)
    g = native.GemmFp8Args()
    g.a_q, g.a_sf, g.b_q, g.b_sf, g.b2_q, g.b2_sf = ptr(a_q), ptr(a_sf), ptr(b_q), ptr(b_sf), ptr(b2_q), ptr(b2_sf)
    g.residual, g.out = ptr(_bf16c(residual, "residual")), ptr(out)
    g.M, g.N, g.K, g.ldo, g.ldres = M, N, K, out.stride(0), (residual.stride(0) if residual is not None else 0)
    g.act = 1 if b2_q is not None else 0
    g.num_sms = native.sm_count(a_q.device.index)
    if _FP8_2CTA and M >= 1024 and N >= 1024:
        check(native.lib().pb_gemm_mxfp8_2cta(C.byref(g), stream_ptr()), "gemm_mxfp8_2cta")
    else:
        check(native.lib().pb_gemm_mxfp8(C.byref(g), stream_ptr()), "gemm_mxfp8")
    return out


def moe_prefill(h: torch.Tensor, norm_w: torch.Tensor, router: torch.Tensor, we_gate: torch.Tensor, we_up: torch.Tensor, we_down: torch.Tensor,
                *, top_k: int, eps: float, out: torch.Tensor, bufs: Optional[dict] = None, add_residual: bool = True) -> torch.Tensor:
    """out = h + MoE(RMSNorm(h)) for any number of rows (``norm_w=None``: ``h`` is normalised already; ``add_residual=False``: the MoE
    term alone — both for tensor-parallel ranks, which hold a slice of every expert's FFN columns), with NO host synchronisation: router kernel -> routing plan on the device
    (destination row of every (token, expert) pair in expert-major order + the tile table of the grouped GEMM) -> gather -> grouped
    tcgen05 GEMM gate/up with the SwiGLU epilogue -> grouped GEMM down -> weighted combine + residual. Reference (a Python loop over
    the experts with masks and index_add): HF MixtralSparseMoeBlock wrapped at src/petals/models/mixtral/block.py:13-19."""
    M, H = h.shape
    E, I, _ = we_gate.shape
    pairs = M * top_k
    cap = pairs // 128 + E + 1  # 128-row tiles over all groups, at most one ragged tail per expert
    bufs = bufs if bufs is not None else {}

    def buf(name, n, dtype):  # grow-only
        t = bufs.get(name)
        if t is None or t.numel() < n or t.dtype != dtype:
            with torch.inference_mode(False):
                t = torch.empty(n, dtype=dtype, device=h.device)
            bufs[name] = t
        return t[:n]

    xn = buf("moep_xn", M * H, torch.bfloat16).view(M, H) if norm_w is not None else _bf16c(h, "h")
    topi, topw = buf("moep_topi", pairs, torch.int32), buf("moep_topw", pairs, torch.float32)
    pos, table = buf("moep_pos", pairs, torch.int32), buf("moep_table", 1 + 3 * cap, torch.int32)
    gathered = buf("moep_gathered", pairs * H, torch.bfloat16).view(pairs, H)
    act = buf("moep_act", pairs * I, torch.bfloat16).view(pairs, I)
    y = buf("moep_y", pairs * H, torch.bfloat16).view(pairs, H)
    lib, st = native.lib(), stream_ptr()
    check(lib.pb_moe_router(ptr(h), ptr(norm_w), ptr(router), ptr(xn) if norm_w is not None else None, ptr(topi), ptr(topw), M, H, E, top_k, eps, st), "moe_router")
    check(lib.pb_moe_plan(ptr(topi), pairs, E, ptr(pos), ptr(table), cap, st), "moe_plan")
    check(lib.pb_moe_gather(ptr(xn), ptr(pos), ptr(gathered), pairs, H, top_k, st), "moe_gather")
    gemm(gathered, we_gate, b2=we_up, act=ACT_SWIGLU, out=act, grp=table, grp_cap=cap, grp_experts=E)
    gemm(act, we_down, out=y, grp=table, grp_cap=cap, grp_experts=E)
    check(lib.pb_moe_combine_pos(ptr(y), ptr(topw), ptr(pos), ptr(h) if add_residual else None, ptr(out), M, H, top_k, st), "moe_combine_pos")
    return out


class DecodeSpanPlan:
    """Everything ``csrc/decode_span.cu`` needs to run one token through a span of Llama-style blocks in ONE persistent launch:
    the device table of per-block pointers, the tagged data-flow buffers and the step counter.

    ``layers``: per block a dict with ``wqkv wo w_gate w_up w_down ln1_w ln2_w`` (this rank's shards) and ``k_pool v_pool``
    ([num_pages, Hkv, PAGE, D]). ``R``/``rank`` + ``oproj`` / ``mlp`` = (push addresses per rank, local receive address) place the
    two all-reduce buffers in a symmetric heap for tensor parallelism; by default (one GPU) they are plain local tensors."""

    def __init__(self, layers: Sequence[dict], *, H: int, Hq: int, Hkv: int, D: int, I: int, eps: float, attn_scale: float, max_chunks: int,
                 device, R: int = 1, rank: int = 0, oproj: Optional[tuple] = None, mlp: Optional[tuple] = None, epoch: Optional[torch.Tensor] = None,
                 error_flag: Optional[torch.Tensor] = None, nvls: Optional[dict] = None):
        """``nvls`` (NVSwitch multicast, tensor parallel only): ``{"mode": "st" | "reduce", "oproj": addr, "mlp": addr}`` with the
        multicast addresses of slot [rank] ("st": one ``multimem.st`` instead of R peer stores) or of slot [0] ("reduce": partials
        stay in the own heap, the slice owners ``multimem.ld_reduce`` them; ``oproj`` / ``mlp`` push lists then hold only this rank's
        slot [0])."""
        self.nvls = nvls or {}
        self.device = torch.device(device)
        self.H, self.Hq, self.Hkv, self.D, self.I, self.eps, self.attn_scale = H, Hq, Hkv, D, I, eps, attn_scale
        self.R, self.rank, self.max_chunks = R, rank, max_chunks
        names = ("wqkv", "wo", "w_gate", "w_up", "w_down", "ln1_w", "ln2_w", "k_pool", "v_pool")
        self._keep = [[_bf16c(l[n], n) for n in names] for l in layers]
        with torch.inference_mode(False):
            self.table = torch.tensor([[t.data_ptr() for t in row] for row in self._keep], dtype=torch.int64, device=self.device)
            z = lambda n: torch.zeros(n, 2, dtype=torch.int32, device=self.device)  # n LL units {payload, tag}; tag 0 is never valid
            self.qkv_ll, self.attn_ll, self.x_ll, self.act_ll = z((Hq + 2 * Hkv) * D // 2), z(Hq * D // 2), z(H // 2), z(I // 2)
            self.attp_ll = z(Hq * max_chunks * (D + 2))
            self.epoch = epoch if epoch is not None else torch.zeros(1, dtype=torch.int64, device=self.device)
            self.err = error_flag if error_flag is not None else torch.zeros(1, dtype=torch.int32, device=self.device)
            if oproj is None:
                self._oproj, self._mlp = z(R * H // 2), z(R * H // 2)
                oproj = ([self._oproj.data_ptr()], self._oproj.data_ptr())
                mlp = ([self._mlp.data_ptr()], self._mlp.data_ptr())
        self.oproj_push, self.oproj_in = oproj
        self.mlp_push, self.mlp_in = mlp
        assert len(self.oproj_push) in (1, R) and len(self.mlp_push) in (1, R)
        self.num_pages = layers[0]["k_pool"].shape[0]
        # validate the shapes and set the kernel attribute now (not under a stream capture, not inside a timed step)
        dummy = torch.zeros(1, H, dtype=torch.bfloat16, device=self.device)
        table = torch.zeros(1, 1, dtype=torch.int32, device=self.device)
        a = self.args(dummy, dummy, table, table.data_ptr(), None, None)
        a.prepare_only = 1
        check(native.lib().pb_decode_span(C.byref(a), stream_ptr()), "decode_span (prepare)", launches=0)

    def args(self, x_in: torch.Tensor, x_out: torch.Tensor, block_table: torch.Tensor, pos_ptr: int, cos, sin, in_flag: int = 0,
             in_per_epoch: int = 0, lo: int = 0, hi: Optional[int] = None):
        from petals_b200.ops.native import DecodeSpanArgs

        hi = self.table.shape[0] if hi is None else hi
        a = DecodeSpanArgs()
        a.layers, a.n_layers = self.table[lo:hi].data_ptr(), hi - lo
        a.H, a.Hq, a.Hkv, a.D, a.I, a.eps, a.attn_scale = self.H, self.Hq, self.Hkv, self.D, self.I, self.eps, self.attn_scale
        a.x_in, a.x_out, a.in_flag, a.in_per_epoch = x_in.data_ptr(), x_out.data_ptr(), in_flag or None, in_per_epoch
        a.block_table, a.max_pages, a.num_pages, a.pos_ptr = block_table.data_ptr(), block_table.shape[1], self.num_pages, pos_ptr
        a.cos, a.sin, a.max_pos = ptr(cos), ptr(sin), (cos.shape[0] if cos is not None else 0)
        a.qkv_ll, a.attp_ll, a.attn_ll, a.x_ll, a.act_ll = (self.qkv_ll.data_ptr(), self.attp_ll.data_ptr(), self.attn_ll.data_ptr(),
                                                            self.x_ll.data_ptr(), self.act_ll.data_ptr())
        a.max_chunks = min(self.max_chunks, block_table.shape[1])
        a.R, a.rank = self.R, self.rank
        for r in range(len(self.oproj_push)):
            a.oproj_push[r], a.mlp_push[r] = self.oproj_push[r], self.mlp_push[r]
        a.oproj_in, a.mlp_in = self.oproj_in, self.mlp_in
        if self.nvls.get("mode") == "st":
            a.oproj_mc_push, a.mlp_mc_push = self.nvls["oproj"], self.nvls["mlp"]
        elif self.nvls.get("mode") == "reduce":
            a.oproj_mc_sum, a.mlp_mc_sum, a.nvls_reduce = self.nvls["oproj"], self.nvls["mlp"], 1
        a.epoch, a.error_flag = self.epoch.data_ptr(), self.err.data_ptr()
        a.num_sms = native.sm_count(self.device.index)
        a.timing = ptr(getattr(self, "timing", None))
        return a


def decode_span_supported(*, H: int, Hq: int, Hkv: int, D: int, I: int) -> bool:
    """Shapes ``csrc/decode_span.cu`` takes (the launcher re-checks and explains)."""
    return D in (64, 128) and Hkv > 0 and Hq % Hkv == 0 and Hq // Hkv <= 16 and H % 64 == 0 and I % 4 == 0 and (Hq * D) % 64 == 0


def decode_span(plan: DecodeSpanPlan, x_in: torch.Tensor, x_out: torch.Tensor, block_table: torch.Tensor, pos_ptr: int, cos, sin, *,
                in_flag: int = 0, in_per_epoch: int = 0, lo: int = 0, hi: Optional[int] = None, bump_epoch: bool = True) -> torch.Tensor:
    """One token (``x_in`` [1, H] -> ``x_out`` [1, H]) through blocks [lo, hi) of the plan: one launch (plus the step-counter bump)."""
    if bump_epoch:
        check(native.lib().pb_bump_epoch(plan.epoch.data_ptr(), stream_ptr()), "bump_epoch")
    a = plan.args(x_in, x_out, block_table, pos_ptr, cos, sin, in_flag, in_per_epoch, lo, hi)
    check(native.lib().pb_decode_span(C.byref(a), stream_ptr()), "decode_span")
    return x_out
