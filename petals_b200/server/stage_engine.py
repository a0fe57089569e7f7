"""Stage engine: executes a contiguous span of transformer blocks on one B200 with the sm_100a kernels.

This is the B200-native counterpart of the reference's per-block ``TransformerBackend`` +
``_MergedInferenceStep`` (src/petals/server/backend.py:24-235): the *whole span* is the unit of execution.

* decode shapes (B*T <= 8 rows): every block is 7 launches — fused norm+QKV GEMV, RoPE+KV-append, paged
  split-KV attention (+combine), O-proj GEMV+residual, fused norm+gate/up GEMV+SwiGLU, down GEMV+residual —
  and the entire span is captured once per (B, T) into a CUDA graph whose only mutable inputs are device
  buffers (activation, block table, cache position). One graph replay per token per stage replaces the
  reference's per-block task-pool round trips and its six tiny per-op graphs (SURVEY.md §2.5(a)).
* prefill / parallel-forward shapes: tcgen05 GEMMs with fused bias/GELU/SwiGLU/residual epilogues, flash
  attention over the paged cache, chunked by ``max_chunk_tokens`` (the pipelining unit).
* no-cache forward (rpc_forward / training forward) reuses the same kernels against a one-layer scratch pool.
* anything without a hand-written kernel yet (MoE experts, backward) runs the oracle math on the same weight
  tensors, so every family is always servable.
"""
from __future__ import annotations

import os

import math
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from petals_b200.models.block_oracle import GenericBlock
from petals_b200.models.spec import BlockSpec, alibi_slopes
from petals_b200.ops import functional as Fn
from petals_b200.ops import native
from petals_b200.ops.functional import PAGE
from petals_b200.server.memory_cache import MemoryCache, SessionCache
from petals_b200.utils.logging import get_logger
from petals_b200.utils.misc import is_dummy

logger = get_logger(__name__)
MAX_DECODE_ROWS = 8


def fast_path_supported(spec: BlockSpec) -> bool:
    """Can the fused sm_100a kernels run this block family end to end?"""
    if spec.head_dim not in (64, 128) or spec.post_ln_residual:
        return False
    if spec.hidden_size % 8 or spec.intermediate_size % 8 or spec.qkv_dim % 8:
        return False
    return spec.mlp in ("swiglu", "gelu", "moe")


class StageEngine:
    FP8_NAMES = ("wqkv", "wo", "w_gate", "w_up", "w_down")

    def __init__(self, spec: BlockSpec, blocks: Sequence[GenericBlock], cache: MemoryCache, *, device,
                 max_chunk_tokens: int = 8192, use_cuda_graphs: bool = True, fp8: bool = False, free_bf16: bool = True):
        self.spec, self.blocks, self.cache = spec, list(blocks), cache
        # Block-scaled FP8 serving (--quant_type fp8): projections are kept as E4M3 payload + UE8M0 scales (ops/quant.py).
        # Decode streams the 1-byte weights directly (csrc/linear_decode_fp8.cu). Prefill quantises the activations to MXFP8 too
        # (fused with the RMSNorm in front of the projection) and multiplies on the block-scaled tensor-core path
        # (csrc/gemm_mxfp8.cu: tcgen05.mma kind::mxf8f6f4.block_scale, twice the bf16 rate); layouts that path does not cover
        # (or PETALS_B200_FP8_PREFILL=dequant) dequantise one projection at a time into a bf16 scratch for the bf16 GEMM.
        self.fp8: Optional[List[Dict[str, Tuple[torch.Tensor, torch.Tensor]]]] = None
        self.fp8_sf: Optional[List[Dict[str, torch.Tensor]]] = None  # weight scales in the tensor cores' block layout
        self.max_decode_rows = MAX_DECODE_ROWS
        if fp8:
            from petals_b200.ops.quant import quantize_mxfp8

            from petals_b200.ops.quant import pack_scales

            self.fp8, self.fp8_sf = [], []
            self.max_decode_rows = 4
            for block in self.blocks:
                entry = {}
                for name in self.FP8_NAMES:
                    p = getattr(block, name, None)
                    if p is None or p.dim() != 2 or p.shape[1] % 32:
                        continue
                    entry[name] = quantize_mxfp8(p.data)
                    if free_bf16:
                        p.data = torch.empty(0, dtype=p.dtype, device=p.device)
                self.fp8.append(entry)
                self.fp8_sf.append({n: pack_scales(e) for n, (q, e) in entry.items() if q.shape[1] % 128 == 0})
            s_ = spec
            self.fp8_w8a8 = (os.environ.get("PETALS_B200_FP8_PREFILL", "w8a8").lower() != "dequant" and torch.device(device).type == "cuda"
                             and s_.norm == "rms" and s_.mlp == "swiglu" and not s_.parallel_attn and not (s_.qkv_bias or s_.out_bias or s_.mlp_bias)
                             and all(set(sf) >= set(self.FP8_NAMES) for sf in self.fp8_sf))
        self.device = torch.device(device)
        self.n_blocks = len(self.blocks)
        self.max_chunk_tokens = max_chunk_tokens
        self.use_cuda_graphs = use_cuda_graphs
        self.dtype = torch.bfloat16
        s = spec
        self.norm_kind = Fn.NORM_RMS if s.norm == "rms" else Fn.NORM_LAYER
        self.act = Fn.ACT_SWIGLU if s.mlp == "swiglu" else (Fn.ACT_GELU_TANH if s.gelu_tanh else Fn.ACT_GELU_ERF)
        self.cos = self.sin = None
        if s.rotary:
            self.cos, self.sin = Fn.rope_tables(s.head_dim, s.max_position, s.rope_theta, s.rope_scaling, device=self.device)
        self.slopes = alibi_slopes(s.num_heads).to(self.device) if s.alibi else None
        self.sms = native.sm_count(self.device.index)
        # device-resident step state shared by all graphs
        self.max_pages = cache.max_pages_per_seq
        self.pos_static = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.err_flag = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.fuse_rope = os.environ.get("PETALS_B200_FUSE_ROPE", "1") != "0"
        # single-token steps of Llama-style spans as ONE persistent data-flow kernel (csrc/decode_span.cu): weights stream through
        # a shared-memory ring across what used to be kernel boundaries, phases are ordered by tagged data instead of launches
        self.use_span_kernel = os.environ.get("PETALS_B200_SPAN_KERNEL", "1") != "0" and self._span_kernel_ok()
        self._span_plans: Dict[Optional[str], Fn.DecodeSpanPlan] = {}  # per adapter (captured graphs keep the plan's table address)
        self._split_ctr = torch.zeros(8192, dtype=torch.int32, device=self.device)  # split-KV arrival counters (self-resetting)
        self._tables: Dict[int, torch.Tensor] = {}  # batch -> static block table
        self._graphs: Dict[Tuple[int, int, int, int], dict] = {}
        self._active: Optional[SessionCache] = None
        self._dev_pos = -1
        self._bufs: Dict[Tuple[str, int], torch.Tensor] = {}
        self._moe_bufs: Dict[str, torch.Tensor] = {}
        # opt-in (PETALS_B200_LORA_ENGINE=1): requests with an active LoRA adapter run on the kernels against per-adapter merged copies
        # of the targeted projections (utils/peft.py:MergedAdapterBlock) instead of falling back to the PyTorch executor. Each adapter
        # has its own weight views and its own captured graphs; activation buffers are shared. Not combined with FP8 weights.
        # PETALS_B200_LORA_ENGINE: "lowrank" (default) = base projection + x.A^T.B^T.scale as two extra skinny launches per adapted projection,
        # no weight copies (reference semantics: utils/peft.py:173-209); "merged" = per-adapter merged copies of the targeted projections;
        # "0" = adapter requests run on the PyTorch executor.
        mode = os.environ.get("PETALS_B200_LORA_ENGINE", "lowrank").lower()
        self.lora_mode = {"1": "merged", "merged": "merged", "lowrank": "lowrank"}.get(mode)
        self.lora_on_engine = self.lora_mode is not None and not fp8
        self._lora_tables: Dict[tuple, Optional[Tuple[torch.Tensor, torch.Tensor]]] = {}
        self._adapter: Optional[str] = None
        self._adapter_state: Dict[Optional[str], tuple] = {}
        # scratch one-layer pool for cache-less forward passes
        n_scratch = max(1, (max_chunk_tokens + PAGE - 1) // PAGE) + 1
        self._scratch_pool = torch.zeros(2, n_scratch, s.num_kv_heads, PAGE, s.head_dim, dtype=self.dtype, device=self.device)
        self._scratch_pages = n_scratch

    # ---- persistent span kernel ---------------------------------------------------------------------------------------
    def _span_kernel_ok(self) -> bool:
        s = self.spec
        return (self.fp8 is None and s.norm == "rms" and s.mlp == "swiglu" and s.rotary and not s.qkv_interleaved and not s.parallel_attn
                and not s.post_ln_residual and not s.alibi and not s.sliding_window and not (s.qkv_bias or s.out_bias or s.mlp_bias)
                and Fn.decode_span_supported(H=s.hidden_size, Hq=s.num_heads, Hkv=s.num_kv_heads, D=s.head_dim, I=s.intermediate_size)
                and all(b._p("bqkv") is None for b in self.blocks))

    def _span_kernel_plan(self) -> "Fn.DecodeSpanPlan":
        if self._adapter not in self._span_plans:
            s = self.spec
            layers = []
            for slot, b in enumerate(self.blocks):
                k_pool, v_pool = self.cache.layer_pools(slot)
                layers.append(dict(wqkv=b.wqkv, wo=b.wo, w_gate=b.w_gate, w_up=b.w_up, w_down=b.w_down, ln1_w=b.ln1_w, ln2_w=b.ln2_w,
                                   k_pool=k_pool, v_pool=v_pool))
            self._span_plans[self._adapter] = Fn.DecodeSpanPlan(layers, H=s.hidden_size, Hq=s.num_heads, Hkv=s.num_kv_heads, D=s.head_dim, I=s.intermediate_size,
                                                eps=s.norm_eps, attn_scale=s.attn_scale, max_chunks=self.max_pages, device=self.device,
                                                error_flag=self.err_flag)
        return self._span_plans[self._adapter]

    # ---- adapters ------------------------------------------------------------------------------------------
    def use_adapter(self, name: Optional[str]) -> None:
        """Switch the weight views and the graph cache to those of ``name`` (``None`` = the base weights)."""
        if name == self._adapter:
            return
        if not self.lora_on_engine and name is not None:
            raise RuntimeError("this engine does not serve adapters (PETALS_B200_LORA_ENGINE=1 enables merged-weight serving)")
        self._adapter_state[self._adapter] = (self.blocks, self._graphs)
        if name not in self._adapter_state:
            base = self._adapter_state[None][0] if None in self._adapter_state else self.blocks
            if self.lora_mode == "merged":
                from petals_b200.utils.peft import MergedAdapterBlock

                with torch.inference_mode(False):
                    views = [MergedAdapterBlock(b, name) for b in base]
                logger.info(f"adapter {name}: merged copies of the targeted projections take {sum(v.merged_bytes for v in views) / 2**20:.0f} MiB")
                self._adapter_state[name] = (views, {})
            else:
                for b in base:
                    if name not in getattr(b, "lora_adapters", {}):
                        raise KeyError(f"Adapter {name!r} is not loaded on this server (available: {sorted(getattr(b, 'lora_adapters', {}))})")
                self._adapter_state[name] = (base, {})  # same weights, own graph cache: the low-rank factors ride next to the base GEMVs
        self.blocks, self._graphs = self._adapter_state[name]
        self._adapter = name

    def _lora(self, slot: int, name: str) -> Optional[Tuple[torch.Tensor, torch.Tensor]]:
        """Low-rank factors of the active adapter for projection ``name`` of block ``slot``: ``(A [r, in], B [out, r])`` with every pair on
        that projection stacked along r (a pair on q_proj only touches the q rows of the fused QKV: its B is zero elsewhere), the
        scale folded into B, r padded to a multiple of 64 with zeros (tile-aligned for both kernels). None: nothing to add."""
        if self._adapter is None or self.lora_mode != "lowrank":
            return None
        key = (self._adapter, slot, name)
        if key not in self._lora_tables:
            entries = getattr(self.blocks[slot], "lora_adapters", {}).get(self._adapter, {}).get(name)
            if not entries:
                self._lora_tables[key] = None
            else:
                w = getattr(self.blocks[slot], name)
                r_tot = sum(A.shape[0] for A, _, _, _ in entries)
                r_pad = (r_tot + 63) // 64 * 64
                with torch.inference_mode(False):
                    A_cat = torch.zeros(r_pad, w.shape[1], dtype=self.dtype, device=self.device)
                    B_cat = torch.zeros(w.shape[0], r_pad, dtype=torch.float32, device=self.device)
                    r0 = 0
                    for A, Bm, scale, rows in entries:
                        r = A.shape[0]
                        A_cat[r0:r0 + r] = A.to(self.device, self.dtype)
                        B_cat[(slice(None) if rows is None else rows), r0:r0 + r] = Bm.to(self.device, torch.float32) * float(scale)
                        r0 += r
                    self._lora_tables[key] = (A_cat, B_cat.to(self.dtype).contiguous())
        return self._lora_tables[key]

    def _lora_add_decode(self, slot: int, name: str, x: torch.Tensor, y: torch.Tensor, **prologue) -> None:
        """y += (prologue(x) A^T) B^T for decode shapes: two skinny weight-streaming launches, the second accumulates into y."""
        ab = self._lora(slot, name)
        if ab is None:
            return
        t = Fn.linear_decode(x, ab[0], out=self._buf("lora_t", x.shape[0], ab[0].shape[0]), **prologue)
        Fn.linear_decode(t, ab[1], residual=y, out=y)

    def _lora_add_prefill(self, slot: int, name: str, xn: torch.Tensor, y: torch.Tensor) -> None:
        ab = self._lora(slot, name)
        if ab is None:
            return
        t = Fn.gemm(xn, ab[0], out=self._buf("lora_t_p", xn.shape[0], ab[0].shape[0]))
        Fn.gemm(t, ab[1], residual=y, out=y)

    def _has_lora(self, slot: int, *names: str) -> bool:
        return any(self._lora(slot, n) is not None for n in names)

    # ---- buffers ---------------------------------------------------------------------------------------
    def _w(self, slot: int, name: str) -> Optional[torch.Tensor]:
        """bf16 view of a projection weight: the block's tensor, or (FP8 serving) a scratch dequantised on the fly."""
        p = getattr(self.blocks[slot], name, None)
        if self.fp8 is None or name not in self.fp8[slot]:
            return p
        if p is not None and p.numel() > 0:
            return p
        q, e = self.fp8[slot][name]
        return Fn.dequant_mxfp8(q, e, out=self._buf("dq_" + name, q.shape[0], q.shape[1]))

    def _lin_decode(self, slot: int, name: str, x: torch.Tensor, name2: Optional[str] = None, **kw) -> torch.Tensor:
        """One decode-shape projection: bf16 weight streamer, or its FP8 twin when this stage serves quantised weights."""
        w = self.blocks[slot]
        if self.fp8 is not None and name in self.fp8[slot]:
            q, e = self.fp8[slot][name]
            q2, e2 = self.fp8[slot][name2] if name2 else (None, None)
            return Fn.linear_decode_fp8(x, q, e, w2_q=q2, w2_scale=e2, **kw)
        return Fn.linear_decode(x, getattr(w, name), w2=getattr(w, name2) if name2 else None, **kw)

    def _buf(self, name: str, rows: int, cols: int, dtype=None) -> torch.Tensor:
        """Persistent activation buffer. Decode-shape buffers are keyed by their full shape and never replaced (captured CUDA
        graphs keep their raw addresses). Prefill / forward buffers (row count = B*T of whatever a client sends) are ONE grow-only
        allocation per name, handed out as views: a client sweeping prompt lengths cannot grow the pool without bound."""
        dtype = dtype or self.dtype
        growable = rows > MAX_DECODE_ROWS and (name.endswith("_p") or name in ("x_fwd", "x_taken") or name.startswith("dq_") or name.startswith("bw_"))
        if growable:
            key, need = (name, dtype), rows * cols
            flat = self._bufs.get(key)
            if flat is None or flat.numel() < need:
                with torch.inference_mode(False):
                    flat = torch.empty(need, dtype=dtype, device=self.device)  # the old one is released in stream order
                self._bufs[key] = flat
            return flat[:need].view(rows, cols)
        key = (name, rows, cols, dtype)
        t = self._bufs.get(key)
        if t is None:
            with torch.inference_mode(False):  # persistent: must stay writable from threads outside inference mode
                t = torch.empty(rows, cols, dtype=dtype, device=self.device)
            self._bufs[key] = t
        return t

    def _table(self, B: int) -> torch.Tensor:
        if B not in self._tables:
            with torch.inference_mode(False):
                self._tables[B] = torch.zeros(B, self.max_pages, dtype=torch.int32, device=self.device)
        return self._tables[B]

    def _splits(self, B: int, T: int) -> int:
        G = self.spec.group_size
        m_tiles = (T * G + 63) // 64
        ctas = B * self.spec.num_kv_heads * m_tiles
        return int(min(16, max(1, (2 * self.sms) // max(1, ctas))))

    def _split_counter(self, B: int, T: int, splits: int) -> Optional[torch.Tensor]:
        """Arrival counters that let the last split CTA merge the split-KV partials inside the attention kernel."""
        if splits <= 1:
            return None
        m_tiles = (T * self.spec.group_size + 63) // 64
        return self._split_ctr if m_tiles * B * self.spec.num_kv_heads <= self._split_ctr.numel() else None

    # ---- one block ---------------------------------------------------------------------------------------
    def _attention(self, qkv: torch.Tensor, slot: int, B: int, T: int, table: torch.Tensor, pos_ptr: int,
                   pools: Tuple[torch.Tensor, torch.Tensor], splits: int, tag: str) -> torch.Tensor:
        s = self.spec
        M = B * T
        w = self.blocks[slot]
        q_buf = self._buf(f"q{tag}", M, s.num_heads * s.head_dim)
        attn = self._buf(f"attn{tag}", M, s.num_heads * s.head_dim)
        if qkv is not None:  # None: RoPE + KV append already happened in the QKV projection's epilogue
            Fn.rope_kv_append(qkv, q_buf, pools[0], pools[1], table, pos_ptr, self.cos, self.sin, B=B, T=T, Hq=s.num_heads,
                              Hkv=s.num_kv_heads, D=s.head_dim, qkv_bias=None, interleaved=s.qkv_interleaved,
                              error_flag=self.err_flag.data_ptr())
        po = pl = None
        if splits > 1:
            po = self._buf(f"po{tag}", splits * M * s.num_heads, s.head_dim, torch.float32)
            pl = self._buf(f"pl{tag}", splits, M * s.num_heads, torch.float32)
        Fn.paged_attention(q_buf, pools[0], pools[1], table, pos_ptr, attn, B=B, T=T, Hq=s.num_heads, Hkv=s.num_kv_heads,
                           D=s.head_dim, scale=s.attn_scale, splits=splits, partial_o=po, partial_lse=pl,
                           alibi_slopes=self.slopes, window=s.sliding_window, split_counter=self._split_counter(B, T, splits))
        return attn

    def _push_kwargs(self, hop: Optional[tuple], gemm: bool = False) -> dict:
        """Epilogue/prologue arguments that turn the span's last kernel into the fused stage hop (see parallel/fabric.py)."""
        if hop is None:
            return {}
        fabric, kind, rank = hop[:3]
        slot = hop[3] if len(hop) > 3 else 0
        data, flag = fabric.zone(kind, rank, slot)
        kw = fabric.begin_push(kind, slot)
        kw.update(push_out=[data], done_counter=fabric.done_counter.data_ptr())
        if gemm:
            kw["push_done_flag"] = [flag]
        else:
            kw["push_flag"] = [flag]
        return kw

    def _block_decode(self, x: torch.Tensor, out: torch.Tensor, slot: int, B: int, T: int, table, pos_ptr, pools, splits,
                      hop: Optional[tuple] = None) -> torch.Tensor:
        """x, out: [M, H] ping-pong residual buffers. Returns the buffer holding the block output."""
        s, w = self.spec, self.blocks[slot]
        M = B * T
        eps = s.norm_eps
        if self.fuse_rope and self.fp8 is None and w._p("bqkv") is None and not s.qkv_interleaved and not self._has_lora(slot, "wqkv"):
            # QKV projection whose epilogue rotates q/k and appends k/v to the cache pages: no RoPE launch, no qkv round trip
            Fn.linear_decode(x, w.wqkv, norm_weight=w.ln1_w, norm_bias=w._p("ln1_b"), norm_kind=self.norm_kind, eps=eps,
                             error_flag=self.err_flag.data_ptr(),
                             rope=dict(q_out=self._buf("q", M, s.num_heads * s.head_dim), k_pool=pools[0], v_pool=pools[1], block_table=table,
                                       pos_ptr=pos_ptr, cos=self.cos, sin=self.sin, T=T, Hq=s.num_heads, Hkv=s.num_kv_heads, D=s.head_dim))
            qkv = None
        else:
            qkv = self._lin_decode(slot, "wqkv", x, bias=w._p("bqkv"), norm_weight=w.ln1_w, norm_bias=w._p("ln1_b"), norm_kind=self.norm_kind,
                                   eps=eps, out=self._buf("qkv", M, s.qkv_dim))
            self._lora_add_decode(slot, "wqkv", x, qkv, norm_weight=w.ln1_w, norm_bias=w._p("ln1_b"), norm_kind=self.norm_kind, eps=eps)
        attn = self._attention(qkv, slot, B, T, table, pos_ptr, pools, splits, "")
        h1 = self._lin_decode(slot, "wo", attn, bias=w._p("bo"), residual=x, out=out)
        self._lora_add_decode(slot, "wo", attn, h1)
        if s.mlp == "moe":
            # router + the k chosen experts' GEMVs + combine: sync-free, so the whole block stays graph-capturable
            return Fn.moe_decode(h1, w.ln2_w, w.router, w.we_gate, w.we_up, w.we_down, top_k=s.top_k, eps=eps, out=x, bufs=self._moe_bufs)
        if s.parallel_attn:
            mlp_in, ln_w, ln_b = x, (w.ln2_w if s.dual_ln else w.ln1_w), (w._p("ln2_b") if s.dual_ln else w._p("ln1_b"))
        else:
            mlp_in, ln_w, ln_b = h1, w.ln2_w, w._p("ln2_b")
        norm_kw = dict(norm_weight=ln_w, norm_bias=ln_b, norm_kind=self.norm_kind, eps=eps)
        if s.mlp == "swiglu" and self._has_lora(slot, "w_gate", "w_up"):
            # the low-rank terms enter before the activation: gate and up separately, then the SwiGLU kernel
            g = self._lin_decode(slot, "w_gate", mlp_in, out=self._buf("lora_g", M, s.intermediate_size), **norm_kw)
            u = self._lin_decode(slot, "w_up", mlp_in, out=self._buf("lora_u", M, s.intermediate_size), **norm_kw)
            self._lora_add_decode(slot, "w_gate", mlp_in, g, **norm_kw)
            self._lora_add_decode(slot, "w_up", mlp_in, u, **norm_kw)
            act = Fn.swiglu(g, u, out=self._buf("act", M, s.intermediate_size))
        elif s.mlp == "swiglu":
            act = self._lin_decode(slot, "w_gate", mlp_in, "w_up", act=Fn.ACT_SWIGLU, out=self._buf("act", M, s.intermediate_size), **norm_kw)
        elif self._has_lora(slot, "w_up"):
            pre = self._lin_decode(slot, "w_up", mlp_in, bias=w._p("b_up"), out=self._buf("lora_u", M, s.intermediate_size), **norm_kw)
            self._lora_add_decode(slot, "w_up", mlp_in, pre, **norm_kw)
            act = Fn.activation(pre, self.act, out=self._buf("act", M, s.intermediate_size))
        else:
            act = self._lin_decode(slot, "w_up", mlp_in, bias=w._p("b_up"), act=self.act, out=self._buf("act", M, s.intermediate_size), **norm_kw)
        # down projection + residual; write into x's buffer (x is dead for sequential blocks, and for
        # parallel blocks h1 already contains x + attn). With `hop`, the same epilogue also stores the rows into the
        # next stage's landing zone over NVLink and publishes its flag: the stage hop costs no extra kernel.
        if self._has_lora(slot, "w_down"):
            y = self._lin_decode(slot, "w_down", act, bias=w._p("b_down"), residual=h1, out=x)
            self._lora_add_decode(slot, "w_down", act, y)
            if hop is not None:
                hop[0].send(y, hop[2], hop[1], *hop[3:4])
            return y
        return self._lin_decode(slot, "w_down", act, bias=w._p("b_down"), residual=h1, out=x, **self._push_kwargs(hop))

    def _quant_rows(self, x: torch.Tensor, norm_w: Optional[torch.Tensor], tag: str) -> Tuple[torch.Tensor, torch.Tensor]:
        """MXFP8 copy of the rows of ``x`` (RMSNorm(x) * norm_w when a weight is given) in grow-only scratch buffers."""
        M, K = x.shape
        q = self._buf(f"q8{tag}_p", M, K, torch.uint8)
        sf = self._buf(f"sf8{tag}_p", ((M + 127) // 128) * (K // 128), 512, torch.uint8)
        return Fn.quant_mxfp8(x, norm_w, self.spec.norm_eps, q=q, sf=sf)

    def _block_prefill_fp8(self, x: torch.Tensor, slot: int, B: int, T: int, table, pos_ptr, pools, hop: Optional[tuple] = None) -> torch.Tensor:
        """The prefill block with every projection on the block-scaled FP8 tensor-core path: activations are quantised per 32 values
        along K right where they are produced (norm outputs: fused with the norm), weights are the stage's MXFP8 payloads."""
        s, w, f, sf = self.spec, self.blocks[slot], self.fp8[slot], self.fp8_sf[slot]
        M = B * T
        aq, asf = self._quant_rows(x, w.ln1_w, "h")
        qkv = Fn.gemm_mxfp8(aq, asf, f["wqkv"][0], sf["wqkv"], out=self._buf("qkv_p", M, s.qkv_dim))
        attn = self._attention(qkv, slot, B, T, table, pos_ptr, pools, 1, "_p")
        aq, asf = self._quant_rows(attn, None, "a")
        h1 = Fn.gemm_mxfp8(aq, asf, f["wo"][0], sf["wo"], residual=x, out=self._buf("h1_p", M, s.hidden_size))
        aq, asf = self._quant_rows(h1, w.ln2_w, "h")
        act = Fn.gemm_mxfp8(aq, asf, f["w_gate"][0], sf["w_gate"], b2_q=f["w_up"][0], b2_sf=sf["w_up"], out=self._buf("act_p", M, s.intermediate_size))
        aq, asf = self._quant_rows(act, None, "i")
        y = Fn.gemm_mxfp8(aq, asf, f["w_down"][0], sf["w_down"], residual=h1, out=x)
        if hop is not None:
            hop[0].send(y, hop[2], hop[1], *hop[3:4])
        return y

    def _block_prefill(self, x: torch.Tensor, slot: int, B: int, T: int, table, pos_ptr, pools, hop: Optional[tuple] = None) -> torch.Tensor:
        """x: [M, H] (overwritten with the block output)."""
        s, w = self.spec, self.blocks[slot]
        M = B * T
        eps = s.norm_eps
        if self.fp8 is not None and self.fp8_w8a8:
            return self._block_prefill_fp8(x, slot, B, T, table, pos_ptr, pools, hop)
        xn = Fn.norm(x, w.ln1_w, w._p("ln1_b"), kind=self.norm_kind, eps=eps, out=self._buf("xn_p", M, s.hidden_size))
        qkv = Fn.gemm(xn, self._w(slot, "wqkv"), bias=w._p("bqkv"), out=self._buf("qkv_p", M, s.qkv_dim))
        self._lora_add_prefill(slot, "wqkv", xn, qkv)
        attn = self._attention(qkv, slot, B, T, table, pos_ptr, pools, 1, "_p")
        h1 = Fn.gemm(attn, self._w(slot, "wo"), bias=w._p("bo"), residual=x, out=self._buf("h1_p", M, s.hidden_size))
        self._lora_add_prefill(slot, "wo", attn, h1)
        if s.mlp == "moe":
            return self._moe_prefill(h1, w, x)
        if s.parallel_attn:
            xn2 = Fn.norm(x, w.ln2_w, w._p("ln2_b"), kind=self.norm_kind, eps=eps, out=xn) if s.dual_ln else xn
        else:
            xn2 = Fn.norm(h1, w.ln2_w, w._p("ln2_b"), kind=self.norm_kind, eps=eps, out=xn)
        act_buf = self._buf("act_p", M, s.intermediate_size)
        if s.mlp == "swiglu" and self._has_lora(slot, "w_gate", "w_up"):
            g = Fn.gemm(xn2, self._w(slot, "w_gate"), out=self._buf("lora_g_p", M, s.intermediate_size))
            u = Fn.gemm(xn2, self._w(slot, "w_up"), out=self._buf("lora_u_p", M, s.intermediate_size))
            self._lora_add_prefill(slot, "w_gate", xn2, g)
            self._lora_add_prefill(slot, "w_up", xn2, u)
            act = Fn.swiglu(g, u, out=act_buf)
        elif s.mlp == "swiglu":
            act = Fn.gemm(xn2, self._w(slot, "w_gate"), b2=self._w(slot, "w_up"), act=Fn.ACT_SWIGLU, out=act_buf)
        elif self._has_lora(slot, "w_up"):
            pre = Fn.gemm(xn2, self._w(slot, "w_up"), bias=w._p("b_up"), out=self._buf("lora_u_p", M, s.intermediate_size))
            self._lora_add_prefill(slot, "w_up", xn2, pre)
            act = Fn.activation(pre, self.act, out=act_buf)
        else:
            act = Fn.gemm(xn2, self._w(slot, "w_up"), bias=w._p("b_up"), act=self.act, out=act_buf)
        if self._has_lora(slot, "w_down"):
            y = Fn.gemm(act, self._w(slot, "w_down"), bias=w._p("b_down"), residual=h1, out=x)
            self._lora_add_prefill(slot, "w_down", act, y)
            if hop is not None:
                hop[0].send(y, hop[2], hop[1], *hop[3:4])
            return y
        return Fn.gemm(act, self._w(slot, "w_down"), bias=w._p("b_down"), residual=h1, out=x, **self._push_kwargs(hop, gemm=True))

    def _moe_prefill(self, h1: torch.Tensor, w: GenericBlock, out: torch.Tensor) -> torch.Tensor:
        """out = h1 + MoE(RMSNorm(h1)) for many tokens, entirely on the device: the routing plan (expert-major row order + the tile
        table of the grouped tcgen05 GEMM) is built by a kernel, so no group size ever travels to the host (ops/functional.py)."""
        s = self.spec
        return Fn.moe_prefill(h1, w.ln2_w, w.router, w.we_gate, w.we_up, w.we_down, top_k=s.top_k, eps=s.norm_eps, out=out, bufs=self._moe_bufs)

    # ---- span execution ------------------------------------------------------------------------------------
    def _sync_session(self, session: SessionCache, B: int) -> torch.Tensor:
        table = self._table(B)
        if self._active is not session or session._synced_version != session._version:
            table.copy_(session.table_dev[:, : self.max_pages], non_blocking=True)
            session._synced_version = session._version
            self._active = session
            self._dev_pos = -1
        if self._dev_pos != session.position:
            self.pos_static.fill_(session.position)
            self._dev_pos = session.position
        return table

    def _run_span(self, x: torch.Tensor, B: int, T: int, lo: int, hi: int, table, pos_ptr, pools_of, prompts, decode: bool, splits: int,
                  hop: Optional[tuple] = None) -> torch.Tensor:
        M = B * T
        if (decode and M == 1 and self.use_span_kernel and prompts is None and hop is None and hi > lo and pools_of == self.cache.layer_pools
                and (self._adapter is None or self.lora_mode == "merged")):
            out = self._buf("h_alt", M, self.spec.hidden_size)
            return Fn.decode_span(self._span_kernel_plan(), x, out, table, pos_ptr, self.cos, self.sin, lo=lo, hi=hi)
        other = self._buf("h_alt", M, self.spec.hidden_size) if decode else None
        cur = x
        for slot in range(lo, hi):
            if prompts is not None and not is_dummy(prompts[slot - lo]):
                Fn.add_prompts(cur.view(B, T, -1), prompts[slot - lo])
            fused_hop = hop if (slot == hi - 1 and self.spec.mlp != "moe" and not (decode and self.fp8 is not None)) else None
            if decode:
                nxt = self._block_decode(cur, other, slot, B, T, table, pos_ptr, pools_of(slot), splits, fused_hop)
                if nxt is not cur:  # MoE path returned the alternate buffer
                    cur, other = nxt, cur
            else:
                cur = self._block_prefill(cur, slot, B, T, table, pos_ptr, pools_of(slot), fused_hop)
        if hop is not None and (self.spec.mlp == "moe" or (decode and self.fp8 is not None)):  # no fused epilogue here yet: host-issued NVLink copy
            hop[0].send(cur, hop[2], hop[1], *hop[3:4])
        return cur

    def inference_step(self, session: SessionCache, hidden: torch.Tensor, prompts: Optional[Sequence[torch.Tensor]] = None,
                       hypo_ids: Optional[torch.Tensor] = None, block_range: Optional[Tuple[int, int]] = None,
                       take_from: Optional[tuple] = None, push_to: Optional[tuple] = None) -> torch.Tensor:
        """One rpc_inference step through blocks [lo, hi) of this stage (reference: backend.py:111-144).

        ``take_from = (fabric, src_rank, B, T[, slot])``: the input was pushed into landing slot ``slot`` of this rank by
        ``src_rank``'s last kernel (``hidden`` is then only a shape carrier). ``push_to = (fabric, kind, rank[, slot])``: the span's
        last kernel stores its output into that landing slot of ``rank``; the returned tensor is then empty."""
        lo, hi = block_range or (0, self.n_blocks)
        if take_from is not None:
            fabric, src_rank, B, T = take_from[:4]
            H = self.spec.hidden_size
            staged = self._buf("x_taken", B * T, H)
            fabric.take(B * T, "x_in", src_rank, staged, *take_from[4:5])
            hidden = staged.view(B, T, H)
        B, T, H = hidden.shape
        if hypo_ids is not None and not is_dummy(hypo_ids):
            session.reorder(hypo_ids)
        if T == 0:
            return hidden
        if hidden.dtype != self.dtype:
            hidden = hidden.to(self.dtype)
        out = torch.empty(B, T, H, dtype=self.dtype, device=self.device)
        has_prompts = prompts is not None and any(not is_dummy(p) for p in prompts)
        # chunked prefill: the chunk is also the unit a downstream stage can start on
        max_t = max(1, self.max_chunk_tokens // B)
        if push_to is not None:
            if T > max_t or B * T > push_to[0].max_tokens:
                raise ValueError("a fused stage hop needs the whole step in one chunk; split the input on the client")
            self._step_chunk(session, hidden, [p[:, :T] if (p is not None and not is_dummy(p)) else None for p in prompts] if has_prompts else None,
                             lo, hi, push_to)
            return hidden[:, :0]
        for t0 in range(0, T, max_t):
            t1 = min(T, t0 + max_t)
            chunk = hidden[:, t0:t1]
            cp = None
            if has_prompts:
                cp = [p[:, t0:t1] if (not is_dummy(p) and t0 < p.shape[1]) else None for p in prompts]
                if all(c is None for c in cp):
                    cp = None
            out[:, t0:t1] = self._step_chunk(session, chunk, cp, lo, hi)
        return out

    def _step_chunk(self, session: SessionCache, hidden: torch.Tensor, prompts, lo: int, hi: int, hop: Optional[tuple] = None) -> torch.Tensor:
        B, T, H = hidden.shape
        M = B * T
        session.prepare_write(T)
        table = self._sync_session(session, B)
        pos_ptr = self.pos_static.data_ptr()
        pools_of = self.cache.layer_pools
        decode = M <= self.max_decode_rows
        if decode and self.use_cuda_graphs and prompts is None:
            key = (B, T, lo, hi) if hop is None else (B, T, lo, hi) + tuple(hop[1:])
            g = self._graphs.get(key)
            if g is None:
                g = self._capture(B, T, lo, hi, table, hop)
            g["x"].copy_(hidden.reshape(M, H))
            g["graph"].replay()
            native.add_launches(g["launches"])
            result = g["out"].view(B, T, H).clone()
        else:
            x = self._buf("x_in" if decode else "x_in_p", M, H)
            x.copy_(hidden.reshape(M, H))
            splits = self._splits(B, T) if decode else 1
            y = self._run_span(x, B, T, lo, hi, table, pos_ptr, pools_of, prompts, decode, splits, hop)
            native.check(native.lib().pb_advance_pos(pos_ptr, T, native.stream_ptr()), "advance_pos")
            result = y.view(B, T, H).clone()
        session.set_position(session.position + T, sync_device=False)
        self._dev_pos = session.position
        return result

    def _capture(self, B: int, T: int, lo: int, hi: int, table: torch.Tensor, hop: Optional[tuple] = None) -> dict:
        """Capture the decode step of blocks [lo, hi) for a (B, T) shape into a CUDA graph."""
        M, H = B * T, self.spec.hidden_size
        with torch.inference_mode(False):
            x = torch.zeros(M, H, dtype=self.dtype, device=self.device)
        pos_ptr = self.pos_static.data_ptr()
        splits = self._splits(B, T)
        saved_pos = self.pos_static.clone()

        def run():
            xin = self._buf("x_in", M, H)
            xin.copy_(x)
            y = self._run_span(xin, B, T, lo, hi, table, pos_ptr, self.cache.layer_pools, None, True, splits, cap_hop[0])
            native.check(native.lib().pb_advance_pos(pos_ptr, T, native.stream_ptr()), "advance_pos")
            return y

        # warm-up on a side stream (sets kernel attributes, allocates buffers), then capture. The warm-up runs WITHOUT the
        # hop: a push would consume a transfer slot on the peer.
        cap_hop = [None]
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            run()
        cap_hop[0] = hop
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize(self.device)
        self.pos_static.copy_(saved_pos)
        graph = torch.cuda.CUDAGraph()
        before = native.launch_count
        with torch.cuda.graph(graph):
            out = run()
        launches = native.launch_count - before
        native.add_launches(-launches)  # captured, not executed
        self.pos_static.copy_(saved_pos)  # capture does not execute, but keep the invariant explicit
        g = dict(graph=graph, x=x, out=out, launches=launches)
        self._graphs[(B, T, lo, hi) if hop is None else (B, T, lo, hi) + tuple(hop[1:])] = g
        logger.debug(f"captured decode graph B={B} T={T} blocks [{lo},{hi}) splits={splits}")
        return g

    # ---- cache-less forward (rpc_forward / training forward) ----------------------------------------------------
    def forward(self, hidden: torch.Tensor, prompts: Optional[Sequence[torch.Tensor]] = None,
                block_range: Optional[Tuple[int, int]] = None, hop: Optional[tuple] = None) -> torch.Tensor:
        """``hop = (fabric, kind, rank[, slot])``: the span output is also stored into that landing slot — by the epilogue of the
        span's last GEMM when the batch is one group (the forward micro-batch hop of training), by a peer copy otherwise."""
        lo, hi = block_range or (0, self.n_blocks)
        B, T, H = hidden.shape
        if T == 0 or B == 0:
            return hidden
        if hidden.dtype != self.dtype:
            hidden = hidden.to(self.dtype)
        out = torch.empty_like(hidden)
        # attention is causal within a sequence, so batch rows are independent: process them in groups that
        # fit the scratch pool
        # every row owns ceil(T / PAGE) WHOLE pages of the scratch pool, so groups are sized in pages, not tokens
        pages_per_seq = (T + PAGE - 1) // PAGE
        if pages_per_seq > self._scratch_pages:
            raise ValueError(f"sequence of {T} tokens exceeds max_chunk_tokens={self.max_chunk_tokens} for a cache-less forward")
        rows_per_group = max(1, self._scratch_pages // pages_per_seq)
        zero = torch.zeros(1, dtype=torch.int32, device=self.device)
        for b0 in range(0, B, rows_per_group):
            b1 = min(B, b0 + rows_per_group)
            nb = b1 - b0
            assert nb * pages_per_seq <= self._scratch_pages
            table = torch.arange(nb * pages_per_seq, dtype=torch.int32, device=self.device).view(nb, pages_per_seq).contiguous()
            x = self._buf("x_fwd", nb * T, H)
            x.copy_(hidden[b0:b1].reshape(nb * T, H))
            pr = None
            if prompts is not None and any(not is_dummy(p) for p in prompts):
                pr = [p if is_dummy(p) or p.shape[0] == 1 else p[b0:b1] for p in prompts]
            scratch = lambda slot: (self._scratch_pool[0], self._scratch_pool[1])
            decode = nb * T <= self.max_decode_rows
            fused = hop if (hop is not None and nb == B and hi > lo) else None
            y = self._run_span(x, nb, T, lo, hi, table, zero.data_ptr(), scratch, pr, decode, 1, fused)
            out[b0:b1] = y.view(nb, T, H)
        if hop is not None and not (rows_per_group >= B and hi > lo):
            hop[0].send(out.view(B * T, H), hop[2], hop[1], *hop[3:4])
        self._active = None  # the static table/pos were not touched, but be conservative
        return out

    # ---- backward (rpc_backward: gradients w.r.t. activations and deep prompts; the blocks are frozen) -----------------------
    def backward_supported(self) -> bool:
        """Block layouts whose backward runs on the kernels end to end (Llama-style: RMSNorm, SwiGLU, rotary GQA, no biases).
        Other families are differentiated by autograd over the oracle block (server/backend.py)."""
        s = self.spec
        return (self.fp8 is None and self._adapter is None and s.norm == "rms" and s.mlp == "swiglu" and s.rotary and not s.qkv_interleaved
                and not s.parallel_attn and not s.post_ln_residual and not s.alibi and not s.sliding_window
                and not (s.qkv_bias or s.out_bias or s.mlp_bias) and s.head_dim in (64, 128) and s.hidden_size % 64 == 0 and s.intermediate_size % 64 == 0 and s.qkv_dim % 64 == 0
                and all(b._p("bqkv") is None for b in self.blocks))

    def _forward_saving(self, x: torch.Tensor, slot: int, nb: int, T: int, table: torch.Tensor, zero_ptr: int) -> Tuple[torch.Tensor, dict]:
        """One block forward on the kernels that keeps what its backward needs: the block input, the rotated queries, this block's
        K/V pages, the attention output with its log-sum-exp, the post-attention residual and the two MLP projections."""
        s, w = self.spec, self.blocks[slot]
        M, dev, bf = nb * T, self.device, torch.bfloat16
        pages = table.numel()
        sv = dict(x=x, q=torch.empty(M, s.num_heads * s.head_dim, dtype=bf, device=dev),
                  # zero-filled: the tail of a sequence's last page is multiplied by exactly-zero probabilities in the tensor cores
                  k_pool=torch.zeros(pages, s.num_kv_heads, PAGE, s.head_dim, dtype=bf, device=dev),
                  v_pool=torch.zeros(pages, s.num_kv_heads, PAGE, s.head_dim, dtype=bf, device=dev),
                  attn=torch.empty(M, s.num_heads * s.head_dim, dtype=bf, device=dev), lse=torch.empty(M * s.num_heads, dtype=torch.float32, device=dev))
        xn = Fn.norm(x, w.ln1_w, None, kind=self.norm_kind, eps=s.norm_eps, out=self._buf("bw_xn_p", M, s.hidden_size))
        qkv = Fn.gemm(xn, w.wqkv, out=self._buf("bw_qkv_p", M, s.qkv_dim))
        Fn.rope_kv_append(qkv, sv["q"], sv["k_pool"], sv["v_pool"], table, zero_ptr, self.cos, self.sin, B=nb, T=T, Hq=s.num_heads, Hkv=s.num_kv_heads,
                          D=s.head_dim, error_flag=self.err_flag.data_ptr())
        Fn.paged_attention(sv["q"], sv["k_pool"], sv["v_pool"], table, zero_ptr, sv["attn"], B=nb, T=T, Hq=s.num_heads, Hkv=s.num_kv_heads, D=s.head_dim,
                           scale=s.attn_scale, splits=1, lse_out=sv["lse"])
        sv["h1"] = Fn.gemm(sv["attn"], w.wo, residual=x)
        xn2 = Fn.norm(sv["h1"], w.ln2_w, None, kind=self.norm_kind, eps=s.norm_eps, out=xn)
        sv["g"], sv["u"] = Fn.gemm(xn2, w.w_gate), Fn.gemm(xn2, w.w_up)
        act = Fn.swiglu(sv["g"], sv["u"], out=self._buf("bw_act_p", M, s.intermediate_size))
        return Fn.gemm(act, w.w_down, residual=sv["h1"]), sv

    def _backward_block(self, dy: torch.Tensor, sv: dict, slot: int, nb: int, T: int, table: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """dL/d(block input) from dL/d(block output): dgrad GEMMs on the untransposed weights (tcgen05, MN-major B), SwiGLU / RMSNorm /
        RoPE backward kernels, flash-attention backward. ``out``: where the block's last kernel stores the result (the previous stage's
        landing slot when this is the gradient hop)."""
        s, w = self.spec, self.blocks[slot]
        M = nb * T
        d_act = Fn.gemm(dy, w.w_down, b_mn_major=True, out=self._buf("bw_act_p", M, s.intermediate_size))
        Fn.swiglu_bwd_(d_act, sv["g"], sv["u"])  # g <- d gate, u <- d up
        d_xn2 = Fn.gemm(sv["g"], w.w_gate, b_mn_major=True, out=self._buf("bw_xn_p", M, s.hidden_size))
        d_xn2 = Fn.gemm(sv["u"], w.w_up, b_mn_major=True, residual=d_xn2, out=d_xn2)
        d_h1 = Fn.rmsnorm_bwd(d_xn2, sv["h1"], w.ln2_w, s.norm_eps, d_res=dy)
        d_attn = Fn.gemm(d_h1, w.wo, b_mn_major=True)
        dq, dk, dv = Fn.attention_bwd(sv["q"], sv["k_pool"], sv["v_pool"], table, sv["attn"], d_attn, sv["lse"], B=nb, T=T, Hq=s.num_heads,
                                      Hkv=s.num_kv_heads, D=s.head_dim, scale=s.attn_scale)
        d_qkv = Fn.qkv_grad_merge(dq, dk, dv, self.cos, self.sin, T=T, Hq=s.num_heads, Hkv=s.num_kv_heads, D=s.head_dim,
                                  out=self._buf("bw_qkv_p", M, s.qkv_dim))
        d_xn1 = Fn.gemm(d_qkv, w.wqkv, b_mn_major=True, out=d_xn2)
        return Fn.rmsnorm_bwd(d_xn1, sv["x"], w.ln1_w, s.norm_eps, d_res=d_h1, out=out)

    def backward(self, hidden: torch.Tensor, grad_out: torch.Tensor, prompts: Optional[Sequence[Optional[torch.Tensor]]] = None,
                 block_range: Optional[Tuple[int, int]] = None, grad_hop: Optional[tuple] = None,
                 grad_ack: Optional[tuple] = None) -> Tuple[torch.Tensor, List[Optional[torch.Tensor]]]:
        """``rpc_backward`` of blocks [lo, hi) on the kernels (reference: src/petals/server/block_functions.py:84-141). One forward that
        saves the per-block intermediates, then the blocks' backward in reverse order — or, when the saved tensors of the whole
        span would not fit the budget, the reference's schedule: remember the block inputs, recompute one block at a time.

        The gradient hop (parallel/fabric.py, kind "g_in"): ``grad_out`` may be the rows of this rank's landing slot, read in place —
        ``grad_ack = (fabric, kind, src_rank, slot)`` acknowledges the slot once the last kernel reading it is enqueued; with
        ``grad_hop = (fabric, kind, rank[, slot])`` the last kernel of the first block's backward (RMSNorm backward + residual gradient)
        stores dL/d(span input) straight into the previous stage's landing slot and the returned tensor is empty."""
        lo, hi = block_range or (0, self.n_blocks)
        B, T, H = hidden.shape
        grad_prompts: List[Optional[torch.Tensor]] = [None] * (hi - lo)
        if B == 0 or T == 0:
            return grad_out, grad_prompts
        hidden, grad_out = hidden.to(self.dtype), grad_out.to(self.dtype)
        s = self.spec
        if hi <= lo:
            grad_hop = self._finish_grad_hop(grad_out.reshape(B * T, H), grad_hop, grad_ack)
            return (grad_out if grad_hop is None else grad_out.new_empty(0)), grad_prompts
        pages_per_seq = (T + PAGE - 1) // PAGE
        per_token = 2 * (3 * s.hidden_size + 2 * s.num_heads * s.head_dim + 2 * s.num_kv_heads * s.head_dim + 2 * s.intermediate_size)
        budget = float(os.environ.get("PETALS_B200_BWD_SAVE_GB", "16")) * 2 ** 30
        if pages_per_seq > self._scratch_pages:
            raise ValueError(f"sequence of {T} tokens exceeds max_chunk_tokens={self.max_chunk_tokens} for a backward pass")
        rows_per_group = max(1, min(B, self._scratch_pages // pages_per_seq))
        first_prompt = prompts is not None and prompts[0] is not None and not is_dummy(prompts[0])
        fused_hop = grad_hop is not None and rows_per_group >= B and not first_prompt  # the prompt gradient is sliced from d: keep it local
        grad_in = torch.empty_like(hidden) if not fused_hop else None
        zero = torch.zeros(1, dtype=torch.int32, device=self.device)
        for b0 in range(0, B, rows_per_group):
            b1 = min(B, b0 + rows_per_group)
            nb, M = b1 - b0, (b1 - b0) * T
            table = torch.arange(nb * pages_per_seq, dtype=torch.int32, device=self.device).view(nb, pages_per_seq).contiguous()
            keep_all = per_token * M * (hi - lo) <= budget
            pr = [None if (prompts is None or prompts[i] is None or is_dummy(prompts[i])) else (prompts[i] if prompts[i].shape[0] == 1 else prompts[i][b0:b1])
                  for i in range(hi - lo)]
            x = hidden[b0:b1].reshape(M, H).clone()
            saves: List[object] = []
            for slot in range(lo, hi):
                if pr[slot - lo] is not None:
                    Fn.add_prompts(x.view(nb, T, H), pr[slot - lo].to(self.dtype).contiguous())
                if keep_all:
                    x, sv = self._forward_saving(x, slot, nb, T, table, zero.data_ptr())
                    saves.append(sv)
                else:
                    saves.append(x)  # the block input (prompt included); everything else is recomputed when its turn comes
                    if slot + 1 < hi:
                        x = self._run_span(x.clone(), nb, T, slot, slot + 1, table, zero.data_ptr(),
                                           lambda _slot: (self._scratch_pool[0], self._scratch_pool[1]), None, False, 1).clone()
            d = grad_out[b0:b1].reshape(M, H).contiguous()
            for slot in reversed(range(lo, hi)):
                sv = saves.pop()
                if not keep_all:
                    _, sv = self._forward_saving(sv, slot, nb, T, table, zero.data_ptr())
                dst = None
                if fused_hop and slot == lo:
                    dst = grad_hop[0].open_push(M, grad_hop[2], grad_hop[1], *grad_hop[3:4])
                d = self._backward_block(d, sv, slot, nb, T, table, out=dst)
                if slot == hi - 1 and b1 == B and grad_ack is not None:  # the landing slot holding grad_out has been read for the last time
                    grad_ack[0].acknowledge(*grad_ack[1:])
                    grad_ack = None
                if dst is not None:
                    grad_hop[0].publish(grad_hop[2], grad_hop[1], *grad_hop[3:4])
                p = pr[slot - lo]
                if p is not None:
                    gp = d.view(nb, T, H)[:, : p.shape[1]]
                    gp = gp.sum(0, keepdim=True) if p.shape[0] == 1 else gp
                    if p.shape[0] == 1:
                        grad_prompts[slot - lo] = gp.clone() if grad_prompts[slot - lo] is None else grad_prompts[slot - lo] + gp
                    else:
                        if grad_prompts[slot - lo] is None:
                            grad_prompts[slot - lo] = torch.zeros(B, p.shape[1], H, dtype=self.dtype, device=self.device)
                        grad_prompts[slot - lo][b0:b1] = gp
            if grad_in is not None:
                grad_in[b0:b1] = d.view(nb, T, H)
        self._active = None
        if fused_hop:
            return hidden.new_empty(0), grad_prompts
        if grad_hop is not None:
            self._finish_grad_hop(grad_in.view(B * T, H), grad_hop, None)
            return hidden.new_empty(0), grad_prompts
        return grad_in, grad_prompts

    @staticmethod
    def _finish_grad_hop(rows: torch.Tensor, grad_hop: Optional[tuple], grad_ack: Optional[tuple]) -> Optional[tuple]:
        """The unfused tail of a gradient hop: a peer copy of finished rows, then the acknowledgement of the slot they came from."""
        if grad_hop is not None:
            grad_hop[0].send(rows, grad_hop[2], grad_hop[1], *grad_hop[3:4])
        if grad_ack is not None:
            grad_ack[0].acknowledge(*grad_ack[1:])
        return grad_hop

    def check_errors(self) -> None:
        code = int(self.err_flag.item())
        if code:
            self.err_flag.zero_()
            raise RuntimeError(f"device-side error flag {code} (1 = peer flag watchdog, 2 = KV page table overflow)")
