"""Tensor parallelism inside a stage: one process per GPU, fused compute + NVLink collectives.

The reference delegates intra-server TP to the ``tensor_parallel`` package: one Python thread per device and an
NCCL/``torch.cuda.comm`` all-reduce after every row-parallel linear (src/petals/utils/convert_block.py:118-135,
SURVEY.md §2.4 X5). Here a TP group is N worker *processes* (rank = GPU) sharing a symmetric heap:

* column-parallel projections (QKV, gate/up) need no communication;
* every row-parallel projection (attention out, MLP down) is a weight-streaming GEMV whose **epilogue stores its
  partial result straight into all peers' HBM over NVLink** and publishes one flag per peer; the *next* kernel
  (fused norm + column-parallel GEMV) **waits on the flag, sums the N partials + residual in its prologue** and goes
  on. That is a one-shot all-reduce with zero extra launches, zero NCCL calls and no host involvement — per layer
  the critical path sees two flag waits (~NVLink latency) instead of two all-reduce kernels;
* KV caches, attention heads and FFN columns are sharded; norms and the residual stream are replicated.

Control plane: the leader (rank 0 of the group, the process that owns the swarm endpoint) broadcasts tiny step
commands through a shared-memory ring (``parallel/control.py``); followers replay the same CUDA graph. Every rank
bumps a device-resident epoch per step; flag targets are ``epoch * n_sources`` so nothing is ever reset.
"""
from __future__ import annotations

import dataclasses
import os
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from petals_b200.models.block_oracle import GenericBlock
from petals_b200.models.spec import BlockSpec
from petals_b200.ops import functional as Fn
from petals_b200.ops import native
from petals_b200.parallel.symmetric import SymmetricHeap, ptr_array
from petals_b200.server.memory_cache import MemoryCache, SessionCache
from petals_b200.utils.logging import get_logger

logger = get_logger(__name__)
MAX_ROWS = 8


def tp_supported(spec: BlockSpec, world: int) -> bool:
    """Layouts the NVLink engine shards itself. Everything else (biases on the projections, ALiBi, fused interleaved QKV, parallel
    attention) is split by the generic path (parallel/tp_generic.py) — `shard_block` below carries no bias tensors. Sparse-MoE blocks
    (Mixtral) are sharded along every expert's FFN dimension with the router replicated."""
    if spec.mlp == "moe" and not (spec.norm == "rms" and 0 < spec.num_experts <= 64 and 0 < spec.top_k <= 8):
        return False
    return (spec.mlp in ("swiglu", "gelu", "moe") and not spec.parallel_attn and not spec.qkv_interleaved and not spec.post_ln_residual
            and not (spec.qkv_bias or spec.out_bias or spec.mlp_bias) and not spec.alibi
            and spec.num_kv_heads % world == 0 and spec.num_heads % world == 0 and spec.intermediate_size % (2 * world) == 0
            and spec.head_dim in (64, 128))


def local_spec(spec: BlockSpec, world: int) -> BlockSpec:
    """The shard's view: 1/world of the heads and FFN columns, full hidden size."""
    return dataclasses.replace(spec, num_heads=spec.num_heads // world, num_kv_heads=spec.num_kv_heads // world,
                               intermediate_size=spec.intermediate_size // world)


def shard_block(block: GenericBlock, spec: BlockSpec, rank: int, world: int, device) -> Dict[str, torch.Tensor]:
    """Megatron-style split of one block's canonical tensors (column-parallel rows / row-parallel columns)."""
    D = spec.head_dim
    hq, hkv, I = spec.num_heads // world, spec.num_kv_heads // world, spec.intermediate_size // world
    q0, k0, v0 = 0, spec.num_heads * D, (spec.num_heads + spec.num_kv_heads) * D
    w = block.wqkv
    out = {
        "wqkv": torch.cat([w[q0 + rank * hq * D: q0 + (rank + 1) * hq * D], w[k0 + rank * hkv * D: k0 + (rank + 1) * hkv * D],
                           w[v0 + rank * hkv * D: v0 + (rank + 1) * hkv * D]], 0),
        "wo": block.wo[:, rank * hq * D: (rank + 1) * hq * D],
        "ln1_w": block.ln1_w, "ln2_w": block.ln2_w,
    }
    if spec.mlp == "moe":  # every rank holds 1/world of EVERY expert's FFN columns; the router is replicated
        out.update(router=block.router, we_gate=block.we_gate[:, rank * I: (rank + 1) * I], we_up=block.we_up[:, rank * I: (rank + 1) * I],
                   we_down=block.we_down[:, :, rank * I: (rank + 1) * I])
    else:
        out.update(w_down=block.w_down[:, rank * I: (rank + 1) * I], w_up=block.w_up[rank * I: (rank + 1) * I])
    if spec.mlp == "swiglu":
        out["w_gate"] = block.w_gate[rank * I: (rank + 1) * I]
    for name in ("ln1_b", "ln2_b"):
        if getattr(block, name, None) is not None:
            out[name] = getattr(block, name)
    return {k: v.detach().to(device).contiguous() for k, v in out.items()}


def random_shard(spec: BlockSpec, rank: int, world: int, layer: int, device, seed: int = 0, std: float = 0.02) -> Dict[str, torch.Tensor]:
    """A random shard generated in place (benchmarks: the full 140 GB model never exists anywhere)."""
    ls = local_spec(spec, world)
    g = torch.Generator(device=device).manual_seed(seed * 1000003 + layer * 64 + rank)
    H = spec.hidden_size

    def rnd(*shape):
        return (torch.randn(*shape, device=device, dtype=torch.float32, generator=g) * std).to(torch.bfloat16)

    out = {"wqkv": rnd(ls.qkv_dim, H), "wo": rnd(H, ls.num_heads * ls.head_dim), "ln1_w": torch.ones(H, device=device, dtype=torch.bfloat16),
           "ln2_w": torch.ones(H, device=device, dtype=torch.bfloat16)}
    if spec.mlp == "moe":
        E, I = spec.num_experts, ls.intermediate_size
        # the router must be IDENTICAL on every rank: its own generator, seeded without the rank
        gr = torch.Generator(device=device).manual_seed(seed * 1000003 + layer * 64 + 63)
        out.update(router=(torch.randn(E, H, device=device, dtype=torch.float32, generator=gr) * std).to(torch.bfloat16),
                   we_gate=rnd(E, I, H), we_up=rnd(E, I, H), we_down=rnd(E, H, I))
    else:
        out.update(w_up=rnd(ls.intermediate_size, H), w_down=rnd(H, ls.intermediate_size))
    if spec.mlp == "swiglu":
        out["w_gate"] = rnd(ls.intermediate_size, H)
    if spec.norm == "layer":
        out["ln1_b"] = torch.zeros(H, device=device, dtype=torch.bfloat16)
        out["ln2_b"] = torch.zeros(H, device=device, dtype=torch.bfloat16)
    return out


def prefill_heap_bytes(hidden_size: int, world: int, n_blocks: int, max_prefill_rows: int) -> int:
    """Symmetric-heap bytes the sequence-parallel prefill path needs (landing zone, partial slots, activations, output, flags)."""
    if max_prefill_rows <= 0:
        return 0
    mo = (max_prefill_rows + world - 1) // world
    row = hidden_size * 2
    return (mo + world * mo + 2 * max_prefill_rows) * row + (4 * n_blocks + 4) * 8 + 8 * 4096


class TPDecodeEngine:
    """Executes a span of blocks sharded over a TP group.

    * decode-shaped steps (B*T <= 8 rows): weight-streaming GEMVs with the all-reduce fused into epilogue + next prologue;
    * prefill-shaped steps (up to ``max_prefill_rows`` rows): sequence-parallel tcgen05 GEMMs whose epilogue performs the
      reduce-scatter over NVLink and whose successor norm kernel performs the all-gather (csrc/seq_parallel.cu)."""

    def __init__(self, spec: BlockSpec, shards: Sequence[Dict[str, torch.Tensor]], heap: SymmetricHeap, cache: MemoryCache, *,
                 use_cuda_graphs: bool = True, max_prefill_rows: int = 4096):
        self.spec, self.shards, self.heap, self.cache = spec, list(shards), heap, cache
        self.rank, self.world = heap.rank, heap.world
        self.ls = local_spec(spec, self.world)
        self.device = heap.device
        self.n_blocks = len(self.shards)
        self.use_cuda_graphs = use_cuda_graphs
        H = spec.hidden_size
        self.norm_kind = Fn.NORM_RMS if spec.norm == "rms" else Fn.NORM_LAYER
        self.act = Fn.ACT_SWIGLU if spec.mlp == "swiglu" else (Fn.ACT_GELU_TANH if spec.gelu_tanh else Fn.ACT_GELU_ERF)
        self.cos = self.sin = None
        if spec.rotary:
            self.cos, self.sin = Fn.rope_tables(spec.head_dim, spec.max_position, spec.rope_theta, spec.rope_scaling, device=self.device)
        self.sms = native.sm_count(self.device.index)
        # ---- symmetric allocations (identical order on every rank) ----------------------------------------------
        R, L = self.world, self.n_blocks
        self.slot_bytes = MAX_ROWS * H * 2
        self.off_x_in = heap.alloc(self.slot_bytes)
        self.off_parts_attn = heap.alloc(R * self.slot_bytes)
        self.off_parts_mlp = heap.alloc(R * self.slot_bytes)
        self.off_flags = heap.alloc((2 * L + 2) * 8)
        # LL all-reduce buffers: [source rank][MAX_ROWS, H/2] x 8-byte {2 x bf16, tag} units (twice the payload bytes)
        self.use_ll = os.environ.get("PETALS_B200_TP_LL", "1") != "0"
        self.ll_slot_bytes = MAX_ROWS * H * 4
        self.off_ll_attn = heap.alloc(R * self.ll_slot_bytes, align=4096)
        self.off_ll_mlp = heap.alloc(R * self.ll_slot_bytes, align=4096)
        self.x_in = heap.tensor(self.off_x_in, (MAX_ROWS, H), torch.bfloat16)
        # single-token steps: the whole span as ONE persistent data-flow kernel per rank (csrc/decode_span.cu). Its two all-reduce
        # buffers are [source rank][H/2] 8-byte LL units on every rank (allocated unconditionally: symmetric order).
        self.span_slot_bytes = H * 4
        self.off_span_attn = heap.alloc(R * self.span_slot_bytes, align=4096)
        self.off_span_mlp = heap.alloc(R * self.span_slot_bytes, align=4096)
        ls_ = self.ls
        self.use_span_kernel = (os.environ.get("PETALS_B200_SPAN_KERNEL", "1") != "0" and self.use_ll and spec.norm == "rms" and spec.mlp == "swiglu" and spec.rotary
                                and not spec.sliding_window
                                and Fn.decode_span_supported(H=H, Hq=ls_.num_heads, Hkv=ls_.num_kv_heads, D=ls_.head_dim, I=ls_.intermediate_size))
        self._span_plan: Optional[Fn.DecodeSpanPlan] = None
        # sequence-parallel prefill: rows are owned in contiguous slices of `mo` rows per rank
        self.max_prefill_rows = P = max(0, max_prefill_rows)
        if P:
            self.p_mo_max = (P + R - 1) // R
            self.p_slot_bytes = self.p_mo_max * H * 2
            self.off_p_x_in = heap.alloc(self.p_slot_bytes, align=4096)        # my residual rows, scattered by the leader
            self.off_p_parts = heap.alloc(R * self.p_slot_bytes, align=4096)    # [src rank][my rows, H] GEMM-epilogue partials
            self.off_p_xn = heap.alloc(P * H * 2, align=4096)                   # all rows, normalised (all-gathered)
            self.off_p_out = heap.alloc(P * H * 2, align=4096)                  # span output, gathered on the leader
            self.off_p_flags = heap.alloc((4 * L + 4) * 8)
            self.p_xn = heap.tensor(self.off_p_xn, (P, H), torch.bfloat16)
            self.p_out = heap.tensor(self.off_p_out, (P, H), torch.bfloat16)
            self.p_x_in = heap.tensor(self.off_p_x_in, (self.p_mo_max, H), torch.bfloat16)
        # ---- local state ----------------------------------------------------------------------------------------------
        dev = self.device
        self.epoch = torch.zeros(1, dtype=torch.int64, device=dev)
        self.epoch_p = torch.zeros(1, dtype=torch.int64, device=dev)  # prefill steps count their own epochs (own flag set)
        # Counter flags target `epoch * sources`, so every step that bumps an epoch must also feed every flag waiting on it. The span
        # kernel feeds only the step-input flag (its partial sums travel as tagged LL units), so the multi-launch path counts the steps
        # of the flag that only IT feeds (last block's MLP partials -> final reduce) in an epoch of its own.
        self.epoch_f = torch.zeros(1, dtype=torch.int64, device=dev) if self.use_span_kernel else self.epoch
        self.err = torch.zeros(1, dtype=torch.int32, device=dev)
        self.done_counter = torch.zeros(1, dtype=torch.int32, device=dev)
        self.fuse_rope = os.environ.get("PETALS_B200_FUSE_ROPE", "1") != "0"
        self._split_ctr = torch.zeros(1024, dtype=torch.int32, device=dev)  # split-KV arrival counters (self-resetting)
        self._moe_bufs: Dict[object, torch.Tensor] = {}  # sparse-MoE scratch (ops/functional.py: moe_decode / moe_prefill)
        self.pos_static = torch.zeros(1, dtype=torch.int32, device=dev)
        self.max_pages = cache.max_pages_per_seq
        self._tables: Dict[int, torch.Tensor] = {}
        self._graphs: Dict[Tuple[int, int], dict] = {}
        self._bufs: Dict[tuple, torch.Tensor] = {}
        self._active: Optional[SessionCache] = None
        self._dev_pos = -1
        self.out = torch.zeros(MAX_ROWS, H, dtype=torch.bfloat16, device=dev)

    # ---- addresses -------------------------------------------------------------------------------------------------
    def flag(self, rank: int, index: int) -> int:
        return self.heap.addr(rank, self.off_flags + 8 * index)

    def flag_attn(self, rank: int, layer: int) -> int:
        return self.flag(rank, 2 + 2 * layer)

    def flag_mlp(self, rank: int, layer: int) -> int:
        return self.flag(rank, 3 + 2 * layer)

    def parts(self, off: int, owner: int, src: int) -> int:
        return self.heap.addr(owner, off + src * self.slot_bytes)

    def _buf(self, name: str, rows: int, cols: int, dtype=torch.bfloat16) -> torch.Tensor:
        # keyed by the full shape and never replaced: captured CUDA graphs keep the raw addresses of these buffers
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

    # ---- one decode step of the whole span (launch sequence; captured into a graph) ------------------------------------
    def _launch_span(self, B: int, T: int, table: torch.Tensor, final_reduce: bool) -> torch.Tensor:
        s, ls, R, me = self.spec, self.ls, self.world, self.rank
        M, H = B * T, s.hidden_size
        eps = s.norm_eps
        ep, err, ctr = self.epoch.data_ptr(), self.err.data_ptr(), self.done_counter.data_ptr()
        pos_ptr = self.pos_static.data_ptr()
        native.check(native.lib().pb_bump_epoch(ep, native.stream_ptr()), "bump_epoch")
        if M == 1 and self.use_span_kernel:
            # one launch for the whole span: waits for the leader's input flag, streams this rank's shards, pushes the partial sums of
            # both row-parallel projections to every rank and finishes the all-reduces itself (the span output lands in self.out)
            Fn.decode_span(self._span_kernel_plan(), self.x_in[:1], self.out[:1], table, pos_ptr, self.cos, self.sin,
                           in_flag=self.flag(me, 0), in_per_epoch=1, bump_epoch=False)
            native.check(native.lib().pb_advance_pos(pos_ptr, T, native.stream_ptr()), "advance_pos")
            return self.out[:M]
        ep_f = self.epoch_f.data_ptr()
        if ep_f != ep:
            native.check(native.lib().pb_bump_epoch(ep_f, native.stream_ptr()), "bump_epoch")
        h = [self._buf("h_a", M, H), self._buf("h_b", M, H)]
        cur = self.x_in[:M]  # residual stream entering layer 0 (pushed by the leader)
        nxt = 0
        qkv_buf = self._buf("qkv", M, ls.qkv_dim)
        q_buf = self._buf("q", M, ls.num_heads * ls.head_dim)
        attn = self._buf("attn", M, ls.num_heads * ls.head_dim)
        act = self._buf("act", M, ls.intermediate_size)
        splits = int(min(16, max(1, (2 * self.sms) // max(1, B * ls.num_kv_heads))))
        po = self._buf("po", splits * M * ls.num_heads, ls.head_dim, torch.float32) if splits > 1 else None
        pl = self._buf("pl", splits, M * ls.num_heads, torch.float32) if splits > 1 else None
        attn_parts = [self.parts(self.off_parts_attn, me, r) for r in range(R)]
        mlp_parts = [self.parts(self.off_parts_mlp, me, r) for r in range(R)]
        # LL protocol (default): partials travel as {payload, tag} units, consumers poll the payload; the flag protocol stays for
        # the step input and for the last layer's MLP (its consumer is the final reduce kernel)
        L, ll = self.n_blocks, self.use_ll
        ll_attn_in = [self.heap.addr(me, self.off_ll_attn + r * self.ll_slot_bytes) for r in range(R)]
        ll_mlp_in = [self.heap.addr(me, self.off_ll_mlp + r * self.ll_slot_bytes) for r in range(R)]
        ll_attn_out = [self.heap.addr(r, self.off_ll_attn + me * self.ll_slot_bytes) for r in range(R)]
        ll_mlp_out = [self.heap.addr(r, self.off_ll_mlp + me * self.ll_slot_bytes) for r in range(R)]
        split_ctr = self._split_ctr if splits > 1 and B * ls.num_kv_heads <= 1024 else None

        def k1_kwargs(l: int, cur, nxt):
            """[all-reduce tail of the previous MLP] + norm + column-parallel QKV; the epilogue rotates q/k and appends k/v to this
            rank's cache pages. Returns (kwargs, residual buffer after the call, next ping-pong index)."""
            w, pools = self.shards[l], self.cache.layer_pools(l)
            kw = dict(x=cur, w=w["wqkv"], norm_weight=w["ln1_w"], norm_bias=w.get("ln1_b"), norm_kind=self.norm_kind, eps=eps, epoch=ep, error_flag=err)
            if self.fuse_rope:
                kw["rope"] = dict(q_out=q_buf, k_pool=pools[0], v_pool=pools[1], block_table=table, pos_ptr=pos_ptr, cos=self.cos, sin=self.sin, T=T,
                                  Hq=ls.num_heads, Hkv=ls.num_kv_heads, D=ls.head_dim)
            else:
                kw["out"] = qkv_buf
            if l == 0:
                kw.update(wait_flag=self.flag(me, 0), wait_per_epoch=1)
                return kw, cur, nxt
            kw.update(dict(ll_parts=ll_mlp_in, ll_tag=(L, l - 1)) if ll else dict(parts=mlp_parts, wait_flag=self.flag_mlp(me, l - 1), wait_per_epoch=R))
            kw["x_out"] = h[nxt]
            return kw, h[nxt], nxt ^ 1

        def launch(kw: dict):
            kw = dict(kw)
            return Fn.linear_decode(kw.pop("x"), kw.pop("w"), **kw)

        kw1, cur, nxt = k1_kwargs(0, cur, nxt)
        launch(kw1)
        for l, w in enumerate(self.shards):
            pools = self.cache.layer_pools(l)
            if not self.fuse_rope:
                Fn.rope_kv_append(qkv_buf, q_buf, pools[0], pools[1], table, pos_ptr, self.cos, self.sin, B=B, T=T, Hq=ls.num_heads,
                                  Hkv=ls.num_kv_heads, D=ls.head_dim, error_flag=err)
            Fn.paged_attention(q_buf, pools[0], pools[1], table, pos_ptr, attn, B=B, T=T, Hq=ls.num_heads, Hkv=ls.num_kv_heads, D=ls.head_dim,
                               scale=s.attn_scale, splits=splits, partial_o=po, partial_lse=pl, window=s.sliding_window, split_counter=split_ctr)
            # K2: row-parallel O-projection; the epilogue sends this rank's partial to every rank's slot [me]
            if ll:
                k2 = dict(x=attn, w=w["wo"], store_local=False, ll_push=ll_attn_out, ll_tag=(L, l), epoch=ep, error_flag=err)
            else:
                k2 = dict(x=attn, w=w["wo"], store_local=False, push_out=[self.parts(self.off_parts_attn, r, me) for r in range(R)],
                          push_flag=[self.flag_attn(r, l) for r in range(R)], done_counter=ctr, error_flag=err)
            if s.mlp == "moe":
                # sparse MoE: no single GEMV consumes / produces the all-reduced vectors, so the two halves of the LL all-reduce run as
                # their own small kernels (csrc/ll_collectives.cu) around the device-routed expert GEMVs (csrc/moe.cu). Every rank sums
                # the partials in the same order -> bit-identical h1 -> identical routing on every rank.
                launch(k2)
                h1 = h[nxt]
                if ll:
                    Fn.ll_reduce(cur, ll_attn_in, (L, l), ep, h1, err)
                else:
                    native.check(native.lib().pb_reduce_parts(cur.data_ptr(), ptr_array(attn_parts), R, self.flag_attn(me, l), R, ep, h1.data_ptr(),
                                                              M * H * 2, err, native.stream_ptr()), "reduce_parts")
                cur, nxt = h1, nxt ^ 1
                part = Fn.moe_decode(cur, w["ln2_w"], w["router"], w["we_gate"], w["we_up"], w["we_down"], top_k=s.top_k, eps=eps,
                                     out=self._buf("moe_part", M, H), bufs=self._moe_bufs, add_residual=False)
                if ll and l + 1 < L:
                    Fn.ll_push(part, ll_mlp_out, (L, l), ep)
                else:
                    native.check(native.lib().pb_push_rows(part.data_ptr(), ptr_array([self.parts(self.off_parts_mlp, r, me) for r in range(R)]),
                                                           ptr_array([self.flag_mlp(r, l) for r in range(R)]), R, M * H * 2, native.stream_ptr()), "push_rows")
                if l + 1 < L:
                    kw1, cur, nxt = k1_kwargs(l + 1, cur, nxt)
                    launch(kw1)
                continue
            # K3: [all-reduce tail of attention] + norm + column-parallel gate/up (+SwiGLU)
            k3 = dict(x=cur, norm_weight=w["ln2_w"], norm_bias=w.get("ln2_b"), norm_kind=self.norm_kind, eps=eps, out=act, epoch=ep, x_out=h[nxt],
                      error_flag=err)
            k3.update(dict(ll_parts=ll_attn_in, ll_tag=(L, l)) if ll else dict(parts=attn_parts, wait_flag=self.flag_attn(me, l), wait_per_epoch=R))
            k3.update(dict(w=w["w_gate"], w2=w["w_up"], act=Fn.ACT_SWIGLU) if s.mlp == "swiglu" else dict(w=w["w_up"], act=self.act))
            cur, nxt = h[nxt], nxt ^ 1
            # K4: row-parallel down projection, sent like K2 (the last block uses the flag protocol: its consumer is the final reduce)
            if ll and l + 1 < L:
                k4 = dict(x=act, w=w["w_down"], store_local=False, ll_push=ll_mlp_out, ll_tag=(L, l), epoch=ep, error_flag=err)
            else:
                k4 = dict(x=act, w=w["w_down"], store_local=False, push_out=[self.parts(self.off_parts_mlp, r, me) for r in range(R)],
                          push_flag=[self.flag_mlp(r, l) for r in range(R)], done_counter=ctr, error_flag=err)
            for kw in (k2, k3, k4):
                launch(kw)
            if l + 1 < L:
                kw1, cur, nxt = k1_kwargs(l + 1, cur, nxt)
                launch(kw1)
        if final_reduce:
            parts = ptr_array(mlp_parts)
            native.check(native.lib().pb_reduce_parts(cur.data_ptr(), parts, R, self.flag_mlp(me, self.n_blocks - 1), R, ep_f, self.out.data_ptr(),
                                                      M * H * 2, err, native.stream_ptr()), "reduce_parts")
        native.check(native.lib().pb_advance_pos(pos_ptr, T, native.stream_ptr()), "advance_pos")
        self._last_residual, self._last_parts = cur, mlp_parts
        return self.out[:M]

    def _span_kernel_plan(self) -> "Fn.DecodeSpanPlan":
        if self._span_plan is None:
            s, ls, R, me = self.spec, self.ls, self.world, self.rank
            layers = []
            for l, w in enumerate(self.shards):
                k_pool, v_pool = self.cache.layer_pools(l)
                layers.append(dict(wqkv=w["wqkv"], wo=w["wo"], w_gate=w["w_gate"], w_up=w["w_up"], w_down=w["w_down"], ln1_w=w["ln1_w"],
                                   ln2_w=w["ln2_w"], k_pool=k_pool, v_pool=v_pool))
            # PETALS_B200_SPAN_NVLS: "0" = unicast peer stores; "st" = one multimem.st per partial (NVSwitch replicates it into every
            # rank's slot); "reduce" = partials stay local, the slice owners multimem.ld_reduce them (in-switch sum). Needs the
            # heap's multicast mapping (parallel/symmetric.py); without it every mode degrades to unicast.
            # Default = what measured fastest on B200 boxes (profiles/r2_2gpu_selftests_and_bench.txt, r2_8gpu_bench_selftests_pipeline.txt):
            # 2 ranks: multimem.st 13.47 ms/token vs 13.59 unicast; 8 ranks: unicast 6.89 vs 7.06 for multimem.st.
            mode = os.environ.get("PETALS_B200_SPAN_NVLS", "st" if R <= 2 else "0").lower()
            mc = getattr(self.heap, "multicast_ptr", 0)
            nvls = None
            push = lambda off: [self.heap.addr(r, off + me * self.span_slot_bytes) for r in range(R)]
            push_attn, push_mlp = push(self.off_span_attn), push(self.off_span_mlp)
            if mc and R > 1 and mode == "st":
                nvls = dict(mode="st", oproj=self.heap.mc_addr(self.off_span_attn + me * self.span_slot_bytes),
                            mlp=self.heap.mc_addr(self.off_span_mlp + me * self.span_slot_bytes))
            elif mc and R > 1 and mode == "reduce":
                nvls = dict(mode="reduce", oproj=self.heap.mc_addr(self.off_span_attn), mlp=self.heap.mc_addr(self.off_span_mlp))
                push_attn, push_mlp = [self.heap.addr(me, self.off_span_attn)], [self.heap.addr(me, self.off_span_mlp)]
            self.span_nvls_mode = nvls["mode"] if nvls else "unicast"
            self._span_plan = Fn.DecodeSpanPlan(
                layers, H=s.hidden_size, Hq=ls.num_heads, Hkv=ls.num_kv_heads, D=ls.head_dim, I=ls.intermediate_size, eps=s.norm_eps,
                attn_scale=s.attn_scale, max_chunks=self.max_pages, device=self.device, R=R, rank=me,
                oproj=(push_attn, self.heap.addr(me, self.off_span_attn)), mlp=(push_mlp, self.heap.addr(me, self.off_span_mlp)),
                epoch=self.epoch, error_flag=self.err, nvls=nvls)
        return self._span_plan

    # ---- sequence-parallel prefill ---------------------------------------------------------------------------------------
    def p_flag(self, rank: int, index: int) -> int:
        return self.heap.addr(rank, self.off_p_flags + 8 * index)

    def _p_layer_flag(self, rank: int, layer: int, which: int) -> int:
        """which: 0 = xn ready (input of QKV), 1 = attention partials landed, 2 = xn2 ready (input of gate/up), 3 = MLP partials landed."""
        return self.p_flag(rank, 4 + 4 * layer + which)

    def _launch_prefill(self, B: int, T: int, table: torch.Tensor) -> torch.Tensor:
        """One prompt chunk of M = B*T rows through the whole span. Per layer and rank: 4 tcgen05 GEMMs, RoPE+KV append, flash
        attention and 2 norm_reduce_gather kernels; the two reduce-scatters ride in GEMM epilogues, the two all-gathers in the norm
        kernels; every wait is a flag spin in the consumer's prologue."""
        s, ls, R, me = self.spec, self.ls, self.world, self.rank
        M, H = B * T, s.hidden_size
        if M > self.max_prefill_rows:
            raise ValueError(f"{M} rows exceed max_prefill_rows={self.max_prefill_rows}")
        mo = (M + R - 1) // R
        my_rows = max(0, min(mo, M - me * mo))
        eps, L = s.norm_eps, self.n_blocks
        ep, err, ctr = self.epoch_p.data_ptr(), self.err.data_ptr(), self.done_counter.data_ptr()
        pos_ptr = self.pos_static.data_ptr()
        native.check(native.lib().pb_bump_epoch(ep, native.stream_ptr()), "bump_epoch")
        x_res = self._buf("p_res", self.p_mo_max, H)
        xn = self.p_xn[:M]
        qkv_buf = self._buf("p_qkv", M, ls.qkv_dim)
        q_buf = self._buf("p_q", M, ls.num_heads * ls.head_dim)
        attn = self._buf("p_attn", M, ls.num_heads * ls.head_dim)
        act = self._buf("p_act", M, ls.intermediate_size)
        row_b = H * 2
        my_parts = [self.heap.addr(me, self.off_p_parts + r * self.p_slot_bytes) for r in range(R)]
        push_parts = [self.heap.addr(r, self.off_p_parts + me * self.p_slot_bytes) for r in range(R)]  # my slot in every owner's buffer
        gather_xn = [self.heap.addr(r, self.off_p_xn + me * mo * row_b) for r in range(R)]
        dev = self.device.index
        common = dict(rows=my_rows, H=H, eps=eps, epoch=ep, done_counter=ctr, error_flag=err, device_index=dev)
        w0 = self.shards[0]
        # layer-0 prologue: my slice of the chunk (scattered by the leader) becomes the residual; its norm is all-gathered
        Fn.norm_reduce_gather(self.p_x_in, x_res, norm_weight=w0["ln1_w"], norm_bias=w0.get("ln1_b"), norm_kind=self.norm_kind,
                              gather_out=gather_xn, gather_flag=[self._p_layer_flag(r, 0, 0) for r in range(R)],
                              wait_flag=self.p_flag(me, 0), wait_per_epoch=1, **common)
        for l, w in enumerate(self.shards):
            pools = self.cache.layer_pools(l)
            Fn.gemm(xn, w["wqkv"], out=qkv_buf, wait_flag=self._p_layer_flag(me, l, 0), wait_per_epoch=R, epoch=ep, error_flag=err)
            Fn.rope_kv_append(qkv_buf, q_buf, pools[0], pools[1], table, pos_ptr, self.cos, self.sin, B=B, T=T, Hq=ls.num_heads,
                              Hkv=ls.num_kv_heads, D=ls.head_dim, error_flag=err)
            Fn.paged_attention(q_buf, pools[0], pools[1], table, pos_ptr, attn, B=B, T=T, Hq=ls.num_heads, Hkv=ls.num_kv_heads, D=ls.head_dim,
                               scale=s.attn_scale, splits=1, window=s.sliding_window)
            # row-parallel O-projection; the epilogue IS the reduce-scatter (row r -> owner r // mo, slot [me])
            Fn.gemm(attn, w["wo"], store_local=False, push_out=push_parts, push_rows_per_owner=mo,
                    push_done_flag=[self._p_layer_flag(r, l, 1) for r in range(R)], done_counter=ctr, error_flag=err)
            Fn.norm_reduce_gather(x_res, x_res, parts=my_parts, norm_weight=w["ln2_w"], norm_bias=w.get("ln2_b"), norm_kind=self.norm_kind,
                                  gather_out=gather_xn, gather_flag=[self._p_layer_flag(r, l, 2) for r in range(R)],
                                  wait_flag=self._p_layer_flag(me, l, 1), wait_per_epoch=R, **common)
            if s.mlp == "moe":
                # every rank routes ALL rows (replicated router on the gathered norm outputs) through its slice of every expert: device-built
                # routing plan + grouped tcgen05 GEMMs (ops/functional.py:moe_prefill); the partial rows then go to their owners' slots
                native.check(native.lib().pb_wait_flag(self._p_layer_flag(me, l, 2), ep, R, 0, err, native.stream_ptr()), "wait_flag")
                part = Fn.moe_prefill(xn, None, w["router"], w["we_gate"], w["we_up"], w["we_down"], top_k=s.top_k, eps=eps,
                                      out=self._buf("p_moe_part", M, H), bufs=self._moe_bufs, add_residual=False)
                for r in range(R):
                    rows = max(0, min(mo, M - r * mo))
                    Fn.norm_reduce_gather(part[r * mo: r * mo + rows] if rows else part[:0], None, rows=rows, H=H, norm_kind=Fn.NORM_NONE,
                                          gather_out=[push_parts[r]], gather_flag=[self._p_layer_flag(r, l, 3)], done_counter=ctr, error_flag=err,
                                          device_index=dev)
            else:
                kw = dict(out=act, wait_flag=self._p_layer_flag(me, l, 2), wait_per_epoch=R, epoch=ep, error_flag=err)
                if s.mlp == "swiglu":
                    Fn.gemm(xn, w["w_gate"], b2=w["w_up"], act=Fn.ACT_SWIGLU, **kw)
                else:
                    Fn.gemm(xn, w["w_up"], act=self.act, **kw)
                Fn.gemm(act, w["w_down"], store_local=False, push_out=push_parts, push_rows_per_owner=mo,
                        push_done_flag=[self._p_layer_flag(r, l, 3) for r in range(R)], done_counter=ctr, error_flag=err)
            if l + 1 < L:
                wn = self.shards[l + 1]
                Fn.norm_reduce_gather(x_res, x_res, parts=my_parts, norm_weight=wn["ln1_w"], norm_bias=wn.get("ln1_b"), norm_kind=self.norm_kind,
                                      gather_out=gather_xn, gather_flag=[self._p_layer_flag(r, l + 1, 0) for r in range(R)],
                                      wait_flag=self._p_layer_flag(me, l, 3), wait_per_epoch=R, **common)
            else:  # span output: raw sum, gathered on the leader only
                Fn.norm_reduce_gather(x_res, None, parts=my_parts, norm_kind=Fn.NORM_NONE,
                                      gather_out=[self.heap.addr(0, self.off_p_out + me * mo * row_b)], gather_flag=[self.p_flag(0, 1)],
                                      wait_flag=self._p_layer_flag(me, l, 3), wait_per_epoch=R, **common)
        if me == 0:
            native.check(native.lib().pb_wait_flag(self.p_flag(0, 1), ep, R, 0, err, native.stream_ptr()), "wait_flag")
        native.check(native.lib().pb_advance_pos(pos_ptr, T, native.stream_ptr()), "advance_pos")
        return self.p_out[:M]

    def push_prefill_inputs(self, hidden: torch.Tensor) -> None:
        """Leader: scatter the chunk's rows to their owners' landing zones over NVLink (one multi-CTA copy + flag per owner)."""
        M, H = hidden.shape
        R = self.world
        mo = (M + R - 1) // R
        src = self._buf("p_stage", self.max_prefill_rows, H)
        src[:M].copy_(hidden)
        for r in range(R):
            rows = max(0, min(mo, M - r * mo))
            Fn.norm_reduce_gather(src[r * mo: r * mo + rows] if rows else src[:0], None, rows=rows, H=H, norm_kind=Fn.NORM_NONE,
                                  gather_out=[self.heap.addr(r, self.off_p_x_in)], gather_flag=[self.p_flag(r, 0)],
                                  done_counter=self.done_counter.data_ptr(), error_flag=self.err.data_ptr(), device_index=self.device.index)

    def run_prefill(self, session: SessionCache, B: int, T: int) -> torch.Tensor:
        """Every rank calls this once per prefill command (the leader after scattering the inputs)."""
        session.prepare_write(T)
        table = self._sync_session(session, B)
        before = native.launch_count
        out = self._launch_prefill(B, T, table)
        self.prefill_launches = native.launch_count - before
        session.set_position(session.position + T)
        self._dev_pos = session.position
        return out

    def _graph(self, B: int, T: int, table: torch.Tensor) -> dict:
        key = (B, T)
        g = self._graphs.get(key)
        if g is not None:
            return g
        # No warm-up replay here: a warm-up would consume flag epochs on this rank only. Kernel attributes were set by
        # `warm_kernels()` (communication-free launches) before any peer traffic.
        graph = torch.cuda.CUDAGraph()
        before = native.launch_count
        with torch.cuda.graph(graph):
            self._launch_span(B, T, table, final_reduce=True)
        launches = native.launch_count - before
        native.add_launches(-launches)
        g = dict(graph=graph, launches=launches)
        self._graphs[key] = g
        return g

    def warm_kernels(self, B: int, T: int) -> None:
        """Launch every kernel variant of a (B, T) step once WITHOUT communication so that lazy module loading,
        cudaFuncSetAttribute and buffer allocation happen before graph capture (which must not allocate)."""
        s, ls = self.spec, self.ls
        M, H = B * T, s.hidden_size
        if self.use_span_kernel:
            self._span_kernel_plan()  # buffers + kernel attribute now: graph capture must not allocate
        w = self.shards[0]
        x = self._buf("h_a", M, H)
        self._buf("h_b", M, H)
        x.zero_()
        table = self._table(B)
        qkv = Fn.linear_decode(x, w["wqkv"], norm_weight=w["ln1_w"], norm_bias=w.get("ln1_b"), norm_kind=self.norm_kind, eps=s.norm_eps,
                               out=self._buf("qkv", M, ls.qkv_dim))
        q_buf, attn = self._buf("q", M, ls.num_heads * ls.head_dim), self._buf("attn", M, ls.num_heads * ls.head_dim)
        if self.fuse_rope:
            # the RoPE-fused QKV variant too; it writes k/v of layer 0 at the positions the real step overwrites right after
            pools = self.cache.layer_pools(0)
            Fn.linear_decode(x, w["wqkv"], norm_weight=w["ln1_w"], norm_bias=w.get("ln1_b"), norm_kind=self.norm_kind, eps=s.norm_eps,
                             error_flag=self.err.data_ptr(),
                             rope=dict(q_out=q_buf, k_pool=pools[0], v_pool=pools[1], block_table=table, pos_ptr=self.pos_static.data_ptr(),
                                       cos=self.cos, sin=self.sin, T=T, Hq=ls.num_heads, Hkv=ls.num_kv_heads, D=ls.head_dim))
        attn.zero_()
        act = self._buf("act", M, ls.intermediate_size)
        splits = int(min(16, max(1, (2 * self.sms) // max(1, B * ls.num_kv_heads))))
        if splits > 1:
            self._buf("po", splits * M * ls.num_heads, ls.head_dim, torch.float32), self._buf("pl", splits, M * ls.num_heads, torch.float32)
        scratch = torch.zeros(M, H, dtype=torch.bfloat16, device=self.device)
        Fn.linear_decode(attn, w["wo"], out=scratch)
        if s.mlp == "moe":
            Fn.moe_decode(x, w["ln2_w"], w["router"], w["we_gate"], w["we_up"], w["we_down"], top_k=s.top_k, eps=s.norm_eps,
                          out=self._buf("moe_part", M, H), bufs=self._moe_bufs, add_residual=False)
            torch.cuda.synchronize(self.device)
            return
        if s.mlp == "swiglu":
            Fn.linear_decode(x, w["w_gate"], w2=w["w_up"], act=Fn.ACT_SWIGLU, norm_weight=w["ln2_w"], norm_kind=self.norm_kind, eps=s.norm_eps,
                             out=act, parts=[scratch], x_out=self._buf("h_b", M, H))
        else:
            Fn.linear_decode(x, w["w_up"], act=self.act, norm_weight=w["ln2_w"], norm_bias=w.get("ln2_b"), norm_kind=self.norm_kind,
                             eps=s.norm_eps, out=act, parts=[scratch], x_out=self._buf("h_b", M, H))
        Fn.linear_decode(act, w["w_down"], out=scratch)
        torch.cuda.synchronize(self.device)

    # ---- session bookkeeping (identical on every rank) ---------------------------------------------------------------------
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

    def run_step(self, session: SessionCache, B: int, T: int) -> torch.Tensor:
        """Every rank calls this once per step command (the leader after pushing the inputs)."""
        assert B * T <= MAX_ROWS
        session.prepare_write(T)
        table = self._sync_session(session, B)
        if (B, T) not in self._graphs:
            self.warm_kernels(B, T)
        if self.use_cuda_graphs:
            g = self._graph(B, T, table)
            g["graph"].replay()
            native.add_launches(g["launches"])
        else:
            self._launch_span(B, T, table, final_reduce=True)
        session.set_position(session.position + T)
        self._dev_pos = session.position
        return self.out[: B * T]

    def push_inputs(self, hidden: torch.Tensor) -> None:
        """Leader: broadcast the step's input rows into every rank's ``x_in`` (+ one flag each) over NVLink."""
        M = hidden.shape[0]
        src = self._buf("x_stage", MAX_ROWS, self.spec.hidden_size)
        src[:M].copy_(hidden)
        R = self.world
        dsts = ptr_array([self.heap.addr(r, self.off_x_in) for r in range(R)])
        flags = ptr_array([self.flag(r, 0) for r in range(R)])
        native.check(native.lib().pb_push_rows(src.data_ptr(), dsts, flags, R, M * self.spec.hidden_size * 2, native.stream_ptr()), "push_rows")

    def check_errors(self) -> None:
        code = int(self.err.item())
        if code:
            self.err.zero_()
            raise RuntimeError(f"rank {self.rank}: device-side error flag {code} (1 = peer flag watchdog expired, 2 = KV page table overflow)")


# ---- CPU oracle of the sharded math (tests; reference: tests/test_tensor_parallel.py) ----------------------------------------
def shard_oracle_blocks(block: GenericBlock, spec: BlockSpec, world: int) -> List[GenericBlock]:
    """One plain-PyTorch block per rank holding exactly the tensors :func:`shard_block` gives that rank."""
    ls = local_spec(spec, world)
    out = []
    for rank in range(world):
        b = GenericBlock(ls, dtype=block.wqkv.dtype, device=block.wqkv.device)
        with torch.no_grad():
            for name, t in shard_block(block, spec, rank, world, block.wqkv.device).items():
                getattr(b, name).copy_(t)
        out.append(b)
    return out


def tp_oracle_forward(shards: Sequence[GenericBlock], hidden: torch.Tensor, caches: Optional[Sequence[Tuple[torch.Tensor, torch.Tensor]]] = None,
                      pos: int = 0) -> torch.Tensor:
    """What the TP engine computes, written with autograd-friendly tensor ops: norms and the residual stream are replicated,
    every rank contributes a partial attention / MLP output and the partials are summed where the engine all-reduces."""
    first = shards[0]
    ln1 = first._norm(hidden, "ln1")
    h = hidden + sum(b.attention(ln1, *(caches[r] if caches is not None else (None, None)), pos) for r, b in enumerate(shards))
    ln2 = first._norm(h, "ln2")
    return h + sum(b.mlp(ln2) for b in shards)
