"""The NVLink activation fabric between pipeline stages (one process per GPU).

In the reference every hop between servers is an RPC that drags the activation through host memory, protobuf and the
libp2p daemon, and the router budgets 18 ms for it (SURVEY.md §0.4; src/petals/client/routing/sequence_manager.py:223).
Here each worker process owns a *landing zone* in a CUDA-IPC symmetric heap:

* ``x_in``  — where the previous stage's **last kernel** (down-projection GEMV or tcgen05 GEMM + residual) stores its
  output tiles directly over NVLink (``push_out`` epilogue), followed by one release-increment of ``in_flag``;
* ``y_ret`` — the same for the last stage returning the final hidden states to the client's GPU (and, in training, for the first
  stage returning the gradient of the span input);
* ``g_in``  — the gradient hop: the **last kernel of stage i+1's backward** (the RMSNorm backward of its first block, which adds
  the residual gradient) stores dL/d(hidden) straight into stage i's landing slot, so ``rpc_backward`` between stages carries no
  tensor bytes either (``server/stage_engine.py:backward``).

The consuming stage's **first kernel** waits on the flag (``ld.acquire.sys``) — so the hop costs one NVLink store stream
overlapped with the producer's math plus a flag latency, and the control RPC between processes carries *no tensor
bytes* (only "your input is in your landing zone"). Flags are monotonic; every consumer keeps a device-resident count
of consumed transfers (the "epoch" passed to the kernels), so nothing is ever reset and CUDA graphs stay valid.

Created once per process: by :func:`join_fabric` when independently started processes of a box rendezvous (``run_server
--fabric_address HOST:PORT --fabric_rank R --fabric_world N``, ``from_pretrained(..., fabric_address=...)`` for a co-located client), or by
:func:`init_fabric` inside a job that is already one ``torch.distributed`` world (benchmarks, self-tests). Stages announce their membership
(:func:`fabric_info`) in ``rpc_info``; clients route hops by those announcements and need no membership themselves. Absent
(``get_fabric()`` is None) otherwise: stages then exchange tensors by reference or over the socket transport. On CPU the same protocol
runs over POSIX shared memory (:class:`HostFabric`)."""
from __future__ import annotations

from typing import Optional

import torch
import torch.distributed as dist

from petals_b200.ops import native
from petals_b200.parallel.symmetric import SymmetricHeap, host_barrier, ptr_array, tensor_from_ptr
from petals_b200.utils.logging import get_logger

logger = get_logger(__name__)
_fabric: Optional["Fabric"] = None


KINDS = {"x_in": 0, "y_ret": 1, "g_in": 2}
NK = len(KINDS)


class Fabric:
    """Landing rings in the symmetric heap. Every rank owns, per kind ("x_in": input of its span, "y_ret": results returned to a
    client on this rank, "g_in": gradient of its span's output), ``n_slots`` landing slots of ``max_tokens x hidden`` bf16 plus, per slot, a data flag (incremented by the
    producer's release after its stores) and an acknowledgement flag ON THE PRODUCER (incremented by the consumer when the slot
    may be overwritten). All counters are monotonic and per slot, so transfers through different slots are independent: a
    producer can have up to ``n_slots`` chunks in flight towards the same consumer (chunked prefill / micro-batches in a
    pipeline), and nothing is ever reset."""

    def __init__(self, hidden_size: int, max_tokens: int = 8192, group=None, extra_bytes: int = (256 << 20) + (1 << 20), n_slots: int = 4):
        self.hidden_size, self.max_tokens, self.n_slots = hidden_size, max_tokens, n_slots
        self.zone_bytes = max_tokens * hidden_size * 2
        self.heap = SymmetricHeap(NK * n_slots * self.zone_bytes + extra_bytes, group=group)
        self.rank, self.world, self.device = self.heap.rank, self.heap.world, self.heap.device
        self.off_zones = self.heap.alloc(NK * n_slots * self.zone_bytes)
        self.off_flags = self.heap.alloc(2 * NK * n_slots * 8 + 64)  # [data | ack][kind][slot] u64
        self._zone_views = {}
        # device-resident counters: transfers consumed per (kind, slot) and pushes issued per (kind, slot)
        self.consumed = torch.zeros(NK, n_slots, dtype=torch.int64, device=self.device)
        self.pushed = torch.zeros(NK, n_slots, dtype=torch.int64, device=self.device)
        self.done_counter = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.err = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._flag_src = torch.zeros(16, dtype=torch.uint8, device=self.device)
        self._scratch_off = self.heap.alloc(64)
        # back-pressure: the pushing kernel's prologue waits for ack >= number of pushes issued through this slot so far; the
        # acknowledgement flags start at 1, so the first push through a slot never waits
        self.heap.tensor(self.off_flags + NK * n_slots * 8, (NK * n_slots,), torch.int64).fill_(1)
        torch.cuda.synchronize(self.device)
        host_barrier(group)

    # ---- addresses ---------------------------------------------------------------------------------------------
    def _zone_off(self, kind: str, slot: int) -> int:
        return self.off_zones + (KINDS[kind] * self.n_slots + slot % self.n_slots) * self.zone_bytes

    def _data_flag_off(self, kind: str, slot: int) -> int:
        return self.off_flags + (KINDS[kind] * self.n_slots + slot % self.n_slots) * 8

    def _ack_flag_off(self, kind: str, slot: int) -> int:
        return self.off_flags + (NK * self.n_slots + KINDS[kind] * self.n_slots + slot % self.n_slots) * 8

    def zone(self, kind: str, rank: int, slot: int = 0):
        """(data address, data-flag address) of landing slot ``slot`` of ``kind`` on ``rank``."""
        if kind not in KINDS:
            raise ValueError(kind)
        return self.heap.addr(rank, self._zone_off(kind, slot)), self.heap.addr(rank, self._data_flag_off(kind, slot))

    def ack_flag_addr(self, rank: int, kind: str = "x_in", slot: int = 0) -> int:
        """Where the consumer of a transfer acknowledges: on the PRODUCER ``rank``, per (kind, slot) of the consumer's ring."""
        return self.heap.addr(rank, self._ack_flag_off(kind, slot))

    def view(self, kind: str, slot: int = 0) -> torch.Tensor:
        """This rank's landing slot as a [max_tokens, hidden] tensor (no copy)."""
        key = (kind, slot % self.n_slots)
        if key not in self._zone_views:
            self._zone_views[key] = self.heap.tensor(self._zone_off(kind, slot), (self.max_tokens, self.hidden_size), torch.bfloat16)
        return self._zone_views[key]

    def begin_push(self, kind: str = "x_in", slot: int = 0) -> dict:
        """Call right before launching a kernel whose epilogue pushes into a peer's landing slot: returns the prologue wait
        arguments that implement the back-pressure described above."""
        counter = self.pushed[KINDS[kind], slot % self.n_slots]
        native.check(native.lib().pb_bump_epoch(counter.data_ptr(), native.stream_ptr()), "bump_epoch")
        return dict(wait_flag=self.ack_flag_addr(self.rank, kind, slot), wait_per_epoch=1, epoch=counter.data_ptr(), error_flag=self.err.data_ptr())

    def wait(self, kind: str = "y_ret", slot: int = 0) -> None:
        """Enqueue a wait for the next transfer into this rank's landing slot (advances the slot's consumed count)."""
        counter = self.consumed[KINDS[kind], slot % self.n_slots]
        _, flag = self.zone(kind, self.rank, slot)
        lib = native.lib()
        native.check(lib.pb_bump_epoch(counter.data_ptr(), native.stream_ptr()), "bump_epoch")
        native.check(lib.pb_wait_flag(flag, counter.data_ptr(), 1, 0, self.err.data_ptr(), native.stream_ptr()), "wait_flag")

    def acknowledge(self, kind: str, src_rank: int, slot: int = 0) -> None:
        """Tell ``src_rank`` that landing slot ``slot`` may be overwritten (stream ordered: after everything that read it)."""
        self._signal(self.ack_flag_addr(src_rank, kind, slot), src_rank)

    def take(self, M: int, kind: str, src_rank: int, out: torch.Tensor, slot: int = 0) -> torch.Tensor:
        """Consume the next transfer into slot ``slot``: wait, copy the rows out, acknowledge to ``src_rank``."""
        self.wait(kind, slot)
        out.copy_(self.view(kind, slot)[:M])
        self.acknowledge(kind, src_rank, slot)
        return out

    # ---- zero-copy halves of a transfer: the consumer reads the landing slot in place, the producer's kernel writes into the peer's ----
    def landing(self, M: int, kind: str, slot: int = 0) -> torch.Tensor:
        """Wait (on the stream) for the next transfer into slot ``slot`` and return its rows IN PLACE. The caller acknowledges
        (:meth:`acknowledge`) once the last kernel that reads them has been enqueued."""
        self.wait(kind, slot)
        return self.view(kind, slot)[:M]

    def open_push(self, M: int, rank: int, kind: str, slot: int = 0) -> torch.Tensor:
        """Rows [M, H] of landing slot ``slot`` on ``rank`` as a tensor a kernel can store into (peer memory over NVLink); the
        back-pressure wait is enqueued first. Follow the producing kernel with :meth:`publish`."""
        if M > self.max_tokens:
            raise ValueError(f"{M} rows exceed the fabric landing zone ({self.max_tokens})")
        data, _ = self.zone(kind, rank, slot)
        kw = self.begin_push(kind, slot)
        native.check(native.lib().pb_wait_flag(kw["wait_flag"], kw["epoch"], 1, 0, kw["error_flag"], native.stream_ptr()), "wait_flag")
        return tensor_from_ptr(data, (M, self.hidden_size), torch.bfloat16, self.device)

    def publish(self, rank: int, kind: str, slot: int = 0) -> None:
        """Release-increment the data flag of the slot :meth:`open_push` handed out (stream ordered after the stores)."""
        self._signal(self.zone(kind, rank, slot)[1], rank)

    def _signal(self, flag_addr: int, rank: int) -> None:
        scratch = ptr_array([self.heap.addr(rank, self._scratch_off)])
        native.check(native.lib().pb_push_rows(self._flag_src.data_ptr(), scratch, ptr_array([flag_addr]), 1, 16, native.stream_ptr()), "fabric signal")

    # ---- host-issued transfers (client -> first stage; anything not produced by a fused epilogue) ---------------------
    def send(self, rows: torch.Tensor, rank: int, kind: str = "x_in", slot: int = 0) -> None:
        """Copy ``rows`` [M, H] into a landing slot of ``rank`` and publish it (stream ordered)."""
        M = rows.shape[0]
        if M > self.max_tokens:
            raise ValueError(f"{M} rows exceed the fabric landing zone ({self.max_tokens})")
        data, flag = self.zone(kind, rank, slot)
        dst = tensor_from_ptr(data, (M, self.hidden_size), torch.bfloat16, self.device)
        kw = self.begin_push(kind, slot)  # honour back-pressure like the fused pushes do
        native.check(native.lib().pb_wait_flag(kw["wait_flag"], kw["epoch"], 1, 0, kw["error_flag"], native.stream_ptr()), "wait_flag")
        dst.copy_(rows.reshape(M, self.hidden_size).to(torch.bfloat16))  # P2P memcpy over NVLink
        self._signal(flag, rank)

    def recv(self, M: int, kind: str, src_rank: int, slot: int = 0) -> torch.Tensor:
        out = torch.empty(M, self.hidden_size, dtype=torch.bfloat16, device=self.device)
        return self.take(M, kind, src_rank, out, slot)

    def check_errors(self) -> None:
        if int(self.err.item()):
            self.err.zero_()
            raise RuntimeError(f"rank {self.rank}: a fabric flag wait timed out (a peer stage is gone or stalled)")

    def close(self) -> None:
        self.heap.close()


class HostFabric:
    """The same protocol over POSIX shared memory, for CPU processes (gloo): lets the multi-process plumbing tests exercise
    the fabric code paths of the client and the handlers (landing rings, per-slot flags, acknowledgements) without GPUs."""

    def __init__(self, hidden_size: int, max_tokens: int = 1024, group=None, dtype: torch.dtype = torch.float32, n_slots: int = 4):
        import time
        from multiprocessing import shared_memory

        import numpy as np

        self.hidden_size, self.max_tokens, self.dtype, self.n_slots = hidden_size, max_tokens, dtype, n_slots
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.device = torch.device("cpu")
        self._time, self._np = time, np
        itemsize = torch.empty(0, dtype=dtype).element_size()
        self._zone_bytes = max_tokens * hidden_size * itemsize
        self._flag_bytes = 2 * NK * n_slots * 8
        per_rank = NK * n_slots * self._zone_bytes + self._flag_bytes
        names = [None]
        if self.rank == 0:
            self._shm = shared_memory.SharedMemory(create=True, size=per_rank * self.world)
            self._shm.buf[: per_rank * self.world] = b"\x00" * (per_rank * self.world)
            names[0] = self._shm.name
        dist.broadcast_object_list(names, src=0, group=group)
        if self.rank != 0:
            from petals_b200.parallel.control import attach_shared_memory

            self._shm = attach_shared_memory(names[0])
        self._per_rank = per_rank
        self._consumed = np.zeros((NK, n_slots), dtype=np.int64)
        self._pushed = np.zeros((NK, n_slots), dtype=np.int64)
        self._open = {}
        if self.rank == 0:
            for r in range(self.world):
                self._flags(r)[NK * n_slots:] = 1  # acknowledgement flags start at 1 (the first push through a slot never waits)
        host_barrier(group)

    def _flags(self, rank: int):
        """u64 [data flags: kind x slot | ack flags: kind x slot] of ``rank``."""
        off = rank * self._per_rank + NK * self.n_slots * self._zone_bytes
        return self._np.ndarray((2 * NK * self.n_slots,), dtype=self._np.uint64, buffer=self._shm.buf, offset=off)

    def _idx(self, kind: str, slot: int) -> int:
        return KINDS[kind] * self.n_slots + slot % self.n_slots

    def _zone(self, kind: str, rank: int, rows: int, slot: int) -> torch.Tensor:
        off = rank * self._per_rank + self._idx(kind, slot) * self._zone_bytes
        flat = torch.frombuffer(self._shm.buf, dtype=self.dtype, count=rows * self.hidden_size, offset=off)
        return flat.view(rows, self.hidden_size)

    def _spin(self, rank: int, idx: int, target: int, what: str, timeout: float = 30.0) -> None:
        deadline = self._time.monotonic() + timeout
        while int(self._flags(rank)[idx]) < target:
            if self._time.monotonic() > deadline:
                raise TimeoutError(f"rank {self.rank}: timed out waiting for {what}")
            self._time.sleep(0)

    def send(self, rows: torch.Tensor, rank: int, kind: str = "x_in", slot: int = 0) -> None:
        M = rows.shape[0]
        if M > self.max_tokens:
            raise ValueError(f"{M} rows exceed the fabric landing zone ({self.max_tokens})")
        i = self._idx(kind, slot)
        self._pushed[KINDS[kind], slot % self.n_slots] += 1
        self._spin(self.rank, NK * self.n_slots + i, int(self._pushed[KINDS[kind], slot % self.n_slots]), "the consumer's acknowledgement")
        self._zone(kind, rank, M, slot).copy_(rows.reshape(M, self.hidden_size).to(self.dtype))
        self._flags(rank)[i] += 1

    def take(self, M: int, kind: str, src_rank: int, out: torch.Tensor, slot: int = 0) -> torch.Tensor:
        i = self._idx(kind, slot)
        self._consumed[KINDS[kind], slot % self.n_slots] += 1
        self._spin(self.rank, i, int(self._consumed[KINDS[kind], slot % self.n_slots]), f"a transfer into {kind}[{slot}]")
        out.copy_(self._zone(kind, self.rank, M, slot))
        self._flags(src_rank)[NK * self.n_slots + i] += 1
        return out

    def landing(self, M: int, kind: str, slot: int = 0) -> torch.Tensor:
        i = self._idx(kind, slot)
        self._consumed[KINDS[kind], slot % self.n_slots] += 1
        self._spin(self.rank, i, int(self._consumed[KINDS[kind], slot % self.n_slots]), f"a transfer into {kind}[{slot}]")
        return self._zone(kind, self.rank, M, slot)

    def acknowledge(self, kind: str, src_rank: int, slot: int = 0) -> None:
        self._flags(src_rank)[NK * self.n_slots + self._idx(kind, slot)] += 1

    def open_push(self, M: int, rank: int, kind: str, slot: int = 0) -> torch.Tensor:
        if M > self.max_tokens:
            raise ValueError(f"{M} rows exceed the fabric landing zone ({self.max_tokens})")
        i = self._idx(kind, slot)
        self._pushed[KINDS[kind], slot % self.n_slots] += 1
        self._spin(self.rank, NK * self.n_slots + i, int(self._pushed[KINDS[kind], slot % self.n_slots]), "the consumer's acknowledgement")
        return self._zone(kind, rank, M, slot)

    def publish(self, rank: int, kind: str, slot: int = 0) -> None:
        self._flags(rank)[self._idx(kind, slot)] += 1

    def recv(self, M: int, kind: str, src_rank: int, slot: int = 0) -> torch.Tensor:
        return self.take(M, kind, src_rank, torch.empty(M, self.hidden_size, dtype=self.dtype), slot)

    def check_errors(self) -> None:
        pass

    def close(self) -> None:
        shm, self._shm = getattr(self, "_shm", None), None
        if shm is None:
            return
        try:
            shm.close()
            if self.rank == 0:
                shm.unlink()
        except Exception:  # noqa: BLE001
            pass


def init_fabric(hidden_size: int, max_tokens: int = 8192, group=None, host_dtype: torch.dtype = torch.float32, n_slots: int = 4,
                cuda: Optional[bool] = None):
    """Collective over ``group``. Returns None when there is nothing to connect (single process). ``cuda``: the landing rings live
    in GPU memory (default: when a CUDA device is visible) or, for members that serve on the CPU, in host shared memory."""
    global _fabric
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) < 2:
        return None
    if cuda is None:
        cuda = torch.cuda.is_available()
    # the landing rings live at the same offsets of every member's heap: every member must size them identically
    mine = (int(hidden_size), int(max_tokens), int(n_slots), bool(cuda))
    everyone = [None] * dist.get_world_size(group)
    try:
        dist.all_gather_object(everyone, mine, group=group)
    except Exception as e:  # noqa: BLE001 - a group without an object-collective path: skip the courtesy check, the rings still work
        logger.warning(f"could not compare the fabric geometry across members: {e!r}")
        everyone = [mine]
    if any(other != mine for other in everyone):
        raise ValueError(f"the members of a fabric must agree on (hidden_size, max_tokens, n_slots, cuda): {everyone}")
    if cuda:
        _fabric = Fabric(hidden_size, max_tokens, group, n_slots=n_slots)
    else:
        _fabric = HostFabric(hidden_size, min(max_tokens, 1024), group, host_dtype, n_slots=n_slots)
    # one identity per fabric: clients learn from `rpc_info` which stages can reach each other's landing rings (two stages hop over NVLink
    # only if they announce the same id), whether or not the client itself is a member
    import uuid

    ident = [uuid.uuid4().hex if dist.get_rank(group) == 0 else None]
    try:
        dist.broadcast_object_list(ident, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
    except Exception as e:  # noqa: BLE001 - no identity: only clients that are members themselves can route over this fabric (legacy behaviour)
        logger.warning(f"could not agree on a fabric identity: {e!r}")
        ident = [None]
    _fabric.fabric_id = ident[0]
    return _fabric


def join_fabric(address: str, rank: int, world: int, hidden_size: int, *, device=None, max_tokens: int = 8192,
                host_dtype: torch.dtype = torch.float32, n_slots: int = 4):
    """Rendezvous of independently started processes of one NVLink box (stage servers: ``run_server --fabric_address ...``; a co-located
    client: ``from_pretrained(..., fabric_address=...)``) into one landing-ring fabric. Collective over the ``world`` processes that call
    it with the same ``address`` ("host:port"); initialises ``torch.distributed`` for them if the process has not done so itself.
    Returns ``(fabric, owns_process_group)``."""
    if rank is None or world is None or not 0 <= rank < world or world < 2:
        raise ValueError("a fabric needs fabric_rank R and fabric_world N with 0 <= R < N and N >= 2")
    if _fabric is not None:
        return _fabric, False
    owns = False
    device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else torch.device("cpu")
    cuda = device.type == "cuda"  # a member that serves on the CPU joins the shared-memory fabric, GPU or not
    if not dist.is_initialized():
        if cuda:
            torch.cuda.set_device(device)
        dist.init_process_group(backend="cpu:gloo,cuda:nccl" if cuda else "gloo", init_method=f"tcp://{address}", rank=rank, world_size=world,
                                **({"device_id": device} if cuda else {}))
        owns = True
    fabric = init_fabric(hidden_size, max_tokens=max_tokens, host_dtype=host_dtype, n_slots=n_slots, cuda=cuda)
    logger.info(f"Joined the NVLink fabric {str(getattr(fabric, 'fabric_id', '?'))[:8]} as member {rank} of {world} ({fabric.max_tokens} rows per landing slot)")
    return fabric, owns


def leave_fabric(owns_process_group: bool) -> None:
    """Undo :func:`join_fabric` (best effort: peers may already be gone)."""
    global _fabric
    try:
        if _fabric is not None:
            _fabric.close()
        _fabric = None
        if owns_process_group and dist.is_initialized():
            dist.destroy_process_group()
    except Exception as e:  # noqa: BLE001
        logger.debug(f"leaving the fabric: {e!r}")


def fabric_info(fabric=None) -> Optional[dict]:
    """What a stage announces about its fabric membership (``rpc_info()["fabric"]``)."""
    fabric = fabric if fabric is not None else _fabric
    if fabric is None:
        return None
    return {"id": getattr(fabric, "fabric_id", None), "rank": fabric.rank, "world": fabric.world, "max_tokens": fabric.max_tokens,
            "hidden_size": fabric.hidden_size, "n_slots": getattr(fabric, "n_slots", 1)}


def get_fabric() -> Optional[Fabric]:
    return _fabric
