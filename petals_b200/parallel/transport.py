"""Control-plane transport between a client and stage workers.

The reference speaks protobuf-over-libp2p through a Go daemon (hivemind P2P; SURVEY.md §2.4). Inside one box
that collapses to two cases:

* same process  -> the "stub" *is* the handler object; tensors are passed by reference (CUDA tensors stay on
  the GPU, nothing is serialised);
* other process -> a Unix-domain-socket RPC with a msgpack header + raw tensor bytes (this is the CPU
  plumbing path used by ``run_server`` swarms and the multi-process tests; the GPU data plane between
  stages never uses it — activations move by fused NVLink stores, see parallel/symmetric.py).

Request = ``{"method", "uids", "meta", "tensors": [{"dtype", "shape"}...]}``; response = ``{"ok", "error",
"meta", "tensors"}``. ``rpc_inference`` keeps its connection open as a bidirectional stream, one request per
step, exactly one response per request, an empty request closes the session (reference
src/petals/client/inference_session.py:198-207).
"""
from __future__ import annotations

import contextlib
import ctypes as C
import errno
import os
import socket
import socketserver
import struct
import threading
import traceback
from typing import Any, Dict, List, Optional, Sequence, Tuple

import msgpack
import torch

from petals_b200.utils.compression import decode as decode_tensor, encode as encode_tensor, normalize_output_compression
from petals_b200.utils.logging import get_logger

logger = get_logger(__name__)

def parse_address(address: str) -> Tuple[str, ...]:
    """``/path/to.sock`` -> ("unix", path); ``tcp://host:port`` or a libp2p-style multiaddr
    (``/ip4/10.0.0.1/tcp/31337[/p2p/<id>]``, ``/dns/name/tcp/31337``; the form the reference prints and accepts as
    ``--initial_peers``) -> ("tcp", host, port)."""
    if address.startswith("tcp://"):
        host, _, port = address[len("tcp://"):].rpartition(":")
        return ("tcp", host.strip("[]") or "127.0.0.1", int(port))
    parts = address.strip("/").split("/")
    if len(parts) >= 4 and parts[0] in ("ip4", "ip6", "dns", "dns4", "dns6") and parts[2] == "tcp":
        return ("tcp", parts[1], int(parts[3]))
    return ("unix", address)


def is_network_address(address: str) -> bool:
    return isinstance(address, str) and parse_address(address)[0] == "tcp"


def format_address(host: str, port: int) -> str:
    return f"tcp://{host}:{port}"


def to_multiaddr(address: str) -> str:
    kind, *rest = parse_address(address)
    if kind != "tcp":
        return address
    host, port = rest
    proto = "ip4" if host.replace(".", "").isdigit() else ("ip6" if ":" in host else "dns")
    return f"/{proto}/{host}/tcp/{port}"


_SUN_PATH_MAX = 107  # bytes of a Unix socket path (sockaddr_un.sun_path holds 108 with the terminating NUL)


@contextlib.contextmanager
def _unix_name(path: str):
    """A name that binds / connects to the Unix socket at ``path`` however deep its directory is (a rendezvous directory may live under
    a long temp path): ``path`` itself when it fits, else the same file reached through a descriptor of its directory."""
    if len(os.fsencode(path)) <= _SUN_PATH_MAX:
        yield path
        return
    fd = os.open(os.path.dirname(path) or ".", os.O_PATH | os.O_DIRECTORY)
    try:
        yield f"/proc/self/fd/{fd}/{os.path.basename(path)}"
    finally:
        os.close(fd)


def open_connection(address: str, connect_timeout: float, request_timeout: Optional[float]) -> socket.socket:
    kind, *rest = parse_address(address)
    if kind == "tcp":
        s = socket.create_connection((rest[0], rest[1]), timeout=connect_timeout)
        s.setsockopt(socket.IPPROTO_TCP, socket.TCP_NODELAY, 1)  # one decode step = one small frame each way
    else:
        s = socket.socket(socket.AF_UNIX, socket.SOCK_STREAM)
        s.settimeout(connect_timeout)
        with _unix_name(rest[0]) as name:
            s.connect(name)
    s.settimeout(request_timeout)
    return s


_DTYPE_NAMES = {torch.float32: "f32", torch.float16: "f16", torch.bfloat16: "bf16", torch.int64: "i64", torch.int32: "i32",
                torch.uint8: "u8", torch.bool: "b1", torch.float64: "f64"}
_DTYPES = {v: k for k, v in _DTYPE_NAMES.items()}


def _native_io():
    """The C++ socket loops (csrc/runtime/socket_io.cpp); ``PETALS_B200_PY_TRANSPORT=1`` forces the pure-Python path."""
    if os.environ.get("PETALS_B200_PY_TRANSPORT", "0") == "1":
        return None
    try:
        from petals_b200.ops import native

        return native.rt()
    except Exception:  # noqa: BLE001 - no compiler on this host: the Python loops below do the same job
        return None


def _raise_io(rc: int, what: str) -> None:
    if rc == -1:
        raise ConnectionError("peer closed the connection")
    if rc == -errno.ETIMEDOUT:
        raise socket.timeout(f"{what} timed out")
    if rc in (-errno.EPIPE, -errno.ECONNRESET, -errno.EBADF, -errno.ENOTCONN):
        raise ConnectionError(f"{what}: {os.strerror(-rc)}")
    raise OSError(-rc, f"{what}: {os.strerror(-rc)}")


def _timeout_of(sock: socket.socket) -> float:
    t = sock.gettimeout()
    return -1.0 if t is None else float(t)


def _recv_exact(sock: socket.socket, n: int) -> bytes:
    chunks, got = [], 0
    while got < n:
        c = sock.recv(min(n - got, 1 << 20))
        if not c:
            raise ConnectionError("peer closed the connection")
        chunks.append(c)
        got += len(c)
    return b"".join(chunks)


def _recv_into(sock: socket.socket, n: int) -> torch.Tensor:
    """n payload bytes -> a fresh flat uint8 tensor, received in place (no intermediate bytes objects)."""
    buf = torch.empty(n, dtype=torch.uint8)
    io = _native_io()
    if io is not None:
        rc = io.pb_sock_recv_exact(sock.fileno(), buf.data_ptr(), n, _timeout_of(sock))
        if rc != 0:
            _raise_io(rc, "recv")
        return buf
    view, got = memoryview(buf.numpy()), 0
    while got < n:
        k = sock.recv_into(view[got:], n - got)
        if k == 0:
            raise ConnectionError("peer closed the connection")
        got += k
    return buf


def send_message(sock: socket.socket, header: Dict[str, Any], tensors: Sequence[torch.Tensor] = (), compression=None) -> None:
    """``compression``: one codec for every tensor or a list with one entry per tensor (utils/compression.py);
    integer/bool tensors and empty tensors always travel raw."""
    metas, blobs = [], []
    per_tensor = list(compression) if isinstance(compression, (list, tuple)) else [compression] * len(tensors)
    for t, codec in zip(tensors, per_tensor):
        if t is None:
            t = torch.empty(0)  # an empty tensor means "argument absent" (utils/misc.py DUMMY convention)
        cmeta, parts = encode_tensor(t, codec)
        metas.append({"dtype": _DTYPE_NAMES[t.dtype], "shape": list(t.shape), "nbytes": sum(b.numel() for b in parts),
                      "parts": [b.numel() for b in parts], "c": cmeta})
        blobs.extend(parts)
    header = dict(header, tensors=metas)
    payload = msgpack.packb(header, use_bin_type=True)
    head = struct.pack("<I", len(payload)) + payload
    io = _native_io()
    if io is None:
        sock.sendall(head + b"".join(b.numpy().tobytes() for b in blobs if b.numel()))
        return
    blobs = [b for b in blobs if b.numel()]  # the tensors stay referenced (alive) until sendmsg has consumed them
    n = 1 + len(blobs)
    ptrs = (C.c_void_p * n)(C.cast(C.c_char_p(head), C.c_void_p), *[b.data_ptr() for b in blobs])
    lens = (C.c_int64 * n)(len(head), *[b.numel() for b in blobs])
    rc = io.pb_sock_send_frames(sock.fileno(), ptrs, lens, n, _timeout_of(sock))
    if rc != 0:
        _raise_io(rc, "send")


MAX_HEADER_BYTES = 16 << 20  # a header is a few hundred bytes; anything huge is a corrupt or foreign stream
MAX_TENSORS_PER_MESSAGE = 256
MAX_PART_BYTES = 8 << 30       # one part of one tensor
MAX_MESSAGE_BYTES = 16 << 30   # all payload bytes of one message (a step's activations are max_batch_size * hidden * 2 bytes: MiB, not GiB)


class ProtocolError(ConnectionError):
    """The peer sent something that is not a frame of this protocol; the connection is dropped."""


def recv_message(sock: socket.socket) -> Tuple[Dict[str, Any], List[torch.Tensor]]:
    (n,) = struct.unpack("<I", _recv_exact(sock, 4))
    if n > MAX_HEADER_BYTES:
        raise ProtocolError(f"header of {n} bytes announced (limit {MAX_HEADER_BYTES})")
    try:
        header = msgpack.unpackb(_recv_exact(sock, n), raw=False)
    except ConnectionError:
        raise
    except Exception as e:  # noqa: BLE001 - msgpack raises several unrelated exception types on garbage
        raise ProtocolError(f"undecodable header: {e!r}") from None
    if not isinstance(header, dict) or not isinstance(header.get("tensors", []), list) or len(header.get("tensors", [])) > MAX_TENSORS_PER_MESSAGE:
        raise ProtocolError("malformed header")
    tensors, total = [], 0
    for m in header.get("tensors", []):
        sizes = m.get("parts", [m.get("nbytes", 0)]) if isinstance(m, dict) else None
        if sizes is None or m.get("dtype") not in _DTYPES or any(not isinstance(k, int) or k < 0 or k > MAX_PART_BYTES for k in sizes):
            raise ProtocolError("malformed tensor descriptor")
        shape = m.get("shape")
        if not isinstance(shape, list) or len(shape) > 8 or any(not isinstance(d, int) or d < 0 for d in shape):
            raise ProtocolError("malformed tensor shape")
        total += sum(sizes)
        if total > MAX_MESSAGE_BYTES:
            raise ProtocolError(f"message announces more than {MAX_MESSAGE_BYTES} payload bytes")
        parts = [_recv_into(sock, k) for k in sizes]
        try:
            tensors.append(decode_tensor(m.get("c", {"codec": "NONE"}), parts, _DTYPES[m["dtype"]], shape))
        except (ValueError, KeyError, TypeError, IndexError, RuntimeError) as e:  # descriptor and payload disagree
            raise ProtocolError(f"tensor descriptor does not match its payload: {e}") from None
    return header, tensors


class RemoteError(RuntimeError):
    """An exception raised by the remote handler, re-raised on the caller's side."""


# ---------------------------------------------------------------------------------------------------------
# server side
# ---------------------------------------------------------------------------------------------------------
class TrackedConn(socketserver.BaseRequestHandler):
    """Registers the connection with its server so that ``RpcServer.shutdown`` can drop established connections too
    (a stopped stage must not keep answering on old streams; clients then fail over like after a crash)."""

    def setup(self) -> None:
        conns = getattr(self.server, "open_conns", None)
        if conns is not None:
            with self.server.open_conns_lock:  # type: ignore[attr-defined]
                conns.add(self.request)

    def finish(self) -> None:
        conns = getattr(self.server, "open_conns", None)
        if conns is not None:
            with self.server.open_conns_lock:  # type: ignore[attr-defined]
                conns.discard(self.request)


class _Conn(TrackedConn):
    def handle(self) -> None:
        handler = self.server.rpc_handler  # type: ignore[attr-defined]
        sock: socket.socket = self.request
        stream, stream_codec = None, None
        try:
            while True:
                try:
                    header, tensors = recv_message(sock)
                except ConnectionError:
                    break
                method = header.get("method")
                try:
                    meta = header.get("meta") or {}
                    default_codec = getattr(handler, "compression", None)
                    if method == "rpc_inference":
                        if stream is None:
                            stream = handler.rpc_inference(header["uids"], header.get("meta", {}))
                            stream_codec = meta.get("output_compression")  # sticky for the whole session
                        if header.get("close") or not tensors:
                            stream.close()
                            stream = None
                            send_message(sock, {"ok": True, "closed": True})
                            continue
                        out = stream.step(*tensors, metadata=header.get("meta", {}))
                        send_message(sock, {"ok": True}, [out],
                                     normalize_output_compression(meta.get("output_compression", stream_codec), 1, default_codec))
                    elif method == "rpc_info":
                        send_message(sock, {"ok": True, "meta": handler.rpc_info(header.get("uids"))})
                    elif method == "rpc_forward":
                        codecs = normalize_output_compression(meta.get("output_compression"), 1, default_codec)
                        out = handler.rpc_forward(header["uids"], *tensors, metadata=header.get("meta", {}))
                        send_message(sock, {"ok": True}, [out], codecs)
                    elif method == "rpc_backward":
                        outs = list(handler.rpc_backward(header["uids"], *tensors, metadata=header.get("meta", {})))
                        send_message(sock, {"ok": True}, outs, normalize_output_compression(meta.get("output_compression"), len(outs), default_codec))
                    elif method == "rpc_push":
                        handler.rpc_push(header["uids"], *tensors, metadata=header.get("meta", {}))
                        send_message(sock, {"ok": True})
                    elif method == "rpc_ping":
                        send_message(sock, {"ok": True})
                    elif method == "rpc_check":
                        send_message(sock, {"ok": True, "meta": bool(handler.rpc_check(meta["check_peer"], float(meta.get("wait_timeout", 5.0))))})
                    else:
                        send_message(sock, {"ok": False, "error": f"unknown method {method!r}", "etype": "ValueError"})
                except Exception as e:  # noqa: BLE001 - report to the caller, keep serving
                    logger.debug("rpc failed:\n" + traceback.format_exc())
                    send_message(sock, {"ok": False, "error": str(e), "etype": type(e).__name__})
        finally:
            if stream is not None:
                stream.close()


class _ThreadedUnixServer(socketserver.ThreadingMixIn, socketserver.UnixStreamServer):
    daemon_threads = True
    allow_reuse_address = True


class _ThreadedTcpServer(socketserver.ThreadingMixIn, socketserver.TCPServer):
    daemon_threads = True
    allow_reuse_address = True
    request_queue_size = 128

    def get_request(self):
        conn, addr = super().get_request()
        conn.setsockopt(socket.IPPROTO_TCP, socket.TCP_NODELAY, 1)
        return conn, addr


class RpcServer:
    """Serves a handler on a Unix socket or on TCP (one thread per connection = one per in-flight request/stream).

    ``address``: a filesystem path, or ``tcp://host:port`` (port 0 = pick a free one; ``self.address`` is the bound one).
    ``conn_class`` lets other services (the swarm registry) reuse the framing with their own dispatcher."""

    def __init__(self, handler, address: str, conn_class=None):
        kind, *rest = parse_address(address)
        self.socket_path = None
        if kind == "tcp":
            self._server = _ThreadedTcpServer((rest[0], rest[1]), conn_class or _Conn)
            host, port = self._server.server_address[:2]
            self.address = format_address(rest[0] if rest[0] not in ("", "0.0.0.0", "::") else host, port)
            self.port = port
        else:
            if os.path.exists(address):
                os.unlink(address)
            self.socket_path = self.address = address
            with _unix_name(address) as name:
                self._server = _ThreadedUnixServer(name, conn_class or _Conn)
        self._server.rpc_handler = handler  # type: ignore[attr-defined]
        self._server.open_conns, self._server.open_conns_lock = set(), threading.Lock()  # type: ignore[attr-defined]
        self._thread = threading.Thread(target=self._server.serve_forever, kwargs=dict(poll_interval=0.1), daemon=True)

    def start(self) -> None:
        self._thread.start()

    def shutdown(self) -> None:
        self._server.shutdown()
        self._server.server_close()
        with self._server.open_conns_lock:  # type: ignore[attr-defined]
            conns = list(self._server.open_conns)  # type: ignore[attr-defined]
        for c in conns:
            try:
                c.shutdown(socket.SHUT_RDWR)
            except OSError:
                pass
        if self.socket_path is not None and os.path.exists(self.socket_path):
            os.unlink(self.socket_path)


# ---------------------------------------------------------------------------------------------------------
# client side
# ---------------------------------------------------------------------------------------------------------
_EXC = {"ValueError": ValueError, "KeyError": KeyError, "TimeoutError": TimeoutError, "RuntimeError": RuntimeError}


def _raise_remote(header: Dict[str, Any]) -> None:
    etype = header.get("etype", "RuntimeError")
    if etype == "AllocationFailed":
        from petals_b200.server.memory_cache import AllocationFailed

        raise AllocationFailed(header.get("error"))
    raise _EXC.get(etype, RemoteError)(header.get("error"))


class _RemoteStream:
    def __init__(self, sock: socket.socket, uids: Sequence[str], metadata: dict, compression=None):
        self._sock, self._uids, self._open_meta, self._first, self.closed = sock, list(uids), metadata, True, False
        self._compression = compression

    def step(self, *tensors: torch.Tensor, metadata: Optional[dict] = None) -> torch.Tensor:
        meta = dict(self._open_meta if self._first else {}, **(metadata or {}))
        self._first = False
        # only the hidden states (first tensor) are compressed; prompts / hypo_ids travel raw
        codecs = [self._compression] + [None] * (len(tensors) - 1)
        send_message(self._sock, {"method": "rpc_inference", "uids": self._uids, "meta": meta}, tensors, codecs)
        header, outs = recv_message(self._sock)
        if not header.get("ok"):
            _raise_remote(header)
        return outs[0]

    def close(self) -> None:
        if self.closed:
            return
        self.closed = True
        try:
            send_message(self._sock, {"method": "rpc_inference", "uids": self._uids, "close": True})
            recv_message(self._sock)
        except (OSError, ConnectionError):
            pass
        finally:
            self._sock.close()


class RemoteHandlerProxy:
    """Client stub for a stage worker living in another process (``socket_path``: unix path or ``tcp://host:port``)."""

    def __init__(self, socket_path: str, connect_timeout: float = 5.0, request_timeout: float = 180.0, compression=None):
        self.socket_path, self.connect_timeout, self.request_timeout = socket_path, connect_timeout, request_timeout
        self.compression = compression  # codec for the activations this client sends (utils/compression.py)

    def _connect(self) -> socket.socket:
        return open_connection(self.socket_path, self.connect_timeout, self.request_timeout)

    def _call(self, header: Dict[str, Any], tensors: Sequence[torch.Tensor] = ()):
        with self._connect() as s:
            send_message(s, header, tensors, self.compression if header.get("method") in ("rpc_forward", "rpc_backward", "rpc_push") else None)
            reply, outs = recv_message(s)
        if not reply.get("ok"):
            _raise_remote(reply)
        return reply, outs

    def rpc_info(self, uids=None) -> dict:
        return self._call({"method": "rpc_info", "uids": uids})[0]["meta"]

    def rpc_ping(self) -> None:
        self._call({"method": "rpc_ping"})

    def rpc_check(self, check_peer: str, wait_timeout: float = 5.0) -> bool:
        return bool(self._call({"method": "rpc_check", "meta": {"check_peer": check_peer, "wait_timeout": wait_timeout}})[0]["meta"])

    def rpc_forward(self, uids, *tensors, metadata=None) -> torch.Tensor:
        return self._call({"method": "rpc_forward", "uids": list(uids), "meta": metadata or {}}, tensors)[1][0]

    def rpc_backward(self, uids, *tensors, metadata=None) -> List[torch.Tensor]:
        return self._call({"method": "rpc_backward", "uids": list(uids), "meta": metadata or {}}, tensors)[1]

    def rpc_push(self, uids, *tensors, metadata=None) -> None:
        self._call({"method": "rpc_push", "uids": list(uids), "meta": metadata or {}}, tensors)

    def rpc_inference(self, uids, metadata=None) -> _RemoteStream:
        return _RemoteStream(self._connect(), uids, metadata or {}, self.compression)
