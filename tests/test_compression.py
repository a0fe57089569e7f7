"""Wire codecs of the socket transport (utils/compression.py).

The reference takes its codecs from hivemind and only tests them indirectly (a server started with
``--compression`` in CI); here they are in-tree, so each one is checked against the uncompressed tensor and the
whole path (client -> socket -> handler -> socket -> client) is exercised with per-request ``output_compression``.
"""
import os
import tempfile

import pytest
import torch

from petals_b200.parallel.transport import RemoteHandlerProxy, RpcServer
from petals_b200.utils.compression import (CompressionType, compressed_nbytes, decode, encode, normalize_output_compression,
                                           parse_compression, roundtrip)


def _hidden(shape=(2, 37, 512), dtype=torch.bfloat16, seed=0, outliers=True):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(*shape, generator=g) * 0.7
    if outliers:
        x[..., 3] *= 40  # an outlier feature, as in real transformer hidden states
    return x.to(dtype)


def test_parse_compression_names_and_numbers():
    assert parse_compression(None) is CompressionType.NONE
    assert parse_compression("float16") is CompressionType.FLOAT16
    assert parse_compression(int(CompressionType.BLOCKWISE_8BIT)) is CompressionType.BLOCKWISE_8BIT
    assert parse_compression(CompressionType.UNIFORM_8BIT) is CompressionType.UNIFORM_8BIT
    with pytest.raises(ValueError):
        parse_compression("zstd")


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
def test_none_is_exact(dtype):
    x = _hidden(dtype=dtype)
    y = roundtrip(x, "NONE")
    assert y.dtype == dtype and torch.equal(x, y)


# relative RMS error a codec may introduce on the synthetic hidden states above. The two global-codebook codecs put
# every outlier into their end buckets (beyond ±6σ / the last 1/256 quantile), so they are only meant for — and
# checked on — outlier-free tensors; the per-row and per-block codecs must cope with the outlier feature.
_GLOBAL_CODEBOOK = ("UNIFORM_8BIT", "QUANTILE_8BIT")
_RMS_BOUND = {"FLOAT16": 1e-3, "MEANSTD_16BIT": 2e-3, "UNIFORM_8BIT": 0.03, "QUANTILE_8BIT": 0.05, "BLOCKWISE_8BIT": 0.03,
              "MXFP8": 0.04}  # E4M3 has 3 mantissa bits: <= 6.25 % per value, ~2.5-3 % RMS; a power-of-two scale per 32 values keeps outliers local


@pytest.mark.parametrize("codec", sorted(_RMS_BOUND))
def test_lossy_codecs_are_close_and_smaller(codec):
    x = _hidden(dtype=torch.float32, outliers=codec not in _GLOBAL_CODEBOOK)
    y = roundtrip(x, codec)
    assert y.shape == x.shape and y.dtype == x.dtype
    rel = ((y - x).pow(2).mean().sqrt() / x.pow(2).mean().sqrt()).item()
    assert rel < _RMS_BOUND[codec], (codec, rel)
    ratio = compressed_nbytes(x, codec) / compressed_nbytes(x, "NONE")
    assert ratio < (0.55 if "16" in codec else 0.30), (codec, ratio)


@pytest.mark.parametrize("codec", sorted(_RMS_BOUND))
def test_codecs_restore_dtype_and_handle_odd_sizes(codec):
    for shape in [(1,), (5, 1), (3, 4099), (1, 1, 7)]:
        x = _hidden(shape=shape, dtype=torch.bfloat16, seed=3) if shape[-1] > 3 else torch.randn(*shape).to(torch.bfloat16)
        y = roundtrip(x, codec)
        assert y.dtype == torch.bfloat16 and y.shape == x.shape
        assert torch.isfinite(y.float()).all()


def test_mxfp8_codec_is_the_tensor_core_format():
    """The MXFP8 wire codec is ops/quant.py's format (E4M3 payload + one UE8M0 exponent per 32 values): what an fp8 stage would feed its
    block-scaled GEMM, so a receiver could consume the payload without a dequantise / requantise round trip."""
    from petals_b200.ops.quant import dequantize_mxfp8, quantize_mxfp8
    from petals_b200.utils.compression import encode

    x = _hidden(shape=(4, 256), dtype=torch.float32, seed=5)
    meta, blobs = encode(x, "MXFP8")
    q, e = quantize_mxfp8(x.reshape(-1, 32))
    assert meta["codec"] == "MXFP8" and torch.equal(blobs[0], q.view(torch.uint8).reshape(-1)) and torch.equal(blobs[1], e.reshape(-1))
    assert torch.equal(roundtrip(x, "MXFP8"), dequantize_mxfp8(q, e, torch.float32).reshape(4, 256))
    assert abs(compressed_nbytes(x, "MXFP8") / x.numel() - (1 + 1 / 32)) < 1e-6


def test_float16_clamps_instead_of_overflowing():
    x = torch.tensor([1e6, -1e6, 1.0])
    y = roundtrip(x, "FLOAT16")
    assert torch.isfinite(y).all() and y[0] > 6e4 and y[1] < -6e4


def test_blockwise_scales_each_block_separately():
    x = torch.cat([torch.randn(4096) * 1e-3, torch.randn(4096) * 1e3])
    y = roundtrip(x, "BLOCKWISE_8BIT")
    for lo in (0, 4096):  # the tiny block is not flushed to zero by the huge one
        seg, ref = y[lo:lo + 4096], x[lo:lo + 4096]
        assert ((seg - ref).pow(2).mean().sqrt() / ref.pow(2).mean().sqrt()) < 0.05


def test_integer_and_empty_tensors_travel_raw():
    ids = torch.arange(10)
    meta, blobs = encode(ids, "QUANTILE_8BIT")
    assert meta["codec"] == "NONE" and torch.equal(decode(meta, blobs, ids.dtype, ids.shape), ids)
    meta, blobs = encode(torch.empty(0), "FLOAT16")
    assert meta["codec"] == "NONE" and decode(meta, blobs, torch.float32, (0,)).numel() == 0


def test_output_compression_validation():
    assert normalize_output_compression(None, 2, "FLOAT16") == [CompressionType.FLOAT16] * 2
    assert normalize_output_compression([0, "UNIFORM_8BIT"], 2) == [CompressionType.NONE, CompressionType.UNIFORM_8BIT]
    with pytest.raises(ValueError):
        normalize_output_compression(2, 1)
    with pytest.raises(ValueError):
        normalize_output_compression([0, 0], 1)
    with pytest.raises(ValueError):
        normalize_output_compression([17], 1)


class _EchoStream:
    def __init__(self):
        self.closed = False

    def step(self, hidden, *rest, metadata=None):
        return hidden * 2

    def close(self):
        self.closed = True


class _EchoHandler:
    compression = None

    def rpc_inference(self, uids, metadata=None):
        return _EchoStream()

    def rpc_forward(self, uids, hidden, *rest, metadata=None):
        return hidden + 1

    def rpc_backward(self, uids, inputs, grads, *rest, metadata=None):
        return [grads, inputs[:, :1]]

    def rpc_info(self, uids=None):
        return {"ok": True}


@pytest.fixture
def echo_server():
    with tempfile.TemporaryDirectory() as d:
        handler = _EchoHandler()
        server = RpcServer(handler, os.path.join(d, "s.sock"))
        server.start()
        try:
            yield handler, server.socket_path
        finally:
            server.shutdown()


def test_transport_default_is_exact(echo_server):
    _, path = echo_server
    x = _hidden()
    out = RemoteHandlerProxy(path).rpc_forward(["m.0"], x)
    assert torch.equal(out, x + 1)


def test_unix_socket_in_a_deep_directory(tmp_path):
    """A rendezvous directory may sit under a long temp path: a socket path longer than sun_path's 108 bytes still serves."""
    deep = tmp_path / ("d" * 60) / ("e" * 60)
    deep.mkdir(parents=True)
    path = str(deep / "s.sock")
    assert len(path) > 108
    server = RpcServer(_EchoHandler(), path)
    server.start()
    try:
        x = _hidden()
        assert torch.equal(RemoteHandlerProxy(path).rpc_forward(["m.0"], x), x + 1)
    finally:
        server.shutdown()
    assert not os.path.exists(path)


def test_transport_server_default_and_per_request_override(echo_server):
    handler, path = echo_server
    x = _hidden(dtype=torch.float32)
    handler.compression = "BLOCKWISE_8BIT"
    proxy = RemoteHandlerProxy(path)
    lossy = proxy.rpc_forward(["m.0"], x)
    assert not torch.equal(lossy, x + 1) and torch.allclose(lossy, x + 1, atol=0.5, rtol=0.05)
    exact = proxy.rpc_forward(["m.0"], x, metadata={"output_compression": [0]})  # the client overrides the server default
    assert torch.equal(exact, x + 1)
    with pytest.raises(Exception, match="output_compression"):
        proxy.rpc_forward(["m.0"], x, metadata={"output_compression": [0, 0]})
    g, gp = proxy.rpc_backward(["m.0"], x, x * 3, metadata={"output_compression": ["FLOAT16", "NONE"]})
    assert torch.allclose(g, x * 3, rtol=2e-3, atol=1e-3) and torch.equal(gp, x[:, :1])


def test_transport_compressed_requests_and_sticky_stream_codec(echo_server):
    _, path = echo_server
    x = _hidden(dtype=torch.bfloat16)
    proxy = RemoteHandlerProxy(path, compression="FLOAT16")  # the client compresses what it sends
    stream = proxy.rpc_inference(["m.0"], {"output_compression": ["MEANSTD_16BIT"], "max_length": 8})
    try:
        hypo = torch.arange(2)
        for _ in range(3):  # the codec asked for when the session was opened applies to every step
            out = stream.step(x, torch.empty(0), hypo, metadata={})
            assert out.dtype == x.dtype
            assert torch.allclose(out.float(), x.float() * 2, rtol=2e-2, atol=2e-2)
    finally:
        stream.close()


def test_descriptor_must_match_payload():
    """The shape in a received header is untrusted: a payload that is shorter (or empty) must never turn into uninitialised
    memory of the announced shape, and meta-driven sizes are checked too."""
    import pytest
    import torch

    from petals_b200.utils.compression import WireFormatError, decode

    with pytest.raises(WireFormatError):
        decode({"codec": "NONE"}, [torch.empty(0, dtype=torch.uint8)], torch.float32, [4, 1024, 8192])
    with pytest.raises(WireFormatError):
        decode({"codec": "NONE"}, [torch.zeros(12, dtype=torch.uint8)], torch.float32, [4])
    with pytest.raises(WireFormatError):
        decode({"codec": "FLOAT16"}, [torch.zeros(6, dtype=torch.uint8)], torch.float32, [4])
    with pytest.raises(WireFormatError):
        decode({"codec": "NONE"}, [torch.zeros(16, dtype=torch.uint8)], torch.float32, [-4, -1])
    with pytest.raises(WireFormatError):
        decode({"codec": "MEANSTD_16BIT", "rows": 3}, [torch.zeros(8, dtype=torch.uint8)] * 3, torch.float32, [4])
    with pytest.raises(WireFormatError):
        decode({"codec": "BLOCKWISE_8BIT", "n": 1 << 40}, [torch.zeros(8, dtype=torch.uint8)] * 2, torch.float32, [4])
    assert decode({"codec": "NONE"}, [torch.empty(0, dtype=torch.uint8)], torch.float32, [0, 8]).shape == (0, 8)  # "argument absent"


def test_socket_frame_with_shape_but_no_bytes_is_a_protocol_error():
    import socket
    import struct

    import msgpack
    import pytest

    from petals_b200.parallel.transport import ProtocolError, recv_message

    a, b = socket.socketpair()
    try:
        header = msgpack.packb({"method": "rpc_forward", "tensors": [{"dtype": "float32", "shape": [2, 64, 8192], "nbytes": 0, "parts": [0], "c": {"codec": "NONE"}}]})
        a.sendall(struct.pack("<I", len(header)) + header)
        with pytest.raises(ProtocolError):
            recv_message(b)
    finally:
        a.close()
        b.close()
