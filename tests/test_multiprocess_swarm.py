"""A real multi-process local swarm on CPU (BASELINE config #1, the reference CI's harness .github/workflows/run-tests.yaml:52-91):
`run_dht` rendezvous + two `run_server` OS processes + a client in this process, talking over the Unix-socket transport."""
import os
import signal
import subprocess
import sys
import time

import pytest
import torch

from petals_b200.utils.auto_config import AutoDistributedConfig, AutoDistributedModelForCausalLM
from tests.utils import checkpoint, local_blocks

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _spawn(args, log):
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""), PETALS_LOGLEVEL="INFO")
    return subprocess.Popen([sys.executable, "-m", *args], stdout=log, stderr=subprocess.STDOUT, env=env, cwd=ROOT)


@pytest.mark.parametrize("family,compression,atol", [("bloom", None, 1e-3), ("llama", "FLOAT16", 3e-2)])
def test_two_server_processes(family, compression, atol, tmp_path):
    path = checkpoint(family)
    rendezvous = str(tmp_path / "swarm")
    subprocess.run([sys.executable, "-m", "petals.cli.run_dht", "--rendezvous", rendezvous, "--once"], check=True, cwd=ROOT,
                   env=dict(os.environ, PYTHONPATH=ROOT))
    logs = [open(tmp_path / f"server{i}.log", "w") for i in range(2)]
    common = ["--initial_peers", rendezvous, "--torch_dtype", "float32", "--device", "cpu", "--throughput", "1", "--update_period", "1"]
    if compression:  # the servers answer over the socket transport in this wire codec (utils/compression.py)
        common += ["--compression", compression]
    procs = [_spawn(["petals.cli.run_server", path, "--block_indices", "0:2", "--peer_id", "stage0", *common], logs[0]),
             _spawn(["petals.cli.run_server", path, "--block_indices", "2:4", "--peer_id", "stage1", "--attn_cache_tokens", "2048",
                     "--max_chunk_size_bytes", "1024", *common], logs[1])]  # tiny chunk size => chunked prefill is exercised
    try:
        model = AutoDistributedModelForCausalLM.from_pretrained(path, initial_peers=[rendezvous], max_retries=150, min_backoff=0.5, max_backoff=1.0)
        config = AutoDistributedConfig.from_pretrained(path)
        ids = torch.randint(0, config.vocab_size, (1, 7), generator=torch.Generator().manual_seed(0))
        with torch.inference_mode():
            parallel = model(ids).logits  # waits (with retries) until both server processes are ONLINE
            assert all(p.poll() is None for p in procs), "a server process died"
            h = model.model.embed(ids)
            for b in local_blocks(path, config.num_hidden_layers):
                h = b(h)[0]
            local = model.lm_head(model.model.final_norm(h))
            embs = model.model.embed(ids)
            with model.model.layers.inference_session(max_length=8) as sess:
                outs = [sess.step(embs[:, :5])] + [sess.step(embs[:, t: t + 1]) for t in range(5, 7)]
                peers = [s.span.peer_id for s in sess._server_sessions]
            step = model.lm_head(model.model.final_norm(torch.cat(outs, 1)))
        assert peers == ["stage0", "stage1"]
        assert torch.allclose(parallel, local, atol=atol) and torch.allclose(step, local, atol=atol)
        assert (compression is None) or not torch.equal(parallel, local)
        # gradients flow through other processes too
        x = torch.randn(2, 3, config.hidden_size, requires_grad=True)
        model.model.layers(x).sum().backward()
        assert x.grad is not None and torch.isfinite(x.grad).all()
        out = model.generate(ids, max_new_tokens=3)
        assert out.shape == (1, 10)
    finally:
        for p in procs:
            p.send_signal(signal.SIGTERM)
        for p in procs:
            try:
                p.wait(timeout=10)
            except subprocess.TimeoutExpired:
                p.kill()
        for f in logs:
            f.close()


@pytest.mark.parametrize("member_client", [False, True])
def test_run_server_processes_join_a_fabric_and_serve_a_client_outside_it(member_client, tmp_path):
    """`run_server --fabric_address/--fabric_rank/--fabric_world`: two independently started stage processes form a landing-ring fabric
    (the shared-memory twin on CPU); a client that is NOT a member learns from `rpc_info` that the stages share a fabric, so hidden
    states, training micro-batches and gradients hop stage to stage through the rings and only the two ends travel with the RPCs."""
    import socket

    path = checkpoint("llama")
    rendezvous = str(tmp_path / "swarm")
    subprocess.run([sys.executable, "-m", "petals.cli.run_dht", "--rendezvous", rendezvous, "--once"], check=True, cwd=ROOT, env=dict(os.environ, PYTHONPATH=ROOT))
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    logs = [open(tmp_path / f"server{i}.log", "w") for i in range(2)]
    common = ["--initial_peers", rendezvous, "--torch_dtype", "float32", "--device", "cpu", "--throughput", "1", "--update_period", "1",
              "--fabric_address", f"127.0.0.1:{port}", "--fabric_world", "3" if member_client else "2", "--fabric_max_tokens", "256"]
    procs = [_spawn(["petals.cli.run_server", path, "--block_indices", "0:2", "--peer_id", "stage0", "--fabric_rank", "0", *common], logs[0]),
             _spawn(["petals.cli.run_server", path, "--block_indices", "2:4", "--peer_id", "stage1", "--fabric_rank", "1", *common], logs[1])]
    try:
        # member_client: this process joins the fabric as its third member (from_pretrained(..., fabric_address=...)): the last stage then
        # returns through the client's own landing ring and the client stores the output gradient into the last stage's ring
        extra = dict(fabric_address=f"127.0.0.1:{port}", fabric_rank=2, fabric_world=3, fabric_max_tokens=256, fabric_device="cpu") if member_client else {}
        model = AutoDistributedModelForCausalLM.from_pretrained(path, initial_peers=[rendezvous], max_retries=150, min_backoff=0.5, max_backoff=1.0, **extra)
        config = AutoDistributedConfig.from_pretrained(path)
        ids = torch.randint(0, config.vocab_size, (2, 9), generator=torch.Generator().manual_seed(0))
        blocks = list(local_blocks(path, config.num_hidden_layers))
        with torch.inference_mode():
            h = model.model.embed(ids)
            for b in blocks:
                h = b(h)[0]
            ref = model.lm_head(model.model.final_norm(h))
            with model.inference_session(max_length=16) as sess:
                a = model(ids[:, :6]).logits
                b_ = model(ids[:, 6:7]).logits
                c = model(ids[:, 7:]).logits
                over_fabric = [s.no_history for s in sess._server_sessions]
                same_fabric = len({s.fabric_info["id"] for s in sess._server_sessions}) == 1
            assert all(p.poll() is None for p in procs), "a server process died"
        assert torch.allclose(torch.cat([a, b_, c], 1), ref, atol=1e-3)
        assert over_fabric == [False, True] and same_fabric  # the second stage never got a tensor from the client
        # a long prompt is cut into chunks that travel as a wavefront through the landing RINGS (one slot per chunk in flight)
        chunky = AutoDistributedModelForCausalLM.from_pretrained(path, initial_peers=[rendezvous], max_retries=150, min_backoff=0.5, max_backoff=1.0,
                                                                 pipeline_chunk_tokens=2)
        chunky.load_state_dict(model.state_dict())
        from petals_b200.client.inference_session import InferenceSession

        waves, original = [], InferenceSession._pipelined_wave

        def counting(self, *a, **k):
            out = original(self, *a, **k)
            waves.append(out is not None)
            return out

        InferenceSession._pipelined_wave = counting
        try:
            with torch.inference_mode(), chunky.inference_session(max_length=16) as sess:
                d = chunky(ids[:, :8]).logits  # 4 chunks of 2 positions over 2 stages
                e = chunky(ids[:, 8:]).logits
                assert [s.no_history for s in sess._server_sessions] == [False, True]
        finally:
            InferenceSession._pipelined_wave = original
        assert waves and waves[0], "the long prompt was not ingested as a wavefront of chunks"
        assert torch.allclose(torch.cat([d, e], 1), ref, atol=1e-3)
        # training: forward micro-batches and gradients hop between the stages, the ends travel with the RPCs
        from petals_b200.client.sequential_autograd import FabricPlan

        x = torch.randn(2, 9, config.hidden_size, requires_grad=True)
        before = dict(FabricPlan.hops_done)
        y = model.model.layers(x)
        y.sum().backward()
        assert {k: FabricPlan.hops_done[k] - before[k] for k in before} == {"forward": 2, "backward": 2}
        x2 = x.detach().clone().requires_grad_(True)
        h = x2
        for b in blocks:
            h = b(h)[0]
        h.sum().backward()
        assert torch.allclose(y, h, atol=1e-4) and torch.allclose(x.grad, x2.grad, atol=1e-3)
    finally:
        for p in procs:
            p.terminate()
        for p in procs:
            try:
                p.wait(timeout=10)
            except subprocess.TimeoutExpired:
                p.kill()
        for log in logs:
            log.close()
        if member_client:
            from petals_b200.parallel.fabric import leave_fabric

            leave_fabric(True)
