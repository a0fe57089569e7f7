#!/usr/bin/env python
"""Headline benchmark (BASELINE.json): Llama-3-70B single-stream decode tokens/s (+ prefill tokens/s) on N B200s.

    python bench.py --gpus 1 --steps 32 --warmup 4
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
    python bench.py --impl reference ...   # the unmodified reference, if it could be installed (it cannot: see DESIGN.md)

Method (mirrors the reference's benchmarks/benchmark_inference.py:44-68): one inference session with
``max_length = seq_len``, then one token per step through the public client API. ``value`` is device-timed over
exactly K steps (CUDA events, barrier + synchronize on both sides, max over ranks) with tokens staying on the
device; ``e2e`` repeats the K steps with, per step, the input token copied from pinned host memory and the sampled
token read back to the host. Weights are random-init bf16 of the named architecture, prompts are synthetic ids. With
N = 1 both come from fixed seeds, so the same arguments give the same inputs, and ``--dump-outputs DIR`` writes what the
timed paths returned in their last step so that two builds can be compared output for output (the N > 1 paths draw
their prompts from the global generator and do not dump).
L2 hygiene: every decode step streams the full ~141 GB weight set (>> 126 MB L2), so inputs are larger than L2.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from petals_b200.utils.bench_common import (BASELINE_TOKENS_PER_S, ClockSampler, device_timed_decode, e2e_decode,  # noqa: E402
                                            metric_name, prime_session)


def reference_arm(args) -> None:
    """Run the UNMODIFIED reference from ``baseline/_ref`` through its own public API (none of this repo's code on that path)."""
    from baseline.reference_arm import run_reference

    line = run_reference(args)
    if int(os.environ.get("RANK", "0")) == 0:
        print(json.dumps(line))


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="llama-3-70b")
    ap.add_argument("--seq-len", type=int, default=2048, help="session max_length (reference benchmark default)")
    ap.add_argument("--prompt-len", type=int, default=128)
    ap.add_argument("--parallelism", default="auto", help="auto | ppN | tpN | ppSxtpT (S pipeline stages of T-way tensor-parallel groups, S*T = --gpus)")
    ap.add_argument("--prefill-seq", type=int, default=4096)
    ap.add_argument("--prefill-batch", type=int, default=8)
    ap.add_argument("--prefill-steps", type=int, default=2)
    ap.add_argument("--skip-prefill", action="store_true")
    ap.add_argument("--tp-prefill-rows", type=int, default=8192, help="rows per sequence-parallel prefill chunk (N > 1, tensor parallel)")
    ap.add_argument("--tp-emulate", type=int, default=0, help="DIAGNOSTIC (not a benchmark result): run the compute of ONE rank of a "
                    "tensor-parallel group of this size on one GPU (heads, KV heads and FFN columns divided), to measure the fixed per-layer costs")
    ap.add_argument("--skip-fp8", action="store_true", help="do not append the block-scaled FP8 decode measurement")
    ap.add_argument("--skip-selftests", action="store_true", help="N > 1: do not run the TP / pipeline numerics self-tests before the timed runs")
    ap.add_argument("--skip-pipeline", action="store_true", help="N > 1: do not append the pipeline-parallel record (same model as N stages)")
    ap.add_argument("--pp-chunk-tokens", type=int, default=256, help="positions per chunk of the pipelined prompt ingestion (pipeline record)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="N = 1: after the timed runs, write what each timed path returned in its last step "
                    "as DIR/<name>.npy (token ids as float64, a fixed sample of prefill hidden-state rows as float32)")
    args = ap.parse_args()
    if args.impl == "reference":
        return reference_arm(args)
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.warmup < 3:
        args.warmup = 3
    # generate() adds nothing once the session is full: make room for the prompt, the warm-up and both K-step loops
    need = args.prompt_len + args.warmup + 2 * args.steps
    if args.seq_len < need:
        print(f"note: --seq-len raised from {args.seq_len} to {need} to hold the prompt, {args.warmup} warm-up and 2 x {args.steps} "
              f"timed steps (decode runs at a longer KV length than requested)", file=sys.stderr)
        args.seq_len = need
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1 or args.gpus > 1:
        if args.dump_outputs:
            ap.error("--dump-outputs is implemented for --gpus 1 only")
        from petals_b200.parallel.multi_gpu_bench import run_multi_gpu

        return run_multi_gpu(args)
    run_single_gpu(args)


def run_single_gpu(args) -> None:
    import torch

    from petals_b200.ops import native
    from petals_b200.parallel.swarm import Swarm
    from petals_b200.utils.peaks import measured_peaks
    from petals_b200.utils.random_model import MODEL_PRESETS, launch_random_stage, random_client_model, write_config_only

    torch.cuda.set_device(0)
    dev = "cuda:0"
    native.lib()
    overrides = None
    if args.tp_emulate > 1:
        pre, R = MODEL_PRESETS[args.model], args.tp_emulate
        overrides = dict(num_attention_heads=pre["num_attention_heads"] // R, num_key_value_heads=max(1, pre["num_key_value_heads"] // R),
                         intermediate_size=pre["intermediate_size"] // R, head_dim=pre["hidden_size"] // pre["num_attention_heads"])
    path = write_config_only(args.model, overrides)
    n_layers = MODEL_PRESETS[args.model]["num_hidden_layers"]
    swarm = Swarm("bench")
    t0 = time.time()
    stage = launch_random_stage(path, range(n_layers), swarm, dev, attn_cache_tokens=max(args.seq_len, args.prefill_seq) + 256,
                                inference_max_length=max(args.seq_len, args.prefill_seq), max_batch_size=1 << 20)
    model = random_client_model(path, swarm, dev)
    torch.cuda.synchronize()
    build_s = time.time() - t0
    K, W = args.steps, args.warmup
    vocab = model.config.vocab_size
    outputs = {}
    prompt = torch.randint(0, vocab, (1, args.prompt_len), device=dev, generator=torch.Generator(dev).manual_seed(0))
    with torch.inference_mode(), model.inference_session(max_length=args.seq_len) as sess:
        prime_session(model, sess, prompt, W)  # prompt ingestion is not part of the single-stream metric, like the reference benchmark
        sampler = ClockSampler(0)
        sampler.start()
        ms, launches = device_timed_decode(model, sess, K)  # tokens never leave the GPU
        clocks = sampler.stop()
        outputs["decode_token_ids"] = sess.output_ids.double().cpu().numpy()  # what the last timed generate() returned
        e2e_s, h2d, d2h = e2e_decode(model, sess, K, dev)  # pinned-host token in, sampled token out, every step
    value = K / (ms / 1e3)
    peaks = measured_peaks()
    spec = model.config.block_spec()
    weight_bytes = (spec.active_params() * n_layers + vocab * spec.hidden_size) * 2
    result = {
        "metric": (metric_name(args.model) if args.tp_emulate <= 1 else
                   f"DIAGNOSTIC: one rank's share of a tp{args.tp_emulate} decode step on one GPU, no communication (NOT a benchmark result)"),
        "value": round(value, 3), "unit": "tokens/s", "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": round(ms / K, 4),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": round(value / BASELINE_TOKENS_PER_S, 3), "dtype": "bf16",
        "data": "synthetic token ids; random-init weights of the named architecture",
        "config": {"model": args.model, "global_batch": 1, "seq_len": args.seq_len, "parallelism": f"pp1 (1 stage x {n_layers} blocks)",
                   "l2": "each step streams the full weight set (>> 126 MB L2): inputs larger than L2", "build_s": round(build_s, 1)},
        "clocks": clocks,
        "e2e": {"value": round(K / e2e_s, 3), "unit": "tokens/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "api": "model.generate(max_new_tokens=1, session=sess) per step; token in from pinned host memory, token out to the host"},
        "gpu_launches": launches,
        "roofline": {"weight_bytes_per_token": weight_bytes, "achieved_GBps": round(weight_bytes * value / 1e9, 1),
                     "frac_of_measured_hbm": round(weight_bytes * value / 1e9 / peaks["hbm_gbs"], 3), "peaks": peaks["source"],
                     "note": "bytes = the weights one token actually reads (dense blocks: all; sparse MoE: router + top-k experts) + LM head"},
    }
    if not args.skip_prefill:
        try:
            result["prefill"] = bench_prefill(model, args, peaks, spec, n_layers, outputs, "prefill")
        except Exception as e:  # noqa: BLE001 - the headline number must survive a failure of an appendix
            result["prefill"] = {"error": repr(e)[:200]}
    stage.shutdown()
    if not args.skip_fp8:
        try:
            del stage
            import gc

            gc.collect()
            torch.cuda.empty_cache()
            result["fp8_weights"] = bench_fp8_decode(args, path, n_layers, swarm, dev, K, W, spec, vocab, peaks, outputs)
        except Exception as e:  # noqa: BLE001
            result["fp8_weights"] = {"error": repr(e)[:200]}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(result))
    if args.dump_outputs:
        expected = ["decode_token_ids"] + ([] if args.skip_prefill else ["prefill_hidden_rows"])
        if not args.skip_fp8:
            expected += ["fp8_decode_token_ids"] + ([] if args.skip_prefill else ["fp8_prefill_hidden_rows"])
        missing = [n for n in expected if n not in outputs]
        if missing:  # an appendix failed (its error is in the JSON line): the dump is incomplete
            sys.exit(f"--dump-outputs: no output from {missing}")


def dump_outputs(directory: str, outputs: dict) -> None:
    import numpy as np

    total = sum(a.nbytes for a in outputs.values())
    if total > 64 << 20:
        raise ValueError(f"{total} bytes of outputs exceed the 64 MB dump budget")
    for name, arr in outputs.items():
        if arr.dtype not in (np.float32, np.float64):
            raise TypeError(f"output {name} is {arr.dtype}, the dump holds float32 / float64 only")
    os.makedirs(directory, exist_ok=True)
    for name, arr in outputs.items():
        np.save(os.path.join(directory, f"{name}.npy"), arr)


def sample_rows(hidden, n: int = 256):
    """A fixed, seeded sample of ``n`` rows of [..., H] hidden states, as float32 on the host (the full output is GBs)."""
    import torch

    flat = hidden.reshape(-1, hidden.shape[-1])
    rows = torch.randperm(flat.shape[0], generator=torch.Generator().manual_seed(0))[:n].sort().values
    return flat[rows.to(flat.device)].float().cpu().numpy()


def bench_fp8_decode(args, path, n_layers, swarm, dev, K, W, spec, vocab, peaks, outputs) -> dict:
    """Same single-stream loop with the blocks served as block-scaled FP8 (MXFP8) weights — what `--quant_type fp8` serves in place
    of the reference's default NF4/INT8 (bitsandbytes has no sm_100 kernels). Compute stays bf16/fp32; reported next to, not
    instead of, the bf16 headline."""
    import torch

    from petals_b200.utils.convert_block import QuantType
    from petals_b200.utils.random_model import launch_random_stage, random_client_model

    stage = launch_random_stage(path, range(n_layers), swarm, dev, attn_cache_tokens=args.seq_len + 256, inference_max_length=args.seq_len,
                                max_batch_size=1 << 20, quant_type=QuantType.FP8, peer_id="fp8-stage")
    try:
        model = random_client_model(path, swarm, dev)
        model.model.layers.sequence_manager.update(wait=True)
        prompt = torch.randint(0, vocab, (1, 8), device=dev, generator=torch.Generator(dev).manual_seed(0))
        with torch.inference_mode(), model.inference_session(max_length=args.seq_len) as sess:
            prime_session(model, sess, prompt, W)
            ms, _ = device_timed_decode(model, sess, K)
            outputs["fp8_decode_token_ids"] = sess.output_ids.double().cpu().numpy()
        value = K / (ms / 1e3)
        weight_bytes = spec.active_params() * n_layers * (1 + 1 / 32) + vocab * spec.hidden_size * 2
        rec = {"tokens_per_s": round(value, 3), "ms_per_step": round(ms / K, 4), "weight_bytes_per_token": int(weight_bytes),
               "frac_of_measured_hbm": round(weight_bytes * value / 1e9 / peaks["hbm_gbs"], 3), "format": "E4M3 + UE8M0 scale per 32 (MXFP8)"}
        if not args.skip_prefill:
            # prompt ingestion with BOTH operands in MXFP8 on the block-scaled tensor-core path (csrc/gemm_mxfp8.cu)
            try:
                pf = bench_prefill(model, args, peaks, spec, n_layers, outputs, "fp8_prefill")
                pf["path"] = ("tcgen05.mma kind::mxf8f6f4.block_scale, activations quantised per 32 values (fused with the RMSNorm)"
                              if getattr(stage.stage.engine, "fp8_w8a8", False) else "weights dequantised per projection, bf16 tcgen05 GEMM")
                rec["prefill"] = pf
            except Exception as e:  # noqa: BLE001
                rec["prefill"] = {"error": repr(e)[:200]}
        return rec
    finally:
        stage.shutdown()


def bench_prefill(model, args, peaks, spec, n_layers, outputs, name) -> dict:
    """Parallel forward (benchmark_forward.py analogue): tokens/s = B*T / step time, no LM head."""
    import torch

    dev = "cuda:0"
    B, T = args.prefill_batch, args.prefill_seq
    ids = torch.randint(0, model.config.vocab_size, (B, T), device=dev, generator=torch.Generator(dev).manual_seed(1))
    with torch.inference_mode():
        for _ in range(1):
            model.model(input_ids=ids)
        torch.cuda.synchronize()
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        for _ in range(args.prefill_steps):
            out = model.model(input_ids=ids)
        end.record()
        torch.cuda.synchronize()
        outputs[f"{name}_hidden_rows"] = sample_rows(out.last_hidden_state)
    ms = start.elapsed_time(end) / args.prefill_steps
    flops = 2.0 * spec.active_params() * n_layers * B * T + 4.0 * n_layers * B * T * T * spec.num_heads * spec.head_dim / 2
    return {"tokens_per_s": round(B * T / (ms / 1e3), 1), "ms_per_step": round(ms, 2), "batch": B, "seq_len": T,
            "TFLOPs": round(flops / ms / 1e9, 1), "frac_of_measured_bf16_sustained": round(flops / ms / 1e9 / peaks["bf16_tflops_sustained"], 3)}


if __name__ == "__main__":
    main()
