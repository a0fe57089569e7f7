"""Numerics of every sm_100a kernel against a plain PyTorch fp32 reference of the same op."""
import math

import pytest
import torch

from petals_b200.ops import functional as Fn

pytestmark = pytest.mark.gpu
_MN_DEFAULT = __import__("os").environ.get("PETALS_B200_GEMM_2CTA_MN", "1") != "0"
DEV = "cuda"


def _rand(*shape, scale=1.0, seed=None):
    if seed is not None:
        torch.manual_seed(seed)
    return (torch.randn(*shape, device=DEV, dtype=torch.float32) * scale).to(torch.bfloat16)


def _close(got, want, atol, rtol, what=""):
    got, want = got.float(), want.float()
    err = (got - want).abs()
    tol = atol + rtol * want.abs()
    bad = (err > tol).float().mean().item()
    assert bad < 1e-3, f"{what}: {bad * 100:.3f}% elements out of tolerance, max err {err.max().item():.4g}"


@pytest.mark.parametrize("M", [1, 2, 3, 4, 8])
@pytest.mark.parametrize("N,K", [(1024, 512), (4096, 4096), (2050, 1032)])
def test_linear_decode_plain(M, N, K):
    torch.manual_seed(0)
    x, w = _rand(M, K), _rand(N, K, scale=K ** -0.5)
    got = Fn.linear_decode(x, w)
    _close(got, Fn.linear_ref(x, w), 2e-2, 2e-2, "plain")


@pytest.mark.parametrize("M", [1, 4])
def test_linear_decode_rmsnorm_residual(M):
    torch.manual_seed(1)
    K, N = 4096, 6144
    x, w, g, res = _rand(M, K), _rand(N, K, scale=K ** -0.5), _rand(K) * 0.1 + 1, _rand(M, N)
    got = Fn.linear_decode(x, w, norm_weight=g, norm_kind=Fn.NORM_RMS, eps=1e-5, residual=res)
    want = Fn.linear_ref(x, w, norm_weight=g, norm_kind=Fn.NORM_RMS, eps=1e-5, residual=res)
    _close(got, want, 3e-2, 2e-2, "rmsnorm+residual")


def test_linear_decode_layernorm_gelu_bias():
    torch.manual_seed(2)
    M, K, N = 2, 1024, 4096
    x, w = _rand(M, K), _rand(N, K, scale=K ** -0.5)
    g, b, bias = _rand(K) * 0.1 + 1, _rand(K) * 0.1, _rand(N) * 0.1
    got = Fn.linear_decode(x, w, norm_weight=g, norm_bias=b, norm_kind=Fn.NORM_LAYER, eps=1e-5, bias=bias, act=Fn.ACT_GELU_TANH)
    want = Fn.linear_ref(x, w, norm_weight=g, norm_bias=b, norm_kind=Fn.NORM_LAYER, eps=1e-5, bias=bias, act=Fn.ACT_GELU_TANH)
    _close(got, want, 2e-2, 2e-2, "layernorm+gelu")


@pytest.mark.parametrize("M", [1, 3])
def test_linear_decode_swiglu(M):
    torch.manual_seed(3)
    K, N = 2048, 5632
    x, wg, wu, g = _rand(M, K), _rand(N, K, scale=K ** -0.5), _rand(N, K, scale=K ** -0.5), _rand(K) * 0.1 + 1
    got = Fn.linear_decode(x, wg, w2=wu, act=Fn.ACT_SWIGLU, norm_weight=g, norm_kind=Fn.NORM_RMS, eps=1e-5)
    want = Fn.linear_ref(x, wg, w2=wu, act=Fn.ACT_SWIGLU, norm_weight=g, norm_kind=Fn.NORM_RMS, eps=1e-5)
    _close(got, want, 2e-2, 3e-2, "swiglu")


def test_linear_decode_reduce_parts():
    """Tensor-parallel prologue: x = residual + sum(parts), written back as the new residual stream."""
    torch.manual_seed(4)
    M, K, N = 2, 2048, 2048
    res, parts = _rand(M, K), [_rand(M, K) for _ in range(4)]
    w, g = _rand(N, K, scale=K ** -0.5), _rand(K) * 0.1 + 1
    x_out = torch.zeros(M, K, device=DEV, dtype=torch.bfloat16)
    got = Fn.linear_decode(res, w, norm_weight=g, norm_kind=Fn.NORM_RMS, eps=1e-5, parts=parts, x_out=x_out)
    xs = (res.float() + sum(p.float() for p in parts)).to(torch.bfloat16)
    _close(x_out, xs, 1e-2, 1e-2, "reduced x")
    _close(got, Fn.linear_ref(xs, w, norm_weight=g, norm_kind=Fn.NORM_RMS, eps=1e-5), 3e-2, 2e-2, "reduce+norm+gemv")


@pytest.mark.parametrize("M,N,K", [(128, 256, 64), (128, 256, 512), (256, 512, 1024), (1000, 4096, 4096), (77, 1024, 2048), (4096, 8192, 1024)])
def test_gemm_plain(M, N, K):
    torch.manual_seed(5)
    a, b = _rand(M, K), _rand(N, K, scale=K ** -0.5)
    got = Fn.gemm(a, b)
    _close(got, Fn.linear_ref(a, b), 2e-2, 2e-2, f"gemm {M}x{N}x{K}")


@pytest.mark.parametrize("M,N,K", [(1024, 1024, 512), (1100, 2048 + 64, 1024), (4096, 8192, 1024), (2048, 1280, 8192)])
def test_gemm_2cta_matches_the_1cta_kernel(M, N, K):
    """csrc/gemm_tcgen05_2cta.cu (tcgen05.mma.cta_group::2: one 256 x 256 tile per SM pair): same products and the same fp32
    accumulation order per output as the 1-CTA kernel, so the results must agree to the bf16 rounding of the output — plain, with the
    residual epilogue, and with the SwiGLU epilogue (gate rows staged by the even CTA, up rows by the odd one). Ragged M and N tails."""
    torch.manual_seed(55)
    a, b, b2, res = _rand(M, K), _rand(N, K, scale=K ** -0.5), _rand(N, K, scale=K ** -0.5), _rand(M, N)
    bt = b.t().contiguous()  # [K, N]: the dgrad view of a weight (B consumed MN-major)

    def run():
        return [Fn.gemm(a, b), Fn.gemm(a, b, residual=res), Fn.gemm(a, b, b2=b2, act=Fn.ACT_SWIGLU), Fn.gemm(a, bt, b_mn_major=True)]

    try:
        Fn.set_gemm_2cta(False)
        want = run()
        Fn.set_gemm_2cta(True)
        got = run()
    finally:
        Fn.set_gemm_2cta(True, fp8=False, mn=_MN_DEFAULT)  # the defaults
    _close(got[0], Fn.linear_ref(a, b), 2e-2, 2e-2, f"2cta gemm {M}x{N}x{K}")
    # the flag-wait prologue (sequence-parallel prefill: the A rows are gathered by peers) with an already satisfied flag
    epoch, flag, err = torch.full((1,), 3, dtype=torch.int64, device=DEV), torch.full((1,), 6, dtype=torch.int64, device=DEV), torch.zeros(1, dtype=torch.int32, device=DEV)
    waited = Fn.gemm(a, b, wait_flag=flag.data_ptr(), wait_per_epoch=2, epoch=epoch.data_ptr(), error_flag=err.data_ptr())
    assert torch.equal(waited, got[0]) and int(err.item()) == 0
    for g, w, what in zip(got, want, ("plain", "residual", "swiglu", "MN-major B")):
        assert (g.float() - w.float()).abs().max().item() <= 2e-2 * w.float().abs().max().item(), what
        assert (g.float() - w.float()).abs().mean().item() <= 2e-3 * w.float().abs().mean().item() + 1e-6, what
    assert (got[3].float() - got[0].float()).abs().max().item() <= 2e-2 * got[0].float().abs().max().item()  # a . (b^T)^T == a . b^T


@pytest.mark.parametrize("bn", [64, 128, 256])
def test_gemm_block_n(bn):
    torch.manual_seed(6)
    M, N, K = 384, 1024, 768
    a, b = _rand(M, K), _rand(N, K, scale=K ** -0.5)
    _close(Fn.gemm(a, b, block_n=bn), Fn.linear_ref(a, b), 2e-2, 2e-2, f"gemm bn={bn}")


def test_gemm_bias_gelu_residual():
    torch.manual_seed(7)
    M, N, K = 300, 2048, 1024
    a, b, bias, res = _rand(M, K), _rand(N, K, scale=K ** -0.5), _rand(N) * 0.1, _rand(M, N)
    got = Fn.gemm(a, b, bias=bias, act=Fn.ACT_GELU_TANH)
    _close(got, Fn.linear_ref(a, b, bias=bias, act=Fn.ACT_GELU_TANH), 2e-2, 2e-2, "bias+gelu")
    got = Fn.gemm(a, b, residual=res)
    _close(got, Fn.linear_ref(a, b, residual=res), 3e-2, 2e-2, "residual")


def test_gemm_swiglu():
    torch.manual_seed(8)
    M, N, K = 520, 2816, 1024
    a, wg, wu = _rand(M, K), _rand(N, K, scale=K ** -0.5), _rand(N, K, scale=K ** -0.5)
    got = Fn.gemm(a, wg, b2=wu, act=Fn.ACT_SWIGLU)
    _close(got, Fn.linear_ref(a, wg, w2=wu, act=Fn.ACT_SWIGLU), 2e-2, 3e-2, "gemm swiglu")


@pytest.mark.parametrize("bn", [64, 256])
def test_gemm_b_transposed(bn):
    """dgrad form: out = a[M,K] @ b[K,N] with b consumed MN-major straight from the nn.Linear weight."""
    torch.manual_seed(9)
    M, N, K = 256, 1024, 512
    a, b = _rand(M, K), _rand(K, N, scale=K ** -0.5)
    got = Fn.gemm(a, b, b_mn_major=True, block_n=bn)
    want = (a.float() @ b.float()).to(torch.bfloat16)
    _close(got, want, 2e-2, 2e-2, "gemm MN-major B")


def test_gemm_fp32_out():
    torch.manual_seed(10)
    M, N, K = 256, 512, 1024
    a, b = _rand(M, K), _rand(N, K, scale=K ** -0.5)
    got = Fn.gemm(a, b, out_fp32=True)
    assert got.dtype == torch.float32
    _close(got, a.float() @ b.float().T, 2e-3, 2e-3, "fp32 out")


@pytest.mark.parametrize("kind", [Fn.NORM_RMS, Fn.NORM_LAYER])
def test_norm(kind):
    torch.manual_seed(11)
    x, res = _rand(37, 4096), _rand(37, 4096)
    w, b = _rand(4096) * 0.1 + 1, (_rand(4096) * 0.1 if kind == Fn.NORM_LAYER else None)
    s = torch.empty_like(x)
    got = Fn.norm(x, w, b, kind=kind, eps=1e-5, residual=res, sum_out=s)
    xs = (x.float() + res.float()).to(torch.bfloat16)
    _close(s, xs, 1e-2, 1e-2, "sum_out")
    _close(got, Fn.norm_ref(xs, w, b, kind, 1e-5), 2e-2, 2e-2, "norm")


def test_elementwise():
    torch.manual_seed(12)
    g, u = _rand(16, 1024), _rand(16, 1024)
    want = (torch.nn.functional.silu(g.float()).to(torch.bfloat16).float() * u.float()).to(torch.bfloat16)
    _close(Fn.swiglu(g, u), want, 1e-2, 2e-2, "swiglu")
    _close(Fn.add(g, u), (g.float() + u.float()).to(torch.bfloat16), 1e-2, 1e-2, "add")
    table = _rand(1000, 512)
    ids = torch.randint(0, 1000, (3, 7), device=DEV)
    assert torch.equal(Fn.embedding(table, ids), table[ids])
    logits = torch.randn(5, 32003, device=DEV)
    assert torch.equal(Fn.argmax(logits), logits.argmax(-1))
    lb = logits.to(torch.bfloat16)
    assert torch.equal(lb.float().max(-1).values, lb.float().gather(-1, Fn.argmax(lb)[:, None])[:, 0])
    h, pr = _rand(2, 5, 256), _rand(2, 3, 256)
    want = h.clone()
    want[:, :3] = (want[:, :3].float() + pr.float()).to(torch.bfloat16)
    _close(Fn.add_prompts(h.clone(), pr), want, 1e-2, 1e-2, "add_prompts")


def _paged_setup(B, L_max, Hkv, D, n_extra_pages=3, seed=0):
    """A pool with shuffled page ids and per-sequence block tables."""
    torch.manual_seed(seed)
    pages_per_seq = (L_max + Fn.PAGE - 1) // Fn.PAGE
    n_pages = B * pages_per_seq + n_extra_pages
    perm = torch.randperm(n_pages)[: B * pages_per_seq].to(torch.int32)
    table = perm.view(B, pages_per_seq).contiguous().to(DEV)
    k_pool = torch.zeros(n_pages, Hkv, Fn.PAGE, D, device=DEV, dtype=torch.bfloat16)
    v_pool = torch.zeros_like(k_pool)
    return k_pool, v_pool, table


def _gather_cache(pool, table, L):
    """[B, L, Hkv, D] view of the paged cache."""
    B = table.shape[0]
    out = []
    for b in range(B):
        pages = pool[table[b].long()]  # [P, Hkv, PAGE, D]
        seq = pages.permute(0, 2, 1, 3).reshape(-1, pool.shape[1], pool.shape[3])
        out.append(seq[:L])
    return torch.stack(out)


@pytest.mark.parametrize("D,Hq,Hkv", [(128, 8, 2), (64, 4, 4)])
@pytest.mark.parametrize("steps", [[10, 1, 1], [70, 3], [130, 1]])
def test_rope_kv_and_attention(D, Hq, Hkv, steps):
    """Multi-step session: append with RoPE, attend; compare with the dense fp32 oracle at every step."""
    torch.manual_seed(13)
    B, L_max = 2, sum(steps)
    k_pool, v_pool, table = _paged_setup(B, L_max, Hkv, D)
    cos, sin = Fn.rope_tables(D, 512, theta=10000.0, device=DEV)
    pos = torch.zeros(1, dtype=torch.int32, device=DEV)
    k_all = torch.zeros(B, 0, Hkv, D, device=DEV, dtype=torch.bfloat16)
    v_all = torch.zeros_like(k_all)
    scale = D ** -0.5
    p0 = 0
    for T in steps:
        qkv = _rand(B, T, (Hq + 2 * Hkv) * D)
        q_out = torch.empty(B, T, Hq, D, device=DEV, dtype=torch.bfloat16)
        Fn.rope_kv_append(qkv, q_out, k_pool, v_pool, table, pos.data_ptr(), cos, sin, B=B, T=T, Hq=Hq, Hkv=Hkv, D=D)
        q, k, v = qkv.view(B, T, Hq + 2 * Hkv, D).split([Hq, Hkv, Hkv], dim=2)
        q_ref = Fn.rope_ref(q, cos[p0:p0 + T], sin[p0:p0 + T])
        k_ref = Fn.rope_ref(k, cos[p0:p0 + T], sin[p0:p0 + T])
        k_all, v_all = torch.cat([k_all, k_ref], 1), torch.cat([v_all, v], 1)
        _close(q_out, q_ref, 1e-2, 1e-2, "rope q")
        _close(_gather_cache(k_pool, table, p0 + T), k_all, 1e-2, 1e-2, "cache k")
        _close(_gather_cache(v_pool, table, p0 + T), v_all, 1e-2, 1e-2, "cache v")
        want = Fn.attention_ref(q_ref, k_all, v_all, pos0=p0, scale=scale)
        for splits in (1, 3):
            out = torch.empty(B, T, Hq, D, device=DEV, dtype=torch.bfloat16)
            po = torch.empty(splits, B * T * Hq, D, device=DEV, dtype=torch.float32)
            pl = torch.empty(splits, B * T * Hq, device=DEV, dtype=torch.float32)
            Fn.paged_attention(q_out, k_pool, v_pool, table, pos.data_ptr(), out, B=B, T=T, Hq=Hq, Hkv=Hkv, D=D,
                               scale=scale, splits=splits, partial_o=po, partial_lse=pl)
            _close(out, want, 2e-2, 2e-2, f"attention T={T} splits={splits}")
            if splits > 1:  # combine fused into the attention kernel (last split CTA merges), twice: the counters self-reset
                ctr = torch.zeros(256, device=DEV, dtype=torch.int32)
                for _ in range(2):
                    out2 = torch.full_like(out, float("nan"))
                    Fn.paged_attention(q_out, k_pool, v_pool, table, pos.data_ptr(), out2, B=B, T=T, Hq=Hq, Hkv=Hkv, D=D,
                                       scale=scale, splits=splits, partial_o=po, partial_lse=pl, split_counter=ctr, impl=1)
                    _close(out2, want, 2e-2, 2e-2, f"attention T={T} splits={splits} fused combine")
                assert int(ctr.abs().sum().item()) == 0
        pos += T
        p0 += T


def test_attention_alibi_window_long():
    torch.manual_seed(14)
    B, T, Hq, Hkv, D = 1, 300, 4, 4, 64
    k_pool, v_pool, table = _paged_setup(B, T, Hkv, D)
    pos = torch.zeros(1, dtype=torch.int32, device=DEV)
    qkv = _rand(B, T, (Hq + 2 * Hkv) * D)
    q_out = torch.empty(B, T, Hq, D, device=DEV, dtype=torch.bfloat16)
    Fn.rope_kv_append(qkv, q_out, k_pool, v_pool, table, pos.data_ptr(), None, None, B=B, T=T, Hq=Hq, Hkv=Hkv, D=D)
    q, k, v = qkv.view(B, T, Hq + 2 * Hkv, D).split([Hq, Hkv, Hkv], dim=2)
    slopes = torch.tensor([2 ** (-8 * (i + 1) / Hq) for i in range(Hq)], device=DEV)
    out = torch.empty_like(q_out)
    Fn.paged_attention(q_out, k_pool, v_pool, table, pos.data_ptr(), out, B=B, T=T, Hq=Hq, Hkv=Hkv, D=D, scale=D ** -0.5, alibi_slopes=slopes)
    _close(out, Fn.attention_ref(q, k, v, pos0=0, scale=D ** -0.5, alibi_slopes=slopes), 2e-2, 2e-2, "alibi")
    Fn.paged_attention(q_out, k_pool, v_pool, table, pos.data_ptr(), out, B=B, T=T, Hq=Hq, Hkv=Hkv, D=D, scale=D ** -0.5, window=100)
    _close(out, Fn.attention_ref(q, k, v, pos0=0, scale=D ** -0.5, window=100), 2e-2, 2e-2, "window")


@pytest.mark.parametrize("M", [1, 3])
def test_linear_decode_fp8(M):
    """Block-scaled FP8 weights: exact vs the dequantised-weight oracle (same weights), close to the bf16 original."""
    from petals_b200.ops.quant import dequantize_mxfp8, quantize_mxfp8

    torch.manual_seed(20)
    K, N = 4096, 3072
    x, g = _rand(M, K), _rand(K) * 0.1 + 1
    w, wu, res = _rand(N, K, scale=K ** -0.5), _rand(N, K, scale=K ** -0.5), _rand(M, N)
    q, e = quantize_mxfp8(w)
    qu, eu = quantize_mxfp8(wu)
    wd, wud = dequantize_mxfp8(q, e), dequantize_mxfp8(qu, eu)
    got = Fn.linear_decode_fp8(x, q, e, norm_weight=g, norm_kind=Fn.NORM_RMS, eps=1e-5, residual=res)
    _close(got, Fn.linear_ref(x, wd, norm_weight=g, norm_kind=Fn.NORM_RMS, eps=1e-5, residual=res), 3e-2, 2e-2, "fp8 plain")
    rel = (got.float() - Fn.linear_ref(x, w, norm_weight=g, norm_kind=Fn.NORM_RMS, eps=1e-5, residual=res).float()).abs().mean() / got.float().abs().mean()
    assert rel < 0.06, f"fp8 quantisation error too large: {rel}"
    got = Fn.linear_decode_fp8(x, q, e, w2_q=qu, w2_scale=eu, act=Fn.ACT_SWIGLU, norm_weight=g, norm_kind=Fn.NORM_RMS, eps=1e-5)
    _close(got, Fn.linear_ref(x, wd, w2=wud, act=Fn.ACT_SWIGLU, norm_weight=g, norm_kind=Fn.NORM_RMS, eps=1e-5), 2e-2, 3e-2, "fp8 swiglu")


def test_dequant_mxfp8():
    from petals_b200.ops.quant import dequantize_mxfp8, quantize_mxfp8

    torch.manual_seed(21)
    w = _rand(512, 1024, scale=0.05)
    q, e = quantize_mxfp8(w)
    assert torch.equal(Fn.dequant_mxfp8(q, e), dequantize_mxfp8(q, e))


@pytest.mark.parametrize("M", [1, 3])
def test_moe_decode(M):
    from petals_b200.models.block_oracle import GenericBlock
    from petals_b200.models.spec import BlockSpec

    torch.manual_seed(22)
    spec = BlockSpec(family="mixtral", hidden_size=1024, num_heads=8, num_kv_heads=2, head_dim=128, intermediate_size=1408, mlp="moe",
                     num_experts=8, top_k=2, norm_eps=1e-5)
    blk = GenericBlock(spec, dtype=torch.bfloat16, device=DEV, init_std=0.03)
    blk.ln2_w.data = (1 + 0.1 * torch.randn(1024, device=DEV)).to(torch.bfloat16)
    h = _rand(M, 1024)
    out = torch.empty_like(h)
    Fn.moe_decode(h, blk.ln2_w, blk.router, blk.we_gate, blk.we_up, blk.we_down, top_k=2, eps=1e-5, out=out)
    want = h + blk.mlp(Fn.norm_ref(h, blk.ln2_w, None, Fn.NORM_RMS, 1e-5).view(1, M, 1024)).view(M, 1024)
    _close(out, want, 3e-2, 3e-2, "moe decode")


@pytest.mark.parametrize("M,skew", [(9, False), (200, False), (777, False), (300, True)])
def test_moe_prefill_grouped_gemm(M, skew):
    """Any number of rows through the sync-free MoE path: device-built routing plan, gather, grouped tcgen05 GEMMs (ragged 128-row
    tiles, some experts empty when the router is skewed), weighted combine. Compared with the oracle block's expert loop."""
    from petals_b200.models.block_oracle import GenericBlock
    from petals_b200.models.spec import BlockSpec

    torch.manual_seed(23)
    spec = BlockSpec(family="mixtral", hidden_size=1024, num_heads=8, num_kv_heads=2, head_dim=128, intermediate_size=1408, mlp="moe",
                     num_experts=8, top_k=2, norm_eps=1e-5)
    blk = GenericBlock(spec, dtype=torch.bfloat16, device=DEV, init_std=0.03)
    blk.ln2_w.data = (1 + 0.1 * torch.randn(1024, device=DEV)).to(torch.bfloat16)
    if skew:  # experts 0..2 take (almost) everything: five groups are empty, three span several tiles
        blk.router.data[3:] = 0
        blk.router.data[:3] *= 4
    h = _rand(M, 1024)
    out = torch.empty_like(h)
    bufs = {}
    Fn.moe_prefill(h, blk.ln2_w, blk.router, blk.we_gate, blk.we_up, blk.we_down, top_k=2, eps=1e-5, out=out, bufs=bufs)
    want = h + blk.mlp(Fn.norm_ref(h, blk.ln2_w, None, Fn.NORM_RMS, 1e-5).view(1, M, 1024)).view(M, 1024)
    _close(out, want, 3e-2, 3e-2, "moe prefill")
    # the plan itself: positions are a permutation of the pairs, grouped by expert in ascending order
    pairs = M * 2
    pos, topi = bufs["moep_pos"][:pairs].long().cpu(), bufs["moep_topi"][:pairs].long().cpu()
    assert sorted(pos.tolist()) == list(range(pairs))
    by_pos = torch.empty(pairs, dtype=torch.long)
    by_pos[pos] = topi
    assert torch.equal(by_pos, by_pos.sort().values)
    again = torch.empty_like(h)  # buffers are reused (grow-only): a second, smaller call must not see stale state
    Fn.moe_prefill(h[: M // 2 + 1], blk.ln2_w, blk.router, blk.we_gate, blk.we_up, blk.we_down, top_k=2, eps=1e-5, out=again[: M // 2 + 1], bufs=bufs)
    _close(again[: M // 2 + 1], want[: M // 2 + 1], 3e-2, 3e-2, "moe prefill (reused buffers)")


# ---- sequence-parallel prefill primitives, in loopback: the "peers" are local buffers (same kernels, same flag protocol) ----
def test_gemm_reduce_scatter_routing_loopback():
    """Row-parallel GEMM whose epilogue routes row r only to owner r // rows_per_owner (at local row r % rows_per_owner) and
    publishes one completion flag per owner (last CTA)."""
    torch.manual_seed(11)
    M, N, K, R = 300, 512, 256, 4  # ragged: 75 rows per owner, tiles straddle owners
    mo = (M + R - 1) // R
    a, b = _rand(M, K), _rand(N, K, scale=K ** -0.5)
    owners = [torch.zeros(mo, N, device=DEV, dtype=torch.bfloat16) for _ in range(R)]
    flags = torch.zeros(R, device=DEV, dtype=torch.int64)
    ctr = torch.zeros(1, device=DEV, dtype=torch.int32)
    err = torch.zeros(1, device=DEV, dtype=torch.int32)
    Fn.gemm(a, b, store_local=False, push_out=[o.data_ptr() for o in owners], push_rows_per_owner=mo,
            push_done_flag=[flags[i:].data_ptr() for i in range(R)], done_counter=ctr.data_ptr(), error_flag=err.data_ptr())
    torch.cuda.synchronize()
    want = Fn.linear_ref(a, b)
    for r in range(R):
        rows = max(0, min(mo, M - r * mo))
        _close(owners[r][:rows], want[r * mo: r * mo + rows], 2e-2, 2e-2, f"owner {r}")
    assert flags.tolist() == [1] * R and int(ctr.item()) == 0 and int(err.item()) == 0


@pytest.mark.parametrize("kind", [Fn.NORM_RMS, Fn.NORM_LAYER, Fn.NORM_NONE])
def test_norm_reduce_gather_loopback(kind):
    """Owner-side reduce (residual + R partials) -> norm -> gather into R destination buffers, gated on an epoch flag."""
    torch.manual_seed(12)
    rows, H, R = 37, 2048, 3
    res = _rand(rows, H)
    parts = [_rand(rows, H) for _ in range(R)]
    w, b = _rand(H) * 0.1 + 1, _rand(H) * 0.1
    res_out = torch.zeros_like(res)
    dsts = [torch.zeros(rows, H, device=DEV, dtype=torch.bfloat16) for _ in range(R)]
    flags = torch.zeros(R + 1, device=DEV, dtype=torch.int64)
    flags[R] = 2 * R  # the wait flag already holds epoch(2) * per_epoch(R)
    epoch = torch.full((1,), 2, device=DEV, dtype=torch.int64)
    ctr = torch.zeros(1, device=DEV, dtype=torch.int32)
    err = torch.zeros(1, device=DEV, dtype=torch.int32)
    Fn.norm_reduce_gather(res, res_out, rows=rows, H=H, parts=[p.data_ptr() for p in parts], norm_weight=None if kind == Fn.NORM_NONE else w,
                          norm_bias=b if kind == Fn.NORM_LAYER else None, norm_kind=kind, eps=1e-5,
                          gather_out=[d.data_ptr() for d in dsts], gather_flag=[flags[i:].data_ptr() for i in range(R)],
                          wait_flag=flags[R:].data_ptr(), wait_per_epoch=R, epoch=epoch.data_ptr(), done_counter=ctr.data_ptr(),
                          error_flag=err.data_ptr())
    torch.cuda.synchronize()
    xs = (res.float() + sum(p.float() for p in parts)).to(torch.bfloat16)
    _close(res_out, xs, 1e-2, 1e-2, "residual")
    want = xs if kind == Fn.NORM_NONE else Fn.norm_ref(xs, w, b if kind == Fn.NORM_LAYER else None, kind=kind, eps=1e-5)
    for d in dsts:
        _close(d, want, 2e-2, 2e-2, "gathered rows")
    assert flags[:R].tolist() == [1] * R and int(err.item()) == 0 and int(ctr.item()) == 0


@pytest.mark.parametrize("D,Hq,Hkv", [(128, 8, 1), (128, 4, 2), (64, 4, 2), (64, 3, 3)])
@pytest.mark.parametrize("chunks", [[256, 200], [130, 300, 77]])
def test_attention_tcgen05_prefill(D, Hq, Hkv, chunks):
    """The tcgen05/TMEM prefill kernel (impl=2) against the fp32 oracle and the mma.sync kernel (impl=1): chunked prefill over a
    shuffled paged cache, ragged last tiles, GQA packing with group sizes 1/2/3/8."""
    torch.manual_seed(21)
    B, L_max = 2, sum(chunks)
    k_pool, v_pool, table = _paged_setup(B, L_max, Hkv, D, seed=3)
    cos, sin = Fn.rope_tables(D, 1024, theta=10000.0, device=DEV)
    pos = torch.zeros(1, dtype=torch.int32, device=DEV)
    k_all = torch.zeros(B, 0, Hkv, D, device=DEV, dtype=torch.bfloat16)
    v_all = torch.zeros_like(k_all)
    scale, p0 = D ** -0.5, 0
    for T in chunks:
        qkv = _rand(B, T, (Hq + 2 * Hkv) * D)
        q_out = torch.empty(B, T, Hq, D, device=DEV, dtype=torch.bfloat16)
        Fn.rope_kv_append(qkv, q_out, k_pool, v_pool, table, pos.data_ptr(), cos, sin, B=B, T=T, Hq=Hq, Hkv=Hkv, D=D)
        q, k, v = qkv.view(B, T, Hq + 2 * Hkv, D).split([Hq, Hkv, Hkv], dim=2)
        q_ref = Fn.rope_ref(q, cos[p0:p0 + T], sin[p0:p0 + T])
        k_all, v_all = torch.cat([k_all, Fn.rope_ref(k, cos[p0:p0 + T], sin[p0:p0 + T])], 1), torch.cat([v_all, v], 1)
        want = Fn.attention_ref(q_ref, k_all, v_all, pos0=p0, scale=scale)
        outs = {}
        for impl in (1, 2):
            out = torch.full((B, T, Hq, D), float("nan"), device=DEV, dtype=torch.bfloat16)
            Fn.paged_attention(q_out, k_pool, v_pool, table, pos.data_ptr(), out, B=B, T=T, Hq=Hq, Hkv=Hkv, D=D, scale=scale, impl=impl)
            outs[impl] = out
            _close(out, want, 2e-2, 2e-2, f"impl={impl} T={T} pos0={p0}")
        _close(outs[2], outs[1], 2e-2, 2e-2, "tcgen05 vs mma.sync")
        pos += T
        p0 += T


def test_attention_tcgen05_alibi_window():
    torch.manual_seed(22)
    B, T, Hq, Hkv, D = 1, 400, 4, 2, 64
    k_pool, v_pool, table = _paged_setup(B, T, Hkv, D)
    pos = torch.zeros(1, dtype=torch.int32, device=DEV)
    qkv = _rand(B, T, (Hq + 2 * Hkv) * D)
    q_out = torch.empty(B, T, Hq, D, device=DEV, dtype=torch.bfloat16)
    Fn.rope_kv_append(qkv, q_out, k_pool, v_pool, table, pos.data_ptr(), None, None, B=B, T=T, Hq=Hq, Hkv=Hkv, D=D)
    q, k, v = qkv.view(B, T, Hq + 2 * Hkv, D).split([Hq, Hkv, Hkv], dim=2)
    slopes = torch.tensor([2 ** (-8 * (i + 1) / Hq) for i in range(Hq)], device=DEV)
    out = torch.empty_like(q_out)
    Fn.paged_attention(q_out, k_pool, v_pool, table, pos.data_ptr(), out, B=B, T=T, Hq=Hq, Hkv=Hkv, D=D, scale=D ** -0.5, alibi_slopes=slopes, impl=2)
    _close(out, Fn.attention_ref(q, k, v, pos0=0, scale=D ** -0.5, alibi_slopes=slopes), 2e-2, 2e-2, "tcgen05 alibi")
    Fn.paged_attention(q_out, k_pool, v_pool, table, pos.data_ptr(), out, B=B, T=T, Hq=Hq, Hkv=Hkv, D=D, scale=D ** -0.5, window=150, impl=2)
    _close(out, Fn.attention_ref(q, k, v, pos0=0, scale=D ** -0.5, window=150), 2e-2, 2e-2, "tcgen05 window")


@pytest.mark.parametrize("D,Hq,Hkv", [(128, 8, 2), (64, 4, 4)])
@pytest.mark.parametrize("B,T", [(1, 1), (2, 3), (1, 8)])
def test_linear_decode_fused_rope_append(D, Hq, Hkv, B, T):
    """QKV projection with the RoPE + paged-KV-append epilogue == (projection -> rope_kv_append kernel), bit for bit."""
    torch.manual_seed(31)
    K, M = 1024, B * T
    N = (Hq + 2 * Hkv) * D
    x, w, g = _rand(M, K), _rand(N, K, scale=K ** -0.5), _rand(K) * 0.1 + 1
    cos, sin = Fn.rope_tables(D, 512, theta=10000.0, device=DEV)
    pos = torch.full((1,), 70, dtype=torch.int32, device=DEV)  # mid-page, second page of each sequence
    kp1, vp1, table = _paged_setup(B, 200, Hkv, D, seed=5)
    kp2, vp2 = kp1.clone(), vp1.clone()
    # unfused reference pipeline
    qkv = Fn.linear_decode(x, w, norm_weight=g, norm_kind=Fn.NORM_RMS, eps=1e-5)
    q1 = torch.empty(M, Hq * D, device=DEV, dtype=torch.bfloat16)
    Fn.rope_kv_append(qkv, q1, kp1, vp1, table, pos.data_ptr(), cos, sin, B=B, T=T, Hq=Hq, Hkv=Hkv, D=D)
    # fused
    q2 = torch.full_like(q1, float("nan"))
    err = torch.zeros(1, dtype=torch.int32, device=DEV)
    Fn.linear_decode(x, w, norm_weight=g, norm_kind=Fn.NORM_RMS, eps=1e-5, error_flag=err.data_ptr(),
                     rope=dict(q_out=q2, k_pool=kp2, v_pool=vp2, block_table=table, pos_ptr=pos.data_ptr(), cos=cos, sin=sin, T=T, Hq=Hq, Hkv=Hkv, D=D))
    torch.cuda.synchronize()
    assert int(err.item()) == 0
    _close(q2, q1, 1e-2, 1e-2, "q")
    _close(kp2, kp1, 1e-2, 1e-2, "k pages")
    _close(vp2, vp1, 1e-2, 1e-2, "v pages")
    assert (kp2 != 0).any() and (vp2 != 0).any()


def test_linear_decode_fp8_activation_outliers():
    """The fp16 staging of x is scaled per token by a power of two: huge and tiny rows (no norm, e.g. the down projection's
    input) must neither overflow the packed-half accumulation nor lose the small row."""
    from petals_b200.ops.quant import dequantize_mxfp8, quantize_mxfp8

    torch.manual_seed(23)
    K, N, M = 2048, 1024, 3
    x = _rand(M, K)
    x[0] *= 300.0          # massive activations
    x[0, 7] = 20000.0      # one outlier
    x[1] *= 1e-3           # tiny row
    w = _rand(N, K, scale=K ** -0.5)
    q, e = quantize_mxfp8(w)
    wd = dequantize_mxfp8(q, e)
    got = Fn.linear_decode_fp8(x, q, e)
    want = Fn.linear_ref(x, wd)
    assert torch.isfinite(got.float()).all()
    for m in range(M):
        err = (got[m].float() - want[m].float()).abs().max() / want[m].float().abs().max()
        assert err < 2e-2, f"row {m}: {err}"


@pytest.mark.parametrize("M", [1, 4])
def test_linear_decode_split_k_small_n(M):
    """Projections with few output columns (tensor-parallel QKV shards) run split-K inside the CTA: 4 warps share a row pair."""
    torch.manual_seed(61)
    # plain + norm, and SwiGLU, at shapes that take the split-K path (N/2 < 12 * SMs, K >= 2048)
    K = 8192
    x, g = _rand(M, K), _rand(K) * 0.1 + 1
    w = _rand(1280, K, scale=K ** -0.5)
    got = Fn.linear_decode(x, w, norm_weight=g, norm_kind=Fn.NORM_RMS, eps=1e-5)
    _close(got, Fn.linear_ref(x, w, norm_weight=g, norm_kind=Fn.NORM_RMS, eps=1e-5), 3e-2, 2e-2, "split-k plain")
    wg, wu = _rand(896, K, scale=K ** -0.5), _rand(896, K, scale=K ** -0.5)
    got = Fn.linear_decode(x, wg, w2=wu, act=Fn.ACT_SWIGLU, norm_weight=g, norm_kind=Fn.NORM_RMS, eps=1e-5)
    _close(got, Fn.linear_ref(x, wg, w2=wu, act=Fn.ACT_SWIGLU, norm_weight=g, norm_kind=Fn.NORM_RMS, eps=1e-5), 2e-2, 3e-2, "split-k swiglu")
    # fused RoPE + KV append epilogue on a one-kv-head shard (8 q heads + 1 k + 1 v, d=128): equals projection -> rope kernel
    if M == 1:
        D, Hq, Hkv = 128, 8, 1
        wq = _rand((Hq + 2 * Hkv) * D, K, scale=K ** -0.5)
        cos, sin = Fn.rope_tables(D, 512, theta=10000.0, device=DEV)
        pos = torch.full((1,), 5, dtype=torch.int32, device=DEV)
        kp1, vp1, table = _paged_setup(1, 64, Hkv, D, seed=9)
        kp2, vp2 = kp1.clone(), vp1.clone()
        qkv = Fn.linear_decode(x, wq, norm_weight=g, norm_kind=Fn.NORM_RMS, eps=1e-5)
        q1 = torch.empty(1, Hq * D, device=DEV, dtype=torch.bfloat16)
        Fn.rope_kv_append(qkv, q1, kp1, vp1, table, pos.data_ptr(), cos, sin, B=1, T=1, Hq=Hq, Hkv=Hkv, D=D)
        q2 = torch.empty_like(q1)
        Fn.linear_decode(x, wq, norm_weight=g, norm_kind=Fn.NORM_RMS, eps=1e-5,
                         rope=dict(q_out=q2, k_pool=kp2, v_pool=vp2, block_table=table, pos_ptr=pos.data_ptr(), cos=cos, sin=sin, T=1, Hq=Hq, Hkv=Hkv, D=D))
        _close(q2, q1, 2e-2, 2e-2, "split-k rope q")
        _close(kp2, kp1, 2e-2, 2e-2, "split-k rope k")
        _close(vp2, vp1, 2e-2, 2e-2, "split-k v")


@pytest.mark.parametrize("M", [2, 4, 8])
def test_linear_decode_skinny_tensor_core_path(M):
    """2..8 rows on mma.sync (tokens as the N dimension, k-permuted fragments, K-sliced row blocks reduced through global scratch)
    against the fp32 oracle and the FMA kernel; the scratch / counters must be left zero by every launch."""
    torch.manual_seed(71)
    prev = (Fn._SKINNY["on"], Fn._SKINNY["force"])
    try:
        Fn.set_skinny_gemm(True)
        # plain + residual
        x, w, res = _rand(M, 4096), _rand(4096, 4096, scale=4096 ** -0.5), _rand(M, 4096)
        got = Fn.linear_decode(x, w, residual=res)
        _close(got, Fn.linear_ref(x, w, residual=res), 3e-2, 2e-2, "skinny plain+residual")
        # RMSNorm + SwiGLU
        x, g = _rand(M, 1024), _rand(1024) * 0.1 + 1
        wg, wu = _rand(2816, 1024, scale=1024 ** -0.5), _rand(2816, 1024, scale=1024 ** -0.5)
        got = Fn.linear_decode(x, wg, w2=wu, act=Fn.ACT_SWIGLU, norm_weight=g, norm_kind=Fn.NORM_RMS, eps=1e-5)
        _close(got, Fn.linear_ref(x, wg, w2=wu, act=Fn.ACT_SWIGLU, norm_weight=g, norm_kind=Fn.NORM_RMS, eps=1e-5), 2e-2, 3e-2, "skinny swiglu")
        # LayerNorm + bias + GELU
        x, g, b = _rand(M, 2048), _rand(2048) * 0.1 + 1, _rand(2048) * 0.1
        w, bias = _rand(1024, 2048, scale=2048 ** -0.5), _rand(1024) * 0.1
        got = Fn.linear_decode(x, w, bias=bias, act=Fn.ACT_GELU_TANH, norm_weight=g, norm_bias=b, norm_kind=Fn.NORM_LAYER, eps=1e-5)
        _close(got, Fn.linear_ref(x, w, bias=bias, act=Fn.ACT_GELU_TANH, norm_weight=g, norm_bias=b, norm_kind=Fn.NORM_LAYER, eps=1e-5), 3e-2, 3e-2, "skinny ln+gelu")
        # very wide K (down projection): x read from global memory, no staging
        x, w, res = _rand(M, 28672, scale=0.3), _rand(1024, 28672, scale=28672 ** -0.5), _rand(M, 1024)
        got = Fn.linear_decode(x, w, residual=res)
        _close(got, Fn.linear_ref(x, w, residual=res), 3e-2, 2e-2, "skinny wide-K")
        for scratch, counters, _cap in Fn._SKINNY["keep"]:
            assert float(scratch.abs().sum().item()) == 0.0 and int(counters.abs().sum().item()) == 0
    finally:
        Fn._SKINNY["on"], Fn._SKINNY["force"] = prev


# ---- backward kernels (csrc/attention_bwd.cu, csrc/train_kernels.cu) against fp32 PyTorch autograd ------------------------------------
def _paged_from_dense(k, v):
    """[B, T, Hkv, D] -> pools [B * pages, Hkv, 64, D] with block table arange."""
    B, T, Hkv, D = k.shape
    pages = (T + 63) // 64
    kp = torch.zeros(B * pages, Hkv, 64, D, dtype=k.dtype, device=k.device)
    vp = torch.zeros_like(kp)
    for b in range(B):
        for p in range(pages):
            n = min(64, T - p * 64)
            kp[b * pages + p, :, :n] = k[b, p * 64: p * 64 + n].transpose(0, 1)
            vp[b * pages + p, :, :n] = v[b, p * 64: p * 64 + n].transpose(0, 1)
    table = torch.arange(B * pages, dtype=torch.int32, device=k.device).view(B, pages).contiguous()
    return kp, vp, table


@pytest.mark.parametrize("B,T,Hq,Hkv,D", [(2, 40, 8, 2, 128), (1, 200, 4, 4, 64), (3, 130, 8, 1, 128), (1, 64, 6, 2, 128)])
def test_attention_backward_matches_autograd(B, T, Hq, Hkv, D):
    torch.manual_seed(5)
    q = (torch.randn(B, T, Hq, D, device=DEV) * 0.8).to(torch.bfloat16)
    k = (torch.randn(B, T, Hkv, D, device=DEV) * 0.8).to(torch.bfloat16)
    v = (torch.randn(B, T, Hkv, D, device=DEV) * 0.8).to(torch.bfloat16)
    d_out = (torch.randn(B, T, Hq, D, device=DEV) * 0.3).to(torch.bfloat16)
    scale = D ** -0.5
    # fp32 reference
    qf, kf, vf = (t.float().clone().requires_grad_(True) for t in (q, k, v))
    G = Hq // Hkv
    kk = kf.repeat_interleave(G, dim=2)
    vv = vf.repeat_interleave(G, dim=2)
    s = torch.einsum("bthd,bshd->bhts", qf, kk) * scale
    mask = torch.ones(T, T, dtype=torch.bool, device=DEV).tril()
    s = s.masked_fill(~mask, float("-inf"))
    o_ref = torch.einsum("bhts,bshd->bthd", s.softmax(-1), vv)
    gq, gk, gv = torch.autograd.grad(o_ref, [qf, kf, vf], d_out.float())
    # kernels: forward (saves lse), then backward
    kp, vp, table = _paged_from_dense(k, v)
    M = B * T
    out = torch.empty(M, Hq * D, dtype=torch.bfloat16, device=DEV)
    lse = torch.empty(M * Hq, dtype=torch.float32, device=DEV)
    Fn.paged_attention(q.view(M, Hq * D), kp, vp, table, None, out, B=B, T=T, Hq=Hq, Hkv=Hkv, D=D, scale=scale, lse_out=lse)
    _close(out.view(B, T, Hq, D), o_ref.detach(), 2e-2, 2e-2, "attention forward (lse path)")
    lse_ref = (torch.logsumexp(s.detach(), dim=-1) * 1.4426950408889634).permute(0, 2, 1).reshape(-1)  # [B, T, Hq], log2 domain
    assert (lse - lse_ref).abs().max().item() < 2e-2
    dq, dk, dv = Fn.attention_bwd(q.view(M, Hq * D), kp, vp, table, out, d_out.view(M, Hq * D).contiguous(), lse, B=B, T=T, Hq=Hq, Hkv=Hkv, D=D, scale=scale)
    torch.cuda.synchronize()
    for name, got, ref in (("dq", dq.view(B, T, Hq, D), gq), ("dk", dk.view(B, T, Hkv, D), gk), ("dv", dv.view(B, T, Hkv, D), gv)):
        rel = ((got.float() - ref).norm() / ref.norm()).item()
        assert rel < 2e-2, (name, rel)
        _close(got, ref, 2e-2 * ref.abs().max().item(), 3e-2, name)


@pytest.mark.parametrize("rows,H", [(37, 1024), (5, 4096), (3, 8192)])
def test_rmsnorm_backward_matches_autograd(rows, H):
    torch.manual_seed(6)
    x = torch.randn(rows, H, device=DEV).to(torch.bfloat16)
    w = (1 + 0.1 * torch.randn(H, device=DEV)).to(torch.bfloat16)
    dy = torch.randn(rows, H, device=DEV).to(torch.bfloat16)
    res = torch.randn(rows, H, device=DEV).to(torch.bfloat16)
    xf = x.float().requires_grad_(True)
    y = xf * torch.rsqrt(xf.pow(2).mean(-1, keepdim=True) + 1e-5) * w.float()
    (g,) = torch.autograd.grad(y, xf, dy.float())
    got = Fn.rmsnorm_bwd(dy, x, w, 1e-5, d_res=res)
    _close(got, g + res.float(), 2e-2, 3e-2, "rmsnorm_bwd")


def test_swiglu_and_rope_backward_match_autograd():
    torch.manual_seed(7)
    g = torch.randn(33, 2816, device=DEV).to(torch.bfloat16)
    u = torch.randn(33, 2816, device=DEV).to(torch.bfloat16)
    d = torch.randn(33, 2816, device=DEV).to(torch.bfloat16)
    gf, uf = g.float().requires_grad_(True), u.float().requires_grad_(True)
    rg, ru = torch.autograd.grad(torch.nn.functional.silu(gf) * uf, [gf, uf], d.float())
    g2, u2 = g.clone(), u.clone()
    Fn.swiglu_bwd_(d, g2, u2)
    _close(g2, rg, 2e-2, 3e-2, "d gate")
    _close(u2, ru, 2e-2, 3e-2, "d up")
    # RoPE backward + merge: <R x, g> == <x, R^T g>
    B, T, Hq, Hkv, D = 2, 9, 4, 2, 128
    M = B * T
    cos, sin = Fn.rope_tables(D, 64, 10000.0, None, device=DEV)
    dq = torch.randn(M, Hq * D, device=DEV).to(torch.bfloat16)
    dk = torch.randn(M, Hkv * D, device=DEV).to(torch.bfloat16)
    dv = torch.randn(M, Hkv * D, device=DEV).to(torch.bfloat16)
    merged = Fn.qkv_grad_merge(dq, dk, dv, cos, sin, T=T, Hq=Hq, Hkv=Hkv, D=D).float().view(B, T, Hq + 2 * Hkv, D)
    xq = torch.randn(B, T, Hq, D, device=DEV, requires_grad=True)
    pos = torch.arange(T, device=DEV)
    c, s_ = torch.cat([cos[pos], cos[pos]], -1)[None, :, None, :], torch.cat([sin[pos], sin[pos]], -1)[None, :, None, :]
    rot = lambda x: x * c + torch.cat([-x[..., D // 2:], x[..., : D // 2]], -1) * s_
    (ref_q,) = torch.autograd.grad(rot(xq), xq, dq.float().view(B, T, Hq, D))
    _close(merged[:, :, :Hq], ref_q, 2e-2, 3e-2, "rope^T dq")
    _close(merged[:, :, Hq + Hkv:], dv.float().view(B, T, Hkv, D), 1e-2, 1e-2, "dv passthrough")


def test_ll_collectives_loopback():
    """csrc/ll_collectives.cu in loop-back (the "peers" are local buffers): ll_push writes {2 x bf16, tag} units, ll_reduce polls them and
    adds them to the residual in source order with one rounding — the stand-alone halves of the all-reduce around a sparse-MoE block."""
    torch.manual_seed(31)
    M, H, R = 3, 1024, 4
    epoch = torch.full((1,), 7, dtype=torch.int64, device=DEV)
    x = _rand(M, H)
    parts = [_rand(M, H) for _ in range(R)]
    slots = [torch.zeros(M * H // 2, 2, dtype=torch.int32, device=DEV) for _ in range(R)]
    for r in range(R):
        Fn.ll_push(parts[r], [slots[r].data_ptr()], (5, 2), epoch.data_ptr())
    tags = torch.stack([s[:, 1] for s in slots])
    assert (tags == 7 * 5 + 2).all()
    out = torch.empty_like(x)
    err = torch.zeros(1, dtype=torch.int32, device=DEV)
    Fn.ll_reduce(x, [s.data_ptr() for s in slots], (5, 2), epoch.data_ptr(), out, err.data_ptr())
    want = (x.float() + sum(p.float() for p in parts)).to(torch.bfloat16)
    torch.cuda.synchronize()
    assert int(err.item()) == 0
    assert (out.float() - want.float()).abs().max().item() <= 2 ** -6 * want.float().abs().max().item()  # summation order may differ from torch's by one rounding
    # one push to several destinations at once
    more = [torch.zeros(M * H // 2, 2, dtype=torch.int32, device=DEV) for _ in range(3)]
    Fn.ll_push(parts[0], [m.data_ptr() for m in more], (5, 3), epoch.data_ptr())
    assert all(torch.equal(m, more[0]) for m in more) and (more[0][:, 1] == 7 * 5 + 3).all()
    assert torch.equal(more[0][:, 0].contiguous().view(torch.bfloat16).view(M, H), parts[0])
