// petals_b200 — C ABI of the native library (loaded from Python through ctypes).
// Every launcher takes raw device pointers plus a cudaStream_t (as void*), returns PB_OK or an error
// code, and never synchronises: the Python layer captures whole pipeline stages into CUDA graphs.
#pragma once
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { PB_OK = 0, PB_ERR_SHAPE = 1, PB_ERR_CUDA = 2, PB_ERR_UNSUPPORTED = 3, PB_ERR_DRIVER = 4 };

#define PB_MAX_PEERS 8

// ---- decode-shape linear (linear_decode.cu) ------------------------------------------------------
typedef struct {
  const void* x; const void* w; const void* w2; const void* bias; const void* bias2;
  const void* residual; void* out; const void* norm_w; const void* norm_b; void* x_out;
  float eps; int norm_kind; int act; int M, N, K;
  int n_parts; const void* parts[PB_MAX_PEERS];
  const void* wait_flag; uint64_t wait_per_epoch; const void* epoch;
  int n_push; void* push_out[PB_MAX_PEERS]; void* push_flag[PB_MAX_PEERS];
  void* error_flag;
  int num_sms; int fixed_grid; int* out_grid;
  void* done_counter;
  // fused RoPE + paged KV append epilogue for the QKV projection (rope_q_out != NULL enables it; see linear_decode.cu)
  void* rope_q_out; void* rope_k_pool; void* rope_v_pool; const void* rope_block_table; const void* rope_pos_ptr;
  const void* rope_cos; const void* rope_sin;
  int rope_T, rope_Hq, rope_Hkv, rope_D, rope_max_pages, rope_max_pos;
  // LL one-shot all-reduce (8-byte {payload, tag} units; see linear_decode.cu): tag = (uint32)*epoch * ll_tag_mul + ll_tag_add
  int n_ll_parts; const void* ll_parts[PB_MAX_PEERS];
  int n_ll_push; void* ll_push[PB_MAX_PEERS];
  uint32_t ll_tag_mul, ll_tag_add;
  int rope_num_pages;           // pages in rope_k_pool / rope_v_pool: a table entry outside [0, num_pages) raises error flag 2
} PbLinearDecodeArgs;
int pb_linear_decode(const PbLinearDecodeArgs* a, void* stream);
// 2..8 rows on the tensor cores (mma.sync m16n8k16, tokens as the N dimension); scratch: fp32 [2*N*8] zeros, counters: u32 [N/16] zeros
int pb_linear_decode_mma(const PbLinearDecodeArgs* a, void* scratch, void* counters, void* stream);

// ---- decode-shape linear over block-scaled FP8 weights (linear_decode_fp8.cu) ---------------------------
typedef struct {
  const void* x; const void* w; const void* w_scale; const void* w2; const void* w2_scale;
  const void* bias; const void* bias2; const void* residual; void* out; const void* norm_w; const void* norm_b;
  float eps; int norm_kind; int act; int M, N, K; int num_sms;
} PbLinearFp8Args;
int pb_linear_decode_fp8(const PbLinearFp8Args* a, void* stream);
int pb_dequant_mxfp8(const void* q, const void* e, void* out_bf16, long n_elems, void* stream);

// ---- tcgen05 GEMM (gemm_tcgen05.cu) -----------------------------------------------------------------
// D[M,N] = epilogue(A[M,K] * B^T) with A K-major [M,K]; B either K-major [N,K] (nn.Linear weight,
// forward) or MN-major [K,N] (the same weight used transposed: dgrad). bf16 in, fp32 accumulate.
typedef struct {
  const void* a; const void* b; const void* b2;  // b2: second weight for fused SwiGLU (gate=b, up=b2)
  const void* bias; const void* bias2; const void* residual; void* out;
  int M, N, K;
  int lda, ldb, ldo, ldres;   // leading dimensions in elements (0 = packed)
  int b_mn_major;             // 0: B is [N,K]; 1: B is [K,N]
  int act;                    // 0 none, 1 SwiGLU (needs b2; out has N columns), 2 GELU tanh, 3 GELU erf
  int out_fp32;               // store fp32 instead of bf16
  int accumulate;             // out += result (fp32 out only)
  // fused stage hop / TP push: also store tiles to peer buffers and bump their flags per tile
  int n_push; void* push_out[PB_MAX_PEERS]; void* push_flag[PB_MAX_PEERS];
  // consumer side: wait for flag >= *epoch * wait_per_epoch before loading A
  const void* wait_flag; uint64_t wait_per_epoch; const void* epoch; void* error_flag;
  int num_sms; int block_n;   // 0 = auto
  void* push_done_flag[PB_MAX_PEERS]; void* done_counter;  // once-per-launch completion flag (last CTA)
  int push_rows_per_owner;    // > 0: reduce-scatter routing of output rows to their owner rank (see gemm_tcgen05.cu)
  // grouped (ragged-M) mode for sparse MoE: `grp` = device table from pb_moe_plan {n_mtiles, expert[cap], row0[cap], rows[cap]};
  // B holds grp_experts matrices of N rows each, stacked along N; M is the total number of (token, expert) rows
  const void* grp; int grp_cap; int grp_experts;
} PbGemmArgs;
int pb_gemm_bf16(const PbGemmArgs* a, void* stream);

// ---- norms / elementwise (elementwise.cu) ---------------------------------------------------------
// out = norm(x [+ residual]); if sum_out != null also stores (x + residual).
int pb_norm(const void* x, const void* residual, const void* weight, const void* bias, void* out,
            void* sum_out, int rows, int cols, float eps, int kind /*1 rms, 2 layernorm*/, void* stream);
int pb_swiglu(const void* gate, const void* up, void* out, long n, void* stream);
int pb_add(const void* a, const void* b, void* out, long n, void* stream);
int pb_embedding(const void* table, const void* ids /*int64*/, void* out, int n_tokens, int hidden,
                 void* stream);
// argmax over vocab of logits [rows, vocab] (bf16 or fp32) -> int64 ids
int pb_argmax(const void* logits, int is_fp32, void* out_ids, int rows, int vocab, void* stream);
int pb_add_prompts(void* hidden /*[B,T,H]*/, const void* prompts /*[Bp,P,H]*/, int B, int T, int H,
                   int Bp, int P, const void* pos_ptr, void* stream);
int pb_gelu(const void* x, void* out, long n, int erf_form, void* stream);
int pb_bump_epoch(void* epoch, void* stream);
int pb_advance_pos(void* pos, int delta, void* stream);

// ---- one-token decode of a span of Llama-style blocks as one persistent data-flow kernel (decode_span.cu) -------------
typedef struct {
  const void* layers;      // device array of n_layers x 9 pointers: wqkv, wo, wgate, wup, wdown, ln1, ln2, k_pool, v_pool
  int n_layers;
  int H, Hq, Hkv, D, I;    // this rank's heads / FFN columns, full hidden size
  float eps, attn_scale;
  const void* x_in; void* x_out;                 // [H] bf16
  const void* in_flag; uint64_t in_per_epoch;    // optional flag wait before x_in is read
  const void* block_table; int max_pages, num_pages; const void* pos_ptr;
  const void* cos; const void* sin; int max_pos;
  void* qkv_ll; void* attp_ll; void* attn_ll; void* x_ll; void* act_ll; int max_chunks;   // local tagged buffers
  int R, rank;
  void* oproj_push[PB_MAX_PEERS]; void* mlp_push[PB_MAX_PEERS];   // slot [rank] of every rank's all-reduce buffers
  const void* oproj_in; const void* mlp_in;                       // local [R][H/2] units
  const void* epoch; void* error_flag;
  int num_sms;
  int prepare_only;        // 1: validate the shapes and set the kernel's shared-memory attribute, launch nothing
  void* timing;            // optional uint64 [n_layers][24]: %globaltimer stamps of CTA 0 at every phase boundary (diagnostics)
  // NVSwitch multicast (all NULL / 0 without a multicast mapping of the heap):
  void* oproj_mc_push; void* mlp_mc_push;            // multicast address of slot [rank]: one multimem.st instead of R peer stores
  const void* oproj_mc_sum; const void* mlp_mc_sum;  // multicast address of slot [0]: owners multimem.ld_reduce the R partials (nvls_reduce)
  int nvls_reduce;
} PbDecodeSpanArgs;
int pb_decode_span(const PbDecodeSpanArgs* a, void* stream);
int pb_decode_span_smem(const PbDecodeSpanArgs* a, int* n_stages, int* vin_elems);

// ---- RoPE + paged KV append (rope_kv.cu) ------------------------------------------------------------
typedef struct {
  const void* qkv;        // [B*T, (Hq + 2*Hkv) * D]
  void* q_out;            // [B*T, Hq * D]
  void* k_pool; void* v_pool;   // this layer's pools: [num_pages, Hkv, PAGE, D]
  const void* block_table;      // int32 [B, max_pages]
  const void* pos_ptr;          // int32 device scalar: tokens already in the cache
  const void* cos; const void* sin;  // fp32 [max_pos, D/2] or null (no rotary: BLOOM/ALiBi)
  const void* qkv_bias;         // optional [ (Hq+2Hkv)*D ]
  int B, T, Hq, Hkv, D, page, max_pages, max_pos;
  int interleaved_qkv;          // 1: Falcon/BLOOM fused layout [Hkv, G+2, D] per token
  void* error_flag;
  int num_pages;                // pages in k_pool / v_pool: a table entry outside [0, num_pages) raises error flag 2
} PbRopeKvArgs;
int pb_rope_kv(const PbRopeKvArgs* a, void* stream);

// ---- owner-side reduce-scatter tail + norm + all-gather for sequence-parallel TP prefill (seq_parallel.cu) ----
typedef struct {
  const void* x_res_in; void* x_res_out;            // [rows, H] bf16 owned residual rows (in may be NULL = zero; out may be NULL)
  int n_parts; const void* parts[PB_MAX_PEERS];     // partial rows written by the peers' GEMM epilogues
  const void* norm_w; const void* norm_b; float eps; int norm_kind;   // 0: gather the raw sum
  int n_gather; void* gather_out[PB_MAX_PEERS]; void* gather_flag[PB_MAX_PEERS];
  const void* wait_flag; uint64_t wait_per_epoch; const void* epoch;
  void* done_counter; void* error_flag;
  int rows, H, num_sms;
} PbNormReduceGatherArgs;
int pb_norm_reduce_gather(const PbNormReduceGatherArgs* a, void* stream);

// ---- flash attention over the paged KV cache (attention.cu) ---------------------------------------
typedef struct {
  const void* q;          // [B*T, Hq*D]
  const void* k_pool; const void* v_pool;
  const void* block_table; const void* pos_ptr;
  void* out;              // [B*T, Hq*D]
  void* partial_o;        // fp32 [splits, B*T*Hq, D] (splits > 1)
  void* partial_lse;      // fp32 [splits, B*T*Hq]
  const void* alibi_slopes;  // fp32 [Hq] or null
  float scale;
  int B, T, Hq, Hkv, D, page, max_pages;
  int window;             // sliding window (0 = none)
  int splits;             // >= 1
  int pos_static;         // used when pos_ptr == null
  int num_pages;          // pages in k_pool / v_pool (bounds the TMA tensor map of the tcgen05 path)
  int impl;               // 0 auto, 1 mma.sync kernel, 2 tcgen05 kernel
  void* split_counter;    // int32 [m_tiles * B * Hkv], zeroed once: fuses the split-KV combine into the attention kernel
  void* lse_out;          // optional fp32 [B*T*Hq]: log2-domain log-sum-exp per query row (training forward; mma.sync kernel, splits == 1)
} PbAttnArgs;
int pb_attention(const PbAttnArgs* a, void* stream);

// ---- backward of the causal attention (attention_bwd.cu): activations only, frozen weights -------------------------------
typedef struct {
  const void* q;            // [B*T, Hq*D] rotated queries (what the forward consumed)
  const void* k_pool; const void* v_pool; const void* block_table;   // the keys/values the forward attended to (paged, PAGE = 64)
  const void* out;          // [B*T, Hq*D] forward output
  const void* d_out;        // [B*T, Hq*D] gradient w.r.t. the output
  const void* lse;          // fp32 [B*T*Hq] from the forward (log2 domain)
  void* delta;              // fp32 [B*T*Hq] scratch: rowsum(d_out * out)
  void* dq;                 // [B*T, Hq*D]
  void* dk; void* dv;       // [B*T, Hkv*D] token-major dense gradients of the (rotated) keys / values
  float scale;
  int B, T, Hq, Hkv, D, max_pages, num_pages;
} PbAttnBwdArgs;
int pb_attention_bwd(const PbAttnBwdArgs* a, void* stream);

// ---- element-wise / row-wise pieces of the block backward (train_kernels.cu) ---------------------------------------------
// dx = [d_res +] rmsnorm_backward(dy, x, w): rows x H, fp32 math. d_res may alias dx_out.
int pb_rmsnorm_bwd(const void* dy, const void* x, const void* w, const void* d_res, void* dx_out, int rows, int H, float eps, void* stream);
// SwiGLU backward in place: g <- d_act * u * silu'(g), u <- d_act * silu(g)  (g, u: the bf16 projections saved by the forward)
int pb_swiglu_bwd(const void* d_act, void* g, void* u, long n, void* stream);
// dqkv[M, (Hq+2Hkv) D] = [R^T dq | R^T dk | dv]: the gradients of the rotated queries / keys are rotated back (transposed RoPE,
// position t = row % T) and written next to dv in the fused projection's column layout, ready for the dgrad GEMM.
int pb_qkv_grad_merge(const void* dq, const void* dk, const void* dv, const void* cos, const void* sin, void* dqkv, int M, int T, int Hq, int Hkv,
                      int D, int max_pos, void* stream);

// ---- sparse MoE decode (moe.cu) ------------------------------------------------------------------------------
int pb_moe_router(const void* h, const void* norm_w, const void* router, void* xn_out, void* topi, void* topw, int M, int H, int E,
                  int topk, float eps, void* stream);
int pb_moe_gemv(const void* x, const void* w_all, const void* w2_all, const void* topi, void* out, int pairs, int N, int K,
                long expert_stride, int x_row_div, int num_sms, void* stream);
int pb_moe_combine(const void* y, const void* topw, const void* residual, void* out, int M, int H, int topk, void* stream);

// prefill-sized MoE without host synchronisation: routing plan (destination rows + grouped-GEMM tile table), gather, combine
int pb_moe_plan(const void* topi, int pairs, int E, void* pos, void* table, int cap, void* stream);
int pb_moe_gather(const void* x, const void* pos, void* out, int pairs, int H, int topk, void* stream);
int pb_moe_combine_pos(const void* y, const void* topw, const void* pos, const void* residual, void* out, int M, int H, int topk, void* stream);

// 2-CTA variant (gemm_tcgen05_2cta.cu): plain K-major GEMMs with optional SwiGLU / residual; PB_ERR_UNSUPPORTED for anything else
int pb_gemm_bf16_2cta(const PbGemmArgs* args, void* stream);

// ---- block-scaled FP8 GEMM (gemm_mxfp8.cu): both operands MXFP8 (E4M3 payload + UE8M0 scale per 32 values along K) -------------
// Scale arrays use the tensor cores' block layout: [K / 128][ceil(rows / 128)][512 B], scale of (row r, K slice c) of a block at
// (r % 32) * 16 + (r / 32) * 4 + c  (ops/quant.py:pack_scales; pb_quant_mxfp8 writes it for activations).
typedef struct {
  const void* a_q;   // [M, K] e4m3
  const void* a_sf;
  const void* b_q;   // [N, K] e4m3 (nn.Linear weight layout)
  const void* b_sf;
  const void* b2_q;  // act == 1: second weight (up_proj); the epilogue emits silu(a b^T) * (a b2^T)
  const void* b2_sf;
  const void* residual;  // bf16 [M, N] or null
  void* out;             // bf16 [M, N]
  int M, N, K;
  int ldo, ldres;        // 0 = N
  int act;               // 0 none, 1 SwiGLU
  int num_sms;
} PbGemmFp8Args;
int pb_gemm_mxfp8(const PbGemmFp8Args* args, void* stream);
int pb_gemm_mxfp8_2cta(const PbGemmFp8Args* args, void* stream);   // cta_group::2: one 256 x 256 tile per SM pair
// x bf16 [M, K] -> q e4m3 [M, K] + scales in the block layout; with norm_w: quantises RMSNorm(x) * norm_w (HF rounding) instead.
int pb_quant_mxfp8(const void* x, const void* norm_w, float eps, void* q, void* sf, int M, int K, void* stream);

// ---- stand-alone halves of the LL all-reduce (ll_collectives.cu): tag = *epoch * mul + add -----------------------------------
int pb_ll_reduce(const void* x, void* const* parts, int R, const void* epoch, unsigned mul, unsigned add, void* out, long n_values,
                 void* error_flag, void* stream);
int pb_ll_push(const void* x, void* const* dst, int R, const void* epoch, unsigned mul, unsigned add, long n_values, void* stream);

// ---- KV cache utilities -----------------------------------------------------------------------------
int pb_kv_copy_pages(void* pool, const void* src_pages, const void* dst_pages, int n, long page_elems,
                     long layer_stride_elems, int n_layer_slabs, void* stream);

// ---- runtime (host) ---------------------------------------------------------------------------------
int pb_device_sm_count(int device);
const char* pb_last_error(void);
int pb_check_launch(const char* what);  // cudaGetLastError -> PB_OK / PB_ERR_CUDA, remembers the message
int pb_version(void);

#ifdef __cplusplus
}
#endif
