// petals_b200 — decode-shape linear layer (1..8 tokens): a pure HBM weight streamer.
//
//   out[m, n] = epilogue( sum_k prologue(x)[m, k] * W[n, k] )          W is the HF nn.Linear layout
//
// At decode time tensor cores are idle and the op is bound by reading W exactly once
// (SURVEY.md §7.3 item 1), so this kernel is built around keeping >= 64 KB of 128-bit
// non-allocating loads in flight per SM and fusing everything around the GEMV into it:
//
//   prologue  : [wait on NVLink peer flag] -> [x = residual + sum of TP partials] ->
//               [RMSNorm | LayerNorm] -> bf16 x staged once in shared memory
//   main loop : one warp owns a pair of output columns and streams their two weight rows
//               (plus the two `up_proj` rows for SwiGLU) with 8 independent 16-byte loads per lane
//   epilogue  : [+bias] -> [SwiGLU | GELU] -> [+residual] -> store to local HBM and/or straight
//               into peer GPUs' buffers over NVLink, then a release-increment of the peers' flags.
//
// The last two items are the decode-time "stage hop" (pipeline) and the one-shot all-reduce
// (tensor parallel) fused into the producing GEMV and the consuming GEMV: no NCCL call and no
// separate communication kernel on the token path (replaces X1/X4/X5 of SURVEY.md §2.5(c),
// reference: src/petals/client/inference_session.py:153-172, utils/convert_block.py:128).
#include "common.cuh"
#include "petals_b200.h"

extern "C" int pb_set_error(const char* msg);

namespace pb {

constexpr int kMaxPeers = 8;

struct LinearDecodeParams {
  const __nv_bfloat16* x;         // [M, K] input / residual-in for the reduce prologue
  const __nv_bfloat16* w;         // [N, K]
  const __nv_bfloat16* w2;        // [N, K] second weight (SwiGLU up_proj) or null
  const __nv_bfloat16* bias;      // [N] or null
  const __nv_bfloat16* bias2;     // [N] or null
  const __nv_bfloat16* residual;  // [M, N] or null (epilogue residual add)
  __nv_bfloat16* out;             // [M, N] local output or null (push only)
  const __nv_bfloat16* norm_w;    // [K] or null
  const __nv_bfloat16* norm_b;    // [K] or null (LayerNorm)
  __nv_bfloat16* x_out;           // [M, K] optional: block 0 writes the reduced (pre-norm) x here
  float eps;
  int norm_kind;                  // 0 none, 1 RMSNorm, 2 LayerNorm
  int act;                        // 0 none, 1 SwiGLU(w, w2), 2 GELU(tanh), 3 GELU(erf)
  int M, N, K;
  // --- fused communication -------------------------------------------------------------
  int n_parts;                                  // reduce prologue: x += sum_r parts[r]
  const __nv_bfloat16* parts[kMaxPeers];        // local buffers written by peers
  const uint64_t* wait_flag;                    // prologue waits until *wait_flag >= *epoch * wait_per_epoch
  uint64_t wait_per_epoch;
  const uint64_t* epoch;                        // device-resident step counter (graph friendly)
  int n_push;                                   // epilogue also stores to these (peer) buffers
  __nv_bfloat16* push_out[kMaxPeers];           // [M, N] each
  uint64_t* push_flag[kMaxPeers];               // incremented (release.sys) ONCE per launch, by the last CTA to finish
  unsigned int* done_counter;                   // local device counter used to elect that last CTA (self-resetting)
  int* error_flag;                              // set to 1 on watchdog expiry
  // ---- LL ("low latency") one-shot all-reduce: every partial is sent as 8-byte {2 x bf16, 32-bit tag} stores, so data and
  // validity arrive in one NVLink transaction and the consumer polls the payload itself. No fence, no last-CTA election, no
  // flag round trip (the flag protocol above costs a release fence + atomic + flag hop per all-reduce). tag = epoch * mul + add
  // identifies (step, layer); buffers are never cleared.
  const uint2* ll_parts[kMaxPeers];             // prologue: local buffers [M, K/2] written by the peers' epilogues
  int n_ll_parts;
  uint2* ll_push[kMaxPeers];                    // epilogue: peers' buffers [M, N/2] (this rank's slot)
  int n_ll_push;
  uint32_t ll_tag_mul, ll_tag_add;
  // ---- fused RoPE + paged KV append (QKV projection of Llama-style blocks): the epilogue rotates q/k with HF's bf16
  // rounding, stores q token-major for the attention kernel and writes k/v straight into the session's cache pages, so the
  // decode step needs no separate RoPE/append launch. Output columns are then processed as rotary pairs (i, i + D/2).
  __nv_bfloat16* rope_q_out;                    // [M, Hq*D]; non-null enables the fusion (template flag ROPE)
  __nv_bfloat16* rope_k_pool;
  __nv_bfloat16* rope_v_pool;
  const int* rope_block_table;                  // [B, max_pages]
  const int* rope_pos_ptr;                      // device-resident position of the first new token
  const float* rope_cos;                        // [max_pos, D/2] fp32 (null: no rotation, append only)
  const float* rope_sin;
  int rope_T, rope_Hq, rope_Hkv, rope_D, rope_max_pages, rope_max_pos, rope_num_pages;
  int split_k;                                  // > 1: that many warps share one row pair, each streaming 1/split_k of K
  int pf_lines;                                 // 128-byte weight lines each warp prefetches into L2 before the prologue
};

PB_DEVICE float gelu_tanh(float x) {
  const float k0 = 0.7978845608028654f, k1 = 0.044715f;
  return 0.5f * x * (1.f + tanhf(k0 * (x + k1 * x * x * x)));
}
PB_DEVICE float gelu_erf(float x) { return 0.5f * x * (1.f + erff(x * 0.7071067811865475f)); }
PB_DEVICE float silu(float x) { return x / (1.f + __expf(-x)); }

// 8 bf16 weights (one uint4) times 8 pre-converted fp32 activations per token. Activations are converted ONCE per load
// slot and reused for every weight row of the slot (2 rows, or 4 with SwiGLU): at M >= 2 the bf16->fp32 unpacking of x would
// otherwise saturate the integer pipe before HBM saturates.
template <int M>
PB_DEVICE void fma8(float (&acc)[M], const uint4& w, const float (&xf)[M][8]) {
  const float w0 = bf16_lo(w.x), w1 = bf16_hi(w.x), w2 = bf16_lo(w.y), w3 = bf16_hi(w.y);
  const float w4 = bf16_lo(w.z), w5 = bf16_hi(w.z), w6 = bf16_lo(w.w), w7 = bf16_hi(w.w);
#pragma unroll
  for (int m = 0; m < M; ++m) {
    float a = acc[m];
    a = fmaf(w0, xf[m][0], a); a = fmaf(w1, xf[m][1], a); a = fmaf(w2, xf[m][2], a); a = fmaf(w3, xf[m][3], a);
    a = fmaf(w4, xf[m][4], a); a = fmaf(w5, xf[m][5], a); a = fmaf(w6, xf[m][6], a); a = fmaf(w7, xf[m][7], a);
    acc[m] = a;
  }
}

// Block-wide sum of `v` (one value per thread) broadcast to all threads. `red` holds >= 32 floats.
PB_DEVICE float block_sum(float v, float* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  v = warp_sum(v);
  __syncthreads();  // protect `red` from the previous use
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float t = (lane < nw) ? red[lane] : 0.f;
  return warp_sum(t);
}

PB_DEVICE float rbf16(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }

// Warm L2 with the head of the first weight rows every warp will stream (weights are never written by a kernel, so this may
// run before the producer of x has finished: behind a programmatic dependency or a peer-flag wait).
template <bool DUAL, bool ROPE>
PB_DEVICE void gemv_prefetch(const LinearDecodeParams& p) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int grid = gridDim.x, bid = blockIdx.x, nwarps = blockDim.x >> 5;
  const int task0 = warp * grid + bid;
  if (warp < nwarps && task0 < (p.N >> 1) && p.pf_lines > 0) {
    constexpr int kRows = DUAL ? 4 : 2;
    const int lines_per_row = p.pf_lines / kRows;
    const int half_d = ROPE ? (p.rope_D >> 1) : 1;
    const int n0 = ROPE ? (task0 / half_d) * p.rope_D + task0 % half_d : task0 << 1;
    for (int i = lane; i < p.pf_lines; i += 32) {
      const int row = i / lines_per_row, k = (i - row * lines_per_row) * 64;
      if (row < kRows && k < p.K) prefetch_l2((row < 2 ? p.w : p.w2) + static_cast<size_t>(n0 + (row & 1) * half_d) * p.K + k);
    }
  }
}

// One decode-shape linear layer; all CTAs of the grid cooperate. M = tokens, DUAL = SwiGLU (two weight matrices),
// XSMEM = x staged in shared memory, ROPE = fused RoPE + KV append epilogue.
template <int M, bool DUAL, bool XSMEM, bool ROPE>
PB_DEVICE void gemv_body(const LinearDecodeParams& p, uint8_t* smem_raw) {
  __nv_bfloat16* xs = reinterpret_cast<__nv_bfloat16*>(smem_raw);
  __shared__ float red[32];
  __shared__ float stat[2 * M];

  const int K = p.K, N = p.N;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int tid = threadIdx.x, nthr = blockDim.x;
  const int grid = gridDim.x, bid = blockIdx.x, nwarps = nthr >> 5;

  // ---- prologue ----------------------------------------------------------------------------
  if (p.wait_flag != nullptr) {
    if (tid == 0) {
      const uint64_t target = *p.epoch * p.wait_per_epoch;
      if (!spin_wait_ge(p.wait_flag, target)) atomicExch(p.error_flag, 1);
    }
    __syncthreads();
  }
  const uint32_t ll_tag = (p.n_ll_parts > 0 || p.n_ll_push > 0) ? static_cast<uint32_t>(*p.epoch) * p.ll_tag_mul + p.ll_tag_add : 0u;
  if (XSMEM) {
    const int kvec = K >> 3;  // 8 bf16 per 16-byte vector
    float ssum[M], ssq[M];
#pragma unroll
    for (int m = 0; m < M; ++m) ssum[m] = ssq[m] = 0.f;
    for (int v = tid; v < kvec; v += nthr) {
#pragma unroll
      for (int m = 0; m < M; ++m) {
        const size_t off = static_cast<size_t>(m) * K + (static_cast<size_t>(v) << 3);
        uint4 xv = __ldcg(reinterpret_cast<const uint4*>(p.x + off));
        if (p.n_parts > 0 || p.n_ll_parts > 0) {
          float f[8] = {bf16_lo(xv.x), bf16_hi(xv.x), bf16_lo(xv.y), bf16_hi(xv.y),
                        bf16_lo(xv.z), bf16_hi(xv.z), bf16_lo(xv.w), bf16_hi(xv.w)};
          for (int r = 0; r < p.n_ll_parts; ++r) {
            // 8 values = 4 LL units = 32 bytes; spin until all four carry this step's tag
            const uint4* src = reinterpret_cast<const uint4*>(p.ll_parts[r] + (off >> 1));
            uint4 a, b;
            unsigned long long t0 = 0;
            for (unsigned spins = 0;; ++spins) {
              a = ld_relaxed_sys_v4(src);
              b = ld_relaxed_sys_v4(src + 1);
              if (a.y == ll_tag && a.w == ll_tag && b.y == ll_tag && b.w == ll_tag) break;
              if ((spins & 1023u) == 1023u) {
                const unsigned long long now = globaltimer_ns();
                if (t0 == 0) t0 = now;
                else if (now - t0 > PB_FLAG_TIMEOUT_NS) { if (p.error_flag != nullptr) atomicExch(p.error_flag, 1); break; }
              }
            }
            f[0] += bf16_lo(a.x); f[1] += bf16_hi(a.x); f[2] += bf16_lo(a.z); f[3] += bf16_hi(a.z);
            f[4] += bf16_lo(b.x); f[5] += bf16_hi(b.x); f[6] += bf16_lo(b.z); f[7] += bf16_hi(b.z);
          }
          for (int r = 0; r < p.n_parts; ++r) {
            uint4 pv = __ldcg(reinterpret_cast<const uint4*>(p.parts[r] + off));
            f[0] += bf16_lo(pv.x); f[1] += bf16_hi(pv.x); f[2] += bf16_lo(pv.y); f[3] += bf16_hi(pv.y);
            f[4] += bf16_lo(pv.z); f[5] += bf16_hi(pv.z); f[6] += bf16_lo(pv.w); f[7] += bf16_hi(pv.w);
          }
          xv.x = pack_bf16(f[0], f[1]); xv.y = pack_bf16(f[2], f[3]);
          xv.z = pack_bf16(f[4], f[5]); xv.w = pack_bf16(f[6], f[7]);
          if (p.x_out != nullptr && bid == 0)
            *reinterpret_cast<uint4*>(p.x_out + off) = xv;
        }
        *reinterpret_cast<uint4*>(xs + off) = xv;
        if (p.norm_kind != 0) {
          const float f0 = bf16_lo(xv.x), f1 = bf16_hi(xv.x), f2 = bf16_lo(xv.y), f3 = bf16_hi(xv.y);
          const float f4 = bf16_lo(xv.z), f5 = bf16_hi(xv.z), f6 = bf16_lo(xv.w), f7 = bf16_hi(xv.w);
          ssum[m] += (f0 + f1) + (f2 + f3) + (f4 + f5) + (f6 + f7);
          ssq[m] += f0 * f0 + f1 * f1 + f2 * f2 + f3 * f3 + f4 * f4 + f5 * f5 + f6 * f6 + f7 * f7;
        }
      }
    }
    if (p.norm_kind != 0) {
#pragma unroll
      for (int m = 0; m < M; ++m) {
        const float s1 = block_sum(ssum[m], red);
        const float s2 = block_sum(ssq[m], red);
        if (tid == 0) {
          if (p.norm_kind == 1) {
            stat[2 * m] = 0.f;
            stat[2 * m + 1] = rsqrtf(s2 / K + p.eps);
          } else {
            const float mean = s1 / K;
            const float var = fmaxf(s2 / K - mean * mean, 0.f);
            stat[2 * m] = mean;
            stat[2 * m + 1] = rsqrtf(var + p.eps);
          }
        }
      }
      __syncthreads();
      for (int v = tid; v < kvec; v += nthr) {
        const uint4 gv = __ldg(reinterpret_cast<const uint4*>(p.norm_w) + v);
        uint4 bv = make_uint4(0, 0, 0, 0);
        if (p.norm_kind == 2 && p.norm_b != nullptr) bv = __ldg(reinterpret_cast<const uint4*>(p.norm_b) + v);
        const float g[8] = {bf16_lo(gv.x), bf16_hi(gv.x), bf16_lo(gv.y), bf16_hi(gv.y),
                            bf16_lo(gv.z), bf16_hi(gv.z), bf16_lo(gv.w), bf16_hi(gv.w)};
        const float b[8] = {bf16_lo(bv.x), bf16_hi(bv.x), bf16_lo(bv.y), bf16_hi(bv.y),
                            bf16_lo(bv.z), bf16_hi(bv.z), bf16_lo(bv.w), bf16_hi(bv.w)};
#pragma unroll
        for (int m = 0; m < M; ++m) {
          const float mean = stat[2 * m], rstd = stat[2 * m + 1];
          uint4* px = reinterpret_cast<uint4*>(xs + static_cast<size_t>(m) * K) + v;
          const uint4 xv = *px;
          float f[8] = {bf16_lo(xv.x), bf16_hi(xv.x), bf16_lo(xv.y), bf16_hi(xv.y),
                        bf16_lo(xv.z), bf16_hi(xv.z), bf16_lo(xv.w), bf16_hi(xv.w)};
          if (p.norm_kind == 1) {
            // HF RMSNorm rounding: weight * bf16(x * rstd)
#pragma unroll
            for (int i = 0; i < 8; ++i)
              f[i] = __bfloat162float(__float2bfloat16_rn(f[i] * rstd)) * g[i];
          } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) f[i] = (f[i] - mean) * rstd * g[i] + b[i];
          }
          uint4 o;
          o.x = pack_bf16(f[0], f[1]); o.y = pack_bf16(f[2], f[3]);
          o.z = pack_bf16(f[4], f[5]); o.w = pack_bf16(f[6], f[7]);
          *px = o;
        }
      }
    }
    __syncthreads();
  }

  // ---- main loop: each warp owns a pair of output columns ------------------------------------
  // A warp's work is the sequence of "slots" (task, it): U 16-byte loads per weight row of row pair `task` at K offset it*kstep.
  // Load slot, multiply, next slot: 24 warps/SM hide the latency by interleaving.
  constexpr int U = DUAL ? 2 : 4;  // 16-byte loads per weight row per slot (8 in flight per lane)
  const int ntasks = N >> 1;
  const int total_warps = grid * nwarps;
  const int kstep = 256 * U;
  const int nit = (K + kstep - 1) / kstep;
  const int half_d = ROPE ? (p.rope_D >> 1) : 1;
  struct Slot { uint4 wa[U], wb[U], ua[U], ub[U]; };
  float a0[M], a1[M], b0[M], b1[M];
#pragma unroll
  for (int m = 0; m < M; ++m) a0[m] = a1[m] = b0[m] = b1[m] = 0.f;

  // plain: adjacent output columns (n0, n0+1); ROPE: the rotary pair (i, i + D/2) of one head
  auto first_col = [&](int task) { return ROPE ? (task / half_d) * p.rope_D + task % half_d : task << 1; };
  auto load_slot = [&](Slot& s, int task, int it) {
    const int n0 = first_col(task);
    const __nv_bfloat16* w0 = p.w + static_cast<size_t>(n0) * K;
    const __nv_bfloat16* w1 = w0 + static_cast<size_t>(half_d) * K;
    const __nv_bfloat16* u0 = DUAL ? p.w2 + static_cast<size_t>(n0) * K : nullptr;
    const __nv_bfloat16* u1 = DUAL ? u0 + K : nullptr;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int k = it * kstep + u * 256 + lane * 8;
      if (k < K) {
        s.wa[u] = ld_stream(w0 + k);
        s.wb[u] = ld_stream(w1 + k);
        if (DUAL) {
          s.ua[u] = ld_stream(u0 + k);
          s.ub[u] = ld_stream(u1 + k);
        }
      }
    }
  };
  auto compute_slot = [&](const Slot& s, int it) {
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int k = it * kstep + u * 256 + lane * 8;
      if (k < K) {
        float xf[M][8];
#pragma unroll
        for (int m = 0; m < M; ++m) {
          uint4 xv;
          if (XSMEM) xv = *reinterpret_cast<const uint4*>(xs + static_cast<size_t>(m) * K + k);
          else xv = ld_cached(p.x + static_cast<size_t>(m) * K + k);
          xf[m][0] = bf16_lo(xv.x); xf[m][1] = bf16_hi(xv.x); xf[m][2] = bf16_lo(xv.y); xf[m][3] = bf16_hi(xv.y);
          xf[m][4] = bf16_lo(xv.z); xf[m][5] = bf16_hi(xv.z); xf[m][6] = bf16_lo(xv.w); xf[m][7] = bf16_hi(xv.w);
        }
        fma8<M>(a0, s.wa[u], xf);
        fma8<M>(a1, s.wb[u], xf);
        if (DUAL) {
          fma8<M>(b0, s.ua[u], xf);
          fma8<M>(b1, s.ub[u], xf);
        }
      }
    }
  };
  // reduce the row pair over the warp, run the epilogue, reset the accumulators
  auto finish_task = [&](int task, bool reduced = false) {
    const int n0 = first_col(task);
    if (!reduced) {  // split-K callers pass sums that are already warp-uniform
#pragma unroll
      for (int m = 0; m < M; ++m) {
        a0[m] = warp_sum(a0[m]);
        a1[m] = warp_sum(a1[m]);
        if (DUAL) {
          b0[m] = warp_sum(b0[m]);
          b1[m] = warp_sum(b1[m]);
        }
      }
    }
    // ---- epilogue: lane m handles token m --------------------------------------------------
    float v0 = 0.f, v1 = 0.f, c0 = 0.f, c1 = 0.f;
#pragma unroll
    for (int m = 0; m < M; ++m) {
      if (lane == m) {
        v0 = a0[m]; v1 = a1[m];
        if (DUAL) { c0 = b0[m]; c1 = b1[m]; }
      }
    }
    if (ROPE) {
      if (lane < M) {
        const int D = p.rope_D, head = n0 / D, i = n0 - head * D;
        const int b = lane / p.rope_T, t = lane - b * p.rope_T;
        const int pos = *p.rope_pos_ptr + t;
        float x0 = rbf16(v0), x1 = rbf16(v1);  // the projection output is a bf16 tensor in the unfused pipeline
        const bool is_v = head >= p.rope_Hq + p.rope_Hkv;
        if (!is_v && p.rope_cos != nullptr) {
          const int pp = pos < p.rope_max_pos ? pos : p.rope_max_pos - 1;
          const float c = rbf16(p.rope_cos[static_cast<size_t>(pp) * half_d + i]);
          const float sn = rbf16(p.rope_sin[static_cast<size_t>(pp) * half_d + i]);
          const float y0 = rbf16(rbf16(x0 * c) + rbf16(-x1 * sn));   // HF rotate_half with bf16 rounding of every product
          const float y1 = rbf16(rbf16(x1 * c) + rbf16(x0 * sn));
          x0 = y0; x1 = y1;
        }
        __nv_bfloat16* dst;
        if (head < p.rope_Hq) {
          dst = p.rope_q_out + (static_cast<size_t>(lane) * p.rope_Hq + head) * D;
        } else {
          const int kvh = is_v ? head - p.rope_Hq - p.rope_Hkv : head - p.rope_Hq;
          const int pg_idx = pos >> 6;  // 64-token pages
          if (pg_idx >= p.rope_max_pages) {
            if (p.error_flag != nullptr) atomicExch(p.error_flag, 2);
            dst = nullptr;
          } else {
            const int pg = p.rope_block_table[static_cast<size_t>(b) * p.rope_max_pages + pg_idx];
            if (pg < 0 || pg >= p.rope_num_pages) {  // never write outside the pool
              if (p.error_flag != nullptr) atomicExch(p.error_flag, 2);
              dst = nullptr;
            } else {
              dst = (is_v ? p.rope_v_pool : p.rope_k_pool) + ((static_cast<size_t>(pg) * p.rope_Hkv + kvh) * 64 + (pos & 63)) * D;
            }
          }
        }
        if (dst != nullptr) {
          dst[i] = __float2bfloat16_rn(x0);
          dst[i + half_d] = __float2bfloat16_rn(x1);
        }
      }
    } else if (lane < M) {
      if (p.bias != nullptr) {
        v0 += __bfloat162float(p.bias[n0]);
        v1 += __bfloat162float(p.bias[n0 + 1]);
      }
      if (DUAL) {
        if (p.bias2 != nullptr) {
          c0 += __bfloat162float(p.bias2[n0]);
          c1 += __bfloat162float(p.bias2[n0 + 1]);
        }
        // HF: act(gate) * up, each projection rounded to bf16 first
        v0 = __bfloat162float(__float2bfloat16_rn(v0));
        v1 = __bfloat162float(__float2bfloat16_rn(v1));
        c0 = __bfloat162float(__float2bfloat16_rn(c0));
        c1 = __bfloat162float(__float2bfloat16_rn(c1));
        v0 = __bfloat162float(__float2bfloat16_rn(silu(v0))) * c0;
        v1 = __bfloat162float(__float2bfloat16_rn(silu(v1))) * c1;
      } else if (p.act == 2) {
        v0 = gelu_tanh(v0); v1 = gelu_tanh(v1);
      } else if (p.act == 3) {
        v0 = gelu_erf(v0); v1 = gelu_erf(v1);
      }
      const size_t o = static_cast<size_t>(lane) * N + n0;
      if (p.residual != nullptr) {
        const uint32_t rv = *reinterpret_cast<const uint32_t*>(p.residual + o);
        // HF: residual + bf16(proj)
        v0 = __bfloat162float(__float2bfloat16_rn(v0)) + bf16_lo(rv);
        v1 = __bfloat162float(__float2bfloat16_rn(v1)) + bf16_hi(rv);
      }
      const uint32_t packed = pack_bf16(v0, v1);
      if (p.out != nullptr) *reinterpret_cast<uint32_t*>(p.out + o) = packed;
      for (int r = 0; r < p.n_push; ++r) *reinterpret_cast<uint32_t*>(p.push_out[r] + o) = packed;
      for (int r = 0; r < p.n_ll_push; ++r) st_relaxed_sys_v2(p.ll_push[r] + (o >> 1), packed, ll_tag);
    }
#pragma unroll
    for (int m = 0; m < M; ++m) a0[m] = a1[m] = b0[m] = b1[m] = 0.f;
  };

  int task = warp < nwarps ? warp * grid + bid : ntasks;
  if (p.split_k > 1) {
    // Split-K inside the CTA for projections with few output columns (tensor-parallel QKV shards): S consecutive warps share one
    // row pair, each streams 1/S of K, partial sums meet in shared memory. Without it such a launch has one warp per row pair
    // in total (e.g. 640 warps for a 21 MB matrix) and is bound by the bytes it can keep in flight, not by HBM.
    __shared__ float sk_part[24][M][4];
    const int S = p.split_k;
    const int groups = nwarps / S;
    const int g = warp / S, sidx = warp - g * S;
    const int spw = (nit + S - 1) / S;  // slots per warp
    for (int tb = bid * groups; tb < ntasks; tb += grid * groups) {  // trip count is CTA-uniform (barriers inside)
      const int t = tb + g;
      const bool active = warp < groups * S && t < ntasks;
      if (active) {
        Slot sl;
        const int it1 = min(nit, (sidx + 1) * spw);
        for (int it = sidx * spw; it < it1; ++it) {
          load_slot(sl, t, it);
          compute_slot(sl, it);
        }
      }
#pragma unroll
      for (int m = 0; m < M; ++m) {
        const float r0 = warp_sum(a0[m]), r1 = warp_sum(a1[m]);
        const float r2 = DUAL ? warp_sum(b0[m]) : 0.f, r3 = DUAL ? warp_sum(b1[m]) : 0.f;
        if (lane == 0) { sk_part[warp][m][0] = r0; sk_part[warp][m][1] = r1; sk_part[warp][m][2] = r2; sk_part[warp][m][3] = r3; }
      }
      __syncthreads();
      if (active && sidx == 0) {
#pragma unroll
        for (int m = 0; m < M; ++m) {
          a0[m] = a1[m] = b0[m] = b1[m] = 0.f;
          for (int q = 0; q < S; ++q) {
            a0[m] += sk_part[warp + q][m][0]; a1[m] += sk_part[warp + q][m][1];
            if (DUAL) { b0[m] += sk_part[warp + q][m][2]; b1[m] += sk_part[warp + q][m][3]; }
          }
        }
        finish_task(t, true);
      }
#pragma unroll
      for (int m = 0; m < M; ++m) a0[m] = a1[m] = b0[m] = b1[m] = 0.f;
      __syncthreads();
    }
  } else {
    Slot s;
    for (; task < ntasks; task += total_warps) {
      for (int it = 0; it < nit; ++it) {
        load_slot(s, task, it);
        compute_slot(s, it);
      }
      finish_task(task);
    }
  }

  // ---- publish: every CTA fences its peer stores and checks in on a local counter; the last one to arrive
  // performs ONE release-increment per peer (so a consumer waits for `n_sources` per step, independent of grids).
  if (p.n_push > 0) {
    __syncthreads();
    if (tid == 0) {
      __threadfence_system();
      const unsigned int prev = atomicAdd(p.done_counter, 1u);
      if (prev == static_cast<unsigned int>(grid) - 1) {
        __threadfence_system();
        *p.done_counter = 0u;
        for (int r = 0; r < p.n_push; ++r)
          if (p.push_flag[r] != nullptr) red_release_sys_add(p.push_flag[r], 1ull);
      }
    }
  }
}

template <int M, bool DUAL, bool XSMEM, bool ROPE = false>
__global__ void __launch_bounds__((M <= 4 ? 768 : 512), 1) linear_decode_kernel(const LinearDecodeParams p) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  // ---- PDL pre-section: while the predecessor kernel drains (and while this kernel then waits for a peer flag and normalises x)
  // every warp pulls the head of its first weight rows into L2, so HBM keeps streaming through the bubble between two GEMVs
  if (threadIdx.x == 0) pdl_trigger();
  gemv_prefetch<DUAL, ROPE>(p);
  // one warp parks on the grid dependency, the rest of the CTA parks on the barrier behind it
  if ((threadIdx.x >> 5) == 0) pdl_wait();
  __syncthreads();
  gemv_body<M, DUAL, XSMEM, ROPE>(p, smem_raw);
}

template <int M, bool DUAL, bool XSMEM, bool ROPE = false>
static cudaError_t launch_one(const LinearDecodeParams& p, int grid, int block, size_t smem,
                              cudaStream_t stream) {
  auto kern = linear_decode_kernel<M, DUAL, XSMEM, ROPE>;
  if (smem > 32 * 1024) {  // static shared memory counts against the 48 KB default too
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         static_cast<int>(smem));
    if (e != cudaSuccess) return e;
  }
  // Programmatic dependent launch pays for small weight matrices (kernel-boundary latency is a visible fraction of a short
  // kernel: 8B-class shapes, tensor-parallel shards) and costs ~4 % on long streaming kernels (70B on one GPU); measured in
  // profiles/r1_pdl_sweep.txt. The cut-over is a byte threshold on the streamed weights.
  static const long max_mb = [] { const char* e = getenv("PETALS_B200_PDL_GEMV_MAX_MB"); return e ? atol(e) : 128L; }();
  const long wbytes = static_cast<long>(p.N) * p.K * 2 * (DUAL ? 2 : 1);
  const int kind = wbytes <= (max_mb << 20) ? (kPdlGemv | kPdlGemvBigSmem | kPdlGemvAuto) : (smem > 32 * 1024 ? kPdlGemvBigSmem : kPdlGemv);
  return launch_pdl(kind, kern, dim3(grid), dim3(block), smem, stream, p);
}

template <int M>
static cudaError_t launch_m(const LinearDecodeParams& p, bool dual, bool xsmem, int grid, int block,
                            size_t smem, cudaStream_t s) {
  if (p.rope_q_out != nullptr) return launch_one<M, false, true, true>(p, grid, block, smem, s);  // validated: !dual && xsmem
  if (dual) return xsmem ? launch_one<M, true, true>(p, grid, block, smem, s)
                         : launch_one<M, true, false>(p, grid, block, smem, s);
  return xsmem ? launch_one<M, false, true>(p, grid, block, smem, s)
               : launch_one<M, false, false>(p, grid, block, smem, s);
}

}  // namespace pb

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
namespace pb {

struct GemvGeom { bool dual, xsmem; size_t smem; int grid, best_w; };

// Validate one linear's arguments, translate them into kernel parameters and pick its launch geometry.
static int gemv_fill(const PbLinearDecodeArgs* a, LinearDecodeParams& p, GemvGeom& g) {
  if (a->M < 1 || a->M > 8 || (a->N & 1) || (a->K & 7)) return PB_ERR_SHAPE;
  if (a->n_parts > kMaxPeers || a->n_push > kMaxPeers) return PB_ERR_SHAPE;
  p = LinearDecodeParams{};
  p.x = static_cast<const __nv_bfloat16*>(a->x);
  p.w = static_cast<const __nv_bfloat16*>(a->w);
  p.w2 = static_cast<const __nv_bfloat16*>(a->w2);
  p.bias = static_cast<const __nv_bfloat16*>(a->bias);
  p.bias2 = static_cast<const __nv_bfloat16*>(a->bias2);
  p.residual = static_cast<const __nv_bfloat16*>(a->residual);
  p.out = static_cast<__nv_bfloat16*>(a->out);
  p.norm_w = static_cast<const __nv_bfloat16*>(a->norm_w);
  p.norm_b = static_cast<const __nv_bfloat16*>(a->norm_b);
  p.x_out = static_cast<__nv_bfloat16*>(a->x_out);
  p.eps = a->eps;
  p.norm_kind = a->norm_kind;
  p.act = a->act;
  p.M = a->M; p.N = a->N; p.K = a->K;
  p.n_parts = a->n_parts;
  for (int i = 0; i < a->n_parts; ++i) p.parts[i] = static_cast<const __nv_bfloat16*>(a->parts[i]);
  p.wait_flag = static_cast<const uint64_t*>(a->wait_flag);
  p.wait_per_epoch = a->wait_per_epoch;
  p.epoch = static_cast<const uint64_t*>(a->epoch);
  p.n_push = a->n_push;
  for (int i = 0; i < a->n_push; ++i) {
    p.push_out[i] = static_cast<__nv_bfloat16*>(a->push_out[i]);
    p.push_flag[i] = static_cast<uint64_t*>(a->push_flag[i]);
  }
  p.error_flag = static_cast<int*>(a->error_flag);
  if (a->n_ll_parts < 0 || a->n_ll_parts > kMaxPeers || a->n_ll_push < 0 || a->n_ll_push > kMaxPeers) return PB_ERR_SHAPE;
  if ((a->n_ll_parts > 0 || a->n_ll_push > 0) && a->epoch == nullptr) return PB_ERR_SHAPE;
  if (a->n_ll_push > 0 && a->act == 1) return PB_ERR_SHAPE;  // LL pushes come from the row-parallel projections
  p.n_ll_parts = a->n_ll_parts; p.n_ll_push = a->n_ll_push;
  for (int i = 0; i < a->n_ll_parts; ++i) p.ll_parts[i] = static_cast<const uint2*>(a->ll_parts[i]);
  for (int i = 0; i < a->n_ll_push; ++i) p.ll_push[i] = static_cast<uint2*>(a->ll_push[i]);
  p.ll_tag_mul = a->ll_tag_mul; p.ll_tag_add = a->ll_tag_add;
  if (a->rope_q_out != nullptr) {
    const int D = a->rope_D, heads = a->rope_Hq + 2 * a->rope_Hkv;
    if (a->act != 0 || a->bias != nullptr || a->residual != nullptr || a->n_push > 0 || D < 2 || (D & 1) || a->N != heads * D || a->rope_T < 1 ||
        a->M % a->rope_T != 0 || a->rope_k_pool == nullptr || a->rope_v_pool == nullptr || a->rope_block_table == nullptr ||
        a->rope_pos_ptr == nullptr || (a->rope_cos != nullptr && a->rope_sin == nullptr))
      return PB_ERR_SHAPE;
    p.rope_q_out = static_cast<__nv_bfloat16*>(a->rope_q_out);
    p.rope_k_pool = static_cast<__nv_bfloat16*>(a->rope_k_pool);
    p.rope_v_pool = static_cast<__nv_bfloat16*>(a->rope_v_pool);
    p.rope_block_table = static_cast<const int*>(a->rope_block_table);
    p.rope_pos_ptr = static_cast<const int*>(a->rope_pos_ptr);
    p.rope_cos = static_cast<const float*>(a->rope_cos);
    p.rope_sin = static_cast<const float*>(a->rope_sin);
    p.rope_T = a->rope_T; p.rope_Hq = a->rope_Hq; p.rope_Hkv = a->rope_Hkv; p.rope_D = D;
    p.rope_max_pages = a->rope_max_pages; p.rope_max_pos = a->rope_max_pos;
    p.rope_num_pages = a->rope_num_pages > 0 ? a->rope_num_pages : 0x7fffffff;
  }
  {
    static const int env_pf = [] { const char* e = getenv("PETALS_B200_PF_LINES"); return e ? atoi(e) : -1; }();
    static const int env_pf_wait = [] { const char* e = getenv("PETALS_B200_PF_LINES_WAIT"); return e ? atoi(e) : -1; }();
    // a kernel that will spin on a peer flag can hide a deep prefetch behind the wait; one that starts right away cannot
    p.pf_lines = (a->wait_flag != nullptr || a->n_ll_parts > 0) ? (env_pf_wait >= 0 ? env_pf_wait : 64) : (env_pf >= 0 ? env_pf : 16);
    if (p.pf_lines > 0 && p.pf_lines < 4) p.pf_lines = 4;
  }
  p.done_counter = static_cast<unsigned int*>(a->done_counter);
  if (a->n_push > 0 && p.done_counter == nullptr) return PB_ERR_SHAPE;

  const bool dual = a->act == 1;
  if (dual && p.w2 == nullptr) return PB_ERR_SHAPE;
  const bool need_smem = a->norm_kind != 0 || a->n_parts > 0 || a->n_ll_parts > 0;
  const size_t xbytes = static_cast<size_t>(a->M) * a->K * 2;
  const bool xsmem = need_smem || xbytes <= 160 * 1024;
  if (need_smem && xbytes > 200 * 1024) return PB_ERR_SHAPE;
  const size_t smem = xsmem ? xbytes : 0;

  // Pick warps/SM in [12, 24] that minimises the last-wave quantisation loss. If a fixed grid
  // was requested (flag accounting across ranks needs identical CTA counts) honour it.
  const int sms = a->fixed_grid > 0 ? a->fixed_grid : (a->num_sms > 0 ? a->num_sms : 148);
  const int ntasks = a->N / 2;
  const int max_w = a->M <= 4 ? 24 : 16;
  int best_w = max_w;
  double best_eff = -1.0;
  for (int w = max_w; w >= max_w / 2; --w) {
    const long tw = static_cast<long>(sms) * w;
    const long rounds = (ntasks + tw - 1) / tw;
    const double eff = static_cast<double>(ntasks) / static_cast<double>(rounds * tw);
    if (eff > best_eff + 1e-9) { best_eff = eff; best_w = w; }
  }
  p.split_k = 1;
  static const int env_splitk = [] { const char* e = getenv("PETALS_B200_GEMV_SPLITK"); return e ? atoi(e) : 1; }();
  if (env_splitk && xsmem && a->M <= 4 && a->fixed_grid <= 0 && ntasks < sms * 12 && a->K >= 2048) {
    // few output columns: spread the row pairs over ALL SMs and let 4 (or 2) warps share each pair along K
    const int groups = (ntasks + sms - 1) / sms;
    const int S = groups * 4 <= 24 ? 4 : (groups * 2 <= 24 ? 2 : 1);
    if (S > 1) {
      p.split_k = S;
      g.dual = a->act == 1; g.xsmem = xsmem; g.smem = smem; g.grid = sms; g.best_w = groups * S;
      return PB_OK;
    }
  }
  int grid = sms;
  if (ntasks < sms * best_w) {  // small problem: do not launch idle CTAs beyond need
    grid = (ntasks + best_w - 1) / best_w;
    if (grid < 1) grid = 1;
    if (grid > sms) grid = sms;
  }
  if (a->fixed_grid > 0) grid = a->fixed_grid;
  g.dual = dual; g.xsmem = xsmem; g.smem = smem; g.grid = grid; g.best_w = best_w;
  return PB_OK;
}

}  // namespace pb

extern "C" int pb_linear_decode(const PbLinearDecodeArgs* a, void* stream) {
  using namespace pb;
  LinearDecodeParams p;
  GemvGeom g;
  const int rc = gemv_fill(a, p, g);
  if (rc != PB_OK) return rc;
  const bool dual = g.dual, xsmem = g.xsmem;
  const size_t smem = g.smem;
  const int grid = g.grid, best_w = g.best_w;
  const int block = best_w * 32;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  cudaError_t e = cudaSuccess;
  switch (a->M) {
    case 1: e = launch_m<1>(p, dual, xsmem, grid, block, smem, s); break;
    case 2: e = launch_m<2>(p, dual, xsmem, grid, block, smem, s); break;
    case 3: e = launch_m<3>(p, dual, xsmem, grid, block, smem, s); break;
    case 4: e = launch_m<4>(p, dual, xsmem, grid, block, smem, s); break;
    case 5: e = launch_m<5>(p, dual, xsmem, grid, block, smem, s); break;
    case 6: e = launch_m<6>(p, dual, xsmem, grid, block, smem, s); break;
    case 7: e = launch_m<7>(p, dual, xsmem, grid, block, smem, s); break;
    case 8: e = launch_m<8>(p, dual, xsmem, grid, block, smem, s); break;
  }
  if (e != cudaSuccess) {
    cudaGetLastError();
    char what[160];
    snprintf(what, sizeof(what), "linear_decode M=%d N=%d K=%d grid=%d block=%d smem=%zu: %s", a->M, a->N, a->K, grid, block, smem, cudaGetErrorString(e));
    pb_set_error(what);
    return PB_ERR_CUDA;
  }
  return a->out_grid ? (*(a->out_grid) = grid, PB_OK) : PB_OK;
}
