// petals_b200 — shared device-side primitives for sm_100a kernels.
//
// Thin inline-PTX wrappers for the Blackwell execution model: mbarrier, TMA
// (cp.async.bulk.tensor), tcgen05 (MMA / TMEM alloc / TMEM load / commit),
// system-scope acquire/release for NVLink peer flags, and small math helpers.
// Nothing here is a port of the reference (which ships no native code at all,
// see SURVEY.md §2.2); the patterns follow /opt/skills/guides/blackwell_cuda_programming.md.
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#define PB_DEVICE __device__ __forceinline__

#include <stdio.h>
#include <stdlib.h>

namespace pb {

// ---------------------------------------------------------------------------
// misc
// ---------------------------------------------------------------------------
PB_DEVICE uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
PB_DEVICE uint32_t lane_id() {
  uint32_t l;
  asm volatile("mov.u32 %0, %%laneid;" : "=r"(l));
  return l;
}
PB_DEVICE bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}
PB_DEVICE uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

PB_DEVICE float bf16_lo(uint32_t v) { return __uint_as_float(v << 16); }
PB_DEVICE float bf16_hi(uint32_t v) { return __uint_as_float(v & 0xffff0000u); }
PB_DEVICE uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
PB_DEVICE float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
PB_DEVICE float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// 128-bit streaming load that does not pollute L1 (weights are read exactly once).
PB_DEVICE uint4 ld_stream(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.L2::128B.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
PB_DEVICE void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// ---- programmatic dependent launch (PDL) -------------------------------------------------------------------------
// A kernel launched with the programmatic-stream-serialization attribute may start while its predecessor in the stream
// is still draining. Everything before pdl_wait() must touch only memory no earlier kernel writes (weights: L2
// prefetch); pdl_wait() returns once the predecessor has completed and its writes are visible. pdl_trigger() lets the
// *next* kernel's CTAs be scheduled as soon as this grid's CTAs have all started (they then park in their pdl_wait()).
// Both are no-ops when the kernel was launched without the attribute.
PB_DEVICE void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
PB_DEVICE void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

PB_DEVICE uint4 ld_cached(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

// ---------------------------------------------------------------------------
// system-scope flags (NVLink peer signalling). Acquire/release protocol:
//   producer: data stores → fence.acq_rel.sys (threadfence_system) → red.release.sys.add flag
//   consumer: ld.acquire.sys flag (spin with watchdog) → data loads
// ---------------------------------------------------------------------------
PB_DEVICE void st_release_sys(uint64_t* p, uint64_t v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
PB_DEVICE void red_release_sys_add(uint64_t* p, uint64_t v) {
  asm volatile("red.release.sys.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
PB_DEVICE uint64_t ld_acquire_sys(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
PB_DEVICE uint4 ld_relaxed_sys_v4(const uint4* p) {
  uint4 r;
  asm volatile("ld.relaxed.sys.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p) : "memory");
  return r;
}
// one 8-byte transaction: payload and validity tag arrive together (the LL protocol's atomicity unit)
PB_DEVICE void st_relaxed_sys_v2(uint2* p, uint32_t data, uint32_t tag) {
  asm volatile("st.relaxed.sys.global.v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(data), "r"(tag) : "memory");
}
PB_DEVICE uint64_t ld_relaxed_sys(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
// Wait until *p >= target. Returns false on watchdog expiry (caller records the error).
// The watchdog is wall-clock based (%globaltimer): a lost peer must never hang the GPU.
#ifndef PB_FLAG_TIMEOUT_NS
#define PB_FLAG_TIMEOUT_NS 20000000000ull  // 20 s
#endif
PB_DEVICE bool spin_wait_ge(const uint64_t* p, uint64_t target) {
  if (ld_acquire_sys(p) >= target) return true;
  const uint64_t t0 = globaltimer_ns();
  unsigned spins = 0;
  while (ld_acquire_sys(p) < target) {
    __nanosleep(32);
    if ((++spins & 0x3ff) == 0 && globaltimer_ns() - t0 > PB_FLAG_TIMEOUT_NS) return false;
  }
  return true;
}

// ---------------------------------------------------------------------------
// mbarrier
// ---------------------------------------------------------------------------
PB_DEVICE void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
PB_DEVICE void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
PB_DEVICE void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
PB_DEVICE void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
PB_DEVICE bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Spin on an mbarrier phase with a wall-clock watchdog; traps instead of hanging the GPU.
PB_DEVICE void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const uint64_t t0 = globaltimer_ns();
  unsigned spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0xff) == 0 && globaltimer_ns() - t0 > 10000000000ull) {  // 10 s
      printf("petals_b200: mbarrier watchdog expired (block %d thread %d)\n", blockIdx.x, threadIdx.x);
      __trap();
    }
  }
}

// ---------------------------------------------------------------------------
// TMA
// ---------------------------------------------------------------------------
PB_DEVICE void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
PB_DEVICE void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// 2-D tiled load: coordinates are (innermost = c0, outer = c1) in elements.
PB_DEVICE void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int32_t c0,
                           int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0),
      "r"(c1)
      : "memory");
}
// 2-D load with an L2 eviction-priority hint (createpolicy result).
PB_DEVICE void tma_load_2d_hint(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int32_t c0,
                                int32_t c1, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0),
      "r"(c1), "l"(policy)
      : "memory");
}
PB_DEVICE uint64_t policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
PB_DEVICE uint64_t policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
// 1-D bulk copy global → shared (no tensor map), completes on an mbarrier.
PB_DEVICE void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
      ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// ---------------------------------------------------------------------------
// tcgen05 / TMEM
// ---------------------------------------------------------------------------
PB_DEVICE void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_result)),
               "r"(ncols)
               : "memory");
}
PB_DEVICE void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
PB_DEVICE void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
PB_DEVICE void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
PB_DEVICE void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// tcgen05.commit: arrive on an mbarrier when all previously issued MMAs complete.
PB_DEVICE void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc], bf16/fp16 inputs, fp32 accumulate.
PB_DEVICE void tc_mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// fp8 (e4m3/e5m2) inputs, fp32 accumulate (non-block-scaled kind::f8f6f4).
PB_DEVICE void tc_mma_f8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                         uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}\n"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// TMEM → registers: 32 lanes × 32 columns of 32-bit (one warp reads its lane quarter).
PB_DEVICE void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
        "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
PB_DEVICE void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
PB_DEVICE void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor for a K-major bf16 tile stored with the TMA 128B swizzle:
// rows of 64 elements (128 B), 8-row core groups 1024 B apart (SBO), LBO unused (=1),
// descriptor version 1 (sm_100), layout type 2 (SWIZZLE_128B).
PB_DEVICE uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3ffffu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;               // leading byte offset (ignored for SW128 K-major)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;       // stride byte offset: 8 rows * 128 B
  d |= static_cast<uint64_t>(1) << 46;               // version = 1 (Blackwell)
  d |= static_cast<uint64_t>(2) << 61;               // SWIZZLE_128B
  return d;
}
// MN-major bf16 tile with 128B swizzle (TMA box = 64 contiguous MN elements × rows of the
// contraction dim): contraction-dim 8-row groups are 1024 B apart (SBO); successive 64-element
// MN blocks are `mn_block_bytes` apart (LBO).
PB_DEVICE uint64_t umma_desc_mn_sw128(uint32_t smem_addr, uint32_t mn_block_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3ffffu) >> 4);
  d |= static_cast<uint64_t>((mn_block_bytes >> 4) & 0x3fff) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// Instruction descriptor for kind::f16 with bf16 A/B, fp32 accumulate.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(uint32_t M, uint32_t N, uint32_t a_mn_major,
                                                       uint32_t b_mn_major) {
  return (1u << 4)                 // c_format = F32
         | (1u << 7)               // a_format = BF16
         | (1u << 10)              // b_format = BF16
         | (a_mn_major << 15)      // a_major
         | (b_mn_major << 16)      // b_major
         | ((N >> 3) << 17)        // n_dim
         | ((M >> 4) << 24);       // m_dim
}
// kind::f8f6f4 with e4m3 A/B, fp32 accumulate (K-major only).
__host__ __device__ constexpr uint32_t umma_idesc_e4m3(uint32_t M, uint32_t N) {
  return (1u << 4) | (0u << 7) | (0u << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

// ---- host: launch with (optional) programmatic dependent launch ------------------------------------------------------
// pb_pdl_enabled() reads PETALS_B200_PDL once (default on). Kernels launched through launch_pdl() MUST call pdl_wait()
// before reading anything an earlier kernel of the stream produced.
enum PdlKind : int { kPdlGemv = 1, kPdlRope = 2, kPdlAttn = 4, kPdlCombine = 8, kPdlGemvBigSmem = 16, kPdlGemvAuto = 32 };
inline int pdl_mask() {
  static const int mask = [] {
    const char* e = getenv("PETALS_B200_PDL");
    if (e != nullptr && e[0] == '0') return 0;
    const char* m = getenv("PETALS_B200_PDL_MASK");
    return m != nullptr ? atoi(m) : (kPdlRope | kPdlAttn | kPdlCombine);  // measured on B200: PDL on the weight-streaming GEMVs costs ~4 % (profiles/r1_pdl_sweep.txt)
  }();
  return mask;
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(int kind, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = (pdl_mask() & kind) ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

}  // namespace pb
