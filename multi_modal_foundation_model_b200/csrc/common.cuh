// Common device helpers for the sm_100a kernels: mbarrier, TMA (cp.async.bulk.tensor), tcgen05
// (TMEM alloc / mma / commit / ld), shared-memory matrix descriptors, Philox dropout stream.
// Everything here is inline PTX; no CUTLASS/CuTe is included.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace mmfm {

typedef __nv_bfloat16 bf16;

#define MMFM_DEVINL __device__ __forceinline__

// ------------------------------------------------------------------------------------------------
// misc
// ------------------------------------------------------------------------------------------------
MMFM_DEVINL uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

MMFM_DEVINL bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P1;\n\t.reg .b32 R1;\n\t"
      "elect.sync R1|P1, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P1;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}

// ------------------------------------------------------------------------------------------------
// programmatic dependent launch: every hot kernel starts with pdl_enter().  The trigger lets the NEXT kernel of the
// stream / graph be scheduled while this one is still running (its CTAs become resident as SMs drain and park at their
// own wait), the wait blocks until every prerequisite grid has completed and its writes are visible -- so kernel-to-
// kernel launch latency and the tail of a persistent grid overlap instead of adding up.  Without the launch attribute
// (host_util.h: launch_pdl; off unless MMFM_PDL=1 -- measured neutral on the default step) both instructions are no-ops.
// ------------------------------------------------------------------------------------------------
MMFM_DEVINL void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
MMFM_DEVINL void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
MMFM_DEVINL void pdl_enter() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
}

// ------------------------------------------------------------------------------------------------
// mbarrier
// ------------------------------------------------------------------------------------------------
MMFM_DEVINL void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
MMFM_DEVINL void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
MMFM_DEVINL void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

MMFM_DEVINL void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
MMFM_DEVINL void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// try_wait suspends the thread in hardware until the phase completes or a time limit expires.  The default limit is
// short: ncu's source page showed 11 % of all issued instructions of the attention forward in try_wait / branch polling
// loops, competing with the math warps of the same scheduler.  MMFM_MBAR_HINT_NS (compile-time, default 20 us) asks for
// a longer suspension; completion still wakes the thread at once.
#ifndef MMFM_MBAR_HINT_NS
#define MMFM_MBAR_HINT_NS 20000
#endif
// polls before a waiter gives up: with the suspend hint one poll lasts up to MMFM_MBAR_HINT_NS, so 2^17 polls are a few
// seconds (a protocol bug must not hold a GPU box for minutes)
#if MMFM_MBAR_HINT_NS > 0
#define MMFM_MBAR_SPIN_LIMIT (1u << 17)
#else
#define MMFM_MBAR_SPIN_LIMIT (1u << 26)
#endif
MMFM_DEVINL bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
#if MMFM_MBAR_HINT_NS > 0
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"((uint32_t)MMFM_MBAR_HINT_NS)
      : "memory");
#else
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
#endif
  return ok != 0;
}
// Bounded wait: a protocol bug traps (-> cudaErrorLaunchFailure) instead of hanging the box.  try_wait suspends the
// thread in hardware for a bounded time, so the loop polls rarely; the bound is an iteration count (no clock reads
// in the loop: a role warp that mostly waits must not steal issue slots from the math warps of its scheduler).
MMFM_DEVINL void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  uint32_t n = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++n > MMFM_MBAR_SPIN_LIMIT) {
      printf("mmfm: mbarrier wait timeout block(%d,%d,%d) thread %d parity %u bar %u\n", blockIdx.x, blockIdx.y,
             blockIdx.z, threadIdx.x, parity, smem_u32(bar));
      __trap();
    }
  }
}
// Same for role warps (TMA producer, MMA issuer) that wait for long stretches: back off between polls.
MMFM_DEVINL void mbar_wait_relaxed(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  uint32_t n = 0;
  while (!mbar_try_wait(bar, parity)) {
    __nanosleep(40);
    if (++n > MMFM_MBAR_SPIN_LIMIT) {
      printf("mmfm: mbarrier wait timeout block(%d,%d,%d) thread %d parity %u bar %u\n", blockIdx.x, blockIdx.y,
             blockIdx.z, threadIdx.x, parity, smem_u32(bar));
      __trap();
    }
  }
}

// ------------------------------------------------------------------------------------------------
// TMA
// ------------------------------------------------------------------------------------------------
MMFM_DEVINL void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}
MMFM_DEVINL void tma_load_2d_addr(uint32_t smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_dst), "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

// Tensor store: one box from shared memory (TMA layout, same swizzle as the map) to global memory; rows / columns
// outside the tensor are clipped.  Completion is tracked by the issuing thread's bulk async-group.
MMFM_DEVINL void tma_store_2d(const CUtensorMap* m, uint32_t smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(m), "r"(smem_src),
               "r"(c0), "r"(c1)
               : "memory");
}
MMFM_DEVINL void tma_store_3d(const CUtensorMap* m, uint32_t smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(m), "r"(smem_src),
               "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
MMFM_DEVINL void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// wait until the SOURCE (shared memory) of all but the newest N committed bulk groups has been read
template <int N>
MMFM_DEVINL void bulk_wait_group_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
MMFM_DEVINL void bulk_wait_group() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// Multicast load: the box lands at the same shared-memory offset of every CTA of the cluster whose rank bit is set in
// `mask`, and completes `bytes` on the mbarrier at the same offset in each of them.
MMFM_DEVINL void tma_load_2d_mc(uint32_t smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_dst), "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(mask)
      : "memory");
}
// tcgen05.commit that arrives on the mbarrier at this offset in every CTA of `mask`
MMFM_DEVINL void umma_commit_mc(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(mask)
               : "memory");
}
MMFM_DEVINL uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
MMFM_DEVINL void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// Pull one box of the tensor into L2 without touching shared memory: issued a tile or two ahead of the real load, it
// turns the ring's HBM latency into L2 latency, so the same bytes in flight sustain a multiple of the bandwidth.
MMFM_DEVINL void tma_prefetch_l2_2d(const CUtensorMap* m, int c0, int c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::"l"(m), "r"(c0), "r"(c1) : "memory");
}

// ------------------------------------------------------------------------------------------------
// tcgen05 / TMEM
// ------------------------------------------------------------------------------------------------
MMFM_DEVINL void tmem_alloc(uint32_t* smem_slot, uint32_t ncols) {  // whole warp, ncols pow2 >= 32
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)),
               "r"(ncols)
               : "memory");
}
MMFM_DEVINL void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
MMFM_DEVINL void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
MMFM_DEVINL void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
MMFM_DEVINL void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem], kind::f16 (bf16 inputs, fp32 accumulate); single thread issues.
MMFM_DEVINL void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Same with the A operand read from tensor memory (lane = row, one 32-bit column = two consecutive K elements).
MMFM_DEVINL void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Make the mbarrier track completion of all previously issued tcgen05.mma of this thread.
MMFM_DEVINL void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// 32 lanes x 32 columns of 32-bit: thread t of the warp gets lane (quadrant*32 + t), 32 consecutive columns.
MMFM_DEVINL void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]),
        "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]),
        "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
MMFM_DEVINL void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
MMFM_DEVINL void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// 32 lanes x 16 columns of 32-bit, registers -> tensor memory (thread t of the warp writes lane quadrant*32 + t)
MMFM_DEVINL void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
MMFM_DEVINL void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
MMFM_DEVINL void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------
// UMMA descriptors (bit layout: cute/arch/mma_sm100_desc.hpp -- SmemDescriptor / InstrDescriptor)
// ------------------------------------------------------------------------------------------------
// Shared-memory matrix descriptor.  addr/lbo/sbo in bytes (multiples of 16); layout: 0 none, 2 = 128B swizzle,
// 4 = 64B swizzle, 6 = 32B swizzle.  version (bits 46-47) = 1 on sm_100.
MMFM_DEVINL uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)(layout & 7) << 61;
  return d;
}
// Instruction descriptor for kind::f16 with bf16 A/B, fp32 D.  a_mn / b_mn: 1 = MN-major operand.
__host__ __device__ inline uint32_t make_idesc_bf16(uint32_t M, uint32_t N, uint32_t a_mn, uint32_t b_mn) {
  uint32_t d = 0;
  d |= 1u << 4;             // D format fp32
  d |= 1u << 7;             // A format bf16
  d |= 1u << 10;            // B format bf16
  d |= (a_mn & 1u) << 15;   // A major
  d |= (b_mn & 1u) << 16;   // B major
  d |= ((N >> 3) & 0x3F) << 17;
  d |= ((M >> 4) & 0x1F) << 24;
  return d;
}

// ------------------------------------------------------------------------------------------------
// Philox dropout stream (restated in oracle/philox_ref.py)
// ------------------------------------------------------------------------------------------------
constexpr int kPhiloxRounds = 7;

MMFM_DEVINL void mulhilo32(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {   // one IMAD.WIDE
  const unsigned long long p = (unsigned long long)a * (unsigned long long)b;
  hi = (uint32_t)(p >> 32);
  lo = (uint32_t)p;
}

MMFM_DEVINL uint4 philox4x32(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < kPhiloxRounds; ++r) {
    uint32_t hi0, lo0, hi1, lo1;
    mulhilo32(0xD2511F53u, c0, hi0, lo0);
    mulhilo32(0xCD9E8D57u, c2, hi1, lo1);
    const uint32_t n0 = hi1 ^ c1 ^ k0;
    const uint32_t n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}

// Four Philox blocks whose counters differ only in the low word c0 (c0, c0+1, c0+2, c0+3 -- the four quad-lane calls of
// one 64-key block) with ONE shared key schedule: 14 key additions per group instead of 56, and four independent
// dependency chains interleaved by construction.  Bit-identical to four philox4x32 calls.
MMFM_DEVINL void philox4x32_x4(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                               uint4 (&out)[4]) {
  uint32_t a0[4], a1[4], a2[4], a3[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) { a0[q] = c0 + q; a1[q] = c1; a2[q] = c2; a3[q] = c3; }
#pragma unroll
  for (int r = 0; r < kPhiloxRounds; ++r) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      uint32_t hi0, lo0, hi1, lo1;
      mulhilo32(0xD2511F53u, a0[q], hi0, lo0);
      mulhilo32(0xCD9E8D57u, a2[q], hi1, lo1);
      const uint32_t n0 = hi1 ^ a1[q] ^ k0;
      const uint32_t n2 = hi0 ^ a3[q] ^ k1;
      a0[q] = n0; a1[q] = lo1; a2[q] = n2; a3[q] = lo0;
    }
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) out[q] = make_uint4(a0[q], a1[q], a2[q], a3[q]);
}

struct DropCfg {
  const unsigned long long* seed;  // device scalar (graph-replay safe); nullptr => dropout off
  uint32_t site;
  uint32_t thresh;                 // drop iff byte < thresh; 0 => off
  float scale;                     // 256 / (256 - thresh)
};

// 16 random bytes for elements [16*g16, 16*g16+16) of row `row` in a (rows, cols) field.
MMFM_DEVINL uint4 drop_bytes16(unsigned long long seed, uint32_t site, uint64_t row, uint32_t groups_per_row,
                               uint32_t g16) {
  uint64_t g = row * (uint64_t)groups_per_row + g16;
  return philox4x32((uint32_t)g, (uint32_t)(g >> 32), site, 0u, (uint32_t)seed, (uint32_t)(seed >> 32));
}
MMFM_DEVINL uint32_t drop_byte(const uint4& w, int b) {  // b in [0,16)
  uint32_t word = (b < 4) ? w.x : (b < 8) ? w.y : (b < 12) ? w.z : w.w;
  return (word >> ((b & 3) * 8)) & 0xFFu;
}

// ------------------------------------------------------------------------------------------------
// small math
// ------------------------------------------------------------------------------------------------
// erf-GELU (transformers ACT2FN['gelu'], mm_utils.py:46) through Abramowitz-Stegun 7.1.26: |erf error| <= 1.5e-7,
// far below the bf16 rounding of the outputs, at roughly half the instructions of erff(); e = exp(-x^2/2) is shared
// with the derivative's Gaussian term.
MMFM_DEVINL float erf_poly(float z, float& e) {   // returns erf(z); e = exp(-z*z)
  const float az = fabsf(z);
  float t, ex;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, az, 1.0f)));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ex) : "f"(-1.4426950408889634f * z * z));
  e = ex;
  const float poly =
      fmaf(fmaf(fmaf(fmaf(1.061405429f, t, -1.453152027f), t, 1.421413741f), t, -0.284496736f), t, 0.254829592f) * t;
  return copysignf(fmaf(-poly, ex, 1.0f), z);
}
MMFM_DEVINL float gelu_erf(float x) {
  float e;
  return 0.5f * x * (1.0f + erf_poly(x * 0.70710678118654752f, e));
}
MMFM_DEVINL float gelu_erf_grad(float x) {
  float e;
  const float cdf = 0.5f * (1.0f + erf_poly(x * 0.70710678118654752f, e));
  return fmaf(x * 0.3989422804014327f, e, cdf);   // Phi(x) + x * phi(x), phi(x) = exp(-x^2/2) / sqrt(2 pi)
}
MMFM_DEVINL void gelu_erf_both(float x, float& g, float& dg) {   // gelu and its derivative from one erf / exp pair
  float e;
  const float cdf = 0.5f * (1.0f + erf_poly(x * 0.70710678118654752f, e));
  g = x * cdf;
  dg = fmaf(x * 0.3989422804014327f, e, cdf);
}
MMFM_DEVINL float softsign(float x) { return x / (1.0f + fabsf(x)); }

MMFM_DEVINL float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

MMFM_DEVINL uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
MMFM_DEVINL float2 unpack_bf16x2(uint32_t u) {
  __nv_bfloat162 v = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(v);
}


// packed fp32 pairs (FFMA2 / FMUL2 / FADD2: one issue slot for two lanes of work)
MMFM_DEVINL uint64_t pack_f2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
MMFM_DEVINL void unpack_f2(uint64_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
MMFM_DEVINL uint64_t ffma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
MMFM_DEVINL uint64_t fmul2(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
MMFM_DEVINL uint64_t fadd2(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}

// gelu and its derivative for a PAIR of arguments with packed fp32 arithmetic (FMUL2 / FFMA2): the same Abramowitz-Stegun
// evaluation as gelu_erf_both, half the issue slots for everything but the two MUFU ops per element.  The MLP-up epilogue
// of the TMA-store GEMM evaluates 26 M of these per launch and is bound by issue slots.
MMFM_DEVINL void gelu_erf_both2(float x0, float x1, float& g0, float& g1, float& d0, float& d1) {
  const uint64_t x = pack_f2(x0, x1);
  const uint64_t z = fmul2(x, pack_f2(0.70710678118654752f, 0.70710678118654752f));
  float z0, z1;
  unpack_f2(z, z0, z1);
  float t0, t1, e0, e1;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t0) : "f"(fmaf(0.3275911f, fabsf(z0), 1.0f)));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t1) : "f"(fmaf(0.3275911f, fabsf(z1), 1.0f)));
  float a0, a1;
  unpack_f2(fmul2(fmul2(z, z), pack_f2(-1.4426950408889634f, -1.4426950408889634f)), a0, a1);
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(a0));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(a1));
  const uint64_t t = pack_f2(t0, t1), e = pack_f2(e0, e1);
  uint64_t q = ffma2(pack_f2(1.061405429f, 1.061405429f), t, pack_f2(-1.453152027f, -1.453152027f));
  q = ffma2(q, t, pack_f2(1.421413741f, 1.421413741f));
  q = ffma2(q, t, pack_f2(-0.284496736f, -0.284496736f));
  q = ffma2(q, t, pack_f2(0.254829592f, 0.254829592f));
  q = fmul2(q, t);
  float r0, r1;
  unpack_f2(ffma2(q, fmul2(e, pack_f2(-1.0f, -1.0f)), pack_f2(1.0f, 1.0f)), r0, r1);   // 1 - poly * exp(-z^2) = erf(|z|)
  const uint64_t erf2 = pack_f2(copysignf(r0, z0), copysignf(r1, z1));
  const uint64_t cdf = ffma2(erf2, pack_f2(0.5f, 0.5f), pack_f2(0.5f, 0.5f));
  unpack_f2(fmul2(x, cdf), g0, g1);
  unpack_f2(ffma2(fmul2(x, pack_f2(0.3989422804014327f, 0.3989422804014327f)), e, cdf), d0, d1);
}

// ------------------------------------------------------------------------------------------------
// warp-level mma.sync path (attention core: d_head 32/64 tiles are softmax-bound, see DESIGN.md)
// ------------------------------------------------------------------------------------------------
MMFM_DEVINL void ldsm_x4(uint32_t (&r)[4], uint32_t saddr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(saddr));
}
MMFM_DEVINL void ldsm_x4_t(uint32_t (&r)[4], uint32_t saddr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(saddr));
}
// D(16x8, fp32) += A(16x16, bf16, row) * B(16x8, bf16, col)
MMFM_DEVINL void mma_16816(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

// D(16x8, fp32) = A * B (zero accumulator input: saves clearing the destination registers)
MMFM_DEVINL void mma_16816_z(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%10,%10,%10};"
      : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]), "f"(0.f));
}

MMFM_DEVINL float quad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  return v;
}
MMFM_DEVINL float quad_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
  return v;
}

// ------------------------------------------------------------------------------------------------
// Deterministic mode (torch.use_deterministic_algorithms): fixed-order fold of per-CTA partial vectors
// ------------------------------------------------------------------------------------------------
MMFM_DEVINL float det_add(float a, float b) { return a + b; }
MMFM_DEVINL double det_add(double a, double b) { return a + b; }
MMFM_DEVINL float4 det_add(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }

// Ticketed pairwise tree over the n_leaves partial vectors slot(i) = ws + i * stride (n elements of V each) of one
// reduction.  Every CTA of the reduction calls it with all its threads after writing slot(leaf) (and after pdl_wait).
// At level l node k covers slot k << l; the nodes 2j and 2j+1 meet at ticket ((2j+1) << l) - 1.  The CTA that arrives
// second adds the two slots into the left one and climbs; the first one exits; an unpaired last node climbs as it is.
// The CTA that completes the root pair calls emit(i, total_i) for i in [0, n) instead of storing it.  The tree's shape
// depends only on n_leaves and a + b == b + a in IEEE arithmetic, so the result does not depend on which CTA arrives
// last, and no CTA ever waits for another.  The second arrival clears its ticket: a launch leaves its n_leaves - 1
// tickets at zero for the next one (graph replays need no memset).
template <typename V, typename Emit>
MMFM_DEVINL void det_tree_fold(V* ws, long long stride, int n, int leaf, int n_leaves, unsigned int* tickets,
                               Emit emit) {
  __shared__ unsigned int s_second;
  int node = leaf;
  for (int l = 0; (1 << l) < n_leaves; ++l) {
    const int width = (n_leaves + (1 << l) - 1) >> l;
    if ((node | 1) >= width) { node >>= 1; continue; }
    const int right = (node | 1) << l;
    __syncthreads();   // this CTA's writes to its slot are done ...
    if (threadIdx.x == 0) {
      __threadfence();   // ... and visible device-wide before the ticket
      const unsigned int t = atomicAdd(tickets + right - 1, 1u);
      if (t != 0u) {
        tickets[right - 1] = 0u;
        __threadfence();   // the partner's slot writes (fenced before its ticket) are visible to this CTA
      }
      s_second = t;
    }
    __syncthreads();
    if (s_second == 0u) return;
    V* a = ws + (long long)((node & ~1) << l) * stride;
    const V* b = ws + (long long)right * stride;
    // kU elements per thread in flight: one CTA moves the whole pair, so the level time is L2 latency-bound otherwise
    constexpr int kU = 8;
    for (int i0 = threadIdx.x; i0 < n; i0 += kU * blockDim.x) {
      V va[kU], vb[kU];
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        const int i = i0 + u * blockDim.x;
        if (i < n) { va[u] = __ldcg(a + i); vb[u] = __ldcg(b + i); }
      }
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        const int i = i0 + u * blockDim.x;
        if (i >= n) break;
        if (width == 2) emit(i, det_add(va[u], vb[u]));
        else a[i] = det_add(va[u], vb[u]);
      }
    }
    if (width == 2) return;
    node >>= 1;
  }
  __syncthreads();   // n_leaves == 1: the total is this CTA's own slot
  for (int i = threadIdx.x; i < n; i += blockDim.x) emit(i, __ldcg(ws + (long long)leaf * stride + i));
}

// one random byte for element (row, col) of a (rows, cols) dropout field (slow path; hot loops fetch 16 at once)
MMFM_DEVINL uint32_t drop_byte_at(unsigned long long seed, uint32_t site, uint64_t row, uint32_t groups_per_row,
                                  uint32_t col) {
  uint4 w = drop_bytes16(seed, site, row, groups_per_row, col >> 4);
  return drop_byte(w, col & 15);
}

}  // namespace mmfm
