// tcgen05 / TMEM / TMA GEMM kernels of the multi-modal encoder/decoder path.
//
//   gemm_tn_kernel    D[M,N] = epilogue(A[M,K] . B[N,K]^T)     both operands K-major (nn.Linear forward + dgrad)
//   gemm_wgrad_kernel dW[NO,KI] += dY[R,NO]^T . X[R,KI]        both operands MN-major, split over R (wgrad)
//
// Replaces the cuBLAS calls under every nn.Linear of the reference path (SURVEY.md 2.2 K1,K3,K10,K12,K14-K17 and
// their autograd backward, K21).  One CTA computes one 128 x BN output tile:
//   warp 0   : TMA producer (one elected lane), STAGES-deep mbarrier ring of 128B-swizzled smem tiles
//   warp 1   : TMEM allocation + tcgen05.mma issue (one elected lane), fp32 accumulator in TMEM
//   warps 2-5: epilogue -- tcgen05.ld of their TMEM lane quadrant, fused bias / activation / dropout /
//              token-zeroing / residual, direct vectorised global stores
// Several CTAs are resident per SM (smem- and TMEM-limited), so one CTA's epilogue overlaps another's main loop.
#include "common.cuh"
#include <stdlib.h>
#include "host_util.h"
#include "../../include/mmfm_b200.h"

namespace mmfm {

constexpr int kBM = 128;
constexpr int kBK = 64;
constexpr int kGemmThreads = 192;

// ------------------------------------------------------------------------------------------------
// Epilogue, two phases per epilogue warp (each warp owns the 32 accumulator rows of its TMEM lane quadrant):
//   A  thread = row : tcgen05.ld 32 columns at a time, + bias (smem broadcast), dropout (the thread holds whole
//      16-column Philox groups of its row), token zeroing -> fp32 staging tile in shared memory (the drained
//      pipeline stages are reused)
//   B  lane = 4 consecutive columns, one row (BN = 128) or two rows (BN = 64) per step: activation / saved-tensor
//      derivative, residual add, 16-byte coalesced global loads and stores (a warp touches one contiguous 512-byte
//      row segment per instruction instead of 32 rows x 16 bytes)
// Only __syncwarp separates the phases: a warp re-reads exactly the rows it staged.
// ------------------------------------------------------------------------------------------------
MMFM_DEVINL float4 ld4_f32(const float* p, bool vec, int nvalid) {
  if (vec) return __ldg(reinterpret_cast<const float4*>(p));
  float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
  if (nvalid > 0) r.x = __ldg(p);
  if (nvalid > 1) r.y = __ldg(p + 1);
  if (nvalid > 2) r.z = __ldg(p + 2);
  if (nvalid > 3) r.w = __ldg(p + 3);
  return r;
}
MMFM_DEVINL float4 ld4_bf16(const bf16* p, bool vec, int nvalid) {
  if (vec) {
    const uint2 u = __ldg(reinterpret_cast<const uint2*>(p));
    const float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y);
    return make_float4(a.x, a.y, b.x, b.y);
  }
  float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
  if (nvalid > 0) r.x = __bfloat162float(p[0]);
  if (nvalid > 1) r.y = __bfloat162float(p[1]);
  if (nvalid > 2) r.z = __bfloat162float(p[2]);
  if (nvalid > 3) r.w = __bfloat162float(p[3]);
  return r;
}
MMFM_DEVINL void st4_f32(float* p, bool vec, int nvalid, const float4& v) {
  if (vec) { *reinterpret_cast<float4*>(p) = v; return; }
  if (nvalid > 0) p[0] = v.x;
  if (nvalid > 1) p[1] = v.y;
  if (nvalid > 2) p[2] = v.z;
  if (nvalid > 3) p[3] = v.w;
}
MMFM_DEVINL void st4_bf16(bf16* p, bool vec, int nvalid, const float4& v) {
  if (vec) { *reinterpret_cast<uint2*>(p) = make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w)); return; }
  if (nvalid > 0) p[0] = __float2bfloat16_rn(v.x);
  if (nvalid > 1) p[1] = __float2bfloat16_rn(v.y);
  if (nvalid > 2) p[2] = __float2bfloat16_rn(v.z);
  if (nvalid > 3) p[3] = __float2bfloat16_rn(v.w);
}

// ------------------------------------------------------------------------------------------------
// TN kernel.  Warp roles: 0 = TMA producer, 1 = TMEM allocator + MMA issuer, 2..9 = epilogue (two warps per TMEM
// lane quadrant, each taking one half of the tile's columns).  The epilogue flavour is a template parameter so the
// per-element code is branch-free; EPI_GENERIC keeps every run-time option (unaligned pitches, odd N).
// ------------------------------------------------------------------------------------------------
constexpr int kEpiWarps = 16;   // four warps per TMEM lane quadrant, each taking a quarter of the tile's columns
constexpr int kTnThreads = 64 + kEpiWarps * 32;

enum EpiKind : int {
  EPI_PLAIN_BF16 = 0,   // D(bf16) = v
  EPI_PLAIN_F32 = 1,    // D(f32) = v
  EPI_RES_F32 = 2,      // D(f32) = v + res                       (dropout / token zeroing / remap allowed)
  EPI_GELU = 3,         // D2(bf16) = v ; D(bf16) = gelu(v)
  EPI_SOFTSIGN = 4,     // D(bf16) = softsign(v) * s
  EPI_DGELU = 5,        // D(bf16) = v * gelu'(aux)
  EPI_DSOFTSIGN = 6,    // D(bf16) = v * s * (1 - |aux/s|)^2
  EPI_GENERIC = 7,
  EPI_GELU_DG = 8,      // D2(bf16) = gelu'(v) ; D(bf16) = gelu(v)
  EPI_MULAUX = 9        // D(bf16) = v * aux
};

// Persistent: one CTA per SM walks the tile list (n fastest, so concurrently running CTAs share A rows in L2).  The
// TMA producer runs ahead across tile boundaries through a STAGES-deep ring; the accumulator is double-buffered in
// TMEM (2 x BN columns) so the MMA of tile i+1 overlaps the epilogue of tile i; the epilogue stages through its own
// shared-memory tile.
template <int BN, int STAGES, int EPI>
__global__ void __launch_bounds__(kTnThreads, 1) gemm_tn_kernel(const __grid_constant__ CUtensorMap tmA,
                                                                 const __grid_constant__ CUtensorMap tmB,
                                                                 const mmfm_gemm_args p, int tiles_n, int n_tiles,
                                                                 int bstat) {
  constexpr uint32_t kABytes = kBM * kBK * 2;  // 16 KB
  constexpr uint32_t kBBytes = BN * kBK * 2;
  constexpr uint32_t kStageBytes = kABytes + kBBytes;
  constexpr uint32_t kTmemCols = 2 * BN;  // 256 or 128: power of two
  constexpr int kPitch = BN + 4;  // fp32 staging pitch (floats): 16-byte rows, conflict-free in both phases
  constexpr int kHalf = BN / (kEpiWarps / 4);   // columns per epilogue warp
  constexpr bool GEN = EPI == EPI_GENERIC;

  // Weight-stationary mode (bstat): the grid is a multiple of tiles_n, so every tile of this CTA has the same column
  // block; its whole K extent of B (<= half of the ring area) is loaded ONCE and stays resident, the ring carries A
  // k-blocks only.  These skinny-K GEMMs are bound by L2 -> SM traffic, which this halves.
  constexpr int kMaxStages = 8;
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[kMaxStages];
  __shared__ __align__(8) uint64_t empty_bar[kMaxStages];
  __shared__ __align__(8) uint64_t b_full;
  __shared__ __align__(8) uint64_t acc_full[2];
  __shared__ __align__(8) uint64_t acc_empty[2];
  __shared__ uint32_t tmem_slot;
  __shared__ __align__(16) float s_bias[kEpiWarps][kHalf];

  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  float* stage_f = reinterpret_cast<float*>(smem_raw + (smem_base - smem_u32(smem_raw)) + STAGES * kStageBytes);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int nkb = (p.K + kBK - 1) / kBK;
  const uint32_t b_res_bytes = bstat ? (uint32_t)nkb * kBBytes : 0u;
  const uint32_t ring_base = smem_base + b_res_bytes;
  const uint32_t st_bytes = bstat ? kABytes : kStageBytes;
  uint32_t nst = bstat ? (STAGES * kStageBytes - b_res_bytes) / kABytes : (uint32_t)STAGES;
  if (nst > (uint32_t)kMaxStages) nst = kMaxStages;

  pdl_trigger();
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
#pragma unroll
    for (int s = 0; s < kMaxStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(&b_full, 1);
    mbar_init(&acc_full[0], 1);
    mbar_init(&acc_full[1], 1);
    mbar_init(&acc_empty[0], kEpiWarps);
    mbar_init(&acc_empty[1], kEpiWarps);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(&tmem_slot, kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;
  pdl_wait();

  if (warp == 0) {
    if (elect_one()) {
      uint32_t it = 0;
      if (bstat) {
        const int n0 = ((int)blockIdx.x % tiles_n) * BN;
        mbar_arrive_expect_tx(&b_full, b_res_bytes);
        for (int kb = 0; kb < nkb; ++kb) tma_load_2d_addr(smem_base + kb * kBBytes, &tmB, &b_full, kb * kBK, n0);
      }
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int m0 = (tile / tiles_n) * kBM, n0 = (tile % tiles_n) * BN;
        // L2 prefetch of the activation rows this CTA needs two tiles from now (the ring itself holds about one
        // tile); the CTA that owns the first column tile of that row block fetches for all its neighbours
        {
          const int t2 = tile + 2 * (int)gridDim.x;
          if (t2 < n_tiles && (t2 % tiles_n == 0 || tiles_n > (int)gridDim.x)) {
            const int m2 = (t2 / tiles_n) * kBM;
            for (int kb = 0; kb < nkb; ++kb) tma_prefetch_l2_2d(&tmA, kb * kBK, m2);
          }
        }
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const uint32_t s = it % nst;
          if (it >= nst) mbar_wait(&empty_bar[s], ((it / nst) - 1) & 1);
          mbar_arrive_expect_tx(&full_bar[s], st_bytes);
          const uint32_t a_dst = ring_base + s * st_bytes;
          tma_load_2d_addr(a_dst, &tmA, &full_bar[s], kb * kBK, m0);
          if (!bstat) tma_load_2d_addr(a_dst + kABytes, &tmB, &full_bar[s], kb * kBK, n0);
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      const uint32_t idesc = make_idesc_bf16(kBM, BN, 0, 0);
      uint32_t it = 0, t = 0;
      if (bstat) mbar_wait(&b_full, 0);
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++t) {
        const uint32_t buf = t & 1u;
        if (t >= 2) mbar_wait(&acc_empty[buf], ((t >> 1) - 1) & 1);   // epilogue drained this TMEM buffer
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + buf * BN;
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const uint32_t s = it % nst;
          mbar_wait(&full_bar[s], (it / nst) & 1);
          tc_fence_after();
          const uint32_t a_addr = ring_base + s * st_bytes;
          const uint32_t b_addr = bstat ? smem_base + kb * kBBytes : a_addr + kABytes;
#pragma unroll
          for (int k = 0; k < kBK / 16; ++k) {
            const uint64_t da = make_smem_desc(a_addr + k * 32, 16, 1024, 2);
            const uint64_t db = make_smem_desc(b_addr + k * 32, 16, 1024, 2);
            umma_bf16(d_tmem, da, db, idesc, (kb > 0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&empty_bar[s]);
        }
        umma_commit(&acc_full[buf]);
      }
    }
  } else {
    // ---------------- epilogue warps: TMEM lane quadrant = warp % 4, column slice = (warp - 2) / 4 ----------
    const int ew = warp - 2;
    const int quad = warp & 3;
    const int half = ew >> 2;
    const int cbase = half * kHalf;
    const int row_l = quad * 32 + lane;            // tile row of this thread (phase A)
    constexpr bool kMayDrop = GEN || EPI == EPI_RES_F32;
    constexpr bool kHasRes = GEN || EPI == EPI_RES_F32;
    constexpr bool kHasAux = GEN || EPI == EPI_DGELU || EPI == EPI_DSOFTSIGN || EPI == EPI_MULAUX;
    bool drop = false;
    unsigned long long seed = 0ull;
    if (kMayDrop) {
      drop = p.drop.thresh != 0u;
      if (drop) seed = *p.drop.seed;
    }
    const uint32_t drop_gpr = (uint32_t)((p.N + 15) >> 4);
    const int act = GEN ? p.act : 0;
    const bool f32out = GEN ? (p.d_fp32 != 0) : (EPI == EPI_PLAIN_F32 || EPI == EPI_RES_F32);
    const float inv_scale = 1.0f / p.act_scale;
    const bool has_res = GEN ? (p.res != nullptr) : (EPI == EPI_RES_F32);
    const bool has_aux = GEN ? (act == MMFM_ACT_DGELU || act == MMFM_ACT_DSOFTSIGN || act == MMFM_ACT_MULAUX) : kHasAux;
    float* my_bias = s_bias[ew];
    static_assert(kHalf <= 64, "bias slice: at most two values per lane");
    // bias slice of this warp's columns, fetched one tile ahead so its latency is never exposed
    auto load_bias = [&](int tile_i, float (&b)[2]) {
      b[0] = b[1] = 0.f;
      if (tile_i < n_tiles && p.bias) {
        const int nn = (tile_i % tiles_n) * BN + cbase;
        if (lane < kHalf && nn + lane < p.N) b[0] = __ldg(p.bias + nn + lane);
        if (lane + 32 < kHalf && nn + lane + 32 < p.N) b[1] = __ldg(p.bias + nn + lane + 32);
      }
    };
    float bias_next[2];
    load_bias(blockIdx.x, bias_next);

    uint32_t t = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++t) {
      const uint32_t buf = t & 1u;
      const int m0 = (tile / tiles_n) * kBM, n0 = (tile % tiles_n) * BN;
      const long long r = (long long)m0 + row_l;     // GEMM row of this thread in phase A
      const bool warp_has_cols = (n0 + cbase) < p.N;
      if (lane < kHalf) my_bias[lane] = bias_next[0];
      if (lane + 32 < kHalf) my_bias[lane + 32] = bias_next[1];
      load_bias(tile + gridDim.x, bias_next);
      bool zero = false;
      if (kMayDrop && p.row_zero && r < p.M) {
        const int pos = p.remap_T > 0 ? p.remap_off + (int)(r % p.remap_T) : (int)(r % p.remap_S);
        zero = p.row_zero[pos] != 0;
      }
      // while the main loop runs: pull this thread's residual / saved-tensor row segment into L2
      if (r < p.M && warp_has_cols) {
        const int ncols = min(kHalf, p.N - n0 - cbase);
        if (kHasRes && p.res) {
          long long orow = r;
          if (p.remap_T > 0) {
            const int bb = (int)r / p.remap_T;
            orow = (long long)bb * p.remap_S + p.remap_off + ((int)r - bb * p.remap_T);
          }
          const char* ptr = reinterpret_cast<const char*>(p.res + orow * p.ldr + n0 + cbase);
          for (int o = 0; o < ncols * 4; o += 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr + o));
        }
        if (kHasAux && p.aux) {
          const char* ptr =
              reinterpret_cast<const char*>(reinterpret_cast<const bf16*>(p.aux) + r * p.ldaux + n0 + cbase);
          for (int o = 0; o < ncols * 2; o += 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr + o));
        }
      }
      __syncwarp();
      mbar_wait(&acc_full[buf], (t >> 1) & 1);
      tc_fence_after();
      // Interior tiles of the two commonest flavours take a straight-line path: no edge / alignment / remap tests, bf16
      // staging for bf16 outputs, 16-byte global accesses (these GEMMs are bound by epilogue instruction issue).
      const bool interior = (m0 + kBM <= p.M) && (n0 + BN <= p.N);
      if ((EPI == EPI_PLAIN_BF16 || EPI == EPI_RES_F32) && interior && p.remap_T == 0 && kHalf == 32) {
        const uint32_t t_row = tmem_base + buf * BN + ((uint32_t)(quad * 32) << 16) + (uint32_t)cbase;
        if (EPI == EPI_PLAIN_BF16) {
          // bf16 staging (half the shared-memory traffic of the fp32 tile; row-strided 16-byte global stores straight
          // from registers were measured 35 % slower than this staged, row-contiguous form)
          constexpr int kPitchH = BN + 8;   // bf16 staging pitch (elements): 16 bytes mod 128 -> phase A conflict-free
          bf16* stage_h = reinterpret_cast<bf16*>(stage_f);
          bf16* my_row_h = stage_h + row_l * kPitchH + cbase;
#pragma unroll
          for (int c0 = 0; c0 < 32; c0 += 16) {
            uint32_t acc[16];
            tmem_ld16(t_row + (uint32_t)c0, acc);
            tmem_ld_wait();
            uint32_t h[8];
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4) {
              const float4 b4 = *reinterpret_cast<const float4*>(&my_bias[c0 + j4 * 4]);
              h[2 * j4] = pack_bf16x2(__uint_as_float(acc[4 * j4]) + b4.x, __uint_as_float(acc[4 * j4 + 1]) + b4.y);
              h[2 * j4 + 1] = pack_bf16x2(__uint_as_float(acc[4 * j4 + 2]) + b4.z, __uint_as_float(acc[4 * j4 + 3]) + b4.w);
            }
            *reinterpret_cast<uint4*>(my_row_h + c0) = make_uint4(h[0], h[1], h[2], h[3]);
            *reinterpret_cast<uint4*>(my_row_h + c0 + 8) = make_uint4(h[4], h[5], h[6], h[7]);
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&acc_empty[buf]);
          // phase B: 4 lanes x 16 bytes per row, 8 rows per step; the two rows of a quarter-warp are 4 apart (64 bytes
          // mod 128 in the staging tile: no bank conflicts)
          const int lr = (lane >> 3) + 4 * ((lane >> 2) & 1), lc = (lane & 3) * 8;
          bf16* dst = reinterpret_cast<bf16*>(p.D) + ((long long)m0 + quad * 32 + lr) * p.ldd + n0 + cbase + lc;
          const bf16* src = stage_h + (quad * 32 + lr) * kPitchH + cbase + lc;
#pragma unroll
          for (int st8 = 0; st8 < 4; ++st8)
            *reinterpret_cast<uint4*>(dst + (long long)st8 * 8 * p.ldd) = *reinterpret_cast<const uint4*>(src + st8 * 8 * kPitchH);
        } else {
          float* my_row = stage_f + row_l * kPitch + cbase;
#pragma unroll
          for (int c0 = 0; c0 < 32; c0 += 16) {
            uint32_t acc[16];
            tmem_ld16(t_row + (uint32_t)c0, acc);
            tmem_ld_wait();
            float v[16];
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4) {
              const float4 b4 = *reinterpret_cast<const float4*>(&my_bias[c0 + j4 * 4]);
              v[4 * j4 + 0] = __uint_as_float(acc[4 * j4 + 0]) + b4.x;
              v[4 * j4 + 1] = __uint_as_float(acc[4 * j4 + 1]) + b4.y;
              v[4 * j4 + 2] = __uint_as_float(acc[4 * j4 + 2]) + b4.z;
              v[4 * j4 + 3] = __uint_as_float(acc[4 * j4 + 3]) + b4.w;
            }
            if (drop) {
              const uint4 w = drop_bytes16(seed, p.drop.site, (uint64_t)r, drop_gpr, (uint32_t)((n0 + cbase + c0) >> 4));
#pragma unroll
              for (int j = 0; j < 16; ++j) v[j] = (drop_byte(w, j) < p.drop.thresh) ? 0.f : v[j] * p.drop.scale;
            }
            if (zero) {
#pragma unroll
              for (int j = 0; j < 16; ++j) v[j] = 0.f;
            }
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4)
              *reinterpret_cast<float4*>(my_row + c0 + j4 * 4) =
                  make_float4(v[4 * j4], v[4 * j4 + 1], v[4 * j4 + 2], v[4 * j4 + 3]);
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&acc_empty[buf]);
          // phase B: 8 lanes x 16 bytes per row, 4 rows per step; the residual rows of all steps are requested first
          const int lr = lane >> 3, lc = (lane & 7) * 4;
          const long long grow = (long long)m0 + quad * 32 + lr;
          const float* rsrc = p.res + grow * p.ldr + n0 + cbase + lc;
          float* dst = reinterpret_cast<float*>(p.D) + grow * p.ldd + n0 + cbase + lc;
          const float* src = stage_f + (quad * 32 + lr) * kPitch + cbase + lc;
          float4 rv[8];
#pragma unroll
          for (int s8 = 0; s8 < 8; ++s8) rv[s8] = __ldg(reinterpret_cast<const float4*>(rsrc + (long long)s8 * 4 * p.ldr));
#pragma unroll
          for (int s8 = 0; s8 < 8; ++s8) {
            const float4 v = *reinterpret_cast<const float4*>(src + s8 * 4 * kPitch);
            *reinterpret_cast<float4*>(dst + (long long)s8 * 4 * p.ldd) =
                make_float4(v.x + rv[s8].x, v.y + rv[s8].y, v.z + rv[s8].z, v.w + rv[s8].w);
          }
        }
        __syncwarp();   // staging rows are re-written by this warp's next tile
        continue;
      }
      if (warp_has_cols) {
        const uint32_t t_row = tmem_base + buf * BN + ((uint32_t)(quad * 32) << 16) + (uint32_t)cbase;
        float* my_row = stage_f + row_l * kPitch + cbase;
        // ---------------- phase A: thread = row ----------------
#pragma unroll
        for (int c0 = 0; c0 < kHalf; c0 += 16) {
          uint32_t acc[16];
          tmem_ld16(t_row + (uint32_t)c0, acc);
          tmem_ld_wait();
          float v[16];
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4) {
            const float4 b4 = *reinterpret_cast<const float4*>(&my_bias[c0 + j4 * 4]);
            v[4 * j4 + 0] = __uint_as_float(acc[4 * j4 + 0]) + b4.x;
            v[4 * j4 + 1] = __uint_as_float(acc[4 * j4 + 1]) + b4.y;
            v[4 * j4 + 2] = __uint_as_float(acc[4 * j4 + 2]) + b4.z;
            v[4 * j4 + 3] = __uint_as_float(acc[4 * j4 + 3]) + b4.w;
          }
          if (kMayDrop) {
            if (drop) {
              const uint4 w = drop_bytes16(seed, p.drop.site, (uint64_t)r, drop_gpr, (uint32_t)((n0 + cbase + c0) >> 4));
#pragma unroll
              for (int j = 0; j < 16; ++j) v[j] = (drop_byte(w, j) < p.drop.thresh) ? 0.f : v[j] * p.drop.scale;
            }
            if (zero) {
#pragma unroll
              for (int j = 0; j < 16; ++j) v[j] = 0.f;
            }
          }
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4)
            *reinterpret_cast<float4*>(my_row + c0 + j4 * 4) =
                make_float4(v[4 * j4], v[4 * j4 + 1], v[4 * j4 + 2], v[4 * j4 + 3]);
        }
      }
      // this warp is done with the TMEM buffer: hand it back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[buf]);
      if (warp_has_cols) {
        // ---------------- phase B: lane = 4 consecutive columns; coalesced global traffic ----------------
        constexpr int kLanesPerRow = kHalf / 4;          // 8 (BN 128) or 4 (BN 64)
        constexpr int kRowsPerStep = 32 / kLanesPerRow;  // 4 or 8
        constexpr int kSteps = 32 / kRowsPerStep;        // 8 or 4
        constexpr int kBatch = kSteps < 8 ? kSteps : 8;  // steps whose global loads are issued together
        const int lcol = cbase + (lane % kLanesPerRow) * 4;
        const int n = n0 + lcol;
        const int nvalid = p.N - n;
        const int lrow = lane / kLanesPerRow;
        // the specialised kernels are only launched when every pointer / pitch is vector-aligned and N % 4 == 0
        const bool vec_d = GEN ? ((p.ldd % 4 == 0) && nvalid >= 4 && ((reinterpret_cast<uintptr_t>(p.D) & (p.d_fp32 ? 15 : 7)) == 0)) : true;
        const bool vec_d2 = GEN ? (p.D2 && (p.ldd % 4 == 0) && nvalid >= 4 && ((reinterpret_cast<uintptr_t>(p.D2) & 7) == 0)) : true;
        const bool vec_r = GEN ? (p.res && (p.ldr % 4 == 0) && nvalid >= 4 && ((reinterpret_cast<uintptr_t>(p.res) & 15) == 0)) : true;
        const bool vec_a = GEN ? (p.aux && (p.ldaux % 4 == 0) && nvalid >= 4 && ((reinterpret_cast<uintptr_t>(p.aux) & 7) == 0)) : true;
        if (nvalid > 0) {
#pragma unroll 1
          for (int it0 = 0; it0 < kSteps; it0 += kBatch) {
            float4 rv[kBatch], av[kBatch];
            long long orow[kBatch];
#pragma unroll
            for (int u = 0; u < kBatch; ++u) {
              const int rl = quad * 32 + (it0 + u) * kRowsPerStep + lrow;
              const long long rr = (long long)m0 + rl;
              orow[u] = rr;
              if (kMayDrop && p.remap_T > 0) {
                const int bb = (int)rr / p.remap_T;
                orow[u] = (long long)bb * p.remap_S + p.remap_off + ((int)rr - bb * p.remap_T);
              }
              if (rr >= p.M) orow[u] = -1;
              rv[u] = make_float4(0.f, 0.f, 0.f, 0.f);
              av[u] = rv[u];
              if (orow[u] >= 0) {
                if (has_res) rv[u] = ld4_f32(p.res + orow[u] * p.ldr + n, vec_r, nvalid);
                if (has_aux) av[u] = ld4_bf16(reinterpret_cast<const bf16*>(p.aux) + rr * p.ldaux + n, vec_a, nvalid);
              }
            }
#pragma unroll
            for (int u = 0; u < kBatch; ++u) {
              if (orow[u] < 0) continue;
              const int rl = quad * 32 + (it0 + u) * kRowsPerStep + lrow;
              float4 v = *reinterpret_cast<const float4*>(stage_f + rl * kPitch + lcol);
              if (EPI == EPI_GELU || (GEN && act == MMFM_ACT_GELU)) {
                if (!GEN || p.D2) st4_bf16(reinterpret_cast<bf16*>(p.D2) + orow[u] * p.ldd + n, vec_d2, nvalid, v);
                v.x = gelu_erf(v.x); v.y = gelu_erf(v.y); v.z = gelu_erf(v.z); v.w = gelu_erf(v.w);
              } else if (EPI == EPI_GELU_DG || (GEN && act == MMFM_ACT_GELU_DG)) {
                float4 dg;
                gelu_erf_both(v.x, v.x, dg.x); gelu_erf_both(v.y, v.y, dg.y);
                gelu_erf_both(v.z, v.z, dg.z); gelu_erf_both(v.w, v.w, dg.w);
                if (!GEN || p.D2) st4_bf16(reinterpret_cast<bf16*>(p.D2) + orow[u] * p.ldd + n, vec_d2, nvalid, dg);
              } else if (EPI == EPI_MULAUX || (GEN && act == MMFM_ACT_MULAUX)) {
                const float4 a = av[u];
                v.x *= a.x; v.y *= a.y; v.z *= a.z; v.w *= a.w;
              } else if (EPI == EPI_SOFTSIGN || (GEN && act == MMFM_ACT_SOFTSIGN)) {
                v.x = softsign(v.x) * p.act_scale; v.y = softsign(v.y) * p.act_scale;
                v.z = softsign(v.z) * p.act_scale; v.w = softsign(v.w) * p.act_scale;
              } else if (EPI == EPI_DGELU || (GEN && act == MMFM_ACT_DGELU)) {
                const float4 a = av[u];
                v.x *= gelu_erf_grad(a.x); v.y *= gelu_erf_grad(a.y); v.z *= gelu_erf_grad(a.z); v.w *= gelu_erf_grad(a.w);
              } else if (EPI == EPI_DSOFTSIGN || (GEN && act == MMFM_ACT_DSOFTSIGN)) {
                const float4 a = av[u];
                float tt;
                tt = 1.0f - fabsf(a.x * inv_scale); v.x *= p.act_scale * tt * tt;
                tt = 1.0f - fabsf(a.y * inv_scale); v.y *= p.act_scale * tt * tt;
                tt = 1.0f - fabsf(a.z * inv_scale); v.z *= p.act_scale * tt * tt;
                tt = 1.0f - fabsf(a.w * inv_scale); v.w *= p.act_scale * tt * tt;
              }
              if (has_res) { v.x += rv[u].x; v.y += rv[u].y; v.z += rv[u].z; v.w += rv[u].w; }
              if (f32out) st4_f32(reinterpret_cast<float*>(p.D) + orow[u] * p.ldd + n, vec_d, nvalid, v);
              else st4_bf16(reinterpret_cast<bf16*>(p.D) + orow[u] * p.ldd + n, vec_d, nvalid, v);
            }
          }
        }
      }
      __syncwarp();   // phase B reads of the staging rows are done before the next tile's phase A overwrites them
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, kTmemCols);
}

// ------------------------------------------------------------------------------------------------
// wgrad kernel: dW[NO,KI] += sum over a slice of rows of dY[r,NO]^T X[r,KI];  optionally db[NO] += colsum(dY)
// (the bias gradient rides on the tensor pipe: one extra N=16 MMA per k-step against a tile of ones)
// ------------------------------------------------------------------------------------------------
// BN = 256 (KI % 256 == 0): one CTA per SM owns a 128 x 256 tile of dW.  As in gemm_ts.cu the main loop is bound by
// shared-memory bandwidth (every operand byte is written once by TMA and read once by the tensor core; a 128 x 128 x 16
// MMA alone reads 128 B/clk), and the wider tile moves 25 % fewer bytes per FLOP and reads every dY box once instead of
// once per 128-column tile.
// DET (deterministic mode, no clusters): instead of red.global, each split CTA writes its fp32 tile and bias column to
// its workspace slot [tile][split] and the splits of a tile are folded by det_tree_fold (common.cuh) into dW / dbias.
template <int BN>
__host__ __device__ constexpr long long wgrad_slot_f4() { return ((long long)kBM * BN + kBM) / 4; }   // float4s per workspace slot

template <int STAGES, int BN, bool DET = false>
__global__ void __launch_bounds__(kGemmThreads) gemm_wgrad_kernel(const __grid_constant__ CUtensorMap tmY,
                                                                   const __grid_constant__ CUtensorMap tmX, int R,
                                                                   int NO, int KI, float* __restrict__ dW,
                                                                   long long ldw, int rows_per_split,
                                                                   float* __restrict__ dbias, int cx, int cy,
                                                                   float4* __restrict__ ws, unsigned int* tickets) {
  // (cx, cy) = thread-block cluster shape over (KI tiles, NO tiles), 1 or 2 each.  The CTAs of a cluster work on the
  // same rows: the two KI tiles of a cluster row share their dY boxes, the two NO tiles of a cluster column share their
  // X boxes, so each CTA loads HALF of what it consumes and TMA-multicasts it to its peer (this kernel is bound by
  // L2 -> SM traffic: every dY box is needed by all KI tiles and every X box by all NO tiles).
  constexpr uint32_t kBoxBytes = 64 * kBK * 2;  // [64 rows(k) x 64 cols(mn)] bf16 = 8 KB
  constexpr uint32_t kABytes = 2 * kBoxBytes;
  constexpr uint32_t kBBytes = (BN / 64) * kBoxBytes;
  constexpr uint32_t kStageBytes = kABytes + kBBytes;
  constexpr uint32_t kOnesBytes = 2048;         // 16 k-rows x 128 B of bf16(1.0)
  constexpr uint32_t kTmemCols = 2 * BN;        // BN (dW tile) + 16 (bias column), power of two
  constexpr int kPitch = BN + 4;
  static_assert((size_t)kBM * kPitch * 4 <= (size_t)STAGES * kStageBytes, "staging tile must fit in the stages");

  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[STAGES];
  __shared__ __align__(8) uint64_t empty_bar[STAGES];
  __shared__ __align__(8) uint64_t accum_bar;
  __shared__ uint32_t tmem_slot;

  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_al = smem_raw + (smem_base - smem_u32(smem_raw));
  float* stage_f = reinterpret_cast<float*>(smem_al);
  const uint32_t ones_addr = smem_base + STAGES * kStageBytes;
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int ki0 = blockIdx.x * BN;
  const int no0 = blockIdx.y * kBM;
  const int r_begin = blockIdx.z * rows_per_split;
  const int r_end = min(R, r_begin + rows_per_split);
  const int nkb = (r_end - r_begin + kBK - 1) / kBK;  // >= 1 by construction of the grid
  const bool do_bias = (dbias != nullptr) && (blockIdx.x == 0);
  // cluster geometry: rank = x_local + cx * y_local; peers along x share dY, peers along y share X
  const bool clustered = cx * cy > 1;
  const uint32_t rank = clustered ? cluster_ctarank() : 0u;
  const int xl = (int)rank % cx, yl = (int)rank / cx;
  const uint16_t mask_x = (uint16_t)(cx == 2 ? (3u << (cx * yl)) : (1u << rank));                 // (0,yl) and (1,yl)
  const uint16_t mask_y = (uint16_t)(cy == 2 ? ((1u << xl) | (1u << (xl + cx))) : (1u << rank));    // (xl,0) and (xl,1)
  const uint16_t mask_free = (uint16_t)(mask_x | mask_y);      // CTAs whose loads land in this CTA's stages
  const uint32_t n_free = (uint32_t)(1 + (cx == 2) + (cy == 2));

  pdl_trigger();
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmY);
    tma_prefetch_desc(&tmX);
#pragma unroll
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], n_free);   // this CTA and the peers it multicasts to have drained the stage
    }
    mbar_init(&accum_bar, 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(&tmem_slot, kTmemCols);
    tmem_relinquish();
  }
  if (do_bias && warp >= 2) {
    uint32_t* ones = reinterpret_cast<uint32_t*>(smem_al + STAGES * kStageBytes);
    for (int i = threadIdx.x - 64; i < (int)(kOnesBytes / 4); i += 128) ones[i] = 0x3F803F80u;
    fence_proxy_async();  // generic-proxy writes -> visible to the tensor core (async proxy)
  }
  tc_fence_before();
  __syncthreads();
  if (clustered) cluster_sync_all();   // every CTA's barriers are initialised before a peer's multicast can touch them
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;
  pdl_wait();

  if (warp == 0) {
    if (elect_one()) {
      constexpr int kAhead = 2 * STAGES;   // L2 prefetch distance in k-blocks (the ring holds STAGES of them)
      for (int kb = 0; kb < nkb; ++kb) {
        const int s = kb % STAGES;
        if (kb + kAhead < nkb) {
          // every dY box is read by all KI tiles, every X box by all NO tiles: one of them prefetches for the others
          const int rp = r_begin + (kb + kAhead) * kBK;
          if (blockIdx.x == 0) { tma_prefetch_l2_2d(&tmY, no0, rp); tma_prefetch_l2_2d(&tmY, no0 + 64, rp); }
          if (blockIdx.y == 0) { tma_prefetch_l2_2d(&tmX, ki0, rp); tma_prefetch_l2_2d(&tmX, ki0 + 64, rp); }
        }
        if (kb >= STAGES) mbar_wait(&empty_bar[s], ((kb / STAGES) - 1) & 1);
        mbar_arrive_expect_tx(&full_bar[s], kStageBytes);
        const uint32_t a_dst = smem_base + s * kStageBytes;
        const int r0 = r_begin + kb * kBK;
        // rows_per_split is a multiple of kBK, so only the global tail (>= R) is zero-filled by TMA
        if (cx == 2) {   // this CTA fetches dY box xl for both KI tiles of its cluster row
          tma_load_2d_mc(a_dst + xl * kBoxBytes, &tmY, &full_bar[s], no0 + 64 * xl, r0, mask_x);
        } else {
          tma_load_2d_addr(a_dst, &tmY, &full_bar[s], no0, r0);
          tma_load_2d_addr(a_dst + kBoxBytes, &tmY, &full_bar[s], no0 + 64, r0);
        }
        if (cy == 2) {   // ... and X box yl for both NO tiles of its cluster column
          tma_load_2d_mc(a_dst + kABytes + yl * kBoxBytes, &tmX, &full_bar[s], ki0 + 64 * yl, r0, mask_y);
        } else {
#pragma unroll
          for (int bx = 0; bx < BN / 64; ++bx)
            tma_load_2d_addr(a_dst + kABytes + bx * kBoxBytes, &tmX, &full_bar[s], ki0 + 64 * bx, r0);
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      const uint32_t idesc = make_idesc_bf16(kBM, BN, 1, 1);
      const uint32_t idesc_b = make_idesc_bf16(kBM, 16, 1, 1);
      for (int kb = 0; kb < nkb; ++kb) {
        const int s = kb % STAGES;
        mbar_wait(&full_bar[s], (kb / STAGES) & 1);
        tc_fence_after();
        const uint32_t a_addr = smem_base + s * kStageBytes;
        const uint32_t b_addr = a_addr + kABytes;
#pragma unroll
        for (int k = 0; k < kBK / 16; ++k) {
          // MN-major, 128B swizzle: 64 mn-elements per 128B row, 8 k-rows per 1024B atom (SBO), next 64
          // mn-elements in the neighbouring TMA box (LBO = box size)
          const uint64_t da = make_smem_desc(a_addr + k * 2048, kBoxBytes, 1024, 2);
          const uint64_t db = make_smem_desc(b_addr + k * 2048, kBoxBytes, 1024, 2);
          umma_bf16(tmem_base, da, db, idesc, (kb > 0 || k > 0) ? 1u : 0u);
          if (do_bias) {
            const uint64_t d1 = make_smem_desc(ones_addr, kBoxBytes, 1024, 2);
            umma_bf16(tmem_base + BN, da, d1, idesc_b, (kb > 0 || k > 0) ? 1u : 0u);
          }
        }
        if (clustered) umma_commit_mc(&empty_bar[s], mask_free);   // frees the stage here and tells the peers that feed it
        else umma_commit(&empty_bar[s]);
      }
      umma_commit(&accum_bar);
    }
  } else {
    const int quad = warp & 3;
    const int row_l = quad * 32 + lane;
    mbar_wait(&accum_bar, 0);
    tc_fence_after();
    const uint32_t t_row = tmem_base + ((uint32_t)(quad * 32) << 16);
    float* my_row = stage_f + row_l * kPitch;
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
      if (ki0 + c0 >= KI) break;
      uint32_t acc[32];
      tmem_ld32(t_row + (uint32_t)c0, acc);
      tmem_ld_wait();
#pragma unroll
      for (int j4 = 0; j4 < 8; ++j4)
        *reinterpret_cast<float4*>(my_row + c0 + j4 * 4) =
            make_float4(__uint_as_float(acc[4 * j4]), __uint_as_float(acc[4 * j4 + 1]),
                        __uint_as_float(acc[4 * j4 + 2]), __uint_as_float(acc[4 * j4 + 3]));
    }
    if (do_bias) {
      uint32_t bacc[16];
      tmem_ld16(t_row + (uint32_t)BN, bacc);
      tmem_ld_wait();
      if constexpr (DET) {
        float* slot = reinterpret_cast<float*>(ws + (blockIdx.z + (long long)gridDim.z * (blockIdx.y * gridDim.x + blockIdx.x)) *
                                                        wgrad_slot_f4<BN>());
        slot[kBM * BN + row_l] = __uint_as_float(bacc[0]);
      } else {
        if (no0 + row_l < NO) atomicAdd(dbias + no0 + row_l, __uint_as_float(bacc[0]));
      }
    }
    __syncwarp();
    // coalesced accumulation: lane = 4 consecutive columns, one row (128 columns of it) per step
#pragma unroll 1
    for (int cp = 0; cp < BN / 128; ++cp) {
      const int lcol = cp * 128 + lane * 4;
      const int kcol = ki0 + lcol;
      const int nvalid = KI - kcol;
      const bool vec = (ldw % 4 == 0) && nvalid >= 4 && ((reinterpret_cast<uintptr_t>(dW) & 15) == 0);
#pragma unroll 4
      for (int it = 0; it < 32; ++it) {
        const int rl = quad * 32 + it;
        const int no = no0 + rl;
        if (no >= NO || nvalid <= 0) continue;
        const float4 v = *reinterpret_cast<const float4*>(stage_f + rl * kPitch + lcol);
        if constexpr (DET) {
          ws[(blockIdx.z + (long long)gridDim.z * (blockIdx.y * gridDim.x + blockIdx.x)) * wgrad_slot_f4<BN>() +
             (rl * BN + lcol) / 4] = v;
          continue;
        }
        float* dst = dW + (long long)no * ldw + kcol;
        if (vec) {
          asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(v.x), "f"(v.y), "f"(v.z),
                       "f"(v.w)
                       : "memory");
        } else {
          if (nvalid > 0) atomicAdd(dst, v.x);
          if (nvalid > 1) atomicAdd(dst + 1, v.y);
          if (nvalid > 2) atomicAdd(dst + 2, v.z);
          if (nvalid > 3) atomicAdd(dst + 3, v.w);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (clustered) cluster_sync_all();   // no CTA leaves while a peer's commit may still arrive on its barriers
  if (warp == 1) tmem_dealloc(tmem_base, kTmemCols);
  if constexpr (DET) {
    const long long tile = blockIdx.y * gridDim.x + blockIdx.x;
    const bool vec = (ldw % 4 == 0) && ((reinterpret_cast<uintptr_t>(dW) & 15) == 0);
    det_tree_fold(ws + tile * gridDim.z * wgrad_slot_f4<BN>(), wgrad_slot_f4<BN>(),
                  (kBM * BN + (do_bias ? kBM : 0)) / 4, blockIdx.z, gridDim.z, tickets + tile * gridDim.z,
                  [&](int i, float4 v) {
                    const int e = 4 * i;
                    if (e >= kBM * BN) {   // bias column
                      const float vv[4] = {v.x, v.y, v.z, v.w};
                      for (int u = 0; u < 4; ++u)
                        if (no0 + e - kBM * BN + u < NO) dbias[no0 + e - kBM * BN + u] += vv[u];
                      return;
                    }
                    const int no = no0 + e / BN, kcol = ki0 + e % BN;
                    if (no >= NO || kcol >= KI) return;
                    float* dst = dW + (long long)no * ldw + kcol;
                    if (vec && kcol + 4 <= KI) {
                      float4 o = *reinterpret_cast<float4*>(dst);
                      *reinterpret_cast<float4*>(dst) = det_add(o, v);
                      return;
                    }
                    const float vv[4] = {v.x, v.y, v.z, v.w};
                    for (int u = 0; u < 4 && kcol + u < KI; ++u) dst[u] += vv[u];
                  });
  }
}

// ------------------------------------------------------------------------------------------------
// bias gradient: out[c] += sum_r dY[r,c]
// ------------------------------------------------------------------------------------------------
constexpr int kColsumRows = 256;
// DET: the CTAs of a column slice (blockIdx.x) fold their 512 column sums with det_tree_fold instead of atomics
template <bool DET = false>
__global__ void __launch_bounds__(256) colsum_bf16_kernel(const bf16* __restrict__ dY, long long ld, int R, int NO,
                                                           float* __restrict__ out, float* __restrict__ ws,
                                                           unsigned int* tickets) {
  const int c = (blockIdx.x * 256 + threadIdx.x) * 2;
  if (!DET && c >= NO) return;
  const int r0 = blockIdx.y * kColsumRows;
  const int r1 = (DET && c >= NO) ? r0 : min(R, r0 + kColsumRows);   // (DET: every thread takes part in the fold)
  float s0 = 0.f, s1 = 0.f;
  if (c + 1 < NO && (ld & 1) == 0) {
    for (int r = r0; r < r1; ++r) {
      uint32_t u = __ldg(reinterpret_cast<const uint32_t*>(dY + (long long)r * ld + c));
      float2 f = unpack_bf16x2(u);
      s0 += f.x;
      s1 += f.y;
    }
  } else {
    for (int r = r0; r < r1; ++r) {
      s0 += __bfloat162float(dY[(long long)r * ld + c]);
      if (c + 1 < NO) s1 += __bfloat162float(dY[(long long)r * ld + c + 1]);
    }
  }
  if constexpr (DET) {
    float* slices = ws + (long long)blockIdx.x * gridDim.y * 512;
    slices[blockIdx.y * 512 + 2 * threadIdx.x] = s0;
    slices[blockIdx.y * 512 + 2 * threadIdx.x + 1] = s1;
    det_tree_fold(slices, 512, 512, blockIdx.y, gridDim.y, tickets + (long long)blockIdx.x * gridDim.y,
                  [&](int i, float v) {
                    if (blockIdx.x * 512 + i < NO) out[blockIdx.x * 512 + i] += v;
                  });
    return;
  }
  atomicAdd(out + c, s0);
  if (c + 1 < NO) atomicAdd(out + c + 1, s1);
}

// ------------------------------------------------------------------------------------------------
// fp32 -> bf16 cast with optional transposed copy (weight shadows, input staging)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) cast_bf16_kernel(const float* __restrict__ x, long long ldx, bf16* __restrict__ y,
                                                         long long ldy, bf16* __restrict__ yt, long long ldyt, int R,
                                                         int C) {
  __shared__ float tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = r0 + ty + i * 8, c = c0 + tx;
    float v = 0.f;
    if (r < R && c < C) {
      v = x[(long long)r * ldx + c];
      if (y) y[(long long)r * ldy + c] = __float2bfloat16_rn(v);
    }
    tile[ty + i * 8][tx] = v;
  }
  if (yt == nullptr) return;
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c = c0 + ty + i * 8, r = r0 + tx;
    if (r < R && c < C) yt[(long long)c * ldyt + r] = __float2bfloat16_rn(tile[tx][ty + i * 8]);
  }
}

}  // namespace mmfm

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
namespace mmfm {
int try_launch_gemm_ts(const mmfm_gemm_args* a, cudaStream_t st);   // gemm_ts.cu
}
using namespace mmfm;

template <int BN, int STAGES, int EPI>
static int launch_tn(const mmfm_gemm_args* a, cudaStream_t st) {
  CUtensorMap tmA, tmB;
  int rc = make_tmap_bf16_2d(&tmA, a->A, (uint64_t)a->M, (uint64_t)a->K, (uint64_t)a->lda, kBK, kBM, TMA_SW_128);
  if (rc) return rc;
  rc = make_tmap_bf16_2d(&tmB, a->B, (uint64_t)a->N, (uint64_t)a->K, (uint64_t)a->ldb, kBK, BN, TMA_SW_128);
  if (rc) return rc;
  constexpr size_t smem = (size_t)STAGES * (kBM * kBK * 2 + BN * kBK * 2) + (size_t)kBM * (BN + 4) * 4 + 1024;
  static bool attr_set = false;
  if (!attr_set) {
    MMFM_CHECK_CUDA(cudaFuncSetAttribute(gemm_tn_kernel<BN, STAGES, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem));
    attr_set = true;
  }
  const int tiles_n = (a->N + BN - 1) / BN, tiles_m = (a->M + kBM - 1) / kBM;
  const int n_tiles = tiles_n * tiles_m;
  int grid = n_tiles < device_sm_count() ? n_tiles : device_sm_count();
  // weight-stationary schedule: B's whole K extent fits half of the ring area and the grid can be a multiple of tiles_n
  // (measured neutral on B200 -- these GEMMs turned out to be bound by epilogue instruction issue, not by L2 -> SM
  // traffic -- so the streamed-B schedule stays the default; MMFM_GEMM_BSTAT=1 enables it for A/B measurements)
  static int bstat_env = -1;
  if (bstat_env < 0) {
    const char* e = getenv("MMFM_GEMM_BSTAT");
    bstat_env = (e && e[0] == '1') ? 1 : 0;
  }
  const int nkb = (a->K + kBK - 1) / kBK;
  int bstat = 0;
  if (bstat_env && (size_t)nkb * BN * kBK * 2 * 2 <= (size_t)STAGES * (kBM * kBK * 2 + BN * kBK * 2) &&
      tiles_n <= device_sm_count() && tiles_m > 1) {
    int per_n = device_sm_count() / tiles_n;
    if (per_n > tiles_m) per_n = tiles_m;
    grid = per_n * tiles_n;
    bstat = 1;
  }
  set_l2_window(a->D, (size_t)a->M * (size_t)a->ldd * (a->d_fp32 ? 4 : 2));   // the output is the next kernel's input
  MMFM_CHECK_CUDA(launch_pdl(gemm_tn_kernel<BN, STAGES, EPI>, dim3(grid), dim3(kTnThreads), smem, st, tmA, tmB, *a, tiles_n,
                             n_tiles, bstat));
  return 0;
}

template <int EPI>
static int launch_tn_bn(const mmfm_gemm_args* a, cudaStream_t st) {
  if (a->N <= 64) return launch_tn<64, 4, EPI>(a, st);
  return launch_tn<128, 4, EPI>(a, st);
}

static bool al(const void* p, uintptr_t m) { return (reinterpret_cast<uintptr_t>(p) & (m - 1)) == 0; }

// pick the branch-free epilogue when the call fits one of the flavours the model uses and everything is aligned
static int pick_epi(const mmfm_gemm_args* a) {
  if (a->N % 4 != 0 || a->ldd % 4 != 0) return EPI_GENERIC;
  const bool f32 = a->d_fp32 != 0;
  if (!al(a->D, f32 ? 16 : 8)) return EPI_GENERIC;
  const bool extras = a->drop.thresh != 0 || a->row_zero != nullptr || a->remap_T > 0;
  if (a->res) {
    if (a->act != MMFM_ACT_NONE || !f32 || a->D2 || a->ldr % 4 != 0 || !al(a->res, 16)) return EPI_GENERIC;
    return EPI_RES_F32;
  }
  if (extras) return EPI_GENERIC;
  switch (a->act) {
    case MMFM_ACT_NONE: return a->D2 ? EPI_GENERIC : (f32 ? EPI_PLAIN_F32 : EPI_PLAIN_BF16);
    case MMFM_ACT_GELU: return (!f32 && a->D2 && al(a->D2, 8)) ? EPI_GELU : EPI_GENERIC;
    case MMFM_ACT_GELU_DG: return (!f32 && a->D2 && al(a->D2, 8)) ? EPI_GELU_DG : EPI_GENERIC;
    case MMFM_ACT_MULAUX:
      if (f32 || a->D2 || a->ldaux % 4 != 0 || !al(a->aux, 8)) return EPI_GENERIC;
      return EPI_MULAUX;
    case MMFM_ACT_SOFTSIGN: return (!f32 && !a->D2) ? EPI_SOFTSIGN : EPI_GENERIC;
    case MMFM_ACT_DGELU:
    case MMFM_ACT_DSOFTSIGN:
      if (f32 || a->D2 || a->ldaux % 4 != 0 || !al(a->aux, 8)) return EPI_GENERIC;
      return a->act == MMFM_ACT_DGELU ? EPI_DGELU : EPI_DSOFTSIGN;
  }
  return EPI_GENERIC;
}

extern "C" int mmfm_gemm_tn(const mmfm_gemm_args* a, void* stream) {
  MMFM_REQUIRE(a != nullptr, "mmfm_gemm_tn: null args");
  MMFM_REQUIRE(a->M > 0 && a->N > 0 && a->K > 0, "mmfm_gemm_tn: bad shape M=%d N=%d K=%d", a->M, a->N, a->K);
  MMFM_REQUIRE(a->A && a->B && a->D, "mmfm_gemm_tn: null operand");
  MMFM_REQUIRE(a->act >= MMFM_ACT_NONE && a->act <= MMFM_ACT_ROWDOT_DROP, "mmfm_gemm_tn: bad act %d", a->act);
  MMFM_REQUIRE(!(a->act == MMFM_ACT_DGELU || a->act == MMFM_ACT_DSOFTSIGN || a->act == MMFM_ACT_MULAUX ||
                 a->act == MMFM_ACT_ROWDOT_DROP) || a->aux,
               "mmfm_gemm_tn: act %d needs aux", a->act);
  MMFM_REQUIRE(a->act != MMFM_ACT_ROWDOT_DROP || (a->rowdot && a->rowdot_S > 0 && a->M % a->rowdot_S == 0),
               "mmfm_gemm_tn: MMFM_ACT_ROWDOT_DROP needs rowdot / rowdot_S with M %% rowdot_S == 0");
  MMFM_REQUIRE(a->act != MMFM_ACT_GELU_DG || a->D2, "mmfm_gemm_tn: MMFM_ACT_GELU_DG needs the D2 buffer");
  MMFM_REQUIRE(a->drop.thresh == 0 || a->drop.seed, "mmfm_gemm_tn: dropout without seed pointer");
  MMFM_REQUIRE(a->drop.thresh < 256, "mmfm_gemm_tn: dropout threshold out of range");
  MMFM_REQUIRE(!(a->row_zero && a->remap_T == 0) || a->remap_S > 0, "mmfm_gemm_tn: row_zero needs remap_S");
  MMFM_REQUIRE(a->act == MMFM_ACT_NONE || a->act == MMFM_ACT_ROWDOT_DROP || (a->drop.thresh == 0 && a->row_zero == nullptr),
               "mmfm_gemm_tn: an activation epilogue cannot be combined with dropout / token zeroing");
  cudaStream_t st = (cudaStream_t)stream;
  // calls without output-row remap go to the TMA-store kernel (gemm_ts.cu); the rest (embedding projection with
  // remap + token zeroing, narrow N, unaligned pitches, legacy activation flavours) stay here
  {
    const int taken = try_launch_gemm_ts(a, st);
    if (taken != 0) return taken > 0 ? 0 : taken;
    MMFM_REQUIRE(a->act != MMFM_ACT_ROWDOT_DROP,
                 "mmfm_gemm_tn: MMFM_ACT_ROWDOT_DROP is built for the TMA-store kernel only (bf16 D, N %% 32 == 0, N > 64, "
                 "16-byte aligned D / aux / pitches, no remap / bias)");
  }
  switch (pick_epi(a)) {
    case EPI_PLAIN_BF16: return launch_tn_bn<EPI_PLAIN_BF16>(a, st);
    case EPI_PLAIN_F32: return launch_tn_bn<EPI_PLAIN_F32>(a, st);
    case EPI_RES_F32: return launch_tn_bn<EPI_RES_F32>(a, st);
    case EPI_GELU: return launch_tn_bn<EPI_GELU>(a, st);
    case EPI_SOFTSIGN: return launch_tn_bn<EPI_SOFTSIGN>(a, st);
    case EPI_DGELU: return launch_tn_bn<EPI_DGELU>(a, st);
    case EPI_DSOFTSIGN: return launch_tn_bn<EPI_DSOFTSIGN>(a, st);
    case EPI_GELU_DG: return launch_tn_bn<EPI_GELU_DG>(a, st);
    case EPI_MULAUX: return launch_tn_bn<EPI_MULAUX>(a, st);
    default: return launch_tn_bn<EPI_GENERIC>(a, st);
  }
}

// split-R arithmetic of the wgrad launch (also the deterministic workspace size: one slot per CTA)
static int wgrad_splits(int R, int NO, int KI, int BN, int* rows_per_split) {
  const int tiles = ((NO + kBM - 1) / kBM) * ((KI + BN - 1) / BN);
  const int kblocks = (R + kBK - 1) / kBK;
  static int waves_x2 = -1;   // MMFM_WGRAD_CTAS_X2: target CTA count in half-SM-counts (default 4 = two CTAs per SM)
  if (waves_x2 < 0) {
    const char* e = getenv("MMFM_WGRAD_CTAS_X2");
    waves_x2 = e ? atoi(e) : 4;
    if (waves_x2 < 1) waves_x2 = 4;
  }
  // all CTAs must be resident at once (two per SM): a split count rounded UP spills a few CTAs into a second wave that
  // costs as much as the first (measured 43 us vs 34 us on the QKV shape), so round down
  // BN 256: one CTA per SM (144 KB of stages, 512 TMEM columns); BN 128: two
  int splits = ((BN == 256 ? 2 : waves_x2) * device_sm_count() / 2) / tiles;
  if (splits > kblocks) splits = kblocks;
  if (splits < 1) splits = 1;
  *rows_per_split = ((kblocks + splits - 1) / splits) * kBK;
  return (R + *rows_per_split - 1) / *rows_per_split;
}

template <int BN>
static int launch_wgrad(const void* dY, long long lddy, const void* X, long long ldx, int R, int NO, int KI, float* dW,
                        long long ldw, float* dbias, void* stream) {
  constexpr int STAGES = 3;
  CUtensorMap tmY, tmX;
  int rc = make_tmap_bf16_2d(&tmY, dY, (uint64_t)R, (uint64_t)NO, (uint64_t)lddy, 64, kBK, TMA_SW_128);
  if (rc) return rc;
  rc = make_tmap_bf16_2d(&tmX, X, (uint64_t)R, (uint64_t)KI, (uint64_t)ldx, 64, kBK, TMA_SW_128);
  if (rc) return rc;
  constexpr size_t smem = (size_t)STAGES * ((2 + BN / 64) * 64 * kBK * 2) + 2048 + 1024;
  static bool attr_set = false;
  if (!attr_set) {
    MMFM_CHECK_CUDA(cudaFuncSetAttribute(gemm_wgrad_kernel<STAGES, BN>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem));
    attr_set = true;
  }
  int rows_per_split = 0;
  const int splits = wgrad_splits(R, NO, KI, BN, &rows_per_split);
  dim3 grid((KI + BN - 1) / BN, (NO + kBM - 1) / kBM, splits);
  static int mc_env = -1;   // MMFM_WGRAD_MULTICAST=1: 2x2 clusters, each CTA loads half of its boxes and multicasts them
  if (mc_env < 0) {
    const char* e = getenv("MMFM_WGRAD_MULTICAST");
    mc_env = (e && e[0] == '1') ? 1 : 0;   // measured slower than independent CTAs (lock-step stages): off by default
  }
  const int cx = (mc_env && BN == 128 && grid.x % 2 == 0) ? 2 : 1, cy = (mc_env && BN == 128 && grid.y % 2 == 0) ? 2 : 1;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = dim3(kGemmThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cx;
  attr[0].val.clusterDim.y = cy;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  MMFM_CHECK_CUDA(cudaLaunchKernelEx(&cfg, gemm_wgrad_kernel<STAGES, BN>, tmY, tmX, R, NO, KI, dW, ldw, rows_per_split, dbias,
                                     cx, cy, (float4*)nullptr, (unsigned int*)nullptr));
  return 0;
}

// deterministic twin: always the 128-wide tile without clusters (MMFM_WGRAD_BN / MMFM_WGRAD_MULTICAST do not apply)
static DetNeed wgrad_det_need(int R, int NO, int KI) {
  int rows_per_split = 0;
  const int splits = wgrad_splits(R, NO, KI, 128, &rows_per_split);
  const long long ctas = (long long)((NO + kBM - 1) / kBM) * ((KI + 127) / 128) * splits;
  return DetNeed{ctas * wgrad_slot_f4<128>() * 16, (int)ctas};
}

static int launch_wgrad_det(const void* dY, long long lddy, const void* X, long long ldx, int R, int NO, int KI,
                            float* dW, long long ldw, float* dbias, const mmfm_det_ws* ws, cudaStream_t st) {
  constexpr int STAGES = 3, BN = 128;
  MMFM_REQUIRE(ws != nullptr, "mmfm_gemm_wgrad_det: null workspace");
  if (int rc = det_ws_check(ws->buf, ws->bytes, ws->tickets, ws->n_tickets, wgrad_det_need(R, NO, KI),
                            "mmfm_gemm_wgrad_det"))
    return rc;
  CUtensorMap tmY, tmX;
  int rc = make_tmap_bf16_2d(&tmY, dY, (uint64_t)R, (uint64_t)NO, (uint64_t)lddy, 64, kBK, TMA_SW_128);
  if (rc) return rc;
  rc = make_tmap_bf16_2d(&tmX, X, (uint64_t)R, (uint64_t)KI, (uint64_t)ldx, 64, kBK, TMA_SW_128);
  if (rc) return rc;
  constexpr size_t smem = (size_t)STAGES * ((2 + BN / 64) * 64 * kBK * 2) + 2048 + 1024;
  static bool attr_set = false;
  if (!attr_set) {
    MMFM_CHECK_CUDA(cudaFuncSetAttribute(gemm_wgrad_kernel<STAGES, BN, true>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set = true;
  }
  int rows_per_split = 0;
  const int splits = wgrad_splits(R, NO, KI, BN, &rows_per_split);
  MMFM_CHECK_CUDA(launch_pdl(gemm_wgrad_kernel<STAGES, BN, true>, dim3((KI + BN - 1) / BN, (NO + kBM - 1) / kBM, splits),
                             dim3(kGemmThreads), smem, st, tmY, tmX, R, NO, KI, dW, ldw, rows_per_split, dbias, 1, 1,
                             (float4*)ws->buf, ws->tickets));
  return 0;
}

static DetNeed colsum_det_need(int R, int NO) {
  const long long slices = (NO + 511) / 512, parts = (R + kColsumRows - 1) / kColsumRows;
  return DetNeed{slices * parts * 512 * 4, (int)(slices * parts)};
}

namespace mmfm {
bool det_need_gemm(int kind, long long d0, long long d1, long long d2, DetNeed* need) {
  if (kind == MMFM_DET_WGRAD) *need = wgrad_det_need((int)d0, (int)d1, (int)d2);
  else if (kind == MMFM_DET_COLSUM) *need = colsum_det_need((int)d0, (int)d1);
  else return false;
  return true;
}
}  // namespace mmfm


extern "C" int mmfm_gemm_wgrad(const void* dY, long long lddy, const void* X, long long ldx, int R, int NO, int KI,
                               float* dW, long long ldw, float* dbias, void* stream) {
  MMFM_REQUIRE(dY && X && dW, "mmfm_gemm_wgrad: null operand");
  MMFM_REQUIRE(R > 0 && NO > 0 && KI > 0, "mmfm_gemm_wgrad: bad shape R=%d NO=%d KI=%d", R, NO, KI);
  static int bn_env = -1;   // MMFM_WGRAD_BN=128 pins the 128-wide dW tile (A/B measurements)
  if (bn_env < 0) {
    const char* e = getenv("MMFM_WGRAD_BN");
    bn_env = e ? atoi(e) : 128;   // the 256-wide tile measured equal (QKV 29.4 vs 29.8 us) to slower (down 25.7 vs 23.4 us)
  }
  if (bn_env == 256 && KI % 256 == 0) return launch_wgrad<256>(dY, lddy, X, ldx, R, NO, KI, dW, ldw, dbias, stream);
  return launch_wgrad<128>(dY, lddy, X, ldx, R, NO, KI, dW, ldw, dbias, stream);
}

extern "C" int mmfm_gemm_wgrad_det(const void* dY, long long lddy, const void* X, long long ldx, int R, int NO, int KI,
                                   float* dW, long long ldw, float* dbias, const mmfm_det_ws* ws, void* stream) {
  MMFM_REQUIRE(dY && X && dW, "mmfm_gemm_wgrad_det: null operand");
  MMFM_REQUIRE(R > 0 && NO > 0 && KI > 0, "mmfm_gemm_wgrad_det: bad shape R=%d NO=%d KI=%d", R, NO, KI);
  return launch_wgrad_det(dY, lddy, X, ldx, R, NO, KI, dW, ldw, dbias, ws, (cudaStream_t)stream);
}

extern "C" int mmfm_colsum_bf16(const void* dY, long long ld, int R, int NO, float* out, void* stream) {
  MMFM_REQUIRE(dY && out && R > 0 && NO > 0, "mmfm_colsum_bf16: bad arguments");
  dim3 grid((NO + 511) / 512, (R + kColsumRows - 1) / kColsumRows);
  colsum_bf16_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const bf16*)dY, ld, R, NO, out, nullptr, nullptr);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_colsum_bf16_det(const void* dY, long long ld, int R, int NO, float* out, const mmfm_det_ws* ws,
                                    void* stream) {
  MMFM_REQUIRE(dY && out && R > 0 && NO > 0 && ws, "mmfm_colsum_bf16_det: bad arguments");
  if (int rc = det_ws_check(ws->buf, ws->bytes, ws->tickets, ws->n_tickets, colsum_det_need(R, NO), "mmfm_colsum_bf16_det"))
    return rc;
  dim3 grid((NO + 511) / 512, (R + kColsumRows - 1) / kColsumRows);
  colsum_bf16_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>((const bf16*)dY, ld, R, NO, out, (float*)ws->buf,
                                                                   ws->tickets);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_cast_bf16(const float* x, long long ldx, void* y, long long ldy, void* yt, long long ldyt, int R,
                              int C, void* stream) {
  MMFM_REQUIRE(x && (y || yt) && R > 0 && C > 0, "mmfm_cast_bf16: bad arguments");
  dim3 grid((C + 31) / 32, (R + 31) / 32);
  MMFM_REQUIRE(grid.y <= 65535, "mmfm_cast_bf16: too many rows (%d)", R);
  cast_bf16_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, ldx, (bf16*)y, ldy, (bf16*)yt, ldyt, R, C);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}
