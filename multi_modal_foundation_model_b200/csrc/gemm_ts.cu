// Persistent tcgen05 GEMM with a TMA-store epilogue: D[M,N] = epilogue(A[M,K] . B[N,K]^T), both operands K-major bf16.
//
// Same contract and main loop as gemm_tn_kernel (gemm.cu) -- nn.Linear forward / dgrad of the reference path
// (mm_utils.py:51-52,107-109,114,145-147,152; encoder_embeddings.py:50; decoder_embeddings.py:107; mm.py:292) -- for the
// calls whose output rows are not remapped.  What changes is the way a finished tile leaves the SM.  The epilogue of
// gemm_tn_kernel costs as much as cuBLAS's whole GEMM on the QKV shape (tools/gemm_bench.py, K = 64 probe: 25 us for
// the 79 MB output): every epilogue warp reads TMEM, stages the tile in shared memory, reads it back row-contiguously and
// issues its own global loads (residual / saved tensor) and stores.  Here
//   * warps 4-19 (epilogue): thread = accumulator row; tcgen05.ld -> bias / activation / dropout -> ONE pass of 16-byte
//     shared-memory stores straight into the TMA box layout (64B swizzle for bf16, 128B for fp32: conflict-free for
//     row-per-thread accesses) -> fence.proxy.async -> mbarrier arrive.  No global memory instruction at all.
//   * warp 2 (store): one elected lane issues cp.async.bulk.tensor stores of the tile's four [128 x 32] boxes (UTMASTG)
//     and recycles the staging buffer when the TMA unit has read it.  Edge tiles are clipped by the tensor map.
//   * warp 3 (input): saved-tensor (bf16) boxes of a tile are TMA-loaded INTO the staging buffer
//     two tiles ahead; the epilogue combines them in place, so they cost neither registers nor extra shared memory.
//   * warp 0 (A/B ring producer) and warp 1 (TMEM allocation + tcgen05.mma issue, double-buffered accumulator) as in
//     gemm_tn_kernel.
// Staging is double-buffered, so the MMA of tile i+1, the epilogue of tile i and the store of tile i-1 overlap.
//
// A and B stream through the ring together.  A weight-stationary schedule (each CTA keeping its column tile's [BN x K]
// weight slab resident, the ring carrying activation k-blocks only) cut the QKV call's L2 -> SM traffic from 393 MB to
// 236 MB but measured neutral to slower on B200: the A-only ring it leaves room for is too shallow.
#include "common.cuh"
#include "host_util.h"
#include "../../include/mmfm_b200.h"

#ifdef MMFM_DBG_TIMING
// per-role clock64 trace of one CTA (tools/micro/gemm_ts_timing.py): g_dbg_ts[role][slot]
__device__ long long g_dbg_ts[8][64];
__device__ __forceinline__ long long dbg_now() {
  long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t) :: "memory");
  return t;
}
#define DBG_TS(role, slot) do { if (blockIdx.x == 5 && (slot) < 64) g_dbg_ts[role][slot] = dbg_now(); } while (0)
__device__ long long g_dbg_cta[160][2];     // entry / exit of every CTA
extern "C" int mmfm_debug_read_gemm_ts(long long* out) {
  return (int)cudaMemcpyFromSymbol(out, g_dbg_ts, sizeof(long long) * 8 * 64);
}
extern "C" int mmfm_debug_read_gemm_cta(long long* out) {
  return (int)cudaMemcpyFromSymbol(out, g_dbg_cta, sizeof(long long) * 160 * 2);
}
#else
#define DBG_TS(role, slot) do { } while (0)
#endif

namespace mmfm {

constexpr int kTsBM = 128, kTsBK = 64;   // tile = 128 x BN (BN = 128 or 256 columns, a template parameter)
constexpr int kTsEpiWarps = 16, kTsFirstEpi = 4;
constexpr int kTsThreads = (kTsFirstEpi + kTsEpiWarps) * 32;   // 640

enum TsEpi : int {
  TS_BF16 = 0,       // D(bf16) = v
  TS_SOFTSIGN = 1,   // D(bf16) = softsign(v) * s
  TS_F32 = 2,        // D(f32)  = v
  TS_GELU = 3,       // D(bf16) = gelu(v)                       (forward-only MLP-up: no derivative stored)
  TS_GELU_DG = 4,    // D(bf16) = gelu(v) ; D2(bf16) = gelu'(v)
  TS_MULAUX = 5,     // D(bf16) = v * aux
  TS_DSOFTSIGN = 6,  // D(bf16) = v * s * (1 - |aux / s|)^2
  TS_ROWDOT = 7      // rowdot[(r / S), group, r % S] = sum_32cols v * aux ; D(bf16) = dropout(v)   (attention-backward prep)
};

template <int EPI>
struct TsCfg {
  static constexpr bool kF32 = EPI == TS_F32;
  static constexpr bool kHasIn = EPI == TS_MULAUX || EPI == TS_DSOFTSIGN || EPI == TS_ROWDOT;
  static constexpr bool kTwoOut = EPI == TS_GELU_DG;
  static constexpr uint32_t kRowBytes = kF32 ? 128u : 64u;          // one box row: 32 columns
  static constexpr uint32_t kSlice = 128u * kRowBytes;              // one [128 x 32] box
  static constexpr uint32_t kOut = 4u * kSlice;                     // one output tile
  static constexpr uint32_t kBuf = kOut * (kTwoOut ? 2u : 1u);      // one staging buffer
};
constexpr int kTsMaxStages = 4;
constexpr size_t kTsMaxSmem = 230400;   // 225 KB dynamic (+ static barriers) of the 227 KB a CTA may own

// BN = 256: the tile is 128 x 256 (fp32 accumulator 2 x 256 TMEM columns).  Every byte of an A / B tile is read from
// shared memory once per tile by the tensor core and written once by TMA, and a 128 x 128 x 16 tcgen05.mma already reads
// 128 B/clk -- the whole shared-memory bandwidth of an SM -- so the main loop of the 128-wide tile runs at half the
// tensor rate (measured: the marginal cost of K is 1.05 PFLOP/s).  The 256-wide tile moves 25 % fewer shared-memory
// bytes per FLOP and re-reads the activation rows half as often.  The epilogue treats it as two 128-column units that
// go through the two staging buffers one after the other.
template <int EPI, int BN>
__global__ void __launch_bounds__(kTsThreads, 1) gemm_tn_ts_kernel(const __grid_constant__ CUtensorMap tmA,
                                                                    const __grid_constant__ CUtensorMap tmB,
                                                                    const __grid_constant__ CUtensorMap tmD,
                                                                    const __grid_constant__ CUtensorMap tmD2,
                                                                    const __grid_constant__ CUtensorMap tmIn,
                                                                    const mmfm_gemm_args p, int tiles_n, int n_tiles,
                                                                    int nst) {
  using Cfg = TsCfg<EPI>;
  constexpr int STAGES = kTsMaxStages;
  constexpr uint32_t kABytes = kTsBM * kTsBK * 2, kBBytes = BN * kTsBK * 2;
  constexpr uint32_t kTsStageBytes = kABytes + kBBytes;
  constexpr int NU = BN / 128;              // 128-column epilogue units per tile
  constexpr int kTsBN = BN;
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[STAGES], empty_bar[STAGES];
  __shared__ __align__(8) uint64_t acc_full[2], acc_empty[2], in_full[2], stg_full[2], stg_free[2];
  __shared__ uint32_t tmem_slot;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkb = (p.K + kTsBK - 1) / kTsBK;
  if (threadIdx.x == 0) DBG_TS(7, 63);     // kernel entry
#ifdef MMFM_DBG_TIMING
  if (threadIdx.x == 0 && blockIdx.x < 160) g_dbg_cta[blockIdx.x][0] = dbg_now();
#endif
  // shared memory: [ring: nst stages of A + B] [2 staging buffers]
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_al = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t stg_off = (uint32_t)nst * kTsStageBytes;
  const uint32_t stg_base = smem_base + stg_off;                      // staging buffers (1024-aligned)
  uint8_t* stg_ptr = smem_al + stg_off;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    tma_prefetch_desc(&tmD);
    if (Cfg::kTwoOut) tma_prefetch_desc(&tmD2);
    if (Cfg::kHasIn) tma_prefetch_desc(&tmIn);
#pragma unroll
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], kTsEpiWarps);
      mbar_init(&in_full[i], 1);
      mbar_init(&stg_full[i], kTsEpiWarps);
      mbar_init(&stg_free[i], 1);
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(&tmem_slot, 2u * BN);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------ A / B ring producer ------------------------------------------
    if (elect_one()) {
      uint32_t it = 0;
      const uint32_t ns = (uint32_t)nst;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int m0 = (tile / tiles_n) * kTsBM, n0 = (tile % tiles_n) * kTsBN;
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const uint32_t s = it % ns;
          if (it >= ns) mbar_wait(&empty_bar[s], ((it / ns) - 1) & 1);
          mbar_arrive_expect_tx(&full_bar[s], kTsStageBytes);
          const uint32_t a_dst = smem_base + s * kTsStageBytes;
          tma_load_2d_addr(a_dst, &tmA, &full_bar[s], kb * kTsBK, m0);
          tma_load_2d_addr(a_dst + kABytes, &tmB, &full_bar[s], kb * kTsBK, n0);
        }
        DBG_TS(0, (int)(it / (uint32_t)nkb) - 1);      // all k-blocks of the tile issued
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------ MMA issuer ----------------------------------------------------
    if (elect_one()) {
      const uint32_t idesc = make_idesc_bf16(kTsBM, kTsBN, 0, 0);
      uint32_t it = 0, t = 0;
      const uint32_t ns = (uint32_t)nst;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++t) {
        const uint32_t buf = t & 1u;
        if (t >= 2) mbar_wait(&acc_empty[buf], ((t >> 1) - 1) & 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + buf * kTsBN;
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const uint32_t s = it % ns;
          mbar_wait(&full_bar[s], (it / ns) & 1);
          tc_fence_after();
          const uint32_t a_addr = smem_base + s * kTsStageBytes;
          const uint32_t b_addr = a_addr + kABytes;
#pragma unroll
          for (int k = 0; k < kTsBK / 16; ++k)
            umma_bf16(d_tmem, make_smem_desc(a_addr + k * 32, 16, 1024, 2), make_smem_desc(b_addr + k * 32, 16, 1024, 2),
                      idesc, (kb > 0 || k > 0) ? 1u : 0u);
          umma_commit(&empty_bar[s]);
          if (kb == 0) DBG_TS(1, (int)t);                 // first k-block of the tile had landed, MMAs issued
        }
        umma_commit(&acc_full[buf]);
        DBG_TS(2, (int)t);                                // last MMA of the tile issued
      }
    }
  } else if (warp == 2) {
    // ------------------------------------------------ store warp ----------------------------------------------------
    if (elect_one()) {
      uint32_t u = 0;       // running count of 128-column units: staging buffer u & 1, barrier phase (u >> 1) & 1
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int m0 = (tile / tiles_n) * kTsBM, n0 = (tile % tiles_n) * kTsBN;
#pragma unroll 1
        for (int hh = 0; hh < NU; ++hh, ++u) {
          const uint32_t sb = u & 1u;
          mbar_wait(&stg_full[sb], (u >> 1) & 1);
          DBG_TS(3, (int)u);
          const uint32_t src = stg_base + sb * Cfg::kBuf;
          const int nu = n0 + 128 * hh;
#pragma unroll
          for (int h = 0; h < 4; ++h) {
            if (nu + 32 * h < p.N) {
              tma_store_2d(&tmD, src + h * Cfg::kSlice, nu + 32 * h, m0);
              if (Cfg::kTwoOut) tma_store_2d(&tmD2, src + Cfg::kOut + h * Cfg::kSlice, nu + 32 * h, m0);
            }
          }
          bulk_commit_group();
          bulk_wait_group_read<0>();        // the TMA unit has read the buffer: it may be refilled
          DBG_TS(4, (int)u);
          mbar_arrive(&stg_free[sb]);
        }
      }
      bulk_wait_group<0>();
    }
  } else if (warp == 3) {
    // ------------------------------------------------ input warp: saved-tensor boxes ------------------------------
    if (Cfg::kHasIn && elect_one()) {
      uint32_t u = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int m0 = (tile / tiles_n) * kTsBM, n0 = (tile % tiles_n) * kTsBN;
#pragma unroll 1
        for (int hh = 0; hh < NU; ++hh, ++u) {
          const uint32_t sb = u & 1u;
          const int nu = n0 + 128 * hh;
          if (nu >= p.N) {                                   // unit past the last column: nothing to load
            if (u >= 2) mbar_wait(&stg_free[sb], ((u >> 1) - 1) & 1);
            mbar_arrive(&in_full[sb]);
            continue;
          }
          if (u >= 2) mbar_wait(&stg_free[sb], ((u >> 1) - 1) & 1);
          int nbox = (p.N - nu + 31) / 32;
          if (nbox > 4) nbox = 4;
          mbar_arrive_expect_tx(&in_full[sb], (uint32_t)nbox * Cfg::kSlice);
          DBG_TS(5, (int)u);
          const uint32_t dst = stg_base + sb * Cfg::kBuf;
          for (int h = 0; h < nbox; ++h) tma_load_2d_addr(dst + h * Cfg::kSlice, &tmIn, &in_full[sb], nu + 32 * h, m0);
        }
      }
    }
  } else {
    // ------------------------------------------------ epilogue warps ------------------------------------------------
    // TMEM lane quadrant = warp % 4 (hardware rule), column slice h = (warp - 4) / 4: 32 columns = one TMA box
    const int ew = warp - kTsFirstEpi;
    const int quad = warp & 3, h = ew >> 2;
    const int row = quad * 32 + lane;
    bool drop = false;
    unsigned long long seed = 0ull;
    if (EPI == TS_ROWDOT) {
      drop = p.drop.thresh != 0u;
      if (drop) seed = *p.drop.seed;
    }
    const uint32_t drop_gpr = (uint32_t)((p.N + 15) >> 4);
    const float act_scale = p.act_scale, inv_scale = 1.0f / p.act_scale;
    // swizzled position of 16-byte chunk c of this thread's box row
    const uint32_t row_off = (uint32_t)row * Cfg::kRowBytes;
    const uint32_t swz = Cfg::kF32 ? (uint32_t)(row & 7) : (uint32_t)((row >> 1) & 3);

    uint32_t t = 0, u = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++t) {
      const uint32_t buf = t & 1u;
      const int m0 = (tile / tiles_n) * kTsBM, n0 = (tile % tiles_n) * kTsBN;
      mbar_wait(&acc_full[buf], (t >> 1) & 1);
      tc_fence_after();
#pragma unroll 1
      for (int hh = 0; hh < NU; ++hh, ++u) {
      const uint32_t sb = u & 1u;
      const int nb = n0 + 128 * hh + 32 * h;            // first column of this warp's box
      const bool has_cols = nb < p.N;
      if (Cfg::kHasIn) mbar_wait(&in_full[sb], (u >> 1) & 1);          // implies the buffer was free
      else if (u >= 2) mbar_wait(&stg_free[sb], ((u >> 1) - 1) & 1);
      if (warp == kTsFirstEpi && lane == 0) DBG_TS(6, (int)u);
      if (has_cols) {
        uint8_t* box = stg_ptr + sb * Cfg::kBuf + h * Cfg::kSlice + row_off;
        const uint32_t t_row = tmem_base + buf * kTsBN + ((uint32_t)(quad * 32) << 16) + (uint32_t)(128 * hh + 32 * h);
        const long long r = (long long)m0 + row;
        float dot = 0.f;       // TS_ROWDOT: <v, aux> over this thread's 32 columns (= one attention head at d_head 32)
#pragma unroll
        for (int c0 = 0; c0 < 32; c0 += 16) {
          uint32_t acc[16];
          tmem_ld16(t_row + (uint32_t)c0, acc);
          tmem_ld_wait();
          float v[16];
          if (p.bias) {
            if (nb + c0 + 16 <= p.N) {
#pragma unroll
              for (int j4 = 0; j4 < 4; ++j4) {
                const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + nb + c0) + j4);
                v[4 * j4 + 0] = __uint_as_float(acc[4 * j4 + 0]) + b4.x;
                v[4 * j4 + 1] = __uint_as_float(acc[4 * j4 + 1]) + b4.y;
                v[4 * j4 + 2] = __uint_as_float(acc[4 * j4 + 2]) + b4.z;
                v[4 * j4 + 3] = __uint_as_float(acc[4 * j4 + 3]) + b4.w;
              }
            } else {
#pragma unroll
              for (int j = 0; j < 16; ++j)
                v[j] = __uint_as_float(acc[j]) + ((nb + c0 + j < p.N) ? __ldg(p.bias + nb + c0 + j) : 0.f);
            }
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(acc[j]);
          }
          if (EPI == TS_F32) {
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4)
              *reinterpret_cast<float4*>(box + ((((uint32_t)(c0 >> 2) + j4) ^ swz) << 4)) =
                  make_float4(v[4 * j4], v[4 * j4 + 1], v[4 * j4 + 2], v[4 * j4 + 3]);
          } else {
            // bf16 outputs: two 16-byte chunks (8 elements each) per 16 columns
            if (EPI == TS_SOFTSIGN) {
#pragma unroll
              for (int j = 0; j < 16; ++j) v[j] = softsign(v[j]) * act_scale;
            }
            float d2[16];
            if (EPI == TS_GELU_DG) {
#pragma unroll
              for (int j = 0; j < 16; j += 2) gelu_erf_both2(v[j], v[j + 1], v[j], v[j + 1], d2[j], d2[j + 1]);
            }
            if (EPI == TS_GELU) {
              // the same evaluation as TS_GELU_DG, so D is bit for bit what that flavour writes; the derivative is dead
#pragma unroll
              for (int j = 0; j < 16; j += 2) {
                float g0, g1;
                gelu_erf_both2(v[j], v[j + 1], v[j], v[j + 1], g0, g1);
              }
            }
            uint4 wdrop = make_uint4(0u, 0u, 0u, 0u);
            if (EPI == TS_ROWDOT && drop)
              wdrop = drop_bytes16(seed, p.drop.site, (uint64_t)r, drop_gpr, (uint32_t)((nb + c0) >> 4));
#pragma unroll
            for (int q8 = 0; q8 < 2; ++q8) {
              uint4* q = reinterpret_cast<uint4*>(box + ((((uint32_t)(c0 >> 3) + q8) ^ swz) << 4));
              if (EPI == TS_ROWDOT) {
                const uint4 a4 = *q;                                  // attention output O, in place
                const uint32_t aw[4] = {a4.x, a4.y, a4.z, a4.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const float2 a2 = unpack_bf16x2(aw[e]);
                  dot = fmaf(v[8 * q8 + 2 * e], a2.x, dot);
                  dot = fmaf(v[8 * q8 + 2 * e + 1], a2.y, dot);
                }
                if (drop) {
#pragma unroll
                  for (int e = 0; e < 8; ++e)
                    v[8 * q8 + e] = (drop_byte(wdrop, 8 * q8 + e) < p.drop.thresh) ? 0.f : v[8 * q8 + e] * p.drop.scale;
                }
              }
              if (EPI == TS_MULAUX || EPI == TS_DSOFTSIGN) {
                const uint4 a4 = *q;                                  // saved tensor, in place
                const uint32_t aw[4] = {a4.x, a4.y, a4.z, a4.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const float2 a2 = unpack_bf16x2(aw[e]);
                  float f0 = a2.x, f1 = a2.y;
                  if (EPI == TS_DSOFTSIGN) {
                    const float t0 = 1.0f - fabsf(f0 * inv_scale), t1 = 1.0f - fabsf(f1 * inv_scale);
                    f0 = act_scale * t0 * t0;
                    f1 = act_scale * t1 * t1;
                  }
                  v[8 * q8 + 2 * e] *= f0;
                  v[8 * q8 + 2 * e + 1] *= f1;
                }
              }
              *q = make_uint4(pack_bf16x2(v[8 * q8], v[8 * q8 + 1]), pack_bf16x2(v[8 * q8 + 2], v[8 * q8 + 3]),
                              pack_bf16x2(v[8 * q8 + 4], v[8 * q8 + 5]), pack_bf16x2(v[8 * q8 + 6], v[8 * q8 + 7]));
              if (EPI == TS_GELU_DG)
                *reinterpret_cast<uint4*>(box + Cfg::kOut + ((((uint32_t)(c0 >> 3) + q8) ^ swz) << 4)) =
                    make_uint4(pack_bf16x2(d2[8 * q8], d2[8 * q8 + 1]), pack_bf16x2(d2[8 * q8 + 2], d2[8 * q8 + 3]),
                               pack_bf16x2(d2[8 * q8 + 4], d2[8 * q8 + 5]), pack_bf16x2(d2[8 * q8 + 6], d2[8 * q8 + 7]));
            }
          }
        }
        if (EPI == TS_ROWDOT && r < p.M) {
          const long long bb = r / p.rowdot_S;
          const int ii = (int)(r - bb * p.rowdot_S);
          p.rowdot[(bb * (p.N >> 5) + (nb >> 5)) * p.rowdot_S + ii] = dot;
        }
      }
      // staged box over to the store warp; after the last unit the accumulator buffer goes back to the MMA warp
      tc_fence_before();
      fence_proxy_async();          // generic-proxy writes -> visible to the TMA unit (async proxy)
      __syncwarp();
      if (lane == 0) {
        if (hh == NU - 1) mbar_arrive(&acc_empty[buf]);
        mbar_arrive(&stg_full[sb]);
        if (warp == kTsFirstEpi) DBG_TS(7, (int)u);
      }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) DBG_TS(7, 62);     // all roles done
#ifdef MMFM_DBG_TIMING
  if (threadIdx.x == 0 && blockIdx.x < 160) { __threadfence(); g_dbg_cta[blockIdx.x][1] = dbg_now(); }
#endif
  if (warp == 1) tmem_dealloc(tmem_base, 2u * BN);
}

}  // namespace mmfm

using namespace mmfm;

template <int EPI, int BN>
static int launch_ts_bn(const mmfm_gemm_args* a, cudaStream_t st) {
  using Cfg = TsCfg<EPI>;
  CUtensorMap tmA, tmB, tmD, tmD2, tmIn;
  memset(&tmD2, 0, sizeof(tmD2));
  memset(&tmIn, 0, sizeof(tmIn));
  int rc = make_tmap_bf16_2d(&tmA, a->A, (uint64_t)a->M, (uint64_t)a->K, (uint64_t)a->lda, kTsBK, kTsBM, TMA_SW_128);
  if (rc) return rc;
  rc = make_tmap_bf16_2d(&tmB, a->B, (uint64_t)a->N, (uint64_t)a->K, (uint64_t)a->ldb, kTsBK, BN, TMA_SW_128);
  if (rc) return rc;
  if (Cfg::kF32) rc = make_tmap_f32_2d(&tmD, a->D, (uint64_t)a->M, (uint64_t)a->N, (uint64_t)a->ldd, 32, 128, TMA_SW_128);
  else rc = make_tmap_bf16_2d(&tmD, a->D, (uint64_t)a->M, (uint64_t)a->N, (uint64_t)a->ldd, 32, 128, TMA_SW_64);
  if (rc) return rc;
  if (Cfg::kTwoOut) {
    rc = make_tmap_bf16_2d(&tmD2, a->D2, (uint64_t)a->M, (uint64_t)a->N, (uint64_t)a->ldd, 32, 128, TMA_SW_64);
    if (rc) return rc;
  }
  if (Cfg::kHasIn) rc = make_tmap_bf16_2d(&tmIn, a->aux, (uint64_t)a->M, (uint64_t)a->N, (uint64_t)a->ldaux, 32, 128, TMA_SW_64);
  if (rc) return rc;
  static bool attr_set = false;
  if (!attr_set) {
    MMFM_CHECK_CUDA(cudaFuncSetAttribute(gemm_tn_ts_kernel<EPI, BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTsMaxSmem));
    attr_set = true;
  }
  const int tiles_n = (a->N + BN - 1) / BN, tiles_m = (a->M + kTsBM - 1) / kTsBM;
  const int n_tiles = tiles_n * tiles_m;
  const int grid = n_tiles < device_sm_count() ? n_tiles : device_sm_count();
  // as many A + B stages as fit beside the two staging buffers (at most kTsMaxStages)
  const size_t stage = (size_t)(kTsBM + BN) * kTsBK * 2;
  const size_t room = (kTsMaxSmem - 1024 - 2 * (size_t)Cfg::kBuf) / stage;
  const int nst = room > (size_t)kTsMaxStages ? kTsMaxStages : (int)room;
  const size_t smem = 1024 + (size_t)nst * stage + 2 * (size_t)Cfg::kBuf;
  gemm_tn_ts_kernel<EPI, BN><<<grid, kTsThreads, smem, st>>>(tmA, tmB, tmD, tmD2, tmIn, *a, tiles_n, n_tiles, nst);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

// 256-wide tiles when N is a multiple of 256 (the model's 256 / 512 / 768-column projections)
template <int EPI>
static int launch_ts(const mmfm_gemm_args* a, cudaStream_t st) {
  if (a->N % 256 == 0) return launch_ts_bn<EPI, 256>(a, st);
  return launch_ts_bn<EPI, 128>(a, st);
}

namespace mmfm {

static bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// Returns 1 when the call was taken by the TMA-store kernel, 0 when it does not fit (the caller falls back to
// gemm_tn_kernel), < 0 on error.
int try_launch_gemm_ts(const mmfm_gemm_args* a, cudaStream_t st) {
  if (a->N <= 64 || a->N % 4 != 0 || a->remap_T > 0 || a->row_zero != nullptr) return 0;
  const bool f32 = a->d_fp32 != 0;
  const int esz = f32 ? 4 : 2;
  if (!al16(a->D) || (a->ldd * esz) % 16 != 0) return 0;
  if (a->bias && !al16(a->bias)) return 0;
  const bool drop = a->drop.thresh != 0;
  // fp32 + residual stays on gemm_tn_kernel: here it measured 2-3 us SLOWER (28.1 vs 26.4 us out-proj, 37.3 vs 34.4 us
  // down-proj, graph-timed): the residual box travels TMA -> shared memory -> registers -> shared memory -> TMA, twice
  // the shared-memory bytes of the staged epilogue, and shared-memory bandwidth is what the main loop competes for.
  if (a->res) return 0;
  if (drop && a->act != MMFM_ACT_ROWDOT_DROP) return 0;
  int epi = -1;
  switch (a->act) {
    case MMFM_ACT_NONE:
      if (a->D2) return 0;
      epi = f32 ? TS_F32 : TS_BF16;
      break;
    case MMFM_ACT_SOFTSIGN:
      if (f32 || a->D2) return 0;
      epi = TS_SOFTSIGN;
      break;
    case MMFM_ACT_GELU:
      if (f32 || a->D2) return 0;        // with D2 (the pre-activation) it stays on gemm_tn_kernel
      epi = TS_GELU;
      break;
    case MMFM_ACT_GELU_DG:
      if (f32 || !a->D2 || !al16(a->D2)) return 0;
      epi = TS_GELU_DG;
      break;
    case MMFM_ACT_MULAUX:
    case MMFM_ACT_DSOFTSIGN:
      if (f32 || a->D2 || !a->aux || !al16(a->aux) || (a->ldaux * 2) % 16 != 0) return 0;
      epi = a->act == MMFM_ACT_MULAUX ? TS_MULAUX : TS_DSOFTSIGN;
      break;
    case MMFM_ACT_ROWDOT_DROP:
      if (f32 || a->D2 || a->bias || !a->aux || !al16(a->aux) || (a->ldaux * 2) % 16 != 0 || a->N % 32 != 0 || !a->rowdot)
        return 0;
      epi = TS_ROWDOT;
      break;
    default:
      return 0;
  }
  int rc = 0;
  switch (epi) {
    case TS_BF16: rc = launch_ts<TS_BF16>(a, st); break;
    case TS_SOFTSIGN: rc = launch_ts<TS_SOFTSIGN>(a, st); break;
    case TS_F32: rc = launch_ts<TS_F32>(a, st); break;
    case TS_GELU: rc = launch_ts<TS_GELU>(a, st); break;
    case TS_GELU_DG: rc = launch_ts<TS_GELU_DG>(a, st); break;
    case TS_MULAUX: rc = launch_ts<TS_MULAUX>(a, st); break;
    case TS_DSOFTSIGN: rc = launch_ts<TS_DSOFTSIGN>(a, st); break;
    case TS_ROWDOT: rc = launch_ts<TS_ROWDOT>(a, st); break;
    default: return 0;
  }
  return rc == 0 ? 1 : rc;
}

}  // namespace mmfm
