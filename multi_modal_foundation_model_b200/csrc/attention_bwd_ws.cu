// Masked multi-head attention backward for the default model (d_head 32, Sq, Sk <= 256): persistent, WARP-SPECIALISED
// tcgen05 / TMEM kernel (autograd of F.scaled_dot_product_attention, reference src/multi_modal/mm_utils.py:105-112,
// :143-150).  One CTA per SM loops over (batch, head) items and computes dQ, dK and dV of an item in one go, so every
// score element goes through the softmax / dropout / dS arithmetic once.
//
// Mathematics: the forward computes O = P_drop V with P_drop = P . keep . s (s = 1 / (1 - dropout p)), so
// dP_drop = dO V^T and the softmax gradient is dS = P . (s keep . dP_drop - delta), where delta = rowsum(dO . O)
// = rowsum(P . dP) comes from the preparation step.  The factor s stays out of the inner loop: the passes compute
// dS / s = (P . keep) . dP_drop - P . (delta / s), and s is applied when dQ / dK / dV leave tensor memory.
//
// Data flow of an item: the key range is split into two 128-key halves, each with its own S / dP buffer in TMEM and its
// own barriers; per 128-query tile the passes run in the order A(h0) A(h1) B(h0) B(h1) and every MMA batch is issued
// right after the pass that produces its operands and waited for one pass later:
//   pass A(h)  p = exp2(s*scale - lse) under the mask, P_drop -> swizzled smem slab ; then  dP_h = dO V_h^T (over the
//              dead S_h), dV_h += P_drop_h^T dO
//   pass B(h)  dS -> the SAME slab (P_drop is dead by then) ; then  dQ += dS_h K_h, dK_h += dS_h^T Q, and the S_h of the
//              next query tile -- or of the NEXT ITEM
// The slabs are the canonical 128-byte-swizzled layout ([128 query rows] x [64 keys] per slab), written with 16-byte
// stores from registers, so one copy of dS serves both the dQ (K-major A) and the dK (MN-major A) products.  The
// operands (K, V, Q, dO) and the per-row side data (lse, delta, keep words -- bulk-copied to shared memory) of item n+1
// are loaded while item n computes.
//
// The block-synchronous form of this kernel took 12.7 us per item (globaltimer trace), of which only ~5.8 us were the
// four probability / dS passes.  Its three serialisations and what replaced them:
//   * the MMA batches were issued by math warp 0 between block-wide barriers, so every pass waited for that warp
//     (0.5 us per query tile)                     -> a dedicated issuer warp; passes hand over through mbarriers only
//   * after the last pass the CTA drained the tensor pipe, staged and copied the six output tiles out (2.4 us) and only
//     then started the next item (1.2 us prologue) -> the read-out of item n runs in the MIDDLE of item n+1 (after its
//     first two probability passes, when item n's products have long completed): dV is double-buffered in tensor memory
//     (512 columns in use), dQ / dK are not overwritten before the first dS pass of item n+1, and the tiles leave
//     through TMA stores issued by the loader warp from the retired operand stage
//   * masked / unmasked template copies of every pass (68 KB of SASS for a 32 KB instruction cache) -> one copy; a
//     chunk that carries a mask first overwrites its masked scores in registers
// Roles (576 threads): warps 0-15 math (thread = query row = TMEM lane; warp quadrant x four 32-key column groups),
// warp 16 tcgen05.mma issuer, warp 17 TMA loader / storer.  Two schedulers host five warps, so ptxas caps the kernel at
// 96 registers per thread.
//
// Measured on B200 (tools/attn_bench.py, default shape, dropout on, preparation kernel included): 201 us for the block-
// synchronous kernel -> 141 us (this structure) -> 135 us with the issuer's MMA batches unrolled (a rolled loop spends
// ~100 clocks of descriptor arithmetic per 41-clock MMA: tools/micro/umma_rate.cu) -> 132 us with every math thread
// arriving on the hand-over barriers itself (a warp-level sync + one elected arrival added latency).  What a globaltimer trace of this
// kernel (tools/micro/bwd_ws_timing.py) shows per item: probability passes at the MUFU bound (0.54 us per 128 x 128
// block = 16 exp2 per clock and SM), dS passes ~0.42 us, and about as much again in hand-over latency between passes.
// Variants that were built, verified and measured SLOWER, so they are not here: eight math warps with 168 registers
// (147 us: one or two warps per scheduler cannot cover the MUFU / tcgen05.ld latencies); two column groups that own one
// key half each and run one pass out of phase, with 8 or 16 math warps (157 - 187 us: same reason); 8-key work units dealt
// evenly to the column groups (the predicated unit bodies cost more instructions than the balance wins); a polynomial
// exp2 on the FMA pipe for a third of the pairs (142 us: packed FFMA2 saves issue slots, not pipe cycles); the product
// -p * delta moved into the probability pass (136 us); setmaxnreg
// (the register pool only holds what a warpgroup released: the math warps cannot get past 112, and a 32-register issuer
// spills inside its MMA batches).
#include "attn_common.cuh"

#ifdef MMFM_DBG_TIMING
__device__ long long g_dbg_ws[64];
#define DBG_WS(slot) do { if (blockIdx.x == 7 && it == 3 && threadIdx.x == 32) { long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_) :: "memory"); g_dbg_ws[slot] = t_; } } while (0)
extern "C" int mmfm_debug_read_bwd_ws(long long* out) {
  return (int)cudaMemcpyFromSymbol(out, g_dbg_ws, sizeof(long long) * 64);
}
#else
#define DBG_WS(slot) do { } while (0)
#endif

namespace mmfm {

constexpr int kWsThreads = 576;   // 18 warps x 112 registers fill the register file
constexpr int kWsMathWarps = 16, kWsMmaWarp = 16, kWsTmaWarp = 17;
constexpr uint32_t kWRow = 64;                       // bytes per operand row (32 bf16), 64-byte swizzle
constexpr uint32_t kWOp = 256 * kWRow;               // one operand buffer: 256 rows
constexpr uint32_t kWStage = 4 * kWOp;               // K, V, Q, dO  (retired stage = staging of the six output tiles)
constexpr uint32_t kWSide = 1024 + 1024 + 8192;      // lse, delta (256 floats each), keep words (256 rows x 4 x 8 B)
constexpr uint32_t kWsSmem = 1024 + 2 * kWStage + 4 * kSlabBytes + 2 * kWSide;
constexpr uint32_t kWTile = 128 * kWRow;             // one staged output tile: 128 rows x 32 bf16

MMFM_DEVINL void bulk_load_ws(uint32_t dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
MMFM_DEVINL void lds_v4(uint32_t addr, uint32_t& a, uint32_t& b, uint32_t& c, uint32_t& d) {
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(addr) : "memory");
}

template <bool DROP>
__global__ void __launch_bounds__(kWsThreads, 1) attn_bwd_ws_kernel(
    const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmdO,
    const __grid_constant__ CUtensorMap tmK, const __grid_constant__ CUtensorMap tmV,
    const __grid_constant__ CUtensorMap tmdQ, const __grid_constant__ CUtensorMap tmdK,
    const __grid_constant__ CUtensorMap tmdV, const AttnParams p, int npad, int n_items) {
  constexpr int D = 32;
  constexpr uint32_t kSbo64 = 512;
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t ld_bar[2], s_bar[2], dp_bar[2], pa_bar[2], ds_bar[2], done_bar, staged_bar;
  __shared__ uint32_t tmem_slot;

  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_al = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t sSlab = smem_base + 2 * kWStage;                 // 4 slabs: P_drop, then dS (64 keys x 128 query rows each)
  const uint32_t side_off = 2 * kWStage + 4 * kSlabBytes;         // byte offset of the side-data stages
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int nqt = (p.Sq + 127) >> 7;
  const int nkh = (npad + 127) >> 7;                 // 128-key halves
  const int wlast = npad - 128 * (nkh - 1);          // width of the last half (multiple of 16)
  const int nch = (npad + 31) >> 5;
  const int nkb = (p.Sk + kTile - 1) / kTile;
  const int my_items = (n_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (tid == 0) {
    tma_prefetch_desc(&tmQ); tma_prefetch_desc(&tmdO); tma_prefetch_desc(&tmK); tma_prefetch_desc(&tmV);
    tma_prefetch_desc(&tmdQ); tma_prefetch_desc(&tmdK); tma_prefetch_desc(&tmdV);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&ld_bar[i], 1);
      mbar_init(&s_bar[i], 1);
      mbar_init(&dp_bar[i], 1);
      mbar_init(&pa_bar[i], kWsMathWarps * 32);
      mbar_init(&ds_bar[i], kWsMathWarps * 32);
    }
    mbar_init(&done_bar, 1);
    mbar_init(&staged_bar, kWsMathWarps);
    fence_mbar_init();
  }
  if (warp == kWsMmaWarp) {
    tmem_alloc(&tmem_slot, 512u);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;
  constexpr uint32_t dq_col = 256u, dk_col = 320u, dv_col = 384u;   // dV: 384 + 64 * (item parity) + 32 * half

  if (warp >= kWsMathWarps) {
    if (warp == kWsTmaWarp) {
      // ------------------------------------------------ loader / storer ------------------------------------------------
      if (lane == 0) {
        const uint32_t lse_bytes = (uint32_t)p.Sq * 4u, keep_bytes = DROP ? (uint32_t)p.Sq * (uint32_t)nkb * 8u : 0u;
        const uint32_t tx_bytes = (uint32_t)(2 * npad) * kWRow + 2u * kWOp + 2u * lse_bytes + keep_bytes;
        auto issue_loads = [&](int item, int st) {
          const int b = item / p.nh, h = item - b * p.nh;
          const long long bh = (long long)item;
          const uint32_t base = smem_base + st * kWStage;
          mbar_arrive_expect_tx(&ld_bar[st], tx_bytes);
          tma_load_2d_addr(base, &tmK, &ld_bar[st], h * D, b * p.Sk);
          tma_load_2d_addr(base + kWOp, &tmV, &ld_bar[st], h * D, b * p.Sk);
          tma_load_2d_addr(base + 2 * kWOp, &tmQ, &ld_bar[st], h * D, b * p.Sq);
          tma_load_2d_addr(base + 2 * kWOp + 128 * kWRow, &tmQ, &ld_bar[st], h * D, b * p.Sq + 128);
          tma_load_2d_addr(base + 3 * kWOp, &tmdO, &ld_bar[st], h * D, b * p.Sq);
          tma_load_2d_addr(base + 3 * kWOp + 128 * kWRow, &tmdO, &ld_bar[st], h * D, b * p.Sq + 128);
          const uint32_t side = smem_base + side_off + st * kWSide;
          bulk_load_ws(side, p.lse + bh * p.Sq, lse_bytes, &ld_bar[st]);
          bulk_load_ws(side + 1024, p.delta + bh * p.Sq, lse_bytes, &ld_bar[st]);
          if (DROP) bulk_load_ws(side + 2048, p.p_keep + bh * p.Sq * nkb * 4, keep_bytes, &ld_bar[st]);
        };
        if (my_items > 0) issue_loads((int)blockIdx.x, 0);
        if (my_items > 1) issue_loads((int)blockIdx.x + (int)gridDim.x, 1);
        for (int it = 0; it < my_items; ++it) {
          const int item = (int)blockIdx.x + it * (int)gridDim.x;
          const int b = item / p.nh, h = item - b * p.nh;
          const uint32_t stage = smem_base + (uint32_t)(it & 1) * kWStage;
          mbar_wait_relaxed(&staged_bar, (uint32_t)(it & 1));     // the six tiles of item `it` sit in its retired stage
          for (int qt = 0; qt < nqt; ++qt) tma_store_3d(&tmdQ, stage + (uint32_t)qt * kWTile, h * D, qt * 128, b);
          for (int kh = 0; kh < nkh; ++kh) {
            tma_store_3d(&tmdK, stage + (uint32_t)(2 + 2 * kh) * kWTile, h * D, kh * 128, b);
            tma_store_3d(&tmdV, stage + (uint32_t)(3 + 2 * kh) * kWTile, h * D, kh * 128, b);
          }
          bulk_commit_group();
          if (it + 2 < my_items) {
            bulk_wait_group_read<0>();                            // the stage may be overwritten
            issue_loads(item + 2 * (int)gridDim.x, it & 1);
          }
        }
        bulk_wait_group<0>();
      }
      __syncwarp();
    } else if (warp == kWsMmaWarp) {
      // ------------------------------------------------ MMA issuer ------------------------------------------------------
      if (elect_one()) {
        const uint32_t idesc_q = make_idesc_bf16(128, D, 0, 1);   // dQ: A K-major (slabs), B MN-major (K tile)
        const uint32_t idesc_t = make_idesc_bf16(128, D, 1, 1);   // dK / dV: A MN-major (slabs), B MN-major
        auto issue_s = [&](int st, int qt, int kh) {     // S_h = Q_qt K_h^T -> buffer kh
          const uint32_t base = smem_base + st * kWStage;
          const uint32_t n = (uint32_t)(kh == nkh - 1 ? wlast : 128);
          const uint32_t idesc = make_idesc_bf16(128, n, 0, 0);
          const uint32_t aq = base + 2 * kWOp + (uint32_t)qt * 128u * kWRow, bk = base + (uint32_t)kh * 128u * kWRow;
#pragma unroll
          for (int k = 0; k < D / 16; ++k)
            umma_bf16(tmem_base + 128u * kh, make_smem_desc(aq + k * 32, 16, kSbo64, 4),
                      make_smem_desc(bk + k * 32, 16, kSbo64, 4), idesc, k > 0 ? 1u : 0u);
          umma_commit(&s_bar[kh]);
        };
        auto issue_dp_dv = [&](int st, int qt, int kh, uint32_t dvc) {  // dP_h = dO_qt V_h^T over S_h ; dV_h += P_drop_h^T dO_qt
          const uint32_t base = smem_base + st * kWStage;
          const uint32_t n = (uint32_t)(kh == nkh - 1 ? wlast : 128);
          const uint32_t idesc = make_idesc_bf16(128, n, 0, 0);
          const uint32_t ad = base + 3 * kWOp + (uint32_t)qt * 128u * kWRow, bv = base + kWOp + (uint32_t)kh * 128u * kWRow;
#pragma unroll
          for (int k = 0; k < D / 16; ++k)
            umma_bf16(tmem_base + 128u * kh, make_smem_desc(ad + k * 32, 16, kSbo64, 4),
                      make_smem_desc(bv + k * 32, 16, kSbo64, 4), idesc, k > 0 ? 1u : 0u);
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
            umma_bf16(tmem_base + dvc + 32u * kh,
                      make_smem_desc(sSlab + (uint32_t)(2 * kh) * kSlabBytes + (uint32_t)kk * 2048u, kSlabBytes, 1024, 2),
                      make_smem_desc(ad + (uint32_t)kk * 16u * kWRow, kSbo64, kSbo64, 4), idesc_t, (qt > 0 || kk > 0) ? 1u : 0u);
          umma_commit(&dp_bar[kh]);
        };
        auto issue_dq_dk = [&](int st, int qt, int kh) {  // dQ_qt += dS_h K_h ; dK_h += dS_h^T Q_qt
          const uint32_t base = smem_base + st * kWStage;
          const int nks = (kh == nkh - 1 ? wlast : 128) >> 4;
          const uint32_t aq = base + 2 * kWOp + (uint32_t)qt * 128u * kWRow;
#pragma unroll 8
          for (int k2 = 0; k2 < nks; ++k2) {
            const int kk = 8 * kh + k2;           // 16-key step inside the whole key range
            umma_bf16(tmem_base + dq_col + 32u * qt,
                      make_smem_desc(sSlab + (uint32_t)(kk >> 2) * kSlabBytes + (uint32_t)(kk & 3) * 32u, 16, 1024, 2),
                      make_smem_desc(base + (uint32_t)kk * 16u * kWRow, kSbo64, kSbo64, 4), idesc_q, (kh > 0 || k2 > 0) ? 1u : 0u);
          }
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
            umma_bf16(tmem_base + dk_col + 32u * kh,
                      make_smem_desc(sSlab + (uint32_t)(2 * kh) * kSlabBytes + (uint32_t)kk * 2048u, kSlabBytes, 1024, 2),
                      make_smem_desc(aq + (uint32_t)kk * 16u * kWRow, kSbo64, kSbo64, 4), idesc_t, (qt > 0 || kk > 0) ? 1u : 0u);
        };

        uint32_t ph = 0;
        for (int it = 0; it < my_items; ++it) {
          const int st = it & 1;
          const uint32_t dvc = dv_col + 64u * (uint32_t)(it & 1);
          const bool has_next = it + 1 < my_items;
          if (it == 0) {
            mbar_wait_relaxed(&ld_bar[0], 0u);
            tc_fence_after();
            for (int kh = 0; kh < nkh; ++kh) issue_s(0, 0, kh);
          }
          for (int qt = 0; qt < nqt; ++qt, ++ph) {
            const uint32_t par = ph & 1u;
            const bool last_q = (qt + 1 == nqt);
            for (int kh = 0; kh < nkh; ++kh) {
              mbar_wait(&pa_bar[kh], par);      // P_drop of this half is in its slabs, S_h has been read
              tc_fence_after();
              issue_dp_dv(st, qt, kh, dvc);
            }
            for (int kh = 0; kh < nkh; ++kh) {
              mbar_wait(&ds_bar[kh], par);      // dS of this half is in its slabs, dP_h has been read (and, at the first
              tc_fence_after();                 // pass of an item, the previous item's accumulators have been read out)
              issue_dq_dk(st, qt, kh);
              if (last_q && kh == nkh - 1) umma_commit(&done_bar);      // every product of this item is issued
              if (!last_q) {
                issue_s(st, qt + 1, kh);                                 // its commit also covers the batch above
              } else if (has_next) {
                if (kh == 0) {
                  mbar_wait_relaxed(&ld_bar[st ^ 1], (uint32_t)(((it + 1) >> 1) & 1));
                  tc_fence_after();
                }
                issue_s(st ^ 1, 0, kh);
              }
            }
          }
        }
      }
      __syncwarp();
    }
  } else {
    // -------------------------------------------------- math warps ------------------------------------------------------
    const int quad = warp & 3, grp = warp >> 2;
    const int row = quad * 32 + lane;
    const int mode = p.mask_mode;
    const float sl2 = p.scale * kLog2e;
    const float dsc = DROP ? p.drop_p.scale : 1.0f;
    const float inv_dsc = 1.0f / dsc;
    const uint32_t t_row = tmem_base + ((uint32_t)(quad * 32) << 16);
    const uint64_t sl2x2 = pack_f2(sl2, sl2);
    const uint32_t slab_row = sSlab + (uint32_t)row * 128u;
    const uint32_t swz = (uint32_t)(row & 7);

    // key-validity bytes of this warp's two 32-key chunks (c = grp, grp + 4), fetched one item ahead
    auto kv_fetch = [&](int item, uint32_t (&v)[2]) {
      const int b = item / p.nh;
      const unsigned char* kvg = p.key_valid + (long long)b * p.Sk;
#pragma unroll
      for (int kh = 0; kh < 2; ++kh) {
        const int j = (grp + 4 * kh) * 32 + lane;
        v[kh] = (j < p.Sk) ? ((mode == MMFM_MASK_CAUSAL) ? 1u : (uint32_t)kvg[j]) : 0u;
      }
    };

    // read-out of a finished item: 16-column pieces over the 4 thread groups
    //   piece 0..3   : dQ of query tile piece/2, column half piece&1          (TMEM lane = query row)
    //   piece 4..11  : (kh, which, half) = ((piece-4)/4, ((piece-4)/2)&1, (piece-4)&1); which 0 dK, 1 dV (lane = key row)
    // staged as six [128 rows][32 bf16] tiles in the TMA 64-byte-swizzle layout inside the item's retired operand stage
    auto read_out = [&](int rit) {
      mbar_wait(&done_bar, (uint32_t)(rit & 1));
      tc_fence_after();
      const uint32_t dvc = dv_col + 64u * (uint32_t)(rit & 1);
      const uint32_t stage = smem_base + (uint32_t)(rit & 1) * kWStage;
      const uint32_t sw4 = (uint32_t)((row >> 1) & 3);
#pragma unroll
      for (int u = 0; u < 3; ++u) {       // one piece at a time: the probabilities of the running item stay in registers
        const int piece = grp + 4 * u;
        uint32_t col;
        int tile, half;
        float fs;
        if (piece < 4) {
          col = dq_col + 32u * (piece >> 1) + 16u * (piece & 1);
          tile = piece >> 1; half = piece & 1; fs = p.scale * dsc;
        } else {
          const int q = piece - 4, kh = q >> 2, which = (q >> 1) & 1;
          col = (which ? dvc : dk_col) + 32u * kh + 16u * (q & 1);
          tile = 2 + 2 * kh + which; half = q & 1; fs = which ? dsc : p.scale * dsc;
        }
        uint32_t r[16];
        tmem_ld16(t_row + col, r);
        tmem_ld_wait();
        const uint32_t dst = stage + (uint32_t)tile * kWTile + (uint32_t)row * kWRow;
#pragma unroll
        for (int k8 = 0; k8 < 2; ++k8) {
          const int k = 8 * k8;
          st_shared_v4(dst + ((((uint32_t)(2 * half + k8)) ^ sw4) << 4),
                       pack_bf16x2(__uint_as_float(r[k]) * fs, __uint_as_float(r[k + 1]) * fs),
                       pack_bf16x2(__uint_as_float(r[k + 2]) * fs, __uint_as_float(r[k + 3]) * fs),
                       pack_bf16x2(__uint_as_float(r[k + 4]) * fs, __uint_as_float(r[k + 5]) * fs),
                       pack_bf16x2(__uint_as_float(r[k + 6]) * fs, __uint_as_float(r[k + 7]) * fs));
        }
      }
      tc_fence_before();
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&staged_bar);
    };

    uint32_t kvb[2] = {0u, 0u};
    if (my_items > 0) kv_fetch((int)blockIdx.x, kvb);
    uint32_t ph = 0;
#pragma unroll 1
    for (int it = 0; it < my_items; ++it) {
      const int item = (int)blockIdx.x + it * (int)gridDim.x;
      const int st = it & 1;
      uint32_t colbits[2];
      colbits[0] = __ballot_sync(0xffffffffu, kvb[0] != 0u);
      colbits[1] = __ballot_sync(0xffffffffu, kvb[1] != 0u);
      if (it + 1 < my_items) kv_fetch(item + (int)gridDim.x, kvb);
      DBG_WS(0);
      mbar_wait(&ld_bar[st], (uint32_t)((it >> 1) & 1));   // side data of this item have landed
      DBG_WS(1);
      const float* s_lse = reinterpret_cast<const float*>(smem_al + side_off + st * kWSide);
      const float* s_dl = s_lse + 256;
      const uint8_t* s_keep = smem_al + side_off + st * kWSide + 2048;

#pragma unroll 1
      for (int qt = 0; qt < nqt; ++qt, ++ph) {
        const uint32_t par = ph & 1u;
        const int i = qt * 128 + row;
        const bool rok = i < p.Sq;
        // a warp whose 32 query rows all lie past Sq (S = 200: the last quadrant of the second tile) only zeroes its part
        // of the slabs: the probability passes are MUFU-bound, so every dead row skipped is time won
        const bool dead = qt * 128 + quad * 32 >= p.Sq;
        float lse2 = INFINITY, ndl = 0.f;
        if (rok) {
          const float l = s_lse[i];
          lse2 = (l == -INFINITY) ? INFINITY : l * kLog2e;   // a fully masked row has no probabilities at all
          ndl = -s_dl[i] * inv_dsc;
        }
        const uint64_t nlse2x2 = pack_f2(-lse2, -lse2), ndlx2 = pack_f2(ndl, ndl);
        uint32_t aws[2] = {0u, 0u};
#pragma unroll
        for (int kh = 0; kh < 2; ++kh) {
          const int c = grp + 4 * kh;
          uint32_t aw = colbits[kh];
          const int rel = i - 32 * c;
          if (mode == MMFM_MASK_KEY_OR_DIAG) {
            if (rel >= 0 && rel < 32 && i < p.Sk) aw |= 1u << rel;
          } else if (mode == MMFM_MASK_CAUSAL) {
            aw &= (rel >= 31) ? 0xFFFFFFFFu : (rel < 0 ? 0u : ((2u << rel) - 1u));
          }
          aws[kh] = aw;
        }
        uint32_t pk[2][16];    // p as packed bf16, kept for the dS pass (p * keep is read back from the slab)

        // ---------------- pass A (both halves): probabilities ----------------
#pragma unroll
        for (int kh = 0; kh < 2; ++kh) {
          if (kh >= nkh) break;
          const int c = grp + 4 * kh;
          DBG_WS(4 + 16 * qt + 4 * kh);
          mbar_wait(&s_bar[kh], par);
          tc_fence_after();
          DBG_WS(5 + 16 * qt + 4 * kh);
          if (c < nch && dead) {
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4)
              st_shared_v4(slab_row + (uint32_t)(c >> 1) * kSlabBytes + ((((uint32_t)((c & 1) * 4 + q4)) ^ swz) << 4), 0u, 0u, 0u, 0u);
          } else if (c < nch) {
            uint32_t rs[32];
            tmem_ld32(t_row + 32u * c, rs);
            uint32_t km[4][2] = {{0u, 0u}, {0u, 0u}, {0u, 0u}, {0u, 0u}};
            if (DROP) {
              uint2 w2 = make_uint2(0xFFFFFFFFu, 0xFFFFFFFFu);
              if (rok) w2 = *reinterpret_cast<const uint2*>(s_keep + ((size_t)i * nkb + (c >> 1)) * 8);
              const int sh = 8 * (c & 1);   // second 32-column chunk of the 64-key block: n-tiles 4..7 -> bits 8..15
              keep_msb_words((w2.x & 0xFFFFu) >> sh, km[0]);
              keep_msb_words((w2.x >> 16) >> sh, km[1]);
              keep_msb_words((w2.y & 0xFFFFu) >> sh, km[2]);
              keep_msb_words((w2.y >> 16) >> sh, km[3]);
            }
            const uint32_t aw = aws[kh];
            tmem_ld_wait();
            if (__any_sync(0xffffffffu, aw != 0xFFFFFFFFu)) {   // masked columns may hold stale TMEM bits: overwrite, never multiply
#pragma unroll
              for (int k = 0; k < 32; ++k)
                if (!((aw >> k) & 1u)) rs[k] = 0xFF800000u;   // -inf -> probability 0
            }
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4) {
              uint32_t pd[4];
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                const int T = 4 * q4 + u;   // pair T of the chunk = columns 2T, 2T+1: n-tile n = T/4, quad lane ql = T%4
                float x0, x1;
                unpack_f2(ffma2(pack_f2(__uint_as_float(rs[2 * T]), __uint_as_float(rs[2 * T + 1])), sl2x2, nlse2x2), x0, x1);
                const uint32_t pp = pack_bf16x2(fast_exp2(x0), fast_exp2(x1));
                pk[kh][T] = pp;
                pd[u] = DROP ? (pp & prmt_b(km[T & 3][(T >> 2) >> 1], ((T >> 2) & 1) ? 0xBBAAu : 0x9988u)) : pp;
              }
              const int j16 = (c & 1) * 4 + q4;
              st_shared_v4(slab_row + (uint32_t)(c >> 1) * kSlabBytes + ((((uint32_t)j16) ^ swz) << 4), pd[0], pd[1], pd[2], pd[3]);
            }
          }
          DBG_WS(6 + 16 * qt + 4 * kh);
          fence_proxy_async();
          tc_fence_before();
          mbar_arrive(&pa_bar[kh]);
        }

        // the previous item's accumulators: its products completed long ago; dQ / dK are first overwritten by the
        // products of the dS pass below, the dV of this item accumulate in the other half of the dV columns
        if (qt == 0 && it > 0) read_out(it - 1);

        // ---------------- pass B (both halves): dS into the slab P_drop just left ----------------
#pragma unroll
        for (int kh = 0; kh < 2; ++kh) {
          if (kh >= nkh) break;
          const int c = grp + 4 * kh;
          DBG_WS(12 + 16 * qt + 4 * kh);
          mbar_wait(&dp_bar[kh], par);   // dP_h is there, and the dV product has finished reading this half's slabs
          tc_fence_after();
          DBG_WS(13 + 16 * qt + 4 * kh);
          if (c < nch && !dead) {          // (a dead warp's slab rows already hold zeros = its dS)
            uint32_t rd[32];
            tmem_ld32(t_row + 32u * c, rd);
            const uint32_t aw = aws[kh];
            tmem_ld_wait();
            if (__any_sync(0xffffffffu, aw != 0xFFFFFFFFu)) {
#pragma unroll
              for (int k = 0; k < 32; ++k)
                if (!((aw >> k) & 1u)) rd[k] = 0u;
            }
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4) {
              const int j16 = (c & 1) * 4 + q4;
              const uint32_t addr = slab_row + (uint32_t)(c >> 1) * kSlabBytes + ((((uint32_t)j16) ^ swz) << 4);
              uint32_t pd[4], ds[4];
              lds_v4(addr, pd[0], pd[1], pd[2], pd[3]);
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                const int T = 4 * q4 + u;
                const uint32_t pp = pk[kh][T];
                const uint64_t t2 = fmul2(pack_f2(__uint_as_float(pp << 16), __uint_as_float(pp & 0xFFFF0000u)), ndlx2);
                float s0, s1;
                unpack_f2(ffma2(pack_f2(__uint_as_float(pd[u] << 16), __uint_as_float(pd[u] & 0xFFFF0000u)),
                                pack_f2(__uint_as_float(rd[2 * T]), __uint_as_float(rd[2 * T + 1])), t2), s0, s1);
                ds[u] = pack_bf16x2(s0, s1);
              }
              st_shared_v4(addr, ds[0], ds[1], ds[2], ds[3]);
            }
          }
          DBG_WS(14 + 16 * qt + 4 * kh);
          fence_proxy_async();
          tc_fence_before();
          mbar_arrive(&ds_bar[kh]);
        }
      }
    }
    if (my_items > 0) read_out(my_items - 1);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kWsMmaWarp) tmem_dealloc(tmem_base, 512u);
}

}  // namespace mmfm

using namespace mmfm;

namespace mmfm {
int launch_attn_bwd_ws(const mmfm_attn_args* a, const AttnParams& p, cudaStream_t st) {
  constexpr int D = 32;
  const int npk = (a->Sk + 15) / 16 * 16;
  const uint64_t width = (uint64_t)a->n_heads * D;
  const bool drop = a->drop_p.thresh != 0u;
  CUtensorMap tq, tdo, tk, tv, tdq, tdk, tdv;
  if (int rc = make_tmap_bf16_2d(&tq, a->q, (uint64_t)a->B * a->Sq, width, (uint64_t)a->ldq, D, 128, TMA_SW_64)) return rc;
  if (int rc = make_tmap_bf16_2d(&tdo, a->d_o, (uint64_t)a->B * a->Sq, width, (uint64_t)a->lddo, D, 128, TMA_SW_64)) return rc;
  if (int rc = make_tmap_bf16_2d(&tk, a->k, (uint64_t)a->B * a->Sk, width, (uint64_t)a->ldk, D, npk, TMA_SW_64)) return rc;
  if (int rc = make_tmap_bf16_2d(&tv, a->v, (uint64_t)a->B * a->Sk, width, (uint64_t)a->ldv, D, npk, TMA_SW_64)) return rc;
  if (int rc = make_tmap_bf16_3d(&tdq, a->dq, (uint64_t)a->B, (uint64_t)a->Sq, width, (uint64_t)a->lddq, D, 128, TMA_SW_64)) return rc;
  if (int rc = make_tmap_bf16_3d(&tdk, a->dk, (uint64_t)a->B, (uint64_t)a->Sk, width, (uint64_t)a->lddk, D, 128, TMA_SW_64)) return rc;
  if (int rc = make_tmap_bf16_3d(&tdv, a->dv, (uint64_t)a->B, (uint64_t)a->Sk, width, (uint64_t)a->lddv, D, 128, TMA_SW_64)) return rc;
  static bool attr_set = false;
  if (!attr_set) {
    MMFM_CHECK_CUDA(cudaFuncSetAttribute(attn_bwd_ws_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWsSmem));
    MMFM_CHECK_CUDA(cudaFuncSetAttribute(attn_bwd_ws_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWsSmem));
    attr_set = true;
  }
  const int n_items = a->B * a->n_heads;
  int grid = device_sm_count();
  if (grid > n_items) grid = n_items;
  if (drop) attn_bwd_ws_kernel<true><<<grid, kWsThreads, kWsSmem, st>>>(tq, tdo, tk, tv, tdq, tdk, tdv, p, npk, n_items);
  else attn_bwd_ws_kernel<false><<<grid, kWsThreads, kWsSmem, st>>>(tq, tdo, tk, tv, tdq, tdk, tdv, p, npk, n_items);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}
}  // namespace mmfm
