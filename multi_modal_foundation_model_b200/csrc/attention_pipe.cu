// Masked multi-head attention forward, persistent warp-specialised tcgen05 / TMEM kernel for any sequence length
// (reference src/multi_modal/mm_utils.py:105-112 self-attention, :143-150 cross-attention; same contract as
// attention.cu, whose header describes the mask descriptors and the dropout stream).
//
// One CTA per SM, looping over work items (batch, head, pair of 128-query tiles A/B).  Roles:
//   warps 0-7   softmax of tile A: thread = query row = TMEM lane; two column groups of 4 warps own alternate 64-column
//               blocks of the row (more math warps per scheduler) and exchange row max / sum through shared memory
//   warps 8-15  softmax of tile B
//   warp  16    tcgen05.mma issuer (one elected lane)
//   warp  17    TMA producer: Q tile pairs (2-stage ring) and K/V blocks (kKvStages-stage ring); its 32 lanes also pack
//               the key-validity bytes of the item's batch entry into bits
// Tensor memory (512 columns): S_A | S_B | O_A | O_B.  Per key block j of a tile:
//   MMA      S = Q K_j^T                                   -> s_full
//   softmax  row max over the block (tcgen05.ld in 32-column chunks), running max / sum update, O rescale when the
//            max moved (only then), p = exp2(s*scale - max), probability dropout on the packed bf16 pairs,
//            tcgen05.st of P over the consumed part of S            -> p_ready
//   MMA      O (+)= P V_j  (A operand read from TMEM, V as MN-major smem operand)   -> pv_done ; then S of the NEXT
//            step of this tile is issued at once, so the two tiles' softmax phases and the tensor pipe overlap
// After the last block the softmax warps normalise O, apply output dropout and store bf16 rows + LSE; this epilogue
// runs while the MMA warp is already computing the next item's scores.  When the whole key range fits the S buffer
// (Sk <= 224 at d_head 32: the model's S = 200) there is one block per item and the softmax is a single exact pass.
// The dropout field and the stored keep words are bit-identical to attention.cu's kernels (same Philox calls).
#include "attn_common.cuh"
#include <stdlib.h>

#ifdef MMFM_DBG_TIMING
__device__ long long g_dbg_p[8][64];
#define DBG_P(slot) do { if (blockIdx.x == 5 && it == 3 && lane == 0 && (warp & 3) == 1) g_dbg_p[warp >> 2][slot] = clock64(); } while (0)
extern "C" int mmfm_debug_read_pipe(long long* out, int n) {
  return (int)cudaMemcpyFromSymbol(out, g_dbg_p, sizeof(long long) * (n < 512 ? n : 512));
}
#else
#define DBG_P(slot) do { } while (0)
#endif

namespace mmfm {

constexpr int kPipeThreads = 576;   // 16 softmax warps + MMA issuer + TMA producer
constexpr int kMmaWarp = 16, kTmaWarp = 17;
constexpr int kKvStages = 3;
constexpr int kMaxColWords = 512;   // key-validity bits: Sk <= 16384

template <int D>
struct PipeCfg {
  static constexpr uint32_t kRowBytes = D * 2;                  // 64 (64B swizzle) or 128 (128B swizzle)
  static constexpr uint32_t kLayout = (D == 32) ? 4u : 2u;      // UMMA smem-descriptor swizzle code
  static constexpr uint32_t kSbo = 8 * kRowBytes;               // 8-row swizzle atom
  static constexpr int kSW = (512 - 2 * D) / 2;                 // width of one S buffer: 224 (D=32) / 192 (D=64)
  static constexpr uint32_t kQTile = 128 * kRowBytes;           // one 128-row query tile
  static constexpr uint32_t kQStage = 2 * kQTile;
  static constexpr uint32_t kKvHalf = (uint32_t)kSW * kRowBytes;   // room for the widest key block
  static constexpr uint32_t kKvStage = 2 * kKvHalf;
  static constexpr uint32_t kSmem = 1024 + 2 * kQStage + kKvStages * kKvStage;
};

// prmt with the sign-replicating selector mode (selector nibble bit 3): result byte = 0xFF / 0x00 from the msb of the
// selected source byte
MMFM_DEVINL uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
  uint32_t d;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
  return d;
}

MMFM_DEVINL void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// msb of byte k of the result = (byte k of x >= thresh); c4 / le128 from keep_consts()
MMFM_DEVINL uint32_t keep_msb(uint32_t x, uint32_t c4, bool le128) {
  const uint32_t y = (x & 0x7F7F7F7Fu) + c4;
  return le128 ? (x | y) : (x & y);
}
// 16 keep bits (bit b = byte b kept) from four msb-form words
MMFM_DEVINL uint32_t msb_bits16(uint32_t m0, uint32_t m1, uint32_t m2, uint32_t m3) {
  const uint32_t k = 0x00204081u;
  return (((m0 & 0x80808080u) * k) >> 28) | ((((m1 & 0x80808080u) * k) >> 24) & 0xF0u) |
         ((((m2 & 0x80808080u) * k) >> 20) & 0xF00u) | ((((m3 & 0x80808080u) * k) >> 16) & 0xF000u);
}

// One 32-column chunk of a score row -> probabilities: p = exp2(s * sl2 - base) under the mask, row-sum update, packed
// bf16 pairs with the probability-dropout keep masks applied.  MASKED is chosen per chunk by a warp vote so that the
// common unmasked chunk carries no predicate instructions at all.
template <bool MASKED, bool DROP, int HF>
MMFM_DEVINL void softmax_chunk(const uint32_t (&r)[32], uint32_t aw, float sl2, float base, float& l,
                               const uint32_t (&mw)[4][4], uint32_t (&pk)[16]) {
  float l0 = 0.f, l1 = 0.f;
#pragma unroll
  for (int t = 0; t < 16; ++t) {
    float e0 = fast_exp2(fmaf(__uint_as_float(r[2 * t]), sl2, -base));
    float e1 = fast_exp2(fmaf(__uint_as_float(r[2 * t + 1]), sl2, -base));
    if (MASKED) {   // select, never multiply: masked columns may hold stale TMEM bits
      if (!((aw >> (2 * t)) & 1u)) e0 = 0.f;
      if (!((aw >> (2 * t + 1)) & 1u)) e1 = 0.f;
    }
    l0 += e0;
    l1 += e1;
    pk[t] = pack_bf16x2(e0, e1);
  }
  l += l0 + l1;
  if (DROP) {
    // pair t covers columns 32c + 2t, +1: n-tile n = 4*hf + t/4, quad lane ql = t%4 -> bytes 2n, 2n+1 of call ql =
    // word 2*hf + t/8, byte pair (t/4)&1; prmt replicates the msb of the selected byte over its half of the mask
#pragma unroll
    for (int t = 0; t < 16; ++t) {
      const uint32_t word = mw[t & 3][2 * HF + (t >> 3)];
      pk[t] &= prmt(word, 0u, ((t >> 2) & 1) ? 0xBBAAu : 0x9988u);
    }
  }
}

template <bool MASKED>
MMFM_DEVINL float chunk_max(const uint32_t (&r)[32], uint32_t aw, float bm) {
  if (!MASKED) {
#pragma unroll
    for (int k = 0; k < 32; k += 2) bm = fmaxf(bm, fmaxf(__uint_as_float(r[k]), __uint_as_float(r[k + 1])));
  } else {
#pragma unroll
    for (int k = 0; k < 32; ++k)
      if ((aw >> k) & 1u) bm = fmaxf(bm, __uint_as_float(r[k]));
  }
  return bm;
}

template <int D, bool DROP>
__global__ void __launch_bounds__(kPipeThreads, 1) attn_fwd_pipe_kernel(const __grid_constant__ CUtensorMap tmQ,
                                                                       const __grid_constant__ CUtensorMap tmK,
                                                                       const __grid_constant__ CUtensorMap tmV,
                                                                       const AttnParams p, int bn, int nb, int n_qp,
                                                                       int n_items) {
  using Cfg = PipeCfg<D>;
  constexpr uint32_t kRowBytes = Cfg::kRowBytes, kLayout = Cfg::kLayout, kSbo = Cfg::kSbo;
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t q_full[2], q_empty[2], kv_full[kKvStages], kv_empty[kKvStages];
  __shared__ __align__(8) uint64_t s_full[2], p_ready[2], pv_done[2];
  __shared__ uint32_t tmem_slot;
  __shared__ uint32_t s_colbits[2][kMaxColWords];
  __shared__ float s_red[2][2][2][128];   // [tile][step parity][column group][row]: block maxima
  __shared__ float s_sum[2][2][2][128];   // [tile][item parity][column group][row]: row sums

  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sQ = smem_base, sKV = sQ + 2 * Cfg::kQStage;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int bl = ((p.Sk - (nb - 1) * bn) + 15) & ~15;   // width of the last key block (multiple of 16)

  if (tid == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&q_full[i], 2);   // TMA transaction (Q tiles) + the producer warp's key-validity bits
      mbar_init(&q_empty[i], 1);
      mbar_init(&s_full[i], 1);
      mbar_init(&p_ready[i], 256);
      mbar_init(&pv_done[i], 1);
    }
    for (int i = 0; i < kKvStages; ++i) {
      mbar_init(&kv_full[i], 1);
      mbar_init(&kv_empty[i], 1);
    }
    fence_mbar_init();
  }
  if (warp == kMmaWarp) {
    tmem_alloc(&tmem_slot, 512u);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;

  // item -> (b, h, q0): query-tile pair fastest, then head, then batch
  auto decode = [&](int item, int& b, int& h, int& q0) {
    int bh = item;
    q0 = 0;
    if (n_qp > 1) {                 // (the default model has one tile pair per (batch, head): no division for it)
      bh = item / n_qp;
      // the pair index is rotated by bh: with a grid that is a multiple of n_qp a CTA would otherwise always get the same
      // pair position, and under the causal mask (blocks walked grow with q0) the CTAs of the last position set the time
      q0 = ((item - bh * n_qp + bh) % n_qp) * 256;
    }
    b = bh / p.nh;
    h = bh - b * p.nh;
  };
  // Mask-aware block skipping: under the causal mask the keys after a tile's last query row are never attended, so a
  // tile only walks the key blocks up to its diagonal (tile A of a pair one block fewer than tile B) and the producer
  // only loads those -- half of all score blocks of a long sequence.  Number of key blocks tile X of the pair at q0 uses:
  const bool causal_skip = p.mask_mode == MMFM_MASK_CAUSAL && nb > 1;
  auto tile_blocks = [&](int q0, int X) -> int {
    const int r0 = q0 + 128 * X;
    if (r0 >= p.Sq) return 0;
    return causal_skip ? min(nb, (r0 + 127) / bn + 1) : nb;
  };

  if (warp == kTmaWarp) {
    // ------------------------------------------------ TMA producer ------------------------------------------------
    // the whole warp loops: one lane drives TMA, all 32 lanes pack the key-validity bytes of the item's batch entry
    // into bits (one ballot per 32 keys) next to the Q stage, so the softmax warps never touch global memory for masks
    int it = 0, t = 0;
    const int ncw = min((p.Sk + 31) >> 5, kMaxColWords);
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
      int b, h, q0;
      decode(item, b, h, q0);
      const int qs = it & 1;
      const bool has_b = q0 + 128 < p.Sq;
      mbar_wait_relaxed(&q_empty[qs], (uint32_t)(((it >> 1) & 1) ^ 1));
      if (lane == 0) {
        mbar_arrive_expect_tx(&q_full[qs], has_b ? 2 * Cfg::kQTile : Cfg::kQTile);
        tma_load_2d_addr(sQ + qs * Cfg::kQStage, &tmQ, &q_full[qs], h * D, b * p.Sq + q0);
        if (has_b) tma_load_2d_addr(sQ + qs * Cfg::kQStage + Cfg::kQTile, &tmQ, &q_full[qs], h * D, b * p.Sq + q0 + 128);
      }
      {
        const unsigned char* kvg = p.key_valid + (long long)b * p.Sk;
        const bool causal = p.mask_mode == MMFM_MASK_CAUSAL;
#pragma unroll 4
        for (int w = 0; w < ncw; ++w) {
          const int j = w * 32 + lane;
          const bool v = (j < p.Sk) && (causal || kvg[j] != 0);
          const uint32_t m = __ballot_sync(0xffffffffu, v);
          if (lane == 0) s_colbits[qs][w] = m;
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&q_full[qs]);
      }
      const int nst = max(tile_blocks(q0, 0), tile_blocks(q0, 1));   // key blocks any tile of this pair needs
      if (lane == 0) {
        for (int j = 0; j < nst; ++j) {
          const int ks = (t + j) % kKvStages;
          mbar_wait_relaxed(&kv_empty[ks], (uint32_t)((((t + j) / kKvStages) & 1) ^ 1));
          mbar_arrive_expect_tx(&kv_full[ks], 2u * (uint32_t)bn * kRowBytes);
          tma_load_2d_addr(sKV + ks * Cfg::kKvStage, &tmK, &kv_full[ks], h * D, b * p.Sk + j * bn);
          tma_load_2d_addr(sKV + ks * Cfg::kKvStage + Cfg::kKvHalf, &tmV, &kv_full[ks], h * D, b * p.Sk + j * bn);
        }
      }
      t += nst;
      __syncwarp();
    }
  } else if (warp == kMmaWarp) {
    // ------------------------------------------------ MMA issuer --------------------------------------------------
    if (elect_one()) {
      const int my_items = (n_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
      const uint32_t idesc_pv = make_idesc_bf16(128, D, 0, 1);   // A = P (TMEM, K-major), B = V MN-major
      uint32_t cnt[2] = {0u, 0u};                                // blocks issued per tile (barrier phases)

      // S of (item it, key block j, tile X) from K/V ring step t
      auto issue_qk = [&](int it, int j, int X, int t) {
        const int qs = it & 1, ks = t % kKvStages;
        mbar_wait_relaxed(&q_full[qs], (uint32_t)((it >> 1) & 1));
        mbar_wait_relaxed(&kv_full[ks], (uint32_t)((t / kKvStages) & 1));
        tc_fence_after();
        const uint32_t n = (uint32_t)(j == nb - 1 ? bl : bn);
        const uint32_t idesc = make_idesc_bf16(128, n, 0, 0);
        const uint32_t aq = sQ + qs * Cfg::kQStage + X * Cfg::kQTile, ak = sKV + ks * Cfg::kKvStage;
#pragma unroll
        for (int k = 0; k < D / 16; ++k)
          umma_bf16(tmem_base + (uint32_t)(X * Cfg::kSW), make_smem_desc(aq + k * 32, 16, kSbo, kLayout),
                    make_smem_desc(ak + k * 32, 16, kSbo, kLayout), idesc, k > 0 ? 1u : 0u);
        umma_commit(&s_full[X]);
      };
      auto item_blocks = [&](int it, int (&nbx)[2]) {
        int b, h, q0;
        decode((int)blockIdx.x + it * (int)gridDim.x, b, h, q0);
        nbx[0] = tile_blocks(q0, 0);
        nbx[1] = tile_blocks(q0, 1);
      };

      // Per tile the stream is S(0), [P.V(j), S(j+1)] ...; the two tiles alternate, so one tile's softmax overlaps the
      // other's products, and the first scores of the next item are issued behind the last P.V of this one.
      int nbx[2] = {0, 0}, nnx[2] = {0, 0};
      int t = 0;                                                 // K/V ring step of (it, j)
      if (my_items > 0) {
        item_blocks(0, nbx);
        issue_qk(0, 0, 0, 0);
        if (nbx[1] > 0) issue_qk(0, 0, 1, 0);
      }
      for (int it = 0; it < my_items; ++it) {
        const int qs = it & 1;
        const int nst = max(nbx[0], nbx[1]);
        const bool has_next = it + 1 < my_items;
        if (has_next) item_blocks(it + 1, nnx);
        for (int j = 0; j < nst; ++j, ++t) {
          const int ks = t % kKvStages;
          const int nks = (j == nb - 1 ? bl : bn) >> 4;
          const uint32_t av = sKV + ks * Cfg::kKvStage + Cfg::kKvHalf;
          const bool last = j + 1 == nst;
          const int lastX = (j < nbx[1]) ? 1 : 0;                // the last tile that reads this K/V stage
          for (int X = 0; X < 2; ++X) {
            if (j < nbx[X]) {
              mbar_wait(&p_ready[X], cnt[X] & 1u);
              ++cnt[X];
              tc_fence_after();
              const uint32_t t_s = tmem_base + (uint32_t)(X * Cfg::kSW), t_o = tmem_base + (uint32_t)(2 * Cfg::kSW + X * D);
              // 16-key steps in pairs with incremental operands: the issue loop is a dependent chain of address arithmetic in
              // ONE thread, and the tile's epilogue waits for the last of these products
              uint64_t dv = make_smem_desc(av, kSbo, kSbo, kLayout);
              const uint64_t dstep = (uint64_t)((16u * kRowBytes) >> 4);
              uint32_t ta = t_s;
              uint32_t acc = j > 0 ? 1u : 0u;
#pragma unroll 1
              for (int kk = 0; kk + 1 < nks; kk += 2) {
                umma_bf16_ts(t_o, ta, dv, idesc_pv, acc);
                umma_bf16_ts(t_o, ta + 8u, dv + dstep, idesc_pv, 1u);
                acc = 1u;
                ta += 32u;
                dv += 2 * dstep;
              }
              if (nks & 1) umma_bf16_ts(t_o, ta, dv, idesc_pv, acc);
              umma_commit(&pv_done[X]);
            }
            if (X == lastX) {      // every MMA that reads this K/V stage (and, on the last block, the Q stage) is issued
              umma_commit(&kv_empty[ks]);
              if (last) umma_commit(&q_empty[qs]);
            }
            // the next scores of this tile: the next key block, or the first block of the next item
            if (!last) {
              if (j + 1 < nbx[X]) issue_qk(it, j + 1, X, t + 1);
            } else if (has_next && nnx[X] > 0) {
              issue_qk(it + 1, 0, X, t + 1);
            }
          }
        }
        nbx[0] = nnx[0];
        nbx[1] = nnx[1];
      }
    }
    __syncwarp();
  } else {
    // ------------------------------------------------ softmax warps -----------------------------------------------
    // warp -> (tile X, column group g, TMEM quadrant wq): the two groups of a tile own alternate 64-column blocks of
    // the same 128 rows (four math warps per scheduler instead of two) and exchange the row maximum / row sum
    // through shared memory with a 256-thread named barrier.
    const int X = warp >> 3, g = (warp >> 2) & 1, wq = warp & 3;
    const int row = wq * 32 + lane;
    const int mode = p.mask_mode;
    const float sl2 = p.scale * kLog2e;
    const uint32_t t_lane = tmem_base + ((uint32_t)(wq * 32) << 16);
    const uint32_t t_s = t_lane + (uint32_t)(X * Cfg::kSW);
    const uint32_t t_o = t_lane + (uint32_t)(2 * Cfg::kSW + X * D + g * (D / 2));   // this group's half of the O row
    const int nkb_tot = (p.Sk + kTile - 1) / kTile;
    const int ncw = min((p.Sk + 31) >> 5, kMaxColWords);
    unsigned long long seed_p = 0ull;
    uint32_t c4 = 0;
    bool le128 = true;
    if (DROP) {
      seed_p = *p.drop_p.seed;
      const uint32_t th = p.drop_p.thresh;
      le128 = th <= 128u;
      c4 = (le128 ? 128u - th : 256u - th) * 0x01010101u;
    }
    const bool drop_o = p.drop_o.thresh != 0u;
    unsigned long long seed_o = 0ull;
    if (drop_o) seed_o = *p.drop_o.seed;
    const uint32_t gpr_o = (uint32_t)((p.nh * D + 15) >> 4);
    uint32_t cnt = 0;
    int it = 0;

    for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
      int b, h, q0;
      decode(item, b, h, q0);
      const int r0 = q0 + X * 128;
      const int nbt = tile_blocks(q0, X);             // key blocks of this tile (fewer under the causal mask)
      if (nbt == 0) continue;                         // tile B of a short item: nothing was issued for it
      const bool active = r0 + wq * 32 < p.Sq;        // warp-uniform: a warp whose 32 rows are all out of range idles
      const int i = r0 + row;
      const long long bh = (long long)b * p.nh + h;

      // key-validity bits of this batch entry: packed by the producer warp next to the Q stage
      const uint32_t* colbits = s_colbits[it & 1];
      DBG_P(0);
      mbar_wait(&q_full[it & 1], (uint32_t)((it >> 1) & 1));
      DBG_P(1);

      auto allowed_word = [&](int cg) -> uint32_t {   // cg = global 32-column chunk index
        uint32_t aw = cg < ncw ? colbits[cg] : 0u;
        const int rel = i - 32 * cg;
        if (mode == MMFM_MASK_KEY_OR_DIAG) {
          if (rel >= 0 && rel < 32 && i < p.Sk) aw |= 1u << rel;
        } else if (mode == MMFM_MASK_CAUSAL) {
          aw &= (rel >= 31) ? 0xFFFFFFFFu : (rel < 0 ? 0u : ((2u << rel) - 1u));
        }
        return aw;
      };

      float m_run = -INFINITY, l = 0.f;
      const unsigned long long prow = (unsigned long long)bh * p.Sq + i;
      for (int j = 0; j < nbt; ++j) {
        const int width = (j == nb - 1) ? bl : bn;
        const int nch = (width + 31) >> 5;
        const int nblk = (nch + 1) >> 1;   // 64-column blocks: one set of Philox calls each
        const int cg0 = (j * bn) >> 5;
        mbar_wait(&s_full[X], cnt & 1u);
        tc_fence_after();
        DBG_P(2);
        // ---------------- pass 1: block maximum over this group's columns, then across the two groups ----------------
        float bm = -INFINITY;
        if (active) {
#pragma unroll 1
          for (int kb = g; kb < nblk; kb += 2) {
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
              const int c = 2 * kb + hf;
              if (c < nch) {
                uint32_t r[32];
                tmem_ld32(t_s + 32u * c, r);
                tmem_ld_wait();
                const uint32_t aw = allowed_word(cg0 + c);
                if (__any_sync(0xffffffffu, aw != 0xFFFFFFFFu)) bm = chunk_max<true>(r, aw, bm);
                else bm = chunk_max<false>(r, aw, bm);
              }
            }
          }
        }
        DBG_P(3);
        s_red[X][cnt & 1u][g][row] = bm;
        named_bar_sync(1 + X, 256);
        DBG_P(4);
        bm = fmaxf(s_red[X][cnt & 1u][0][row], s_red[X][cnt & 1u][1][row]);
        if (active) {
          const float m_new = fmaxf(m_run, bm);
          const float base = (m_new == -INFINITY) ? 0.f : m_new * sl2;
          if (j > 0) {
            const float alpha = (m_run == -INFINITY) ? ((m_new == -INFINITY) ? 1.f : 0.f) : fast_exp2(m_run * sl2 - base);
            l *= alpha;
            if (__any_sync(0xffffffffu, alpha != 1.f)) {
              // the running maximum of some row moved: bring its partial output to the new reference
              mbar_wait(&pv_done[X], (cnt - 1u) & 1u);
              tc_fence_after();
#pragma unroll
              for (int u = 0; u < D / 32; ++u) {
                uint32_t o[16];
                tmem_ld16(t_o + 16u * u, o);
                tmem_ld_wait();
#pragma unroll
                for (int k = 0; k < 16; ++k) o[k] = __float_as_uint(__uint_as_float(o[k]) * alpha);
                tmem_st16(t_o + 16u * u, o);
              }
            }
          }
          m_run = m_new;
          // ---------------- pass 2: probabilities ----------------
#pragma unroll 1
          for (int kb = g; kb < nblk; kb += 2) {
            uint32_t mw[4][4];   // keep words (msb of each byte) of this block: [quad lane ql][word]
            if (DROP) {
              const uint32_t kbg = (uint32_t)((j * bn) >> 6) + (uint32_t)kb;
              uint4 w4[4];
              pdrop_bytes_x4(seed_p, p.drop_p.site, prow, (uint32_t)nkb_tot, kbg, w4);
#pragma unroll
              for (int ql = 0; ql < 4; ++ql) {
                mw[ql][0] = keep_msb(w4[ql].x, c4, le128);
                mw[ql][1] = keep_msb(w4[ql].y, c4, le128);
                mw[ql][2] = keep_msb(w4[ql].z, c4, le128);
                mw[ql][3] = keep_msb(w4[ql].w, c4, le128);
              }
              if (i < p.Sq)
                *reinterpret_cast<uint2*>(p.p_keep + ((bh * p.Sq + i) * nkb_tot + kbg) * 4) =
                    make_uint2(msb_bits16(mw[0][0], mw[0][1], mw[0][2], mw[0][3]) |
                                   (msb_bits16(mw[1][0], mw[1][1], mw[1][2], mw[1][3]) << 16),
                               msb_bits16(mw[2][0], mw[2][1], mw[2][2], mw[2][3]) |
                                   (msb_bits16(mw[3][0], mw[3][1], mw[3][2], mw[3][3]) << 16));
            }
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
              const int c = 2 * kb + hf;
              if (c < nch) {
                uint32_t r[32];
                tmem_ld32(t_s + 32u * c, r);
                tmem_ld_wait();
                const uint32_t aw = allowed_word(cg0 + c);
                uint32_t pk[16];
                if (__any_sync(0xffffffffu, aw != 0xFFFFFFFFu)) {
                  if (hf == 0) softmax_chunk<true, DROP, 0>(r, aw, sl2, base, l, mw, pk);
                  else softmax_chunk<true, DROP, 1>(r, aw, sl2, base, l, mw, pk);
                } else {
                  if (hf == 0) softmax_chunk<false, DROP, 0>(r, aw, sl2, base, l, mw, pk);
                  else softmax_chunk<false, DROP, 1>(r, aw, sl2, base, l, mw, pk);
                }
                tmem_st16(t_s + 32u * c, pk);       // in place: bf16 chunk c over the first 16 columns of fp32 chunk c
              }
            }
          }
          tmem_st_wait();
        }
        DBG_P(5);
        tc_fence_before();
        mbar_arrive(&p_ready[X]);
        ++cnt;
      }

      // ---------------- epilogue: O / l, output dropout, bf16 rows + LSE (each group stores half of the row) ----------
      s_sum[X][it & 1][g][row] = l;
      named_bar_sync(1 + X, 256);
      DBG_P(6);
      l = s_sum[X][it & 1][0][row] + s_sum[X][it & 1][1][row];
      mbar_wait(&pv_done[X], (cnt - 1u) & 1u);
      tc_fence_after();
      DBG_P(7);
      if (active) {
        float inv = l > 0.f ? 1.0f / l : 0.f;
        if (DROP) inv *= p.drop_p.scale;
        const bool ok = i < p.Sq;
        if (ok && g == 0) p.lse[bh * p.Sq + i] = (l > 0.f) ? (m_run * sl2 + log2f(l)) * kLn2 : -INFINITY;
        const int col0 = h * D + g * (D / 2);
        bf16* dst = p.o + ((long long)b * p.Sq + i) * p.ldo + col0;
#pragma unroll
        for (int u = 0; u < D / 32; ++u) {
          uint32_t o[16];
          tmem_ld16(t_o + 16u * u, o);
          tmem_ld_wait();
          float v[16];
#pragma unroll
          for (int k = 0; k < 16; ++k) v[k] = __uint_as_float(o[k]) * inv;
          if (drop_o) {
            const uint4 w = drop_bytes16(seed_o, p.drop_o.site, (uint64_t)((long long)b * p.Sq + i), gpr_o,
                                         (uint32_t)((col0 + 16 * u) >> 4));
#pragma unroll
            for (int k = 0; k < 16; ++k) v[k] = drop_byte(w, k) < p.drop_o.thresh ? 0.f : v[k] * p.drop_o.scale;
          }
          if (ok) {
#pragma unroll
            for (int k = 0; k < 16; k += 8)
              *reinterpret_cast<uint4*>(dst + 16 * u + k) =
                  make_uint4(pack_bf16x2(v[k], v[k + 1]), pack_bf16x2(v[k + 2], v[k + 3]),
                             pack_bf16x2(v[k + 4], v[k + 5]), pack_bf16x2(v[k + 6], v[k + 7]));
          }
        }
      }
      DBG_P(8);
      tc_fence_before();   // O was read out: the next item's first P.V may overwrite it once p_ready fires
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) tmem_dealloc(tmem_base, 512u);
}

}  // namespace mmfm

using namespace mmfm;

template <int D>
static int launch_fwd_pipe_d(const mmfm_attn_args* a, const AttnParams& p, cudaStream_t st) {
  using Cfg = PipeCfg<D>;
  const int npad = (a->Sk + 15) / 16 * 16;
  int bn, nb;
  if (npad <= Cfg::kSW) {
    bn = npad;
    nb = 1;
  } else {
    bn = 128;
    nb = (a->Sk + 127) / 128;
  }
  const TmaSwizzle sw = (D == 32) ? TMA_SW_64 : TMA_SW_128;
  CUtensorMap tq, tk, tv;
  const uint64_t width = (uint64_t)a->n_heads * D;
  if (int rc = make_tmap_bf16_2d(&tq, a->q, (uint64_t)a->B * a->Sq, width, (uint64_t)a->ldq, D, 128, sw)) return rc;
  if (int rc = make_tmap_bf16_2d(&tk, a->k, (uint64_t)a->B * a->Sk, width, (uint64_t)a->ldk, D, bn, sw)) return rc;
  if (int rc = make_tmap_bf16_2d(&tv, a->v, (uint64_t)a->B * a->Sk, width, (uint64_t)a->ldv, D, bn, sw)) return rc;
  const bool drop = a->drop_p.thresh != 0u;
  static bool attr_set = false;
  if (!attr_set) {
    MMFM_CHECK_CUDA(cudaFuncSetAttribute(attn_fwd_pipe_kernel<D, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::kSmem));
    MMFM_CHECK_CUDA(cudaFuncSetAttribute(attn_fwd_pipe_kernel<D, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::kSmem));
    attr_set = true;
  }
  const int n_qp = (a->Sq + 255) / 256;
  const long long n_items_ll = (long long)a->B * a->n_heads * n_qp;
  MMFM_REQUIRE(n_items_ll < (1ll << 30), "mmfm_attention_fwd: too many work items");
  const int n_items = (int)n_items_ll;
  int grid = device_sm_count();
  if (grid > n_items) grid = n_items;
  if (drop) attn_fwd_pipe_kernel<D, true><<<grid, kPipeThreads, Cfg::kSmem, st>>>(tq, tk, tv, p, bn, nb, n_qp, n_items);
  else attn_fwd_pipe_kernel<D, false><<<grid, kPipeThreads, Cfg::kSmem, st>>>(tq, tk, tv, p, bn, nb, n_qp, n_items);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

namespace mmfm {
// entry used by attention.cu's dispatcher; the caller has validated the arguments (no modality-separation mask,
// 16-byte aligned operands, Sk <= 16384)
int launch_attn_fwd_pipe(const mmfm_attn_args* a, const AttnParams& p, cudaStream_t st) {
  return a->d_head == 32 ? launch_fwd_pipe_d<32>(a, p, st) : launch_fwd_pipe_d<64>(a, p, st);
}
}  // namespace mmfm
