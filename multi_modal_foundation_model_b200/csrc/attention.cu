// Masked multi-head attention, forward and backward (flash-style: no (B,h,S,S) score / mask tensors in HBM).
//
// Replaces F.scaled_dot_product_attention(q, k, v, attn_mask=bool (B,h,S,S), dropout_p) and its autograd backward
// (reference src/multi_modal/mm_utils.py:105-112 self-attention, :143-150 cross-attention).  The (B,S,S) int64 masks
// the reference materialises (mm.py:152-158 encoder / cross, :178-194 decoder) are evaluated as predicates from
// compact descriptors: per-key validity bytes (B,Sk) -> one bit per key packed once per CTA, a diagonal flag, a
// causal flag and optional modality ids.
//
// Tiling: one CTA = 64 rows (4 warps x 16) of one (batch, head); it streams 64-wide column blocks through a
// double-buffered cp.async pipeline; scores live in mma.sync accumulators, the online-softmax state in registers.
// Every (row block, column block) pair is classified once, CTA-uniformly:
//   skip  - the mask rules the pair out entirely (padded key blocks, blocks above the causal diagonal)
//   fast  - every element is allowed: no predicate work at all
//   mixed - per-element test of a per-thread 16-bit column mask (+ one compare for the diagonal / causal rule)
// and columns past Sk / warps past Sq do no work (S = 200 is not a multiple of 64).
// At d_head = 32 the kernel is bound by the exp / ALU work of the softmax (one exp per 128 MACs), not by the tensor
// pipe -- see DESIGN.md -- so the inner loop is written for instruction count: scores are scaled inside the exp2
// FFMA, the dropout scale is applied once to the output accumulators, keep decisions are 16-bit masks built with
// byte-wise SIMD compares, and the backward reads those bits back instead of regenerating Philox output.
//   fwd       rows = queries, cols = keys : S = Q K^T -> P -> O += P V ; writes O (after output dropout), LSE, keep bits
//   bwd prep  delta = rowsum(dO * O), dO <- dO * output-dropout mask
//   bwd dq    rows = queries, cols = keys : dQ += (P * (dP - delta)) K
//   bwd dkv   rows = keys, cols = queries : dV += P_drop^T dO ; dK += dS^T Q
#include "attn_common.cuh"

namespace mmfm {

MMFM_DEVINL void cp_async16(uint32_t dst, const void* src, bool valid) {
  const int sz = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(sz) : "memory");
}
MMFM_DEVINL void cp_async8(uint32_t dst, const void* src, bool valid) {
  const int sz = valid ? 8 : 0;
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(dst), "l"(src), "r"(sz) : "memory");
}
MMFM_DEVINL void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
MMFM_DEVINL void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}


template <int D>
struct TileCfg {
  static constexpr int kPitch = D + 8;              // elements; keeps ldmatrix rows on distinct banks
  static constexpr int kBytes = kTile * kPitch * 2;  // one 64 x D tile
};

// 64 x D bf16 tile: rows row0 .. row0+63 of a matrix with `nrows` valid rows (others zero-filled)
template <int D>
MMFM_DEVINL void load_tile(uint32_t sdst, const bf16* g, long long ld, int row0, int nrows) {
  constexpr int kChunks = D / 8;
#pragma unroll
  for (int c = threadIdx.x; c < kTile * kChunks; c += kAttnThreads) {
    const int r = c / kChunks, cc = c - r * kChunks;
    const bool ok = (row0 + r) < nrows;
    const bf16* src = g + (long long)(ok ? row0 + r : 0) * ld + cc * 8;
    cp_async16(sdst + (uint32_t)(r * TileCfg<D>::kPitch + cc * 8) * 2, src, ok);
  }
}

// A fragments (16 rows of this warp x D) from a row-major tile
template <int D>
MMFM_DEVINL void load_a_frags(uint32_t stile, int warp, int lane, uint32_t (&f)[D / 16][4]) {
  const int r = warp * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;
#pragma unroll
  for (int ks = 0; ks < D / 16; ++ks) {
    const int c = ks * 16 + (lane >> 4) * 8;
    ldsm_x4(f[ks], stile + (uint32_t)(r * TileCfg<D>::kPitch + c) * 2);
  }
}

// acc[8][4] (16 x 64) = A(16 x D) . T^T where T is a 64 x D row-major tile (n = tile row, k = tile column);
// only the first `npairs` pairs of 8-column tiles are computed
template <int D>
MMFM_DEVINL void mma_rowtile_nt(float (&acc)[8][4], const uint32_t (&a)[D / 16][4], uint32_t stile, int lane,
                                int npairs) {
#pragma unroll
  for (int np = 0; np < 4; ++np) {
    if (np < npairs) {
#pragma unroll
      for (int ks = 0; ks < D / 16; ++ks) {
        uint32_t b[4];
        const int r = np * 16 + (lane >> 4) * 8 + (lane & 7);
        const int c = ks * 16 + ((lane >> 3) & 1) * 8;
        ldsm_x4(b, stile + (uint32_t)(r * TileCfg<D>::kPitch + c) * 2);
        const uint32_t b0[2] = {b[0], b[1]}, b1[2] = {b[2], b[3]};
        if (ks == 0) {   // the accumulator tile starts from zero: no clearing pass
          mma_16816_z(acc[2 * np], a[ks], b0);
          mma_16816_z(acc[2 * np + 1], a[ks], b1);
        } else {
          mma_16816(acc[2 * np], a[ks], b0);
          mma_16816(acc[2 * np + 1], a[ks], b1);
        }
      }
    } else {
      acc[2 * np][0] = acc[2 * np][1] = acc[2 * np][2] = acc[2 * np][3] = 0.f;
      acc[2 * np + 1][0] = acc[2 * np + 1][1] = acc[2 * np + 1][2] = acc[2 * np + 1][3] = 0.f;
    }
  }
}

// out[D/8][4] (16 x D) += P(16 x 64, packed bf16 A fragments) . T where T is a 64 x D row-major tile (k = tile row);
// only the first `nk16` groups of 16 tile rows contribute
template <int D>
MMFM_DEVINL void mma_rowtile_nn(float (&out)[D / 8][4], const uint32_t (&p)[4][4], uint32_t stile, int lane,
                                int nk16) {
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    if (t < nk16) {
#pragma unroll
      for (int dp = 0; dp < D / 16; ++dp) {
        uint32_t b[4];
        const int r = t * 16 + ((lane >> 3) & 1) * 8 + (lane & 7);
        const int c = dp * 16 + (lane >> 4) * 8;
        ldsm_x4_t(b, stile + (uint32_t)(r * TileCfg<D>::kPitch + c) * 2);
        const uint32_t b0[2] = {b[0], b[1]}, b1[2] = {b[2], b[3]};
        mma_16816(out[2 * dp], p[t], b0);
        mma_16816(out[2 * dp + 1], p[t], b1);
      }
    }
  }
}

MMFM_DEVINL void pack_p(const float (&s)[8][4], uint32_t (&p)[4][4]) {
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    p[t][0] = pack_bf16x2(s[2 * t][0], s[2 * t][1]);
    p[t][1] = pack_bf16x2(s[2 * t][2], s[2 * t][3]);
    p[t][2] = pack_bf16x2(s[2 * t + 1][0], s[2 * t + 1][1]);
    p[t][3] = pack_bf16x2(s[2 * t + 1][2], s[2 * t + 1][3]);
  }
}

// ------------------------------------------------------------------------------------------------------------
// mask machinery
// ------------------------------------------------------------------------------------------------------------
// Pack validity bytes into bits: word w bit l = (flags[w*32+l] != 0) for index < n.  Whole CTA; caller syncs.
MMFM_DEVINL void pack_valid_bits(const unsigned char* __restrict__ flags, int n, uint32_t* sbits, int nwords) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int w = warp; w < nwords; w += kAttnThreads / 32) {
    const int j = w * 32 + lane;
    const bool v = (j < n) && (flags[j] != 0);
    const uint32_t m = __ballot_sync(0xffffffffu, v);
    if (lane == 0) sbits[w] = m;
  }
}

// Classification of one (row block r0, column block c0) pair; everything here is CTA-uniform.
// ROWS_ARE_KEYS = false: rows are queries, columns keys (fwd, dq); true: rows keys, columns queries (dkv).
struct Blk {
  unsigned long long colmask;  // allowed-by-column bits (key validity / in-range) for the 64 columns
  int ncols;                   // columns in range
  bool skip, fast, diag, causal;
};

template <bool ROWS_ARE_KEYS>
MMFM_DEVINL Blk classify(int mode, bool sep, int r0, int c0, int ncols_total, unsigned long long col_valid_bits,
                         bool rows_all_valid, bool rows_any_valid) {
  Blk b;
  b.ncols = min(kTile, ncols_total - c0);
  const unsigned long long inrange = b.ncols >= 64 ? ~0ull : ((1ull << b.ncols) - 1ull);
  const bool cross = (c0 < r0 + kTile) && (c0 + kTile > r0);  // block touches the diagonal i == j
  b.diag = false;
  b.causal = false;
  if (mode == MMFM_MASK_CAUSAL) {
    b.colmask = inrange;
    // query i, key j: allowed iff j <= i
    const bool none = ROWS_ARE_KEYS ? (r0 > c0 + kTile - 1) : (c0 > r0 + kTile - 1);
    const bool all = ROWS_ARE_KEYS ? (r0 + kTile - 1 <= c0) : (c0 + kTile - 1 <= r0);
    b.skip = none && !sep;
    b.causal = !all;
    b.fast = all && b.ncols == 64 && !sep;
    return b;
  }
  if (!ROWS_ARE_KEYS) {
    b.colmask = col_valid_bits & inrange;
    const bool need_diag = (mode == MMFM_MASK_KEY_OR_DIAG) && cross && (b.colmask != inrange);
    b.diag = need_diag;
    b.skip = !sep && (b.colmask == 0ull) && !need_diag;
    b.fast = !sep && (b.colmask == ~0ull);
  } else {
    // columns are queries: always "valid" when in range; the key validity is a ROW property
    b.colmask = inrange;
    const bool need_diag = (mode == MMFM_MASK_KEY_OR_DIAG) && cross && !rows_all_valid;
    b.diag = need_diag;
    b.skip = !sep && !rows_any_valid && !need_diag;
    b.fast = !sep && rows_all_valid && (b.ncols == 64);
  }
  return b;
}

// the 16 columns one thread owns inside a 64-column block: bit (2n+e) <- colmask bit (8n + 2*ql + e)
MMFM_DEVINL uint32_t my_col_bits(unsigned long long colmask, int ql) {
  const unsigned long long t = colmask >> (2 * ql);
  uint32_t r = 0;
#pragma unroll
  for (int n = 0; n < 8; ++n) r |= ((uint32_t)(t >> (8 * n)) & 3u) << (2 * n);
  return r;
}

// 16 keep bits from four byte-mask words (0xFF / 0x00 per byte)
MMFM_DEVINL uint32_t mask_bits16(const uint32_t (&m)[4]) {
  return (((m[0] & 0x01010101u) * 0x01020408u) >> 24) | ((((m[1] & 0x01010101u) * 0x01020408u) >> 24) << 4) |
         ((((m[2] & 0x01010101u) * 0x01020408u) >> 24) << 8) | ((((m[3] & 0x01010101u) * 0x01020408u) >> 24) << 12);
}

// Per-thread allowed bits (2 x 16) for the mixed path.  The thread owns rows (ra, ra+8) and the 16 columns
// c0 + 8n + 2ql + e.  ROWS_ARE_KEYS selects which index is the query.
template <bool ROWS_ARE_KEYS, bool SEP>
MMFM_DEVINL void mixed_bits(const AttnParams& p, const Blk& bk, int mode, int ql, int ra, int c0, bool rowok0,
                            bool rowok1, uint32_t& a0, uint32_t& a1) {
  const uint32_t cb = my_col_bits(bk.colmask, ql);
  const uint32_t inr = my_col_bits(bk.ncols >= 64 ? ~0ull : ((1ull << bk.ncols) - 1ull), ql);
  a0 = cb;
  a1 = cb;
  if (ROWS_ARE_KEYS && mode != MMFM_MASK_CAUSAL) {
    a0 = rowok0 ? cb : 0u;
    a1 = rowok1 ? cb : 0u;
  }
  if (bk.diag || bk.causal) {
    // column offset (8n + e) at which column index == row index, for row ra: dd = ra - (c0 + 2ql)
    const int dd0 = ra - (c0 + 2 * ql), dd1 = dd0 + 8;
    uint32_t eq0 = 0, eq1 = 0, le0 = 0, le1 = 0;  // bit (2n+e): col == row ; col <= row
#pragma unroll
    for (int n = 0; n < 8; ++n) {
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int off = 8 * n + e;
        eq0 |= (off == dd0 ? 1u : 0u) << (2 * n + e);
        eq1 |= (off == dd1 ? 1u : 0u) << (2 * n + e);
        le0 |= (off <= dd0 ? 1u : 0u) << (2 * n + e);
        le1 |= (off <= dd1 ? 1u : 0u) << (2 * n + e);
      }
    }
    if (bk.diag) {
      a0 |= eq0 & inr;
      a1 |= eq1 & inr;
    } else {
      // causal: query i, key j allowed iff j <= i
      if (!ROWS_ARE_KEYS) {  // rows = queries, cols = keys: col <= row
        a0 &= le0;
        a1 &= le1;
      } else {               // rows = keys, cols = queries: row <= col  <=>  !(col < row)  <=>  !(le & !eq)
        a0 &= ~(le0 & ~eq0);
        a1 &= ~(le1 & ~eq1);
      }
    }
  }
  if (SEP) {
    // allowed |= modality(query) != modality(key); both indices must be in range
    uint32_t s0 = 0, s1 = 0;
    const int nrows_tot = ROWS_ARE_KEYS ? p.Sk : p.Sq;
#pragma unroll
    for (int n = 0; n < 8; ++n) {
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int c = c0 + 8 * n + 2 * ql + e;
        if (8 * n + 2 * ql + e < bk.ncols) {
          const short mc = ROWS_ARE_KEYS ? p.mod_q[c] : p.mod_k[c];
          if (ra < nrows_tot) s0 |= ((ROWS_ARE_KEYS ? p.mod_k[ra] : p.mod_q[ra]) != mc ? 1u : 0u) << (2 * n + e);
          if (ra + 8 < nrows_tot)
            s1 |= ((ROWS_ARE_KEYS ? p.mod_k[ra + 8] : p.mod_q[ra + 8]) != mc ? 1u : 0u) << (2 * n + e);
        }
      }
    }
    a0 |= s0;
    a1 |= s1;
  }
}

// ------------------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------------------
template <int D, bool DROP, bool SEP>
__global__ void __launch_bounds__(kAttnThreads, D == 32 ? 4 : 2) attn_fwd_kernel(const AttnParams p) {
  using TC = TileCfg<D>;
  extern __shared__ __align__(16) uint8_t smem_dyn[];
  const uint32_t sQ = smem_u32(smem_dyn);
  const uint32_t sK = sQ + TC::kBytes, sV = sQ + 3 * TC::kBytes;  // two stages each
  uint32_t* sBits = reinterpret_cast<uint32_t*>(smem_dyn + 5 * TC::kBytes);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, ql = lane & 3;
  const int q0 = blockIdx.x * kTile, h = blockIdx.y, b = blockIdx.z;
  const int nkb = (p.Sk + kTile - 1) / kTile;
  const int mode = p.mask_mode;
  const bf16* qg = p.q + (long long)b * p.Sq * p.ldq + h * D;
  const bf16* kg = p.k + (long long)b * p.Sk * p.ldk + h * D;
  const bf16* vg = p.v + (long long)b * p.Sk * p.ldv + h * D;

  load_tile<D>(sQ, qg, p.ldq, q0, p.Sq);
  load_tile<D>(sK, kg, p.ldk, 0, p.Sk);
  load_tile<D>(sV, vg, p.ldv, 0, p.Sk);
  cp_async_commit();
  pack_valid_bits(p.key_valid + (long long)b * p.Sk, p.Sk, sBits, 2 * nkb);

  const int i0 = q0 + warp * 16 + g;
  const bool warp_active = (q0 + warp * 16) < p.Sq;
  const float sl2 = p.scale * kLog2e;
  float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;  // running max in raw-score units
  float o[D / 8][4];
#pragma unroll
  for (int n = 0; n < D / 8; ++n) o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f;
  uint32_t qf[D / 16][4];

  unsigned long long seed_p = 0ull;
  uint32_t thresh4 = 0;
  if (DROP) {
    seed_p = *p.drop_p.seed;
    thresh4 = p.drop_p.thresh * 0x01010101u;
  }
  const long long bh = (long long)(b * p.nh + h);
  const unsigned long long prow0 = (unsigned long long)bh * p.Sq + i0;

  for (int kb = 0; kb < nkb; ++kb) {
    const int st = kb & 1;
    if (kb + 1 < nkb) {
      load_tile<D>(sK + (st ^ 1) * TC::kBytes, kg, p.ldk, (kb + 1) * kTile, p.Sk);
      load_tile<D>(sV + (st ^ 1) * TC::kBytes, vg, p.ldv, (kb + 1) * kTile, p.Sk);
    }
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    if (kb == 0) load_a_frags<D>(sQ, warp, lane, qf);
    const unsigned long long cvb = (unsigned long long)sBits[2 * kb] | ((unsigned long long)sBits[2 * kb + 1] << 32);
    const Blk bk = classify<false>(mode, SEP, q0, kb * kTile, p.Sk, cvb, true, true);
    if (!bk.skip && warp_active) {
      const int npairs = (bk.ncols + 15) >> 4;
      const int nt = 2 * npairs;
      float s[8][4];
      mma_rowtile_nt<D>(s, qf, sK + st * TC::kBytes, lane, npairs);
      if (!bk.fast) {
        uint32_t a0, a1;
        mixed_bits<false, SEP>(p, bk, mode, ql, i0, kb * kTile, true, true, a0, a1);
#pragma unroll
        for (int n = 0; n < 8; ++n) {
          if (n >= nt) break;  // warp-uniform: columns past the block edge do no work
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            if (!((a0 >> (2 * n + e)) & 1u)) s[n][e] = -INFINITY;
            if (!((a1 >> (2 * n + e)) & 1u)) s[n][2 + e] = -INFINITY;
          }
        }
      }
      float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
      for (int n = 0; n < 8; ++n) {
        if (n >= nt) break;  // warp-uniform: columns past the block edge do no work
        mx0 = fmaxf(mx0, fmaxf(s[n][0], s[n][1]));
        mx1 = fmaxf(mx1, fmaxf(s[n][2], s[n][3]));
      }
      mx0 = quad_max(mx0);
      mx1 = quad_max(mx1);
      const float mn0 = fmaxf(m0, mx0), mn1 = fmaxf(m1, mx1);
      const float base0 = (mn0 == -INFINITY) ? 0.f : mn0 * sl2, base1 = (mn1 == -INFINITY) ? 0.f : mn1 * sl2;
      const float al0 = fast_exp2(m0 * sl2 - base0), al1 = fast_exp2(m1 * sl2 - base1);
      m0 = mn0;
      m1 = mn1;
      float rs0 = 0.f, rs1 = 0.f;
#pragma unroll
      for (int n = 0; n < 8; ++n) {
        if (n >= nt) break;  // warp-uniform: columns past the block edge do no work
        s[n][0] = fast_exp2(fmaf(s[n][0], sl2, -base0));
        s[n][1] = fast_exp2(fmaf(s[n][1], sl2, -base0));
        s[n][2] = fast_exp2(fmaf(s[n][2], sl2, -base1));
        s[n][3] = fast_exp2(fmaf(s[n][3], sl2, -base1));
        rs0 += s[n][0] + s[n][1];
        rs1 += s[n][2] + s[n][3];
      }
      l0 = fmaf(l0, al0, rs0);
      l1 = fmaf(l1, al1, rs1);
#pragma unroll
      for (int n = 0; n < D / 8; ++n) {
        o[n][0] *= al0; o[n][1] *= al0; o[n][2] *= al1; o[n][3] *= al1;
      }
      uint32_t pf[4][4];
      pack_p(s, pf);
      if (DROP) {
        // keep decisions as byte masks (0xFF keep / 0x00 drop); survivors are rescaled once, on the output.
        // Element (n-tile n, e) of row g reads byte 2n+e: word n/2, bytes 2(n%2)+e -> one PRMT widens two bytes into
        // the two halves of the packed bf16x2 register, one LOP3 applies them.
        const uint4 w0 = pdrop_bytes(seed_p, p.drop_p.site, prow0, (uint32_t)nkb, (uint32_t)kb, (uint32_t)ql);
        const uint4 w1 = pdrop_bytes(seed_p, p.drop_p.site, prow0 + 8, (uint32_t)nkb, (uint32_t)kb, (uint32_t)ql);
        const uint32_t ma[4] = {__vcmpgeu4(w0.x, thresh4), __vcmpgeu4(w0.y, thresh4), __vcmpgeu4(w0.z, thresh4),
                                __vcmpgeu4(w0.w, thresh4)};
        const uint32_t mb[4] = {__vcmpgeu4(w1.x, thresh4), __vcmpgeu4(w1.y, thresh4), __vcmpgeu4(w1.z, thresh4),
                                __vcmpgeu4(w1.w, thresh4)};
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          pf[t][0] &= __byte_perm(ma[t], 0u, 0x1100u);
          pf[t][1] &= __byte_perm(mb[t], 0u, 0x1100u);
          pf[t][2] &= __byte_perm(ma[t], 0u, 0x3322u);
          pf[t][3] &= __byte_perm(mb[t], 0u, 0x3322u);
        }
        const uint32_t k0 = mask_bits16(ma), k1 = mask_bits16(mb);
        if (i0 < p.Sq) p.p_keep[((bh * p.Sq + i0) * nkb + kb) * 4 + ql] = (unsigned short)k0;
        if (i0 + 8 < p.Sq) p.p_keep[((bh * p.Sq + i0 + 8) * nkb + kb) * 4 + ql] = (unsigned short)k1;
      }
      mma_rowtile_nn<D>(o, pf, sV + st * TC::kBytes, lane, npairs);
    }
    __syncthreads();
  }
  if (!warp_active) return;

  l0 = quad_sum(l0);
  l1 = quad_sum(l1);
  const int i1 = i0 + 8;
  float inv0 = l0 > 0.f ? 1.0f / l0 : 0.f, inv1 = l1 > 0.f ? 1.0f / l1 : 0.f;
  if (ql == 0) {
    float* lse = p.lse + bh * p.Sq;
    if (i0 < p.Sq) lse[i0] = (l0 > 0.f) ? (m0 * sl2 + log2f(l0)) * kLn2 : -INFINITY;
    if (i1 < p.Sq) lse[i1] = (l1 > 0.f) ? (m1 * sl2 + log2f(l1)) * kLn2 : -INFINITY;
  }
  if (DROP) {
    inv0 *= p.drop_p.scale;
    inv1 *= p.drop_p.scale;
  }
  unsigned long long seed_o = 0ull;
  const bool drop_o = p.drop_o.thresh != 0u;
  if (drop_o) seed_o = *p.drop_o.seed;
  const uint32_t gpr_o = (uint32_t)((p.nh * D + 15) >> 4);
#pragma unroll
  for (int n = 0; n < D / 8; ++n) {
    float v00 = o[n][0] * inv0, v01 = o[n][1] * inv0, v10 = o[n][2] * inv1, v11 = o[n][3] * inv1;
    const int col = h * D + 8 * n + 2 * ql;
    if (drop_o) {
      const uint4 w0 = drop_bytes16(seed_o, p.drop_o.site, (uint64_t)((long long)b * p.Sq + i0), gpr_o, (uint32_t)(col >> 4));
      const uint4 w1 = drop_bytes16(seed_o, p.drop_o.site, (uint64_t)((long long)b * p.Sq + i1), gpr_o, (uint32_t)(col >> 4));
      const int bb = col & 15;
      v00 = drop_byte(w0, bb) < p.drop_o.thresh ? 0.f : v00 * p.drop_o.scale;
      v01 = drop_byte(w0, bb + 1) < p.drop_o.thresh ? 0.f : v01 * p.drop_o.scale;
      v10 = drop_byte(w1, bb) < p.drop_o.thresh ? 0.f : v10 * p.drop_o.scale;
      v11 = drop_byte(w1, bb + 1) < p.drop_o.thresh ? 0.f : v11 * p.drop_o.scale;
    }
    if (i0 < p.Sq)
      *reinterpret_cast<uint32_t*>(p.o + ((long long)b * p.Sq + i0) * p.ldo + col) = pack_bf16x2(v00, v01);
    if (i1 < p.Sq)
      *reinterpret_cast<uint32_t*>(p.o + ((long long)b * p.Sq + i1) * p.ldo + col) = pack_bf16x2(v10, v11);
  }
}

// ------------------------------------------------------------------------------------------------------------
// backward prep: delta[b,h,i] = sum_c dO[b,i,hD+c] * O[b,i,hD+c]; dO <- dO * (output dropout mask * scale)
// ------------------------------------------------------------------------------------------------------------
template <int D>
__global__ void __launch_bounds__(256) attn_bwd_prep_kernel(const AttnParams p) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int H = p.nh * D;
  const long long R = (long long)p.B * p.Sq;
  const bool drop_o = p.drop_o.thresh != 0u;
  unsigned long long seed_o = 0ull;
  if (drop_o) seed_o = *p.drop_o.seed;
  const uint32_t gpr_o = (uint32_t)((H + 15) >> 4);
  for (long long r = (long long)blockIdx.x * 8 + warp; r < R; r += (long long)gridDim.x * 8) {
    const long long b = r / p.Sq;
    const int i = (int)(r - b * p.Sq);
    for (int c = lane * 8; c < H; c += 256) {
      uint4 dv = *reinterpret_cast<const uint4*>(p.d_o + r * p.lddo + c);
      const uint4 ov = *reinterpret_cast<const uint4*>(p.o + r * p.ldo + c);
      float2 d[4] = {unpack_bf16x2(dv.x), unpack_bf16x2(dv.y), unpack_bf16x2(dv.z), unpack_bf16x2(dv.w)};
      const float2 oo[4] = {unpack_bf16x2(ov.x), unpack_bf16x2(ov.y), unpack_bf16x2(ov.z), unpack_bf16x2(ov.w)};
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) s += d[j].x * oo[j].x + d[j].y * oo[j].y;
#pragma unroll
      for (int off = 1; off < D / 8; off <<= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
      if ((lane & (D / 8 - 1)) == 0) p.delta[(b * p.nh + c / D) * p.Sq + i] = s;
      if (drop_o) {
        const uint4 w = drop_bytes16(seed_o, p.drop_o.site, (uint64_t)r, gpr_o, (uint32_t)(c >> 4));
        const int bb = c & 15;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          d[j].x = drop_byte(w, bb + 2 * j) < p.drop_o.thresh ? 0.f : d[j].x * p.drop_o.scale;
          d[j].y = drop_byte(w, bb + 2 * j + 1) < p.drop_o.thresh ? 0.f : d[j].y * p.drop_o.scale;
        }
        dv.x = pack_bf16x2(d[0].x, d[0].y);
        dv.y = pack_bf16x2(d[1].x, d[1].y);
        dv.z = pack_bf16x2(d[2].x, d[2].y);
        dv.w = pack_bf16x2(d[3].x, d[3].y);
        *reinterpret_cast<uint4*>(p.d_o + r * p.lddo + c) = dv;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// backward dQ: rows = queries, cols = keys
// ------------------------------------------------------------------------------------------------------------
template <int D, bool DROP, bool SEP>
__global__ void __launch_bounds__(kAttnThreads, D == 32 ? 4 : 2) attn_bwd_dq_kernel(const AttnParams p) {
  using TC = TileCfg<D>;
  extern __shared__ __align__(16) uint8_t smem_dyn[];
  const uint32_t sQ = smem_u32(smem_dyn), sdO = sQ + TC::kBytes;
  const uint32_t sK = sQ + 2 * TC::kBytes, sV = sQ + 4 * TC::kBytes;
  uint32_t* sBits = reinterpret_cast<uint32_t*>(smem_dyn + 6 * TC::kBytes);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, ql = lane & 3;
  const int q0 = blockIdx.x * kTile, h = blockIdx.y, b = blockIdx.z;
  const int nkb = (p.Sk + kTile - 1) / kTile;
  const int mode = p.mask_mode;
  const bf16* qg = p.q + (long long)b * p.Sq * p.ldq + h * D;
  const bf16* dog = p.d_o + (long long)b * p.Sq * p.lddo + h * D;
  const bf16* kg = p.k + (long long)b * p.Sk * p.ldk + h * D;
  const bf16* vg = p.v + (long long)b * p.Sk * p.ldv + h * D;

  load_tile<D>(sQ, qg, p.ldq, q0, p.Sq);
  load_tile<D>(sdO, dog, p.lddo, q0, p.Sq);
  load_tile<D>(sK, kg, p.ldk, 0, p.Sk);
  load_tile<D>(sV, vg, p.ldv, 0, p.Sk);
  cp_async_commit();
  pack_valid_bits(p.key_valid + (long long)b * p.Sk, p.Sk, sBits, 2 * nkb);

  const int i0 = q0 + warp * 16 + g, i1 = i0 + 8;
  const bool warp_active = (q0 + warp * 16) < p.Sq;
  const float sl2 = p.scale * kLog2e;
  const long long bh = (long long)(b * p.nh + h);
  const float lse0 = (i0 < p.Sq) ? p.lse[bh * p.Sq + i0] * kLog2e : INFINITY;
  const float lse1 = (i1 < p.Sq) ? p.lse[bh * p.Sq + i1] * kLog2e : INFINITY;
  const float dsc = DROP ? p.drop_p.scale : 1.0f;
  // dS = P * (keep * dsc * dP - delta) -> fold dsc: work with dP' = keep * dP and delta' = delta / dsc, rescale at the end
  const float dl0 = ((i0 < p.Sq) ? p.delta[bh * p.Sq + i0] : 0.f) / dsc;
  const float dl1 = ((i1 < p.Sq) ? p.delta[bh * p.Sq + i1] : 0.f) / dsc;
  float dq[D / 8][4];
#pragma unroll
  for (int n = 0; n < D / 8; ++n) dq[n][0] = dq[n][1] = dq[n][2] = dq[n][3] = 0.f;
  uint32_t qf[D / 16][4], dof[D / 16][4];

  for (int kb = 0; kb < nkb; ++kb) {
    const int st = kb & 1;
    if (kb + 1 < nkb) {
      load_tile<D>(sK + (st ^ 1) * TC::kBytes, kg, p.ldk, (kb + 1) * kTile, p.Sk);
      load_tile<D>(sV + (st ^ 1) * TC::kBytes, vg, p.ldv, (kb + 1) * kTile, p.Sk);
    }
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    if (kb == 0) {
      load_a_frags<D>(sQ, warp, lane, qf);
      load_a_frags<D>(sdO, warp, lane, dof);
    }
    const unsigned long long cvb = (unsigned long long)sBits[2 * kb] | ((unsigned long long)sBits[2 * kb + 1] << 32);
    const Blk bk = classify<false>(mode, SEP, q0, kb * kTile, p.Sk, cvb, true, true);
    if (!bk.skip && warp_active) {
      const int npairs = (bk.ncols + 15) >> 4;
      const int nt = 2 * npairs;
      float s[8][4], dp[8][4];
      mma_rowtile_nt<D>(s, qf, sK + st * TC::kBytes, lane, npairs);
      mma_rowtile_nt<D>(dp, dof, sV + st * TC::kBytes, lane, npairs);
      uint32_t a0 = 0xFFFFu, a1 = 0xFFFFu;
      if (!bk.fast) mixed_bits<false, SEP>(p, bk, mode, ql, i0, kb * kTile, true, true, a0, a1);
      uint32_t k0 = 0xFFFFu, k1 = 0xFFFFu;
      if (DROP) {
        if (i0 < p.Sq) k0 = p.p_keep[((bh * p.Sq + i0) * nkb + kb) * 4 + ql];
        if (i1 < p.Sq) k1 = p.p_keep[((bh * p.Sq + i1) * nkb + kb) * 4 + ql];
      }
#pragma unroll
      for (int n = 0; n < 8; ++n) {
        if (n >= nt) break;  // warp-uniform: columns past the block edge do no work
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int bit = 2 * n + e;
          float p0 = fast_exp2(fmaf(s[n][e], sl2, -lse0));
          float p1 = fast_exp2(fmaf(s[n][2 + e], sl2, -lse1));
          if (!bk.fast) {
            if (!((a0 >> bit) & 1u)) p0 = 0.f;
            if (!((a1 >> bit) & 1u)) p1 = 0.f;
          }
          float dp0 = dp[n][e], dp1 = dp[n][2 + e];
          if (DROP) {
            if (!((k0 >> bit) & 1u)) dp0 = 0.f;
            if (!((k1 >> bit) & 1u)) dp1 = 0.f;
          }
          s[n][e] = p0 * (dp0 - dl0);
          s[n][2 + e] = p1 * (dp1 - dl1);
        }
      }
      uint32_t pf[4][4];
      pack_p(s, pf);
      mma_rowtile_nn<D>(dq, pf, sK + st * TC::kBytes, lane, npairs);
    }
    __syncthreads();
  }
  if (!warp_active) return;
  const float fs = p.scale * dsc;
#pragma unroll
  for (int n = 0; n < D / 8; ++n) {
    const int col = h * D + 8 * n + 2 * ql;
    if (i0 < p.Sq)
      *reinterpret_cast<uint32_t*>(p.dq + ((long long)b * p.Sq + i0) * p.lddq + col) =
          pack_bf16x2(dq[n][0] * fs, dq[n][1] * fs);
    if (i1 < p.Sq)
      *reinterpret_cast<uint32_t*>(p.dq + ((long long)b * p.Sq + i1) * p.lddq + col) =
          pack_bf16x2(dq[n][2] * fs, dq[n][3] * fs);
  }
}

// ------------------------------------------------------------------------------------------------------------
// backward dK, dV: rows = keys, cols = queries
// ------------------------------------------------------------------------------------------------------------
template <int D, bool DROP, bool SEP>
__global__ void __launch_bounds__(kAttnThreads, D == 32 ? 3 : 2) attn_bwd_dkv_kernel(const AttnParams p) {
  using TC = TileCfg<D>;
  extern __shared__ __align__(16) uint8_t smem_dyn[];
  const uint32_t sK = smem_u32(smem_dyn), sV = sK + TC::kBytes;
  const uint32_t sQ = sK + 2 * TC::kBytes, sdO = sK + 4 * TC::kBytes;  // two stages each
  uint8_t* tail = smem_dyn + 6 * TC::kBytes;
  float* sLse = reinterpret_cast<float*>(tail);                          // [2][64]
  float* sDelta = reinterpret_cast<float*>(tail + 2 * kTile * 4);        // [2][64]
  unsigned short* sKeep = reinterpret_cast<unsigned short*>(tail + 4 * kTile * 4);  // [2][64][4]
  __shared__ uint32_t sRowBits[2];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, ql = lane & 3;
  const int kblk = blockIdx.x, k0 = kblk * kTile, h = blockIdx.y, b = blockIdx.z;
  const int nqb = (p.Sq + kTile - 1) / kTile;
  const int nkb = (p.Sk + kTile - 1) / kTile;
  const int mode = p.mask_mode;
  const long long bh = (long long)(b * p.nh + h);
  const bf16* qg = p.q + (long long)b * p.Sq * p.ldq + h * D;
  const bf16* dog = p.d_o + (long long)b * p.Sq * p.lddo + h * D;
  const bf16* kg = p.k + (long long)b * p.Sk * p.ldk + h * D;
  const bf16* vg = p.v + (long long)b * p.Sk * p.ldv + h * D;
  const unsigned char* kvg = p.key_valid + (long long)b * p.Sk;
  const float dsc = DROP ? p.drop_p.scale : 1.0f;
  const float inv_dsc = 1.0f / dsc;

  auto load_q = [&](int qb, int st) {
    load_tile<D>(sQ + st * TC::kBytes, qg, p.ldq, qb * kTile, p.Sq);
    load_tile<D>(sdO + st * TC::kBytes, dog, p.lddo, qb * kTile, p.Sq);
    if (threadIdx.x < kTile) {
      const int i = qb * kTile + threadIdx.x;
      sLse[st * kTile + threadIdx.x] = (i < p.Sq) ? p.lse[bh * p.Sq + i] * kLog2e : INFINITY;
      sDelta[st * kTile + threadIdx.x] = (i < p.Sq) ? p.delta[bh * p.Sq + i] * inv_dsc : 0.f;
      if (DROP) {
        const bool ok = i < p.Sq;
        const unsigned short* src = p.p_keep + ((bh * p.Sq + (ok ? i : 0)) * nkb + kblk) * 4;
        cp_async8(smem_u32(sKeep + (st * kTile + threadIdx.x) * 4), src, ok);
      }
    }
  };
  load_tile<D>(sK, kg, p.ldk, k0, p.Sk);
  load_tile<D>(sV, vg, p.ldv, k0, p.Sk);
  load_q(0, 0);
  cp_async_commit();
  if (warp < 2) {
    const int j = k0 + warp * 32 + lane;
    const uint32_t m = __ballot_sync(0xffffffffu, (j < p.Sk) && (kvg[j] != 0));
    if (lane == 0) sRowBits[warp] = m;
  }
  __syncthreads();
  const unsigned long long rowbits = (unsigned long long)sRowBits[0] | ((unsigned long long)sRowBits[1] << 32);
  const int nrows = min(kTile, p.Sk - k0);
  const unsigned long long rows_inrange = nrows >= 64 ? ~0ull : ((1ull << nrows) - 1ull);
  const bool rows_all_valid = (rowbits == ~0ull);
  const bool rows_any_valid = (mode == MMFM_MASK_CAUSAL) ? true : (rowbits != 0ull);
  (void)rows_inrange;

  const int j0 = k0 + warp * 16 + g, j1 = j0 + 8;  // this thread's key rows
  const bool warp_active = (k0 + warp * 16) < p.Sk;
  const bool kv0 = (rowbits >> (warp * 16 + g)) & 1ull, kv1 = (rowbits >> (warp * 16 + g + 8)) & 1ull;
  const float sl2 = p.scale * kLog2e;
  float dk[D / 8][4], dv[D / 8][4];
#pragma unroll
  for (int n = 0; n < D / 8; ++n) {
    dk[n][0] = dk[n][1] = dk[n][2] = dk[n][3] = 0.f;
    dv[n][0] = dv[n][1] = dv[n][2] = dv[n][3] = 0.f;
  }
  uint32_t kf[D / 16][4], vf[D / 16][4];
  // keep-bit addressing: word (query i, quad (key%8)/2), bit ((key%64)/8)*2 + key%2
  const int kq = g >> 1;
  const int bit0 = (warp * 2) * 2 + (g & 1), bit1 = bit0 + 2;

  for (int qb = 0; qb < nqb; ++qb) {
    const int st = qb & 1;
    if (qb + 1 < nqb) load_q(qb + 1, st ^ 1);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    if (qb == 0) {
      load_a_frags<D>(sK, warp, lane, kf);
      load_a_frags<D>(sV, warp, lane, vf);
    }
    const Blk bk = classify<true>(mode, SEP, k0, qb * kTile, p.Sq, 0ull, rows_all_valid, rows_any_valid);
    if (!bk.skip && warp_active) {
      const int npairs = (bk.ncols + 15) >> 4;
      const int nt = 2 * npairs;
      float s[8][4], dp[8][4];
      mma_rowtile_nt<D>(s, kf, sQ + st * TC::kBytes, lane, npairs);     // S^T[key, query]
      mma_rowtile_nt<D>(dp, vf, sdO + st * TC::kBytes, lane, npairs);   // dP^T[key, query]
      uint32_t a0 = 0xFFFFu, a1 = 0xFFFFu;
      if (!bk.fast) mixed_bits<true, SEP>(p, bk, mode, ql, j0, qb * kTile, kv0, kv1, a0, a1);
      float pd[8][4];  // dropped probabilities (for dV)
      const float* lsep = sLse + st * kTile + 2 * ql;
      const float* dlp = sDelta + st * kTile + 2 * ql;
      const unsigned short* kp = sKeep + (st * kTile + 2 * ql) * 4 + kq;
#pragma unroll
      for (int n = 0; n < 8; ++n) {
        if (n >= nt) break;  // warp-uniform: columns past the block edge do no work
        const float2 lse2 = *reinterpret_cast<const float2*>(lsep + 8 * n);
        const float2 dl2 = *reinterpret_cast<const float2*>(dlp + 8 * n);
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int bit = 2 * n + e;
          const float lse = e ? lse2.y : lse2.x, dl = e ? dl2.y : dl2.x;
          float p0 = fast_exp2(fmaf(s[n][e], sl2, -lse));
          float p1 = fast_exp2(fmaf(s[n][2 + e], sl2, -lse));
          if (!bk.fast) {
            if (!((a0 >> bit) & 1u)) p0 = 0.f;
            if (!((a1 >> bit) & 1u)) p1 = 0.f;
          }
          float dp0 = dp[n][e], dp1 = dp[n][2 + e];
          float pd0 = p0, pd1 = p1;
          if (DROP) {
            const uint32_t wbits = kp[(8 * n + e) * 4];
            if (!((wbits >> bit0) & 1u)) { dp0 = 0.f; pd0 = 0.f; }
            if (!((wbits >> bit1) & 1u)) { dp1 = 0.f; pd1 = 0.f; }
          }
          pd[n][e] = pd0;
          pd[n][2 + e] = pd1;
          s[n][e] = p0 * (dp0 - dl);
          s[n][2 + e] = p1 * (dp1 - dl);
        }
      }
      uint32_t pf[4][4];
      pack_p(pd, pf);
      mma_rowtile_nn<D>(dv, pf, sdO + st * TC::kBytes, lane, npairs);
      pack_p(s, pf);
      mma_rowtile_nn<D>(dk, pf, sQ + st * TC::kBytes, lane, npairs);
    }
    __syncthreads();
  }
  if (!warp_active) return;
  const float fk = p.scale * dsc;
#pragma unroll
  for (int n = 0; n < D / 8; ++n) {
    const int col = h * D + 8 * n + 2 * ql;
    if (j0 < p.Sk) {
      *reinterpret_cast<uint32_t*>(p.dk + ((long long)b * p.Sk + j0) * p.lddk + col) =
          pack_bf16x2(dk[n][0] * fk, dk[n][1] * fk);
      *reinterpret_cast<uint32_t*>(p.dv + ((long long)b * p.Sk + j0) * p.lddv + col) =
          pack_bf16x2(dv[n][0] * dsc, dv[n][1] * dsc);
    }
    if (j1 < p.Sk) {
      *reinterpret_cast<uint32_t*>(p.dk + ((long long)b * p.Sk + j1) * p.lddk + col) =
          pack_bf16x2(dk[n][2] * fk, dk[n][3] * fk);
      *reinterpret_cast<uint32_t*>(p.dv + ((long long)b * p.Sk + j1) * p.lddv + col) =
          pack_bf16x2(dv[n][2] * dsc, dv[n][3] * dsc);
    }
  }
}

}  // namespace mmfm

// ------------------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------------------
using namespace mmfm;

template <void (*KERNEL)(const AttnParams)>
static int launch_k(const AttnParams& p, dim3 grid, int smem, cudaStream_t st) {
  static int attr_smem = 0;
  if (smem > attr_smem) {
    if (smem > 48 * 1024)
      MMFM_CHECK_CUDA(cudaFuncSetAttribute(KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr_smem = smem;
  }
  KERNEL<<<grid, kAttnThreads, smem, st>>>(p);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

static int check_common(const mmfm_attn_args* a, const char* who) {
  MMFM_REQUIRE(a != nullptr, "%s: null args", who);
  MMFM_REQUIRE(a->q && a->k && a->v && a->o && a->lse && a->key_valid, "%s: null operand", who);
  MMFM_REQUIRE(a->B > 0 && a->n_heads > 0 && a->Sq > 0 && a->Sk > 0, "%s: bad shape", who);
  MMFM_REQUIRE(a->Sk <= 16384 && a->Sq <= 16384, "%s: sequence too long (%d, %d)", who, a->Sq, a->Sk);
  MMFM_REQUIRE(a->d_head == 32 || a->d_head == 64, "%s: d_head %d not supported (32 or 64)", who, a->d_head);
  MMFM_REQUIRE(a->mask_mode >= MMFM_MASK_KEY && a->mask_mode <= MMFM_MASK_CAUSAL, "%s: bad mask mode %d", who,
               a->mask_mode);
  MMFM_REQUIRE((a->mod_q == nullptr) == (a->mod_k == nullptr), "%s: mod_q and mod_k must be given together", who);
  MMFM_REQUIRE(a->ldq % 8 == 0 && a->ldk % 8 == 0 && a->ldv % 8 == 0 && a->ldo % 8 == 0,
               "%s: row pitches must be multiples of 8 elements", who);
  MMFM_REQUIRE(a->drop_p.thresh < 256u && a->drop_o.thresh < 256u, "%s: dropout threshold out of range", who);
  MMFM_REQUIRE(a->drop_p.thresh == 0u || a->drop_p.seed, "%s: probability dropout without seed", who);
  MMFM_REQUIRE(a->drop_o.thresh == 0u || a->drop_o.seed, "%s: output dropout without seed", who);
  MMFM_REQUIRE(a->drop_p.thresh == 0u || a->p_keep, "%s: probability dropout needs the p_keep buffer", who);
  MMFM_REQUIRE(a->B <= 65535 && a->n_heads <= 65535, "%s: grid too large", who);
  return 0;
}

static AttnParams to_params(const mmfm_attn_args* a) {
  AttnParams p;
  p.q = (const bf16*)a->q; p.ldq = a->ldq;
  p.k = (const bf16*)a->k; p.ldk = a->ldk;
  p.v = (const bf16*)a->v; p.ldv = a->ldv;
  p.o = (bf16*)a->o; p.ldo = a->ldo;
  p.lse = a->lse;
  p.key_valid = a->key_valid;
  p.mod_q = a->mod_q; p.mod_k = a->mod_k;
  p.B = a->B; p.nh = a->n_heads; p.Sq = a->Sq; p.Sk = a->Sk;
  p.mask_mode = a->mask_mode;
  p.scale = a->scale;
  p.drop_p = DropCfg{a->drop_p.seed, a->drop_p.site, a->drop_p.thresh, a->drop_p.scale};
  p.drop_o = DropCfg{a->drop_o.seed, a->drop_o.site, a->drop_o.thresh, a->drop_o.scale};
  p.p_keep = a->p_keep;
  p.d_o = (bf16*)a->d_o; p.lddo = a->lddo;
  p.delta = a->delta;
  p.dq = (bf16*)a->dq; p.lddq = a->lddq;
  p.dk = (bf16*)a->dk; p.lddk = a->lddk;
  p.dv = (bf16*)a->dv; p.lddv = a->lddv;
  return p;
}

// dispatch on (d_head, dropout, modality-separation)
#define ATTN_DISPATCH(KERNEL, grid, smem_expr)                                                    \
  do {                                                                                            \
    if (a->d_head == 32) {                                                                        \
      constexpr int D = 32;                                                                       \
      const int smem = (smem_expr);                                                               \
      if (drop) { if (sep) return launch_k<KERNEL<32, true, true>>(p, grid, smem, st);            \
                  return launch_k<KERNEL<32, true, false>>(p, grid, smem, st); }                  \
      if (sep) return launch_k<KERNEL<32, false, true>>(p, grid, smem, st);                       \
      return launch_k<KERNEL<32, false, false>>(p, grid, smem, st);                               \
    } else {                                                                                      \
      constexpr int D = 64;                                                                       \
      const int smem = (smem_expr);                                                               \
      if (drop) { if (sep) return launch_k<KERNEL<64, true, true>>(p, grid, smem, st);            \
                  return launch_k<KERNEL<64, true, false>>(p, grid, smem, st); }                  \
      if (sep) return launch_k<KERNEL<64, false, true>>(p, grid, smem, st);                       \
      return launch_k<KERNEL<64, false, false>>(p, grid, smem, st);                               \
    }                                                                                             \
  } while (0)

// Forward dispatch:
//   no modality-separation mask, 16-byte aligned operands -> persistent warp-specialised tcgen05 kernel (attention_pipe.cu)
//   otherwise                                             -> mma.sync flash kernel (modality ids, odd alignments)
extern "C" int mmfm_attention_fwd(const mmfm_attn_args* a, void* stream) {
  if (int rc = check_common(a, "mmfm_attention_fwd")) return rc;
  const bool drop = a->drop_p.thresh != 0u, sep = a->mod_q != nullptr;
  const AttnParams p = to_params(a);
  const bool al16 = ((reinterpret_cast<uintptr_t>(a->q) | reinterpret_cast<uintptr_t>(a->k) |
                      reinterpret_cast<uintptr_t>(a->v) | reinterpret_cast<uintptr_t>(a->o)) & 15) == 0;
  if (!sep && al16) return launch_attn_fwd_pipe(a, p, (cudaStream_t)stream);
  dim3 grid((a->Sq + kTile - 1) / kTile, a->n_heads, a->B);
  cudaStream_t st = (cudaStream_t)stream;
  const int nkb = (a->Sk + kTile - 1) / kTile;
  ATTN_DISPATCH(attn_fwd_kernel, grid, 5 * TileCfg<D>::kBytes + 2 * nkb * 4);
}

static int launch_dq(const mmfm_attn_args* a, const AttnParams& p, cudaStream_t st) {
  const bool drop = a->drop_p.thresh != 0u, sep = a->mod_q != nullptr;
  dim3 grid((a->Sq + kTile - 1) / kTile, a->n_heads, a->B);
  const int nkb = (a->Sk + kTile - 1) / kTile;
  ATTN_DISPATCH(attn_bwd_dq_kernel, grid, 6 * TileCfg<D>::kBytes + 2 * nkb * 4);
}
static int launch_dkv(const mmfm_attn_args* a, const AttnParams& p, cudaStream_t st) {
  const bool drop = a->drop_p.thresh != 0u, sep = a->mod_q != nullptr;
  dim3 grid((a->Sk + kTile - 1) / kTile, a->n_heads, a->B);
  ATTN_DISPATCH(attn_bwd_dkv_kernel, grid, 6 * TileCfg<D>::kBytes + 4 * kTile * 4 + 2 * kTile * 4 * 2);
}

// Backward dispatch (after the prep kernel: delta = rowsum(dO * O), dO <- dO * output-dropout mask):
//   d_head 32, Sq, Sk <= 256 (the default model), 16-byte aligned lse / delta / p_keep, Sq % 4 == 0
//                                                  -> persistent warp-specialised fused kernel (attention_bwd_ws.cu)
//   any other shape without modality-separation    -> streamed tcgen05 dq / dkv pair (attention_bwd_stream.cu)
//   modality-separation mask, odd alignments        -> mma.sync dq / dkv pair
extern "C" int mmfm_attention_bwd(const mmfm_attn_args* a, void* stream) {
  if (int rc = check_common(a, "mmfm_attention_bwd")) return rc;
  MMFM_REQUIRE(a->d_o && a->delta && a->dq && a->dk && a->dv, "mmfm_attention_bwd: null gradient buffer");
  MMFM_REQUIRE(a->lddo % 8 == 0 && a->lddq % 8 == 0 && a->lddk % 8 == 0 && a->lddv % 8 == 0,
               "mmfm_attention_bwd: row pitches must be multiples of 8 elements");
  const AttnParams p = to_params(a);
  cudaStream_t st = (cudaStream_t)stream;
  const long long R = (long long)a->B * a->Sq;
  int pgrid = (int)((R + 7) / 8);
  const int cap = device_sm_count() * 8;
  if (pgrid > cap) pgrid = cap;
  if (!a->prep_done) {   // else: delta and the masked d_o come from the out-projection dgrad GEMM (MMFM_ACT_ROWDOT_DROP)
    if (a->d_head == 32) attn_bwd_prep_kernel<32><<<pgrid, 256, 0, st>>>(p);
    else attn_bwd_prep_kernel<64><<<pgrid, 256, 0, st>>>(p);
    MMFM_CHECK_CUDA(cudaGetLastError());
  }

  const bool al16 = ((reinterpret_cast<uintptr_t>(a->q) | reinterpret_cast<uintptr_t>(a->k) |
                      reinterpret_cast<uintptr_t>(a->v) | reinterpret_cast<uintptr_t>(a->d_o) |
                      reinterpret_cast<uintptr_t>(a->dq) | reinterpret_cast<uintptr_t>(a->dk) |
                      reinterpret_cast<uintptr_t>(a->dv)) & 15) == 0;
  if (a->mod_q == nullptr && al16) {
    const bool side_al = ((reinterpret_cast<uintptr_t>(a->lse) | reinterpret_cast<uintptr_t>(a->delta) |
                           reinterpret_cast<uintptr_t>(a->p_keep)) & 15) == 0;
    if (a->d_head == 32 && a->Sq <= 256 && a->Sk <= 256 && a->Sq % 4 == 0 && side_al) return launch_attn_bwd_ws(a, p, st);
    return launch_attn_bwd_stream(a, p, st);
  }
  if (int rc = launch_dq(a, p, st)) return rc;
  return launch_dkv(a, p, st);
}
