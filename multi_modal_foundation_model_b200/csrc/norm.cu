// LayerNorm forward / backward (nn.LayerNorm(H), eps 1e-5, affine): bandwidth kernels.
//
// Replaces ATen's vectorized_layer_norm_kernel / layer_norm_backward under every LayerNorm of the reference path
// (encoder_embeddings.py:98-100,112,114; decoder_embeddings.py:116-126,141-145; mm.py:72,77,202,212).
//
// One warp owns one row: the fp32 row is read once with 16-byte loads into registers (H <= 2048 and H % 128 == 0
// take the register path; other widths re-read through L1), mean/variance are warp-shuffle reductions, the bf16
// output is written with 8-byte stores.  The backward kernel fuses the residual-gradient add, the optional
// dropout-masked bf16 copy that feeds the next dgrad GEMM, and the dgamma/dbeta column sums (register partials per
// lane -> shared-memory reduction per CTA -> one red.global per column per CTA).
#include "common.cuh"
#include "host_util.h"
#include "../../include/mmfm_b200.h"

namespace mmfm {

constexpr int kLnWarps = 8;  // rows per CTA pass

MMFM_DEVINL long long ln_out_row(long long r, int modmajor_T, int S, long long BT) {
  if (modmajor_T <= 0) return r;
  const long long b = r / S;
  const int s = (int)(r - b * S);
  const int m = s / modmajor_T;
  return (long long)m * BT + b * modmajor_T + (s - m * modmajor_T);
}

// NV = number of float4 chunks per lane (H = 128 * NV); NV == 0 -> generic width (H % 4 == 0), re-reading x.
template <int NV>
__global__ void __launch_bounds__(kLnWarps * 32) layernorm_fwd_kernel(const float* __restrict__ x,
                                                                       const float* __restrict__ gamma,
                                                                       const float* __restrict__ beta,
                                                                       bf16* __restrict__ y, float* __restrict__ mean,
                                                                       float* __restrict__ rstd, int R, int H,
                                                                       float eps, int modmajor_T, int S) {
  pdl_enter();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long BT = modmajor_T > 0 ? (long long)(R / S) * modmajor_T : 0;
  const float invH = 1.0f / (float)H;
  if constexpr (NV > 0 && NV <= 4) {
    // register path, kLnRows rows per warp in flight: all rows' loads are issued before the first reduction starts
    // (NV <= 2: four rows, 64 KB in flight per SM at full occupancy -- the two-row form reached 62 % of the HBM peak)
    constexpr int U = NV <= 2 ? 4 : 2;
    for (long long r0 = ((long long)blockIdx.x * kLnWarps + warp) * U; r0 < R; r0 += (long long)gridDim.x * kLnWarps * U) {
      float4 v[U][NV];
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int j = 0; j < NV; ++j)
          v[u][j] = (r0 + u < R) ? __ldg(reinterpret_cast<const float4*>(x + (r0 + u) * H) + lane + 32 * j)
                                 : make_float4(0.f, 0.f, 0.f, 0.f);
      float mu[U], rs[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < NV; ++j) s += (v[u][j].x + v[u][j].y) + (v[u][j].z + v[u][j].w);
        mu[u] = warp_sum(s) * invH;
        float q = 0.f;
#pragma unroll
        for (int j = 0; j < NV; ++j) {
          const float a = v[u][j].x - mu[u], b = v[u][j].y - mu[u], c = v[u][j].z - mu[u], d = v[u][j].w - mu[u];
          q += (a * a + b * b) + (c * c + d * d);
        }
        rs[u] = rsqrtf(warp_sum(q) * invH + eps);
      }
      float4 gm[NV], bt[NV];
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        gm[j] = __ldg(reinterpret_cast<const float4*>(gamma) + lane + 32 * j);
        bt[j] = __ldg(reinterpret_cast<const float4*>(beta) + lane + 32 * j);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long r = r0 + u;
        if (r >= R) break;
        if (lane == 0) {
          mean[r] = mu[u];
          rstd[r] = rs[u];
        }
        bf16* yr = y + ln_out_row(r, modmajor_T, S, BT) * H;
#pragma unroll
        for (int j = 0; j < NV; ++j) {
          uint2 o;
          o.x = pack_bf16x2((v[u][j].x - mu[u]) * rs[u] * gm[j].x + bt[j].x, (v[u][j].y - mu[u]) * rs[u] * gm[j].y + bt[j].y);
          o.y = pack_bf16x2((v[u][j].z - mu[u]) * rs[u] * gm[j].z + bt[j].z, (v[u][j].w - mu[u]) * rs[u] * gm[j].w + bt[j].w);
          reinterpret_cast<uint2*>(yr)[lane + 32 * j] = o;
        }
      }
    }
  } else {
  for (long long r = (long long)blockIdx.x * kLnWarps + warp; r < R; r += (long long)gridDim.x * kLnWarps) {
    const float* xr = x + r * H;
    bf16* yr = y + ln_out_row(r, modmajor_T, S, BT) * H;
    if constexpr (NV > 0) {
      float4 v[NV];
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        v[j] = __ldg(reinterpret_cast<const float4*>(xr) + lane + 32 * j);
        s += (v[j].x + v[j].y) + (v[j].z + v[j].w);
      }
      const float mu = warp_sum(s) * invH;
      float q = 0.f;
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        const float a = v[j].x - mu, b = v[j].y - mu, c = v[j].z - mu, d = v[j].w - mu;
        q += (a * a + b * b) + (c * c + d * d);
      }
      const float rs = rsqrtf(warp_sum(q) * invH + eps);
      if (lane == 0) {
        mean[r] = mu;
        rstd[r] = rs;
      }
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + lane + 32 * j);
        const float4 b = __ldg(reinterpret_cast<const float4*>(beta) + lane + 32 * j);
        uint2 o;
        o.x = pack_bf16x2((v[j].x - mu) * rs * g.x + b.x, (v[j].y - mu) * rs * g.y + b.y);
        o.y = pack_bf16x2((v[j].z - mu) * rs * g.z + b.z, (v[j].w - mu) * rs * g.w + b.w);
        reinterpret_cast<uint2*>(yr)[lane + 32 * j] = o;
      }
    } else {
      float s = 0.f;
      for (int c = lane * 4; c < H; c += 128) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(xr + c));
        s += (t.x + t.y) + (t.z + t.w);
      }
      const float mu = warp_sum(s) * invH;
      float q = 0.f;
      for (int c = lane * 4; c < H; c += 128) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(xr + c));
        const float a = t.x - mu, b = t.y - mu, cc = t.z - mu, d = t.w - mu;
        q += (a * a + b * b) + (cc * cc + d * d);
      }
      const float rs = rsqrtf(warp_sum(q) * invH + eps);
      if (lane == 0) {
        mean[r] = mu;
        rstd[r] = rs;
      }
      for (int c = lane * 4; c < H; c += 128) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(xr + c));
        const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + c));
        const float4 b = __ldg(reinterpret_cast<const float4*>(beta + c));
        uint2 o;
        o.x = pack_bf16x2((t.x - mu) * rs * g.x + b.x, (t.y - mu) * rs * g.y + b.y);
        o.y = pack_bf16x2((t.z - mu) * rs * g.z + b.z, (t.w - mu) * rs * g.w + b.w);
        *reinterpret_cast<uint2*>(yr + c) = o;
      }
    }
  }
  }
}

// dx = dres + rstd * (g*dy - mean(g*dy) - xhat * mean(g*dy*xhat));  dgamma += sum dy*xhat; dbeta += sum dy
// DET: the CTA's column sums go to its workspace slot [dgamma H | dbeta H] and det_tree_fold adds them up
template <int NV, bool DET = false>
__global__ void __launch_bounds__(kLnWarps * 32) layernorm_bwd_kernel(
    const bf16* __restrict__ dy, const float* __restrict__ x, const float* __restrict__ mean,
    const float* __restrict__ rstd, const float* __restrict__ gamma, const float* dres, float* dx,
    bf16* __restrict__ dxb, DropCfg drop, float* __restrict__ dgamma, float* __restrict__ dbeta, int R, int H,
    int modmajor_T, int S, float* __restrict__ ws, unsigned int* tickets) {
  static_assert(NV > 0, "register path only");
  pdl_enter();
  __shared__ float red[kLnWarps][NV * 128 + 4];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long BT = modmajor_T > 0 ? (long long)(R / S) * modmajor_T : 0;
  const float invH = 1.0f / (float)H;
  unsigned long long seed = 0ull;
  if (drop.thresh != 0u) seed = *drop.seed;
  const uint32_t gpr = (uint32_t)((H + 15) >> 4);

  float4 gam[NV], accg[NV], accb[NV];
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    gam[j] = __ldg(reinterpret_cast<const float4*>(gamma) + lane + 32 * j);
    accg[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    accb[j] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  for (long long r = (long long)blockIdx.x * kLnWarps + warp; r < R; r += (long long)gridDim.x * kLnWarps) {
    const float* xr = x + r * H;
    const bf16* dyr = dy + ln_out_row(r, modmajor_T, S, BT) * H;
    const float mu = __ldg(mean + r), rs = __ldg(rstd + r);
    float4 xh[NV], gd[NV], dr[NV];
    float s1 = 0.f, s2 = 0.f;
    if (dres) {   // issued up front: in flight together with x / dy instead of after the two reductions
#pragma unroll
      for (int j = 0; j < NV; ++j) dr[j] = reinterpret_cast<const float4*>(dres + r * H)[lane + 32 * j];
    }
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      const float4 xv = __ldg(reinterpret_cast<const float4*>(xr) + lane + 32 * j);
      const uint2 dv = __ldg(reinterpret_cast<const uint2*>(dyr) + lane + 32 * j);
      const float2 d01 = unpack_bf16x2(dv.x), d23 = unpack_bf16x2(dv.y);
      xh[j] = make_float4((xv.x - mu) * rs, (xv.y - mu) * rs, (xv.z - mu) * rs, (xv.w - mu) * rs);
      accb[j].x += d01.x; accb[j].y += d01.y; accb[j].z += d23.x; accb[j].w += d23.y;
      accg[j].x += d01.x * xh[j].x; accg[j].y += d01.y * xh[j].y;
      accg[j].z += d23.x * xh[j].z; accg[j].w += d23.y * xh[j].w;
      gd[j] = make_float4(d01.x * gam[j].x, d01.y * gam[j].y, d23.x * gam[j].z, d23.y * gam[j].w);
      s1 += (gd[j].x + gd[j].y) + (gd[j].z + gd[j].w);
      s2 += (gd[j].x * xh[j].x + gd[j].y * xh[j].y) + (gd[j].z * xh[j].z + gd[j].w * xh[j].w);
    }
    const float m1 = warp_sum(s1) * invH, m2 = warp_sum(s2) * invH;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      float4 o;
      o.x = rs * (gd[j].x - m1 - xh[j].x * m2);
      o.y = rs * (gd[j].y - m1 - xh[j].y * m2);
      o.z = rs * (gd[j].z - m1 - xh[j].z * m2);
      o.w = rs * (gd[j].w - m1 - xh[j].w * m2);
      if (dres) { o.x += dr[j].x; o.y += dr[j].y; o.z += dr[j].z; o.w += dr[j].w; }
      if (dx) reinterpret_cast<float4*>(dx + r * H)[lane + 32 * j] = o;
      if (dxb) {
        if (drop.thresh != 0u) {
          const int c = (lane + 32 * j) * 4;
          const uint4 w = drop_bytes16(seed, drop.site, (uint64_t)r, gpr, (uint32_t)(c >> 4));
          const int b0 = c & 15;
          o.x = (drop_byte(w, b0) < drop.thresh) ? 0.f : o.x * drop.scale;
          o.y = (drop_byte(w, b0 + 1) < drop.thresh) ? 0.f : o.y * drop.scale;
          o.z = (drop_byte(w, b0 + 2) < drop.thresh) ? 0.f : o.z * drop.scale;
          o.w = (drop_byte(w, b0 + 3) < drop.thresh) ? 0.f : o.w * drop.scale;
        }
        uint2 p;
        p.x = pack_bf16x2(o.x, o.y);
        p.y = pack_bf16x2(o.z, o.w);
        reinterpret_cast<uint2*>(dxb + r * H)[lane + 32 * j] = p;
      }
    }
  }
  // CTA reduction of the column partials, then one atomic per column per CTA
#pragma unroll 1
  for (int pass = 0; pass < 2; ++pass) {
    if (pass == 1) __syncthreads();
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      const float4 a = pass == 0 ? accg[j] : accb[j];
      float* dst = &red[warp][(lane + 32 * j) * 4];
      dst[0] = a.x; dst[1] = a.y; dst[2] = a.z; dst[3] = a.w;
    }
    __syncthreads();
    float* out = pass == 0 ? dgamma : dbeta;
    if (out) {
      for (int c = threadIdx.x; c < H; c += kLnWarps * 32) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < kLnWarps; ++w) s += red[w][c];
        if constexpr (DET) ws[(long long)blockIdx.x * 2 * H + pass * H + c] = s;
        else atomicAdd(out + c, s);
      }
    }
  }
  if constexpr (DET) {
    det_tree_fold(ws, 2 * H, 2 * H, blockIdx.x, gridDim.x, tickets, [&](int i, float v) {
      float* out = i < H ? dgamma : dbeta;
      if (out) out[i < H ? i : i - H] += v;
    });
  }
}

// ------------------------------------------------------------------------------------------------------------
// Several LayerNorms over one input (the decoder layers' context_norm, decoder_embeddings.py:141-145): see the header.
// Warp = row as above; H = 128 * NV.
// ------------------------------------------------------------------------------------------------------------
template <int NV>
__global__ void __launch_bounds__(kLnWarps * 32) layernorm_fwd_multi_kernel(const mmfm_ln_multi_args a) {
  pdl_enter();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int R = a.R, H = a.H;
  const float invH = 1.0f / (float)H;
  constexpr int U = 2;   // rows per warp in flight
  for (long long r0 = ((long long)blockIdx.x * kLnWarps + warp) * U; r0 < R; r0 += (long long)gridDim.x * kLnWarps * U) {
    float4 v[U][NV];
#pragma unroll
    for (int u = 0; u < U; ++u)
#pragma unroll
      for (int j = 0; j < NV; ++j)
        v[u][j] = (r0 + u < R) ? __ldg(reinterpret_cast<const float4*>(a.x + (r0 + u) * H) + lane + 32 * j)
                               : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int u = 0; u < U; ++u) {
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < NV; ++j) s += (v[u][j].x + v[u][j].y) + (v[u][j].z + v[u][j].w);
      const float mu = warp_sum(s) * invH;
      float q = 0.f;
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        v[u][j].x -= mu; v[u][j].y -= mu; v[u][j].z -= mu; v[u][j].w -= mu;
        q += (v[u][j].x * v[u][j].x + v[u][j].y * v[u][j].y) + (v[u][j].z * v[u][j].z + v[u][j].w * v[u][j].w);
      }
      const float rs = rsqrtf(warp_sum(q) * invH + a.eps);
#pragma unroll
      for (int j = 0; j < NV; ++j) { v[u][j].x *= rs; v[u][j].y *= rs; v[u][j].z *= rs; v[u][j].w *= rs; }   // x-hat
      if (lane == 0 && r0 + u < R) {
        a.mean[r0 + u] = mu;
        a.rstd[r0 + u] = rs;
      }
    }
    for (int l = 0; l < a.n; ++l) {
      float4 gm[NV], bt[NV];
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        gm[j] = __ldg(reinterpret_cast<const float4*>(a.gamma[l]) + lane + 32 * j);
        bt[j] = __ldg(reinterpret_cast<const float4*>(a.beta[l]) + lane + 32 * j);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (r0 + u >= R) break;
        bf16* yr = reinterpret_cast<bf16*>(a.y[l]) + (r0 + u) * H;
#pragma unroll
        for (int j = 0; j < NV; ++j) {
          uint2 o;
          o.x = pack_bf16x2(fmaf(v[u][j].x, gm[j].x, bt[j].x), fmaf(v[u][j].y, gm[j].y, bt[j].y));
          o.y = pack_bf16x2(fmaf(v[u][j].z, gm[j].z, bt[j].z), fmaf(v[u][j].w, gm[j].w, bt[j].w));
          reinterpret_cast<uint2*>(yr)[lane + 32 * j] = o;
        }
      }
    }
  }
}

template <int NV, int NL, bool DET = false>
__global__ void __launch_bounds__(kLnWarps * 32) layernorm_bwd_multi_kernel(const mmfm_ln_multi_args a,
                                                                            float* __restrict__ ws,
                                                                            unsigned int* tickets) {
  pdl_enter();
  __shared__ float red[kLnWarps][128 * NV + 4];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int R = a.R, H = a.H;
  const float invH = 1.0f / (float)H;
  constexpr int U = (NV * NL <= 10) ? 2 : 1;   // rows per warp in flight (their loads are issued before the first reduction)
  float4 accg[NL][NV], accb[NL][NV];
#pragma unroll
  for (int l = 0; l < NL; ++l)
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      accg[l][j] = make_float4(0.f, 0.f, 0.f, 0.f);
      accb[l][j] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  for (long long r0 = ((long long)blockIdx.x * kLnWarps + warp) * U; r0 < R; r0 += (long long)gridDim.x * kLnWarps * U) {
    uint2 dv[U][NL][NV];
    float4 xv[U][NV];
    float mu[U], rs[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long r = (r0 + u < R) ? r0 + u : r0;   // (a row past the end re-reads row r0 and is not written)
      mu[u] = __ldg(a.mean + r);
      rs[u] = __ldg(a.rstd + r);
#pragma unroll
      for (int l = 0; l < NL; ++l)
#pragma unroll
        for (int j = 0; j < NV; ++j)
          dv[u][l][j] = __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const bf16*>(a.dy[l]) + r * H) + lane + 32 * j);
#pragma unroll
      for (int j = 0; j < NV; ++j) xv[u][j] = __ldg(reinterpret_cast<const float4*>(a.x + r * H) + lane + 32 * j);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (r0 + u >= R) break;
      const long long r = r0 + u;
      float4 xh[NV], gd[NV];
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        xh[j] = make_float4((xv[u][j].x - mu[u]) * rs[u], (xv[u][j].y - mu[u]) * rs[u], (xv[u][j].z - mu[u]) * rs[u],
                            (xv[u][j].w - mu[u]) * rs[u]);
        gd[j] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int l = 0; l < NL; ++l)
#pragma unroll
        for (int j = 0; j < NV; ++j) {
          const float4 gm = __ldg(reinterpret_cast<const float4*>(a.gamma[l]) + lane + 32 * j);
          const float2 d01 = unpack_bf16x2(dv[u][l][j].x), d23 = unpack_bf16x2(dv[u][l][j].y);
          accb[l][j].x += d01.x; accb[l][j].y += d01.y; accb[l][j].z += d23.x; accb[l][j].w += d23.y;
          accg[l][j].x = fmaf(d01.x, xh[j].x, accg[l][j].x); accg[l][j].y = fmaf(d01.y, xh[j].y, accg[l][j].y);
          accg[l][j].z = fmaf(d23.x, xh[j].z, accg[l][j].z); accg[l][j].w = fmaf(d23.y, xh[j].w, accg[l][j].w);
          gd[j].x = fmaf(d01.x, gm.x, gd[j].x); gd[j].y = fmaf(d01.y, gm.y, gd[j].y);
          gd[j].z = fmaf(d23.x, gm.z, gd[j].z); gd[j].w = fmaf(d23.y, gm.w, gd[j].w);
        }
      float s1 = 0.f, s2 = 0.f;
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        s1 += (gd[j].x + gd[j].y) + (gd[j].z + gd[j].w);
        s2 += (gd[j].x * xh[j].x + gd[j].y * xh[j].y) + (gd[j].z * xh[j].z + gd[j].w * xh[j].w);
      }
      const float m1 = warp_sum(s1) * invH, m2 = warp_sum(s2) * invH;
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        float4 o;
        o.x = rs[u] * (gd[j].x - m1 - xh[j].x * m2);
        o.y = rs[u] * (gd[j].y - m1 - xh[j].y * m2);
        o.z = rs[u] * (gd[j].z - m1 - xh[j].z * m2);
        o.w = rs[u] * (gd[j].w - m1 - xh[j].w * m2);
        reinterpret_cast<float4*>(a.dx + r * H)[lane + 32 * j] = o;
        if (a.dxb) {
          uint2 pk;
          pk.x = pack_bf16x2(o.x, o.y);
          pk.y = pack_bf16x2(o.z, o.w);
          reinterpret_cast<uint2*>(reinterpret_cast<bf16*>(a.dxb) + r * H)[lane + 32 * j] = pk;
        }
      }
    }
  }
  // CTA reduction of the column partials, then one atomic per column per CTA and layer
#pragma unroll 1
  for (int pass = 0; pass < 2 * NL; ++pass) {
    if (pass > 0) __syncthreads();
    const int l = pass >> 1;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int ll = 0; ll < NL; ++ll)
        if (ll == l) v = (pass & 1) ? accb[ll][j] : accg[ll][j];
      float* dst = &red[warp][(lane + 32 * j) * 4];
      dst[0] = v.x; dst[1] = v.y; dst[2] = v.z; dst[3] = v.w;
    }
    __syncthreads();
    float* out = (pass & 1) ? a.dbeta[l] : a.dgamma[l];
    if (out) {
      for (int c = threadIdx.x; c < H; c += kLnWarps * 32) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < kLnWarps; ++w) s += red[w][c];
        if constexpr (DET) ws[(long long)blockIdx.x * 2 * NL * H + pass * H + c] = s;
        else atomicAdd(out + c, s);
      }
    }
  }
  if constexpr (DET) {   // slot = [dgamma_0 | dbeta_0 | dgamma_1 | ...], H each
    det_tree_fold(ws, 2 * NL * H, 2 * NL * H, blockIdx.x, gridDim.x, tickets, [&](int i, float v) {
      const int pass = i / H;
      float* out = (pass & 1) ? a.dbeta[pass >> 1] : a.dgamma[pass >> 1];
      if (out) out[i - pass * H] += v;
    });
  }
}

// ------------------------------------------------------------------------------------------------------------
// ScaleNorm (mm_utils.py:31-39, `use_scalenorm: true`): y = x * g / max(||x||_2, eps), g a scalar parameter.
// Warp per row, any H % 4 == 0 (the row is re-read through L1 for the second pass).  Off the default config's path
// (mm.yaml:41 ships use_scalenorm: false), so these are plain bandwidth kernels without the register-path variants.
// rnorm[r] = 1 / max(||x_r||, eps) is saved for the backward.
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kLnWarps * 32) scalenorm_fwd_kernel(const float* __restrict__ x,
                                                                       const float* __restrict__ g,
                                                                       bf16* __restrict__ y, float* __restrict__ rnorm,
                                                                       int R, int H, float eps) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float gs = __ldg(g);
  for (long long r = (long long)blockIdx.x * kLnWarps + warp; r < R; r += (long long)gridDim.x * kLnWarps) {
    const float* xr = x + r * H;
    float q = 0.f;
    for (int c = lane * 4; c < H; c += 128) {
      const float4 t = __ldg(reinterpret_cast<const float4*>(xr + c));
      q += (t.x * t.x + t.y * t.y) + (t.z * t.z + t.w * t.w);
    }
    const float rn = 1.0f / fmaxf(sqrtf(warp_sum(q)), eps);
    if (lane == 0) rnorm[r] = rn;
    const float k = gs * rn;
    for (int c = lane * 4; c < H; c += 128) {
      const float4 t = __ldg(reinterpret_cast<const float4*>(xr + c));
      uint2 o;
      o.x = pack_bf16x2(t.x * k, t.y * k);
      o.y = pack_bf16x2(t.z * k, t.w * k);
      *reinterpret_cast<uint2*>(y + r * H + c) = o;
    }
  }
}

// dx = dres + g * rn * (dy - xhat * <dy, xhat>), xhat = x * rn  (the projection term vanishes where the norm was clamped
// to eps: there the scale g / eps is a constant);  dg += sum_rows <dy, xhat>
template <bool DET = false>
__global__ void __launch_bounds__(kLnWarps * 32) scalenorm_bwd_kernel(const bf16* __restrict__ dy,
                                                                       const float* __restrict__ x,
                                                                       const float* __restrict__ rnorm,
                                                                       const float* __restrict__ g, const float* dres,
                                                                       float* dx, bf16* __restrict__ dxb, DropCfg drop,
                                                                       float* __restrict__ dg, int R, int H, float eps,
                                                                       float* __restrict__ ws, unsigned int* tickets) {
  __shared__ float red[kLnWarps];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float gs = __ldg(g);
  unsigned long long seed = 0ull;
  if (drop.thresh != 0u) seed = *drop.seed;
  const uint32_t gpr = (uint32_t)((H + 15) >> 4);
  float acc_g = 0.f;
  for (long long r = (long long)blockIdx.x * kLnWarps + warp; r < R; r += (long long)gridDim.x * kLnWarps) {
    const float* xr = x + r * H;
    const bf16* dyr = dy + r * H;
    const float rn = __ldg(rnorm + r);
    float s = 0.f;
    for (int c = lane * 4; c < H; c += 128) {
      const float4 t = __ldg(reinterpret_cast<const float4*>(xr + c));
      const uint2 dv = __ldg(reinterpret_cast<const uint2*>(dyr + c));
      const float2 d01 = unpack_bf16x2(dv.x), d23 = unpack_bf16x2(dv.y);
      s += (d01.x * t.x + d01.y * t.y) + (d23.x * t.z + d23.y * t.w);
    }
    const float dot = warp_sum(s) * rn;            // <dy, xhat>
    acc_g += dot;
    const bool clamped = rn >= 1.0f / eps;         // ||x|| <= eps
    const float proj = clamped ? 0.f : dot * rn;   // xhat * <dy, xhat> = x * (rn * dot)
    const float k = gs * rn;
    for (int c = lane * 4; c < H; c += 128) {
      const float4 t = __ldg(reinterpret_cast<const float4*>(xr + c));
      const uint2 dv = __ldg(reinterpret_cast<const uint2*>(dyr + c));
      const float2 d01 = unpack_bf16x2(dv.x), d23 = unpack_bf16x2(dv.y);
      float4 o;
      o.x = k * (d01.x - t.x * proj); o.y = k * (d01.y - t.y * proj);
      o.z = k * (d23.x - t.z * proj); o.w = k * (d23.y - t.w * proj);
      if (dres) {
        const float4 dr = *reinterpret_cast<const float4*>(dres + r * H + c);
        o.x += dr.x; o.y += dr.y; o.z += dr.z; o.w += dr.w;
      }
      if (dx) *reinterpret_cast<float4*>(dx + r * H + c) = o;
      if (dxb) {
        if (drop.thresh != 0u) {
          const uint4 w = drop_bytes16(seed, drop.site, (uint64_t)r, gpr, (uint32_t)(c >> 4));
          const int b0 = c & 15;
          o.x = (drop_byte(w, b0) < drop.thresh) ? 0.f : o.x * drop.scale;
          o.y = (drop_byte(w, b0 + 1) < drop.thresh) ? 0.f : o.y * drop.scale;
          o.z = (drop_byte(w, b0 + 2) < drop.thresh) ? 0.f : o.z * drop.scale;
          o.w = (drop_byte(w, b0 + 3) < drop.thresh) ? 0.f : o.w * drop.scale;
        }
        uint2 pk;
        pk.x = pack_bf16x2(o.x, o.y);
        pk.y = pack_bf16x2(o.z, o.w);
        *reinterpret_cast<uint2*>(dxb + r * H + c) = pk;
      }
    }
  }
  if (lane == 0) red[warp] = acc_g;
  __syncthreads();
  if (threadIdx.x == 0 && (DET || dg)) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kLnWarps; ++w) t += red[w];
    if constexpr (DET) ws[blockIdx.x] = t;
    else atomicAdd(dg, t);
  }
  if constexpr (DET) {
    det_tree_fold(ws, 1, 1, blockIdx.x, gridDim.x, tickets, [&](int, float v) {
      if (dg) *dg += v;
    });
  }
}

}  // namespace mmfm

using namespace mmfm;

static int ln_grid(int R) {
  // no cap: the block scheduler balances better than a grid-stride loop with a ragged tail
  return (R + kLnWarps - 1) / kLnWarps;
}
static int ln_grid_fwd(int R, int H) {
  // register path: four (H <= 256) or two (H == 512) rows per warp (see the kernel), so fewer CTAs
  if (H == 128 || H == 256) return (R + 4 * kLnWarps - 1) / (4 * kLnWarps);
  if (H == 512) return (R + 2 * kLnWarps - 1) / (2 * kLnWarps);
  return ln_grid(R);
}

// CTAs that are resident at once (whole waves only: the backward ends with per-CTA atomics, so fat CTAs)
template <typename K>
static int resident_ctas(K kernel, int threads) {
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, 0) != cudaSuccess || per_sm < 1) per_sm = 1;
  return per_sm * device_sm_count();
}

extern "C" int mmfm_layernorm_fwd(const float* x, const float* gamma, const float* beta, void* y, float* mean,
                                  float* rstd, int R, int H, float eps, int modmajor_T, int S, void* stream) {
  MMFM_REQUIRE(x && gamma && beta && y && mean && rstd, "mmfm_layernorm_fwd: null pointer");
  MMFM_REQUIRE(R > 0 && H > 0 && H % 4 == 0, "mmfm_layernorm_fwd: bad shape R=%d H=%d (H must be a multiple of 4)", R, H);
  MMFM_REQUIRE(modmajor_T <= 0 || (S > 0 && S % modmajor_T == 0 && R % S == 0),
               "mmfm_layernorm_fwd: modality-major remap needs S %% T == 0 and R %% S == 0");
  cudaStream_t st = (cudaStream_t)stream;
  const int grid = ln_grid_fwd(R, H);
  set_l2_window(y, (size_t)R * H * 2);   // read next by the projection GEMM
#define LN_FWD(NV) \
  MMFM_CHECK_CUDA(launch_pdl(layernorm_fwd_kernel<NV>, dim3(grid), dim3(kLnWarps * 32), 0, st, x, gamma, beta, (bf16*)y, mean, rstd, R, H, eps, modmajor_T, S))
  switch (H) {
    case 128: LN_FWD(1); break;
    case 256: LN_FWD(2); break;
    case 512: LN_FWD(4); break;
    case 1024: LN_FWD(8); break;
    default: LN_FWD(0); break;
  }
#undef LN_FWD
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_layernorm_bwd(const void* dy, const float* x, const float* mean, const float* rstd,
                                  const float* gamma, const float* dres, float* dx, void* dxb,
                                  const mmfm_dropout* drop, float* dgamma, float* dbeta, int R, int H, int modmajor_T,
                                  int S, void* stream) {
  MMFM_REQUIRE(dy && x && mean && rstd && gamma, "mmfm_layernorm_bwd: null pointer");
  MMFM_REQUIRE(dx || dxb, "mmfm_layernorm_bwd: no output requested");
  MMFM_REQUIRE(R > 0 && (H == 128 || H == 256 || H == 512 || H == 1024),
               "mmfm_layernorm_bwd: hidden size %d not supported (128/256/512/1024)", H);
  MMFM_REQUIRE(modmajor_T <= 0 || (S > 0 && S % modmajor_T == 0 && R % S == 0),
               "mmfm_layernorm_bwd: modality-major remap needs S %% T == 0 and R %% S == 0");
  DropCfg dc{nullptr, 0u, 0u, 1.0f};
  if (drop && drop->thresh != 0u) {
    MMFM_REQUIRE(drop->seed != nullptr && drop->thresh < 256u, "mmfm_layernorm_bwd: bad dropout config");
    dc = DropCfg{drop->seed, drop->site, drop->thresh, drop->scale};
  }
  cudaStream_t st = (cudaStream_t)stream;
  // fewer, fatter CTAs than the forward (every CTA ends with 2*H atomics); exactly one resident wave
  const int want = (R + kLnWarps * 4 - 1) / (kLnWarps * 4);
  if (dxb) set_l2_window(dxb, (size_t)R * H * 2);   // read next by a dgrad GEMM
#define LN_BWD(NV)                                                                                                \
  do {                                                                                                            \
    static int cap = 0;                                                                                           \
    if (cap == 0) cap = resident_ctas(layernorm_bwd_kernel<NV>, kLnWarps * 32);                                   \
    const int grid = want < cap ? (want < 1 ? 1 : want) : cap;                                                    \
    MMFM_CHECK_CUDA(launch_pdl(layernorm_bwd_kernel<NV>, dim3(grid), dim3(kLnWarps * 32), 0, st, (const bf16*)dy, x, mean,  \
                               rstd, gamma, dres, dx, (bf16*)dxb, dc, dgamma, dbeta, R, H, modmajor_T, S, nullptr, nullptr)); \
  } while (0)
  switch (H) {
    case 128: LN_BWD(1); break;
    case 256: LN_BWD(2); break;
    case 512: LN_BWD(4); break;
    default: LN_BWD(8); break;
  }
#undef LN_BWD
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

static int ln_multi_check(const mmfm_ln_multi_args* a, const char* who, bool bwd) {
  MMFM_REQUIRE(a != nullptr, "%s: null args", who);
  MMFM_REQUIRE(a->x && a->mean && a->rstd, "%s: null pointer", who);
  MMFM_REQUIRE(a->n >= 1 && a->n <= MMFM_MAX_LN, "%s: n=%d outside [1,%d]", who, a->n, MMFM_MAX_LN);
  MMFM_REQUIRE(a->R > 0 && (a->H == 128 || a->H == 256 || a->H == 512), "%s: bad shape R=%d H=%d (H in {128, 256, 512})", who,
               a->R, a->H);
  // the backward keeps 2 * n * (H / 128) float4 column partials in registers
  MMFM_REQUIRE((a->H / 128) * a->n <= 12, "%s: n=%d LayerNorms of width %d exceed the register budget (n * H / 128 <= 12)", who,
               a->n, a->H);
  for (int l = 0; l < a->n; ++l) {
    MMFM_REQUIRE(a->gamma[l] != nullptr, "%s: layer %d has no gamma", who, l);
    if (bwd) MMFM_REQUIRE(a->dy[l] != nullptr, "%s: layer %d has no upstream gradient", who, l);
    else MMFM_REQUIRE(a->beta[l] && a->y[l], "%s: layer %d has no beta / output", who, l);
  }
  if (bwd) MMFM_REQUIRE(a->dx != nullptr, "%s: null dx", who);
  return 0;
}

extern "C" int mmfm_layernorm_fwd_multi(const mmfm_ln_multi_args* a, void* stream) {
  if (int rc = ln_multi_check(a, "mmfm_layernorm_fwd_multi", false)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int grid = ln_grid_fwd(a->R, a->H);
  switch (a->H) {
    case 128: MMFM_CHECK_CUDA(launch_pdl(layernorm_fwd_multi_kernel<1>, dim3(grid), dim3(kLnWarps * 32), 0, st, *a)); break;
    case 256: MMFM_CHECK_CUDA(launch_pdl(layernorm_fwd_multi_kernel<2>, dim3(grid), dim3(kLnWarps * 32), 0, st, *a)); break;
    default: MMFM_CHECK_CUDA(launch_pdl(layernorm_fwd_multi_kernel<4>, dim3(grid), dim3(kLnWarps * 32), 0, st, *a)); break;
  }
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

// one resident wave: the register-heavy kernel (2 * n * NV float4 accumulators) fits one or two CTAs per SM
static int ln_bwd_multi_grid(int R, int H, int n) {
  const int grid = device_sm_count() * ((H / 128) * n <= 4 ? 2 : 1);
  const int max_grid = (R + kLnWarps - 1) / kLnWarps;
  return grid > max_grid ? max_grid : grid;
}

template <int NV, bool DET>
static int ln_bwd_multi_launch(const mmfm_ln_multi_args* a, cudaStream_t st, float* ws_buf, unsigned int* tickets) {
  const int grid = ln_bwd_multi_grid(a->R, a->H, a->n);
#define LNB(NL)                                                                                                  \
  MMFM_CHECK_CUDA(DET ? launch_pdl(layernorm_bwd_multi_kernel<NV, NL, true>, dim3(grid), dim3(kLnWarps * 32), 0, st, *a, \
                                   ws_buf, tickets)                                                               \
                      : launch_pdl(layernorm_bwd_multi_kernel<NV, NL>, dim3(grid), dim3(kLnWarps * 32), 0, st, *a,   \
                                   (float*)nullptr, (unsigned int*)nullptr))
  switch (a->n) {
    case 1: LNB(1); break;
    case 2: LNB(2); break;
    case 3: LNB(3); break;
    case 4: LNB(4); break;
    case 5: LNB(5); break;
    case 6: LNB(6); break;
    case 7: LNB(7); break;
    default: LNB(8); break;
  }
#undef LNB
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_layernorm_bwd_multi(const mmfm_ln_multi_args* a, void* stream) {
  if (int rc = ln_multi_check(a, "mmfm_layernorm_bwd_multi", true)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  switch (a->H) {
    case 128: return ln_bwd_multi_launch<1, false>(a, st, nullptr, nullptr);
    case 256: return ln_bwd_multi_launch<2, false>(a, st, nullptr, nullptr);
    default: return ln_bwd_multi_launch<4, false>(a, st, nullptr, nullptr);
  }
}

// ---- deterministic twins (column sums folded by det_tree_fold; one workspace slot per CTA) ----
static int ln_bwd_det_grid(int R) {
  const int want = (R + kLnWarps * 4 - 1) / (kLnWarps * 4);
  const int cap = 2 * device_sm_count();
  return want < 1 ? 1 : (want < cap ? want : cap);
}
static int scalenorm_bwd_grid(int R, int cap) {
  int grid = (R + kLnWarps * 4 - 1) / (kLnWarps * 4);
  if (grid > cap) grid = cap;
  return grid < 1 ? 1 : grid;
}

namespace mmfm {
bool det_need_norm(int kind, long long d0, long long d1, long long d2, DetNeed* need) {
  const int R = (int)d0, H = (int)d1;
  if (kind == MMFM_DET_LN_BWD) {
    const int g = ln_bwd_det_grid(R);
    *need = DetNeed{(long long)g * 2 * H * 4, g};
  } else if (kind == MMFM_DET_LN_BWD_MULTI) {
    const int g = ln_bwd_multi_grid(R, H, (int)d2);
    *need = DetNeed{(long long)g * 2 * d2 * H * 4, g};
  } else if (kind == MMFM_DET_SCALENORM_BWD) {
    const int g = scalenorm_bwd_grid(R, 2 * device_sm_count());
    *need = DetNeed{(long long)g * 4, g};
  } else {
    return false;
  }
  return true;
}
}  // namespace mmfm

extern "C" int mmfm_layernorm_bwd_det(const void* dy, const float* x, const float* mean, const float* rstd,
                                      const float* gamma, const float* dres, float* dx, void* dxb,
                                      const mmfm_dropout* drop, float* dgamma, float* dbeta, int R, int H,
                                      int modmajor_T, int S, const mmfm_det_ws* ws, void* stream) {
  MMFM_REQUIRE(dy && x && mean && rstd && gamma && ws, "mmfm_layernorm_bwd_det: null pointer");
  MMFM_REQUIRE(dx || dxb, "mmfm_layernorm_bwd_det: no output requested");
  MMFM_REQUIRE(R > 0 && (H == 128 || H == 256 || H == 512 || H == 1024),
               "mmfm_layernorm_bwd_det: hidden size %d not supported (128/256/512/1024)", H);
  MMFM_REQUIRE(modmajor_T <= 0 || (S > 0 && S % modmajor_T == 0 && R % S == 0),
               "mmfm_layernorm_bwd_det: modality-major remap needs S %% T == 0 and R %% S == 0");
  DetNeed need{0, 0};
  det_need_norm(MMFM_DET_LN_BWD, R, H, 0, &need);
  if (int rc = det_ws_check(ws->buf, ws->bytes, ws->tickets, ws->n_tickets, need, "mmfm_layernorm_bwd_det")) return rc;
  DropCfg dc{nullptr, 0u, 0u, 1.0f};
  if (drop && drop->thresh != 0u) {
    MMFM_REQUIRE(drop->seed != nullptr && drop->thresh < 256u, "mmfm_layernorm_bwd_det: bad dropout config");
    dc = DropCfg{drop->seed, drop->site, drop->thresh, drop->scale};
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int grid = ln_bwd_det_grid(R);
  if (dxb) set_l2_window(dxb, (size_t)R * H * 2);
#define LN_BWD_DET(NV)                                                                                            \
  MMFM_CHECK_CUDA(launch_pdl(layernorm_bwd_kernel<NV, true>, dim3(grid), dim3(kLnWarps * 32), 0, st, (const bf16*)dy, x, \
                             mean, rstd, gamma, dres, dx, (bf16*)dxb, dc, dgamma, dbeta, R, H, modmajor_T, S,      \
                             (float*)ws->buf, ws->tickets))
  switch (H) {
    case 128: LN_BWD_DET(1); break;
    case 256: LN_BWD_DET(2); break;
    case 512: LN_BWD_DET(4); break;
    default: LN_BWD_DET(8); break;
  }
#undef LN_BWD_DET
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_layernorm_bwd_multi_det(const mmfm_ln_multi_args* a, const mmfm_det_ws* ws, void* stream) {
  if (int rc = ln_multi_check(a, "mmfm_layernorm_bwd_multi_det", true)) return rc;
  MMFM_REQUIRE(ws != nullptr, "mmfm_layernorm_bwd_multi_det: null workspace");
  DetNeed need{0, 0};
  det_need_norm(MMFM_DET_LN_BWD_MULTI, a->R, a->H, a->n, &need);
  if (int rc = det_ws_check(ws->buf, ws->bytes, ws->tickets, ws->n_tickets, need, "mmfm_layernorm_bwd_multi_det"))
    return rc;
  cudaStream_t st = (cudaStream_t)stream;
  float* buf = (float*)ws->buf;
  switch (a->H) {
    case 128: return ln_bwd_multi_launch<1, true>(a, st, buf, ws->tickets);
    case 256: return ln_bwd_multi_launch<2, true>(a, st, buf, ws->tickets);
    default: return ln_bwd_multi_launch<4, true>(a, st, buf, ws->tickets);
  }
}

extern "C" int mmfm_scalenorm_fwd(const float* x, const float* g, void* y, float* rnorm, int R, int H, float eps,
                                  void* stream) {
  MMFM_REQUIRE(x && g && y && rnorm, "mmfm_scalenorm_fwd: null pointer");
  MMFM_REQUIRE(R > 0 && H > 0 && H % 4 == 0, "mmfm_scalenorm_fwd: bad shape R=%d H=%d (H must be a multiple of 4)", R, H);
  scalenorm_fwd_kernel<<<ln_grid(R), kLnWarps * 32, 0, (cudaStream_t)stream>>>(x, g, (bf16*)y, rnorm, R, H, eps);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_scalenorm_bwd(const void* dy, const float* x, const float* rnorm, const float* g, const float* dres,
                                  float* dx, void* dxb, const mmfm_dropout* drop, float* dg, int R, int H, float eps,
                                  void* stream) {
  MMFM_REQUIRE(dy && x && rnorm && g, "mmfm_scalenorm_bwd: null pointer");
  MMFM_REQUIRE(dx || dxb, "mmfm_scalenorm_bwd: no output requested");
  MMFM_REQUIRE(R > 0 && H > 0 && H % 4 == 0, "mmfm_scalenorm_bwd: bad shape R=%d H=%d", R, H);
  DropCfg dc{nullptr, 0u, 0u, 1.0f};
  if (drop && drop->thresh != 0u) {
    MMFM_REQUIRE(drop->seed != nullptr && drop->thresh < 256u, "mmfm_scalenorm_bwd: bad dropout config");
    dc = DropCfg{drop->seed, drop->site, drop->thresh, drop->scale};
  }
  static int cap = 0;
  if (cap == 0) cap = resident_ctas(scalenorm_bwd_kernel<false>, kLnWarps * 32);
  const int grid = scalenorm_bwd_grid(R, cap);
  scalenorm_bwd_kernel<<<grid, kLnWarps * 32, 0, (cudaStream_t)stream>>>((const bf16*)dy, x, rnorm, g, dres, dx, (bf16*)dxb,
                                                                        dc, dg, R, H, eps, nullptr, nullptr);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_scalenorm_bwd_det(const void* dy, const float* x, const float* rnorm, const float* g,
                                      const float* dres, float* dx, void* dxb, const mmfm_dropout* drop, float* dg,
                                      int R, int H, float eps, const mmfm_det_ws* ws, void* stream) {
  MMFM_REQUIRE(dy && x && rnorm && g && ws, "mmfm_scalenorm_bwd_det: null pointer");
  MMFM_REQUIRE(dx || dxb, "mmfm_scalenorm_bwd_det: no output requested");
  MMFM_REQUIRE(R > 0 && H > 0 && H % 4 == 0, "mmfm_scalenorm_bwd_det: bad shape R=%d H=%d", R, H);
  DetNeed need{0, 0};
  det_need_norm(MMFM_DET_SCALENORM_BWD, R, H, 0, &need);
  if (int rc = det_ws_check(ws->buf, ws->bytes, ws->tickets, ws->n_tickets, need, "mmfm_scalenorm_bwd_det")) return rc;
  DropCfg dc{nullptr, 0u, 0u, 1.0f};
  if (drop && drop->thresh != 0u) {
    MMFM_REQUIRE(drop->seed != nullptr && drop->thresh < 256u, "mmfm_scalenorm_bwd_det: bad dropout config");
    dc = DropCfg{drop->seed, drop->site, drop->thresh, drop->scale};
  }
  const int grid = scalenorm_bwd_grid(R, 2 * device_sm_count());
  scalenorm_bwd_kernel<true><<<grid, kLnWarps * 32, 0, (cudaStream_t)stream>>>(
      (const bf16*)dy, x, rnorm, g, dres, dx, (bf16*)dxb, dc, dg, R, H, eps, (float*)ws->buf, ws->tickets);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}
