// Bandwidth kernels around the GEMM / attention core: mask preparation, embedding assembly and its gradient,
// the small-channel (C <= 8) embedder / head, the fused masked loss + gradient, multi-tensor fp32 -> bf16 casts.
//
// Reference call sites replaced (paths relative to the reference root):
//   mask_prep            mm.py:266-275 (mask[:,:,0] & attn), :147,169 (argwhere(mask[0]==1)), :231,237 (counts)
//   embed_assemble(+bwd) encoder_embeddings.py:56-59 / decoder_embeddings.py:56-59 (mod_emb + pos_embed gather)
//   embed_grad_prep      autograd of the in-place token zeroing (mm.py:149,171) and embedding dropout (:61)
//   smallc_*             encoder_embeddings.py:50-61 and decoder_embeddings.py:105-107 for C <= 8 (behaviour, C = 2)
//   loss_fwd_bwd         mm.py:217-239 with nn.PoissonNLLLoss(log_input=True) (:80) and nn.MSELoss (:81)
#include "common.cuh"
#include <math.h>
#include "host_util.h"
#include "../../include/mmfm_b200.h"

namespace mmfm {

MMFM_DEVINL float block_sum(float v, float* sh) {  // sh: >= 32 floats
  v = warp_sum(v);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
  __syncthreads();
  if (lane == 0) sh[warp] = v;
  __syncthreads();
  float t = (threadIdx.x < nw) ? sh[threadIdx.x] : 0.f;
  if (warp == 0) t = warp_sum(t);
  if (threadIdx.x == 0) sh[0] = t;
  __syncthreads();
  return sh[0];
}

// ------------------------------------------------------------------------------------------------------------
// mask preparation (B*S elements).  grid = (slices, modalities): the step's first kernel sits on the critical path of
// everything else, and as a single CTA it spent 44 us on 25 dependent rounds of strided int64 loads.  Every CTA adds its
// masked-token count to a per-modality counter; the last one to finish (ticket) turns the counters into n_examples /
// inv_n and leaves counters and ticket at zero for the next launch.  Counts are integers: the result does not depend on
// the arrival order.  (One mask_prep in flight per device at a time: the engine issues it on its single stream.)
// ------------------------------------------------------------------------------------------------------------
__device__ unsigned int g_mp_count[MMFM_MAX_MOD];
__device__ unsigned int g_mp_ticket;

__global__ void __launch_bounds__(256) mask_prep_kernel(const mmfm_mask_args a, unsigned char* __restrict__ zero_flags,
                                                         unsigned char* __restrict__ key_valid,
                                                         unsigned char* __restrict__ tok_mask,
                                                         long long* __restrict__ n_examples,
                                                         float* __restrict__ inv_n) {
  __shared__ float sh[32];
  const int S = a.n_mod * a.T;
  const int m = blockIdx.y;
  int cnt = 0;
  const uint32_t thresh = a.sample_thresh ? a.sample_thresh[m] : 0u;
  const unsigned long long seed = (thresh && a.seed) ? *a.seed : 0ull;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < a.B * a.T; e += gridDim.x * blockDim.x) {
    const int b = e / a.T, t = e - b * a.T;
    const long long at = a.attn[m][(long long)b * a.attn_sb[m] + (long long)t * a.attn_st[m]];
    long long mk;
    if (thresh) {   // device-side Bernoulli(ratio) field (Masker temporal mode, models/masker.py:85-86,132)
      const uint4 w = philox4x32((uint32_t)(e >> 2), 0u, MMFM_MASK_SITE + (uint32_t)m, 2u, (uint32_t)seed,
                                 (uint32_t)(seed >> 32));
      const uint32_t word = (e & 3) == 0 ? w.x : (e & 3) == 1 ? w.y : (e & 3) == 2 ? w.z : w.w;
      mk = word < thresh;
    } else {
      mk = a.mask[m] ? a.mask[m][(long long)b * a.mask_sb[m] + (long long)t * a.mask_st[m]] : 0;
    }
    mk &= at;  // mm.py:270
    const long long o = (long long)b * S + m * a.T + t;
    key_valid[o] = at != 0;
    tok_mask[o] = (unsigned char)(mk != 0);
    if (b == 0) zero_flags[m * a.T + t] = (mk == 1);
    cnt += (int)mk;  // mask entries are 0/1 (mm.py:231 sums the expanded mask)
  }
  const float c = block_sum((float)cnt, sh);  // exact: counts < 2^24
  if (threadIdx.x == 0) {
    atomicAdd(&g_mp_count[m], (unsigned int)(c + 0.5f));
    __threadfence();
    const unsigned int ticket = atomicAdd(&g_mp_ticket, 1u);
    if (ticket == gridDim.x * gridDim.y - 1) {   // every other CTA's count is in
      __threadfence();
      long long total = 0;
      for (int mm = 0; mm < a.n_mod; ++mm) {
        const long long n = (long long)atomicExch(&g_mp_count[mm], 0u) * a.channels[mm];
        n_examples[mm] = n;
        total += n;
      }
      inv_n[0] = 1.0f / (float)total;  // total == 0 -> inf (reference: NaN loss)
      g_mp_ticket = 0u;
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// embedding assembly
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) embed_assemble_kernel(const float* __restrict__ mod_row,
                                                              const float* __restrict__ pos,
                                                              const long long* __restrict__ ts, float* __restrict__ emb,
                                                              int B, int T, int S, int off, int H) {
  const int hv = H >> 2;
  const long long total = (long long)B * T * hv;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long r = e / hv;
    const int c = (int)(e - r * hv);
    const long long b = r / T;
    const int t = (int)(r - b * T);
    float4 v = __ldg(reinterpret_cast<const float4*>(mod_row) + c);
    if (pos) {
      const float4 pv = __ldg(reinterpret_cast<const float4*>(pos + ts[r] * H) + c);
      v.x += pv.x; v.y += pv.y; v.z += pv.z; v.w += pv.w;
    }
    reinterpret_cast<float4*>(emb + (b * S + off + t) * H)[c] = v;
  }
}

// grid (T, B-chunks); block = (H/4 float4 column groups) x kAsmLanes sample lanes: lane l walks samples b0+l, b0+l+L, ..
// so several independent row loads are in flight per column group.  Consecutive samples of a lane that hit the same
// position row are summed in registers before one red.global per column; the modality-embedding sums of the lanes are
// combined in shared memory (one atomic per column per CTA).
constexpr int kAsmLanes = 4;
constexpr int kModReplicas = 16;
__device__ float g_dmod_scratch[kModReplicas][1024];   // H <= 1024 (checked by the launcher); all zero between launches
__device__ unsigned int g_dmod_ticket;
// DET (called with dpos == NULL; embed_pos_bwd_det_kernel below owns dpos): the CTA's modality-embedding sum goes to
// its workspace slot and det_tree_fold adds the slots up, instead of the scratch replicas.
template <bool DET = false>
__global__ void embed_assemble_bwd_kernel(const float* __restrict__ g, const float* __restrict__ g2,
                                          const long long* __restrict__ ts, float* __restrict__ dpos,
                                          float* __restrict__ dmod, int B, int T, int S, int off, int H, int bchunk,
                                          float4* __restrict__ ws, unsigned int* tickets) {
  extern __shared__ float4 sm_acc[];                      // [kAsmLanes][H/4]
  const int t = blockIdx.x;
  const int b0 = blockIdx.y * bchunk, b1 = min(B, b0 + bchunk);
  const int ncol = H >> 2;
  const int c = threadIdx.x % ncol, sl = threadIdx.x / ncol;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f), accm = acc;
  long long cur = -1;
  if (sl < kAsmLanes) {
    // four samples per round: all their row loads are issued before the first use (same summation order)
    constexpr int kU = 4;
    for (int bb = b0 + sl; bb < b1; bb += kAsmLanes * kU) {
      float4 v[kU];
      long long id[kU];
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        const int b = bb + u * kAsmLanes;
        v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        id[u] = -1;
        if (b < b1) {
          const long long row = ((long long)b * S + off + t) * H;
          v[u] = __ldg(reinterpret_cast<const float4*>(g + row) + c);
          if (g2) {
            const float4 w = __ldg(reinterpret_cast<const float4*>(g2 + row) + c);
            v[u].x += w.x; v[u].y += w.y; v[u].z += w.z; v[u].w += w.w;
          }
          if (!DET && dpos) id[u] = ts[(long long)b * T + t];
        }
      }
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        if (bb + u * kAsmLanes >= b1) break;
        accm.x += v[u].x; accm.y += v[u].y; accm.z += v[u].z; accm.w += v[u].w;
        if (!DET && dpos) {
          const long long idx = id[u];
          if (idx != cur) {
            if (cur >= 0) {
              float* d = dpos + cur * H + c * 4;
              atomicAdd(d, acc.x); atomicAdd(d + 1, acc.y); atomicAdd(d + 2, acc.z); atomicAdd(d + 3, acc.w);
            }
            cur = idx;
            acc = make_float4(0.f, 0.f, 0.f, 0.f);
          }
          acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w;
        }
      }
    }
    if (!DET && dpos && cur >= 0) {
      float* d = dpos + cur * H + c * 4;
      atomicAdd(d, acc.x); atomicAdd(d + 1, acc.y); atomicAdd(d + 2, acc.z); atomicAdd(d + 3, acc.w);
    }
    sm_acc[sl * ncol + c] = accm;
  }
  __syncthreads();
  if constexpr (DET) {
    const int leaf = blockIdx.x + blockIdx.y * gridDim.x;
    if (sl == 0) {
      float4 tot = sm_acc[c];
#pragma unroll
      for (int l = 1; l < kAsmLanes; ++l) tot = det_add(tot, sm_acc[l * ncol + c]);
      ws[(long long)leaf * ncol + c] = tot;
    }
    det_tree_fold(ws, ncol, ncol, leaf, gridDim.x * gridDim.y, tickets, [&](int i, float4 v) {
      float4* d = reinterpret_cast<float4*>(dmod) + i;
      *d = det_add(*d, v);
    });
    return;
  }
  // Modality-embedding gradient = sum over ALL rows: hundreds of CTAs adding to the same H addresses serialise in L2
  // (600 atomics per address at B = 256), so the CTAs spread their sums over kModReplicas scratch copies and the last
  // CTA to finish (ticket) folds the copies into dmod and clears them for the next launch.  (One launch in flight per
  // device at a time: the engine issues them on its single stream.)
  __shared__ bool s_last;
  if (sl == 0) {
    float4 tot = sm_acc[c];
#pragma unroll
    for (int l = 1; l < kAsmLanes; ++l) {
      const float4 o = sm_acc[l * ncol + c];
      tot.x += o.x; tot.y += o.y; tot.z += o.z; tot.w += o.w;
    }
    float* dm = g_dmod_scratch[(blockIdx.x + blockIdx.y * gridDim.x) % kModReplicas] + c * 4;
    atomicAdd(dm, tot.x); atomicAdd(dm + 1, tot.y); atomicAdd(dm + 2, tot.z); atomicAdd(dm + 3, tot.w);
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(&g_dmod_ticket, 1u) == gridDim.x * gridDim.y - 1;
  __syncthreads();
  if (s_last) {
    __threadfence();
    for (int col = threadIdx.x; col < H; col += blockDim.x) {
      float sum = 0.f;
#pragma unroll
      for (int r = 0; r < kModReplicas; ++r) sum += atomicExch(&g_dmod_scratch[r][col], 0.f);
      atomicAdd(dmod + col, sum);
    }
    if (threadIdx.x == 0) g_dmod_ticket = 0u;
  }
}

// Deterministic position-embedding gradient: CTA p owns row p of dpos and sums the gradient rows of every (b, t) with
// ts[b, t] == p.  The CTA scans ts in chunks of 1024 (b * T + t order), compacts the hits of a chunk in order, and its
// thread groups (256 / (H/4) of them, one float4 column per thread) take the hits round-robin; the group sums are added
// in group order at the end.  The summation order depends only on ts, so repeated and permuted timestamps are fine.
constexpr int kPosScan = 4;   // ts entries per thread per chunk
__global__ void __launch_bounds__(256) embed_pos_bwd_det_kernel(const float* __restrict__ g, const float* __restrict__ g2,
                                                                const long long* __restrict__ ts, float* __restrict__ dpos,
                                                                int B, int T, int S, int off, int H) {
  __shared__ int list[256 * kPosScan];
  __shared__ int wsum[8];
  __shared__ float4 gsum[256];
  const int p = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ncol = H >> 2, groups = 256 / ncol;
  const int grp = threadIdx.x / ncol, c = threadIdx.x - grp * ncol;
  const int BT = B * T;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int e0 = 0; e0 < BT; e0 += 256 * kPosScan) {
    const int eb = e0 + threadIdx.x * kPosScan;
    unsigned int hit = 0u;
#pragma unroll
    for (int u = 0; u < kPosScan; ++u)
      if (eb + u < BT && __ldg(ts + eb + u) == p) hit |= 1u << u;
    const int nh = __popc(hit);
    int x = nh;   // inclusive warp scan of the hit counts
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) wsum[warp] = x;
    __syncthreads();
    int pos = x - nh, total = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
      if (w < warp) pos += wsum[w];
      total += wsum[w];
    }
#pragma unroll
    for (int u = 0; u < kPosScan; ++u)
      if (hit & (1u << u)) list[pos++] = eb + u;
    __syncthreads();
    if (grp < groups) {
      for (int k = grp; k < total; k += groups) {
        const int e = list[k];
        const int b = e / T, t = e - b * T;
        const long long row = ((long long)b * S + off + t) * H;
        float4 v = __ldg(reinterpret_cast<const float4*>(g + row) + c);
        if (g2) v = det_add(v, __ldg(reinterpret_cast<const float4*>(g2 + row) + c));
        acc = det_add(acc, v);
      }
    }
    __syncthreads();   // list / wsum are rewritten by the next chunk
  }
  if (grp < groups) gsum[threadIdx.x] = acc;
  __syncthreads();
  if (grp == 0) {
    float4 tot = gsum[c];
    for (int j = 1; j < groups; ++j) tot = det_add(tot, gsum[j * ncol + c]);
    float4* d = reinterpret_cast<float4*>(dpos + (long long)p * H) + c;
    *d = det_add(*d, tot);
  }
}

__global__ void __launch_bounds__(256) embed_grad_prep_kernel(const float* __restrict__ dx, bf16* __restrict__ dtok,
                                                               const unsigned char* __restrict__ row_zero, DropCfg drop,
                                                               int B, int T, int S, int off, int H) {
  const int hv = H >> 2;
  const long long total = (long long)B * T * hv;
  unsigned long long seed = 0ull;
  if (drop.thresh != 0u) seed = *drop.seed;
  const uint32_t gpr = (uint32_t)((H + 15) >> 4);
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long r = e / hv;
    const int c = (int)(e - r * hv) * 4;
    const long long b = r / T;
    const int t = (int)(r - b * T);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!(row_zero && row_zero[off + t])) {
      v = __ldg(reinterpret_cast<const float4*>(dx + (b * S + off + t) * H + c));
      if (drop.thresh != 0u) {
        const uint4 w = drop_bytes16(seed, drop.site, (uint64_t)r, gpr, (uint32_t)(c >> 4));
        const int b0 = c & 15;
        v.x = drop_byte(w, b0) < drop.thresh ? 0.f : v.x * drop.scale;
        v.y = drop_byte(w, b0 + 1) < drop.thresh ? 0.f : v.y * drop.scale;
        v.z = drop_byte(w, b0 + 2) < drop.thresh ? 0.f : v.z * drop.scale;
        v.w = drop_byte(w, b0 + 3) < drop.thresh ? 0.f : v.w * drop.scale;
      }
    }
    uint2 o;
    o.x = pack_bf16x2(v.x, v.y);
    o.y = pack_bf16x2(v.z, v.w);
    *reinterpret_cast<uint2*>(dtok + r * H + c) = o;
  }
}

// ------------------------------------------------------------------------------------------------------------
// small-channel embedder (C <= 8 -> hidden 2C <= 16): SIMT
// ------------------------------------------------------------------------------------------------------------
constexpr int kMaxC = 8;
constexpr int kMaxC2 = 16;

MMFM_DEVINL float act_fwd(float v, int act, float scale) {
  if (act == MMFM_ACT_SOFTSIGN) v = softsign(v);
  return v * scale;
}

// one CTA per token row; threads stride over H
__global__ void __launch_bounds__(256) smallc_embed_fwd_kernel(const float* __restrict__ in, const float* __restrict__ W1,
                                                                const float* __restrict__ b1, const float* __restrict__ W2,
                                                                const float* __restrict__ b2, const float* __restrict__ emb,
                                                                float* __restrict__ x, float* __restrict__ hid,
                                                                const unsigned char* __restrict__ row_zero, DropCfg drop,
                                                                float act_scale, int act, int B, int T, int S, int off,
                                                                int C, int H) {
  __shared__ float sh[kMaxC2];
  const long long r = blockIdx.x;
  const long long b = r / T;
  const int t = (int)(r - b * T);
  const int C2 = 2 * C;
  if (threadIdx.x < C2) {
    float a = b1 ? b1[threadIdx.x] : 0.f;
    for (int c = 0; c < C; ++c) a += in[r * C + c] * W1[threadIdx.x * C + c];
    a = act_fwd(a, act, act_scale);
    sh[threadIdx.x] = a;
    hid[r * C2 + threadIdx.x] = a;
  }
  __syncthreads();
  const bool zero = row_zero && row_zero[off + t];
  unsigned long long seed = 0ull;
  if (drop.thresh != 0u) seed = *drop.seed;
  const uint32_t gpr = (uint32_t)((H + 15) >> 4);
  const long long orow = (b * S + off + t) * H;
  for (int h = threadIdx.x; h < H; h += blockDim.x) {
    float v = b2 ? b2[h] : 0.f;
    for (int j = 0; j < C2; ++j) v += sh[j] * W2[h * C2 + j];
    if (drop.thresh != 0u)
      v = drop_byte_at(seed, drop.site, (uint64_t)r, gpr, (uint32_t)h) < drop.thresh ? 0.f : v * drop.scale;
    if (zero) v = 0.f;
    x[orow + h] = v + emb[orow + h];
  }
}

// CTA = chunk of rows, thread = hidden column h (blockDim == H <= 1024).  Register partials for dW2/db2 (thread h)
// and dW1/db1 (threads j < 2C); flushed with atomics at the end.
// Deterministic mode: a CTA's partial gradients go to its workspace slot laid out as the outputs,
// [db2 (H) | dW2 (H x 2C) | db1 (2C) | dW1 (2C x C)], and det_tree_fold adds the slots into them.
MMFM_DEVINL int smallc_embed_slot(int H, int C) { return H * (1 + 2 * C) + 2 * C * (1 + C); }
MMFM_DEVINL void smallc_embed_emit(int i, float v, int H, int C, float* dW1, float* db1, float* dW2, float* db2) {
  const int C2 = 2 * C;
  if (i < H) db2[i] += v;
  else if ((i -= H) < H * C2) dW2[i] += v;
  else if ((i -= H * C2) < C2) db1[i] += v;
  else dW1[i - C2] += v;
}

template <bool DET = false>
__global__ void smallc_embed_bwd_kernel(const float* __restrict__ in, const float* __restrict__ hid,
                                        const float* __restrict__ W2, const float* __restrict__ dx,
                                        const unsigned char* __restrict__ row_zero, DropCfg drop, float act_scale, int act,
                                        float* __restrict__ dW1, float* __restrict__ db1, float* __restrict__ dW2,
                                        float* __restrict__ db2, int B, int T, int S, int off, int C, int H,
                                        int rows_per_cta, float* __restrict__ ws, unsigned int* tickets) {
  __shared__ float red[32][kMaxC2 + 1];
  const int h = threadIdx.x, warp = h >> 5, lane = h & 31, nw = blockDim.x >> 5;
  const int C2 = 2 * C;
  const long long R = (long long)B * T;
  const long long r0 = (long long)blockIdx.x * rows_per_cta, r1 = min(R, r0 + rows_per_cta);
  unsigned long long seed = 0ull;
  if (drop.thresh != 0u) seed = *drop.seed;
  const uint32_t gpr = (uint32_t)((H + 15) >> 4);
  float w2[kMaxC2], aw2[kMaxC2], aw1[kMaxC];
  float ab2 = 0.f, ab1 = 0.f;
#pragma unroll
  for (int j = 0; j < kMaxC2; ++j) {
    w2[j] = (j < C2) ? W2[h * C2 + j] : 0.f;
    aw2[j] = 0.f;
  }
#pragma unroll
  for (int c = 0; c < kMaxC; ++c) aw1[c] = 0.f;
  for (long long r = r0; r < r1; ++r) {
    const long long b = r / T;
    const int t = (int)(r - b * T);
    float d = 0.f;
    if (!(row_zero && row_zero[off + t])) {
      d = dx[(b * S + off + t) * H + h];
      if (drop.thresh != 0u)
        d = drop_byte_at(seed, drop.site, (uint64_t)r, gpr, (uint32_t)h) < drop.thresh ? 0.f : d * drop.scale;
    }
    ab2 += d;
#pragma unroll
    for (int j = 0; j < kMaxC2; ++j) {
      if (j < C2) {
        aw2[j] += d * __ldg(hid + r * C2 + j);
        const float pj = warp_sum(d * w2[j]);
        if (lane == 0) red[warp][j] = pj;
      }
    }
    __syncthreads();
    if (h < C2) {
      float dh = 0.f;
      for (int w = 0; w < nw; ++w) dh += red[w][h];
      // derivative of act(v)*scale expressed through the saved output a = hid
      if (act == MMFM_ACT_SOFTSIGN) {
        const float a = hid[r * C2 + h];
        const float tt = 1.0f - fabsf(a / act_scale);
        dh *= act_scale * tt * tt;
      } else {
        dh *= act_scale;
      }
      ab1 += dh;
#pragma unroll
      for (int c = 0; c < kMaxC; ++c)
        if (c < C) aw1[c] += dh * in[r * C + c];
    }
    __syncthreads();
  }
  if constexpr (DET) {
    const int n = smallc_embed_slot(H, C);
    float* slot = ws + (long long)blockIdx.x * n;
    slot[h] = ab2;
#pragma unroll
    for (int j = 0; j < kMaxC2; ++j)
      if (j < C2) slot[H + h * C2 + j] = aw2[j];
    if (h < C2) {
      slot[H + H * C2 + h] = ab1;
#pragma unroll
      for (int c = 0; c < kMaxC; ++c)
        if (c < C) slot[H + H * C2 + C2 + h * C + c] = aw1[c];
    }
    det_tree_fold(ws, n, n, blockIdx.x, gridDim.x, tickets,
                  [&](int i, float v) { smallc_embed_emit(i, v, H, C, dW1, db1, dW2, db2); });
    return;
  }
  atomicAdd(db2 + h, ab2);
#pragma unroll
  for (int j = 0; j < kMaxC2; ++j)
    if (j < C2) atomicAdd(dW2 + h * C2 + j, aw2[j]);
  if (h < C2) {
    atomicAdd(db1 + h, ab1);
#pragma unroll
    for (int c = 0; c < kMaxC; ++c)
      if (c < C) atomicAdd(dW1 + h * C + c, aw1[c]);
  }
}

// ---- fast path of the small-channel embedder for C <= 2 (the model's behaviour streams): a thread owns 16 consecutive
// hidden columns of a row, i.e. exactly one Philox group, so the dropout stream costs one Philox call per 16 outputs
// (the row-per-CTA kernels above run one call per output element and are bound by it).  gridDim * blockDim is a multiple
// of the groups per row, so a thread's column group -- and with it its slice of W2 -- is fixed for the whole loop.
template <int C>
__global__ void __launch_bounds__(256) smallc_embed_fwd16_kernel(
    const float* __restrict__ in, const float* __restrict__ W1, const float* __restrict__ b1, const float* __restrict__ W2,
    const float* __restrict__ b2, const float* __restrict__ emb, float* __restrict__ x, float* __restrict__ hid,
    const unsigned char* __restrict__ row_zero, DropCfg drop, float act_scale, int act, int B, int T, int S, int off, int H) {
  constexpr int C2 = 2 * C;
  const int gpr = H >> 4;                                   // 16-column groups per row
  const long long slots = (long long)B * T * gpr;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long slot0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int g = (int)(slot0 % gpr);
  unsigned long long seed = 0ull;
  if (drop.thresh != 0u) seed = *drop.seed;
  float w1[C2][C], bb1[C2], w2[16][C2], bb2[16];
#pragma unroll
  for (int j = 0; j < C2; ++j) {
    bb1[j] = b1 ? b1[j] : 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) w1[j][c] = W1[j * C + c];
  }
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    bb2[k] = b2 ? b2[16 * g + k] : 0.f;
#pragma unroll
    for (int j = 0; j < C2; ++j) w2[k][j] = W2[(16 * g + k) * C2 + j];
  }
  for (long long slot = slot0; slot < slots; slot += stride) {
    const long long r = slot / gpr;
    const long long b = r / T;
    const int t = (int)(r - b * T);
    float hj[C2];
#pragma unroll
    for (int j = 0; j < C2; ++j) {
      float a = bb1[j];
#pragma unroll
      for (int c = 0; c < C; ++c) a = fmaf(__ldg(in + r * C + c), w1[j][c], a);
      hj[j] = act_fwd(a, act, act_scale);
      if (g == 0) hid[r * C2 + j] = hj[j];
    }
    const bool zero = row_zero && row_zero[off + t];
    uint4 w = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
    if (drop.thresh != 0u) w = drop_bytes16(seed, drop.site, (uint64_t)r, (uint32_t)gpr, (uint32_t)g);
    const long long orow = (b * S + off + t) * H + 16 * g;
#pragma unroll
    for (int k4 = 0; k4 < 16; k4 += 4) {
      const float4 e = __ldg(reinterpret_cast<const float4*>(emb + orow + k4));
      float v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        float a = bb2[k4 + u];
#pragma unroll
        for (int j = 0; j < C2; ++j) a = fmaf(hj[j], w2[k4 + u][j], a);
        if (drop.thresh != 0u) a = drop_byte(w, k4 + u) < drop.thresh ? 0.f : a * drop.scale;
        v[u] = zero ? 0.f : a;
      }
      *reinterpret_cast<float4*>(x + orow + k4) = make_float4(v[0] + e.x, v[1] + e.y, v[2] + e.z, v[3] + e.w);
    }
  }
}

template <int C, bool DET = false>
__global__ void __launch_bounds__(256) smallc_embed_bwd16_kernel(
    const float* __restrict__ in, const float* __restrict__ hid, const float* __restrict__ W2, const float* __restrict__ dx,
    const unsigned char* __restrict__ row_zero, DropCfg drop, float act_scale, int act, float* __restrict__ dW1,
    float* __restrict__ db1, float* __restrict__ dW2, float* __restrict__ db2, int B, int T, int S, int off, int H,
    float* __restrict__ ws, unsigned int* tickets) {
  constexpr int C2 = 2 * C;
  __shared__ float red[4096 + 256];                         // [CTA row slot][H + 1]: (256/gpr) * (16 gpr + 1) floats
  const int gpr = H >> 4;                                   // 16-column groups per row: a power of two <= 32
  const long long slots = (long long)B * T * gpr;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const int lane = threadIdx.x & 31;
  const long long slot0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int g = (int)(slot0 % gpr);
  unsigned long long seed = 0ull;
  if (drop.thresh != 0u) seed = *drop.seed;
  float w2[16][C2], ab2[16], aw2[16][C2], aw1[C2][C], ab1[C2];
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    ab2[k] = 0.f;
#pragma unroll
    for (int j = 0; j < C2; ++j) aw2[k][j] = 0.f;
  }
  {   // this thread's slice of W2 (16 rows x C2) is contiguous: vector loads instead of 16 * C2 scalar ones
    const float* wsrc = W2 + (size_t)16 * g * C2;
    if constexpr (C2 % 4 == 0) {
#pragma unroll
      for (int q = 0; q < 16 * C2 / 4; ++q) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(wsrc) + q);
        w2[(4 * q) / C2][(4 * q) % C2] = t.x; w2[(4 * q + 1) / C2][(4 * q + 1) % C2] = t.y;
        w2[(4 * q + 2) / C2][(4 * q + 2) % C2] = t.z; w2[(4 * q + 3) / C2][(4 * q + 3) % C2] = t.w;
      }
    } else {
#pragma unroll
      for (int q = 0; q < 16 * C2 / 2; ++q) {
        const float2 t = __ldg(reinterpret_cast<const float2*>(wsrc) + q);
        w2[(2 * q) / C2][(2 * q) % C2] = t.x; w2[(2 * q + 1) / C2][(2 * q + 1) % C2] = t.y;
      }
    }
  }
#pragma unroll
  for (int j = 0; j < C2; ++j) {
    ab1[j] = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) aw1[j][c] = 0.f;
  }
  // the loop bound is warp-uniform (the shuffles below need all 32 lanes); a row past the end contributes zeros
  for (long long wb = slot0 - lane; wb < slots; wb += stride) {
    const long long slot = wb + lane;
    const bool valid = slot < slots;
    const int gshift = 31 - __clz(gpr);                       // gpr is a power of two
    const long long r = valid ? (slot >> gshift) : 0;
    const int b = (int)r / T;                                  // B * T < 2^31
    const int t = (int)r - b * T;
    float d[16];
    const bool zero = !valid || (row_zero && row_zero[off + t]);
    const long long orow = ((long long)b * S + off + t) * H + 16 * g;
#pragma unroll
    for (int k4 = 0; k4 < 16; k4 += 4) {
      const float4 v = zero ? make_float4(0.f, 0.f, 0.f, 0.f) : __ldg(reinterpret_cast<const float4*>(dx + orow + k4));
      d[k4] = v.x; d[k4 + 1] = v.y; d[k4 + 2] = v.z; d[k4 + 3] = v.w;
    }
    if (drop.thresh != 0u && !zero) {
      const uint4 w = drop_bytes16(seed, drop.site, (uint64_t)r, (uint32_t)gpr, (uint32_t)g);
#pragma unroll
      for (int k = 0; k < 16; ++k) d[k] = drop_byte(w, k) < drop.thresh ? 0.f : d[k] * drop.scale;
    }
    float hj[C2], dh[C2], xin[C];
#pragma unroll
    for (int j = 0; j < C2; ++j) { hj[j] = __ldg(hid + r * C2 + j); dh[j] = 0.f; }
#pragma unroll
    for (int c = 0; c < C; ++c) xin[c] = __ldg(in + r * C + c);   // (in flight with the rest: its consumer waited 16 % of the kernel)
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      ab2[k] += d[k];
#pragma unroll
      for (int j = 0; j < C2; ++j) {
        aw2[k][j] = fmaf(d[k], hj[j], aw2[k][j]);
        dh[j] = fmaf(d[k], w2[k][j], dh[j]);
      }
    }
    // sum dh over the gpr lanes of the row
#pragma unroll
    for (int j = 0; j < C2; ++j)
      for (int o = gpr >> 1; o > 0; o >>= 1) dh[j] += __shfl_xor_sync(0xffffffffu, dh[j], o);
    if (g == 0 && valid) {
#pragma unroll
      for (int j = 0; j < C2; ++j) {
        float v = dh[j];
        if (act == MMFM_ACT_SOFTSIGN) {   // derivative of act(v)*scale through the saved output a = hid
          const float tt = 1.0f - fabsf(hj[j] / act_scale);
          v *= act_scale * tt * tt;
        } else {
          v *= act_scale;
        }
        ab1[j] += v;
#pragma unroll
        for (int c = 0; c < C; ++c) aw1[j][c] = fmaf(v, xin[c], aw1[j][c]);
      }
    }
  }
  // ---- flush: (1 + C2) CTA-wide column reductions over the threads that share a column group, one atomic per column ----
  const int trow = threadIdx.x / gpr, nrow = 256 / gpr, pitch = H + 1;
#pragma unroll
  for (int q = 0; q <= C2; ++q) {
#pragma unroll
    for (int k = 0; k < 16; ++k) red[trow * pitch + 16 * g + k] = (q == 0) ? ab2[k] : aw2[k][q == 0 ? 0 : q - 1];
    __syncthreads();
    for (int col = threadIdx.x; col < H; col += 256) {
      float sum = 0.f;
      for (int rr = 0; rr < nrow; ++rr) sum += red[rr * pitch + col];
      if constexpr (DET) ws[(long long)blockIdx.x * smallc_embed_slot(H, C) + (q == 0 ? col : H + col * C2 + (q - 1))] = sum;
      else if (q == 0) atomicAdd(db2 + col, sum);
      else atomicAdd(dW2 + col * C2 + (q - 1), sum);
    }
    __syncthreads();
  }
  if constexpr (DET) {   // the embedder-input gradients of the g == 0 threads, reduced in thread order
    constexpr int kIn = C2 * (1 + C);
    if (g == 0) {
#pragma unroll
      for (int j = 0; j < C2; ++j) {
        red[trow * kIn + j] = ab1[j];
#pragma unroll
        for (int c = 0; c < C; ++c) red[trow * kIn + C2 + j * C + c] = aw1[j][c];
      }
    }
    __syncthreads();
    const int n = smallc_embed_slot(H, C);
    if (threadIdx.x < kIn) {
      float sum = 0.f;
      for (int rr = 0; rr < nrow; ++rr) sum += red[rr * kIn + threadIdx.x];
      ws[(long long)blockIdx.x * n + H * (1 + C2) + threadIdx.x] = sum;
    }
    det_tree_fold(ws, n, n, blockIdx.x, gridDim.x, tickets,
                  [&](int i, float v) { smallc_embed_emit(i, v, H, C, dW1, db1, dW2, db2); });
    return;
  }
  if (g == 0) {
#pragma unroll
    for (int j = 0; j < C2; ++j) {
      atomicAdd(db1 + j, ab1[j]);
#pragma unroll
      for (int c = 0; c < C; ++c) atomicAdd(dW1 + j * C + c, aw1[j][c]);
    }
  }
}

// head forward, C <= 8: warp per row
__global__ void __launch_bounds__(256) smallc_head_fwd_kernel(const bf16* __restrict__ y, const float* __restrict__ W,
                                                               const float* __restrict__ bias, float* __restrict__ preds,
                                                               int R, int H, int C) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (long long r = (long long)blockIdx.x * 8 + warp; r < R; r += (long long)gridDim.x * 8) {
    float acc[kMaxC];
#pragma unroll
    for (int c = 0; c < kMaxC; ++c) acc[c] = 0.f;
    for (int h0 = lane * 8; h0 < H; h0 += 256) {
      const uint4 v = __ldg(reinterpret_cast<const uint4*>(y + r * H + h0));
      const float2 f[4] = {unpack_bf16x2(v.x), unpack_bf16x2(v.y), unpack_bf16x2(v.z), unpack_bf16x2(v.w)};
#pragma unroll
      for (int c = 0; c < kMaxC; ++c) {
        if (c < C) {
          const float* w = W + (long long)c * H + h0;
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[c] += f[j].x * __ldg(w + 2 * j) + f[j].y * __ldg(w + 2 * j + 1);
        }
      }
    }
#pragma unroll
    for (int c = 0; c < kMaxC; ++c) {
      if (c < C) {
        const float s = warp_sum(acc[c]);
        if (lane == 0) preds[r * C + c] = s + (bias ? bias[c] : 0.f);
      }
    }
  }
}

// head backward, C <= 8: grid (row chunks, H/256); lane owns 8 consecutive columns of the 256-wide slice
// DET: workspace slot per CTA = [dW slice (kMaxC x 256) | db (kMaxC)]; one tree per 256-column slice (blockIdx.y)
constexpr int kHeadSlot = kMaxC * 256 + kMaxC;
template <bool DET = false>
__global__ void __launch_bounds__(256) smallc_head_bwd_kernel(const bf16* __restrict__ y, const float* __restrict__ W,
                                                               const bf16* __restrict__ dp, long long lddp,
                                                               bf16* __restrict__ dy, float* __restrict__ dW,
                                                               float* __restrict__ db, int R, int H, int C,
                                                               float* __restrict__ ws, unsigned int* tickets) {
  __shared__ float red[8][256 + 1];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h0 = blockIdx.y * 256 + lane * 8;
  const bool hok = h0 < H;
  float w[kMaxC][8], aw[kMaxC][8], ab[kMaxC];
#pragma unroll
  for (int c = 0; c < kMaxC; ++c) {
    ab[c] = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      w[c][j] = (c < C && hok) ? W[(long long)c * H + h0 + j] : 0.f;
      aw[c][j] = 0.f;
    }
  }
  for (long long r = (long long)blockIdx.x * 8 + warp; r < R; r += (long long)gridDim.x * 8) {
    float d[kMaxC];
#pragma unroll
    for (int c = 0; c < kMaxC; ++c) {
      d[c] = (c < C) ? __bfloat162float(dp[r * lddp + c]) : 0.f;
      ab[c] += d[c];
    }
    if (hok) {
      const uint4 v = __ldg(reinterpret_cast<const uint4*>(y + r * H + h0));
      const float2 f[4] = {unpack_bf16x2(v.x), unpack_bf16x2(v.y), unpack_bf16x2(v.z), unpack_bf16x2(v.w)};
      float o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = 0.f;
#pragma unroll
      for (int c = 0; c < kMaxC; ++c) {
        if (c < C) {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            aw[c][2 * j] += d[c] * f[j].x;
            aw[c][2 * j + 1] += d[c] * f[j].y;
            o[2 * j] += d[c] * w[c][2 * j];
            o[2 * j + 1] += d[c] * w[c][2 * j + 1];
          }
        }
      }
      uint4 ov;
      ov.x = pack_bf16x2(o[0], o[1]); ov.y = pack_bf16x2(o[2], o[3]);
      ov.z = pack_bf16x2(o[4], o[5]); ov.w = pack_bf16x2(o[6], o[7]);
      *reinterpret_cast<uint4*>(dy + r * H + h0) = ov;
    }
  }
#pragma unroll
  for (int c = 0; c < kMaxC; ++c) {
    if (c < C) {
#pragma unroll
      for (int j = 0; j < 8; ++j) red[warp][lane * 8 + j] = aw[c][j];
      __syncthreads();
      const int hh = threadIdx.x;
      float s = 0.f;
#pragma unroll
      for (int wv = 0; wv < 8; ++wv) s += red[wv][hh];
      if constexpr (DET) ws[((long long)blockIdx.y * gridDim.x + blockIdx.x) * kHeadSlot + c * 256 + hh] = s;
      else if (blockIdx.y * 256 + hh < H) atomicAdd(dW + (long long)c * H + blockIdx.y * 256 + hh, s);
      __syncthreads();
    }
  }
  if constexpr (DET) {
    float* slot = ws + ((long long)blockIdx.y * gridDim.x + blockIdx.x) * kHeadSlot;
    if (lane == 0) {
#pragma unroll
      for (int c = 0; c < kMaxC; ++c) red[warp][c] = ab[c];
    }
    __syncthreads();
    if (threadIdx.x < kMaxC) {
      float s = 0.f;
#pragma unroll
      for (int wv = 0; wv < 8; ++wv) s += red[wv][threadIdx.x];
      slot[kMaxC * 256 + threadIdx.x] = s;
    }
    det_tree_fold(ws + (long long)blockIdx.y * gridDim.x * kHeadSlot, kHeadSlot, kHeadSlot, blockIdx.x, gridDim.x,
                  tickets + (long long)blockIdx.y * gridDim.x, [&](int i, float v) {
                    const int c = i >> 8, hh = blockIdx.y * 256 + (i & 255);
                    if (i >= kMaxC * 256) {
                      if (blockIdx.y == 0 && i - kMaxC * 256 < C) db[i - kMaxC * 256] += v;
                    } else if (c < C && hh < H) {
                      dW[(long long)c * H + hh] += v;
                    }
                  });
    return;
  }
  if (blockIdx.y == 0 && lane == 0) {
#pragma unroll
    for (int c = 0; c < kMaxC; ++c)
      if (c < C) atomicAdd(db + c, ab[c]);
  }
}

// ------------------------------------------------------------------------------------------------------------
// fused masked loss + gradient
// ------------------------------------------------------------------------------------------------------------
template <int KIND>
MMFM_DEVINL void loss_elem(float pr, float tg, float& ell, float& grad) {
  if (KIND == MMFM_LOSS_POISSON) {
    const float e = __expf(pr);
    ell = e - tg * pr;
    grad = e - tg;
  } else {
    const float d = pr - tg;
    ell = d * d;
    grad = 2.0f * d;
  }
}

template <int KIND, bool VEC>
__global__ void __launch_bounds__(256) loss_kernel(const float* __restrict__ preds, const float* __restrict__ targets,
                                                    const unsigned char* __restrict__ tok_mask, int S, int off,
                                                    const float* __restrict__ inv_n, int B, int T, int C,
                                                    float* __restrict__ partials, bf16* __restrict__ dpreds,
                                                    long long lddp) {
  __shared__ float sh[32];
  const float invn = __ldg(inv_n);
  float acc = 0.f;
  if (VEC) {
    const int cv = C >> 2;
    const long long total = (long long)B * T * cv;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
      const long long r = e / cv;
      const int c = (int)(e - r * cv) * 4;
      const long long b = r / T;
      const int t = (int)(r - b * T);
      const bool mk = tok_mask[b * S + off + t] != 0;
      float g[4] = {0.f, 0.f, 0.f, 0.f};
      if (mk) {
        const float4 pv = __ldg(reinterpret_cast<const float4*>(preds + r * C + c));
        const float4 tv = __ldg(reinterpret_cast<const float4*>(targets + r * C + c));
        float l0, l1, l2, l3;
        loss_elem<KIND>(pv.x, tv.x, l0, g[0]);
        loss_elem<KIND>(pv.y, tv.y, l1, g[1]);
        loss_elem<KIND>(pv.z, tv.z, l2, g[2]);
        loss_elem<KIND>(pv.w, tv.w, l3, g[3]);
        acc += (l0 + l1) + (l2 + l3);
      }
      uint2 o;
      o.x = pack_bf16x2(g[0] * invn, g[1] * invn);
      o.y = pack_bf16x2(g[2] * invn, g[3] * invn);
      *reinterpret_cast<uint2*>(dpreds + r * lddp + c) = o;
    }
  } else {
    const long long total = (long long)B * T * C;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
      const long long r = e / C;
      const int c = (int)(e - r * C);
      const long long b = r / T;
      const int t = (int)(r - b * T);
      float g = 0.f;
      if (tok_mask[b * S + off + t]) {
        float l;
        loss_elem<KIND>(preds[e], targets[e], l, g);
        acc += l;
      }
      dpreds[r * lddp + c] = __float2bfloat16_rn(g * invn);
    }
  }
  const float s = block_sum(acc, sh);
  if (threadIdx.x == 0) partials[blockIdx.x] = s;
}

// Masked categorical cross-entropy over the class axis (the choice / block streams; BASELINE.json north_star -- an
// extension: the reference has no categorical modality, SURVEY.md section 0).  The loss module slots into the
// reference's forward_loss unchanged (mm.py:229-231): ell[b,t,k] = -targets[b,t,k] * log_softmax(preds[b,t,:])[k],
// summed under the (B,T)->(B,T,K) expanded mask and normalised by the expanded mask count like every other modality.
// thread = one token row (K <= kMaxClasses classes in registers); grad = mask * inv_n * (softmax * sum_k t_k - t).
constexpr int kMaxClasses = 64;
// d ell / d preds[c] of one row, from the row's max, 1 / sum_c exp(preds - max) and sum_c targets
MMFM_DEVINL float ce_grad_elem(float p, float t, float mx, float inv_se, float tsum) {
  return __expf(p - mx) * inv_se * tsum - t;
}
__global__ void __launch_bounds__(256) loss_ce_kernel(const float* __restrict__ preds, const float* __restrict__ targets,
                                                       const unsigned char* __restrict__ tok_mask, int S, int off,
                                                       const float* __restrict__ inv_n, int B, int T, int C,
                                                       float* __restrict__ partials, bf16* __restrict__ dpreds,
                                                       long long lddp) {
  __shared__ float sh[32];
  const float invn = __ldg(inv_n);
  float acc = 0.f;
  const long long rows = (long long)B * T;
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += (long long)gridDim.x * blockDim.x) {
    const long long b = r / T;
    const int t = (int)(r - b * T);
    const bool mk = tok_mask[b * S + off + t] != 0;
    const float* pr = preds + r * C;
    const float* tg = targets + r * C;
    bf16* dp = dpreds + r * lddp;
    if (!mk) {
      for (int c = 0; c < C; ++c) dp[c] = __float2bfloat16_rn(0.f);
      continue;
    }
    float mx = -INFINITY, tsum = 0.f;
    for (int c = 0; c < C; ++c) mx = fmaxf(mx, pr[c]);
    float se = 0.f;
    for (int c = 0; c < C; ++c) se += __expf(pr[c] - mx);
    const float lse = mx + __logf(se);
    for (int c = 0; c < C; ++c) {
      const float tc = tg[c];
      tsum += tc;
      acc -= tc * (pr[c] - lse);
    }
    const float inv_se = 1.0f / se;
    for (int c = 0; c < C; ++c) dp[c] = __float2bfloat16_rn(ce_grad_elem(pr[c], tg[c], mx, inv_se, tsum) * invn);
  }
  const float s = block_sum(acc, sh);
  if (threadIdx.x == 0) partials[blockIdx.x] = s;
}

__global__ void __launch_bounds__(256) loss_finalize_kernel(const float* __restrict__ partials, int n_partials, int n_mod,
                                                             const float* __restrict__ inv_n, float* __restrict__ mod_loss,
                                                             float* __restrict__ loss) {
  __shared__ float sh[32];
  float tot = 0.f;
  for (int m = 0; m < n_mod; ++m) {
    float a = 0.f;
    for (int i = threadIdx.x; i < n_partials; i += blockDim.x) a += partials[m * n_partials + i];
    const float s = block_sum(a, sh);
    if (threadIdx.x == 0) mod_loss[m] = s;
    tot += s;
  }
  if (threadIdx.x == 0) loss[0] = tot * inv_n[0];
}

// Head gradient for arbitrary upstream gradients of the step outputs (autograd of loss, mod_loss[m] and preds):
// dpreds = mask * ell' * (g_loss * inv_n + g_mod) + g_preds.  ell' comes from the device code of the two loss kernels
// above, so g_loss = 1 alone gives their dpreds bit for bit.  A term whose upstream gradient is absent is never
// evaluated (inv_n is inf when no token is masked).  g_preds is read through element strides: autograd hands the
// gradients of sum() / mean() over as stride-0 broadcasts.
MMFM_DEVINL float loss_grad_coef(const float* g_loss, const float* g_mod, const float* inv_n) {
  float coef = 0.f;
  if (g_loss) coef = __ldg(g_loss) * __ldg(inv_n);
  if (g_mod) coef += __ldg(g_mod);
  return coef;
}

template <int KIND>
__global__ void __launch_bounds__(256) loss_grad_kernel(const float* __restrict__ preds, const float* __restrict__ targets,
                                                         const unsigned char* __restrict__ tok_mask, int S, int off,
                                                         const float* __restrict__ inv_n, const float* g_loss,
                                                         const float* g_mod, const float* __restrict__ g_preds,
                                                         long long gp_sb, long long gp_st, long long gp_sc, int B, int T,
                                                         int C, bf16* __restrict__ dpreds, long long lddp) {
  const bool head = g_loss != nullptr || g_mod != nullptr;
  const float coef = head ? loss_grad_coef(g_loss, g_mod, inv_n) : 0.f;
  const long long total = (long long)B * T * C;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long r = e / C;
    const int c = (int)(e - r * C);
    const long long b = r / T;
    const int t = (int)(r - b * T);
    float v = 0.f;
    if (head && tok_mask[b * S + off + t]) {
      float l, g;
      loss_elem<KIND>(__ldg(preds + e), __ldg(targets + e), l, g);
      v = g * coef;
    }
    if (g_preds) v += __ldg(g_preds + b * gp_sb + t * gp_st + c * gp_sc);
    dpreds[r * lddp + c] = __float2bfloat16_rn(v);
  }
}

// categorical variant: thread = one token row, as loss_ce_kernel
__global__ void __launch_bounds__(256) loss_grad_ce_kernel(const float* __restrict__ preds, const float* __restrict__ targets,
                                                            const unsigned char* __restrict__ tok_mask, int S, int off,
                                                            const float* __restrict__ inv_n, const float* g_loss,
                                                            const float* g_mod, const float* __restrict__ g_preds,
                                                            long long gp_sb, long long gp_st, long long gp_sc, int B,
                                                            int T, int C, bf16* __restrict__ dpreds, long long lddp) {
  const bool head = g_loss != nullptr || g_mod != nullptr;
  const float coef = head ? loss_grad_coef(g_loss, g_mod, inv_n) : 0.f;
  const long long rows = (long long)B * T;
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += (long long)gridDim.x * blockDim.x) {
    const long long b = r / T;
    const int t = (int)(r - b * T);
    const float* pr = preds + r * C;
    const float* tg = targets + r * C;
    const float* gp = g_preds ? g_preds + b * gp_sb + t * gp_st : nullptr;
    bf16* dp = dpreds + r * lddp;
    if (head && tok_mask[b * S + off + t]) {
      float mx = -INFINITY, se = 0.f, tsum = 0.f;
      for (int c = 0; c < C; ++c) mx = fmaxf(mx, pr[c]);
      for (int c = 0; c < C; ++c) se += __expf(pr[c] - mx);
      for (int c = 0; c < C; ++c) tsum += tg[c];
      const float inv_se = 1.0f / se;
      for (int c = 0; c < C; ++c) {
        float v = ce_grad_elem(pr[c], tg[c], mx, inv_se, tsum) * coef;
        if (gp) v += gp[c * gp_sc];
        dp[c] = __float2bfloat16_rn(v);
      }
    } else {
      for (int c = 0; c < C; ++c) dp[c] = __float2bfloat16_rn(gp ? gp[c * gp_sc] : 0.f);
    }
  }
}

// Input gradient of the small-channel embedder: warp = one token row.  The lanes stride over H for the 2C dot products
// with W2 (butterfly sums, fixed order), then lane c < C forms dX[r, c] from the 2C hidden gradients.
__global__ void __launch_bounds__(256) smallc_embed_dx_kernel(const float* __restrict__ hid, const float* __restrict__ W1,
                                                               const float* __restrict__ W2, const float* __restrict__ dx,
                                                               const unsigned char* __restrict__ row_zero, DropCfg drop,
                                                               float act_scale, int act, float* __restrict__ dX,
                                                               long long lddx, int accumulate, int B, int T, int S,
                                                               int off, int C, int H) {
  const int lane = threadIdx.x & 31;
  const int C2 = 2 * C;
  const long long R = (long long)B * T;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  unsigned long long seed = 0ull;
  if (drop.thresh != 0u) seed = *drop.seed;
  const uint32_t gpr = (uint32_t)((H + 15) >> 4);
  for (long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < R; r += nwarps) {
    const long long b = r / T;
    const int t = (int)(r - b * T);
    float acc[kMaxC2];
#pragma unroll
    for (int j = 0; j < kMaxC2; ++j) acc[j] = 0.f;
    if (!(row_zero && row_zero[off + t])) {
      for (int h = lane; h < H; h += 32) {
        float d = __ldg(dx + (b * S + off + t) * H + h);
        if (drop.thresh != 0u)
          d = drop_byte_at(seed, drop.site, (uint64_t)r, gpr, (uint32_t)h) < drop.thresh ? 0.f : d * drop.scale;
#pragma unroll
        for (int j = 0; j < kMaxC2; ++j)
          if (j < C2) acc[j] += d * __ldg(W2 + h * C2 + j);
      }
    }
#pragma unroll
    for (int j = 0; j < kMaxC2; ++j) {
      if (j < C2) {
        float dh = warp_sum(acc[j]);
        // derivative of act(v)*scale expressed through the saved output a = hid (as smallc_embed_bwd_kernel)
        if (act == MMFM_ACT_SOFTSIGN) {
          const float tt = 1.0f - fabsf(__ldg(hid + r * C2 + j) / act_scale);
          dh *= act_scale * tt * tt;
        } else {
          dh *= act_scale;
        }
        acc[j] = dh;
      }
    }
    if (lane < C) {
      float v = 0.f;
#pragma unroll
      for (int j = 0; j < kMaxC2; ++j)
        if (j < C2) v += acc[j] * __ldg(W1 + j * C + lane);
      float* o = dX + r * lddx + lane;
      *o = accumulate ? *o + v : v;
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// multi-tensor fp32 -> bf16 cast (weight shadows): one launch for the whole parameter set
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) cast_multi_kernel(const mmfm_cast_item* __restrict__ items, int n_items) {
  __shared__ float tile[32][33];
  // locate the item of this tile (tile_start is an exclusive prefix sum)
  int lo = 0, hi = n_items - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (items[mid].tile_start <= (int)blockIdx.x) lo = mid; else hi = mid - 1;
  }
  const mmfm_cast_item it = items[lo];
  const int tl = blockIdx.x - it.tile_start;
  const int tcols = (it.cols + 31) >> 5;
  const int r0 = (tl / tcols) * 32, c0 = (tl % tcols) * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  bf16* y = reinterpret_cast<bf16*>(it.dst);
  bf16* yt = reinterpret_cast<bf16*>(it.dst_t);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = r0 + ty + i * 8, c = c0 + tx;
    float v = 0.f;
    if (r < it.rows && c < it.cols) {
      v = it.src[(long long)r * it.ld_src + c];
      if (y) y[(long long)r * it.ld_dst + c] = __float2bfloat16_rn(v);
    }
    tile[ty + i * 8][tx] = v;
  }
  if (yt == nullptr) return;
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c = c0 + ty + i * 8, r = r0 + tx;
    if (r < it.rows && c < it.cols) yt[(long long)c * it.ld_dst_t + r] = __float2bfloat16_rn(tile[tx][ty + i * 8]);
  }
}

// x[i] *= *scale (no-op launch when *scale == 1): applies the upstream gradient of the scalar loss
__global__ void __launch_bounds__(256) scale_inplace_kernel(float* __restrict__ x, long long n,
                                                             const float* __restrict__ scale) {
  const float s = __ldg(scale);
  if (s == 1.0f) return;
  const long long n4 = n >> 2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    float4 v = reinterpret_cast<float4*>(x)[i];
    v.x *= s; v.y *= s; v.z *= s; v.w *= s;
    reinterpret_cast<float4*>(x)[i] = v;
  }
  for (long long i = (n4 << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    x[i] *= s;
}

// Data-parallel multi-session step: every rank all-gathered its session id and its session's gradient slab (the
// session's ranges of the flat gradient, back to back).  Row y of the grid serves gathered slab y; only the first rank
// carrying a session writes it, as inv_world * (sum over the ranks carrying it, in ascending order, from 0.0f).  No
// atomics, and every rank computes the same bits.  Sessions no rank carries are neither read nor written.
__device__ __forceinline__ float4 f4_add(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }

__global__ void __launch_bounds__(256) session_grad_combine_kernel(float* __restrict__ grad,
                                                                   const float* __restrict__ gathered, int world,
                                                                   long long stride, const int* __restrict__ ids,
                                                                   const long long* __restrict__ ranges, int n_sessions,
                                                                   float inv_world) {
  const int r0 = blockIdx.y;
  const int s = ids[r0];
  if (s < 0 || s >= n_sessions) return;
  for (int r = 0; r < r0; ++r)
    if (ids[r] == s) return;                      // an earlier rank's CTA row writes this session
  const long long* rg = ranges + 4LL * s;
  const long long lo0 = rg[0], hi0 = rg[1], lo1 = rg[2], hi1 = rg[3];
  if (lo0 < 0 || hi0 < lo0 || lo1 < 0 || hi1 < lo1 || (hi0 - lo0) + (hi1 - lo1) > stride) return;   // malformed table
  const long long step = (long long)gridDim.x * blockDim.x, t0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long soff = 0;                             // position of the range inside the slab
  for (int part = 0; part < 2; ++part) {
    const long long lo = part ? lo1 : lo0, n = (part ? hi1 : hi0) - lo;
    float* dst = grad + lo;
    const float* src = gathered + soff;
    long long done = 0;
    if (((lo | soff | stride) & 3) == 0 && (((uintptr_t)grad | (uintptr_t)gathered) & 15) == 0) {
      const long long n4 = n >> 2;
      for (long long i = t0; i < n4; i += step) {
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int r = r0; r < world; ++r)
          if (ids[r] == s) acc = f4_add(acc, __ldg(reinterpret_cast<const float4*>(src + r * stride) + i));
        reinterpret_cast<float4*>(dst)[i] = make_float4(acc.x * inv_world, acc.y * inv_world, acc.z * inv_world,
                                                        acc.w * inv_world);
      }
      done = n4 << 2;
    }
    for (long long i = done + t0; i < n; i += step) {
      float acc = 0.f;
      for (int r = r0; r < world; ++r)
        if (ids[r] == s) acc += __ldg(src + r * stride + i);
      dst[i] = acc * inv_world;
    }
    soff += n;
  }
}

// Fused multi-tensor AdamW over the flat master-parameter / gradient buffers (torch.optim.AdamW semantics,
// reference train_multi_modal.py:197-202): p *= 1 - lr*wd ; m = b1 m + (1-b1) g ; v = b2 v + (1-b2) g^2 ;
// p -= (lr / bc1) * m / (sqrt(v) / sqrt(bc2) + eps).  One pass, 28 bytes of traffic per parameter.
// The update runs over segments [lo, hi) of the buffers, each with the hyper-parameters of its class (one parameter
// group at one step count); elements outside every segment are neither read nor written.  Work is split into chunks
// of MMFM_ADAMW_CHUNK4 float4 per segment (grid-stride over chunks; a chunk finds its segment by binary search over
// chunk0); the scalar tail of a segment belongs to its last chunk.  Classes travel by value in the parameter space.
struct AdamwClass {
  float lr, beta1, beta2, eps, wd, inv_bc1, inv_sqrt_bc2;
};
struct AdamwParams {
  const mmfm_adamw_seg* segs;   // device table; nullptr = the single segment `one`
  mmfm_adamw_seg one;
  int n_segs, n_chunks, n_classes;
  long long n;
  AdamwClass cls[MMFM_ADAMW_MAX_CLASSES];
};

__global__ void __launch_bounds__(256) adamw_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                     float* __restrict__ m, float* __restrict__ v,
                                                     const __grid_constant__ AdamwParams P) {
  for (int c = blockIdx.x; c < P.n_chunks; c += gridDim.x) {
    int s = 0;
    if (P.segs != nullptr) {      // last segment with chunk0 <= c
      int lo_s = 0, hi_s = P.n_segs - 1;
      while (lo_s < hi_s) {
        const int mid = (lo_s + hi_s + 1) >> 1;
        if (P.segs[mid].chunk0 <= c) lo_s = mid; else hi_s = mid - 1;
      }
      s = lo_s;
    }
    const mmfm_adamw_seg sg = P.segs != nullptr ? P.segs[s] : P.one;
    if (sg.cls < 0 || sg.cls >= P.n_classes || sg.lo < 0 || sg.hi > P.n || sg.lo >= sg.hi || (sg.lo & 3)) continue;
    const AdamwClass& k = P.cls[sg.cls];
    const float decay = 1.0f - k.lr * k.wd, step = k.lr * k.inv_bc1, c1 = 1.0f - k.beta1, c2 = 1.0f - k.beta2;
    const float beta1 = k.beta1, beta2 = k.beta2, eps = k.eps, inv_sqrt_bc2 = k.inv_sqrt_bc2;
    auto upd = [&](float& pp, float gg, float& mm, float& vv) {
      pp *= decay;
      mm = fmaf(beta1, mm, c1 * gg);
      vv = fmaf(beta2, vv, c2 * gg * gg);
      pp -= step * mm / (sqrtf(vv) * inv_sqrt_bc2 + eps);
    };
    const long long v_lo = sg.lo >> 2, v_hi = sg.hi >> 2;          // float4 range of the segment
    const long long k0 = (long long)(c - sg.chunk0) * MMFM_ADAMW_CHUNK4;
    if (k0 < 0 || (k0 > 0 && v_lo + k0 >= v_hi)) continue;   // a chunk past the segment's end (malformed table)
    const long long i0 = v_lo + k0, i1 = min(v_hi, i0 + MMFM_ADAMW_CHUNK4);
    for (long long i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
      float4 Pv = reinterpret_cast<float4*>(p)[i], M = reinterpret_cast<float4*>(m)[i], V = reinterpret_cast<float4*>(v)[i];
      const float4 G = reinterpret_cast<const float4*>(g)[i];
      upd(Pv.x, G.x, M.x, V.x); upd(Pv.y, G.y, M.y, V.y); upd(Pv.z, G.z, M.z, V.z); upd(Pv.w, G.w, M.w, V.w);
      reinterpret_cast<float4*>(p)[i] = Pv;
      reinterpret_cast<float4*>(m)[i] = M;
      reinterpret_cast<float4*>(v)[i] = V;
    }
    if (i1 == v_hi) {                                               // last chunk: the scalar tail
      const long long e = (v_hi << 2) + threadIdx.x;
      if (e < sg.hi) upd(p[e], g[e], m[e], v[e]);
    }
  }
}

// uint8 spike counts -> fp32 and / or bf16 (SURVEY section 8f rank 2: the loader's counts are small non-negative
// integers stored as sparse ubyte, dataset_utils.py:29; shipping them as bytes cuts the H2D copy 4x and both
// conversions are exact).
// VEC: C, both row pitches and all base pointers are multiples of 4 elements -> one thread converts 4 consecutive bytes
// of a row (uchar4 in, float4 / 2 x bf16x2 out); otherwise one byte per thread.
template <bool VEC>
__global__ void __launch_bounds__(256) u8_expand_kernel(const unsigned char* __restrict__ x, long long R, int C,
                                                         float* __restrict__ y32, long long ld32, bf16* __restrict__ y16,
                                                         long long ld16) {
  const int per_row = VEC ? (C >> 2) : C;
  const long long total = R * per_row;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long r = e / per_row;
    const int c = (int)(e - r * per_row) * (VEC ? 4 : 1);
    if (VEC) {
      const uchar4 v = __ldg(reinterpret_cast<const uchar4*>(x + r * C + c));
      const float4 f = make_float4((float)v.x, (float)v.y, (float)v.z, (float)v.w);
      if (y32) *reinterpret_cast<float4*>(y32 + r * ld32 + c) = f;
      if (y16) *reinterpret_cast<uint2*>(y16 + r * ld16 + c) = make_uint2(pack_bf16x2(f.x, f.y), pack_bf16x2(f.z, f.w));
    } else {
      const float f = (float)x[r * C + c];
      if (y32) y32[r * ld32 + c] = f;
      if (y16) y16[r * ld16 + c] = __float2bfloat16_rn(f);
    }
  }
}

// Evaluation metrics (SURVEY section 8f rank 4): one pass over predictions p and targets y [R, C] -> four float64 sums
// per column, [s_y | s_yy | s_err | s_nll] with s_err = sum (y - p)^2 and s_nll = sum (rate - y * log rate), rate = exp(p)
// for log-rate predictions (zero rates become 1e-9 as in eval_utils.py:1086-1091 otherwise).  Bits per spike per neuron
// and R^2 per channel follow from these sums (metrics.py).  CTA = a slab of rows, thread = column (strided), double
// accumulators, one atomicAdd per column per CTA.
// DET: the CTA's 4 * C sums go to its workspace slot and det_tree_fold adds the slots into out
template <bool DET = false>
__global__ void __launch_bounds__(256) column_stats_kernel(const float* __restrict__ p, const float* __restrict__ y,
                                                            long long R, int C, int log_rate, int rows_per_cta,
                                                            double* __restrict__ out, double* __restrict__ ws,
                                                            unsigned int* tickets) {
  const long long r0 = (long long)blockIdx.x * rows_per_cta, r1 = min(R, r0 + rows_per_cta);
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    double sy = 0.0, syy = 0.0, se = 0.0, sn = 0.0;
    for (long long r = r0; r < r1; ++r) {
      const float yv = y[r * C + c], pv = p[r * C + c];
      float rate, lr;
      if (log_rate) { lr = pv; rate = expf(pv); }
      else { rate = pv == 0.f ? 1e-9f : pv; lr = logf(rate); }
      const float d = yv - pv;
      sy += yv;
      syy += (double)yv * yv;
      se += (double)d * d;
      sn += (double)rate - (double)yv * lr;
    }
    if constexpr (DET) {
      double* slot = ws + (long long)blockIdx.x * 4 * C;
      slot[c] = sy;
      slot[C + c] = syy;
      slot[2ll * C + c] = se;
      slot[3ll * C + c] = sn;
      continue;
    }
    atomicAdd(out + c, sy);
    atomicAdd(out + C + c, syy);
    atomicAdd(out + 2ll * C + c, se);
    atomicAdd(out + 3ll * C + c, sn);
  }
  if constexpr (DET) det_tree_fold(ws, 4ll * C, 4 * C, blockIdx.x, gridDim.x, tickets, [&](int i, double v) { out[i] += v; });
}

// CSR ubyte -> dense uint8 (SURVEY section 8f rank 2; dataset_utils.py:38-43 rebuilds each trial with scipy on the host).
// One warp per (trial, bin) row: the row is zero-filled with 16-byte stores where alignment allows, then its
// non-zeros are scattered.  Column indices outside [0, N) are ignored (scipy would raise; the host checks shapes).
__global__ void __launch_bounds__(256) csr_to_dense_u8_kernel(const unsigned char* __restrict__ data,
                                                               const int* __restrict__ indices,
                                                               const long long* __restrict__ row_ptr, long long n_rows,
                                                               int N, unsigned char* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long r = warp0; r < n_rows; r += nwarps) {
    unsigned char* row = out + r * N;
    // zero fill: head bytes up to 16-byte alignment, 16-byte body, tail
    const int head = (int)((16 - (reinterpret_cast<uintptr_t>(row) & 15)) & 15);
    const int h = head < N ? head : N;
    for (int c = lane; c < h; c += 32) row[c] = 0;
    const int body = (N - h) >> 4;
    for (int c = lane; c < body; c += 32) reinterpret_cast<uint4*>(row + h)[c] = make_uint4(0u, 0u, 0u, 0u);
    for (int c = h + (body << 4) + lane; c < N; c += 32) row[c] = 0;
    __syncwarp();
    const long long k0 = row_ptr[r], k1 = row_ptr[r + 1];
    for (long long k = k0 + lane; k < k1; k += 32) {
      const int c = indices[k];
      if (c >= 0 && c < N) row[c] = data[k];
    }
  }
}

}  // namespace mmfm

// ------------------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------------------
using namespace mmfm;

static DropCfg to_drop(const mmfm_dropout* d) {
  if (d == nullptr || d->thresh == 0u) return DropCfg{nullptr, 0u, 0u, 1.0f};
  return DropCfg{d->seed, d->site, d->thresh, d->scale};
}
static int ew_grid(long long work_items, int threads) {
  long long g = (work_items + threads - 1) / threads;
  const long long cap = (long long)device_sm_count() * 8;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

extern "C" int mmfm_mask_prep(const mmfm_mask_args* a, unsigned char* zero_flags, unsigned char* key_valid,
                              unsigned char* tok_mask, long long* n_examples, float* inv_n, void* stream) {
  MMFM_REQUIRE(a && zero_flags && key_valid && tok_mask && n_examples && inv_n, "mmfm_mask_prep: null pointer");
  MMFM_REQUIRE(a->n_mod >= 1 && a->n_mod <= MMFM_MAX_MOD && a->B > 0 && a->T > 0, "mmfm_mask_prep: bad shape");
  for (int m = 0; m < a->n_mod; ++m) {
    MMFM_REQUIRE(a->attn[m] != nullptr, "mmfm_mask_prep: modality %d has no attention mask", m);
    MMFM_REQUIRE(a->channels[m] > 0, "mmfm_mask_prep: modality %d has no channels", m);
  }
  int slices = (a->B * a->T + 255) / 256;
  if (slices > 64) slices = 64;
  mask_prep_kernel<<<dim3(slices, a->n_mod), 256, 0, (cudaStream_t)stream>>>(*a, zero_flags, key_valid, tok_mask, n_examples, inv_n);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_embed_assemble(const float* mod_emb_row, const float* pos_embed, const long long* ts, float* emb,
                                   int B, int T, int S, int off, int H, void* stream) {
  MMFM_REQUIRE(mod_emb_row && emb && (pos_embed == nullptr || ts), "mmfm_embed_assemble: null pointer");
  MMFM_REQUIRE(B > 0 && T > 0 && H % 4 == 0 && off >= 0 && off + T <= S, "mmfm_embed_assemble: bad shape");
  embed_assemble_kernel<<<ew_grid((long long)B * T * (H / 4), 256), 256, 0, (cudaStream_t)stream>>>(
      mod_emb_row, pos_embed, ts, emb, B, T, S, off, H);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

static int embed_bwd_chunks(int B, int T, int* bchunk) {
  int chunks = (4 * device_sm_count() + T - 1) / T;
  if (chunks > B) chunks = B;
  if (chunks < 1) chunks = 1;
  *bchunk = (B + chunks - 1) / chunks;
  return (B + *bchunk - 1) / *bchunk;
}

extern "C" int mmfm_embed_assemble_bwd(const float* g, const float* g2, const long long* ts, float* dpos, float* dmod,
                                       int B, int T, int S, int off, int H, void* stream) {
  MMFM_REQUIRE(g && dmod && (dpos == nullptr || ts), "mmfm_embed_assemble_bwd: null pointer");
  MMFM_REQUIRE(B > 0 && T > 0 && H % 4 == 0 && off >= 0 && off + T <= S, "mmfm_embed_assemble_bwd: bad shape");
  int bchunk = 0;
  const int chunks = embed_bwd_chunks(B, T, &bchunk);
  MMFM_REQUIRE(H % 4 == 0 && H / 4 * kAsmLanes <= 1024, "mmfm_embed_assemble_bwd: H=%d not supported (H %% 4, H <= 1024)", H);
  const int threads = H / 4 * kAsmLanes;
  embed_assemble_bwd_kernel<<<dim3(T, chunks), threads, (size_t)threads * sizeof(float4), (cudaStream_t)stream>>>(
      g, g2, ts, dpos, dmod, B, T, S, off, H, bchunk, nullptr, nullptr);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_embed_grad_prep(const float* dx, void* dtok, const unsigned char* row_zero, const mmfm_dropout* drop,
                                    int B, int T, int S, int off, int H, void* stream) {
  MMFM_REQUIRE(dx && dtok, "mmfm_embed_grad_prep: null pointer");
  MMFM_REQUIRE(B > 0 && T > 0 && H % 4 == 0 && off >= 0 && off + T <= S, "mmfm_embed_grad_prep: bad shape");
  embed_grad_prep_kernel<<<ew_grid((long long)B * T * (H / 4), 256), 256, 0, (cudaStream_t)stream>>>(
      dx, (bf16*)dtok, row_zero, to_drop(drop), B, T, S, off, H);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_smallc_embed_fwd(const float* in, const float* W1, const float* b1, const float* W2, const float* b2,
                                     const float* emb, float* x, float* hid, const unsigned char* row_zero,
                                     const mmfm_dropout* drop, float act_scale, int act, int B, int T, int S, int off,
                                     int C, int H, void* stream) {
  MMFM_REQUIRE(in && W1 && W2 && emb && x && hid, "mmfm_smallc_embed_fwd: null pointer");
  MMFM_REQUIRE(C >= 1 && C <= kMaxC, "mmfm_smallc_embed_fwd: C=%d outside [1,%d]", C, kMaxC);
  MMFM_REQUIRE(act == MMFM_ACT_NONE || act == MMFM_ACT_SOFTSIGN, "mmfm_smallc_embed_fwd: bad act %d", act);
  MMFM_REQUIRE(B > 0 && T > 0 && H > 0 && off >= 0 && off + T <= S, "mmfm_smallc_embed_fwd: bad shape");
  const int gpr = H / 16;
  if (C <= 2 && H % 16 == 0 && gpr <= 256 && 256 % gpr == 0 && (((uintptr_t)emb | (uintptr_t)x) & 15) == 0) {
    // thread = one 16-column group: grid sized to a whole number of resident waves, a multiple of the groups per row
    const long long slots = (long long)B * T * gpr;
    int grid = 4 * device_sm_count();
    if ((long long)grid * 256 > slots) grid = (int)((slots + 255) / 256);
    if (C == 1) smallc_embed_fwd16_kernel<1><<<grid, 256, 0, (cudaStream_t)stream>>>(in, W1, b1, W2, b2, emb, x, hid, row_zero, to_drop(drop), act_scale, act, B, T, S, off, H);
    else smallc_embed_fwd16_kernel<2><<<grid, 256, 0, (cudaStream_t)stream>>>(in, W1, b1, W2, b2, emb, x, hid, row_zero, to_drop(drop), act_scale, act, B, T, S, off, H);
    MMFM_CHECK_CUDA(cudaGetLastError());
    return 0;
  }
  smallc_embed_fwd_kernel<<<B * T, 256, 0, (cudaStream_t)stream>>>(in, W1, b1, W2, b2, emb, x, hid, row_zero,
                                                                   to_drop(drop), act_scale, act, B, T, S, off, C, H);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_smallc_embed_bwd(const float* in, const float* hid, const float* W2, const float* dx,
                                     const unsigned char* row_zero, const mmfm_dropout* drop, float act_scale, int act,
                                     float* dW1, float* db1, float* dW2, float* db2, int B, int T, int S, int off, int C,
                                     int H, void* stream) {
  MMFM_REQUIRE(in && hid && W2 && dx && dW1 && db1 && dW2 && db2, "mmfm_smallc_embed_bwd: null pointer");
  MMFM_REQUIRE(C >= 1 && C <= kMaxC, "mmfm_smallc_embed_bwd: C=%d outside [1,%d]", C, kMaxC);
  MMFM_REQUIRE(H % 32 == 0 && H <= 1024, "mmfm_smallc_embed_bwd: H=%d must be a multiple of 32 and <= 1024", H);
  MMFM_REQUIRE(B > 0 && T > 0 && off >= 0 && off + T <= S, "mmfm_smallc_embed_bwd: bad shape");
  const int gpr = H / 16;
  if (C <= 2 && H % 16 == 0 && gpr <= 32 && 32 % gpr == 0 && ((uintptr_t)dx & 15) == 0) {
    const long long slots = (long long)B * T * gpr;
    int grid = device_sm_count();        // ~230 registers per thread: one CTA per SM, one wave
    if ((long long)grid * 256 > slots) grid = (int)((slots + 255) / 256);
    if (C == 1) smallc_embed_bwd16_kernel<1><<<grid, 256, 0, (cudaStream_t)stream>>>(in, hid, W2, dx, row_zero, to_drop(drop), act_scale, act, dW1, db1, dW2, db2, B, T, S, off, H, nullptr, nullptr);
    else smallc_embed_bwd16_kernel<2><<<grid, 256, 0, (cudaStream_t)stream>>>(in, hid, W2, dx, row_zero, to_drop(drop), act_scale, act, dW1, db1, dW2, db2, B, T, S, off, H, nullptr, nullptr);
    MMFM_CHECK_CUDA(cudaGetLastError());
    return 0;
  }
  const long long R = (long long)B * T;
  int ctas = 2 * device_sm_count();
  int rows_per_cta = (int)((R + ctas - 1) / ctas);
  if (rows_per_cta < 16) rows_per_cta = 16;
  ctas = (int)((R + rows_per_cta - 1) / rows_per_cta);
  smallc_embed_bwd_kernel<<<ctas, H, 0, (cudaStream_t)stream>>>(in, hid, W2, dx, row_zero, to_drop(drop), act_scale, act,
                                                                dW1, db1, dW2, db2, B, T, S, off, C, H, rows_per_cta,
                                                                nullptr, nullptr);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_smallc_head_fwd(const void* y, const float* W, const float* b, float* preds, int R, int H, int C,
                                    void* stream) {
  MMFM_REQUIRE(y && W && preds, "mmfm_smallc_head_fwd: null pointer");
  MMFM_REQUIRE(C >= 1 && C <= kMaxC && R > 0 && H % 8 == 0, "mmfm_smallc_head_fwd: bad shape R=%d H=%d C=%d", R, H, C);
  smallc_head_fwd_kernel<<<ew_grid(R, 8), 256, 0, (cudaStream_t)stream>>>((const bf16*)y, W, b, preds, R, H, C);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_smallc_head_bwd(const void* y, const float* W, const void* dpreds, long long lddp, void* dy,
                                    float* dW, float* db, int R, int H, int C, void* stream) {
  MMFM_REQUIRE(y && W && dpreds && dy && dW && db, "mmfm_smallc_head_bwd: null pointer");
  MMFM_REQUIRE(C >= 1 && C <= kMaxC && R > 0 && H % 8 == 0, "mmfm_smallc_head_bwd: bad shape R=%d H=%d C=%d", R, H, C);
  int gx = (R + 63) / 64;
  const int cap = 2 * device_sm_count();
  if (gx > cap) gx = cap;
  smallc_head_bwd_kernel<<<dim3(gx, (H + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      (const bf16*)y, W, (const bf16*)dpreds, lddp, (bf16*)dy, dW, db, R, H, C, nullptr, nullptr);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_loss_fwd_bwd(const float* preds, const float* targets, const unsigned char* tok_mask, int S, int off,
                                 const float* inv_n, int kind, int B, int T, int C, float* partials, int n_partials,
                                 void* dpreds, long long lddp, void* stream) {
  MMFM_REQUIRE(preds && targets && tok_mask && inv_n && partials && dpreds, "mmfm_loss_fwd_bwd: null pointer");
  MMFM_REQUIRE(kind == MMFM_LOSS_POISSON || kind == MMFM_LOSS_MSE || kind == MMFM_LOSS_CE, "mmfm_loss_fwd_bwd: bad loss kind %d", kind);
  MMFM_REQUIRE(B > 0 && T > 0 && C > 0 && n_partials > 0 && lddp >= C, "mmfm_loss_fwd_bwd: bad shape");
  const bool vec = (C % 4 == 0) && (lddp % 4 == 0);
  cudaStream_t st = (cudaStream_t)stream;
  bf16* dp = (bf16*)dpreds;
#define LOSS(K, V) loss_kernel<K, V><<<n_partials, 256, 0, st>>>(preds, targets, tok_mask, S, off, inv_n, B, T, C, partials, dp, lddp)
  if (kind == MMFM_LOSS_CE) {
    MMFM_REQUIRE(C <= kMaxClasses, "mmfm_loss_fwd_bwd: cross-entropy supports up to %d classes (got %d)", kMaxClasses, C);
    loss_ce_kernel<<<n_partials, 256, 0, st>>>(preds, targets, tok_mask, S, off, inv_n, B, T, C, partials, dp, lddp);
  } else if (kind == MMFM_LOSS_POISSON) { if (vec) LOSS(MMFM_LOSS_POISSON, true); else LOSS(MMFM_LOSS_POISSON, false); }
  else { if (vec) LOSS(MMFM_LOSS_MSE, true); else LOSS(MMFM_LOSS_MSE, false); }
#undef LOSS
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_loss_finalize(const float* partials, int n_partials, int n_mod, const float* inv_n, float* mod_loss,
                                  float* loss, void* stream) {
  MMFM_REQUIRE(partials && inv_n && mod_loss && loss && n_partials > 0 && n_mod > 0, "mmfm_loss_finalize: bad arguments");
  loss_finalize_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(partials, n_partials, n_mod, inv_n, mod_loss, loss);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_loss_grad(const float* preds, const float* targets, const unsigned char* tok_mask, int S, int off,
                              const float* inv_n, const float* g_loss, const float* g_mod, const float* g_preds,
                              long long gp_sb, long long gp_st, long long gp_sc, int kind, int B, int T, int C,
                              void* dpreds, long long lddp, void* stream) {
  MMFM_REQUIRE(preds && targets && tok_mask && inv_n && dpreds, "mmfm_loss_grad: null pointer");
  MMFM_REQUIRE(kind == MMFM_LOSS_POISSON || kind == MMFM_LOSS_MSE || kind == MMFM_LOSS_CE, "mmfm_loss_grad: bad loss kind %d", kind);
  MMFM_REQUIRE(B > 0 && T > 0 && C > 0 && lddp >= C && off >= 0 && off + T <= S, "mmfm_loss_grad: bad shape");
  MMFM_REQUIRE(gp_sb >= 0 && gp_st >= 0 && gp_sc >= 0, "mmfm_loss_grad: negative g_preds stride");
  cudaStream_t st = (cudaStream_t)stream;
  bf16* dp = (bf16*)dpreds;
  if (kind == MMFM_LOSS_CE) {
    MMFM_REQUIRE(C <= kMaxClasses, "mmfm_loss_grad: cross-entropy supports up to %d classes (got %d)", kMaxClasses, C);
    loss_grad_ce_kernel<<<ew_grid((long long)B * T, 256), 256, 0, st>>>(preds, targets, tok_mask, S, off, inv_n, g_loss,
                                                                         g_mod, g_preds, gp_sb, gp_st, gp_sc, B, T, C, dp, lddp);
  } else {
    const int grid = ew_grid((long long)B * T * C, 256);
#define LGRAD(K) loss_grad_kernel<K><<<grid, 256, 0, st>>>(preds, targets, tok_mask, S, off, inv_n, g_loss, g_mod, g_preds, \
                                                          gp_sb, gp_st, gp_sc, B, T, C, dp, lddp)
    if (kind == MMFM_LOSS_POISSON) LGRAD(MMFM_LOSS_POISSON); else LGRAD(MMFM_LOSS_MSE);
#undef LGRAD
  }
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_smallc_embed_dx(const float* hid, const float* W1, const float* W2, const float* dx,
                                    const unsigned char* row_zero, const mmfm_dropout* drop, float act_scale, int act,
                                    float* dX, long long lddx, int accumulate, int B, int T, int S, int off, int C, int H,
                                    void* stream) {
  MMFM_REQUIRE(hid && W1 && W2 && dx && dX, "mmfm_smallc_embed_dx: null pointer");
  MMFM_REQUIRE(C >= 1 && C <= kMaxC, "mmfm_smallc_embed_dx: C=%d outside [1,%d]", C, kMaxC);
  MMFM_REQUIRE(act == MMFM_ACT_NONE || act == MMFM_ACT_SOFTSIGN, "mmfm_smallc_embed_dx: bad act %d", act);
  MMFM_REQUIRE(B > 0 && T > 0 && H > 0 && off >= 0 && off + T <= S && lddx >= C, "mmfm_smallc_embed_dx: bad shape");
  MMFM_REQUIRE(drop == nullptr || drop->thresh == 0u || drop->seed, "mmfm_smallc_embed_dx: dropout without seed pointer");
  smallc_embed_dx_kernel<<<ew_grid((long long)B * T * 32, 256), 256, 0, (cudaStream_t)stream>>>(
      hid, W1, W2, dx, row_zero, to_drop(drop), act_scale, act, dX, lddx, accumulate, B, T, S, off, C, H);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_cast_bf16_multi(const mmfm_cast_item* items_dev, int n_items, int total_tiles, void* stream) {
  MMFM_REQUIRE(items_dev && n_items > 0 && total_tiles > 0, "mmfm_cast_bf16_multi: bad arguments");
  cast_multi_kernel<<<total_tiles, 256, 0, (cudaStream_t)stream>>>(items_dev, n_items);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_scale_inplace(float* x, long long n, const float* scale_dev, void* stream) {
  MMFM_REQUIRE(x && scale_dev && n > 0, "mmfm_scale_inplace: bad arguments");
  MMFM_REQUIRE(((uintptr_t)x & 15) == 0, "mmfm_scale_inplace: buffer must be 16-byte aligned");
  scale_inplace_kernel<<<ew_grid(n / 4 + 1, 256), 256, 0, (cudaStream_t)stream>>>(x, n, scale_dev);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_session_grad_combine(float* grad, const float* gathered, int world, long long slab_stride,
                                         const int* ids_dev, const long long* ranges_dev, int n_sessions,
                                         float inv_world, void* stream) {
  MMFM_REQUIRE(grad && gathered && ids_dev && ranges_dev, "mmfm_session_grad_combine: null pointer");
  MMFM_REQUIRE(world >= 1 && world <= 65535, "mmfm_session_grad_combine: world=%d outside [1, 65535]", world);
  MMFM_REQUIRE(slab_stride >= 1 && n_sessions >= 1, "mmfm_session_grad_combine: bad slab stride or session count");
  MMFM_REQUIRE(isfinite(inv_world), "mmfm_session_grad_combine: inv_world must be finite");
  const dim3 grid(ew_grid((slab_stride + 3) / 4, 256), world);
  session_grad_combine_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(grad, gathered, world, slab_stride, ids_dev,
                                                                       ranges_dev, n_sessions, inv_world);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

static int adamw_class(const mmfm_adamw_class& c, AdamwClass* out) {
  MMFM_REQUIRE(c.step >= 1, "mmfm_adamw: step must be >= 1");
  const double bc1 = 1.0 - pow((double)c.beta1, (double)c.step), bc2 = 1.0 - pow((double)c.beta2, (double)c.step);
  *out = AdamwClass{c.lr, c.beta1, c.beta2, c.eps, c.weight_decay, (float)(1.0 / bc1), (float)(1.0 / sqrt(bc2))};
  return 0;
}

static int adamw_launch(float* p, const float* g, float* exp_avg, float* exp_avg_sq, AdamwParams& P, void* stream) {
  MMFM_REQUIRE(p && g && exp_avg && exp_avg_sq && P.n > 0, "mmfm_adamw: bad arguments");
  MMFM_REQUIRE((((uintptr_t)p | (uintptr_t)g | (uintptr_t)exp_avg | (uintptr_t)exp_avg_sq) & 15) == 0,
               "mmfm_adamw: buffers must be 16-byte aligned");
  adamw_kernel<<<ew_grid((long long)P.n_chunks * 256, 256), 256, 0, (cudaStream_t)stream>>>(p, g, exp_avg, exp_avg_sq, P);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_adamw_step(float* p, const float* g, float* exp_avg, float* exp_avg_sq, long long n, float lr,
                               float beta1, float beta2, float eps, float weight_decay, long long step, void* stream) {
  MMFM_REQUIRE(p && g && exp_avg && exp_avg_sq && n > 0 && step >= 1, "mmfm_adamw_step: bad arguments");
  AdamwParams P{};
  const long long chunks = ((n >> 2) + MMFM_ADAMW_CHUNK4 - 1) / MMFM_ADAMW_CHUNK4;
  MMFM_REQUIRE(chunks < (1LL << 31), "mmfm_adamw_step: n too large");
  P.segs = nullptr;
  P.one = mmfm_adamw_seg{0, n, 0, 0};
  P.n_segs = 1;
  P.n_chunks = chunks > 0 ? (int)chunks : 1;
  P.n_classes = 1;
  P.n = n;
  if (adamw_class(mmfm_adamw_class{lr, beta1, beta2, eps, weight_decay, 0, step}, &P.cls[0]) != 0) return -1;
  return adamw_launch(p, g, exp_avg, exp_avg_sq, P, stream);
}

extern "C" int mmfm_adamw_multi(float* p, const float* g, float* exp_avg, float* exp_avg_sq, long long n,
                                const mmfm_adamw_seg* segs_dev, int n_segs, int n_chunks,
                                const mmfm_adamw_class* classes, int n_classes, void* stream) {
  MMFM_REQUIRE(segs_dev && classes, "mmfm_adamw_multi: null pointer");
  MMFM_REQUIRE(n_segs >= 1 && n_chunks >= n_segs, "mmfm_adamw_multi: bad segment count");
  MMFM_REQUIRE(n_classes >= 1 && n_classes <= MMFM_ADAMW_MAX_CLASSES,
               "mmfm_adamw_multi: n_classes must be in [1, MMFM_ADAMW_MAX_CLASSES]");
  AdamwParams P{};
  P.segs = segs_dev;
  P.n_segs = n_segs;
  P.n_chunks = n_chunks;
  P.n_classes = n_classes;
  P.n = n;
  for (int i = 0; i < n_classes; ++i)
    if (adamw_class(classes[i], &P.cls[i]) != 0) return -1;
  return adamw_launch(p, g, exp_avg, exp_avg_sq, P, stream);
}

extern "C" int mmfm_u8_expand(const unsigned char* x, long long R, int C, float* y32, long long ld32, void* y16,
                              long long ld16, void* stream) {
  MMFM_REQUIRE(x && (y32 || y16) && R > 0 && C > 0, "mmfm_u8_expand: bad arguments");
  MMFM_REQUIRE((!y32 || ld32 >= C) && (!y16 || ld16 >= C), "mmfm_u8_expand: row pitch smaller than the row");
  const bool vec = C % 4 == 0 && ld32 % 4 == 0 && ld16 % 4 == 0 && ((uintptr_t)x & 3) == 0 && ((uintptr_t)y32 & 15) == 0 &&
                   ((uintptr_t)y16 & 7) == 0;
  if (vec) u8_expand_kernel<true><<<ew_grid(R * (C / 4), 256), 256, 0, (cudaStream_t)stream>>>(x, R, C, y32, ld32, (bf16*)y16, ld16);
  else u8_expand_kernel<false><<<ew_grid(R * (long long)C, 256), 256, 0, (cudaStream_t)stream>>>(x, R, C, y32, ld32, (bf16*)y16, ld16);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_column_stats(const float* pred, const float* y, long long R, int C, int log_rate, double* out,
                                 void* stream) {
  MMFM_REQUIRE(pred && y && out && R > 0 && C > 0, "mmfm_column_stats: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  MMFM_CHECK_CUDA(cudaMemsetAsync(out, 0, sizeof(double) * 4 * (size_t)C, st));
  int ctas = 4 * device_sm_count();
  int rows_per_cta = (int)((R + ctas - 1) / ctas);
  if (rows_per_cta < 8) rows_per_cta = 8;
  ctas = (int)((R + rows_per_cta - 1) / rows_per_cta);
  column_stats_kernel<<<ctas, 256, 0, st>>>(pred, y, R, C, log_rate, rows_per_cta, out, nullptr, nullptr);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_csr_to_dense_u8(const unsigned char* data, const int* indices, const long long* row_ptr,
                                    long long n_rows, int N, unsigned char* out, void* stream) {
  MMFM_REQUIRE(row_ptr && out && n_rows > 0 && N > 0, "mmfm_csr_to_dense_u8: bad arguments");
  csr_to_dense_u8_kernel<<<ew_grid(n_rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(data, indices, row_ptr, n_rows, N, out);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------------------
// deterministic twins (column sums folded by det_tree_fold; one workspace slot per CTA, same grids as above)
// ------------------------------------------------------------------------------------------------------------
static bool smallc_fast16(int C, int H) { return C <= 2 && H % 16 == 0 && H / 16 <= 32 && 32 % (H / 16) == 0; }
static int smallc_fast16_grid(long long R, int H) {
  const long long slots = R * (H / 16);
  int grid = device_sm_count();
  if ((long long)grid * 256 > slots) grid = (int)((slots + 255) / 256);
  return grid;
}
static int smallc_generic_ctas(long long R, int* rows_per_cta) {
  int ctas = 2 * device_sm_count();
  *rows_per_cta = (int)((R + ctas - 1) / ctas);
  if (*rows_per_cta < 16) *rows_per_cta = 16;
  return (int)((R + *rows_per_cta - 1) / *rows_per_cta);
}
static int head_bwd_gx(int R) {
  const int gx = (R + 63) / 64, cap = 2 * device_sm_count();
  return gx > cap ? cap : gx;
}
static int column_stats_ctas(long long R, int* rows_per_cta) {
  int ctas = 4 * device_sm_count();
  *rows_per_cta = (int)((R + ctas - 1) / ctas);
  if (*rows_per_cta < 8) *rows_per_cta = 8;
  return (int)((R + *rows_per_cta - 1) / *rows_per_cta);
}

namespace mmfm {
bool det_need_glue(int kind, long long d0, long long d1, long long d2, DetNeed* need) {
  if (kind == MMFM_DET_EMBED_ASM_BWD) {   // (B, T, H)
    int bchunk = 0;
    const long long ctas = (long long)embed_bwd_chunks((int)d0, (int)d1, &bchunk) * d1;
    *need = DetNeed{ctas * d2 * 4, (int)ctas};
  } else if (kind == MMFM_DET_SMALLC_EMBED_BWD) {   // (B*T, C, H): the larger of the two kernels' needs
    const int C = (int)d1, H = (int)d2;
    int rows = 0;
    long long ctas = smallc_generic_ctas(d0, &rows);
    if (smallc_fast16(C, H)) {
      const long long f = smallc_fast16_grid(d0, H);
      if (f > ctas) ctas = f;
    }
    *need = DetNeed{ctas * (H * (1 + 2 * C) + 2 * C * (1 + C)) * 4, (int)ctas};
  } else if (kind == MMFM_DET_SMALLC_HEAD_BWD) {   // (R, H, C)
    const long long ctas = (long long)head_bwd_gx((int)d0) * ((d1 + 255) / 256);
    *need = DetNeed{ctas * kHeadSlot * 4, (int)ctas};
  } else if (kind == MMFM_DET_COLUMN_STATS) {   // (R, C)
    int rows = 0;
    const long long ctas = column_stats_ctas(d0, &rows);
    *need = DetNeed{ctas * 4 * d1 * 8, (int)ctas};
  } else {
    return false;
  }
  return true;
}
}  // namespace mmfm

#define DET_WS_CHECK(kind, d0, d1, d2, who)                                                       \
  do {                                                                                          \
    MMFM_REQUIRE(ws != nullptr, "%s: null workspace", who);                                     \
    DetNeed need{0, 0};                                                                         \
    det_need_glue(kind, d0, d1, d2, &need);                                                     \
    if (int rc = det_ws_check(ws->buf, ws->bytes, ws->tickets, ws->n_tickets, need, who)) return rc; \
  } while (0)

extern "C" int mmfm_embed_assemble_bwd_det(const float* g, const float* g2, const long long* ts, float* dpos, float* dmod,
                                           int B, int T, int S, int off, int H, int n_pos, const mmfm_det_ws* ws,
                                           void* stream) {
  MMFM_REQUIRE(g && dmod && (dpos == nullptr || (ts && n_pos > 0)), "mmfm_embed_assemble_bwd_det: null pointer");
  MMFM_REQUIRE(B > 0 && T > 0 && H % 4 == 0 && H <= 1024 && off >= 0 && off + T <= S,
               "mmfm_embed_assemble_bwd_det: bad shape (H %% 4 == 0, H <= 1024)");
  MMFM_REQUIRE(((uintptr_t)g | (uintptr_t)dmod | (uintptr_t)g2 | (uintptr_t)dpos) % 16 == 0,
               "mmfm_embed_assemble_bwd_det: buffers must be 16-byte aligned");
  DET_WS_CHECK(MMFM_DET_EMBED_ASM_BWD, B, T, H, "mmfm_embed_assemble_bwd_det");
  cudaStream_t st = (cudaStream_t)stream;
  int bchunk = 0;
  const int chunks = embed_bwd_chunks(B, T, &bchunk);
  const int threads = H / 4 * kAsmLanes;
  embed_assemble_bwd_kernel<true><<<dim3(T, chunks), threads, (size_t)threads * sizeof(float4), st>>>(
      g, g2, ts, nullptr, dmod, B, T, S, off, H, bchunk, (float4*)ws->buf, ws->tickets);
  MMFM_CHECK_CUDA(cudaGetLastError());
  if (dpos) {
    embed_pos_bwd_det_kernel<<<n_pos, 256, 0, st>>>(g, g2, ts, dpos, B, T, S, off, H);
    MMFM_CHECK_CUDA(cudaGetLastError());
  }
  return 0;
}

extern "C" int mmfm_smallc_embed_bwd_det(const float* in, const float* hid, const float* W2, const float* dx,
                                         const unsigned char* row_zero, const mmfm_dropout* drop, float act_scale, int act,
                                         float* dW1, float* db1, float* dW2, float* db2, int B, int T, int S, int off,
                                         int C, int H, const mmfm_det_ws* ws, void* stream) {
  MMFM_REQUIRE(in && hid && W2 && dx && dW1 && db1 && dW2 && db2, "mmfm_smallc_embed_bwd_det: null pointer");
  MMFM_REQUIRE(C >= 1 && C <= kMaxC, "mmfm_smallc_embed_bwd_det: C=%d outside [1,%d]", C, kMaxC);
  MMFM_REQUIRE(H % 32 == 0 && H <= 1024, "mmfm_smallc_embed_bwd_det: H=%d must be a multiple of 32 and <= 1024", H);
  MMFM_REQUIRE(B > 0 && T > 0 && off >= 0 && off + T <= S, "mmfm_smallc_embed_bwd_det: bad shape");
  const long long R = (long long)B * T;
  DET_WS_CHECK(MMFM_DET_SMALLC_EMBED_BWD, R, C, H, "mmfm_smallc_embed_bwd_det");
  cudaStream_t st = (cudaStream_t)stream;
  float* buf = (float*)ws->buf;
  if (smallc_fast16(C, H) && ((uintptr_t)dx & 15) == 0) {
    const int grid = smallc_fast16_grid(R, H);
    if (C == 1) smallc_embed_bwd16_kernel<1, true><<<grid, 256, 0, st>>>(in, hid, W2, dx, row_zero, to_drop(drop), act_scale, act, dW1, db1, dW2, db2, B, T, S, off, H, buf, ws->tickets);
    else smallc_embed_bwd16_kernel<2, true><<<grid, 256, 0, st>>>(in, hid, W2, dx, row_zero, to_drop(drop), act_scale, act, dW1, db1, dW2, db2, B, T, S, off, H, buf, ws->tickets);
    MMFM_CHECK_CUDA(cudaGetLastError());
    return 0;
  }
  int rows_per_cta = 0;
  const int ctas = smallc_generic_ctas(R, &rows_per_cta);
  smallc_embed_bwd_kernel<true><<<ctas, H, 0, st>>>(in, hid, W2, dx, row_zero, to_drop(drop), act_scale, act, dW1, db1,
                                                    dW2, db2, B, T, S, off, C, H, rows_per_cta, buf, ws->tickets);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_smallc_head_bwd_det(const void* y, const float* W, const void* dpreds, long long lddp, void* dy,
                                        float* dW, float* db, int R, int H, int C, const mmfm_det_ws* ws, void* stream) {
  MMFM_REQUIRE(y && W && dpreds && dy && dW && db, "mmfm_smallc_head_bwd_det: null pointer");
  MMFM_REQUIRE(C >= 1 && C <= kMaxC && R > 0 && H % 8 == 0, "mmfm_smallc_head_bwd_det: bad shape R=%d H=%d C=%d", R, H, C);
  DET_WS_CHECK(MMFM_DET_SMALLC_HEAD_BWD, R, H, C, "mmfm_smallc_head_bwd_det");
  smallc_head_bwd_kernel<true><<<dim3(head_bwd_gx(R), (H + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      (const bf16*)y, W, (const bf16*)dpreds, lddp, (bf16*)dy, dW, db, R, H, C, (float*)ws->buf, ws->tickets);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mmfm_column_stats_det(const float* pred, const float* y, long long R, int C, int log_rate, double* out,
                                     const mmfm_det_ws* ws, void* stream) {
  MMFM_REQUIRE(pred && y && out && R > 0 && C > 0, "mmfm_column_stats_det: bad arguments");
  DET_WS_CHECK(MMFM_DET_COLUMN_STATS, R, C, 0, "mmfm_column_stats_det");
  cudaStream_t st = (cudaStream_t)stream;
  MMFM_CHECK_CUDA(cudaMemsetAsync(out, 0, sizeof(double) * 4 * (size_t)C, st));
  int rows_per_cta = 0;
  const int ctas = column_stats_ctas(R, &rows_per_cta);
  column_stats_kernel<true><<<ctas, 256, 0, st>>>(pred, y, R, C, log_rate, rows_per_cta, out, (double*)ws->buf,
                                                  ws->tickets);
  MMFM_CHECK_CUDA(cudaGetLastError());
  return 0;
}
