// Shared by the attention translation units: kernel parameter block, constants, the probability-dropout stream.
#pragma once
#include "common.cuh"
#include "host_util.h"
#include "../../include/mmfm_b200.h"

namespace mmfm {

constexpr int kAttnThreads = 128;
constexpr int kTile = 64;
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

MMFM_DEVINL float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

struct AttnParams {
  const bf16* q; long long ldq;
  const bf16* k; long long ldk;
  const bf16* v; long long ldv;
  bf16* o; long long ldo;
  float* lse;
  const unsigned char* key_valid;
  const short* mod_q;
  const short* mod_k;
  int B, nh, Sq, Sk;
  int mask_mode;
  float scale;
  DropCfg drop_p, drop_o;
  unsigned short* p_keep;
  // backward
  bf16* d_o; long long lddo;
  float* delta;
  bf16* dq; long long lddq;
  bf16* dk; long long lddk;
  bf16* dv; long long lddv;
};

// 16 random bytes of the probability-dropout field: row = (b*nh+h)*Sq + i, 64-column block blk, quad lane ql
MMFM_DEVINL uint4 pdrop_bytes(unsigned long long seed, uint32_t site, unsigned long long row, uint32_t nblk,
                              uint32_t blk, uint32_t ql) {
  const unsigned long long g = (row * nblk + blk) * 4ull + ql;
  return philox4x32((uint32_t)g, (uint32_t)(g >> 32), site, 1u, (uint32_t)seed, (uint32_t)(seed >> 32));
}

constexpr uint32_t kSlabBytes = 128 * 128;   // 128 query rows x 64 keys (bf16)

MMFM_DEVINL void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}



// ---- helpers of the fused backward: keep bits -> byte-msb words -> 32-bit pair masks (no per-element bit tests) ----
MMFM_DEVINL uint32_t prmt_b(uint32_t a, uint32_t sel) {   // prmt, sign-replicating selector mode (nibble bit 3)
  uint32_t d;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(0u), "r"(sel));
  return d;
}
// 8 keep bits (n-tile n = 0..3 of this 32-column chunk, e = 0/1 at bit 2n+e) -> two words whose byte msbs carry them:
// word 0 <- bits 0..3 (n = 0, 1), word 1 <- bits 4..7 (n = 2, 3).  x * 0x10204080 moves bit k to bit 8k+7 (k < 4)
// and the partial products never collide, so the msbs are exact.
MMFM_DEVINL void keep_msb_words(uint32_t bits8, uint32_t (&w)[2]) {
  w[0] = (bits8 & 0xFu) * 0x10204080u;
  w[1] = ((bits8 >> 4) & 0xFu) * 0x10204080u;
}

// the four quad-lane calls of one 64-key block at once (g = (row*nblk + blk)*4 + ql: the low two counter bits are ql and
// g is a multiple of 4, so the +ql never carries into the high word)
MMFM_DEVINL void pdrop_bytes_x4(unsigned long long seed, uint32_t site, unsigned long long row, uint32_t nblk,
                                uint32_t blk, uint4 (&w)[4]) {
  const unsigned long long g = (row * nblk + blk) * 4ull;
  philox4x32_x4((uint32_t)g, (uint32_t)(g >> 32), site, 1u, (uint32_t)seed, (uint32_t)(seed >> 32), w);
}

// attention_pipe.cu: persistent warp-specialised tcgen05 forward (any Sk; no modality-separation mask)
int launch_attn_fwd_pipe(const mmfm_attn_args* a, const AttnParams& p, cudaStream_t st);
// attention_bwd_stream.cu: tcgen05 backward pair for long sequences (runs after the prep kernel)
int launch_attn_bwd_stream(const mmfm_attn_args* a, const AttnParams& p, cudaStream_t st);
// attention_bwd_ws.cu: persistent warp-specialised fused backward (d_head 32, Sq, Sk <= 256, Sq % 4 == 0)
int launch_attn_bwd_ws(const mmfm_attn_args* a, const AttnParams& p, cudaStream_t st);

}  // namespace mmfm
