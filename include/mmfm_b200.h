/* mmfm_b200.h -- C ABI of libmmfm_b200.so: the sm_100a kernels behind the forward/backward pass of the
 * masked multi-modal encoder/decoder.
 *
 * The reference (yzhang511/multi_modal_foundation_model) has no FFI: its boundary for this path is the
 * torch.nn.Module call `MultiModal.forward(mod_dict)` + `loss.backward()` (src/multi_modal/mm.py:242-308,
 * src/trainer/base.py:103,194-195), and every arithmetic step under it is a PyTorch library call.  Each entry
 * point below replaces one group of those library call sites (cited per function, paths relative to the
 * reference root) and is what the Python host layer (multi_modal_foundation_model_b200/ops.py, ctypes) binds.
 *
 * Conventions
 *  - plain pointers and sizes only; every pointer is a DEVICE pointer unless stated; all buffers are owned by
 *    the caller; the library allocates nothing on the device, never synchronises, and launches only on `stream`
 *    (a cudaStream_t passed as void*).
 *  - matrices are row-major; `ld*` are row pitches in ELEMENTS.  bf16 operands of the tensor-core kernels need
 *    16-byte aligned base pointers and pitches that are multiples of 8 elements (TMA).
 *  - return value 0 = launched; <0 = rejected (message via mmfm_last_error(), thread local).
 */
#ifndef MMFM_B200_H_
#define MMFM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MMFM_ABI_VERSION 7

const char* mmfm_last_error(void);
int mmfm_abi_version(void);
/* number of SMs of the current device (grid sizing); <=0 when no device */
int mmfm_sm_count(void);

/* Counter-based dropout stream shared by all kernels (restated in oracle/philox_ref.py).  Replaces the
 * nn.Dropout / SDPA dropout_p draws of mm_utils.py:52,111,114 and encoder_embeddings.py:61. */
typedef struct mmfm_dropout {
  const unsigned long long* seed; /* device scalar (graph-replay safe); NULL = dropout off */
  uint32_t site;                  /* stream id of the dropout site */
  uint32_t thresh;                /* element dropped iff random byte < thresh; 0 = off */
  float scale;                    /* 256 / (256 - thresh) */
} mmfm_dropout;

/* ---- tensor-core GEMM (tcgen05 / TMEM / TMA) ------------------------------------------------------------ */
enum mmfm_act {
  MMFM_ACT_NONE = 0,
  MMFM_ACT_GELU = 1,      /* D <- gelu_erf(v); D2 (optional) <- v   (mm_utils.py:51) */
  MMFM_ACT_SOFTSIGN = 2,  /* D <- softsign(v) * act_scale           (encoder_embeddings.py:52) */
  MMFM_ACT_DGELU = 3,     /* D <- v * gelu'(aux)                    (backward of mm_utils.py:51) */
  MMFM_ACT_DSOFTSIGN = 4, /* D <- v * act_scale * (1-|aux/act_scale|)^2   (backward of encoder_embeddings.py:52) */
  MMFM_ACT_GELU_DG = 5,   /* D <- gelu_erf(v); D2 <- gelu_erf'(v): the derivative is saved instead of the pre-activation
                             (erf and the Gaussian term are shared), so the backward epilogue is one multiply */
  MMFM_ACT_MULAUX = 6,    /* D <- v * aux                           (backward of MMFM_ACT_GELU_DG) */
  MMFM_ACT_ROWDOT_DROP = 7 /* out-projection dgrad fused with the attention-backward preparation (autograd of
                             mm_utils.py:111-114): rowdot[(r / S) * G + g][r % S] <- sum over the 32 columns of group g of
                             v * aux  (= delta of head g: rowsum(dO * O)), then D <- dropout(v) (the output-dropout mask
                             of the forward, args->drop).  N % 32 == 0, d_head == 32 (one head = one column group); bf16 D */
};

typedef struct mmfm_gemm_args {
  const void* A; long long lda;  /* bf16 [M,K] */
  const void* B; long long ldb;  /* bf16 [N,K]  (an nn.Linear weight, or its transpose for dgrad) */
  int M, N, K;
  void* D; long long ldd;        /* [M_out, N] bf16 or fp32 */
  int d_fp32;
  void* D2;                      /* optional bf16 second output, pitch ldd */
  const float* bias;             /* [N] or NULL */
  const float* res; long long ldr; /* optional fp32 [M_out, >=N], added last, indexed by the OUTPUT row */
  const void* aux; long long ldaux; /* bf16 [M, >=N] for DGELU / DSOFTSIGN */
  int act; float act_scale;
  mmfm_dropout drop;             /* over the (M,N) field, applied after the activation */
  /* output row remap of the token-embedding GEMM (writes modality m's tokens straight into the packed
   * (B, S=M*T, H) layout, replacing torch.cat of mm.py:98-108):  out_row = (r / remap_T) * remap_S + remap_off +
   * r % remap_T ; remap_T == 0 = identity */
  int remap_T, remap_S, remap_off;
  /* optional [S] flags: token position p = remap_off + r % remap_T (or r % remap_S when remap_T == 0) is zeroed
   * before `res` is added (mm.py:147-149,169-171) */
  const unsigned char* row_zero;
  /* MMFM_ACT_ROWDOT_DROP side output: fp32 [M / rowdot_S, N / 32, rowdot_S] (the attention kernels' delta[B, h, Sq]) */
  float* rowdot; int rowdot_S;
} mmfm_gemm_args;

/* D = epilogue(A . B^T).  Replaces nn.Linear forward (mm_utils.py:51-52,107-109,114,145-147,152;
 * encoder_embeddings.py:50,54; decoder_embeddings.py:50,54,107; mm.py:292) and its autograd dgrad. */
int mmfm_gemm_tn(const mmfm_gemm_args* args, void* stream);

/* dW[NO,KI] += dY[R,NO]^T . X[R,KI]  (fp32 accumulate with red.global.add; caller zeroes dW once per step);
 * dbias (optional, [NO]) += column sums of dY, computed on the tensor pipe in the same pass.
 * Replaces the autograd wgrad (weight and bias) of every nn.Linear on the path. */
int mmfm_gemm_wgrad(const void* dY, long long lddy, const void* X, long long ldx, int R, int NO, int KI, float* dW,
                    long long ldw, float* dbias, void* stream);
/* out[c] += sum_r dY[r,c]  (bias gradient) */
int mmfm_colsum_bf16(const void* dY, long long ld, int R, int NO, float* out, void* stream);

/* ---- conversions ------------------------------------------------------------------------------------- */
/* fp32 [R,C] (pitch ldx) -> bf16 [R,C] (pitch ldy); optional transposed copy yt [C,R] (pitch ldyt) */
int mmfm_cast_bf16(const float* x, long long ldx, void* y, long long ldy, void* yt, long long ldyt, int R, int C,
                   void* stream);

/* ---- LayerNorm (nn.LayerNorm(H), eps 1e-5: encoder_embeddings.py:98-100, decoder_embeddings.py:116-126,
 *      mm.py:72,77) -------------------------------------------------------------------------------------- */
/* y(bf16) = LN(x) ; mean/rstd saved.  modmajor_T > 0: row (b,s) of x is written to row (s/T)*(B*T) + b*T + s%T
 * (modality-major layout feeding the per-modality heads, decoder_embeddings.py:105-107), B = R/S. */
int mmfm_layernorm_fwd(const float* x, const float* gamma, const float* beta, void* y, float* mean, float* rstd,
                       int R, int H, float eps, int modmajor_T, int S, void* stream);
/* dx = dres + LN'(dy) ; optional bf16 copy dxb = bf16(dropout(dx)) ; dgamma/dbeta += column sums.
 * dy is read through the same modality-major remap when modmajor_T > 0. */
int mmfm_layernorm_bwd(const void* dy, const float* x, const float* mean, const float* rstd, const float* gamma,
                       const float* dres, float* dx, void* dxb, const mmfm_dropout* drop, float* dgamma,
                       float* dbeta, int R, int H, int modmajor_T, int S, void* stream);

/* ---- Several LayerNorms over ONE input: the `context_norm` of every decoder layer normalises the same encoder context
 *      (decoder_embeddings.py:141-145 inside the layer loop of :133-147), so x-hat, mean and rstd are shared and only
 *      the affine pairs differ.  Forward: x is read once, n bf16 outputs are written, mean / rstd are saved once.
 *      Backward: dx = LN'(sum_l dy_l . gamma_l) -- LN' is linear in its upstream gradient, so one normalisation of the
 *      gamma-weighted sum replaces n backward passes over x and n read-modify-writes of dx -- with the optional bf16
 *      copy dxb; dgamma[l] / dbeta[l] += column sums of dy_l . x-hat / dy_l.  H in {128, 256, 512}, n <= MMFM_MAX_LN. */
#define MMFM_MAX_LN 8
typedef struct {
  const float* x;                      /* [R, H] fp32 */
  int R, H, n;
  float eps;
  const float* gamma[MMFM_MAX_LN];
  const float* beta[MMFM_MAX_LN];      /* forward only */
  void* y[MMFM_MAX_LN];                /* forward: bf16 [R, H] outputs */
  float* mean;                         /* [R] saved by the forward, read by the backward */
  float* rstd;
  const void* dy[MMFM_MAX_LN];         /* backward: bf16 [R, H] upstream gradients */
  float* dgamma[MMFM_MAX_LN];
  float* dbeta[MMFM_MAX_LN];
  float* dx;                           /* backward: fp32 [R, H] (written, not accumulated) */
  void* dxb;                           /* backward: optional bf16 copy of dx */
} mmfm_ln_multi_args;
int mmfm_layernorm_fwd_multi(const mmfm_ln_multi_args* a, void* stream);
int mmfm_layernorm_bwd_multi(const mmfm_ln_multi_args* a, void* stream);

/* ---- ScaleNorm (mm_utils.py:31-39, config `use_scalenorm: true`): y(bf16) = x * g[0] / max(||x||_2, eps); the
 *      reciprocal norms are saved in rnorm[R].  Backward: dx = dres + g*rnorm*(dy - xhat <dy,xhat>), optional
 *      dropout-masked bf16 copy dxb (as in mmfm_layernorm_bwd), dg[0] += sum_rows <dy, xhat>. ------------------- */
int mmfm_scalenorm_fwd(const float* x, const float* g, void* y, float* rnorm, int R, int H, float eps, void* stream);
int mmfm_scalenorm_bwd(const void* dy, const float* x, const float* rnorm, const float* g, const float* dres, float* dx,
                       void* dxb, const mmfm_dropout* drop, float* dg, int R, int H, float eps, void* stream);

/* ---- masked attention (flash-style; F.scaled_dot_product_attention with the (B,S,S) bool masks of
 *      mm.py:152-158,178-194 evaluated as predicates; mm_utils.py:105-112,143-150) ------------------------ */
enum mmfm_mask_mode {
  MMFM_MASK_KEY = 0,       /* allowed(i,j) = key_valid[b,j]                      (decoder self, default) */
  MMFM_MASK_KEY_OR_DIAG = 1, /* key_valid[b,j] | (i == j)                       (encoder self + cross) */
  MMFM_MASK_CAUSAL = 2     /* j <= i  (key padding dropped, mm.py:183-185) */
};
typedef struct mmfm_attn_args {
  const void* q; long long ldq;   /* bf16 rows (b*Sq + i), head h at columns [h*d, (h+1)*d) */
  const void* k; long long ldk;   /* bf16 rows (b*Sk + j) */
  const void* v; long long ldv;
  void* o; long long ldo;         /* bf16 [B*Sq, h*d], after the output dropout (mm_utils.py:114) */
  float* lse;                     /* [B, h, Sq] log-sum-exp of the scaled masked scores */
  const unsigned char* key_valid; /* [B, Sk] */
  const short* mod_q; const short* mod_k; /* optional [Sq],[Sk] modality ids: allowed |= mod_q[i] != mod_k[j] (sep) */
  int B, n_heads, Sq, Sk, d_head;
  int mask_mode;
  float scale;                    /* 1/sqrt(d_head) */
  mmfm_dropout drop_p;            /* on the probabilities: rows (b*h+hh)*Sq+i, cols Sk */
  mmfm_dropout drop_o;            /* on the output: rows b*Sq+i, cols h*d */
  unsigned short* p_keep;         /* [B, h, Sq, ceil(Sk/64), 4] keep bits of the probability dropout (written by
                                     fwd, read by bwd); may be NULL when drop_p is off */
  /* backward only */
  void* d_o; long long lddo;      /* bf16 [B*Sq, h*d]: in = gradient wrt `o`; overwritten with the gradient wrt the
                                     attention output before the output dropout */
  float* delta;                   /* scratch [B, h, Sq]: rowsum(dO * O) */
  void* dq; long long lddq;
  void* dk; long long lddk;
  void* dv; long long lddv;
  /* backward: non-zero = `delta` is already filled and `d_o` already carries the output-dropout mask (both produced by
   * the out-projection dgrad GEMM, MMFM_ACT_ROWDOT_DROP); the preparation kernel is skipped */
  int prep_done;
} mmfm_attn_args;
int mmfm_attention_fwd(const mmfm_attn_args* args, void* stream);
int mmfm_attention_bwd(const mmfm_attn_args* args, void* stream);

/* ---- token embedding glue ---------------------------------------------------------------------------- */
#define MMFM_MAX_MOD 8
/* Per-modality (B,T) int64 masks as strided views (element strides), so `eval_mask[:, :, 0]` of a (B,T,C) tensor
 * (mm.py:269-270) is passed without a copy.  mask[m] == NULL means "nothing masked". */
typedef struct mmfm_mask_args {
  int n_mod, B, T;
  const long long* mask[MMFM_MAX_MOD]; long long mask_sb[MMFM_MAX_MOD]; long long mask_st[MMFM_MAX_MOD];
  const long long* attn[MMFM_MAX_MOD]; long long attn_sb[MMFM_MAX_MOD]; long long attn_st[MMFM_MAX_MOD];
  int channels[MMFM_MAX_MOD];
  /* Device-side token masking (the Masker's temporal mode, models/masker.py:85-86,132: an i.i.d. Bernoulli(ratio) field
   * over (B,T)) without any host work: when sample_thresh != NULL and sample_thresh[m] (a DEVICE array of n_mod uint32,
   * so a captured graph sees per-step changes) is non-zero, modality m's mask is drawn here instead of read from
   * mask[m]: element e = b*T + t is masked iff word (e & 3) of Philox(counter = (e >> 2, 0, MMFM_MASK_SITE + m, 2),
   * key = *seed) < sample_thresh[m]  (thresh = floor(ratio * 2^32); restated in oracle/philox_ref.py:mask_bernoulli). */
  const unsigned int* sample_thresh;
  const unsigned long long* seed;
} mmfm_mask_args;
#define MMFM_MASK_SITE 8192u
/* With S = n_mod*T and mk = mask & attn (mm.py:270):
 *   zero_flags[s]   = (mk[0,s] == 1)      (mm.py:147,169 -- sample 0's mask zeroes the whole batch)
 *   key_valid[b,s]  = attn[b,s] != 0      (mm.py:152-158,178-194)
 *   tok_mask[b,s]   = mk[b,s] != 0        (loss weights, mm.py:229)
 *   n_examples[m]   = channels[m] * sum(mk[:, m*T:(m+1)*T])   (mm.py:231)
 *   inv_n[0]        = 1 / sum_m n_examples[m]                  (mm.py:237) */
int mmfm_mask_prep(const mmfm_mask_args* args, unsigned char* zero_flags, unsigned char* key_valid,
                   unsigned char* tok_mask, long long* n_examples, float* inv_n, void* stream);
/* emb[b, off+t, :] = mod_emb_row[:] + pos_embed[ts[b,t], :]  (encoder_embeddings.py:56-59); pos_embed may be NULL */
int mmfm_embed_assemble(const float* mod_emb_row, const float* pos_embed, const long long* ts, float* emb, int B,
                        int T, int S, int off, int H, void* stream);
/* gradient of the above: dpos[ts[b,t], :] += g[b, off+t, :] (+ g2) ; dmod[:] += sum_{b,t} (same) */
int mmfm_embed_assemble_bwd(const float* g, const float* g2, const long long* ts, float* dpos, float* dmod, int B,
                            int T, int S, int off, int H, void* stream);
/* d_tok (bf16 [B*T, H]) = dropout_mask( row_zero ? 0 : dx[b, off+t, :] )  -- backward of the embedding epilogue */
int mmfm_embed_grad_prep(const float* dx, void* dtok, const unsigned char* row_zero, const mmfm_dropout* drop, int B,
                         int T, int S, int off, int H, void* stream);
/* small-channel modality (C <= 8, e.g. behaviour C=2): the whole embedder / head as SIMT kernels
 * (encoder_embeddings.py:50-61; decoder_embeddings.py:105-107) */
int mmfm_smallc_embed_fwd(const float* in, const float* W1, const float* b1, const float* W2, const float* b2,
                          const float* emb, float* x, float* hid, const unsigned char* row_zero,
                          const mmfm_dropout* drop, float act_scale, int act, int B, int T, int S, int off, int C,
                          int H, void* stream);
int mmfm_smallc_embed_bwd(const float* in, const float* hid, const float* W2, const float* dx,
                          const unsigned char* row_zero, const mmfm_dropout* drop, float act_scale, int act,
                          float* dW1, float* db1, float* dW2, float* db2, int B, int T, int S, int off, int C, int H,
                          void* stream);
int mmfm_smallc_head_fwd(const void* y, const float* W, const float* b, float* preds, int R, int H, int C,
                         void* stream);
int mmfm_smallc_head_bwd(const void* y, const float* W, const void* dpreds, long long lddp, void* dy, float* dW,
                         float* db, int R, int H, int C, void* stream);

/* ---- fused masked loss + gradient (mm.py:217-239; nn.PoissonNLLLoss(log_input=True) :80, nn.MSELoss :81) -- */
enum mmfm_loss_kind {
  MMFM_LOSS_POISSON = 0, MMFM_LOSS_MSE = 1,
  /* categorical stream (choice / block -- an extension, the reference has none): targets = one-hot / class
   * probabilities over the C classes; ell[.,k] = -t_k * log_softmax(preds)_k, C <= 64 */
  MMFM_LOSS_CE = 2
};
/* preds, targets fp32 [B*T, C] contiguous; tok_mask [B,S] bytes, this modality at columns off..off+T-1.
 * partials[i] = CTA i's share of sum(mask * ell(preds, targets)) (n_partials CTAs, fixed-order finalize);
 * dpreds (bf16, pitch lddp) = mask * ell' * inv_n[0]. */
int mmfm_loss_fwd_bwd(const float* preds, const float* targets, const unsigned char* tok_mask, int S, int off,
                      const float* inv_n, int kind, int B, int T, int C, float* partials, int n_partials, void* dpreds,
                      long long lddp, void* stream);
/* mod_loss[m] = sum of partials[m*n_partials ...]; loss = sum_m mod_loss[m] * inv_n[0] */
int mmfm_loss_finalize(const float* partials, int n_partials, int n_mod, const float* inv_n, float* mod_loss,
                       float* loss, void* stream);
/* Head gradient for arbitrary upstream gradients of loss, mod_loss[m] and preds (autograd of every step output):
 *   dpreds = mask * ell'(preds, targets) * (g_loss[0] * inv_n[0] + g_mod[0]) + g_preds
 * preds / targets / tok_mask / S / off / kind as in mmfm_loss_fwd_bwd.  g_loss, g_mod: device scalars, NULL = that
 * upstream gradient is absent (its term is not evaluated, so inv_n = inf with g_loss NULL stays finite).  g_preds:
 * fp32 upstream gradient of preds with ELEMENT strides (gp_sb, gp_st, gp_sc) over (b, t, c) -- 0 for broadcast
 * dimensions -- or NULL.  ell' is the same device code as mmfm_loss_fwd_bwd: g_loss = 1 alone reproduces its dpreds
 * bit for bit.  Elementwise, no atomics. */
int mmfm_loss_grad(const float* preds, const float* targets, const unsigned char* tok_mask, int S, int off,
                   const float* inv_n, const float* g_loss, const float* g_mod, const float* g_preds, long long gp_sb,
                   long long gp_st, long long gp_sc, int kind, int B, int T, int C, void* dpreds, long long lddp,
                   void* stream);
/* Input gradient of the small-channel embedder (the backward of mmfm_smallc_embed_fwd with respect to `in`), from the
 * saved `hid` and upstream rows that mmfm_smallc_embed_bwd reads, plus W1 [2C, C] (the inputs themselves are not needed):
 *   dX[b,t,:] (+)= W1^T . (act'(hid[b,t,:]) * (W2^T . dropout(row_zero ? 0 : dx[b, off+t, :])))
 * dX fp32 [B*T, C] at pitch lddx; accumulate != 0 adds to it.  One warp per row, no atomics (deterministic). */
int mmfm_smallc_embed_dx(const float* hid, const float* W1, const float* W2, const float* dx,
                         const unsigned char* row_zero, const mmfm_dropout* drop, float act_scale, int act, float* dX,
                         long long lddx, int accumulate, int B, int T, int S, int off, int C, int H, void* stream);

/* ---- multi-tensor cast: bf16 shadows (and transposed shadows for dgrad) of all fp32 weights in one launch -- */
typedef struct mmfm_cast_item {
  const float* src; long long ld_src;   /* fp32 [rows, cols] */
  void* dst; long long ld_dst;          /* bf16 [rows, cols] or NULL */
  void* dst_t; long long ld_dst_t;      /* bf16 [cols, rows] or NULL */
  int rows, cols;
  int tile_start;                       /* exclusive prefix sum of ceil(rows/32)*ceil(cols/32) over the items */
  int pad_;
} mmfm_cast_item;
int mmfm_cast_bf16_multi(const mmfm_cast_item* items_dev, int n_items, int total_tiles, void* stream);
/* x[0..n) *= scale_dev[0]; returns at once on the device when the scale is exactly 1 (upstream gradient of the
 * scalar loss, trainer/base.py:195 always passes 1) */
int mmfm_scale_inplace(float* x, long long n, const float* scale_dev, void* stream);

/* ---- batch wire format (SURVEY section 8f rank 2: spike counts are small non-negative integers, stored as ubyte by
 *      the reference's datasets, dataset_utils.py:29; the dense fp32 (B,T,N) batch of loader/base.py:436-450 can be
 *      shipped as bytes) ------------------------------------------------------------------------------------------ */
/* CSR pieces of a batch (get_binned_spikes_from_sparse, dataset_utils.py:38-43, rebuilds them with scipy on the host):
 * data / indices of all trials concatenated, row_ptr[n_rows + 1] = global offsets of every (trial, bin) row.
 * out: dense uint8 [n_rows, N], fully written (zero fill + scatter). */
int mmfm_csr_to_dense_u8(const unsigned char* data, const int* indices, const long long* row_ptr, long long n_rows, int N,
                         unsigned char* out, void* stream);
/* x: R rows of C bytes (dense).  y32 (optional) fp32 [R, ld32]; y16 (optional) bf16 [R, ld16].  Exact conversions. */
int mmfm_u8_expand(const unsigned char* x, long long R, int C, float* y32, long long ld32, void* y16, long long ld16,
                   void* stream);

/* ---- evaluation metrics (SURVEY section 8f rank 4: bits_per_spike / neg_log_likelihood of src/utils/eval_utils.py:
 *      1052-1119, evaluated per neuron at :201,300,405,608,849, and r2_score per channel, :1539-1549) --------------- */
/* pred, y: fp32 [R, C] dense.  out: 4*C doubles (zeroed here): [sum y | sum y^2 | sum (y-pred)^2 | sum (rate - y log rate)]
 * per column, rate = exp(pred) if log_rate else pred (0 -> 1e-9). */
int mmfm_column_stats(const float* pred, const float* y, long long R, int C, int log_rate, double* out, void* stream);

/* ---- optimizer step (SURVEY section 8f rank 1: torch.optim.AdamW of train_multi_modal.py:197-202 over the flat
 *      master-parameter / gradient buffers; runs right after backward, trainer/base.py:196-198) ------------------- */
/* p, g, exp_avg, exp_avg_sq: n fp32 elements each (16-byte aligned).  step >= 1 is the 1-based update count used for
 * the bias corrections.  Decoupled weight decay, no amsgrad, maximize = false. */
int mmfm_adamw_step(float* p, const float* g, float* exp_avg, float* exp_avg_sq, long long n, float lr, float beta1,
                    float beta2, float eps, float weight_decay, long long step, void* stream);

/* Parameter groups and subsets (ABI 7): one launch updates the segments [lo, hi) of the same four flat buffers, each
 * with the hyper-parameters of its class; elements outside every segment are neither read nor written.  A class is
 * one (parameter group, step count) pair; the bias corrections are computed from `step` on the host in double
 * precision, as mmfm_adamw_step does (which is the one-segment case of the same kernel).
 * segs_dev: n_segs segments in device memory, sorted, non-overlapping, lo a multiple of 4, and chunk0 the prefix sum
 * over the preceding segments of max(1, ceil((hi/4 - lo/4) / MMFM_ADAMW_CHUNK4)); n_chunks is the total.  The table
 * is read by the kernel only: it can be uploaded once and reused while the parameter set stays the same.  A segment
 * with an out-of-range class or bounds is skipped.  classes: n_classes (1..MMFM_ADAMW_MAX_CLASSES) host structs,
 * passed to the kernel by value, so the host array may be reused as soon as the call returns. */
#define MMFM_ADAMW_MAX_CLASSES 64
#define MMFM_ADAMW_CHUNK4 1024
typedef struct {
  long long lo, hi;   /* element range of the flat buffers */
  int cls;            /* index into classes */
  int chunk0;         /* first work chunk of this segment */
} mmfm_adamw_seg;
typedef struct {
  float lr, beta1, beta2, eps, weight_decay;
  int pad_;
  long long step;     /* >= 1: the 1-based update count of the class's parameters */
} mmfm_adamw_class;
int mmfm_adamw_multi(float* p, const float* g, float* exp_avg, float* exp_avg_sq, long long n,
                     const mmfm_adamw_seg* segs_dev, int n_segs, int n_chunks, const mmfm_adamw_class* classes,
                     int n_classes, void* stream);

/* ---- deterministic mode (torch.use_deterministic_algorithms(True)) ---------------------------------------------
 * The entry points above that reduce across CTAs with float atomics have a *_det twin with the same arguments plus a
 * caller-owned workspace.  There every CTA writes its partial to the workspace and a ticketed pairwise tree folds the
 * partials in an order fixed by the grid, so results are bitwise reproducible for the same inputs, shapes and device
 * (the grid depends on the SM count).  No CTA waits for another.  The outputs accumulate (+=) exactly as in the
 * default entry points; they differ from them in the last bits.
 * The workspace: buf (16-byte aligned) of at least the size reported by mmfm_det_ws_bytes, and that many tickets,
 * zeroed once by the caller; every launch leaves its tickets at zero again.  Calls on one stream may share one
 * workspace.  A workspace that is too small is rejected (return -1), never overrun. */
typedef struct mmfm_det_ws {
  void* buf;
  long long bytes;
  unsigned int* tickets;
  int n_tickets;
} mmfm_det_ws;
enum mmfm_det_kind {              /* (d0, d1, d2) of mmfm_det_ws_bytes */
  MMFM_DET_WGRAD = 0,             /* (R, NO, KI) */
  MMFM_DET_COLSUM = 1,            /* (R, NO, -) */
  MMFM_DET_LN_BWD = 2,            /* (R, H, -) */
  MMFM_DET_LN_BWD_MULTI = 3,      /* (R, H, n) */
  MMFM_DET_SCALENORM_BWD = 4,     /* (R, H, -) */
  MMFM_DET_EMBED_ASM_BWD = 5,     /* (B, T, H) */
  MMFM_DET_SMALLC_EMBED_BWD = 6,  /* (B*T, C, H) */
  MMFM_DET_SMALLC_HEAD_BWD = 7,   /* (R, H, C) */
  MMFM_DET_COLUMN_STATS = 8       /* (R, C, -) */
};
/* Host only (queries the device's SM count, launches nothing): workspace bytes and tickets one *_det call of `kind`
 * at these sizes needs, from the same grid arithmetic as its launcher.  Returns 0, or -1 on a bad kind / shape. */
int mmfm_det_ws_bytes(int kind, long long d0, long long d1, long long d2, long long* bytes, int* n_tickets);
int mmfm_gemm_wgrad_det(const void* dY, long long lddy, const void* X, long long ldx, int R, int NO, int KI, float* dW,
                        long long ldw, float* dbias, const mmfm_det_ws* ws, void* stream);
int mmfm_colsum_bf16_det(const void* dY, long long ld, int R, int NO, float* out, const mmfm_det_ws* ws, void* stream);
int mmfm_layernorm_bwd_det(const void* dy, const float* x, const float* mean, const float* rstd, const float* gamma,
                           const float* dres, float* dx, void* dxb, const mmfm_dropout* drop, float* dgamma,
                           float* dbeta, int R, int H, int modmajor_T, int S, const mmfm_det_ws* ws, void* stream);
int mmfm_layernorm_bwd_multi_det(const mmfm_ln_multi_args* a, const mmfm_det_ws* ws, void* stream);
int mmfm_scalenorm_bwd_det(const void* dy, const float* x, const float* rnorm, const float* g, const float* dres,
                           float* dx, void* dxb, const mmfm_dropout* drop, float* dg, int R, int H, float eps,
                           const mmfm_det_ws* ws, void* stream);
/* n_pos = rows of dpos: timestamps outside [0, n_pos) contribute to dmod only.  dpos rows are summed over (b, t) in
 * increasing b * T + t order by one CTA per row. */
int mmfm_embed_assemble_bwd_det(const float* g, const float* g2, const long long* ts, float* dpos, float* dmod, int B,
                                int T, int S, int off, int H, int n_pos, const mmfm_det_ws* ws, void* stream);
int mmfm_smallc_embed_bwd_det(const float* in, const float* hid, const float* W2, const float* dx,
                              const unsigned char* row_zero, const mmfm_dropout* drop, float act_scale, int act,
                              float* dW1, float* db1, float* dW2, float* db2, int B, int T, int S, int off, int C, int H,
                              const mmfm_det_ws* ws, void* stream);
int mmfm_smallc_head_bwd_det(const void* y, const float* W, const void* dpreds, long long lddp, void* dy, float* dW,
                             float* db, int R, int H, int C, const mmfm_det_ws* ws, void* stream);
int mmfm_column_stats_det(const float* pred, const float* y, long long R, int C, int log_rate, double* out,
                          const mmfm_det_ws* ws, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MMFM_B200_H_ */
