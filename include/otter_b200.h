/* otter_b200 — C ABI of the B200-native vision-fusion hot path.
 *
 * The reference (Luodian/Otter) ships no native code and therefore has no FFI; the operations
 * below are the torch calls its hot-path modules make, restated as a C ABI so that a Python host
 * (ctypes, see otter_b200/_lib.py and INTEGRATION.md) can bind them.  Each entry point cites the
 * reference lines it replaces (paths relative to /root/reference).
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless stated otherwise; the caller owns every buffer
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream)
 *   - return value: 0 = ok, non-zero = error; otb_last_error() returns a thread-local message
 *   - no entry point allocates device memory, synchronises the device, or throws
 *   - bf16 = IEEE bfloat16 (2 bytes); "K-major" = reduction dimension contiguous in memory
 */
#ifndef OTTER_B200_H
#define OTTER_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OTB_OK 0
#define OTB_ERR_INVALID 1
#define OTB_ERR_CUDA 2
#define OTB_ERR_UNSUPPORTED 3

const char* otb_last_error(void);
/* Library/ABI version and the SM architecture the kernels were compiled for (100 = sm_100a). */
int otb_version(void);
int otb_compiled_arch(void);
/* Number of kernels this library has launched in the calling process (bench.py "gpu_launches"). */
long long otb_launch_count(void);
/* TMA descriptor cache statistics (which = 0: hits, 1: misses).  Descriptors are cached by (base, shape, pitch, box)
 * under a mutex (SURVEY.md 8b "no global mutable state beyond a mutex-guarded descriptor cache"). */
long long otb_tmap_cache_stat(int which);
/* sizeof() of the ABI structs as the C compiler laid them out: 0 otb_gemm_epilogue, 1 otb_attn_desc,
 * 2 otb_attn_grads, 3 otb_lm_attn_desc, 4 otb_lm_attn_grads (binding self-check for FFI hosts). */
int otb_abi_sizeof(int which);

/* ---------------------------------------------------------------------------------------------
 * GEMM:  D[M,N] = epilogue( A[M,K] . B[N,K]^T )      bf16 operands, fp32 accumulate in TMEM
 * Replaces every nn.Linear / F.linear on the path (modeling_otter.py:139-148,164-167,180-184,
 * 253-256,284-288,340,363-370; xformers_model/clip.py:106-134,145-149) and their autograd
 * dgrad/wgrad.  tcgen05.mma + TMA, persistent, warp-specialised.
 *
 * Operand layouts (ld* in elements):
 *   a_mn_major = 0 : A is stored [M][K] row-major (lda >= K)         (activations, dY for dgrad)
 *   a_mn_major = 1 : A is stored [K][M] row-major (lda >= M)         (dY^T for wgrad, no transpose copy)
 *   b_mn_major = 0 : B is stored [N][K] row-major (ldb >= K)         (nn.Linear weight for forward)
 *   b_mn_major = 1 : B is stored [K][N] row-major (ldb >= N)         (weight for dgrad, X for wgrad)
 * Requirements: lda, ldb, ld_out, ld_aux, ld_res multiples of 8; A, B, out, bias, residual, aux_in and aux_out
 *   16-byte aligned (otherwise OTB_ERR_INVALID naming the operand);
 *   N multiple of 8; for an MN-major operand its MN extent must be a multiple of 8.
 *
 * Epilogue (all optional, applied in this order on the fp32 accumulator v):
 *   v += bias[n]                                   (fp32 [N])
 *   aux_out[m,n] = bf16(v)                         (pre-activation, kept for backward)
 *   v = act(v)             act: 0 none, 1 GELU(erf) (modeling_otter.py:146,367), 2 quick-GELU (CLIP),
 *                               3 relu(v)^2 (Persimmon "relu2", fuyu/modeling_persimmon.py:187-193) — skipped when
 *                               aux_in is given: then `act` names the activation whose DERIVATIVE is applied
 *   v *= act'(aux_in[m,n])                         (backward: aux_in = saved pre-activation; act 3 -> 2 relu(z),
 *                                                   any other value -> gelu'(z))
 *   v *= alpha * (scale_ptr ? (scale_tanh ? tanh(*scale_ptr) : *scale_ptr) : 1)
 *                                                  (tanh gate, modeling_otter.py:387-388,393)
 *   v += residual[m,n]                             (bf16)
 *   out[m,n] = (accumulate ? out[m,n] : 0) + v     (bf16, or fp32 when out_fp32; accumulate needs fp32)
 * ------------------------------------------------------------------------------------------- */
typedef struct otb_gemm_epilogue {
  const float* bias;
  const void* aux_in;
  void* aux_out;
  const float* scale_ptr;
  const void* residual;
  void* out;
  int64_t ld_out, ld_aux_in, ld_aux_out, ld_res;
  int32_t act;
  int32_t scale_tanh;
  int32_t out_fp32;
  int32_t accumulate;
  float alpha;
  int32_t res_fp32; /* residual is fp32 [M][N] instead of bf16 (fp32-grade parity path; needs out_fp32) */
} otb_gemm_epilogue;

int otb_gemm_bf16(const void* A, int a_mn_major, int64_t lda, const void* B, int b_mn_major, int64_t ldb, int M,
                  int N, int K, const otb_gemm_epilogue* epi, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Fused attention cores (tcgen05 QK^T / PV, online fp32 softmax, TMA-staged K/V tiles).
 *   (A) perceiver  latent x (vision ++ latents)   modeling_otter.py:168-179  (Sk2 > 0: second key source)
 *   (B) gated x-attn text x latents, media mask   modeling_otter.py:290-333  (text_time != NULL)
 *   (C) CLIP self-attention                       xformers_model/clip.py:112-128
 * Tensors are addressed in place inside the projection outputs: a matrix is [P*S rows][cols] bf16
 * with row pitch ld; head h lives at columns col0 + h*64.  `*_cols` is the logical column count of the
 * matrix (TMA bound).  Problem p uses rows [p*S, (p+1)*S).  head_dim must be 64.
 *   out[p*Sq+i, out_col0+h*64+d] = sum_j softmax_j(scale * q_i.k_j + mask) v_j[d]
 *   lse [P][H][Sq] fp32 (may be NULL for inference) is what the backward needs.
 * Mask (B): text_time int32 [P][Sq] from otb_text_time(); key j belongs to media slot j / n_per_media.
 *   tt==0 -> row zeroed; 1<=tt<=T_img -> only slot tt-1; tt>T_img -> uniform over all keys.
 * ------------------------------------------------------------------------------------------- */
typedef struct otb_attn_desc {
  const void* q;
  const void* kv1;
  const void* kv2; /* optional second key/value source (perceiver latents), NULL if Sk2 == 0 */
  void* out;
  float* lse;
  const int32_t* text_time;
  int64_t ldq, ldkv1, ldkv2, ld_out;
  int32_t q_cols, kv1_cols, kv2_cols;
  int32_t q_col0, k1_col0, v1_col0, k2_col0, v2_col0, out_col0;
  int32_t n_per_media, T_img;
  int32_t P, H, Sq, Sk1, Sk2, head_dim;
  float scale;
  int32_t mask_ge; /* media mask with torch.ge instead of torch.eq (only_attend_immediate_media=False, :317): keys of
                      media slots 1..text_time; rows with text_time == 0 are then uniform, not zeroed (:326 guard) */
  int32_t causal;  /* self-attention only (Sq == Sk1, no media mask): key j participates iff j <= query row */
} otb_attn_desc;

typedef struct otb_attn_grads {
  const void* dout; /* [P*Sq][..] bf16, same head layout as out */
  void* dq;         /* [P*Sq][..] bf16 */
  void* dkv1;       /* [P*Sk1][..] bf16 : dK at dk1_col0 + h*64, dV at dv1_col0 + h*64 */
  void* dkv2;       /* [P*Sk2][..] bf16 or NULL */
  float* dq_ws;     /* fp32 [P*Sq][H*64] scratch, required when the keys span more than one 128-key tile */
  int64_t ld_dout, ld_dq, ld_dkv1, ld_dkv2;
  int32_t dout_cols, dout_col0, dq_col0, dk1_col0, dv1_col0, dk2_col0, dv2_col0;
  int32_t _pad;
} otb_attn_grads;

int otb_attn_fwd(const otb_attn_desc* d, void* stream);
int otb_attn_bwd(const otb_attn_desc* d, const otb_attn_grads* g, void* stream);

/* ---------------------------------------------------------------------------------------------
 * The north star's single fused kernel (SURVEY.md 7 option (a)): masked cross-attention core + to_out projection +
 * tanh gate + residual, modeling_otter.py:290-340 and :380-389:
 *     y = ( softmax(mask(q k^T * scale)) v  Wo^T ) * tanh(*gate) + residual
 * d: the attention problem as for otb_attn_fwd (one key source, Sk1 = T_img * n <= 64, H <= 8 heads of 64); d->out
 * [P*Sq][H*64] and d->lse still receive O and the log-sum-exp (the backward pass reads them).  wo: bf16 [D][H*64] (the
 * nn.Linear weight, row pitch ld_wo); aux (optional): bf16 [P*Sq][D] pre-gate branch output O Wo^T (for the gate
 * gradient); y: bf16 [P*Sq][D].  D must be a multiple of 512. */
int otb_xattn_out_fused(const otb_attn_desc* d, const void* wo, int64_t ld_wo, const float* gate, const void* residual,
                        int64_t ld_res, void* aux, int64_t ld_aux, void* y, int64_t ld_y, int D, void* stream);

/* ---------------------------------------------------------------------------------------------
 * SURVEY.md §8f rank 1 — causal self-attention of the frozen LM decoder layers (head_dim 128: MPT-7B / LLaMA-7B).
 *   mpt/attention.py:22-84 (scaled_multihead_dot_product_attention), :457-464 (ALiBi key bias), :68-75 (causal mask)
 * qkv is the fused Wqkv GEMM output [B*S][qkv_cols] bf16 (row pitch ld_qkv): head h of Q / K / V at columns
 * q_col0 / k_col0 / v_col0 + h*128.  out [B*S][..] bf16, head h at out_col0 + h*128; lse fp32 [B][H][S].
 *   score(i,j) = scale * q_i.k_j + alibi_slopes[h] * (j - (S-1))      (alibi_slopes NULL: no bias)
 *   causal != 0: keys j > i are masked.
 * Backward returns activation gradients only (the LM is frozen): dqkv has the layout of qkv.
 * ------------------------------------------------------------------------------------------- */
typedef struct otb_lm_attn_desc {
  const void* qkv;
  void* out;
  float* lse;
  const float* alibi_slopes; /* fp32 [H] or NULL */
  int64_t ld_qkv, ld_out;
  int32_t qkv_cols, q_col0, k_col0, v_col0, out_col0;
  int32_t B, H, S, head_dim, causal;
  float scale;
} otb_lm_attn_desc;

typedef struct otb_lm_attn_grads {
  const void* dout; /* [B*S][dout_cols] bf16, head h at dout_col0 + h*128 */
  void* dqkv;       /* [B*S][..] bf16: dQ / dK / dV of head h at dq_col0 / dk_col0 / dv_col0 + h*128 */
  float* dq_ws;     /* fp32 [B*S][H*128] scratch, required when S > 128 */
  int64_t ld_dout, ld_dqkv;
  int32_t dout_cols, dout_col0, dq_col0, dk_col0, dv_col0;
  int32_t _pad;
} otb_lm_attn_grads;

int otb_lm_attn_fwd(const otb_lm_attn_desc* d, void* stream);
int otb_lm_attn_bwd(const otb_lm_attn_desc* d, const otb_lm_attn_grads* g, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Index / mask construction (integer, bit-exact):  modeling_otter.py:296-311
 *   text_time[b,i] = cumsum(media_locations[b,:])[i]; if !attend_previous: +1 on non-media tokens,
 *   then entries > count_nonzero(media_locations[b]) wrap to 0.
 * ------------------------------------------------------------------------------------------- */
int otb_text_time(const uint8_t* media_locations, int B, int L, int attend_previous, int32_t* text_time,
                  void* stream);

/* ---------------------------------------------------------------------------------------------
 * LayerNorm (eps, affine; fp32 statistics)  nn.LayerNorm on the path: modeling_otter.py:136-137,144,
 * 208,251,364; clip.py:160,162,404.  x,y bf16 [rows][D]; gamma/beta fp32 [D]; mean/rstd fp32 [rows].
 * Backward: dx (+ optional `add`, the residual-branch gradient, fused) and per-column parameter
 * gradients via a deterministic two-stage reduction (ws: fp32 [2][chunks][D], chunks = otb_ln_chunks()).
 * ------------------------------------------------------------------------------------------- */
int otb_layernorm_fwd(const void* x, int64_t ldx, const float* gamma, const float* beta, void* y, int64_t ldy,
                      float* mean, float* rstd, int rows, int D, float eps, void* stream);
int otb_ln_chunks(int rows, int D);
int otb_layernorm_bwd(const void* dy, int64_t lddy, const void* x, int64_t ldx, const float* mean,
                      const float* rstd, const float* gamma, const void* add, int64_t ldadd, void* dx,
                      int64_t lddx, float* dgamma, float* dbeta, int accumulate, float* ws, int rows, int D,
                      void* stream);

/* ---------------------------------------------------------------------------------------------
 * Small HBM-bound passes around the GEMMs.
 * ------------------------------------------------------------------------------------------- */
/* dst(bf16)[i] = src(fp32)[i]  — bf16 shadow of fp32 master weights (autocast-equivalent). */
int otb_cast_f32_bf16(const float* src, void* dst, int64_t n, void* stream);
int otb_cast_bf16_f32(const void* src, float* dst, int64_t n, void* stream);
/* dst = float(src) * scale — the up-cast after a bf16 all-reduce(SUM) with 1/world_size folded in (otter_b200/dp.py). */
int otb_cast_bf16_f32_scale(const void* src, float* dst, int64_t n, float scale, void* stream);
/* The same cast for a LIST of tensors in one launch (all trainable weights after an optimizer step).
 * table: device array of n_tensors records {const float* src; bf16* dst; int64 n; int64 first_block}, 32 bytes each,
 * sorted by first_block; tensor t owns blocks [first_block_t, first_block_t + ceil(n_t / 4096)); total_blocks is
 * their sum.  src / dst must be 16-byte aligned. */
int otb_cast_f32_bf16_multi(const void* table, int n_tensors, int64_t total_blocks, void* stream);
/* out[r,:] = bf16(src[(r / div) % mod, :])  fp32 [mod][D] -> bf16 [rows][D]; latents repeat (:232). */
int otb_bcast_rows(const float* src, int div, int mod, void* out, int rows, int D, void* stream);
/* out[r,:] = x[r,:] + bias[(r / div) % mod, :]   bf16 [rows][D] + fp32 [mod][D]  (frame_embs add, :224-226) */
int otb_add_rowbias(const void* x, const float* bias, int div, int mod, void* out, int rows, int D, void* stream);
/* out[g,:] (+)= sum_{r : (r/div)%mod == g} x[r,:]   bf16 [rows][D] -> fp32 [mod][D]
 * (gradient of latents repeat (:232) and of the frame_embs broadcast (:224-226)). Deterministic. */
int otb_grouped_colsum(const void* x, int64_t ldx, int rows, int D, int div, int mod, float* out, int accumulate,
                       void* stream);
/* Tanh-gate gradient (modeling_otter.py:387-388,393):  *dgate (+)= (1 - tanh(*gate)^2) * sum(dy . a)
 * dy, a bf16 [n]; ws fp32 [otb_dot_blocks()] scratch. Deterministic two-stage reduction. */
int otb_dot_blocks(void);
int otb_gate_grad(const void* dy, const void* a, int64_t n, const float* gate, float* dgate, int accumulate,
                  float* ws, void* stream);
/* loss = mean(x^2) (fp32, *loss written), dx = 2 x / n  — the M1 harness loss (BASELINE.md §2). */
int otb_sqmean_loss(const void* x, int64_t n, float* loss, void* dx, float* ws, void* stream);

/* ---------------------------------------------------------------------------------------------
 * fp32-grade forward path (parity mode, csrc/otb_fp32.cu): reproduces the reference's fp32 forward within
 * 1e-3 rel / 1e-5 abs.  GEMMs stay on otb_gemm_bf16: x = x0+x1+x2 (bf16 terms), six cross products as one
 * GEMM over K' = 6K.  otb_split3_concat builds the [rows][6K] operand: pattern 0 = [x0 x0 x1 x1 x0 x2]
 * (A side), pattern 1 = [y0 y1 y0 y1 y2 y0] (B side).  otb_attn_fwd_f32 takes the same descriptor with fp32
 * q/kv/out matrices (lse ignored).
 * ------------------------------------------------------------------------------------------- */
int otb_split3_concat(const float* src, int64_t ld, int rows, int K, int pattern, void* dst, void* stream);
int otb_layernorm_fwd_f32(const float* x, int64_t ldx, const float* gamma, const float* beta, float* y, int64_t ldy,
                          int rows, int D, float eps, void* stream);
int otb_add_rowbias_f32(const float* x, const float* bias, int div, int mod, float* out, int rows, int D,
                        void* stream);
int otb_attn_fwd_f32(const otb_attn_desc* d, void* stream);
/* out = act(acc + bias[n]) * gate + residual   (fp32 [M][N] contiguous; same order as the fused GEMM epilogue) */
int otb_epilogue_f32(const float* acc, const float* bias, int act, const float* scale_ptr, int scale_tanh,
                     const float* residual, float* out, int M, int N, void* stream);

/* fp32-grade BACKWARD passes (csrc/otb_fp32_bwd.cu; dgrad / wgrad reuse the split GEMM): gradients of the path within 1e-3
 * of the reference's fp32 autograd.  All matrices fp32; deterministic (no atomics).
 *   otb_layernorm_bwd_f32  dx (may be NULL) and dgamma / dbeta (both or neither); ws: fp32 [2*rows] scratch
 *   otb_act_bwd_f32        out = dy * act'(pre), act 1 = exact GELU, 2 = quick-GELU
 *   otb_gate_grad_f32      out[0] = (1 - tanh(*gate)^2) * sum(dy * f)     (modeling_otter.py:380-389, the two tanh gates)
 *   otb_rowbias_grad_f32   gradient of otb_add_rowbias_f32's table: out [out_rows][D], rows >= mod are zero
 *   otb_attn_bwd_f32       d as for otb_attn_fwd_f32 with d->out = the forward output; g holds fp32 dout / dq / dkv1 / dkv2
 *                          (dK at dk*_col0 + h*64, dV at dv*_col0 + h*64) and g->dq_ws = fp32 [P*H*Sq*3] scratch */
int otb_layernorm_bwd_f32(const float* dy, int64_t lddy, const float* x, int64_t ldx, const float* gamma, float* dx,
                          int64_t lddx, float* dgamma, float* dbeta, float* ws, int rows, int D, float eps, void* stream);
int otb_act_bwd_f32(const float* dy, const float* pre, int act, float* out, int64_t n, void* stream);
int otb_gate_grad_f32(const float* dy, const float* f, int64_t n, const float* gate, float* out, void* stream);
int otb_rowbias_grad_f32(const float* dy, int div, int mod, int rows, int D, int out_rows, float* out, void* stream);
int otb_attn_bwd_f32(const otb_attn_desc* d, const otb_attn_grads* g, void* stream);

/* CLIP embeddings (xformers_model/clip.py:73-81): */
/* im2col of non-overlapping patches: pixels [N][3][H][W] (fp32 if pix_fp32 else bf16) ->
 * out bf16 [N*(H/p)*(W/p)][Kpad], column c*p*p + i*p + j, zero padded to Kpad. */
int otb_im2col_patches(const void* pixels, int pix_fp32, int N, int H, int W, int patch, void* out, int Kpad,
                       void* stream);
/* h[n,0,:] = cls + pos[0]; h[n,1+t,:] = patch[n*np+t,:] + pos[1+t]   -> bf16 [N][np+1][D] */
int otb_clip_assemble(const void* patch_emb, const float* cls, const float* pos, void* out, int N, int np, int D,
                      void* stream);
/* media[img*v + t, :] = hidden[img, 1+t, :] (+ frame_embs[img % F])  (modeling_otter.py:991,224-227) */
int otb_media_from_clip(const void* hidden, const float* frame_embs, int F, void* out, int n_img, int v, int D,
                        void* stream);
/* Fuyu patch scatter (fuyu/modeling_fuyu.py:65-77): for s with 0 <= idx[b,s] < n_b:
 * out[b,s,:] = cont[b_off[b] + idx[b,s], :] ; else out[b,s,:] = word[b,s,:]. bf16, D % 8 == 0.
 * b_off: int64 [B+1] prefix offsets of the samples' rows inside `cont` (n_b = b_off[b+1] - b_off[b]); ids >= n_b never
 * read out of bounds (the host wrapper raises the reference's ValueError for them before launching). */
int otb_fuyu_scatter(const void* word, const void* cont, const int64_t* idx, const int64_t* b_off, void* out,
                     int B, int S, int D, void* stream);

/* ---------------------------------------------------------------------------------------------
 * SURVEY.md 8f rank 1 — LLaMA decoder layer (the LM of OTTER-Video-LLaMA7B), element-wise passes around the GEMMs and
 * otb_lm_attn_*:  xformers_model/llama.py:74-89 (LlamaRMSNorm), :150-166 (rotate_half rotary embedding), :169-185 (SwiGLU MLP).
 *   otb_rmsnorm_fwd   y = x * rsqrt(mean(x^2) + eps) * weight ; rstd fp32 [rows] kept for backward (may be NULL)
 *   otb_rmsnorm_bwd   dx (+ add) — the LM is frozen, no weight gradient
 *   otb_rope128       in place on `nblk` column blocks of H heads x 128 (q and k of a [rows][3*H*128] buffer); position of
 *                     a row = row % S; backward != 0 applies the transposed rotation
 *   otb_swiglu_fwd/bwd  h = silu(g) * u ; dg, du from dh.   All bf16, row pitches in elements (multiples of 8). */
int otb_rmsnorm_fwd(const void* x, int64_t ldx, const float* weight, void* y, int64_t ldy, float* rstd, int rows, int D,
                    float eps, void* stream);
int otb_rmsnorm_bwd(const void* dy, int64_t lddy, const void* x, int64_t ldx, const float* rstd, const float* weight,
                    const void* add, int64_t ldadd, void* dx, int64_t lddx, int rows, int D, void* stream);
int otb_rope128(void* buf, int64_t ld, int64_t rows, int H, int S, int nblk, float rope_theta, int backward, void* stream);
int otb_swiglu_fwd(const void* g, int64_t ldg, const void* u, int64_t ldu, void* h, int64_t ldh, int64_t rows, int I,
                   void* stream);
int otb_swiglu_bwd(const void* dh, int64_t lddh, const void* g, int64_t ldg, const void* u, int64_t ldu, void* dg,
                   int64_t lddg, void* du, int64_t lddu, int64_t rows, int I, void* stream);

/* ---------------------------------------------------------------------------------------------
 * SURVEY.md 8f rank 3 — Persimmon / Fuyu decoder layer: split + qk-LayerNorm + partial rotary embedding.
 * Replaces fuyu/modeling_persimmon.py:277-303 (`_split_heads`, fused_layer_norm on q and k, fused_apply_rotary_emb on
 * the first rotary_dims of every head, non-interleaved).  fused: bf16 [rows][H][3][64] (query_key_value output);
 * qkv: bf16 [rows][3*H*64] = q | k | v column blocks, head h at columns h*64 of its block (the layout otb_attn_* reads);
 * stats: fp32 [rows][H][4] = mean_q, rstd_q, mean_k, rstd_k (kept for backward); position of a row = row % S.
 * Backward: dqkv -> dfused (same layouts) and the four [64] affine gradients through a deterministic two-stage
 * reduction; ws: otb_qkln_rope_ws_floats() floats. */
int otb_qkln_rope_ws_floats(void);
int otb_qkln_rope_fwd(const void* fused, int64_t ld_fused, const float* q_gamma, const float* q_beta,
                      const float* k_gamma, const float* k_beta, void* qkv, int64_t ld_qkv, float* stats, int64_t rows,
                      int H, int S, int rotary_dims, float rope_theta, float eps, void* stream);
int otb_qkln_rope_bwd(const void* dqkv, int64_t ld_dqkv, const void* fused, int64_t ld_fused, const float* stats,
                      const float* q_gamma, const float* k_gamma, void* dfused, int64_t ld_dfused, float* dq_gamma,
                      float* dq_beta, float* dk_gamma, float* dk_beta, int accumulate, float* ws, int64_t rows, int H,
                      int S, int rotary_dims, float rope_theta, void* stream);

/* ---------------------------------------------------------------------------------------------
 * SURVEY.md 8f rank 4 — input pipeline on the device.  Replaces the per-image host transform
 * Resize((S,S), BICUBIC) -> ToTensor -> Normalize of pipeline/mimicit_utils/mimicit_dataset.py:132-143,329-350
 * and the fp32 stack + bf16 cast of :510-549 / instruction_following.py:99.
 * table: device int64 [N][10] = {src ptr (uint8 HWC, 3 channels), H, W, h-bounds offset, h-coefficient offset,
 * h ksize, v-bounds offset, v-coefficient offset, v ksize, byte offset of this image's [H][S][3] intermediate in tmp};
 * coef: device int32 pool holding, per distinct (in, out) size pair, bounds [S][2] = (first tap, tap count) and the
 * 22-bit fixed-point weights [S][ksize] (Pillow's precompute_coeffs + normalize_coeffs_8bpc, computed by the host
 * binding in float64).  out: [N][3][S][S] bf16 (or fp32).  Bit-exact w.r.t. Pillow / torchvision.  */
int otb_preprocess_images(const int64_t* table, const int32_t* coef, int N, int max_h, int S, void* tmp, float mean0,
                          float mean1, float mean2, float std0, float std1, float std2, void* out, int out_fp32,
                          void* stream);

/* ---------------------------------------------------------------------------------------------
 * SURVEY.md §8f row 2 — the steps immediately either side of the hot path in the training step.
 * Label masking (integer, bit-exact): pipeline/train/instruction_following.py:163-190.
 *   labels = where(ids == eos, eos, mask_val); for every <answer> the span up to and including its matching
 *   <|endofchunk|> copies the ids (both pairing passes of the reference); labels[:, 0] = mask_val.
 * Shifted cross-entropy: src/otter_ai/models/mpt/modeling_mpt.py:430-436 (HF LLaMA computes the same shift):
 *   target[b,t] = labels[b,t+1], last position and -100 ignored; loss = mean over supervised targets;
 *   dlogits (optional, same dtype as logits) = d loss / d logits.  ws: fp32 [1 + B*L].
 * ------------------------------------------------------------------------------------------- */
int otb_label_mask(const int64_t* input_ids, int B, int L, int64_t eos_id, int64_t answer_id, int64_t eoc_id,
                   int64_t mask_val, int64_t* labels, void* stream);
int otb_shifted_cross_entropy(const void* logits, int logits_fp32, int64_t ld, const int64_t* labels, int B, int L,
                              int V, float* loss, void* dlogits, int64_t ldd, float* ws, void* stream);
/* x *= *scalar (device scalar; bf16 or fp32 x) — applies the upstream loss gradient without a host sync. */
int otb_scale_by_scalar(void* x, int x_fp32, int64_t n, const float* scalar, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* OTTER_B200_H */
