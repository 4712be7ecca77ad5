/*
 * icd_b200.h — C ABI of libicd_b200.so: the B200 (sm_100a) captioning-decoder hot path.
 *
 * The reference (SarahAlkhateeb/Image-Captioning-with-Different-Decoders) is pure Python/PyTorch and
 * has no FFI of its own; the "operator interface" of this path is the nn.Module surface
 *   models/attention.py:18-61   SoftAttention.forward
 *   models/attention.py:151-164 AttentionDecoder.init_hidden_state
 *   models/attention.py:218-284 AttentionDecoder.forward (+ its autograd backward)
 *   models/baseline.py:81-111   BaselineDecoder.forward  (+ its autograd backward)
 *   gen_captions.py:16-131      attention_caption_image_beam_search (+ the same search over BaselineDecoder steps)
 *                               and seeded caption sampling (temperature, top-k) over both decoders' steps
 *   train_utils.py:2-12 + models/attention.py:417-430   clamp(+-grad_clip) + Adam step
 * Each entry point below names the reference lines it replaces.  A reference maintainer binds
 * them with ctypes (see INTEGRATION.md); no torch types cross this boundary.
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name ends in _host;
 *   - row-major, element strides given explicitly where a tensor may be a slice;
 *   - `stream` is a cudaStream_t passed as void*; every call is stream-ordered and asynchronous,
 *     never synchronises the device, never allocates: all workspace is caller-provided;
 *   - return value: 0 ok; <0 bad argument / unsupported shape (see icd_last_error_string);
 *     >0 a cudaError_t;
 *   - thread-compatible: no global mutable state except the per-thread last-error string.
 */
#ifndef ICD_B200_H
#define ICD_B200_H

#include <stdint.h>

#if defined(__GNUC__)
#define ICD_API __attribute__((visibility("default")))
#else
#define ICD_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define ICD_B200_ABI_VERSION 18
#define ICD_MAX_STEPS 256

ICD_API int icd_version(void);                       /* ICD_B200_ABI_VERSION the library was built with */
ICD_API const char* icd_last_error_string(void);     /* per-thread, valid until the next failing call     */
ICD_API int icd_sizeof_att_desc(void);               /* sizeof(icd_att_desc_t)  — struct-layout self check */
ICD_API int icd_sizeof_base_desc(void);
ICD_API int icd_sizeof_beam_desc(void);
ICD_API int icd_sizeof_base_beam_desc(void);
ICD_API int icd_sizeof_sample_desc(void);
ICD_API int icd_sizeof_base_sample_desc(void);
ICD_API int icd_has_tensor_core_gemm(void);          /* 1 if the tcgen05/TMA GEMM path was compiled in     */
/* Tile pairing of the tensor-core contraction (also env ICD_GEMM_PAIR): 0 single-CTA tiles, 1 CTA pairs sharing the B tile
 * by TMA multicast, 2 CTA pairs on one 256-row tile with tcgen05.mma.cta_group::2; any other value restores the built-in
 * policy (cta_group::2 pairs for long-K shapes, single CTAs otherwise).  Returns the previous forced mode or -1. */
ICD_API int icd_gemm_set_pair_mode(int mode);
ICD_API int64_t icd_launch_count(void);              /* kernels launched by this library so far (process-wide) */

/* Optional device-side timing of the attention-step kernels (bench.py's roofline line).  icd_prof_enable(n), n >= 1:
 * every n-th icd_attention_step_fwd / _bwd launch (per direction) is bracketed by a cudaEvent pair on its own stream
 * (an event record between two kernels costs a few microseconds and suppresses their programmatic overlap, so a
 * timed region samples with n > 1); icd_prof_enable(0) switches it off.  icd_prof_collect waits for the recorded
 * events, sums elapsed milliseconds / launches / rows per direction over the SAMPLED launches and resets. */
ICD_API int icd_prof_enable(int on);
ICD_API int icd_prof_collect(double* fwd_ms, int64_t* fwd_launches, int64_t* fwd_rows,
                     double* bwd_ms, int64_t* bwd_launches, int64_t* bwd_rows);

/* ------------------------------------------------------------------------------------------------
 * Dense contraction  C[M,N] = A[M,K] * B[N,K]^T (+ epilogue), fp32 storage.
 *   A(m,k) = A[m*sam + k*sak], B(n,k) = B[n*sbn + k*sbk]  (one stride of each operand must be 1)
 *   C(m,n) = C[m*ldc + n]
 *   epilogue: v = acc + bias1[n] + bias2[n] + add1[m*ld1+n] + add2[m*ld2+n]; (any may be NULL)
 *             if (row_mask && !row_mask[m]) v = 0;   C = v + beta*C
 *   precision: ICD_PREC_FP32  — fp32 FMA (parity tier),
 *              ICD_PREC_BF16  — bf16 operands on tcgen05 tensor cores, fp32 accumulate (fast tier)
 *              ICD_PREC_FP32X3 — 3-term bf16 split on the tensor cores, fp32-grade accuracy
 * Replaces every nn.Linear / LSTMCell matmul on the path (models/attention.py:54,55,161-163,
 * 270,277-279; models/baseline.py:106,109).
 * ---------------------------------------------------------------------------------------------- */
#define ICD_PREC_FP32 0
#define ICD_PREC_BF16 1
/* fp32-grade contraction on the bf16 tensor cores: every fp32 operand is split into three bf16 terms (x = x1 + x2 + x3,
 * 24 mantissa bits) and the six significant cross terms x1y1 + x1y2 + x2y1 + x1y3 + x3y1 + x2y2 are accumulated in fp32
 * by ONE tcgen05 contraction over a 6x longer K (the terms are concatenated along K).  Operand rounding is eliminated;
 * the remaining error is the tensor core's truncating fp32 accumulator (~6e-6 norm-wise at K = 512: ~70x tighter than
 * single-pass TF32, ~500x tighter than bf16 operands) at ~2.5x the speed of the fp32 FMA kernel.  Used by caption
 * generation (identical beam captions need fp32-grade logits); accepted by icd_gemm and icd_beam_search. */
#define ICD_PREC_FP32X3 2
/* allow split-K with atomic accumulation (run-to-run summation order not fixed): used only for the weight-gradient
 * contractions whose M x N is small and K = B*T or B*196; every forward contraction is deterministic */
#define ICD_GEMM_ALLOW_SPLITK 1

typedef struct {
    const float* A; int64_t sam, sak;
    const float* B; int64_t sbn, sbk;
    float* C; int64_t ldc;
    int32_t M, N, K;
    const float* bias1; const float* bias2;
    const float* add1; int64_t ld1;
    const float* add2; int64_t ld2;
    const uint8_t* row_mask;
    float beta;
    int32_t precision;
    int32_t flags;                /* ICD_GEMM_* bits */
    void* ws; int64_t ws_bytes;   /* ICD_PREC_BF16 / FP32X3: >= icd_gemm_ws_bytes(M,N,K,precision) bytes for the bf16 operand copies */
} icd_gemm_desc_t;

ICD_API int64_t icd_gemm_ws_bytes(int32_t M, int32_t N, int32_t K, int32_t precision);
ICD_API int icd_gemm(const icd_gemm_desc_t* d, void* stream);

/* The tensor-core contraction on operands that are ALREADY bf16 (no staging pass): C[M,N] (fp32, optional) and / or
 * C16[M,N] (bf16, optional) = A * B^T + bias1[n] + add1[m,n], rows with row_mask[m] == 0 forced to 0.
 *   a_mn = 0: A is K-major, stored [M][K] with lda elements between rows;  a_mn = 1: MN-major, stored [K][M] with lda
 *   elements between k rows (a row-major activation used as the dY^T operand of dW = dY^T X).  Same for B / b_mn.
 *   lda / ldb multiples of 8, operands 16-byte aligned.  splitk_ws: optional icd_gemm_bf16_splitk_ws_floats(M,N,K)
 *   floats enabling deterministic split-K for small M x N.
 */
ICD_API int64_t icd_gemm_bf16_splitk_ws_floats(int32_t M, int32_t N, int32_t K);
ICD_API int icd_gemm_bf16_operands(const void* A16, int64_t lda, int32_t a_mn, const void* B16, int64_t ldb, int32_t b_mn,
                           float* C, int64_t ldc, void* C16, int64_t ldc16, int32_t M, int32_t N, int32_t K,
                           const float* bias1, const float* add1, int64_t ld1, const uint8_t* row_mask,
                           float* splitk_ws, int64_t splitk_ws_floats, void* stream);

/* ------------------------------------------------------------------------------------------------
 * SoftAttention step, forward (models/attention.py:55-60 with att_enc hoisted, + :270-271 gate).
 *   rows      : number of decoder rows processed (batch_size_t, or images*beams)
 *   img_index : optional [rows] int32 — row r attends over image img_index[r] (beam search);
 *               NULL => row r uses image r
 *   enc       : (n_img, P, C) fp32 channel-last feature maps
 *   att_enc   : (n_img, P, A) fp32  = enc_att(enc)            (models/attention.py:54)
 *   att_dec   : row r at att_dec + r*ld_dec, A floats         (dec_att(h), :55)
 *   fbeta_pre : row r at fbeta_pre + r*ld_fb, C floats        (f_beta(h) before sigmoid, :270)
 *   alpha     : out, row r at alpha + r*ld_alpha, P floats    (softmax over pixels, :58)
 *   awe_raw, gate, gated : out (rows, C) each, any may be NULL:
 *        awe_raw = sum_p alpha*enc (:59-60), gate = sigmoid(fbeta_pre), gated = gate*awe_raw (:271)
 * ---------------------------------------------------------------------------------------------- */
ICD_API int icd_attention_step_fwd(int rows, int P, int C, int A,
                           const int32_t* img_index,
                           const float* enc, const float* att_enc,
                           const float* att_dec, int64_t ld_dec,
                           const float* w_full, const float* b_full,
                           const float* fbeta_pre, int64_t ld_fb,
                           float* alpha, int64_t ld_alpha,
                           float* awe_raw, float* gate, float* gated,
                           void* stream);

/* Backward of the step above for the recurrent path.
 *   in : d_gated (rows,C); gate, awe_raw (rows,C) and alpha saved by the forward;
 *        d_alpha_ext: optional upstream gradient on alpha itself (row stride ld_dalpha)
 *   out: d_att_dec row r at d_att_dec + r*ld_ddec (A floats)
 *        d_fbeta_pre row r at d_fbeta_pre + r*ld_dfb (C floats)
 *        d_e row r at d_e + r*ld_de (P floats)  — gradient w.r.t. the pre-softmax scores; consumed
 *        after the time loop by icd_attention_proj_bwd (d_att_enc is NOT read-modify-written per step)
 *        d_awe_out (rows,C), optional: d(loss)/d(awe_raw) = d_gated*gate, kept when the gradient w.r.t. the encoder
 *        features is wanted (icd_attention_enc_grad)
 */
ICD_API int icd_attention_step_bwd(int rows, int P, int C, int A,
                           const float* enc, const float* att_enc,
                           const float* att_dec, int64_t ld_dec,
                           const float* w_full,
                           const float* alpha, int64_t ld_alpha,
                           const float* d_alpha_ext, int64_t ld_dalpha,
                           const float* gate, const float* awe_raw, const float* d_gated,
                           float* d_att_dec, int64_t ld_ddec,
                           float* d_fbeta_pre, int64_t ld_dfb,
                           float* d_e, int64_t ld_de, float* d_awe_out,
                           void* stream);

/* Encoder-feature gradient, attention + initial-state part (models/attention.py:59-60, :161; the reference reaches it
 * when --fine_tune_encoder unfreezes ResNet blocks, train.py:39):
 *   d_enc[b,p,c] = sum_t alpha[b,t,p] * d_awe[t,b,c] + d_mean[b,c] / P        (d_enc is WRITTEN; d_mean may be NULL)
 * alphas (B,T,P), d_awe_all (T,B,C) as saved by icd_attention_step_bwd, bt_host[T] optional (NULL => all rows active in
 * all steps) with row_len_ws = B ints of scratch.  The enc_att part d_att_enc * W_e is added by a contraction (beta 1).
 */
ICD_API int icd_attention_enc_grad(int B, int T, int P, int C, const int32_t* bt_host,
                           const float* alphas, const float* d_awe_all, const float* d_mean,
                           float* d_enc, int32_t* row_len_ws, void* stream);

/* After the time loop: d_att_enc[b,p,a] = w_full[a] * sum_t d_e[b,t,p] * [att_enc[b,p,a]+att_dec[t,b,a] > 0]
 * plus the full_att parameter gradients (d_w_full[A], d_b_full[1]) and, from the same pass, the enc_att bias
 * gradient d_b_enc[A] = sum_{b,p} d_att_enc[b,p,:] (may be NULL).
 *   att_dec_all: (T, B, *) with row (t,b) at att_dec_all + (t*B+b)*ld_dec ; d_e: (B, T, P)
 *   bt_host[T]: rows active at step t;   partial: workspace of icd_attention_proj_bwd_ws_floats() floats
 */
ICD_API int64_t icd_attention_proj_bwd_ws_floats(int B, int P, int A);
ICD_API int icd_attention_proj_bwd(int B, int T, int P, int A, const int32_t* bt_host,
                           const float* att_enc, const float* att_dec_all, int64_t ld_dec,
                           const float* w_full, const float* d_e,
                           float* d_att_enc, float* d_w_full, float* d_b_full, float* d_b_enc,
                           float* partial, void* stream);

/* bf16-STORED feature variants of the three entry points above (tensor-core tier): enc16 (n_img,P,C) and att_enc16
 * (n_img,P,A) are bf16, all arithmetic and every other tensor stay fp32.  Optional bf16 copies of results that feed
 * the next tensor-core contraction: gated16 (rows,C); dz16 row r at dz16 + r*ld_dz16: [d_att_dec (A) | d_fbeta_pre (C)].
 */
ICD_API int icd_attention_step_fwd_bf16(int rows, int P, int C, int A, const int32_t* img_index,
                                const void* enc16, const void* att_enc16,
                                const float* att_dec, int64_t ld_dec,
                                const float* w_full, const float* b_full,
                                const float* fbeta_pre, int64_t ld_fb,
                                float* alpha, int64_t ld_alpha,
                                float* awe_raw, float* gate, float* gated, void* gated16, void* stream);
ICD_API int icd_attention_step_bwd_bf16(int rows, int P, int C, int A,
                                const void* enc16, const void* att_enc16,
                                const float* att_dec, int64_t ld_dec, const float* w_full,
                                const float* alpha, int64_t ld_alpha,
                                const float* d_alpha_ext, int64_t ld_dalpha,
                                const float* gate, const float* awe_raw, const float* d_gated,
                                float* d_att_dec, int64_t ld_ddec,
                                float* d_fbeta_pre, int64_t ld_dfb,
                                float* d_e, int64_t ld_de,
                                void* dz16, int64_t ld_dz16, float* d_awe_out, void* stream);
/* Host-only (no GPU needed): the launch form the two entry points above choose for `rows` rows per launch — the shrinking
 * batch_size_t of models/attention.py:261-265 and small batches (DESIGN.md 5.1, "few rows per launch" / "row balance").
 * direction 0 = forward, 1 = backward.  out4[0] = CTAs per row of the rows that run shared (1: none), out4[1] = rows that run
 * shared (forward: 0 or all; backward: the last n rows, as two half-row CTAs each), out4[2] = CTAs of the launch,
 * out4[3] = 1 if the 128-register instantiation is used (at most two CTAs per SM).  The ICD_ATT_* environment overrides
 * (INTEGRATION.md) are honoured. */
ICD_API int icd_attention_step_launch_plan_bf16(int direction, int rows, int P, int C, int A, int32_t* out4);
/* d_att_enc (fp32) and d_att_enc16 (bf16) are both optional outputs (at least one should be given) */
ICD_API int icd_attention_proj_bwd_bf16(int B, int T, int P, int A, const int32_t* bt_host,
                                const void* att_enc16, const float* att_dec_all, int64_t ld_dec,
                                const float* w_full, const float* d_e,
                                float* d_att_enc, void* d_att_enc16, float* d_w_full, float* d_b_full,
                                float* d_b_enc, float* partial, void* stream);
/* the same with d_att_dec_all (T*B, A; leading dimension ld_ddec; rows of inactive (t, b) zero) = the gradient w.r.t. att_dec
 * written by icd_attention_step_bwd_bf16: d full_att.weight is then formed as  sum att_enc * S + (sum att_dec * d_att_dec) / w
 * (S = the masked d_e sums the kernel needs anyway) — 2 instead of 5 instructions per (pixel, channel, step).  NULL: as above. */
ICD_API int icd_attention_proj_bwd_bf16_ex(int B, int T, int P, int A, const int32_t* bt_host,
                                const void* att_enc16, const float* att_dec_all, int64_t ld_dec,
                                const float* w_full, const float* d_e,
                                float* d_att_enc, void* d_att_enc16, float* d_w_full, float* d_b_full,
                                float* d_b_enc, float* partial, const float* d_att_dec_all, int64_t ld_ddec, void* stream);

/* ------------------------------------------------------------------------------------------------
 * AttentionDecoder.forward / backward, teacher-forced (models/attention.py:218-284).
 * One descriptor carries inputs, weights, outputs, tensors saved for backward and scratch.
 * Shapes: B batch, T = max(decode_lengths), L caption columns, P pixels, C encoder dim,
 *         A attention dim, D decoder dim, E embed size, V vocab, NZ = A + C + 4*D.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t B, T, L, P, C, A, D, E, V;
    int32_t precision;            /* ICD_PREC_* for the dense contractions                      */
    int32_t emb_is_f64;           /* embedding table (and its gradient) are float64 (GloVe path)  */
    int32_t bt_host[ICD_MAX_STEPS]; /* batch_size_t = sum(l > t), first-rows semantics (:261-265)  */
    /* inputs */
    const float* enc;             /* (B,P,C) */
    const void* enc16;            /* optional, ICD_PREC_BF16 only: the features already stored as bf16 (B,P,C), e.g. the
                                     output of an encoder run under autocast; `enc` may then be NULL */
    const int64_t* captions;      /* (B,L)   */
    const uint8_t* drop_mask;     /* (T,B,D) keep-mask or NULL (eval / p=0)   (:279)              */
    float drop_scale;             /* 1/(1-p) */
    /* weights, state_dict order of SURVEY.md 8b */
    const float *enc_att_w, *enc_att_b, *dec_att_w, *dec_att_b, *full_att_w, *full_att_b;
    const float *w_ih, *w_hh, *b_ih, *b_hh;
    const float *h_lin_w, *h_lin_b, *c_lin_w, *c_lin_b;
    const float *f_beta_w, *f_beta_b, *fc_w, *fc_b;
    const void* emb_w;            /* (V,E) fp32 or fp64; NULL => emb_x below already holds pre-computed embeddings (T,B,E)
                                     (use_bert branch, models/attention.py:242-244), no embedding gradient */
    /* outputs */
    float* predictions;           /* (B,T,V) rows >= batch_size_t are exactly 0 (:253,280)        */
    float* alphas;                /* (B,T,P)                                    (:257,281)        */
    /* saved for backward (fwd writes, bwd reads) */
    float* att_enc;               /* (B,P,A)  */
    float* mean_enc;              /* (B,C)    */
    float* emb_x;                 /* (T,B,E)  */
    float* xg;                    /* (T,B,4D) */
    float* w_cat;                 /* (NZ,D) = [dec_att_w; f_beta_w; w_hh] */
    float* b_cat;                 /* (NZ)   = [dec_att_b; f_beta_b; 0]    */
    float* z;                     /* (T,B,NZ) */
    float* awe_raw;               /* (T,B,C)  */
    float* gate;                  /* (T,B,C)  */
    float* gated;                 /* (T,B,C)  */
    float* gates_act;             /* (T,B,4D) */
    float* h_all;                 /* (T+1,B,D) */
    float* c_all;                 /* (T+1,B,D) */
    float* hdrop;                 /* (B,T,D)  */
    uint8_t* row_valid;           /* (B*T)    */
    float* gates_pre;             /* (B,4D) scratch */
    /* ---- backward only ---- */
    const float* d_predictions;   /* (B,T,V) */
    const void* d_predictions16;  /* optional bf16 copy of d_predictions, row stride ld_dpred16 (multiple of 8), as written
                                     by icd_cross_entropy_bwd; ICD_PREC_BF16 only; NULL => converted internally */
    int64_t ld_dpred16;
    const float* d_alphas;        /* (B,T,P) or NULL */
    float *d_enc_att_w, *d_enc_att_b;
    float *d_w_cat, *d_b_cat;     /* (NZ,D),(NZ): rows [0,A) dec_att, [A,A+C) f_beta, [A+C,NZ) w_hh / b_hh(=b_ih) */
    float *d_full_att_w, *d_full_att_b;
    float *d_w_ih;                /* (4D,E+C) */
    float *d_h_lin_w, *d_h_lin_b, *d_c_lin_w, *d_c_lin_b;
    float *d_fc_w, *d_fc_b;
    void* d_emb_w;                /* (V,E) fp32/fp64, pre-zeroed by this call; NULL => embedding frozen */
    /* backward scratch */
    float* d_hdrop;               /* (B,T,D)  */
    float* dz;                    /* (T,B,NZ) */
    float* d_e;                   /* (B,T,P)  */
    float* dh;                    /* (B,D)    */
    float* dc;                    /* (B,D)    */
    float* d_gated;               /* (B,C)    */
    float* d_att_enc;             /* (B,P,A)  ICD_PREC_FP32 only (the bf16 tier keeps a bf16 copy in tc_ws) */
    float* d_emb_x;               /* (T,B,E)  */
    /* optional: gradient w.r.t. the encoder features (encoder_out.requires_grad, --fine_tune_encoder) */
    float* d_enc;                 /* (B,P,C) output; NULL => not computed                          */
    float* d_awe_all;             /* (T,B,C) scratch, required with d_enc                          */
    float* d_mean;                /* (B,C)   scratch, required with d_enc                          */
    float* proj_partial;          /* icd_attention_proj_bwd_ws_floats(B,P,A) floats */
    /* ICD_PREC_BF16 only: arena for the bf16 operand copies, shared by fwd and bwd of the same step */
    void* tc_ws; int64_t tc_ws_bytes;   /* >= icd_attention_decoder_ws_bytes(desc) */
    /* backward only, optional (NULL = not recorded): cudaEvent_t handles recorded on `stream` as soon as a group of weight
     * gradients is final, so that a data-parallel caller can start all-reducing them while the rest of the backward runs:
     *   ev_fc_ready  — d_fc_w, d_fc_b (right after the vocabulary-layer contractions, BEFORE the time loop);
     *   ev_rec_ready — d_h_lin_*, d_c_lin_*, d_w_cat, d_b_cat, d_w_ih, d_emb_w (after the hoisted recurrent weight gradients,
     *                  before the attention-projection pass that produces d_full_att_*, d_enc_att_*). */
    void* ev_fc_ready; void* ev_rec_ready;
} icd_att_desc_t;

ICD_API int64_t icd_attention_decoder_ws_bytes(const icd_att_desc_t* d);
ICD_API int icd_attention_decoder_fwd(const icd_att_desc_t* d, void* stream);
ICD_API int icd_attention_decoder_bwd(const icd_att_desc_t* d, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Captions that share images (several reference captions per image, self-critical samples): the teacher-forced forward and
 * backward above with caption row r attending over image img_index[r] of n_img images.  The result is by definition that of
 * the plain calls on the replicated features enc[img_index]; the features are never replicated.
 * In an indexed call these fields of icd_att_desc_t hold ONE ENTRY PER IMAGE (n_img leading rows instead of B):
 *   enc / enc16 (n_img,P,C), att_enc (n_img,P,A), d_enc (n_img,P,C) (the sum over each image's rows), d_att_enc (n_img,P,A).
 * Every other field stays per row (B), mean_enc included: it is computed once per image and written to each of its rows, so
 * the h_lin / c_lin contractions and their gradients do not change.
 * img_row_ptr / img_rows: the rows of image i are img_rows[img_row_ptr[i] .. img_row_ptr[i+1]), ascending — every per-image
 * sum (d_att_enc, d enc_att.*, d_enc) adds its rows in that order, then steps in order: the result is deterministic.
 * The device-side index is not validated (values must lie in [0, n_img) and agree with the CSR); the host wrappers check it.
 * A NULL index makes the _indexed entry points identical to the plain ones.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t n_img;                /* images (>= 1); an image may have no rows */
    const int32_t* img_index;     /* (B)         device: image of each caption row      */
    const int32_t* img_row_ptr;   /* (n_img + 1) device: CSR offsets, [0] = 0, [n_img] = B */
    const int32_t* img_rows;      /* (B)         device: rows of each image, ascending    */
} icd_att_index_t;

ICD_API int icd_sizeof_att_index(void);
ICD_API int64_t icd_attention_decoder_ws_bytes_indexed(const icd_att_desc_t* d, const icd_att_index_t* ix);
ICD_API int icd_attention_decoder_fwd_indexed(const icd_att_desc_t* d, const icd_att_index_t* ix, void* stream);
ICD_API int icd_attention_decoder_bwd_indexed(const icd_att_desc_t* d, const icd_att_index_t* ix, void* stream);
/* floats of desc->proj_partial an indexed backward needs (B caption rows, n_img images) */
ICD_API int64_t icd_attention_proj_bwd_ws_floats_indexed(int B, int n_img, int P, int A);

/* init_hidden_state (models/attention.py:151-164): mean over pixels, h_lin, c_lin.  h, c: (B,D).
 * Stand-alone entry point (caption generation): precision must be ICD_PREC_FP32 — the tensor-core tiers need a
 * workspace and are reached through icd_attention_decoder_fwd / icd_beam_search. */
ICD_API int icd_init_hidden_state(int B, int P, int C, int D, int precision, const float* enc,
                          const float* h_lin_w, const float* h_lin_b,
                          const float* c_lin_w, const float* c_lin_b,
                          float* mean_enc, float* h, float* c, void* stream);

/* ------------------------------------------------------------------------------------------------
 * BaselineDecoder.forward / backward (models/baseline.py:81-111): embedding of captions[:, :-1],
 * image feature prepended as step 0, 1-layer LSTM from zero state (gate order i,f,g,o), vocab linear.
 * B batch, L caption columns (= LSTM steps), E embed, H hidden, V vocab.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t B, L, E, H, V;
    int32_t precision;
    int32_t emb_is_f64;
    const float* img_features;    /* (B,E)   */
    const int64_t* captions;      /* (B,L)   */
    const void* emb_w;            /* (V,E)   */
    const float *w_ih, *w_hh, *b_ih, *b_hh;   /* (4H,E) (4H,H) (4H) (4H) */
    const float *lin_w, *lin_b;   /* (V,H) (V) */
    float* outputs;               /* (B,L,V) */
    /* saved */
    float* x;                     /* (L,B,E)  step-major LSTM input  */
    float* xg;                    /* (L,B,4H) */
    float* gates_act;             /* (L,B,4H) */
    float* h_all;                 /* (L+1,B,H) */
    float* c_all;                 /* (L+1,B,H) */
    float* hout;                  /* (B,L,H)  */
    float* gates_pre;             /* (B,4H) scratch */
    /* backward */
    const float* d_outputs;       /* (B,L,V) */
    float *d_w_ih, *d_w_hh, *d_b, *d_lin_w, *d_lin_b;   /* d_b = d_b_ih = d_b_hh */
    void* d_emb_w;                /* (V,E) or NULL */
    float* d_img_features;        /* (B,E) or NULL */
    float* d_hout;                /* (B,L,H) */
    float* dg;                    /* (L,B,4H) */
    float* dh;                    /* (B,H) */
    float* dc;                    /* (B,H) */
    float* d_x;                   /* (L,B,E) */
    /* ICD_PREC_BF16 only: arena for the bf16 operand copies, shared by fwd and bwd of the same step */
    void* tc_ws; int64_t tc_ws_bytes;   /* >= icd_baseline_decoder_ws_bytes(desc) */
} icd_base_desc_t;

ICD_API int64_t icd_baseline_decoder_ws_bytes(const icd_base_desc_t* d);
ICD_API int icd_baseline_decoder_fwd(const icd_base_desc_t* d, void* stream);
ICD_API int icd_baseline_decoder_bwd(const icd_base_desc_t* d, void* stream);

/* ------------------------------------------------------------------------------------------------
 * The recurrence of a 1-layer nn.LSTM over L steps from a zero state (models/baseline.py:106) on its own — K8, ONE
 * persistent cooperative kernel per direction (W_hh slices resident in shared memory for all steps, tcgen05 contraction of
 * the step's activation, LSTM cell math in the epilogue, a grid barrier between steps).  The caller hoists the input
 * contraction: xg (L,B,4H) = x W_ih^T + b_ih + b_hh.  Gate order i,f,g,o.  bf16 operands, fp32 accumulation / state.
 *   forward : gates_act (L,B,4H), c_all / h_all (L+1,B,H) [block 0 = the zero state, written here], hout (B,L,H),
 *             h16 ((L+1)*B, H) bf16 scratch (h_t as the next step's operand), hout16 (B*L, H) bf16 copy of hout or NULL
 *   backward: d_hout (B,L,H) in; gates_act, c_all from the forward; dc_ws (B,H) scratch; dg (L,B,4H) fp32 and
 *             dg16 (L*B, 4H) bf16 out — d(loss)/d(gates_pre), the operand of every weight / input gradient contraction
 *   barrier_ws: >= 4 bytes of device memory (the grid-barrier counter).
 * icd_lstm_seq_shape_ok: the pure shape rules, no device needed: L >= 1, H a multiple of 16, H/4 <= 148 (one forward CTA per
 * SM), B <= 512 (4 row tiles of 128), and room for the resident weight slice.
 * icd_lstm_seq_supported: 1 if (B, L, H) passes the shape rules AND both grids are co-resident on the current device at the
 * shared memory they launch with (forward: H/4 CTAs; backward: H/16 clusters of 4 CTAs), as the occupancy calculator says;
 * cached per (row tiles, H).  Otherwise callers keep a per-step launch chain (icd_baseline_decoder_fwd does that by itself).
 * icd_lstm_seq_residency: diagnostic, launches nothing — how many forward CTAs (blocks per SM x SMs) and how many
 * backward 4-CTA clusters the device can hold at once at the shared memory (B, H) launches with.
 * ---------------------------------------------------------------------------------------------- */
ICD_API int icd_lstm_seq_shape_ok(int B, int L, int H);
ICD_API int icd_lstm_seq_supported(int B, int L, int H);
ICD_API int icd_lstm_seq_residency(int B, int H, int* fwd_ctas, int* bwd_clusters);
/* diagnostic: how the last backward recurrence was launched — 0 not yet, 1 cooperative + 4-CTA clusters (co-residency
 * guaranteed by the driver), 2 plain cluster launch (a driver that refuses the combination; only for a grid the occupancy
 * query found co-resident) */
ICD_API int icd_lstm_seq_bwd_launch_mode(void);
ICD_API int icd_lstm_seq_fwd(int B, int L, int H, const float* w_hh, const float* xg, float* gates_act, float* c_all,
                     float* h_all, float* hout, void* h16, void* hout16, void* barrier_ws, void* stream);
ICD_API int icd_lstm_seq_bwd(int B, int L, int H, const float* w_hh, const float* d_hout, const float* gates_act,
                     const float* c_all, float* dc_ws, float* dg, void* dg16, void* barrier_ws, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Batched beam search (gen_captions.py:16-131; state machine in SURVEY.md Appendix C), n_img
 * independent images x k beam slots, fully device-side (no per-step host sync).
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t n_img, k, max_steps;  /* loop body runs for step = 1 .. max_steps+1 (gen_captions.py:119) */
    int32_t P, C, A, D, E, V;
    int32_t precision, emb_is_f64;
    int32_t start_id, end_id;
    const float* enc;             /* (n_img,P,C) */
    const float *enc_att_w, *enc_att_b, *dec_att_w, *dec_att_b, *full_att_w, *full_att_b;
    const float *w_ih, *w_hh, *b_ih, *b_hh;
    const float *h_lin_w, *h_lin_b, *c_lin_w, *c_lin_b;
    const float *f_beta_w, *f_beta_b, *fc_w, *fc_b;
    const void* emb_w;
    /* results (device) */
    int32_t* out_len;             /* (n_img)   length of best completed caption incl. <start>/<end>; 0 => none completed */
    int32_t* out_seq;             /* (n_img, max_steps+2) */
    float* out_score;             /* (n_img)   raw summed log-prob of the winner */
    float* out_alpha;             /* (n_img, max_steps+2, P) frame 0 = ones; may be NULL */
    int32_t* trace_words;         /* (max_steps+1, n_img, k) next-word ids per step, -1 = empty slot; may be NULL */
    /* workspace (device) */
    void* ws; int64_t ws_bytes;   /* >= icd_beam_search_ws_bytes(desc) */
} icd_beam_desc_t;

ICD_API int64_t icd_beam_search_ws_bytes(const icd_beam_desc_t* d);
ICD_API int icd_beam_search(const icd_beam_desc_t* d, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Batched beam search for the BaselineDecoder (models/baseline.py:81-111 run autoregressively; the reference has no
 * generation function for this decoder).  The state machine is that of icd_beam_search; the decoder step is the
 * baseline's: the image feature is LSTM step 0 from the zero state (its logits are not scored, position 0 of every
 * caption is <start>), then steps 1 .. max_steps+1 feed emb(previous word), with <start> at step 1, through one LSTM step
 * (gate order i,f,g,o, b_ih + b_hh) and the vocabulary layer.  k = 1 is greedy decoding.  An fp64 embedding table is
 * cast to fp32 once per call (what the forward does with its rows, models/baseline.py:101).
 * precision: ICD_PREC_FP32 or ICD_PREC_FP32X3 (identical captions need fp32-grade logits).
 * Every argument is validated before the first CUDA call.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t n_img, k, max_steps;  /* k in 1..8, n_img*k <= 65535; loop body runs for step = 1 .. max_steps+1 */
    int32_t E, H, V;              /* E, H multiples of 4; V >= k */
    int32_t precision, emb_is_f64;
    int32_t start_id, end_id;
    const float* img_features;    /* (n_img,E) fp32 */
    const void* emb_w;            /* (V,E) fp32 or fp64 */
    const float *w_ih, *w_hh, *b_ih, *b_hh;   /* (4H,E) (4H,H) (4H) (4H) */
    const float *lin_w, *lin_b;   /* (V,H) (V) */
    /* results (device), as in icd_beam_desc_t */
    int32_t* out_len;             /* (n_img)   length of best completed caption incl. <start>/<end>; 0 => none completed */
    int32_t* out_seq;             /* (n_img, max_steps+2) */
    float* out_score;             /* (n_img)   raw summed log-prob of the winner (steps >= 1) */
    int32_t* trace_words;         /* (max_steps+1, n_img, k) next-word ids per step, -1 = empty slot; may be NULL */
    /* workspace (device) */
    void* ws; int64_t ws_bytes;   /* >= icd_baseline_beam_search_ws_bytes(desc) */
} icd_base_beam_desc_t;

ICD_API int64_t icd_baseline_beam_search_ws_bytes(const icd_base_beam_desc_t* d);   /* -1: shape refused (see the error string) */
ICD_API int icd_baseline_beam_search(const icd_base_beam_desc_t* d, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Seeded, batched caption sampling (temperature, top-k) for the attention decoder (icd_sample_captions) and the
 * BaselineDecoder (icd_baseline_sample_captions).  n_img images x m samples, fully device-side (no per-step host sync).
 * Sample j of image i starts from the decoder's start state exactly as the beam searches above do, and runs steps
 * s = 1 .. max_steps+1; step 1 runs one row per image and draws all m tokens from it.  At each step, with the fp32-grade
 * logits l (V):
 *   lp  = log_softmax(l) at temperature 1 over the full vocabulary (the quantity the beam score sums);
 *   candidates: every token when top_k == 0 (or top_k == V), else the top_k largest l (ties: the lower token id first);
 *   temperature == 0: the token is argmax l (lowest id on a tie);
 *   else Gumbel-max: the candidate with the largest key_v = l_v / temperature + g_v (IEEE fp32 division; lower id on a tie),
 *     g_v = -log(-log(u_v)), u_v = ((bits >> 8) + 0.5) * 2^-24 in (0, 1), bits = word v % 4 of
 *     Philox4x32-10(counter = (v / 4, s, img_base + i, sample_base + j), key = (seed lo, seed hi)).  In fp32, -log(u) is
 *     logf of the exact u below 1/2 and -log1pf(-(1 - u)) (exact 1 - u) above, so it never rounds to 0.
 *   The noise depends on (seed, image, sample, step, token) only: not on chunking, compaction or which images share a call.
 * A sample that draws end_id ends: len = its length incl. <start> and <end>, ended = 1.  One that has not ended after step
 * max_steps+1 keeps its truncated caption: len = max_steps+2, ended = 0.  score = sum of lp[token] over steps 1 .. len-1,
 * fp32 in step order; logp[i, j, s-1] holds each term.  seq beyond len and logp beyond len-1 are 0; every entry is written.
 * m in 1..8, n_img*m <= 65535, temperature finite and >= 0, top_k in 0..V, precision ICD_PREC_FP32 or ICD_PREC_FP32X3.
 * Every argument is validated before the first CUDA call; the size queries return -1 for a refused shape.  The workspace
 * holds one step of state (no per-step history): it does not grow with max_steps.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t n_img, m, max_steps;  /* m samples per image; steps 1 .. max_steps+1 */
    int32_t P, C, A, D, E, V;
    int32_t precision, emb_is_f64;
    int32_t start_id, end_id;
    int32_t top_k;                /* 0 = the whole vocabulary */
    int32_t img_base, sample_base;   /* global index of image 0 and of sample 0 of this call (noise counters) */
    float temperature;            /* 0 = greedy */
    uint64_t seed;
    /* inputs and weights, as in icd_beam_desc_t */
    const float* enc;             /* (n_img,P,C) */
    const float *enc_att_w, *enc_att_b, *dec_att_w, *dec_att_b, *full_att_w, *full_att_b;
    const float *w_ih, *w_hh, *b_ih, *b_hh;
    const float *h_lin_w, *h_lin_b, *c_lin_w, *c_lin_b;
    const float *f_beta_w, *f_beta_b, *fc_w, *fc_b;
    const void* emb_w;
    /* results (device) */
    int32_t* out_seq;             /* (n_img, m, max_steps+2), [.., 0] = <start> */
    int32_t* out_len;             /* (n_img, m) */
    uint8_t* out_ended;           /* (n_img, m) 1 = drew <end> */
    float* out_score;             /* (n_img, m) */
    float* out_logp;              /* (n_img, m, max_steps+1); may be NULL */
    /* workspace (device) */
    void* ws; int64_t ws_bytes;   /* >= icd_sample_captions_ws_bytes(desc) */
} icd_sample_desc_t;

ICD_API int64_t icd_sample_captions_ws_bytes(const icd_sample_desc_t* d);     /* -1: shape refused (see the error string) */
ICD_API int icd_sample_captions(const icd_sample_desc_t* d, void* stream);

typedef struct {
    int32_t n_img, m, max_steps;
    int32_t E, H, V;
    int32_t precision, emb_is_f64;
    int32_t start_id, end_id;
    int32_t top_k;
    int32_t img_base, sample_base;
    float temperature;
    uint64_t seed;
    /* inputs and weights, as in icd_base_beam_desc_t */
    const float* img_features;    /* (n_img,E) fp32 */
    const void* emb_w;            /* (V,E) fp32 or fp64 */
    const float *w_ih, *w_hh, *b_ih, *b_hh;
    const float *lin_w, *lin_b;
    /* results (device), as in icd_sample_desc_t */
    int32_t* out_seq;
    int32_t* out_len;
    uint8_t* out_ended;
    float* out_score;
    float* out_logp;
    void* ws; int64_t ws_bytes;   /* >= icd_baseline_sample_captions_ws_bytes(desc) */
} icd_base_sample_desc_t;

ICD_API int64_t icd_baseline_sample_captions_ws_bytes(const icd_base_sample_desc_t* d);
ICD_API int icd_baseline_sample_captions(const icd_base_sample_desc_t* d, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Optimiser glue: element-wise gradient clamp to +-grad_clip (train_utils.py:2-12) fused with the
 * torch.optim.Adam(lr, betas=(0.9,0.999), eps=1e-8, weight_decay=0) update (models/attention.py:352-355,
 * 423-428) over a flat fp32 buffer; grad_scale multiplies the gradient first (1/world_size after all-reduce).
 * step is the 1-based Adam step count.
 * ---------------------------------------------------------------------------------------------- */
ICD_API int icd_clip_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq,
                       int64_t n, float grad_scale, float grad_clip, float lr, float beta1, float beta2,
                       float eps, int32_t step, void* stream);

/* Keep-mask generator for nn.Dropout (Philox4x32-10, counter-based): out[i] = uniform > p ? 1 : 0 */
ICD_API int icd_dropout_mask(uint8_t* out, int64_t n, float p, uint64_t seed, uint64_t offset, void* stream);

/* Token-level loss glue (models/attention.py:401-411; models/baseline.py:224-225) fused:
 * forward : row_loss[r] = logsumexp(logits[r,:]) - logits[r, targets[r]], lse[r] saved; targets[r] < 0 => row ignored
 *           (row_loss 0) — these are the rows pack_padded_sequence drops / ignore_index skips;
 * backward: d_logits[r,v] = (exp(logits[r,v] - lse[r]) - [v == targets[r]]) * inv_count * (*upstream)  (0 for ignored
 *           rows); `upstream` is a DEVICE scalar (d loss, read by the kernel: no host sync); d_logits16 is an optional
 *           bf16 copy with row stride ld16 (multiple of 8) — the A operand of the vocabulary-layer backward contractions.
 */
ICD_API int icd_cross_entropy_fwd(int64_t R, int V, const float* logits, const int64_t* targets,
                          float* row_loss, float* lse, void* stream);
ICD_API int icd_cross_entropy_bwd(int64_t R, int V, const float* logits, const int64_t* targets, const float* lse,
                          const float* upstream, float inv_count, float* d_logits, void* d_logits16, int64_t ld16,
                          void* stream);
/* training fast path of the bf16 tier: forward AND the bf16 gradient (exp(x - lse) - onehot) * inv_count in ONE pass over the
 * logits (each row is parked in shared memory between the two; V <= ~50 000) — the upstream gradient of the loss is applied
 * afterwards with icd_scale_bf16_by_device_scalar (x16[i] *= *scale; returns at once when *scale == 1). */
ICD_API int icd_cross_entropy_fwd_grad16(int64_t R, int V, const float* logits, const int64_t* targets, float inv_count,
                          float* row_loss, float* lse, void* d_logits16, int64_t ld16, void* stream);
ICD_API int icd_scale_bf16_by_device_scalar(void* x16, int64_t n, const float* scale, void* stream);
/* Per-row weighted gradients (sequence-level training: a reward advantage per caption token): the same kernels with the
 * gradient of row r also multiplied by weights[r] (R fp32 values on the device, any sign, 0 allowed):
 *   bwd      : d_logits[r,v] = (exp(logits[r,v] - lse[r]) - [v == targets[r]]) * ((inv_count * (*upstream)) * weights[r])
 *   fwd_grad16: the bf16 gradient is (exp(x - lse) - onehot) * (inv_count * weights[r]); row_loss and lse stay unweighted.
 * weights == 1 reproduces the unweighted results bit for bit; a row of weight 0 is written as zeros; rows with targets[r] < 0
 * are zero as before.  Every argument (null weights, ld16, V of the one-pass kernel) is checked before any CUDA call. */
ICD_API int icd_weighted_cross_entropy_bwd(int64_t R, int V, const float* logits, const int64_t* targets, const float* lse,
                          const float* upstream, float inv_count, const float* weights, float* d_logits, void* d_logits16,
                          int64_t ld16, void* stream);
ICD_API int icd_weighted_cross_entropy_fwd_grad16(int64_t R, int V, const float* logits, const int64_t* targets,
                          float inv_count, const float* weights, float* row_loss, float* lse, void* d_logits16, int64_t ld16,
                          void* stream);

/* Doubly stochastic attention regulariser (models/attention.py:413-414): reg = mean_{b,p} (alpha_c - sum_t alphas[b,t,p])^2.
 * forward : resid[b,p] = alpha_c - sum_t alphas[b,t,p] (saved for the backward); reg[0] = the mean (summed in a fixed order:
 *           per-block partials in `partial`, ceil(B*P/256) floats, then one reduction);
 * backward: d_alphas[b,t,p] = -2 * resid[b,p] / (B*P) * (*upstream) for every t; `upstream` is a DEVICE scalar. */
ICD_API int icd_alpha_regulariser_fwd(int B, int T, int P, const float* alphas, float alpha_c, float* resid,
                              float* partial, float* reg, void* stream);
ICD_API int icd_alpha_regulariser_bwd(int B, int T, int P, const float* resid, const float* upstream, float* d_alphas,
                              void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ICD_B200_H */
