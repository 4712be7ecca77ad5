// AttentionDecoder.forward / backward (models/attention.py:218-284), teacher forced, as one stream-ordered
// sequence of kernels issued from a single C-ABI call (no Python, no host sync between steps).
//
// Restructuring relative to the reference (SURVEY.md 7.2), numerically the same operations:
//   * enc_att(encoder_out) is time-invariant: computed once per batch, not once per step (:54);
//   * the embedding half of the LSTMCell input contraction, emb_t * W_ih[:, :E]^T + b_ih + b_hh, is hoisted
//     over all steps; only awe_t * W_ih[:, E:]^T stays in the loop (:273-278; the fp64 cat round-trip is exact);
//   * dec_att(h), f_beta(h) and h * W_hh^T share their input: one contraction with [W_dec; W_fbeta; W_hh] (:55,270,277);
//   * fc over dropout(h_t) does not feed back under teacher forcing: one contraction after the loop (:279-280),
//     written straight into predictions (B,T,V) with rows >= batch_size_t forced to exactly 0 (:253).
// Backward is the hand-derived adjoint of the same graph (BPTT), with all weight-gradient contractions hoisted
// out of the loop (one per weight over the T*B stacked rows).
#include "common.cuh"
#include <algorithm>

namespace {

struct BtPack { int v[ICD_MAX_STEPS]; };

__global__ void row_valid_kernel(int B, int T, const BtPack bt, unsigned char* __restrict__ valid) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * T) return;
    const int b = i / T, t = i % T;
    valid[i] = (b < bt.v[t]) ? 1 : 0;
}

int check_common(const icd_att_desc_t* d) {
    ICD_CHECK_ARG(d != nullptr, "attention_decoder: null descriptor");
    ICD_CHECK_ARG(d->B > 0 && d->T > 0 && d->T <= ICD_MAX_STEPS, "attention_decoder: B=%d T=%d out of range", d->B, d->T);
    ICD_CHECK_ARG(d->L >= d->T, "attention_decoder: captions need at least T columns (L=%d T=%d)", d->L, d->T);
    ICD_CHECK_ARG(d->A % 4 == 0 && d->C % 4 == 0 && d->D % 4 == 0 && d->E % 4 == 0,
                  "attention_decoder: A,C,D,E must be multiples of 4 (A=%d C=%d D=%d E=%d)", d->A, d->C, d->D, d->E);
    for (int t = 0; t < d->T; ++t) {
        ICD_CHECK_ARG(d->bt_host[t] >= 0 && d->bt_host[t] <= d->B, "attention_decoder: bt[%d]=%d out of range", t, d->bt_host[t]);
        ICD_CHECK_ARG(t == 0 || d->bt_host[t] <= d->bt_host[t - 1], "attention_decoder: bt must be non-increasing");
    }
    return 0;
}

}  // namespace

// captions that share images (icd_att_index_t): the index is checked here, its device contents are the caller's
int icd_check_att_index(const icd_att_desc_t* d, const icd_att_index_t* ix) {
    if (!ix) return 0;
    ICD_CHECK_ARG(ix->n_img > 0 && ix->n_img <= 65535, "attention_decoder: n_img=%d out of range (1..65535)", ix->n_img);
    ICD_CHECK_ARG(ix->img_index && ix->img_row_ptr && ix->img_rows, "attention_decoder: the image index needs img_index, img_row_ptr and img_rows");
    ICD_CHECK_ARG(d->d_enc == nullptr || d->d_awe_all != nullptr, "attention_decoder: d_enc needs the d_awe_all scratch buffer");
    return 0;
}

extern "C" int icd_init_hidden_state(int B, int P, int C, int D, int precision, const float* enc,
                                     const float* h_lin_w, const float* h_lin_b,
                                     const float* c_lin_w, const float* c_lin_b,
                                     float* mean_enc, float* h, float* c, void* stream) {
    cudaStream_t s = icd_stream(stream);
    ICD_CHECK_ARG(precision == ICD_PREC_FP32 || precision == ICD_PREC_FP32X3, "init_hidden_state: precision %d not supported here", precision);
    // mean over pixels (:161) — same streaming kernel as the attention-weighted sum, uniform weights
    ICD_TRY(icd_weighted_pixel_sum(B, P, C, nullptr, enc, nullptr, 0, nullptr, 0, mean_enc, nullptr, nullptr, s));
    ICD_TRY(icd_gemm_simple(precision, mean_enc, C, 1, h_lin_w, C, 1, h, D, B, D, C, h_lin_b, nullptr,
                            nullptr, 0, nullptr, 0, nullptr, 0.f, s));                       // :162
    ICD_TRY(icd_gemm_simple(precision, mean_enc, C, 1, c_lin_w, C, 1, c, D, B, D, C, c_lin_b, nullptr,
                            nullptr, 0, nullptr, 0, nullptr, 0.f, s));                       // :163
    return 0;
}

int64_t icd_att_tc_ws_bytes(const icd_att_desc_t* d, int n_img);             // decoder_loop_bf16.cu
int icd_attention_decoder_fwd_bf16(const icd_att_desc_t* d, const icd_att_index_t* ix, cudaStream_t s);
int icd_attention_decoder_bwd_bf16(const icd_att_desc_t* d, const icd_att_index_t* ix, cudaStream_t s);

// fp32-grade tier: the splits of the two weight matrices every step of the time loop reads ([W_dec; W_fbeta; W_hh] and
// W_ih[:, E:], K-major in the forward loop, MN-major in the BPTT) are made once per call and kept at the tail of tc_ws
// (they were 26 % of the tier's train step when every contraction re-split them: profiles/r02_fp32x3_split_cache.txt)
static int64_t x3_cache_bytes(const icd_att_desc_t* d) {
    if (d->precision != ICD_PREC_FP32X3) return 0;
    const int64_t NZ = (int64_t)d->A + d->C + 4 * (int64_t)d->D;
    return icd_x3_split_bytes(NZ, d->D) + icd_x3_split_bytes(4 * (int64_t)d->D, d->C) + 512;
}

static int64_t ws_bytes(const icd_att_desc_t* d, const icd_att_index_t* ix) {
    if (!d) return 0;
    const int64_t n_img = ix ? ix->n_img : d->B;        // the rows of the per-image contractions are n_img * P pixel rows
    if (d->precision == ICD_PREC_BF16) return icd_att_tc_ws_bytes(d, (int)n_img);
    if (d->precision != ICD_PREC_FP32X3) return 0;
    // fp32-grade tensor-core tier: every contraction splits its two operands on the fly (gemm_tc.cu); size for the largest
    const int64_t B = d->B, T = d->T, P = d->P, C = d->C, A = d->A, D = d->D, E = d->E, V = d->V, NZ = A + C + 4 * D, TB = T * B;
    const int64_t NP = n_img * P;
    const int64_t shapes[][3] = {
        {NP, A, C}, {B, D, C}, {TB, 4 * D, E}, {B, NZ, D}, {B, 4 * D, C}, {B * T, V, D},
        {B * T, D, V}, {V, D, B * T}, {B, C, 4 * D}, {B, D, NZ}, {D, C, B}, {NZ, D, TB}, {4 * D, E, TB}, {4 * D, C, TB},
        {TB, E, 4 * D}, {A, C, NP}, {B, C, D}, {NP, C, A}};
    int64_t need = 0;
    for (const auto& sh : shapes) need = std::max(need, icd_gemm_ws_bytes((int)sh[0], (int)sh[1], (int)sh[2], ICD_PREC_FP32X3));
    return need + x3_cache_bytes(d);
}

extern "C" int64_t icd_attention_decoder_ws_bytes(const icd_att_desc_t* d) { return ws_bytes(d, nullptr); }
extern "C" int64_t icd_attention_decoder_ws_bytes_indexed(const icd_att_desc_t* d, const icd_att_index_t* ix) { return ws_bytes(d, ix); }

static int decoder_fwd(const icd_att_desc_t* d, const icd_att_index_t* ix, void* stream) {
    ICD_TRY(check_common(d));
    ICD_TRY(icd_check_att_index(d, ix));
    cudaStream_t s = icd_stream(stream);
    if (d->precision == ICD_PREC_BF16) return icd_attention_decoder_fwd_bf16(d, ix, s);
    ICD_CHECK_ARG(d->precision == ICD_PREC_FP32 || d->precision == ICD_PREC_FP32X3, "attention_decoder: unknown precision %d", d->precision);
    ICD_CHECK_ARG(d->enc != nullptr, "attention_decoder(fp32): enc is required (bf16-stored features need ICD_PREC_BF16)");
    IcdSimpleWsScope ws_scope(d->tc_ws, d->tc_ws_bytes, x3_cache_bytes(d));   // ICD_PREC_FP32X3: operand splits live in the caller's arena
    icd_x3_cache_mark(d->w_cat);
    icd_x3_cache_mark(d->w_ih + d->E);
    const int B = d->B, T = d->T, P = d->P, C = d->C, A = d->A, D = d->D, E = d->E, V = d->V;
    const int NZ = A + C + 4 * D;
    const int prec = d->precision;
    const long long BD = (long long)B * D;
    const int n_img = ix ? ix->n_img : B;
    const int32_t* img_index = ix ? ix->img_index : nullptr;

    BtPack pack;
    for (int t = 0; t < ICD_MAX_STEPS; ++t) pack.v[t] = t < T ? d->bt_host[t] : 0;
    row_valid_kernel<<<(B * T + 255) / 256, 256, 0, s>>>(B, T, pack, d->row_valid);
    ICD_LAUNCH_CHECK();

    // buffers whose inactive rows are read later (as zero contributions) must not hold NaN garbage
    ICD_CUDA(cudaMemsetAsync(d->alphas, 0, sizeof(float) * (size_t)B * T * P, s));          // :257
    ICD_CUDA(cudaMemsetAsync(d->hdrop, 0, sizeof(float) * (size_t)B * T * D, s));
    if (d->bt_host[T - 1] < B) {
        ICD_CUDA(cudaMemsetAsync(d->h_all, 0, sizeof(float) * (size_t)(T + 1) * BD, s));
        ICD_CUDA(cudaMemsetAsync(d->c_all, 0, sizeof(float) * (size_t)(T + 1) * BD, s));
        ICD_CUDA(cudaMemsetAsync(d->gated, 0, sizeof(float) * (size_t)T * B * C, s));
        ICD_CUDA(cudaMemsetAsync(d->z, 0, sizeof(float) * (size_t)T * B * NZ, s));
    }

    // [W_dec; W_fbeta; W_hh] and its bias (b_hh rides with the hoisted embedding term instead)
    ICD_CUDA(cudaMemcpyAsync(d->w_cat, d->dec_att_w, sizeof(float) * (size_t)A * D, cudaMemcpyDeviceToDevice, s));
    ICD_CUDA(cudaMemcpyAsync(d->w_cat + (size_t)A * D, d->f_beta_w, sizeof(float) * (size_t)C * D, cudaMemcpyDeviceToDevice, s));
    ICD_CUDA(cudaMemcpyAsync(d->w_cat + (size_t)(A + C) * D, d->w_hh, sizeof(float) * (size_t)4 * D * D, cudaMemcpyDeviceToDevice, s));
    ICD_CUDA(cudaMemcpyAsync(d->b_cat, d->dec_att_b, sizeof(float) * A, cudaMemcpyDeviceToDevice, s));
    ICD_CUDA(cudaMemcpyAsync(d->b_cat + A, d->f_beta_b, sizeof(float) * C, cudaMemcpyDeviceToDevice, s));
    ICD_CUDA(cudaMemsetAsync(d->b_cat + A + C, 0, sizeof(float) * 4 * D, s));

    // K1: att_enc = enc_att(encoder_out), once per batch (:54)
    ICD_TRY(icd_gemm_simple(prec, d->enc, C, 1, d->enc_att_w, C, 1, d->att_enc, A, n_img * P, A, C,
                            d->enc_att_b, nullptr, nullptr, 0, nullptr, 0, nullptr, 0.f, s));
    // K7: init_hidden_state (:250); with an image index the pixel mean is formed once per image and written to its rows
    if (ix) {
        ICD_TRY(icd_weighted_pixel_sum(n_img, P, C, nullptr, d->enc, nullptr, 0, nullptr, 0, d->mean_enc, nullptr, nullptr, s,
                                       ix->img_row_ptr, ix->img_rows));
        ICD_TRY(icd_gemm_simple(prec, d->mean_enc, C, 1, d->h_lin_w, C, 1, d->h_all, D, B, D, C, d->h_lin_b, nullptr,
                                nullptr, 0, nullptr, 0, nullptr, 0.f, s));
        ICD_TRY(icd_gemm_simple(prec, d->mean_enc, C, 1, d->c_lin_w, C, 1, d->c_all, D, B, D, C, d->c_lin_b, nullptr,
                                nullptr, 0, nullptr, 0, nullptr, 0.f, s));
    } else
        ICD_TRY(icd_init_hidden_state(B, P, C, D, prec, d->enc, d->h_lin_w, d->h_lin_b, d->c_lin_w, d->c_lin_b,
                                      d->mean_enc, d->h_all, d->c_all, s));
    // K5: embedding lookup (:247) + hoisted input contraction
    // emb_w == NULL: emb_x (T,B,E) was filled by the caller with pre-computed embeddings (the reference's use_bert branch,
    // models/attention.py:242-244: (B,L,768) BERT vectors instead of the table lookup); they carry no gradient
    if (d->emb_w) ICD_TRY(icd_embed_gather(d->emb_w, d->emb_is_f64, d->captions, B, d->L, T, E, V, d->emb_x, s));
    ICD_TRY(icd_gemm_simple(prec, d->emb_x, E, 1, d->w_ih, E + C, 1, d->xg, 4 * D, T * B, 4 * D, E,
                            d->b_ih, d->b_hh, nullptr, 0, nullptr, 0, nullptr, 0.f, s));

    for (int t = 0; t < T; ++t) {                                                            // :260
        const int bt = d->bt_host[t];                                                        // :261
        if (bt == 0) break;
        const float* h_prev = d->h_all + (size_t)t * BD;
        const float* c_prev = d->c_all + (size_t)t * BD;
        float* zt = d->z + (size_t)t * B * NZ;
        // K2: z = h * [W_dec; W_fbeta; W_hh]^T + [b_dec; b_fbeta; 0]
        ICD_TRY(icd_gemm_simple(prec, h_prev, D, 1, d->w_cat, D, 1, zt, NZ, bt, NZ, D, d->b_cat, nullptr,
                                nullptr, 0, nullptr, 0, nullptr, 0.f, s));
        // K3: attention + gate (:267-271); alpha goes straight into attention_weights[:bt, t, :] (:281)
        ICD_TRY(icd_attention_step_fwd(bt, P, C, A, img_index, d->enc, d->att_enc, zt, NZ,
                                       d->full_att_w, d->full_att_b, zt + A, NZ,
                                       d->alphas + (size_t)t * P, (int64_t)T * P,
                                       d->awe_raw + (size_t)t * B * C, d->gate + (size_t)t * B * C,
                                       d->gated + (size_t)t * B * C, s));
        // K4: gates = xg_t + gated * W_ih[:, E:]^T + z_hh  (:277)
        ICD_TRY(icd_gemm_simple(prec, d->gated + (size_t)t * B * C, C, 1, d->w_ih + E, E + C, 1,
                                d->gates_pre, 4 * D, bt, 4 * D, C, nullptr, nullptr,
                                d->xg + (size_t)t * B * 4 * D, 4 * D, zt + A + C, NZ, nullptr, 0.f, s));
        //     LSTMCell pointwise (:277-278) + dropout on the fc input (:279)
        ICD_TRY(icd_lstm_pointwise_fwd(bt, D, d->gates_pre, c_prev, d->gates_act + (size_t)t * B * 4 * D,
                                       d->c_all + (size_t)(t + 1) * BD, d->h_all + (size_t)(t + 1) * BD,
                                       d->hdrop + (size_t)t * D, (int64_t)T * D,
                                       d->drop_mask ? d->drop_mask + (size_t)t * BD : nullptr, d->drop_scale, s));
    }
    // K6: predictions = fc(dropout(h)) for every (b,t) at once; inactive rows exactly 0 (:253,279-280)
    ICD_TRY(icd_gemm_simple(prec, d->hdrop, D, 1, d->fc_w, D, 1, d->predictions, V, B * T, V, D, d->fc_b, nullptr,
                            nullptr, 0, nullptr, 0, d->row_valid, 0.f, s));
    return 0;
}

extern "C" int icd_attention_decoder_fwd(const icd_att_desc_t* d, void* stream) { return decoder_fwd(d, nullptr, stream); }
extern "C" int icd_attention_decoder_fwd_indexed(const icd_att_desc_t* d, const icd_att_index_t* ix, void* stream) {
    return decoder_fwd(d, ix, stream);
}

static int decoder_bwd(const icd_att_desc_t* d, const icd_att_index_t* ix, void* stream) {
    ICD_TRY(check_common(d));
    ICD_TRY(icd_check_att_index(d, ix));
    cudaStream_t s = icd_stream(stream);
    if (d->precision == ICD_PREC_BF16) return icd_attention_decoder_bwd_bf16(d, ix, s);
    IcdSimpleWsScope ws_scope(d->tc_ws, d->tc_ws_bytes, x3_cache_bytes(d));
    icd_x3_cache_mark(d->w_cat);
    icd_x3_cache_mark(d->w_ih + d->E);
    const int B = d->B, T = d->T, P = d->P, C = d->C, A = d->A, D = d->D, E = d->E, V = d->V;
    const int NZ = A + C + 4 * D;
    const int prec = d->precision;
    const long long BD = (long long)B * D;
    const int TB = T * B;
    const int n_img = ix ? ix->n_img : B;
    const int32_t* img_index = ix ? ix->img_index : nullptr;

    ICD_CUDA(cudaMemsetAsync(d->dz, 0, sizeof(float) * (size_t)TB * NZ, s));
    ICD_CUDA(cudaMemsetAsync(d->d_e, 0, sizeof(float) * (size_t)B * T * P, s));
    ICD_CUDA(cudaMemsetAsync(d->dh, 0, sizeof(float) * (size_t)BD, s));
    ICD_CUDA(cudaMemsetAsync(d->dc, 0, sizeof(float) * (size_t)BD, s));

    // ---- fc (:279): d_hdrop = dY * W_fc ; dW_fc = dY^T * hdrop ; db_fc = masked column sum of dY ----
    ICD_TRY(icd_gemm_simple(prec, d->d_predictions, V, 1, d->fc_w, 1, D, d->d_hdrop, D, B * T, D, V,
                            nullptr, nullptr, nullptr, 0, nullptr, 0, nullptr, 0.f, s));
    ICD_TRY(icd_gemm_simple(prec, d->d_predictions, 1, V, d->hdrop, 1, D, d->d_fc_w, D, V, D, B * T,
                            nullptr, nullptr, nullptr, 0, nullptr, 0, nullptr, 0.f, s, ICD_GEMM_ALLOW_SPLITK));
    ICD_TRY(icd_colsum(d->d_predictions, V, (int64_t)B * T, V, d->row_valid, d->d_fc_b, s));
    if (d->ev_fc_ready) ICD_CUDA(cudaEventRecord(reinterpret_cast<cudaEvent_t>(d->ev_fc_ready), s));

    // ---- BPTT ----
    for (int t = T - 1; t >= 0; --t) {
        const int bt = d->bt_host[t];
        if (bt == 0) continue;
        float* dzt = d->dz + (size_t)t * B * NZ;
        const float* zt = d->z + (size_t)t * B * NZ;
        // LSTMCell pointwise adjoint; dh carries d(loss)/d(h_{t+1}) from step t+1, fc path added here
        ICD_TRY(icd_lstm_pointwise_bwd(bt, D, d->dh, d->d_hdrop + (size_t)t * D, (int64_t)T * D,
                                       d->drop_mask ? d->drop_mask + (size_t)t * BD : nullptr, d->drop_scale,
                                       d->dc, d->gates_act + (size_t)t * B * 4 * D,
                                       d->c_all + (size_t)t * BD, d->c_all + (size_t)(t + 1) * BD,
                                       dzt + A + C, NZ, s));
        // d_gated = dgates * W_ih[:, E:]
        ICD_TRY(icd_gemm_simple(prec, dzt + A + C, NZ, 1, d->w_ih + E, 1, E + C, d->d_gated, C, bt, C, 4 * D,
                                nullptr, nullptr, nullptr, 0, nullptr, 0, nullptr, 0.f, s));
        // attention + gate adjoint -> dz[:, 0:A] (d att_dec), dz[:, A:A+C] (d fbeta_pre), d_e saved
        ICD_TRY(icd_attention_step_bwd_idx(bt, P, C, A, img_index, d->enc, d->att_enc, zt, NZ, d->full_att_w,
                                       d->alphas + (size_t)t * P, (int64_t)T * P,
                                       d->d_alphas ? d->d_alphas + (size_t)t * P : nullptr, (int64_t)T * P,
                                       d->gate + (size_t)t * B * C, d->awe_raw + (size_t)t * B * C, d->d_gated,
                                       dzt, NZ, dzt + A, NZ, d->d_e + (size_t)t * P, (int64_t)T * P,
                                       d->d_enc ? d->d_awe_all + (size_t)t * B * C : nullptr, s));
        // dh_{t} = dz * [W_dec; W_fbeta; W_hh]
        ICD_TRY(icd_gemm_simple(prec, dzt, NZ, 1, d->w_cat, 1, D, d->dh, D, bt, D, NZ,
                                nullptr, nullptr, nullptr, 0, nullptr, 0, nullptr, 0.f, s));
    }

    // ---- init_hidden_state (:161-163): dh, dc now hold d h0, d c0 ----
    ICD_TRY(icd_gemm_simple(prec, d->dh, 1, D, d->mean_enc, 1, C, d->d_h_lin_w, C, D, C, B,
                            nullptr, nullptr, nullptr, 0, nullptr, 0, nullptr, 0.f, s, ICD_GEMM_ALLOW_SPLITK));
    ICD_TRY(icd_colsum(d->dh, D, B, D, nullptr, d->d_h_lin_b, s));
    ICD_TRY(icd_gemm_simple(prec, d->dc, 1, D, d->mean_enc, 1, C, d->d_c_lin_w, C, D, C, B,
                            nullptr, nullptr, nullptr, 0, nullptr, 0, nullptr, 0.f, s, ICD_GEMM_ALLOW_SPLITK));
    ICD_TRY(icd_colsum(d->dc, D, B, D, nullptr, d->d_c_lin_b, s));

    // ---- hoisted weight gradients over the T*B stacked rows ----
    // d[W_dec; W_fbeta; W_hh] = dz^T * h_prev_all ; d[b_dec; b_fbeta; b_hh] = colsum(dz)
    ICD_TRY(icd_gemm_simple(prec, d->dz, 1, NZ, d->h_all, 1, D, d->d_w_cat, D, NZ, D, TB,
                            nullptr, nullptr, nullptr, 0, nullptr, 0, nullptr, 0.f, s, ICD_GEMM_ALLOW_SPLITK));
    ICD_TRY(icd_colsum(d->dz, NZ, TB, NZ, nullptr, d->d_b_cat, s));
    // dW_ih = [dG^T * emb_x | dG^T * gated]
    const float* dG = d->dz + A + C;
    ICD_TRY(icd_gemm_simple(prec, dG, 1, NZ, d->emb_x, 1, E, d->d_w_ih, E + C, 4 * D, E, TB,
                            nullptr, nullptr, nullptr, 0, nullptr, 0, nullptr, 0.f, s, ICD_GEMM_ALLOW_SPLITK));
    ICD_TRY(icd_gemm_simple(prec, dG, 1, NZ, d->gated, 1, C, d->d_w_ih + E, E + C, 4 * D, C, TB,
                            nullptr, nullptr, nullptr, 0, nullptr, 0, nullptr, 0.f, s, ICD_GEMM_ALLOW_SPLITK));
    // embedding gradient (:247) when fine-tuned: d_emb_x = dG * W_ih[:, :E], scatter-added by token id
    if (d->d_emb_w) {
        ICD_TRY(icd_gemm_simple(prec, dG, NZ, 1, d->w_ih, 1, E + C, d->d_emb_x, E, TB, E, 4 * D,
                                nullptr, nullptr, nullptr, 0, nullptr, 0, nullptr, 0.f, s));
        ICD_CUDA(cudaMemsetAsync(d->d_emb_w, 0, (d->emb_is_f64 ? sizeof(double) : sizeof(float)) * (size_t)V * E, s));
        // (d_gated is free after the time loop: it serves as the sort workspace of the deterministic scatter)
        ICD_TRY(icd_embed_scatter_add(d->d_emb_w, d->emb_is_f64, d->captions, B, d->L, T, E, V, d->bt_host, d->d_emb_x, s,
                                      d->d_gated, (int64_t)sizeof(float) * B * C));
    }
    if (d->ev_rec_ready) ICD_CUDA(cudaEventRecord(reinterpret_cast<cudaEvent_t>(d->ev_rec_ready), s));
    // attention projections: d_att_enc for all steps at once, full_att grads, then enc_att grads (:54)
    if (ix)          // per image: d_att_enc (n_img,P,A) summed over each image's (row, step) pairs
        ICD_TRY(icd_attention_proj_bwd_indexed(B, n_img, T, P, A, d->bt_host, ix->img_row_ptr, ix->img_rows, d->att_enc, d->z, NZ,
                                               d->full_att_w, d->d_e, d->d_att_enc, d->d_full_att_w, d->d_full_att_b,
                                               d->d_enc_att_b, d->proj_partial, s));
    else
        ICD_TRY(icd_attention_proj_bwd(B, T, P, A, d->bt_host, d->att_enc, d->z, NZ, d->full_att_w, d->d_e,
                                       d->d_att_enc, d->d_full_att_w, d->d_full_att_b, d->d_enc_att_b, d->proj_partial,
                                       stream));
    ICD_TRY(icd_gemm_simple(prec, d->d_att_enc, 1, A, d->enc, 1, C, d->d_enc_att_w, C, A, C, n_img * P,
                            nullptr, nullptr, nullptr, 0, nullptr, 0, nullptr, 0.f, s, ICD_GEMM_ALLOW_SPLITK));
    // ---- optional: gradient w.r.t. the encoder features (--fine_tune_encoder) ----
    if (d->d_enc) {
        ICD_CHECK_ARG(d->d_awe_all && d->d_mean, "attention_decoder: d_enc needs the d_awe_all and d_mean scratch buffers");
        // d_mean = d h0 W_h + d c0 W_c  (:161-163)
        ICD_TRY(icd_gemm_simple(prec, d->dh, D, 1, d->h_lin_w, 1, C, d->d_mean, C, B, C, D,
                                nullptr, nullptr, nullptr, 0, nullptr, 0, nullptr, 0.f, s));
        ICD_TRY(icd_gemm_simple(prec, d->dc, D, 1, d->c_lin_w, 1, C, d->d_mean, C, B, C, D,
                                nullptr, nullptr, nullptr, 0, nullptr, 0, nullptr, 1.f, s));
        int32_t* row_len_ws = reinterpret_cast<int32_t*>(d->proj_partial);       // free again after the projection pass
        ICD_TRY(icd_attention_enc_grad_indexed(B, n_img, T, P, C, d->bt_host, ix ? ix->img_row_ptr : nullptr,
                                               ix ? ix->img_rows : nullptr, d->alphas, d->d_awe_all, d->d_mean, d->d_enc,
                                               row_len_ws, s));
        // + d_att_enc W_e  (:54)
        ICD_TRY(icd_gemm_simple(prec, d->d_att_enc, A, 1, d->enc_att_w, 1, C, d->d_enc, C, n_img * P, C, A,
                                nullptr, nullptr, nullptr, 0, nullptr, 0, nullptr, 1.f, s));
    }
    return 0;
}

extern "C" int icd_attention_decoder_bwd(const icd_att_desc_t* d, void* stream) { return decoder_bwd(d, nullptr, stream); }
extern "C" int icd_attention_decoder_bwd_indexed(const icd_att_desc_t* d, const icd_att_index_t* ix, void* stream) {
    return decoder_bwd(d, ix, stream);
}
