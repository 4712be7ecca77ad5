// bf16 tensor-core tier of AttentionDecoder.forward / backward (BASELINE.json configs[2]: "bf16 GEMMs").
//
// Same dataflow as decoder_loop.cu (the fp32 parity tier); every dense contraction runs on the tcgen05/TMA kernel
// of gemm_tc.cu with bf16 operands and fp32 accumulation, everything else (attention step, softmax, LSTM gate math,
// reductions, all saved activations and all gradients) stays fp32.  bf16 K-major operand copies live in a
// caller-provided arena (desc->tc_ws):
//   forward, kept for backward : weights (W_e, [W_dec;W_fb;W_hh], W_ih split at E, W_h, W_c, W_fc), enc, mean, emb_x,
//                                h_t, gated_t, dropout(h)
//   backward                   : transposed weight copies for the dX contractions, dY and dY^T, per-step dz,
//                                and the transposed activation stacks feeding the hoisted dW contractions.
// The transposes are produced by the fp32->bf16 conversion pass itself (convert_transpose_kernel), so the tensor-core
// kernel only ever sees K-major operands.
#include "common.cuh"
#include "gemm_tc.cuh"
#include <stdlib.h>

namespace {

struct BtPack { int v[ICD_MAX_STEPS]; };

__global__ void row_valid_kernel16(int B, int T, const BtPack bt, unsigned char* __restrict__ valid) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * T) return;
    const int b = i / T, t = i % T;
    valid[i] = (b < bt.v[t]) ? 1 : 0;
}

inline int64_t up8(int64_t x) { return (x + 7) / 8 * 8; }

// bump allocator over the caller's arena
struct Arena {
    char* base; int64_t cap, off; bool ok;
    void* take_bytes(int64_t bytes) {
        bytes = (bytes + 255) / 256 * 256;
        void* p = base ? base + off : nullptr;
        off += bytes;
        if (base && off > cap) ok = false;
        return p;
    }
    void* take(int64_t rows, int64_t ld) { return take_bytes(rows * ld * 2); }      // bf16 elements
};

// every bf16 buffer of the tier, carved in a fixed order so forward and backward agree on the layout.
// No transposed copies exist: the tensor-core kernel consumes MN-major operands directly (gemm_tc.cu).
struct Bufs {
    void *We, *Wcat, *WihE, *WihC, *Wh, *Wc, *Wfc;                 // weights [out, in] (K-major for y = x W^T, MN-major B for dX = dY W)
    void *WihCp;                                                   // W_ih[:, E:] with gate-permuted rows (fused LSTMCell epilogue)
    void *enc, *att_enc, *mean, *embx, *h, *gated, *hdrop;         // forward activations [rows, features]
    void *dY, *dz, *dh, *dc, *dae;                                 // backward: [rows, features]
    float* splitk; int64_t splitk_floats;                          // deterministic split-K slices
    float* colsum_ws;                                              // partial column sums of the bf16 dY
    int64_t ldE, ldV;
};

// n_img: images of the features (= B, or icd_att_index_t.n_img when captions share images): enc, att_enc and d_att_enc are per image
void carve(const icd_att_desc_t* d, int64_t n_img, Arena& a, Bufs& b) {
    const int64_t B = d->B, T = d->T, P = d->P, C = d->C, A = d->A, D = d->D, E = d->E, V = d->V;
    const int64_t NZ = A + C + 4 * D, TB = T * B;
    b.ldE = up8(E); b.ldV = up8(V);
    b.We = a.take(A, C); b.Wcat = a.take(NZ, D); b.WihE = a.take(4 * D, b.ldE); b.WihC = a.take(4 * D, C);
    b.Wh = a.take(D, C); b.Wc = a.take(D, C); b.Wfc = a.take(V, D);
    b.WihCp = a.take(4 * D, C);
    b.enc = d->enc16 ? const_cast<void*>(d->enc16) : a.take(n_img * P, C);      // caller-provided bf16 features are used in place
    b.att_enc = a.take(n_img * P, A); b.mean = a.take(B, C); b.embx = a.take(TB, b.ldE);
    b.h = a.take(TB + B, D);
    b.gated = a.take(TB, C); b.hdrop = a.take(B * T, D);
    b.dY = a.take(B * T, b.ldV); b.dz = a.take(TB, NZ); b.dh = a.take(B, D); b.dc = a.take(B, D);
    b.dae = a.take(n_img * P, A);
    // split-K workspace: the largest request among the contractions that may split
    const int shapes[][3] = {
        {(int)B, (int)D, (int)C},            // h_lin / c_lin
        {(int)B, (int)NZ, (int)D},           // z = h W_cat^T
        {(int)B, (int)(4 * D), (int)C},      // gates
        {(int)B, (int)C, (int)(4 * D)},      // d_gated
        {(int)B, (int)D, (int)NZ},           // dh
        {(int)D, (int)C, (int)B},            // d h_lin / c_lin weights
        {(int)NZ, (int)D, (int)TB},          // d W_cat
        {(int)(4 * D), (int)E, (int)TB},     // d W_ih (embedding part)
        {(int)(4 * D), (int)C, (int)TB},     // d W_ih (awe part)
        {(int)TB, (int)E, (int)(4 * D)},     // d emb_x
        {(int)A, (int)C, (int)(n_img * P)},  // d enc_att.weight
        {(int)V, (int)D, (int)(B * T)},      // d fc.weight
        {(int)(B * T), (int)D, (int)V},      // d hdrop
    };
    int64_t f = 0;
    for (const auto& sh : shapes) { const int64_t n = icd_gemm_bf16_splitk_floats(sh[0], sh[1], sh[2]); if (n > f) f = n; }
    b.splitk_floats = f;
    b.splitk = reinterpret_cast<float*>(a.take_bytes(f * 4));
    b.colsum_ws = reinterpret_cast<float*>(a.take_bytes(icd_colsum_bf16_ws_floats(B * T, (int)V) * 4));
}

int check16(const icd_att_desc_t* d, int n_img, Arena& a, Bufs& b) {
    ICD_CHECK_ARG(d->A % 8 == 0 && d->C % 8 == 0 && d->D % 8 == 0 && d->E % 4 == 0,
                  "attention_decoder(bf16): A, C, D must be multiples of 8 and E of 4 (A=%d C=%d D=%d E=%d)", d->A, d->C, d->D, d->E);
    a.base = reinterpret_cast<char*>(d->tc_ws); a.cap = d->tc_ws_bytes; a.off = 0; a.ok = true;
    carve(d, n_img, a, b);
    ICD_CHECK_ARG(d->tc_ws != nullptr && a.ok, "attention_decoder(bf16): tc_ws too small (%lld bytes given, %lld needed)",
                  (long long)d->tc_ws_bytes, (long long)a.off);
    return 0;
}

#define CVT(src, sr, rows, cols, dst, ld) ICD_TRY(icd_convert_bf16((src), (sr), 1, (rows), (cols), (dst), (ld), s))
// C[M,N] (+ optional bf16 copy) = A * B^T + epilogue; amn / bmn: operand stored [K][M] / [K][N] (MN-major)
#define MMX(A16, lda, amn, B16, ldb, bmn, Cp, ldc, M, N, K, b1, b2, a1, l1, a2, l2, mask, C16, ldc16) \
    ICD_TRY(icd_gemm_bf16_ex((A16), (lda), (amn), (B16), (ldb), (bmn), (Cp), (ldc), (M), (N), (K), (b1), (b2), (a1), (l1), \
                             (a2), (l2), (mask), 0.f, s, (C16), (ldc16), u.splitk, u.splitk_floats))

inline char* at16(void* p, int64_t elem_off) { return reinterpret_cast<char*>(p) + elem_off * 2; }

}  // namespace

// B images -> pixel means; row_ptr / rows (optional): the mean of image b is written to rows[row_ptr[b] .. row_ptr[b+1])
int icd_convert_features_bf16(int B, int P, int C, const float* enc, void* enc16, float* mean, void* mean16, cudaStream_t s,
                              const int32_t* row_ptr, const int32_t* rows);
int icd_feature_mean_bf16(int B, int P, int C, const void* enc16, float* mean, void* mean16, cudaStream_t s,
                          const int32_t* row_ptr, const int32_t* rows);

int64_t icd_att_tc_ws_bytes(const icd_att_desc_t* d, int n_img) {
    Arena a; a.base = nullptr; a.cap = 0; a.off = 0; a.ok = true;
    Bufs b;
    carve(d, n_img, a, b);
    return a.off;
}

int icd_attention_decoder_fwd_bf16(const icd_att_desc_t* d, const icd_att_index_t* ix, cudaStream_t s) {
    const int n_img = ix ? ix->n_img : d->B;
    const int32_t* img_index = ix ? ix->img_index : nullptr;
    Arena ar; Bufs u;
    ICD_TRY(check16(d, n_img, ar, u));
    const int B = d->B, T = d->T, P = d->P, C = d->C, A = d->A, D = d->D, E = d->E, V = d->V;
    const int NZ = A + C + 4 * D, TB = T * B;
    const long long BD = (long long)B * D;

    BtPack pack;
    for (int t = 0; t < ICD_MAX_STEPS; ++t) pack.v[t] = t < T ? d->bt_host[t] : 0;
    row_valid_kernel16<<<(B * T + 255) / 256, 256, 0, s>>>(B, T, pack, d->row_valid);
    ICD_LAUNCH_CHECK();
    ICD_CUDA(cudaMemsetAsync(d->alphas, 0, sizeof(float) * (size_t)B * T * P, s));
    if (d->bt_host[T - 1] < B) {          // ragged batch: rows that go inactive must read as zeros later
        ICD_CUDA(cudaMemsetAsync(d->hdrop, 0, sizeof(float) * (size_t)B * T * D, s));
        ICD_CUDA(cudaMemsetAsync(u.hdrop, 0, (size_t)B * T * D * 2, s));
        ICD_CUDA(cudaMemsetAsync(d->h_all, 0, sizeof(float) * (size_t)(T + 1) * BD, s));
        ICD_CUDA(cudaMemsetAsync(d->c_all, 0, sizeof(float) * (size_t)(T + 1) * BD, s));
        ICD_CUDA(cudaMemsetAsync(d->gated, 0, sizeof(float) * (size_t)T * B * C, s));
        ICD_CUDA(cudaMemsetAsync(d->z, 0, sizeof(float) * (size_t)T * B * NZ, s));
        ICD_CUDA(cudaMemsetAsync(u.h, 0, (size_t)(TB + B) * D * 2, s));
        ICD_CUDA(cudaMemsetAsync(u.gated, 0, (size_t)TB * C * 2, s));
    }
    // fp32 [b_dec; b_fbeta; 0] (b_hh rides with the hoisted embedding term); the fp32 w_cat copy is kept for callers
    // that inspect it but the tier itself only needs the bf16 stack
    ICD_CUDA(cudaMemcpyAsync(d->b_cat, d->dec_att_b, sizeof(float) * A, cudaMemcpyDeviceToDevice, s));
    ICD_CUDA(cudaMemcpyAsync(d->b_cat + A, d->f_beta_b, sizeof(float) * C, cudaMemcpyDeviceToDevice, s));
    ICD_CUDA(cudaMemsetAsync(d->b_cat + A + C, 0, sizeof(float) * 4 * D, s));

    // ---- bf16 copies of the weights (they change every optimiser step) ----
    // (one launch for all of them: icd_convert_bf16_batch)
    static const bool fused_cell_env = [] { const char* e = getenv("ICD_FUSED_CELL"); return !e || e[0] != '0'; }();
    const bool fused_cell = fused_cell_env && D % 16 == 0 && (E + C) % 4 == 0 && E % 4 == 0 && NZ % 4 == 0 &&
                            (!d->drop_mask || D % 8 == 0) && (T * D) % 8 == 0;
    {
        const IcdCvtSeg segs[9] = {
            {d->enc_att_w, C, A, C, u.We, C},
            {d->dec_att_w, D, A, D, u.Wcat, D},                                               // [W_dec; W_fbeta; W_hh]
            {d->f_beta_w, D, C, D, at16(u.Wcat, (int64_t)A * D), D},
            {d->w_hh, D, 4 * D, D, at16(u.Wcat, (int64_t)(A + C) * D), D},
            {d->w_ih, E + C, 4 * D, E, u.WihE, u.ldE},
            {d->w_ih + E, E + C, 4 * D, C, u.WihC, C},
            {d->h_lin_w, C, D, C, u.Wh, C},
            {d->c_lin_w, C, D, C, u.Wc, C},
            {d->fc_w, D, V, D, u.Wfc, D}};
        ICD_TRY(icd_convert_bf16_batch(segs, 9, s));
    }
    if (fused_cell) ICD_TRY(icd_convert_bf16_gateperm(d->w_ih + E, E + C, D, C, u.WihCp, C, s));
    // ---- features: fp32 -> bf16 and the pixel mean (:161) in one pass over encoder_out ----
    //    (captions that share images: once per image, the mean written to each of the image's rows)
    const int32_t* mrow_ptr = ix ? ix->img_row_ptr : nullptr;
    const int32_t* mrows = ix ? ix->img_rows : nullptr;
    if (d->enc16) ICD_TRY(icd_feature_mean_bf16(n_img, P, C, d->enc16, d->mean_enc, u.mean, s, mrow_ptr, mrows));
    else {
        ICD_CHECK_ARG(d->enc != nullptr, "attention_decoder(bf16): neither enc nor enc16 given");
        ICD_TRY(icd_convert_features_bf16(n_img, P, C, d->enc, u.enc, d->mean_enc, u.mean, s, mrow_ptr, mrows));
    }

    // K1: att_enc = enc_att(encoder_out), once per batch (models/attention.py:54); stored bf16 only
    MMX(u.enc, C, 0, u.We, C, 0, nullptr, 0, n_img * P, A, C, d->enc_att_b, nullptr, nullptr, 0, nullptr, 0, nullptr, u.att_enc, A);
    // K7: init_hidden_state (:162-163); h_0 also emitted as bf16 (operand of the first step)
    MMX(u.mean, C, 0, u.Wh, C, 0, d->h_all, D, B, D, C, d->h_lin_b, nullptr, nullptr, 0, nullptr, 0, nullptr, u.h, D);
    MMX(u.mean, C, 0, u.Wc, C, 0, d->c_all, D, B, D, C, d->c_lin_b, nullptr, nullptr, 0, nullptr, 0, nullptr, nullptr, 0);
    // K5: embedding lookup (:247) + hoisted input contraction
    // emb_w == NULL: emb_x (T,B,E) was filled by the caller with pre-computed embeddings (the reference's use_bert branch,
    // models/attention.py:242-244: (B,L,768) BERT vectors instead of the table lookup); they carry no gradient
    if (d->emb_w) ICD_TRY(icd_embed_gather(d->emb_w, d->emb_is_f64, d->captions, B, d->L, T, E, V, d->emb_x, s));
    CVT(d->emb_x, E, TB, E, u.embx, u.ldE);
    MMX(u.embx, u.ldE, 0, u.WihE, u.ldE, 0, d->xg, 4 * D, TB, 4 * D, E, d->b_ih, d->b_hh, nullptr, 0, nullptr, 0, nullptr, nullptr, 0);

    for (int t = 0; t < T; ++t) {
        const int bt = d->bt_host[t];
        if (bt == 0) break;
        const float* c_prev = d->c_all + (size_t)t * BD;
        float* zt = d->z + (size_t)t * B * NZ;
        char* h16 = at16(u.h, (int64_t)t * B * D);
        char* g16 = at16(u.gated, (int64_t)t * B * C);
        icd_gemm_next_feeds_attention();       // the attention-step grid is staged behind K2 and placed when K2's last CTA exits
        MMX(h16, D, 0, u.Wcat, D, 0, zt, NZ, bt, NZ, D, d->b_cat, nullptr, nullptr, 0, nullptr, 0, nullptr, nullptr, 0);   // K2
        ICD_TRY(icd_attention_step_fwd_bf16(bt, P, C, A, img_index, u.enc, u.att_enc, zt, NZ, d->full_att_w, d->full_att_b,
                                            zt + A, NZ, d->alphas + (size_t)t * P, (int64_t)T * P,
                                            d->awe_raw + (size_t)t * B * C, d->gate + (size_t)t * B * C,
                                            d->gated + (size_t)t * B * C, g16, (void*)s));                         // K3
        if (fused_cell) {                                                                                           // K4 + LSTMCell
            ICD_TRY(icd_gemm_bf16_lstm_cell(g16, C, u.WihCp, C, bt, D, C, d->xg + (size_t)t * B * 4 * D, 4 * D, zt + A + C, NZ, c_prev,
                                            d->gates_act + (size_t)t * B * 4 * D, d->c_all + (size_t)(t + 1) * BD,
                                            d->h_all + (size_t)(t + 1) * BD, d->hdrop + (size_t)t * D, (int64_t)T * D,
                                            d->drop_mask ? d->drop_mask + (size_t)t * BD : nullptr, d->drop_scale,
                                            at16(u.h, (int64_t)(t + 1) * B * D), at16(u.hdrop, (int64_t)t * D), s));
            continue;
        }
        MMX(g16, C, 0, u.WihC, C, 0, d->gates_pre, 4 * D, bt, 4 * D, C, nullptr, nullptr,
            d->xg + (size_t)t * B * 4 * D, 4 * D, zt + A + C, NZ, nullptr, nullptr, 0);                            // K4
        ICD_TRY(icd_lstm_pointwise_fwd(bt, D, d->gates_pre, c_prev, d->gates_act + (size_t)t * B * 4 * D,
                                       d->c_all + (size_t)(t + 1) * BD, d->h_all + (size_t)(t + 1) * BD,
                                       d->hdrop + (size_t)t * D, (int64_t)T * D,
                                       d->drop_mask ? d->drop_mask + (size_t)t * BD : nullptr, d->drop_scale, s,
                                       at16(u.h, (int64_t)(t + 1) * B * D), at16(u.hdrop, (int64_t)t * D)));
    }
    // K6: predictions = fc(dropout(h)) for every (b,t) at once (:279-280); inactive rows exactly 0 (:253)
    MMX(u.hdrop, D, 0, u.Wfc, D, 0, d->predictions, V, B * T, V, D, d->fc_b, nullptr, nullptr, 0, nullptr, 0, d->row_valid, nullptr, 0);
    return 0;
}

int icd_attention_decoder_bwd_bf16(const icd_att_desc_t* d, const icd_att_index_t* ix, cudaStream_t s) {
    const int n_img = ix ? ix->n_img : d->B;
    const int32_t* img_index = ix ? ix->img_index : nullptr;
    Arena ar; Bufs u;
    ICD_TRY(check16(d, n_img, ar, u));
    const int B = d->B, T = d->T, P = d->P, C = d->C, A = d->A, D = d->D, E = d->E, V = d->V;
    const int NZ = A + C + 4 * D, TB = T * B, BT = B * T, BP = n_img * P;      // BP: pixel rows of the per-image tensors
    const long long BD = (long long)B * D;
    const float* NF = nullptr;

    if (d->bt_host[T - 1] < B) {          // ragged batch: inactive rows of the stacked gradients contribute zeros
        ICD_CUDA(cudaMemsetAsync(d->dz, 0, sizeof(float) * (size_t)TB * NZ, s));
        ICD_CUDA(cudaMemsetAsync(u.dz, 0, (size_t)TB * NZ * 2, s));
        ICD_CUDA(cudaMemsetAsync(d->d_e, 0, sizeof(float) * (size_t)B * T * P, s));
    }
    ICD_CUDA(cudaMemsetAsync(d->dh, 0, sizeof(float) * (size_t)BD, s));
    ICD_CUDA(cudaMemsetAsync(d->dc, 0, sizeof(float) * (size_t)BD, s));

    // ---- fc (:279): d_hdrop = dY W_fc ; dW_fc = dY^T hdrop ; db_fc = masked column sum of dY ----
    const void* dY16 = d->d_predictions16;
    int64_t ldY = d->ld_dpred16;
    if (!dY16) { CVT(d->d_predictions, V, BT, V, u.dY, u.ldV); dY16 = u.dY; ldY = u.ldV; }
    MMX(dY16, ldY, 0, u.Wfc, D, 1, d->d_hdrop, D, BT, D, V, NF, NF, NF, 0, NF, 0, nullptr, nullptr, 0);
    MMX(dY16, ldY, 1, u.hdrop, D, 1, d->d_fc_w, D, V, D, BT, NF, NF, NF, 0, NF, 0, nullptr, nullptr, 0);
    ICD_TRY(icd_colsum_bf16(dY16, ldY, (int64_t)BT, V, d->row_valid, d->d_fc_b, u.colsum_ws, s));
    if (d->ev_fc_ready) ICD_CUDA(cudaEventRecord(reinterpret_cast<cudaEvent_t>(d->ev_fc_ready), s));   // fc gradients final

    // ---- BPTT ----
    // The dh contraction (M = batch, N = D, K = NZ) runs split-K; its reduce pass is deferred into the next step's LSTM
    // gate kernel, which sums the K-slice planes while it reads dh anyway (one launch less per step).
    int dh_splits = 0, dh_rows = 0;            // > 0: dh of the previous iteration lives in u.splitk as dh_splits planes of dh_rows rows
    for (int t = T - 1; t >= 0; --t) {
        const int bt = d->bt_host[t];
        if (bt == 0) continue;
        float* dzt = d->dz + (size_t)t * B * NZ;
        const float* zt = d->z + (size_t)t * B * NZ;
        char* dz16 = at16(u.dz, (int64_t)t * B * NZ);
        ICD_TRY(icd_lstm_pointwise_bwd(bt, D, d->dh, d->d_hdrop + (size_t)t * D, (int64_t)T * D,
                                       d->drop_mask ? d->drop_mask + (size_t)t * BD : nullptr, d->drop_scale,
                                       d->dc, d->gates_act + (size_t)t * B * 4 * D,
                                       d->c_all + (size_t)t * BD, d->c_all + (size_t)(t + 1) * BD,
                                       dzt + A + C, NZ, s, at16(dz16, A + C), NZ,     // dG also emitted as bf16
                                       u.splitk, dh_splits, dh_rows));
        // d_gated = dG W_ih[:, E:]           (W_ih[:, E:] stored [4D, C] = MN-major B, N = C, K = 4D)
        icd_gemm_next_feeds_attention();
        MMX(at16(dz16, A + C), NZ, 0, u.WihC, C, 1, d->d_gated, C, bt, C, 4 * D, NF, NF, NF, 0, NF, 0, nullptr, nullptr, 0);
        ICD_TRY(icd_attention_step_bwd_bf16_idx(bt, P, C, A, img_index, u.enc, u.att_enc, zt, NZ, d->full_att_w,
                                            d->alphas + (size_t)t * P, (int64_t)T * P,
                                            d->d_alphas ? d->d_alphas + (size_t)t * P : nullptr, (int64_t)T * P,
                                            d->gate + (size_t)t * B * C, d->awe_raw + (size_t)t * B * C, d->d_gated,
                                            dzt, NZ, dzt + A, NZ, d->d_e + (size_t)t * P, (int64_t)T * P,
                                            dz16, NZ, d->d_enc ? d->d_awe_all + (size_t)t * B * C : nullptr,
                                            (void*)s));                             // d att_dec | d fbeta_pre (+ bf16)
        // dh_t = dz [W_dec; W_fbeta; W_hh]    (stack stored [NZ, D] = MN-major B, N = D, K = NZ); reduce deferred (see above)
        ICD_TRY(icd_gemm_bf16_ex(dz16, NZ, 0, u.Wcat, D, 1, d->dh, D, bt, D, NZ, NF, NF, NF, 0, NF, 0, nullptr, 0.f, s,
                                 nullptr, 0, u.splitk, u.splitk_floats, &dh_splits));
        dh_rows = bt;
    }
    if (dh_splits > 0) ICD_TRY(icd_splitk_finish(u.splitk, dh_splits, dh_rows, D, d->dh, D, nullptr, 0, s));   // d h0

    // ---- init_hidden_state (:161-163): dh, dc now hold d h0, d c0 ----
    CVT(d->dh, D, B, D, u.dh, D);
    CVT(d->dc, D, B, D, u.dc, D);
    MMX(u.dh, D, 1, u.mean, C, 1, d->d_h_lin_w, C, D, C, B, NF, NF, NF, 0, NF, 0, nullptr, nullptr, 0);
    ICD_TRY(icd_colsum(d->dh, D, B, D, nullptr, d->d_h_lin_b, s));
    MMX(u.dc, D, 1, u.mean, C, 1, d->d_c_lin_w, C, D, C, B, NF, NF, NF, 0, NF, 0, nullptr, nullptr, 0);
    ICD_TRY(icd_colsum(d->dc, D, B, D, nullptr, d->d_c_lin_b, s));

    // ---- hoisted weight gradients over the T*B stacked rows: dW = dY^T X, both operands MN-major as stored ----
    MMX(u.dz, NZ, 1, u.h, D, 1, d->d_w_cat, D, NZ, D, TB, NF, NF, NF, 0, NF, 0, nullptr, nullptr, 0);
    ICD_TRY(icd_colsum(d->dz, NZ, TB, NZ, nullptr, d->d_b_cat, s));
    char* dG16 = at16(u.dz, A + C);                                // columns [A+C, NZ) of dz = dG  [TB x 4D], ld NZ
    MMX(dG16, NZ, 1, u.embx, u.ldE, 1, d->d_w_ih, E + C, 4 * D, E, TB, NF, NF, NF, 0, NF, 0, nullptr, nullptr, 0);
    MMX(dG16, NZ, 1, u.gated, C, 1, d->d_w_ih + E, E + C, 4 * D, C, TB, NF, NF, NF, 0, NF, 0, nullptr, nullptr, 0);
    if (d->d_emb_w) {
        MMX(dG16, NZ, 0, u.WihE, u.ldE, 1, d->d_emb_x, E, TB, E, 4 * D, NF, NF, NF, 0, NF, 0, nullptr, nullptr, 0);
        ICD_CUDA(cudaMemsetAsync(d->d_emb_w, 0, (d->emb_is_f64 ? sizeof(double) : sizeof(float)) * (size_t)V * E, s));
        // (d_gated is free after the time loop: it serves as the sort workspace of the deterministic scatter)
        ICD_TRY(icd_embed_scatter_add(d->d_emb_w, d->emb_is_f64, d->captions, B, d->L, T, E, V, d->bt_host, d->d_emb_x, s,
                                      d->d_gated, (int64_t)sizeof(float) * B * C));
    }
    if (d->ev_rec_ready) ICD_CUDA(cudaEventRecord(reinterpret_cast<cudaEvent_t>(d->ev_rec_ready), s)); // recurrent gradients final
    // attention projections: d_att_enc for all steps at once (bf16 only: it is just the A operand of the next
    // contraction), full_att grads and the enc_att bias grad from the same pass, then the enc_att weight grad (:54)
    if (ix)          // per image: d_att_enc (n_img,P,A) summed over each image's (row, step) pairs
        ICD_TRY(icd_attention_proj_bwd_bf16_indexed(B, n_img, T, P, A, d->bt_host, ix->img_row_ptr, ix->img_rows, u.att_enc, d->z, NZ,
                                                    d->full_att_w, d->d_e, u.dae, d->d_full_att_w, d->d_full_att_b,
                                                    d->d_enc_att_b, d->proj_partial, d->dz, NZ, s));
    else
        ICD_TRY(icd_attention_proj_bwd_bf16_ex(B, T, P, A, d->bt_host, u.att_enc, d->z, NZ, d->full_att_w, d->d_e,
                                               nullptr, u.dae, d->d_full_att_w, d->d_full_att_b, d->d_enc_att_b,
                                               d->proj_partial, d->dz, NZ, (void*)s));
    MMX(u.dae, A, 1, u.enc, C, 1, d->d_enc_att_w, C, A, C, BP, NF, NF, NF, 0, NF, 0, nullptr, nullptr, 0);
    // ---- optional: gradient w.r.t. the encoder features (--fine_tune_encoder) ----
    if (d->d_enc) {
        ICD_CHECK_ARG(d->d_awe_all && d->d_mean, "attention_decoder: d_enc needs the d_awe_all and d_mean scratch buffers");
        // d_mean = d h0 W_h + d c0 W_c (:161-163): W_h / W_c stored [D, C] = MN-major B (N = C, K = D); u.dh / u.dc hold d h0 / d c0
        MMX(u.dh, D, 0, u.Wh, C, 1, d->d_mean, C, B, C, D, NF, NF, NF, 0, NF, 0, nullptr, nullptr, 0);
        ICD_TRY(icd_gemm_bf16_ex(u.dc, D, 0, u.Wc, C, 1, d->d_mean, C, B, C, D, NF, NF, NF, 0, NF, 0, nullptr, 1.f, s,
                                 nullptr, 0, u.splitk, u.splitk_floats));
        int32_t* row_len_ws = reinterpret_cast<int32_t*>(d->proj_partial);       // free again after the projection pass
        ICD_TRY(icd_attention_enc_grad_indexed(B, n_img, T, P, C, d->bt_host, ix ? ix->img_row_ptr : nullptr,
                                               ix ? ix->img_rows : nullptr, d->alphas, d->d_awe_all, d->d_mean, d->d_enc,
                                               row_len_ws, s));
        // + d_att_enc W_e (:54): W_e stored [A, C] = MN-major B (N = C, K = A)
        ICD_TRY(icd_gemm_bf16_ex(u.dae, A, 0, u.We, C, 1, d->d_enc, C, BP, C, A, NF, NF, NF, 0, NF, 0, nullptr, 1.f, s,
                                 nullptr, 0, nullptr, 0));
    }
    return 0;
}
