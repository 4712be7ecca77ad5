// Batched, device-side beam search (gen_captions.py:16-131; state machine of SURVEY.md Appendix C).
//
// n_img independent images x k beam slots are decoded together: every step is one round of
//   embedding gather -> [W_dec;W_fbeta;W_hh] contraction -> fused attention step (features indexed per image,
//   never gathered/copied as at gen_captions.py:111, enc_att computed once per image instead of per beam per
//   step) -> LSTMCell -> fc -> per-image warp/block top-k over the (live beams x V) candidates -> beam reorder.
// No host synchronisation inside the loop; sequences and alpha frames are reconstructed at the end by
// back-tracking parent pointers, so no per-step copy of the growing (k, step, 14, 14) alpha tensor (:89).
//
// Finished images leave the working set (the reference stops an image's loop at k == 0, :118): the decoder state lives in
// SLOTS (one per unfinished image) whose live beams occupy consecutive rows; after every step both the slots and the rows
// of the surviving beams are compacted to the front (device-side scans),
// and every kernel of the next step — including the tensor-core contractions, which read their row count from device
// memory — only touches the live slots.  Per-image results (history, alpha frames, winners) stay indexed by image.
//
// Reference semantics kept: step 1 candidates come from beam 0 only (:78-79); later steps take the top
// k_live (= remaining beams) of the flattened (k_live * V) scores, sorted descending (:82); scores are raw
// summed log-probs (:74-76); beams that emit <end> leave the beam and are never replaced (:93-104); the winner is
// the first completed beam with the maximal score (:127); the loop body runs for step = 1..max_steps+1 (:119).
//
// icd_baseline_beam_search runs the same state machine (the same top-k, compaction, reorder and finalize kernels) over the
// BaselineDecoder's step: the image feature as LSTM step 0 from the zero state, then per step h W_hh^T on the live rows, one fused
// kernel for the embg gather + LSTMCell (+ the split of h for the fp32-grade vocabulary contraction), and the vocabulary layer.
#include "beam.cuh"
#include "gemm_tc.cuh"
#include <cuda_bf16.h>
#include <stdlib.h>

namespace {

constexpr int TOPK_NL = 19;     // 64-bit loads per thread of the register-resident top-k pass: rows of up to 2 * 256 * 19 = 9728 logits
constexpr int TOPK_CAP = 512;   // shared candidate list of that pass (logits >= tau of one row); more (massive ties): the streaming pass
constexpr int KMAX = 8;          // beam slots per image supported by the top-k kernel

inline long long up8ll(long long x) { return (x + 7) / 8 * 8; }
constexpr int X3_IMG_CHUNK = 64;          // most images per enc_att projection pass (bounds the split activation scratch)
// Images per pass: the projection runs as 256 x 256 super tiles on 74 CTA pairs, so a pass costs ceil(super tiles / 74) rounds whatever
// its row count.  64 images x 196 pixels are 98 super tiles = 2 rounds for 1.3 rounds of work; 48 images are 74 = exactly one.
// Pick the count (<= X3_IMG_CHUNK) with the most images per round.
inline int x3_img_chunk(int P, int A) {
    int best = X3_IMG_CHUNK;
    double best_score = 0.0;
    for (int ni = X3_IMG_CHUNK; ni >= 8; --ni) {
        const long long tiles_m = ((long long)ni * P + 127) / 128, st = ((tiles_m + 1) / 2) * ((A + 255) / 256);
        const long long rounds = (st + ICD_NUM_SMS / 2 - 1) / (ICD_NUM_SMS / 2);
        const double score = (double)ni / (double)rounds;
        if (score > best_score * 1.0001) { best_score = score; best = ni; }
    }
    return best;
}

}  // namespace

size_t carve(const icd_beam_desc_t* d, BeamWs* w, char* base, bool history) {
    const size_t R = (size_t)d->n_img * d->k, S = (size_t)d->max_steps + 1;
    const int P = d->P, C = d->C, A = d->A, D = d->D, E = d->E, V = d->V, NZ = A + C + 4 * D;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~(size_t)255; return base ? base + o : (char*)nullptr; };
    float* f;
#define TAKE_F(name, n) f = (float*)take(sizeof(float) * (n)); if (w) w->name = f;
    TAKE_F(att_enc, (size_t)d->n_img * P * A)
    TAKE_F(mean, (size_t)d->n_img * C)
    TAKE_F(h0, (size_t)d->n_img * D)
    TAKE_F(c0, (size_t)d->n_img * D)
    TAKE_F(h, R * D) TAKE_F(c, R * D) TAKE_F(h_tmp, R * D) TAKE_F(c_tmp, R * D)
    TAKE_F(w_cat, (size_t)NZ * D) TAKE_F(b_cat, (size_t)NZ)
    TAKE_F(emb_x, R * E) TAKE_F(z, R * NZ) TAKE_F(gated, R * C) TAKE_F(gates_pre, R * 4 * D)
    TAKE_F(logits, R * V)
    TAKE_F(embg, d->emb_is_f64 ? 0 : (size_t)V * 4 * D)       // embedding row x W_ih[:, :E]^T + b_ih for EVERY token, once per call
    TAKE_F(alpha_steps, (history ? S : 1) * R * P)
    TAKE_F(score, R) TAKE_F(score_tmp, R) TAKE_F(best_score, (size_t)d->n_img)
#undef TAKE_F
    int* ip;
#define TAKE_I(name, n) ip = (int*)take(sizeof(int) * (n)); if (w) w->name = ip;
    TAKE_I(img_index, R) TAKE_I(prev_word, R) TAKE_I(k_live, (size_t)d->n_img) TAKE_I(src, R)
    TAKE_I(parent, history ? S * R : 0) TAKE_I(word, history ? S * R : 0) TAKE_I(best_step, (size_t)d->n_img)
    TAKE_I(best_parent, (size_t)d->n_img)
    TAKE_I(slot_img, (size_t)d->n_img) TAKE_I(slot_img_tmp, (size_t)d->n_img) TAKE_I(k_live_tmp, (size_t)d->n_img)
    TAKE_I(new_slot, (size_t)d->n_img) TAKE_I(n_live, 4) TAKE_I(word_tmp, R) TAKE_I(ring_ticket, S + 2)
    ip = (int*)take(sizeof(int) * (size_t)d->n_img); if (w) w->row_off[0] = ip;
    ip = (int*)take(sizeof(int) * (size_t)d->n_img); if (w) w->row_off[1] = ip;
    if (w) w->tag = w->tag_tmp = nullptr;
    if (!history) { TAKE_I(tag, R) TAKE_I(tag_tmp, R) }
#undef TAKE_I
    long long* lp = (long long*)take(sizeof(long long) * R); if (w) w->tok64 = lp;
    if (d->precision == ICD_PREC_FP32X3) {
        auto takev = [&](size_t bytes) { return (void*)take(bytes); };
        void* v;
#define TAKE_X3(name, rows, K) v = takev((size_t)(rows) * 6 * up8ll(K) * 2); if (w) w->name = v;
        TAKE_X3(x3_We, A, C) TAKE_X3(x3_Wcat, NZ, D) TAKE_X3(x3_WihE, 4 * D, E) TAKE_X3(x3_WihC, 4 * D, C)
        TAKE_X3(x3_Wh, D, C) TAKE_X3(x3_Wc, D, C) TAKE_X3(x3_Wfc, V, D)
#undef TAKE_X3
        const size_t act_rows = R > (size_t)X3_IMG_CHUNK * P ? R : (size_t)X3_IMG_CHUNK * P;
        v = takev(act_rows * 6 * up8ll(C) * 2); if (w) w->x3_act = v;
        long long f = 0;
        const long long shapes[][3] = {{(long long)X3_IMG_CHUNK * P, A, 6 * up8ll(C)}, {(long long)d->n_img, D, 6 * up8ll(C)},
                                       {(long long)R, NZ, 6 * up8ll(D)}, {(long long)R, 4 * D, 6 * up8ll(E)},
                                       {(long long)R, 4 * D, 6 * up8ll(C)}, {(long long)R, V, 6 * up8ll(D)}};
        for (const auto& sh : shapes) { const long long n = icd_gemm_bf16_splitk_floats((int)sh[0], (int)sh[1], (int)sh[2]); if (n > f) f = n; }
        float* fp = (float*)take(sizeof(float) * (size_t)f);
        if (w) { w->x3_splitk = fp; w->x3_splitk_floats = f; }
    }
    return off;
}

namespace {

__global__ void beam_init_kernel(int n_img, int k, int D, int start_id, const float* __restrict__ h0,
                                 const float* __restrict__ c0, float* __restrict__ h, float* __restrict__ c,
                                 int* __restrict__ img_index, int* __restrict__ prev_word, long long* __restrict__ tok64,
                                 float* __restrict__ score, int* __restrict__ k_live, float* __restrict__ best_score,
                                 int* __restrict__ best_step, int* __restrict__ best_parent,
                                 int* __restrict__ slot_img, int* __restrict__ n_live, int* __restrict__ row_off) {
    // The reference starts every image with k IDENTICAL beams (:44-62) and takes the first top-k from beam 0 only (:78-79).
    // Here step 1 runs ONE state row per image (k_live = 1); the first top-k still selects k candidates from it, after which
    // the slot holds up to k distinct rows.  Same results, a fifth of the first (and most expensive) step's work.
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long R = (long long)n_img * k;
    if (i < (long long)n_img * D) { h[i] = h0[i]; c[i] = c0[i]; }
    if (i < R) img_index[i] = (int)(i / k);
    if (i < n_img) {
        prev_word[i] = start_id; tok64[i] = start_id; score[i] = 0.f;                                           // :47-52
        k_live[i] = 1; best_score[i] = -INFINITY; best_step[i] = 0; best_parent[i] = 0; slot_img[i] = (int)i; row_off[i] = (int)i;
    }
    if (i == 0) { n_live[0] = n_img; n_live[1] = n_img; }
}

__device__ __forceinline__ bool better(float v, int i, float bv, int bi) {
    return v > bv || (v == bv && i < bi);
}

// A lower bound tau of the KT-th largest value of a row, from the 256 per-thread maxima of the CTA: the KT-th largest of those maxima
// (KT distinct elements of the row are >= it).  Every thread returns the same value.  scratch: 8 * KT + 1 floats (8 * KT <= 64).
template <int KT>
__device__ __forceinline__ float block_kth_of_thread_max(float tm, float* scratch) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    float cur = tm;
#pragma unroll
    for (int r = 0; r < KT; ++r) {                                    // warp: its KT largest lane maxima, one knocked out per round
        const float wm = warp_max(cur);
        const unsigned hit = __ballot_sync(0xffffffffu, cur == wm);
        if (lane == 0) scratch[w * KT + r] = wm;
        if (lane == __ffs(hit) - 1) cur = -INFINITY;
    }
    __syncthreads();
    if (w == 0) {                                                      // warp 0: the KT-th largest of the 8 * KT warp candidates
        float c0 = (lane < 8 * KT) ? scratch[lane] : -INFINITY;
        float c1 = (lane + 32 < 8 * KT) ? scratch[lane + 32] : -INFINITY;
        float kth = -INFINITY;
#pragma unroll
        for (int r = 0; r < KT; ++r) {
            const float wm = warp_max(fmaxf(c0, c1));
            const unsigned hit = __ballot_sync(0xffffffffu, c0 == wm || c1 == wm);
            if (lane == __ffs(hit) - 1) { if (c0 == wm) c0 = -INFINITY; else c1 = -INFINITY; }
            kth = wm;
        }
        if (lane == 0) scratch[8 * KT] = kth;
    }
    __syncthreads();
    return scratch[8 * KT];
}

// One CTA per live slot.  log_softmax over V for each live row, add the running score, top-k_live over the
// flattened candidates (ties: lower flat index first), then the beam bookkeeping of gen_captions.py:85-116.
// State of the surviving beams goes to the *_tmp arrays (slot rows; beam_reorder_kernel moves it to the compacted slots),
// history (parent / word / trace) and winners are written per IMAGE.
template <int KT>      // KT >= k: length of the per-thread candidate lists (a shorter list = far fewer sorted insertions)
__global__ void __launch_bounds__(256, 4) beam_topk_kernel(
        int k, int V, int step, int end_id, const float* __restrict__ logits,
        const float* __restrict__ score, const int* __restrict__ k_live, const int* __restrict__ slot_img,
        const int* __restrict__ n_live, const int* __restrict__ row_off,
        float* __restrict__ score_tmp, int* __restrict__ word_tmp, int* __restrict__ k_live_tmp,
        int* __restrict__ slot_img_tmp, int* __restrict__ src,
        int* __restrict__ parent_s, int* __restrict__ word_s, int* __restrict__ trace_s,
        float* __restrict__ best_score, int* __restrict__ best_step, int* __restrict__ best_parent, int stream_only) {
    __shared__ float s_red[40];
    __shared__ float s_tau[8 * KT + 1];
    __shared__ float s_candx[TOPK_CAP];
    __shared__ int s_candi[TOPK_CAP];
    __shared__ int s_cnt;
    __shared__ float s_cv[256 * KT];
    __shared__ int s_ci[256 * KT];
    __shared__ float s_topv[KMAX];
    __shared__ int s_topi[KMAX];
    const int slot = blockIdx.x;
    if (slot >= n_live[0]) return;                                   // trace rows of finished images were preset to -1
    const int img = slot_img[slot];
    const int kl = k_live[slot];                                     // live state rows of this slot (> 0; 1 at step 1)
    const int nrows = kl;                                                                    // :78-82
    const int ksel = (step == 1) ? k : kl;                           // candidates to select (:79: k from the single first row)
    const int row0 = row_off[slot];                                  // first state row of this slot
    const float* lg = logits + (long long)row0 * V;
    const bool even = (V & 1) == 0;
    const int V2 = V >> 1;
    // thread-local top-KT over this thread's slice of the flattened (nrows*V) candidates (flat index f = i*V + v)
    float tv[KT]; int ti[KT];
#pragma unroll
    for (int j = 0; j < KT; ++j) { tv[j] = -INFINITY; ti[j] = 0x7fffffff; }
    auto flat_insert = [&](float v, int f) {                          // (v, lower flat index first) into the thread's flat top-KT
        if (better(v, f, tv[KT - 1], ti[KT - 1])) {
            tv[KT - 1] = v; ti[KT - 1] = f;
#pragma unroll
            for (int j = KT - 1; j > 0; --j) {
                if (better(tv[j], ti[j], tv[j - 1], ti[j - 1])) {
                    const float a = tv[j]; tv[j] = tv[j - 1]; tv[j - 1] = a;
                    const int b2 = ti[j]; ti[j] = ti[j - 1]; ti[j - 1] = b2;
                }
            }
        }
    };
    for (int i = 0; i < nrows; ++i) {
        if (!stream_only && even && V2 <= TOPK_NL * 256 && 8 * KT <= 64) {
            // Rows of up to 2 * 256 * TOPK_NL logits (V = 9490): the thread's slice of the row stays in registers.  Pass A: thread
            // maximum and sum of exp(x - maximum), five instructions per logit.  Then tau, a lower bound of the row's KT-th largest
            // logit (block_kth_of_thread_max), and pass B puts only the logits >= tau on a shared candidate list; candidate c is
            // valued and inserted by thread c.  (A thread sees 37 logits of a row: with per-thread sorted lists fed by every logit
            // — the streaming pass below — SOME lane of each warp inserts on nearly every element and the whole warp walks the
            // insertion path: 83 instructions per logit measured, the kernel was issue-bound at 190 us per step.)  Every logit that
            // can be among the row's KT best is >= tau, so the selected candidates are those of the streaming pass.
            const float2* x2r = reinterpret_cast<const float2*>(lg + (long long)i * V);
            float2 a[TOPK_NL];
#pragma unroll
            for (int u = 0; u < TOPK_NL; ++u) {
                const int j = threadIdx.x + u * 256;
                a[u] = (j < V2) ? x2r[j] : make_float2(-INFINITY, -INFINITY);
            }
            float tm = -INFINITY, tsum = 0.f;
#pragma unroll
            for (int u = 0; u < TOPK_NL; ++u) tm = fmaxf(tm, fmaxf(a[u].x, a[u].y));
            if (tm > -INFINITY) {
#pragma unroll
                for (int u = 0; u < TOPK_NL; ++u) tsum += __expf(a[u].x - tm) + __expf(a[u].y - tm);      // padding: exp(-inf) = 0
            }
            if (threadIdx.x == 0) s_cnt = 0;
            const float tau = block_kth_of_thread_max<KT>(tm, s_tau);      // (its barriers also publish s_cnt = 0)
#pragma unroll
            for (int u = 0; u < TOPK_NL; ++u) {
                const int j = threadIdx.x + u * 256;
                if (j < V2) {
                    if (a[u].x >= tau) { const int c = atomicAdd(&s_cnt, 1); if (c < TOPK_CAP) { s_candx[c] = a[u].x; s_candi[c] = 2 * j; } }
                    if (a[u].y >= tau) { const int c = atomicAdd(&s_cnt, 1); if (c < TOPK_CAP) { s_candx[c] = a[u].y; s_candi[c] = 2 * j + 1; } }
                }
            }
            const float rmax = block_max(tm, s_red);                        // (barriers: the candidate list is complete)
            const float sum = block_sum((tm == -INFINITY) ? 0.f : tsum * expf(tm - rmax), s_red);
            const int cnt = s_cnt;
            __syncthreads();                                                // every thread has read s_cnt before the next row resets it
            if (cnt <= TOPK_CAP) {
                const float rlsum = logf(sum), rscore = score[row0 + i];
                for (int c = threadIdx.x; c < cnt; c += 256) flat_insert(rscore + ((s_candx[c] - rmax) - rlsum), i * V + s_candi[c]);
                __syncthreads();                                            // the list is free again
                continue;
            }
        }
        // ONE streaming pass per row: online log-sum-exp (running max m, sum s of exp(x - m)) and, in the same pass, the
        // thread's top-KT RAW logits of the row.  log_softmax + score is monotone in the logit within a row, so the row's
        // best candidates are its largest logits; their values v = score + (x - max) - log(sum) (:74-76) are formed once the
        // row statistics are known and merged into the thread's flat top-KT by (v, lower flat index first).  (Selecting by
        // x instead of v inside a row can only differ if two DISTINCT logits among one thread's best k of a row collapse onto the
        // same fp32 v exactly at the selection boundary: a tie whose order torch.topk leaves unspecified too.)
        const float* x = lg + (long long)i * V;
        const float2* x2 = reinterpret_cast<const float2*>(x);
        float m = -INFINITY, ssum = 0.f;
        float rx[KT]; int rv[KT];
#pragma unroll
        for (int j = 0; j < KT; ++j) { rx[j] = -INFINITY; rv[j] = 0x7fffffff; }
        auto keep = [&](float xv, int v) {                            // thread-local top-KT raw logits of this row
            if (better(xv, v, rx[KT - 1], rv[KT - 1])) {
                rx[KT - 1] = xv; rv[KT - 1] = v;
#pragma unroll
                for (int j = KT - 1; j > 0; --j) {
                    if (better(rx[j], rv[j], rx[j - 1], rv[j - 1])) {
                        const float a = rx[j]; rx[j] = rx[j - 1]; rx[j - 1] = a;
                        const int b2 = rv[j]; rv[j] = rv[j - 1]; rv[j - 1] = b2;
                    }
                }
            }
        };
        if (even) {
            int j = threadIdx.x;
            for (; j + 3 * 256 < V2; j += 4 * 256) {
                float2 a[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) a[u] = x2[j + u * 256];
                // the running maximum moves at most once per 8 values: one rescale, then eight plain exp(x - m) terms
                const float cm = fmaxf(fmaxf(fmaxf(a[0].x, a[0].y), fmaxf(a[1].x, a[1].y)), fmaxf(fmaxf(a[2].x, a[2].y), fmaxf(a[3].x, a[3].y)));
                if (cm > m) { ssum *= __expf(m - cm); m = cm; }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    ssum += __expf(a[u].x - m) + __expf(a[u].y - m);
                    keep(a[u].x, 2 * (j + u * 256)); keep(a[u].y, 2 * (j + u * 256) + 1);
                }
            }
            for (; j < V2; j += 256) {
                const float2 a = x2[j];
                const float cm = fmaxf(a.x, a.y);
                if (cm > m) { ssum *= __expf(m - cm); m = cm; }
                ssum += __expf(a.x - m) + __expf(a.y - m);
                keep(a.x, 2 * j); keep(a.y, 2 * j + 1);
            }
        } else {
            for (int v = threadIdx.x; v < V; v += blockDim.x) {
                const float xv = x[v];
                if (xv > m) { ssum *= __expf(m - xv); m = xv; }
                ssum += __expf(xv - m);
                keep(xv, v);
            }
        }
        const float rmax = block_max(m, s_red);
        const float sum = block_sum((m == -INFINITY) ? 0.f : ssum * expf(m - rmax), s_red);
        const float rlsum = logf(sum), rscore = score[row0 + i];
        const int f0 = i * V;
#pragma unroll
        for (int q = 0; q < KT; ++q) {
            if (rv[q] == 0x7fffffff) continue;
            flat_insert(rscore + ((rx[q] - rmax) - rlsum), f0 + rv[q]);
        }
    }
#pragma unroll
    for (int j = 0; j < KT; ++j) { s_cv[threadIdx.x * KT + j] = tv[j]; s_ci[threadIdx.x * KT + j] = ti[j]; }
    __syncthreads();
    if (threadIdx.x < 32) {                                          // warp 0: kl rounds of arg-best
        const int lane = threadIdx.x;
        for (int round = 0; round < ksel; ++round) {
            float bv = -INFINITY; int bi = 0x7fffffff, bpos = -1;
            for (int q = lane; q < 256 * KT; q += 32)
                if (better(s_cv[q], s_ci[q], bv, bi)) { bv = s_cv[q]; bi = s_ci[q]; bpos = q; }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
                const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                const int op = __shfl_xor_sync(0xffffffffu, bpos, o);
                if (better(ov, oi, bv, bi)) { bv = ov; bi = oi; bpos = op; }
            }
            if (lane == 0) { s_topv[round] = bv; s_topi[round] = bi; if (bpos >= 0) { s_cv[bpos] = -INFINITY; s_ci[bpos] = 0x7fffffff; } }
            __syncwarp();
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int nlive = 0;
        float bs = best_score[img];
        for (int j = 0; j < ksel; ++j) {
            const int idx = s_topi[j];
            const float val = s_topv[j];
            const int prev = idx / V, next = idx % V;                                        // :85-86
            if (trace_s) trace_s[img * k + j] = next;                                        // :91
            if (next == end_id) {                                                            // :93-103
                if (val > bs) { bs = val; best_score[img] = val; best_step[img] = step; best_parent[img] = prev; }
            } else {                                                                         // :109-116
                const int r = slot * k + nlive, ri = img * k + nlive;
                src[r] = prev; score_tmp[r] = val; word_tmp[r] = next;
                parent_s[ri] = prev; word_s[ri] = next;
                ++nlive;
            }
        }
        k_live_tmp[slot] = nlive;                                                            // :104
        slot_img_tmp[slot] = img;
    }
}

// Compaction map after a step: new_slot[s] = rank of slot s among the slots that still have live beams (-1: finished or
// beyond the previous live count); n_live = {live slots, live rows}.  One CTA, block-wide scan in chunks of 1024 slots.
__global__ void __launch_bounds__(1024) beam_compact_kernel(int n_img, int k, const int* __restrict__ k_live_tmp,
                                                            int* __restrict__ new_slot, int* __restrict__ n_live,
                                                            int* __restrict__ row_off_new) {
    __shared__ int s_warp[32], s_wrow[32];
    __shared__ int s_carry, s_rcarry;
    const int n_prev = n_live[0];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) { s_carry = 0; s_rcarry = 0; }
    __syncthreads();
    for (int base = 0; base < n_img; base += 1024) {
        const int s = base + threadIdx.x;
        const int kl = (s < n_prev) ? k_live_tmp[s] : 0;
        const int flag = kl > 0 ? 1 : 0;
        int incl = flag, rincl = kl;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o), rv = __shfl_up_sync(0xffffffffu, rincl, o);
            if (lane >= o) { incl += v; rincl += rv; }
        }
        if (lane == 31) { s_warp[warp] = incl; s_wrow[warp] = rincl; }
        __syncthreads();
        if (warp == 0) {
            int w = s_warp[lane], rw = s_wrow[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_up_sync(0xffffffffu, w, o), rv = __shfl_up_sync(0xffffffffu, rw, o);
                if (lane >= o) { w += v; rw += rv; }
            }
            s_warp[lane] = w; s_wrow[lane] = rw;
        }
        __syncthreads();
        const int before = s_carry + (warp > 0 ? s_warp[warp - 1] : 0) + incl - flag;
        const int rbefore = s_rcarry + (warp > 0 ? s_wrow[warp - 1] : 0) + rincl - kl;
        if (s < n_img) new_slot[s] = flag ? before : -1;
        if (flag) row_off_new[before] = rbefore;                     // first state row of the compacted slot
        __syncthreads();
        if (threadIdx.x == 1023) { s_carry += s_warp[31]; s_rcarry += s_wrow[31]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { n_live[0] = s_carry; n_live[1] = s_rcarry; }
}

// Move the surviving beams of old slot s to its compacted slot new_slot[s]: h / c rows follow the parent pointers (:109-110),
// the small per-row state (score, previous word) and the per-slot state (live count, image) move with them.  Reads only
// *_tmp / h_tmp / c_tmp, writes only the current arrays, so the moves of different slots never collide.
__global__ void beam_reorder_kernel(int k, int D, const int* __restrict__ new_slot, const int* __restrict__ k_live_tmp,
                                    const int* __restrict__ slot_img_tmp, const int* __restrict__ src,
                                    const float* __restrict__ score_tmp, const int* __restrict__ word_tmp,
                                    const float* __restrict__ h_tmp, const float* __restrict__ c_tmp,
                                    float* __restrict__ h, float* __restrict__ c, float* __restrict__ score,
                                    int* __restrict__ prev_word, long long* __restrict__ tok64,
                                    int* __restrict__ k_live, int* __restrict__ slot_img,
                                    const int* __restrict__ row_off_old, const int* __restrict__ row_off_new,
                                    const int* __restrict__ tag_tmp, int* __restrict__ tag) {   // tag: optional (sampler)
    const int r = blockIdx.x;                       // (old slot, surviving beam j): index into the *_tmp arrays
    const int s = r / k, j = r % k;
    const int dslot = new_slot[s];
    if (dslot < 0) return;
    const int kl = k_live_tmp[s];
    if (j >= kl) return;
    const int dr = row_off_new[dslot] + j;
    const long long so = ((long long)row_off_old[s] + src[r]) * D, dst = (long long)dr * D;
    for (int dd = threadIdx.x; dd < D; dd += blockDim.x) { h[dst + dd] = h_tmp[so + dd]; c[dst + dd] = c_tmp[so + dd]; }
    if (threadIdx.x == 0) {
        score[dr] = score_tmp[r];
        prev_word[dr] = word_tmp[r]; tok64[dr] = word_tmp[r];
        if (tag) tag[dr] = tag_tmp[r];
        if (j == 0) { k_live[dslot] = kl; slot_img[dslot] = slot_img_tmp[s]; }
    }
}

// Back-track the winner of each image.
__global__ void beam_finalize_kernel(int k, int P, int S1 /* max_steps+1 */, long long R, int start_id, int end_id,
                                     const float* __restrict__ best_score, const int* __restrict__ best_step,
                                     const int* __restrict__ best_parent, const int* __restrict__ parent,
                                     const int* __restrict__ word, const float* __restrict__ alpha_steps,
                                     int* __restrict__ out_len, int* __restrict__ out_seq, float* __restrict__ out_score,
                                     float* __restrict__ out_alpha) {
    const int img = blockIdx.x;
    const int S = best_step[img];
    const int W = S1 + 1;                           // out_seq row width = max_steps + 2
    __shared__ int s_slot[ICD_MAX_STEPS + 2];       // s_slot[s] = row (within image) whose alpha is frame s
    if (threadIdx.x == 0) {
        out_score[img] = best_score[img];
        if (S == 0) { out_len[img] = 0; }
        else {
            out_len[img] = S + 1;
            int* seq = out_seq + (long long)img * W;
            seq[0] = start_id; seq[S] = end_id;
            int cur = best_parent[img];             // slot (step S-1 numbering) the winner extended
            s_slot[S] = cur;
            for (int s = S - 1; s >= 1; --s) {
                const long long o = (long long)(s - 1) * R + (long long)img * k + cur;
                seq[s] = word[o];
                cur = parent[o];
                s_slot[s] = cur;
            }
        }
    }
    __syncthreads();
    if (S == 0 || !out_alpha) return;
    float* oa = out_alpha + (long long)img * W * P;
    for (int p = threadIdx.x; p < P; p += blockDim.x) oa[p] = 1.f;                           // :54 frame of ones
    for (int s = 1; s <= S; ++s) {
        const float* a = alpha_steps + ((long long)(s - 1) * R + (long long)img * k + s_slot[s]) * P;
        for (int p = threadIdx.x; p < P; p += blockDim.x) oa[(long long)s * P + p] = a[p];
    }
}

__global__ void gather_rows_kernel(const float* __restrict__ table_f32, const double* __restrict__ table_f64,
                                   const long long* __restrict__ tok, int E, float* __restrict__ out,
                                   const int* __restrict__ n_live) {
    const long long r = blockIdx.x;
    if (r >= n_live[1]) return;
    const long long t = tok[r];
    for (int e = threadIdx.x; e < E; e += blockDim.x)
        out[r * E + e] = table_f64 ? (float)table_f64[t * E + e] : table_f32[t * E + e];
}

// gates_pre[r, :] = embg[token_r, :] (= embedding(token) W_ih[:, :E]^T + b_ih, precomputed for the whole vocabulary) + the
// h W_hh^T + b_hh part of z: what the per-step embedding contraction produced, as one gather (:65, :70-71).
__global__ void beam_gates_init_kernel(const float* __restrict__ embg, const long long* __restrict__ tok, int G,
                                       const float* __restrict__ zhh, long long ldz, float* __restrict__ gates_pre,
                                       const int* __restrict__ n_live) {
    const long long r = blockIdx.x;
    if (r >= n_live[1]) return;
    const float4* src = reinterpret_cast<const float4*>(embg + tok[r] * G);
    const float4* zz = reinterpret_cast<const float4*>(zhh + r * ldz);
    float4* dst = reinterpret_cast<float4*>(gates_pre + r * G);
    for (int e = threadIdx.x; e < (G >> 2); e += blockDim.x) {
        const float4 a = src[e], b = zz[e];
        dst[e] = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
    }
}

// fp32-grade tier, once per call: ONE pass over a chunk of feature maps writes the 3-term bf16 split of every pixel row (the A
// operand of the enc_att projection, layout [a1 | a1 | a2 | a1 | a3 | a2] along K with segment length C, gemm_tc.cu) AND the pixel
// mean of init_hidden_state (gen_captions.py:62 -> models/attention.py:161) — the features are read once instead of twice.
// grid = (ceil(C/256), images), block = 256 = 4 pixel groups x 64 float4 lanes; the mean is summed exactly like
// weighted_pixel_sum_kernel (pixels p = g, g+4, ... per group, then g0 + g1 + g2 + g3, then / P): bit-identical to it.
__global__ void __launch_bounds__(256) split3_mean_kernel(int P, int C, const float* __restrict__ enc,
                                                          unsigned short* __restrict__ x3, float* __restrict__ mean,
                                                          int nseg /* 6: K-concatenated segments, 3: stored planes [a1 | a2 | a3] */) {
    __shared__ float4 s_part[3 * 64];
    const int img = blockIdx.y;
    const int lane = threadIdx.x & 63, grp = threadIdx.x >> 6;
    const int c = blockIdx.x * 256 + lane * 4;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c < C) {
        const float* base = enc + (long long)img * P * C + c;
        unsigned short* ob = x3 + (long long)img * P * nseg * C + c;
        const int pat[6] = {0, 0, 1, 0, 2, 1};
        for (int p0 = grp; p0 < P; p0 += 16) {
            float4 x[4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
                x[u] = (p0 + 4 * u < P) ? ld_stream_f4(base + (long long)(p0 + 4 * u) * C) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int p = p0 + 4 * u;
                if (p >= P) break;
                acc.x = fmaf(1.f, x[u].x, acc.x); acc.y = fmaf(1.f, x[u].y, acc.y);
                acc.z = fmaf(1.f, x[u].z, acc.z); acc.w = fmaf(1.f, x[u].w, acc.w);
                const float xs[4] = {x[u].x, x[u].y, x[u].z, x[u].w};
                unsigned short t[3][4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const __nv_bfloat16 b1 = __float2bfloat16_rn(xs[q]);
                    const float r1 = xs[q] - __bfloat162float(b1);
                    const __nv_bfloat16 b2 = __float2bfloat16_rn(r1);
                    const __nv_bfloat16 b3 = __float2bfloat16_rn(r1 - __bfloat162float(b2));
                    t[0][q] = __bfloat16_as_ushort(b1); t[1][q] = __bfloat16_as_ushort(b2); t[2][q] = __bfloat16_as_ushort(b3);
                }
                unsigned short* dst = ob + (long long)p * nseg * C;
#pragma unroll
                for (int sg = 0; sg < 6; ++sg) {
                    if (sg >= nseg) break;
                    const unsigned short* tt = t[nseg == 3 ? sg : pat[sg]];
                    *reinterpret_cast<uint2*>(dst + (long long)sg * C) =
                        make_uint2((unsigned)tt[0] | ((unsigned)tt[1] << 16), (unsigned)tt[2] | ((unsigned)tt[3] << 16));
                }
            }
        }
    }
    if (grp > 0) s_part[(grp - 1) * 64 + lane] = acc;
    __syncthreads();
    if (grp == 0 && c < C) {
#pragma unroll
        for (int g = 0; g < 3; ++g) { const float4 o = s_part[g * 64 + lane]; acc.x += o.x; acc.y += o.y; acc.z += o.z; acc.w += o.w; }
        const float inv = (float)P;
        acc.x /= inv; acc.y /= inv; acc.z /= inv; acc.w /= inv;
        *reinterpret_cast<float4*>(mean + (long long)img * C + c) = acc;
    }
}

// ---------------------------------------------------------------------------------------------- BaselineDecoder beam search
// Workspace of icd_baseline_beam_search: the fields of BeamWs the baseline step uses (state rows of H, z = h W_hh^T of 4H, logits, the
// whole-vocabulary embg, the bookkeeping of the shared top-k / compaction / reorder / finalize kernels) and the fp32x3 splits of
// W_ih (x3_WihE), W_hh (x3_Whh) and the vocabulary layer (x3_Wfc).
constexpr int BASE_EMBG_ROWS = 4096;      // vocabulary rows per embg pass (bounds the split activation scratch)

}  // namespace

size_t carve_base(const icd_base_beam_desc_t* d, BeamWs* w, char* base, bool history) {
    const size_t R = (size_t)d->n_img * d->k, S = (size_t)d->max_steps + 1;
    const int E = d->E, H = d->H, V = d->V, G = 4 * H;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~(size_t)255; return base ? base + o : (char*)nullptr; };
    float* f;
#define TAKE_F(name, n) f = (float*)take(sizeof(float) * (n)); if (w) w->name = f;
    TAKE_F(h0, (size_t)d->n_img * H) TAKE_F(c0, (size_t)d->n_img * H)
    TAKE_F(h, R * H) TAKE_F(c, R * H) TAKE_F(h_tmp, R * H) TAKE_F(c_tmp, R * H)
    TAKE_F(z, R * G)                                          // also the gates of the image step (n_img rows)
    TAKE_F(logits, R * V)
    TAKE_F(embg, (size_t)V * G)                               // embedding row x W_ih^T + b_ih + b_hh for EVERY token, once per call
    TAKE_F(emb32, d->emb_is_f64 ? (size_t)V * E : 0)
    TAKE_F(score, R) TAKE_F(score_tmp, R) TAKE_F(best_score, (size_t)d->n_img)
#undef TAKE_F
    int* ip;
#define TAKE_I(name, n) ip = (int*)take(sizeof(int) * (n)); if (w) w->name = ip;
    TAKE_I(img_index, R) TAKE_I(prev_word, R) TAKE_I(k_live, (size_t)d->n_img) TAKE_I(src, R)
    TAKE_I(parent, history ? S * R : 0) TAKE_I(word, history ? S * R : 0) TAKE_I(best_step, (size_t)d->n_img)
    TAKE_I(best_parent, (size_t)d->n_img)
    TAKE_I(slot_img, (size_t)d->n_img) TAKE_I(slot_img_tmp, (size_t)d->n_img) TAKE_I(k_live_tmp, (size_t)d->n_img)
    TAKE_I(new_slot, (size_t)d->n_img) TAKE_I(n_live, 4) TAKE_I(word_tmp, R)
    ip = (int*)take(sizeof(int) * (size_t)d->n_img); if (w) w->row_off[0] = ip;
    ip = (int*)take(sizeof(int) * (size_t)d->n_img); if (w) w->row_off[1] = ip;
    if (w) w->tag = w->tag_tmp = nullptr;
    if (!history) { TAKE_I(tag, R) TAKE_I(tag_tmp, R) }
#undef TAKE_I
    long long* lp = (long long*)take(sizeof(long long) * R); if (w) w->tok64 = lp;
    if (d->precision == ICD_PREC_FP32X3) {
        void* v;
#define TAKE_X3(name, rows, K) v = (void*)take((size_t)(rows) * 6 * up8ll(K) * 2); if (w) w->name = v;
        TAKE_X3(x3_WihE, G, E) TAKE_X3(x3_Whh, G, H) TAKE_X3(x3_Wfc, V, H)
#undef TAKE_X3
        const size_t ve = (size_t)(V < BASE_EMBG_ROWS ? V : BASE_EMBG_ROWS);
        size_t act_rows = R > ve ? R : ve;
        const long long kmax = E > H ? E : H;
        v = (void*)take(act_rows * 6 * up8ll(kmax) * 2); if (w) w->x3_act = v;
        long long nf = 0;
        const long long shapes[][3] = {{(long long)ve, G, 6 * up8ll(E)}, {(long long)d->n_img, G, 6 * up8ll(E)},
                                       {(long long)R, G, 6 * up8ll(H)}, {(long long)R, V, 6 * up8ll(H)}};
        for (const auto& sh : shapes) { const long long n = icd_gemm_bf16_splitk_floats((int)sh[0], (int)sh[1], (int)sh[2]); if (n > nf) nf = n; }
        float* fp = (float*)take(sizeof(float) * (size_t)nf);
        if (w) { w->x3_splitk = fp; w->x3_splitk_floats = nf; }
    }
    return off;
}

namespace {

// The baseline decoder's step after the W_hh contraction, one CTA per live row r:
//   gates = embg[tok[r]] + z[r]   (embg = emb W_ih^T + b_ih + b_hh for the whole vocabulary, z = h W_hh^T of this step)
// then the LSTMCell with the activation code of lstm_pointwise_fwd_kernel (pointwise.cu) -> h_new, c_new.  In the fp32-grade tier
// it also writes the 3-term bf16 split of h_new (rounding of icd_split3_bf16) into x3 — rows of nseg * up8(H): 3 stored planes
// [t1 | t2 | t3] or the 6-segment A pattern [a1 | a1 | a2 | a1 | a3 | a2] (gemm_tc.cu), pad columns zero — which the vocabulary
// contraction then consumes with pre_split.  embg == NULL: gates = z[r] (the image step); c_prev == NULL: the zero state.
__global__ void __launch_bounds__(128) baseline_beam_cell_kernel(int H, const float* __restrict__ embg,
                                                                  const long long* __restrict__ tok, const float* __restrict__ z,
                                                                  const float* __restrict__ c_prev, float* __restrict__ c_new,
                                                                  float* __restrict__ h_new, unsigned short* __restrict__ x3,
                                                                  int nseg, const int* __restrict__ n_live) {
    const long long r = blockIdx.x;
    if (n_live && r >= n_live[1]) return;
    const int G = 4 * H, seg = (H + 7) / 8 * 8;
    const float* e = embg ? embg + tok[r] * G : nullptr;
    const float* zr = z + r * G;
    for (int col = 4 * threadIdx.x; col < seg; col += 4 * blockDim.x) {
        float hv[4] = {0.f, 0.f, 0.f, 0.f};
        if (col < H) {                                        // H % 4 == 0: a group of four is all data or all padding
            float4 g[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                g[q] = *reinterpret_cast<const float4*>(zr + q * H + col);
                if (e) {
                    const float4 a = *reinterpret_cast<const float4*>(e + q * H + col);
                    g[q] = make_float4(a.x + g[q].x, a.y + g[q].y, a.z + g[q].z, a.w + g[q].w);
                }
            }
            const float4 cp = c_prev ? *reinterpret_cast<const float4*>(c_prev + r * H + col) : make_float4(0.f, 0.f, 0.f, 0.f);
            const float gi[4] = {g[0].x, g[0].y, g[0].z, g[0].w}, gf[4] = {g[1].x, g[1].y, g[1].z, g[1].w};
            const float gg[4] = {g[2].x, g[2].y, g[2].z, g[2].w}, go[4] = {g[3].x, g[3].y, g[3].z, g[3].w};
            const float cpv[4] = {cp.x, cp.y, cp.z, cp.w};
            float cv[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float i = sigmoidf_(gi[u]);
                const float f = sigmoidf_(gf[u]);
                const float gt = tanhf(gg[u]);
                const float o = sigmoidf_(go[u]);
                cv[u] = f * cpv[u] + i * gt;
                hv[u] = o * tanhf(cv[u]);
            }
            *reinterpret_cast<float4*>(c_new + r * H + col) = make_float4(cv[0], cv[1], cv[2], cv[3]);
            *reinterpret_cast<float4*>(h_new + r * H + col) = make_float4(hv[0], hv[1], hv[2], hv[3]);
        }
        if (x3) {
            unsigned short t[3][4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const __nv_bfloat16 b1 = __float2bfloat16_rn(hv[u]);
                const float r1 = hv[u] - __bfloat162float(b1);
                const __nv_bfloat16 b2 = __float2bfloat16_rn(r1);
                const __nv_bfloat16 b3 = __float2bfloat16_rn(r1 - __bfloat162float(b2));
                t[0][u] = __bfloat16_as_ushort(b1); t[1][u] = __bfloat16_as_ushort(b2); t[2][u] = __bfloat16_as_ushort(b3);
            }
            const int pat[6] = {0, 0, 1, 0, 2, 1};
            unsigned short* dst = x3 + r * nseg * seg + col;
#pragma unroll
            for (int sg = 0; sg < 6; ++sg) {
                if (sg >= nseg) break;
                const unsigned short* tt = t[nseg == 3 ? sg : pat[sg]];
                *reinterpret_cast<uint2*>(dst + (long long)sg * seg) =
                    make_uint2((unsigned)tt[0] | ((unsigned)tt[1] << 16), (unsigned)tt[2] | ((unsigned)tt[3] << 16));
            }
        }
    }
}

__global__ void f64_to_f32_kernel(const double* __restrict__ src, long long n, float* __restrict__ dst) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        dst[i] = (float)src[i];
}

}  // namespace

// y[rows, N] = x[rows, K] * W[N, K]^T (+ bias + add + beta*y): fp32 FMA kernel, or the fp32-grade tensor-core tier with the
// activation split on the fly and the weight split `w16x3` prepared once per call.
int beam_mm(int prec, const BeamWs& w, const float* x, long long ldx, int rows, int K, const float* W, long long ldw,
            const void* w16x3, float* y, long long ldy, int N, const float* bias, const float* add, long long ldadd,
            float beta, cudaStream_t s, const int* m_live = nullptr, bool pre_split = false, const float* bias2 = nullptr) {
    // m_live: device-side count of live rows (compacted to the front).  The tensor-core tier computes only those; the fp32
    // FMA tier computes all `rows` (rows beyond the live count hold stale, finite state and are never read back).
    if (prec != ICD_PREC_FP32X3)
        return icd_gemm_simple(ICD_PREC_FP32, x, ldx, 1, W, ldw, 1, y, ldy, rows, N, K, bias, bias2, add, ldadd, nullptr, 0,
                               nullptr, beta, s);
    // three stored planes per operand where a segment is a whole number of k-blocks (gemm_tc.cuh), else the six-segment layout;
    // the weight splits of the call (w16x3) and the fused producers of w.x3_act follow the same rule
    const long long seg = up8ll(K);
    const bool p3 = icd_x3_three_planes(K);
    const long long ld3 = (p3 ? 3 : 6) * seg;
    if (!pre_split) ICD_TRY(icd_split3_bf16(x, ldx, rows, K, w.x3_act, p3 ? 2 : 0, s, m_live));   // (pre_split: the producer wrote w.x3_act)
    if (p3) icd_gemm_x3_planes((int)(seg / 64), (int)(seg / 64));
    const int rc = icd_gemm_bf16_ex(w.x3_act, ld3, 0, w16x3, ld3, 0, y, ldy, rows, N, (int)(6 * seg), bias, bias2, add, ldadd,
                                    nullptr, 0, nullptr, beta, s, nullptr, 0, w.x3_splitk, w.x3_splitk_floats, nullptr, m_live);
    icd_gemm_x3_planes(0, 0);
    return rc;
}

int beam_att_prologue(const icd_beam_desc_t* d, BeamWs& w, bool* use_embg_out, cudaStream_t s) {
    const int n_img = d->n_img, P = d->P, C = d->C, A = d->A, D = d->D, E = d->E, V = d->V;
    const int NZ = A + C + 4 * D, prec = d->precision;
    ICD_CUDA(cudaMemcpyAsync(w.w_cat, d->dec_att_w, sizeof(float) * (size_t)A * D, cudaMemcpyDeviceToDevice, s));
    ICD_CUDA(cudaMemcpyAsync(w.w_cat + (size_t)A * D, d->f_beta_w, sizeof(float) * (size_t)C * D, cudaMemcpyDeviceToDevice, s));
    ICD_CUDA(cudaMemcpyAsync(w.w_cat + (size_t)(A + C) * D, d->w_hh, sizeof(float) * (size_t)4 * D * D, cudaMemcpyDeviceToDevice, s));
    ICD_CUDA(cudaMemcpyAsync(w.b_cat, d->dec_att_b, sizeof(float) * A, cudaMemcpyDeviceToDevice, s));
    ICD_CUDA(cudaMemcpyAsync(w.b_cat + A, d->f_beta_b, sizeof(float) * C, cudaMemcpyDeviceToDevice, s));
    ICD_CUDA(cudaMemcpyAsync(w.b_cat + A + C, d->b_hh, sizeof(float) * 4 * D, cudaMemcpyDeviceToDevice, s));

    // once per image: enc_att projection and the initial state (:62)
    ICD_CHECK_ARG(prec == ICD_PREC_FP32 || prec == ICD_PREC_FP32X3, "beam_search: precision must be ICD_PREC_FP32 or ICD_PREC_FP32X3");
    if (prec == ICD_PREC_FP32X3) {            // weights are constant over the whole search: split them once
        ICD_TRY(icd_split3_bf16(d->enc_att_w, C, A, C, w.x3_We, icd_x3_three_planes(C) ? 2 : 1, s));
        ICD_TRY(icd_split3_bf16(w.w_cat, D, NZ, D, w.x3_Wcat, icd_x3_three_planes(D) ? 2 : 1, s));
        ICD_TRY(icd_split3_bf16(d->w_ih, E + C, 4 * D, E, w.x3_WihE, icd_x3_three_planes(E) ? 2 : 1, s));
        ICD_TRY(icd_split3_bf16(d->w_ih + E, E + C, 4 * D, C, w.x3_WihC, icd_x3_three_planes(C) ? 2 : 1, s));
        ICD_TRY(icd_split3_bf16(d->h_lin_w, C, D, C, w.x3_Wh, icd_x3_three_planes(C) ? 2 : 1, s));
        ICD_TRY(icd_split3_bf16(d->c_lin_w, C, D, C, w.x3_Wc, icd_x3_three_planes(C) ? 2 : 1, s));
        ICD_TRY(icd_split3_bf16(d->fc_w, D, V, D, w.x3_Wfc, icd_x3_three_planes(D) ? 2 : 1, s));
    }
    // embedding -> gate contribution for the whole vocabulary, once per call: V rows instead of (live rows) x (steps) rows, and
    // no per-step activation split of the embedding rows (fp32 tables; an fp64 GloVe table keeps the per-step contraction)
    const bool use_embg = !d->emb_is_f64 && (NZ % 4 == 0) && ((A + C) % 4 == 0);
    *use_embg_out = use_embg;
    if (use_embg) {
        const int VC = 4096;                                 // rows per pass: bounds the split scratch (x3_act holds >= 64*P rows of C)
        for (int v0 = 0; v0 < V; v0 += VC) {
            const int nv = V - v0 < VC ? V - v0 : VC;
            ICD_TRY(beam_mm(prec, w, (const float*)d->emb_w + (size_t)v0 * E, E, nv, E, d->w_ih, E + C, w.x3_WihE,
                            w.embg + (size_t)v0 * 4 * D, 4 * D, 4 * D, d->b_ih, nullptr, 0, 0.f, s));
        }
    }
    const int img_chunk = prec == ICD_PREC_FP32X3 ? x3_img_chunk(P, A) : X3_IMG_CHUNK;
    const bool fused_mean = prec == ICD_PREC_FP32X3 && C % 8 == 0 && (reinterpret_cast<uintptr_t>(d->enc) & 15) == 0 &&
                            getenv("ICD_BEAM_FUSED_MEAN_OFF") == nullptr;
    for (int i0 = 0; i0 < n_img; i0 += img_chunk) {          // att_enc = enc_att(enc), once per image
        const int ni = n_img - i0 < img_chunk ? n_img - i0 : img_chunk;
        if (fused_mean) {                 // split of the chunk's pixel rows + the pixel mean of its images in one pass over the features
            split3_mean_kernel<<<dim3((unsigned)((C + 255) / 256), (unsigned)ni), 256, 0, s>>>(
                P, C, d->enc + (size_t)i0 * P * C, reinterpret_cast<unsigned short*>(w.x3_act), w.mean + (size_t)i0 * C,
                icd_x3_three_planes(C) ? 3 : 6);
            ICD_LAUNCH_CHECK();
        }
        ICD_TRY(beam_mm(prec, w, d->enc + (size_t)i0 * P * C, C, ni * P, C, d->enc_att_w, C, w.x3_We,
                        w.att_enc + (size_t)i0 * P * A, A, A, d->enc_att_b, nullptr, 0, 0.f, s, nullptr, fused_mean));
    }
    // initial state (:62): pixel mean, h_lin, c_lin
    if (!fused_mean)
        ICD_TRY(icd_weighted_pixel_sum(n_img, P, C, nullptr, d->enc, nullptr, 0, nullptr, 0, w.mean, nullptr, nullptr, s));
    ICD_TRY(beam_mm(prec, w, w.mean, C, n_img, C, d->h_lin_w, C, w.x3_Wh, w.h0, D, D, d->h_lin_b, nullptr, 0, 0.f, s));
    ICD_TRY(beam_mm(prec, w, w.mean, C, n_img, C, d->c_lin_w, C, w.x3_Wc, w.c0, D, D, d->c_lin_b, nullptr, 0, 0.f, s));
    return 0;
}

int beam_att_step(const icd_beam_desc_t* d, BeamWs& w, int step, bool use_embg, const int* row_off, float* alpha_s, cudaStream_t s) {
    const int n_img = d->n_img, k = d->k, P = d->P, C = d->C, A = d->A, D = d->D, E = d->E, V = d->V;
    const int NZ = A + C + 4 * D, prec = d->precision;
    const long long R = (long long)n_img * k;
    const int* live_rows = w.n_live + 1;
    if (!use_embg) {
        gather_rows_kernel<<<(unsigned)R, 128, 0, s>>>(d->emb_is_f64 ? nullptr : (const float*)d->emb_w,
                                                       d->emb_is_f64 ? (const double*)d->emb_w : nullptr,
                                                       w.tok64, E, w.emb_x, w.n_live);       // :65
        ICD_LAUNCH_CHECK();
    }
    ICD_TRY(beam_mm(prec, w, w.h, D, (int)R, D, w.w_cat, D, w.x3_Wcat, w.z, NZ, NZ, w.b_cat, nullptr, 0, 0.f, s, live_rows));
    // :66-69 — one CTA per live slot serves all of its live beams (features read once per image and step)
    // fp32-grade tensor-core tier: the attention kernel emits the 3-term bf16 split of `gated` itself (the A operand of the
    // gate contraction below), so neither the fp32 copy nor a split pass over (rows, C) is needed
    const bool fused_split = prec == ICD_PREC_FP32X3 && use_embg && (C % 8 == 0);
    ICD_TRY(icd_attention_step_fwd_grouped(n_img, k, P, C, A, w.k_live, d->enc, w.att_enc, w.z, NZ, d->full_att_w,
                                           d->full_att_b, w.z + A, NZ, alpha_s, P, fused_split ? nullptr : w.gated, w.slot_img,
                                           w.n_live, row_off, s, fused_split ? w.x3_act : nullptr, w.ring_ticket + step,
                                           icd_x3_three_planes(C) ? 3 : 6));
    if (use_embg) {
        beam_gates_init_kernel<<<(unsigned)R, 128, 0, s>>>(w.embg, w.tok64, 4 * D, w.z + A + C, NZ, w.gates_pre, w.n_live);
        ICD_LAUNCH_CHECK();
    } else
        ICD_TRY(beam_mm(prec, w, w.emb_x, E, (int)R, E, d->w_ih, E + C, w.x3_WihE, w.gates_pre, 4 * D, 4 * D,
                        d->b_ih, w.z + A + C, NZ, 0.f, s, live_rows));
    ICD_TRY(beam_mm(prec, w, w.gated, C, (int)R, C, d->w_ih + E, E + C, w.x3_WihC, w.gates_pre, 4 * D, 4 * D,
                    nullptr, nullptr, 0, 1.f, s, live_rows, fused_split));               // :70-71
    ICD_TRY(icd_lstm_pointwise_fwd((int)R, D, w.gates_pre, w.c, nullptr, w.c_tmp, w.h_tmp, nullptr, 0, nullptr, 1.f, s,
                                   nullptr, nullptr, live_rows));
    ICD_TRY(beam_mm(prec, w, w.h_tmp, D, (int)R, D, d->fc_w, D, w.x3_Wfc, w.logits, V, V, d->fc_b, nullptr, 0, 0.f, s, live_rows));   // :72
    return 0;
}

int beam_launch_init(int n_img, int k, int D, int start_id, BeamWs& w, cudaStream_t s) {
    const long long n = (long long)n_img * k * D;
    beam_init_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(n_img, k, D, start_id, w.h0, w.c0, w.h, w.c,
                                                                  w.img_index, w.prev_word, w.tok64, w.score, w.k_live,
                                                                  w.best_score, w.best_step, w.best_parent,
                                                                  w.slot_img, w.n_live, w.row_off[0]);
    ICD_LAUNCH_CHECK();
    return 0;
}

int beam_launch_advance(int n_img, int k, int D, BeamWs& w, const int* row_off, int* row_off_next, cudaStream_t s) {
    beam_compact_kernel<<<1, 1024, 0, s>>>(n_img, k, w.k_live_tmp, w.new_slot, w.n_live, row_off_next);
    ICD_LAUNCH_CHECK();
    beam_reorder_kernel<<<(unsigned)((long long)n_img * k), 128, 0, s>>>(k, D, w.new_slot, w.k_live_tmp, w.slot_img_tmp, w.src,
                                                                         w.score_tmp, w.word_tmp, w.h_tmp, w.c_tmp, w.h, w.c,
                                                                         w.score, w.prev_word, w.tok64, w.k_live, w.slot_img,
                                                                         row_off, row_off_next, w.tag_tmp, w.tag);
    ICD_LAUNCH_CHECK();
    return 0;
}

extern "C" int64_t icd_beam_search_ws_bytes(const icd_beam_desc_t* d) {
    if (!d) return -1;
    return (int64_t)carve(d, nullptr, nullptr);
}

extern "C" int icd_beam_search(const icd_beam_desc_t* d, void* stream) {
    ICD_CHECK_ARG(d != nullptr, "beam_search: null descriptor");
    ICD_CHECK_ARG(d->n_img > 0 && d->k >= 1 && d->k <= KMAX, "beam_search: n_img=%d k=%d (k <= %d)", d->n_img, d->k, KMAX);
    ICD_CHECK_ARG(d->max_steps >= 1 && d->max_steps + 1 <= ICD_MAX_STEPS, "beam_search: max_steps=%d out of range", d->max_steps);
    ICD_CHECK_ARG(d->V >= d->k, "beam_search: vocabulary smaller than the beam");
    ICD_CHECK_ARG(d->A % 4 == 0 && d->C % 4 == 0 && d->D % 4 == 0 && d->E % 4 == 0, "beam_search: dims must be multiples of 4");
    ICD_CHECK_ARG(d->ws && d->ws_bytes >= icd_beam_search_ws_bytes(d), "beam_search: workspace too small");
    cudaStream_t s = icd_stream(stream);
    BeamWs w;
    carve(d, &w, (char*)d->ws);
    const int n_img = d->n_img, k = d->k, P = d->P, D = d->D, V = d->V;
    const long long R = (long long)n_img * k;
    ICD_CHECK_ARG(R <= 65535, "beam_search: n_img*k=%lld exceeds 65535 rows per call (chunk the images)", R);
    const int S1 = d->max_steps + 1;

    bool use_embg = false;
    ICD_TRY(beam_att_prologue(d, w, &use_embg, s));
    ICD_TRY(beam_launch_init(n_img, k, D, d->start_id, w, s));
    // candidate words of images that are already finished at a step stay -1 (:91 prints nothing for them)
    if (d->trace_words) ICD_CUDA(cudaMemsetAsync(d->trace_words, 0xff, sizeof(int32_t) * (size_t)S1 * R, s));
    ICD_CUDA(cudaMemsetAsync(w.ring_ticket, 0, sizeof(int) * (size_t)(S1 + 2), s));
    for (int step = 1; step <= S1; ++step) {
        float* alpha_s = w.alpha_steps + (size_t)(step - 1) * R * P;
        const int* row_off = w.row_off[(step - 1) & 1];
        int* row_off_next = w.row_off[step & 1];
        ICD_TRY(beam_att_step(d, w, step, use_embg, row_off, alpha_s, s));
#define ICD_TOPK(KT) beam_topk_kernel<KT><<<n_img, 256, 0, s>>>(k, V, step, d->end_id, w.logits, w.score, w.k_live, w.slot_img, w.n_live, \
                                               row_off, w.score_tmp, w.word_tmp, w.k_live_tmp, w.slot_img_tmp, w.src,                   \
                                               w.parent + (size_t)(step - 1) * R, w.word + (size_t)(step - 1) * R,                      \
                                               d->trace_words ? d->trace_words + (size_t)(step - 1) * R : nullptr,                      \
                                               w.best_score, w.best_step, w.best_parent, topk_stream_only)
        const int topk_stream_only = getenv("ICD_BEAM_TOPK_STREAM") != nullptr;      // test hook: the streaming pass for every row
        switch (k) {
            case 1: ICD_TOPK(1); break;
            case 2: ICD_TOPK(2); break;
            case 3: ICD_TOPK(3); break;
            case 4: ICD_TOPK(4); break;
            case 5: ICD_TOPK(5); break;
            case 6: ICD_TOPK(6); break;
            default: ICD_TOPK(8); break;
        }
#undef ICD_TOPK
        ICD_LAUNCH_CHECK();
        ICD_TRY(beam_launch_advance(n_img, k, D, w, row_off, row_off_next, s));
    }
    beam_finalize_kernel<<<n_img, 128, 0, s>>>(k, P, S1, R, d->start_id, d->end_id, w.best_score, w.best_step,
                                               w.best_parent, w.parent, w.word, w.alpha_steps, d->out_len, d->out_seq,
                                               d->out_score, d->out_alpha);
    ICD_LAUNCH_CHECK();
    return 0;
}

static int base_beam_shape_check(const icd_base_beam_desc_t* d) {
    ICD_CHECK_ARG(d != nullptr, "baseline_beam_search: null descriptor");
    ICD_CHECK_ARG(d->n_img > 0 && d->k >= 1 && d->k <= KMAX, "baseline_beam_search: n_img=%d k=%d (k in 1..%d)", d->n_img, d->k, KMAX);
    ICD_CHECK_ARG(d->max_steps >= 1 && d->max_steps + 1 <= ICD_MAX_STEPS, "baseline_beam_search: max_steps=%d out of range", d->max_steps);
    ICD_CHECK_ARG(d->V >= d->k, "baseline_beam_search: vocabulary (%d) smaller than the beam (%d)", d->V, d->k);
    ICD_CHECK_ARG(d->E > 0 && d->H > 0 && d->E % 4 == 0 && d->H % 4 == 0, "baseline_beam_search: E=%d H=%d must be positive multiples of 4",
                  d->E, d->H);
    ICD_CHECK_ARG((long long)d->n_img * d->k <= 65535, "baseline_beam_search: n_img*k=%lld exceeds 65535 rows per call (chunk the images)",
                  (long long)d->n_img * d->k);
    ICD_CHECK_ARG(d->precision == ICD_PREC_FP32 || d->precision == ICD_PREC_FP32X3,
                  "baseline_beam_search: precision must be ICD_PREC_FP32 or ICD_PREC_FP32X3 (identical captions need fp32-grade logits)");
    return 0;
}

static int base_beam_check(const icd_base_beam_desc_t* d) {
    ICD_TRY(base_beam_shape_check(d));
    ICD_CHECK_ARG(d->start_id >= 0 && d->start_id < d->V && d->end_id >= 0 && d->end_id < d->V,
                  "baseline_beam_search: start_id / end_id outside the vocabulary");
    ICD_CHECK_ARG(d->img_features && d->emb_w && d->w_ih && d->w_hh && d->b_ih && d->b_hh && d->lin_w && d->lin_b,
                  "baseline_beam_search: null input or weight");
    ICD_CHECK_ARG(d->out_len && d->out_seq && d->out_score, "baseline_beam_search: null result pointer");
    ICD_CHECK_ARG(d->ws && d->ws_bytes >= (int64_t)carve_base(d, nullptr, nullptr), "baseline_beam_search: workspace too small");
    return 0;
}

extern "C" int64_t icd_baseline_beam_search_ws_bytes(const icd_base_beam_desc_t* d) {
    if (base_beam_shape_check(d) != 0) return -1;         // (the reason is in icd_last_error_string)
    return (int64_t)carve_base(d, nullptr, nullptr);
}

int beam_base_prologue(const icd_base_beam_desc_t* d, BeamWs& w, cudaStream_t s) {
    const int n_img = d->n_img, E = d->E, H = d->H, V = d->V, G = 4 * H, prec = d->precision;
    if (prec == ICD_PREC_FP32X3) {                        // weights are constant over the whole search: split them once
        ICD_TRY(icd_split3_bf16(d->w_ih, E, G, E, w.x3_WihE, icd_x3_three_planes(E) ? 2 : 1, s));
        ICD_TRY(icd_split3_bf16(d->w_hh, H, G, H, w.x3_Whh, icd_x3_three_planes(H) ? 2 : 1, s));
        ICD_TRY(icd_split3_bf16(d->lin_w, H, V, H, w.x3_Wfc, icd_x3_three_planes(H) ? 2 : 1, s));
    }
    // an fp64 table is cast to fp32 once (the forward casts the rows it reads, models/baseline.py:101), so it takes the embg path too
    const float* emb = (const float*)d->emb_w;
    if (d->emb_is_f64) {
        const long long n = (long long)V * E;
        const long long blocks = (n + 255) / 256 < 4 * ICD_NUM_SMS ? (n + 255) / 256 : 4 * ICD_NUM_SMS;
        f64_to_f32_kernel<<<(unsigned)blocks, 256, 0, s>>>((const double*)d->emb_w, n, w.emb32);
        ICD_LAUNCH_CHECK();
        emb = w.emb32;
    }
    // embg = emb W_ih^T + b_ih + b_hh for the whole vocabulary, once per call: the per-step input contraction becomes a row gather
    for (int v0 = 0; v0 < V; v0 += BASE_EMBG_ROWS) {
        const int nv = V - v0 < BASE_EMBG_ROWS ? V - v0 : BASE_EMBG_ROWS;
        ICD_TRY(beam_mm(prec, w, emb + (size_t)v0 * E, E, nv, E, d->w_ih, E, w.x3_WihE, w.embg + (size_t)v0 * G, G, G, d->b_ih,
                        nullptr, 0, 0.f, s, nullptr, false, d->b_hh));
    }
    // step 0 (models/baseline.py:101,106): the image feature through one LSTM step from the zero state; its logits are not scored
    ICD_TRY(beam_mm(prec, w, d->img_features, E, n_img, E, d->w_ih, E, w.x3_WihE, w.z, G, G, d->b_ih, nullptr, 0, 0.f, s, nullptr,
                    false, d->b_hh));
    baseline_beam_cell_kernel<<<(unsigned)n_img, 128, 0, s>>>(H, nullptr, nullptr, w.z, nullptr, w.c0, w.h0, nullptr, 0, nullptr);
    ICD_LAUNCH_CHECK();
    return 0;
}

int beam_base_step(const icd_base_beam_desc_t* d, BeamWs& w, cudaStream_t s) {
    const int H = d->H, V = d->V, G = 4 * H, prec = d->precision;
    const long long R = (long long)d->n_img * d->k;
    const bool x3 = prec == ICD_PREC_FP32X3;
    const int nseg = icd_x3_three_planes(H) ? 3 : 6;     // layout of the split of h_tmp the cell kernel writes (= beam_mm's)
    const int* live_rows = w.n_live + 1;
    ICD_TRY(beam_mm(prec, w, w.h, H, (int)R, H, d->w_hh, H, w.x3_Whh, w.z, G, G, nullptr, nullptr, 0, 0.f, s, live_rows));
    baseline_beam_cell_kernel<<<(unsigned)R, 128, 0, s>>>(H, w.embg, w.tok64, w.z, w.c, w.c_tmp, w.h_tmp,
                                                          x3 ? reinterpret_cast<unsigned short*>(w.x3_act) : nullptr, nseg, w.n_live);
    ICD_LAUNCH_CHECK();
    ICD_TRY(beam_mm(prec, w, w.h_tmp, H, (int)R, H, d->lin_w, H, w.x3_Wfc, w.logits, V, V, d->lin_b, nullptr, 0, 0.f, s, live_rows,
                    x3));
    return 0;
}

extern "C" int icd_baseline_beam_search(const icd_base_beam_desc_t* d, void* stream) {
    ICD_TRY(base_beam_check(d));                          // every argument before the first CUDA call
    cudaStream_t s = icd_stream(stream);
    BeamWs w;
    carve_base(d, &w, (char*)d->ws);
    const int n_img = d->n_img, k = d->k, H = d->H, V = d->V;
    const long long R = (long long)n_img * k;
    const int S1 = d->max_steps + 1;

    ICD_TRY(beam_base_prologue(d, w, s));
    ICD_TRY(beam_launch_init(n_img, k, H, d->start_id, w, s));
    if (d->trace_words) ICD_CUDA(cudaMemsetAsync(d->trace_words, 0xff, sizeof(int32_t) * (size_t)S1 * R, s));
    for (int step = 1; step <= S1; ++step) {               // steps 1 .. max_steps+1: the state machine of icd_beam_search
        const int* row_off = w.row_off[(step - 1) & 1];
        int* row_off_next = w.row_off[step & 1];
        ICD_TRY(beam_base_step(d, w, s));
#define ICD_BASE_TOPK(KT) beam_topk_kernel<KT><<<n_img, 256, 0, s>>>(k, V, step, d->end_id, w.logits, w.score, w.k_live, w.slot_img,     \
                                               w.n_live, row_off, w.score_tmp, w.word_tmp, w.k_live_tmp, w.slot_img_tmp, w.src,      \
                                               w.parent + (size_t)(step - 1) * R, w.word + (size_t)(step - 1) * R,                   \
                                               d->trace_words ? d->trace_words + (size_t)(step - 1) * R : nullptr,                   \
                                               w.best_score, w.best_step, w.best_parent, 0)
        switch (k) {
            case 1: ICD_BASE_TOPK(1); break;
            case 2: ICD_BASE_TOPK(2); break;
            case 3: ICD_BASE_TOPK(3); break;
            case 4: ICD_BASE_TOPK(4); break;
            case 5: ICD_BASE_TOPK(5); break;
            case 6: ICD_BASE_TOPK(6); break;
            default: ICD_BASE_TOPK(8); break;
        }
#undef ICD_BASE_TOPK
        ICD_LAUNCH_CHECK();
        ICD_TRY(beam_launch_advance(n_img, k, H, w, row_off, row_off_next, s));
    }
    beam_finalize_kernel<<<n_img, 128, 0, s>>>(k, 0, S1, R, d->start_id, d->end_id, w.best_score, w.best_step, w.best_parent,
                                               w.parent, w.word, nullptr, d->out_len, d->out_seq, d->out_score, nullptr);
    ICD_LAUNCH_CHECK();
    return 0;
}
