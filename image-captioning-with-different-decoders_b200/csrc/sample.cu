// Seeded, batched caption sampling (temperature, top-k) for both decoders: icd_sample_captions (attention decoder) and
// icd_baseline_sample_captions (BaselineDecoder).  The definition of a sample is in include/icd_b200.h.
//
// The decoder computation is the beam search's (beam.cuh): the same once-per-call prologue, the same per-step contractions,
// attention / cell kernels and vocabulary layer on the live rows, and the same slot state machine — one slot per unfinished
// image whose live rows (here: samples) occupy consecutive rows, compacted after every step by beam_compact_kernel /
// beam_reorder_kernel, with each row's sample index travelling in w.tag.  Only the selection differs: sample_select_kernel
// draws instead of ranking, and writes each sample's tokens, log-probabilities and end state straight into the outputs, so the
// workspace holds no per-step history.  No host synchronisation inside the loop.
#include "beam.cuh"
#include <math.h>
#include <string.h>

namespace {

constexpr int SEL_THREADS = 256;
constexpr int SEL_NL = 19;            // = beam_topk_kernel's TOPK_NL: rows of up to 2 * 256 * 19 logits stay in registers
constexpr int MMAX = 8;               // samples per image: the grouped attention kernel's rows-per-slot range

__device__ __forceinline__ bool better_key(float v, int i, float bv, int bi) { return v > bv || (v == bv && i < bi); }

// fp32 -> uint32 with the same order (-0 folded onto +0, so equal values give equal keys)
__device__ __forceinline__ uint32_t ord_key(float x) {
    uint32_t b = __float_as_uint(x);
    if (b == 0x80000000u) b = 0u;
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

// Row maximum and log(sum exp(l - max)) with the arithmetic of beam_topk_kernel (register pass for even V <= 2*256*SEL_NL, the
// streaming online pass otherwise), so that lp = (l - max) - lsum is bit-identical to the beam search's log-probability.
__device__ __forceinline__ void row_log_softmax_stats(const float* __restrict__ x, int V, float* s_red, float& rmax, float& rlsum) {
    const bool even = (V & 1) == 0;
    const int V2 = V >> 1;
    const float2* x2 = reinterpret_cast<const float2*>(x);
    float sum;
    if (even && V2 <= SEL_NL * SEL_THREADS) {
        float2 a[SEL_NL];
#pragma unroll
        for (int u = 0; u < SEL_NL; ++u) {
            const int j = threadIdx.x + u * SEL_THREADS;
            a[u] = (j < V2) ? x2[j] : make_float2(-INFINITY, -INFINITY);
        }
        float tm = -INFINITY, tsum = 0.f;
#pragma unroll
        for (int u = 0; u < SEL_NL; ++u) tm = fmaxf(tm, fmaxf(a[u].x, a[u].y));
        if (tm > -INFINITY) {
#pragma unroll
            for (int u = 0; u < SEL_NL; ++u) tsum += __expf(a[u].x - tm) + __expf(a[u].y - tm);
        }
        rmax = block_max(tm, s_red);
        sum = block_sum((tm == -INFINITY) ? 0.f : tsum * expf(tm - rmax), s_red);
    } else {
        float m = -INFINITY, ssum = 0.f;
        if (even) {
            int j = threadIdx.x;
            for (; j + 3 * SEL_THREADS < V2; j += 4 * SEL_THREADS) {
                float2 a[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) a[u] = x2[j + u * SEL_THREADS];
                const float cm = fmaxf(fmaxf(fmaxf(a[0].x, a[0].y), fmaxf(a[1].x, a[1].y)), fmaxf(fmaxf(a[2].x, a[2].y), fmaxf(a[3].x, a[3].y)));
                if (cm > m) { ssum *= __expf(m - cm); m = cm; }
#pragma unroll
                for (int u = 0; u < 4; ++u) ssum += __expf(a[u].x - m) + __expf(a[u].y - m);
            }
            for (; j < V2; j += SEL_THREADS) {
                const float2 a = x2[j];
                const float cm = fmaxf(a.x, a.y);
                if (cm > m) { ssum *= __expf(m - cm); m = cm; }
                ssum += __expf(a.x - m) + __expf(a.y - m);
            }
        } else {
            for (int v = threadIdx.x; v < V; v += SEL_THREADS) {
                const float xv = x[v];
                if (xv > m) { ssum *= __expf(m - xv); m = xv; }
                ssum += __expf(xv - m);
            }
        }
        rmax = block_max(m, s_red);
        sum = block_sum((m == -INFINITY) ? 0.f : ssum * expf(m - rmax), s_red);
    }
    rlsum = logf(sum);
}

// Inclusive prefix sum over the CTA (thread order).  s_w: 8 ints.
__device__ __forceinline__ int block_incl_scan(int v, int* s_w) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v += t; }
    __syncthreads();
    if (lane == 31) s_w[w] = v;
    __syncthreads();
    int off = 0;
    for (int q = 0; q < w; ++q) off += s_w[q];
    return v + off;
}

// Exact top-K boundary of a row (1 <= K < V) under the order (larger l first, then lower id): radix select over ord_key in four
// 8-bit digits gives the K-th largest key thr; the candidates are every v with key > thr, and those with key == thr up to the
// id idx_cut (the ids of equal keys are taken in increasing order).
__device__ void topk_boundary(const float* __restrict__ x, int V, int K, unsigned* s_hist, int* s_w, int* s_misc,
                              uint32_t& thr, int& idx_cut) {
    uint32_t prefix = 0u, mask = 0u;
    int rem = K, eq = 0;
    for (int shift = 24; shift >= 0; shift -= 8) {
        s_hist[threadIdx.x] = 0u;
        __syncthreads();
        for (int v = threadIdx.x; v < V; v += SEL_THREADS) {
            const uint32_t u = ord_key(x[v]);
            if ((u & mask) == prefix) atomicAdd(&s_hist[(u >> shift) & 255u], 1u);
        }
        __syncthreads();
        const int h = (int)s_hist[255 - threadIdx.x];          // digits in decreasing order
        const int ge = block_incl_scan(h, s_w);                // elements with this digit or a larger one
        if (ge >= rem && ge - h < rem) { s_misc[0] = 255 - (int)threadIdx.x; s_misc[1] = rem - (ge - h); s_misc[2] = h; }
        __syncthreads();
        prefix |= (uint32_t)s_misc[0] << shift; mask |= 255u << shift;
        rem = s_misc[1]; eq = s_misc[2];
        __syncthreads();
    }
    thr = prefix;
    if (rem == eq) { idx_cut = 0x7fffffff; return; }          // every element equal to the boundary is a candidate
    // the rem-th smallest id among the keys equal to thr: ordered count over chunks of 256 consecutive ids
    if (threadIdx.x == 0) s_misc[3] = -1;
    int carry = 0;
    for (int base = 0; base < V; base += SEL_THREADS) {
        const int v = base + threadIdx.x;
        const int f = (v < V && ord_key(x[v]) == thr) ? 1 : 0;
        const int incl = block_incl_scan(f, s_w);
        if (f && carry + incl == rem) s_misc[3] = v;
        const int total = s_w[0] + s_w[1] + s_w[2] + s_w[3] + s_w[4] + s_w[5] + s_w[6] + s_w[7];
        carry += total;
        __syncthreads();
        if (s_misc[3] >= 0) break;
    }
    idx_cut = s_misc[3];
}

// Block-wide arg-best of (key, id) pairs: the largest key, the lowest id on a tie.  Every thread returns the winner's id.
__device__ __forceinline__ int block_argbest(float bk, int bi, float* s_k, int* s_i) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ok = __shfl_xor_sync(0xffffffffu, bk, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (better_key(ok, oi, bk, bi)) { bk = ok; bi = oi; }
    }
    __syncthreads();
    if (lane == 0) { s_k[w] = bk; s_i[w] = bi; }
    __syncthreads();
    if (w == 0) {
        bk = lane < SEL_THREADS / 32 ? s_k[lane] : -INFINITY;
        bi = lane < SEL_THREADS / 32 ? s_i[lane] : 0x7fffffff;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ok = __shfl_xor_sync(0xffffffffu, bk, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (better_key(ok, oi, bk, bi)) { bk = ok; bi = oi; }
        }
        if (lane == 0) s_i[SEL_THREADS / 32] = bi;
    }
    __syncthreads();
    return s_i[SEL_THREADS / 32];
}

// Gumbel noise of token v from its Philox word: g = -log(-log(u)), u = ((bits >> 8) + 0.5) * 2^-24.  -log(u) is formed from an
// exact fp32 operand on both halves: logf(u) below 1/2, log1pf(-(1 - u)) above (where u itself would round to 1).
__device__ __forceinline__ float gumbel_from_bits(uint32_t bits) {
    const uint32_t x = bits >> 8;
    const float e = (x < (1u << 23)) ? -logf(((float)x + 0.5f) * 0x1p-24f)
                                     : -log1pf(-(((float)((1u << 24) - x) - 0.5f) * 0x1p-24f));
    return -logf(e);
}

// One CTA per live slot (image).  For each live row of the slot: the log-softmax statistics, the top-k boundary (if any), and
// the draw(s) — m draws from the single row of step 1, one draw per row afterwards — then the per-sample outputs and the
// bookkeeping of the slot state machine (surviving rows into the *_tmp arrays in row order, their sample index into tag_tmp).
__global__ void __launch_bounds__(SEL_THREADS) sample_select_kernel(
        int m, int V, int step, int S1 /* max_steps+1 */, int start_id, int end_id, float temperature, int top_k,
        uint32_t seed_lo, uint32_t seed_hi, int img_base, int sample_base,
        const float* __restrict__ logits, const float* __restrict__ score, const int* __restrict__ k_live,
        const int* __restrict__ slot_img, const int* __restrict__ n_live, const int* __restrict__ row_off,
        const int* __restrict__ tag, float* __restrict__ score_tmp, int* __restrict__ word_tmp, int* __restrict__ k_live_tmp,
        int* __restrict__ slot_img_tmp, int* __restrict__ src, int* __restrict__ tag_tmp,
        int* __restrict__ out_seq, int* __restrict__ out_len, unsigned char* __restrict__ out_ended,
        float* __restrict__ out_score, float* __restrict__ out_logp) {
    __shared__ float s_red[40];
    __shared__ unsigned s_hist[256];
    __shared__ int s_w[8], s_misc[4];
    __shared__ float s_k[SEL_THREADS / 32];
    __shared__ int s_i[SEL_THREADS / 32 + 1];
    const int slot = blockIdx.x;
    if (slot >= n_live[0]) return;
    const int img = slot_img[slot];
    const int kl = k_live[slot];
    const int row0 = row_off[slot];
    const bool greedy = temperature == 0.f;
    const bool restrict_k = !greedy && top_k > 0 && top_k < V;
    const int nq = (V + 3) >> 2;
    int nlive = 0;                                                   // (thread 0)
    for (int i = 0; i < kl; ++i) {
        const float* x = logits + (long long)(row0 + i) * V;
        float rmax, rlsum;
        row_log_softmax_stats(x, V, s_red, rmax, rlsum);
        uint32_t thr = 0u; int idx_cut = 0x7fffffff;
        if (restrict_k) topk_boundary(x, V, top_k, s_hist, s_w, s_misc, thr, idx_cut);
        const int ndraw = (step == 1) ? m : 1;                       // step 1: the slot's single row serves all m samples
        int greedy_tok = -1;
        for (int dr = 0; dr < ndraw; ++dr) {
            const int j = (step == 1) ? dr : tag[row0 + i];          // sample index within the call
            int tok;
            if (greedy) {
                if (greedy_tok < 0) {
                    float bk = -INFINITY; int bi = 0x7fffffff;
                    for (int v = threadIdx.x; v < V; v += SEL_THREADS) { const float l = x[v]; if (better_key(l, v, bk, bi)) { bk = l; bi = v; } }
                    greedy_tok = block_argbest(bk, bi, s_k, s_i);
                }
                tok = greedy_tok;
            } else {
                float bk = -INFINITY; int bi = 0x7fffffff;
                for (int q = threadIdx.x; q < nq; q += SEL_THREADS) {
                    uint32_t c[4] = {(uint32_t)q, (uint32_t)step, (uint32_t)(img_base + img), (uint32_t)(sample_base + j)};
                    philox4x32_10(c, seed_lo, seed_hi);
#pragma unroll
                    for (int wd = 0; wd < 4; ++wd) {
                        const int v = 4 * q + wd;
                        if (v >= V) break;
                        const float l = x[v];
                        if (restrict_k) { const uint32_t u = ord_key(l); if (u < thr || (u == thr && v > idx_cut)) continue; }
                        const float key = __fadd_rn(__fdiv_rn(l, temperature), gumbel_from_bits(c[wd]));
                        if (better_key(key, v, bk, bi)) { bk = key; bi = v; }
                    }
                }
                tok = block_argbest(bk, bi, s_k, s_i);
            }
            if (threadIdx.x == 0) {
                const float lp = (x[tok] - rmax) - rlsum;
                const float ns = score[row0 + i] + lp;
                const long long o = (long long)img * m + j;
                int* seq = out_seq + o * (S1 + 1);
                if (step == 1) seq[0] = start_id;
                seq[step] = tok;
                if (out_logp) out_logp[o * S1 + step - 1] = lp;
                if (tok == end_id || step == S1) {                   // ended, or truncated after the last step
                    out_len[o] = step + 1; out_ended[o] = tok == end_id ? 1 : 0; out_score[o] = ns;
                } else {
                    const int r = slot * m + nlive;
                    src[r] = i; score_tmp[r] = ns; word_tmp[r] = tok; tag_tmp[r] = j;
                    ++nlive;
                }
            }
        }
    }
    if (threadIdx.x == 0) { k_live_tmp[slot] = nlive; slot_img_tmp[slot] = img; }
}

int launch_select(int n_img, int m, int V, int step, int S1, int start_id, int end_id, float temperature, int top_k,
                  uint64_t seed, int img_base, int sample_base, BeamWs& w, const int* row_off, int* out_seq, int* out_len,
                  uint8_t* out_ended, float* out_score, float* out_logp, cudaStream_t s) {
    sample_select_kernel<<<n_img, SEL_THREADS, 0, s>>>(m, V, step, S1, start_id, end_id, temperature, top_k, (uint32_t)seed,
                                                       (uint32_t)(seed >> 32), img_base, sample_base, w.logits, w.score,
                                                       w.k_live, w.slot_img, w.n_live, row_off, w.tag, w.score_tmp, w.word_tmp,
                                                       w.k_live_tmp, w.slot_img_tmp, w.src, w.tag_tmp, out_seq, out_len,
                                                       out_ended, out_score, out_logp);
    ICD_LAUNCH_CHECK();
    return 0;
}

int sample_common_check(const char* who, int n_img, int m, int max_steps, int V, float temperature, int top_k, int precision,
                        int img_base, int sample_base) {
    ICD_CHECK_ARG(n_img > 0 && m >= 1 && m <= MMAX, "%s: n_img=%d m=%d (m in 1..%d)", who, n_img, m, MMAX);
    ICD_CHECK_ARG(max_steps >= 1 && max_steps + 1 <= ICD_MAX_STEPS, "%s: max_steps=%d out of range", who, max_steps);
    ICD_CHECK_ARG(V >= 1, "%s: empty vocabulary", who);
    ICD_CHECK_ARG(isfinite(temperature) && temperature >= 0.f, "%s: temperature must be finite and >= 0 (got %g)", who,
                  (double)temperature);
    ICD_CHECK_ARG(top_k >= 0 && top_k <= V, "%s: top_k=%d outside 0..V (V=%d)", who, top_k, V);
    ICD_CHECK_ARG(img_base >= 0 && sample_base >= 0, "%s: img_base / sample_base must be >= 0", who);
    ICD_CHECK_ARG((long long)n_img * m <= 65535, "%s: n_img*m=%lld exceeds 65535 rows per call (chunk the images)", who,
                  (long long)n_img * m);
    ICD_CHECK_ARG(precision == ICD_PREC_FP32 || precision == ICD_PREC_FP32X3,
                  "%s: precision must be ICD_PREC_FP32 or ICD_PREC_FP32X3 (the log-probabilities need fp32-grade logits)", who);
    return 0;
}

// The sampler's descriptor seen as a beam descriptor (k = m): the shared prologue / step / workspace code reads that.
icd_beam_desc_t as_beam(const icd_sample_desc_t* d) {
    icd_beam_desc_t b;
    memset(&b, 0, sizeof(b));
    b.n_img = d->n_img; b.k = d->m; b.max_steps = d->max_steps;
    b.P = d->P; b.C = d->C; b.A = d->A; b.D = d->D; b.E = d->E; b.V = d->V;
    b.precision = d->precision; b.emb_is_f64 = d->emb_is_f64; b.start_id = d->start_id; b.end_id = d->end_id;
    b.enc = d->enc; b.enc_att_w = d->enc_att_w; b.enc_att_b = d->enc_att_b; b.dec_att_w = d->dec_att_w; b.dec_att_b = d->dec_att_b;
    b.full_att_w = d->full_att_w; b.full_att_b = d->full_att_b; b.w_ih = d->w_ih; b.w_hh = d->w_hh; b.b_ih = d->b_ih;
    b.b_hh = d->b_hh; b.h_lin_w = d->h_lin_w; b.h_lin_b = d->h_lin_b; b.c_lin_w = d->c_lin_w; b.c_lin_b = d->c_lin_b;
    b.f_beta_w = d->f_beta_w; b.f_beta_b = d->f_beta_b; b.fc_w = d->fc_w; b.fc_b = d->fc_b; b.emb_w = d->emb_w;
    b.ws = d->ws; b.ws_bytes = d->ws_bytes;
    return b;
}

icd_base_beam_desc_t as_base_beam(const icd_base_sample_desc_t* d) {
    icd_base_beam_desc_t b;
    memset(&b, 0, sizeof(b));
    b.n_img = d->n_img; b.k = d->m; b.max_steps = d->max_steps; b.E = d->E; b.H = d->H; b.V = d->V;
    b.precision = d->precision; b.emb_is_f64 = d->emb_is_f64; b.start_id = d->start_id; b.end_id = d->end_id;
    b.img_features = d->img_features; b.emb_w = d->emb_w; b.w_ih = d->w_ih; b.w_hh = d->w_hh; b.b_ih = d->b_ih; b.b_hh = d->b_hh;
    b.lin_w = d->lin_w; b.lin_b = d->lin_b;
    b.ws = d->ws; b.ws_bytes = d->ws_bytes;
    return b;
}

int att_sample_shape_check(const icd_sample_desc_t* d) {
    ICD_CHECK_ARG(d != nullptr, "sample_captions: null descriptor");
    ICD_TRY(sample_common_check("sample_captions", d->n_img, d->m, d->max_steps, d->V, d->temperature, d->top_k, d->precision,
                                d->img_base, d->sample_base));
    ICD_CHECK_ARG(d->P > 0 && d->C > 0 && d->A > 0 && d->D > 0 && d->E > 0, "sample_captions: non-positive dimension");
    ICD_CHECK_ARG(d->A % 4 == 0 && d->C % 4 == 0 && d->D % 4 == 0 && d->E % 4 == 0, "sample_captions: dims must be multiples of 4");
    return 0;
}

int att_sample_check(const icd_sample_desc_t* d) {
    ICD_TRY(att_sample_shape_check(d));
    ICD_CHECK_ARG(d->start_id >= 0 && d->start_id < d->V && d->end_id >= 0 && d->end_id < d->V,
                  "sample_captions: start_id / end_id outside the vocabulary");
    ICD_CHECK_ARG(d->enc && d->enc_att_w && d->enc_att_b && d->dec_att_w && d->dec_att_b && d->full_att_w && d->full_att_b &&
                  d->w_ih && d->w_hh && d->b_ih && d->b_hh && d->h_lin_w && d->h_lin_b && d->c_lin_w && d->c_lin_b &&
                  d->f_beta_w && d->f_beta_b && d->fc_w && d->fc_b && d->emb_w, "sample_captions: null input or weight");
    ICD_CHECK_ARG(d->out_seq && d->out_len && d->out_ended && d->out_score, "sample_captions: null result pointer");
    const icd_beam_desc_t b = as_beam(d);
    ICD_CHECK_ARG(d->ws && d->ws_bytes >= (int64_t)carve(&b, nullptr, nullptr, false), "sample_captions: workspace too small");
    return 0;
}

int base_sample_shape_check(const icd_base_sample_desc_t* d) {
    ICD_CHECK_ARG(d != nullptr, "baseline_sample_captions: null descriptor");
    ICD_TRY(sample_common_check("baseline_sample_captions", d->n_img, d->m, d->max_steps, d->V, d->temperature, d->top_k,
                                d->precision, d->img_base, d->sample_base));
    ICD_CHECK_ARG(d->E > 0 && d->H > 0 && d->E % 4 == 0 && d->H % 4 == 0,
                  "baseline_sample_captions: E=%d H=%d must be positive multiples of 4", d->E, d->H);
    return 0;
}

int base_sample_check(const icd_base_sample_desc_t* d) {
    ICD_TRY(base_sample_shape_check(d));
    ICD_CHECK_ARG(d->start_id >= 0 && d->start_id < d->V && d->end_id >= 0 && d->end_id < d->V,
                  "baseline_sample_captions: start_id / end_id outside the vocabulary");
    ICD_CHECK_ARG(d->img_features && d->emb_w && d->w_ih && d->w_hh && d->b_ih && d->b_hh && d->lin_w && d->lin_b,
                  "baseline_sample_captions: null input or weight");
    ICD_CHECK_ARG(d->out_seq && d->out_len && d->out_ended && d->out_score, "baseline_sample_captions: null result pointer");
    const icd_base_beam_desc_t b = as_base_beam(d);
    ICD_CHECK_ARG(d->ws && d->ws_bytes >= (int64_t)carve_base(&b, nullptr, nullptr, false),
                  "baseline_sample_captions: workspace too small");
    return 0;
}

}  // namespace

extern "C" int64_t icd_sample_captions_ws_bytes(const icd_sample_desc_t* d) {
    if (att_sample_shape_check(d) != 0) return -1;        // (the reason is in icd_last_error_string)
    const icd_beam_desc_t b = as_beam(d);
    return (int64_t)carve(&b, nullptr, nullptr, false);
}

extern "C" int icd_sample_captions(const icd_sample_desc_t* d, void* stream) {
    ICD_TRY(att_sample_check(d));                         // every argument before the first CUDA call
    cudaStream_t s = icd_stream(stream);
    const icd_beam_desc_t b = as_beam(d);
    BeamWs w;
    carve(&b, &w, (char*)d->ws, false);
    const int n_img = d->n_img, m = d->m, D = d->D, V = d->V, S1 = d->max_steps + 1;
    const long long R = (long long)n_img * m;
    ICD_CUDA(cudaMemsetAsync(d->out_seq, 0, sizeof(int32_t) * (size_t)R * (S1 + 1), s));
    if (d->out_logp) ICD_CUDA(cudaMemsetAsync(d->out_logp, 0, sizeof(float) * (size_t)R * S1, s));
    bool use_embg = false;
    ICD_TRY(beam_att_prologue(&b, w, &use_embg, s));
    ICD_TRY(beam_launch_init(n_img, m, D, d->start_id, w, s));
    ICD_CUDA(cudaMemsetAsync(w.ring_ticket, 0, sizeof(int) * (size_t)(S1 + 2), s));
    for (int step = 1; step <= S1; ++step) {
        const int* row_off = w.row_off[(step - 1) & 1];
        int* row_off_next = w.row_off[step & 1];
        ICD_TRY(beam_att_step(&b, w, step, use_embg, row_off, w.alpha_steps, s));   // (alpha of one step, not kept)
        ICD_TRY(launch_select(n_img, m, V, step, S1, d->start_id, d->end_id, d->temperature, d->top_k, d->seed, d->img_base,
                              d->sample_base, w, row_off, d->out_seq, d->out_len, d->out_ended, d->out_score, d->out_logp, s));
        ICD_TRY(beam_launch_advance(n_img, m, D, w, row_off, row_off_next, s));
    }
    return 0;
}

extern "C" int64_t icd_baseline_sample_captions_ws_bytes(const icd_base_sample_desc_t* d) {
    if (base_sample_shape_check(d) != 0) return -1;
    const icd_base_beam_desc_t b = as_base_beam(d);
    return (int64_t)carve_base(&b, nullptr, nullptr, false);
}

extern "C" int icd_baseline_sample_captions(const icd_base_sample_desc_t* d, void* stream) {
    ICD_TRY(base_sample_check(d));                        // every argument before the first CUDA call
    cudaStream_t s = icd_stream(stream);
    const icd_base_beam_desc_t b = as_base_beam(d);
    BeamWs w;
    carve_base(&b, &w, (char*)d->ws, false);
    const int n_img = d->n_img, m = d->m, H = d->H, V = d->V, S1 = d->max_steps + 1;
    const long long R = (long long)n_img * m;
    ICD_CUDA(cudaMemsetAsync(d->out_seq, 0, sizeof(int32_t) * (size_t)R * (S1 + 1), s));
    if (d->out_logp) ICD_CUDA(cudaMemsetAsync(d->out_logp, 0, sizeof(float) * (size_t)R * S1, s));
    ICD_TRY(beam_base_prologue(&b, w, s));
    ICD_TRY(beam_launch_init(n_img, m, H, d->start_id, w, s));
    for (int step = 1; step <= S1; ++step) {
        const int* row_off = w.row_off[(step - 1) & 1];
        int* row_off_next = w.row_off[step & 1];
        ICD_TRY(beam_base_step(&b, w, s));
        ICD_TRY(launch_select(n_img, m, V, step, S1, d->start_id, d->end_id, d->temperature, d->top_k, d->seed, d->img_base,
                              d->sample_base, w, row_off, d->out_seq, d->out_len, d->out_ended, d->out_score, d->out_logp, s));
        ICD_TRY(beam_launch_advance(n_img, m, H, w, row_off, row_off_next, s));
    }
    return 0;
}
