// Fused additive-attention step kernels (HBM-bound).  Reference: models/attention.py:55-60, 270-271.
//
// Forward, per decoder row r (image b = img_index ? img_index[r] : r):
//   scores kernel : e[p] = sum_a relu(att_enc[b,p,a] + att_dec[r,a]) * w_full[a] + b_full     (:55-57)
//                   alpha = softmax_p(e)                                                        (:58)
//                   one CTA per row streams the 196x512 att_enc tile once (401 KB), warp-per-pixel rows,
//                   128-bit coalesced loads, warp-shuffle dot, block softmax.
//   weighted-sum  : awe[c] = sum_p alpha[p] * enc[b,p,c]; gate = sigmoid(fbeta_pre); gated = gate*awe
//                   grid (C/256, rows): a CTA streams a 196 x 1 KB column panel of enc with 4 pixel
//                   groups x 64 float4 lanes, 7 independent 128-bit loads in flight per thread,
//                   cross-group reduce in shared memory, gate fused in the epilogue.   (:59-60, 270-271)
// The (B,196,2048) `enc*alpha` temporary of the reference (:59) is never materialised.
//
// Backward, per row: d_awe = d_gated*gate, d_fbeta_pre = d_gated*awe_raw*gate*(1-gate),
//   d_alpha[p] = <d_awe, enc[b,p,:]> (+ upstream), softmax backward in centred form,
//   d_att_dec[a] = w_full[a] * sum_p d_e[p] * [att_enc[b,p,a]+att_dec[a] > 0].
// d_att_enc is NOT read-modify-written per step: d_e is saved per step and one kernel after the time
// loop (attention_proj_bwd) forms d_att_enc and d_w_full for all steps at once.
#include "common.cuh"
#include "tc_common.cuh"
#include <cuda_bf16.h>
#include <stdlib.h>

namespace {

// ------------------------------------------------------------------------------------------------
// Fused attention step, forward: ONE kernel per decode step.  grid = rows, block = 256 (8 warps).
//   phase 1  scores: warp per pixel row of att_enc (A floats), two rows per iteration => 2*(A/128) independent
//            128-bit loads in flight per lane; relu(att_enc + att_dec) . w_full via warp shuffle
//   phase 2  softmax over the P scores in shared memory (expf, block reductions); alpha written out
//   phase 3  awe[c] = sum_p alpha[p] * enc[p, c]: thread t owns float4 columns t and t+256 (C = 2048 => two
//            columns), 2 x 4 independent 128-bit loads in flight, each pixel row read as two contiguous 4 KB runs
//   epilogue gate = sigmoid(fbeta_pre), gated = gate * awe
// Algorithmic bytes per row: P*A*4 (att_enc) + P*C*4 (enc) + small = 2 026 256 B for P=196, A=512, C=2048.
// smem: 2*A + P + 40 floats.
// ------------------------------------------------------------------------------------------------
constexpr int FW_UNROLL = 4;

__global__ void __launch_bounds__(256, 4) att_step_fwd_kernel(
        int P, int C, int A, const int* __restrict__ img_index,
        const float* __restrict__ enc, const float* __restrict__ att_enc,
        const float* __restrict__ att_dec, long long ld_dec,
        const float* __restrict__ w_full, const float* __restrict__ b_full,
        const float* __restrict__ fbeta_pre, long long ld_fb,
        float* __restrict__ alpha, long long ld_alpha,
        float* __restrict__ awe_raw, float* __restrict__ gate, float* __restrict__ gated) {
    extern __shared__ __align__(16) float sm[];
    float* s_dec = sm;            // A
    float* s_wf = sm + A;         // A
    float* s_e = sm + 2 * A;      // P  (scores, then alpha)
    float* s_red = s_e + ((P + 3) & ~3);       // 40
    const int r = blockIdx.x;
    const int img = img_index ? img_index[r] : r;
    const float* ae = att_enc + (long long)img * P * A;
    const float* dec = att_dec + (long long)r * ld_dec;
    for (int a = threadIdx.x; a < A; a += blockDim.x) { s_dec[a] = dec[a]; s_wf[a] = w_full[a]; }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    const float bfull = b_full ? b_full[0] : 0.f;
    const int A4 = A >> 2;
    for (int p = warp; p < P; p += 2 * nwarp) {
        const int p2 = p + nwarp;
        const bool has2 = p2 < P;
        const float* row0 = ae + (long long)p * A;
        const float* row1 = ae + (long long)(has2 ? p2 : p) * A;
        float acc0 = 0.f, acc1 = 0.f;
        for (int j = lane; j < A4; j += 32) {
            const float4 x0 = ld_stream_f4(row0 + 4 * j);
            const float4 x1 = ld_stream_f4(row1 + 4 * j);
            const float4 d = *reinterpret_cast<const float4*>(s_dec + 4 * j);
            const float4 w = *reinterpret_cast<const float4*>(s_wf + 4 * j);
            acc0 = fmaf(fmaxf(x0.x + d.x, 0.f), w.x, acc0);
            acc0 = fmaf(fmaxf(x0.y + d.y, 0.f), w.y, acc0);
            acc0 = fmaf(fmaxf(x0.z + d.z, 0.f), w.z, acc0);
            acc0 = fmaf(fmaxf(x0.w + d.w, 0.f), w.w, acc0);
            acc1 = fmaf(fmaxf(x1.x + d.x, 0.f), w.x, acc1);
            acc1 = fmaf(fmaxf(x1.y + d.y, 0.f), w.y, acc1);
            acc1 = fmaf(fmaxf(x1.z + d.z, 0.f), w.z, acc1);
            acc1 = fmaf(fmaxf(x1.w + d.w, 0.f), w.w, acc1);
        }
        acc0 = warp_sum(acc0);
        acc1 = warp_sum(acc1);
        if (lane == 0) { s_e[p] = acc0 + bfull; if (has2) s_e[p2] = acc1 + bfull; }
    }
    __syncthreads();
    float m = -INFINITY;
    for (int p = threadIdx.x; p < P; p += blockDim.x) m = fmaxf(m, s_e[p]);
    m = block_max(m, s_red);
    float sum = 0.f;
    for (int p = threadIdx.x; p < P; p += blockDim.x) { const float ex = expf(s_e[p] - m); s_e[p] = ex; sum += ex; }
    sum = block_sum(sum, s_red);
    {
        float* out = alpha + (long long)r * ld_alpha;
        for (int p = threadIdx.x; p < P; p += blockDim.x) { const float al = s_e[p] / sum; s_e[p] = al; out[p] = al; }
    }
    __syncthreads();

    // phase 3: alpha-weighted sum over pixels, two float4 columns per thread per pass
    const float* eb = enc + (long long)img * P * C;
    const int stride = blockDim.x * 4;                         // 1024 floats between a thread's two columns
    for (int c0 = threadIdx.x * 4; c0 < C; c0 += 2 * stride) {
        const int c1 = c0 + stride;
        const bool has1 = c1 < C;
        const float* b0 = eb + c0;
        const float* b1 = eb + (has1 ? c1 : c0);
        float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = make_float4(0.f, 0.f, 0.f, 0.f);
        int p = 0;
        for (; p + FW_UNROLL <= P; p += FW_UNROLL) {
            float4 x0[FW_UNROLL], x1[FW_UNROLL];
#pragma unroll
            for (int u = 0; u < FW_UNROLL; ++u) {
                x0[u] = ld_stream_f4(b0 + (long long)(p + u) * C);
                x1[u] = ld_stream_f4(b1 + (long long)(p + u) * C);
            }
#pragma unroll
            for (int u = 0; u < FW_UNROLL; ++u) {
                const float al = s_e[p + u];
                a0.x = fmaf(al, x0[u].x, a0.x); a0.y = fmaf(al, x0[u].y, a0.y);
                a0.z = fmaf(al, x0[u].z, a0.z); a0.w = fmaf(al, x0[u].w, a0.w);
                a1.x = fmaf(al, x1[u].x, a1.x); a1.y = fmaf(al, x1[u].y, a1.y);
                a1.z = fmaf(al, x1[u].z, a1.z); a1.w = fmaf(al, x1[u].w, a1.w);
            }
        }
        for (; p < P; ++p) {
            const float4 x0 = ld_stream_f4(b0 + (long long)p * C);
            const float4 x1 = ld_stream_f4(b1 + (long long)p * C);
            const float al = s_e[p];
            a0.x = fmaf(al, x0.x, a0.x); a0.y = fmaf(al, x0.y, a0.y);
            a0.z = fmaf(al, x0.z, a0.z); a0.w = fmaf(al, x0.w, a0.w);
            a1.x = fmaf(al, x1.x, a1.x); a1.y = fmaf(al, x1.y, a1.y);
            a1.z = fmaf(al, x1.z, a1.z); a1.w = fmaf(al, x1.w, a1.w);
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            if (h == 1 && !has1) break;
            const int c = h ? c1 : c0;
            const float4 acc = h ? a1 : a0;
            const long long o = (long long)r * C + c;
            if (awe_raw) *reinterpret_cast<float4*>(awe_raw + o) = acc;
            if (fbeta_pre) {
                const float4 f = *reinterpret_cast<const float4*>(fbeta_pre + (long long)r * ld_fb + c);
                const float4 g = make_float4(sigmoidf_(f.x), sigmoidf_(f.y), sigmoidf_(f.z), sigmoidf_(f.w));
                if (gate) *reinterpret_cast<float4*>(gate + o) = g;
                if (gated) *reinterpret_cast<float4*>(gated + o) =
                        make_float4(g.x * acc.x, g.y * acc.y, g.z * acc.z, g.w * acc.w);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Grouped forward for caption generation: the K beam rows of ONE image share its feature map, so one CTA serves all
// live beams of an image and reads att_enc / enc ONCE per step instead of once per beam (gen_captions.py:44 expands the
// features to k copies and :111 re-gathers them every step).  grid = n_img, block = 256; rows img*k + j, j < k_live[img];
// images with no live beam exit immediately.  Per row the arithmetic (lane partition of the score dot, sequential pixel
// order of the weighted sum) is that of att_step_fwd_kernel, so results are bit-identical to the per-row kernel.
// smem: K*A (att_dec) + A (w_full) + K*Ppad (scores / alpha) floats.
// ------------------------------------------------------------------------------------------------
#ifndef ICD_ATT_GROUPED_MINB
#define ICD_ATT_GROUPED_MINB 3
#endif
template <int K>
__global__ void __launch_bounds__(256, ICD_ATT_GROUPED_MINB) att_step_fwd_grouped_kernel(
        int k, int P, int C, int A, const int* __restrict__ k_live,
        const float* __restrict__ enc, const float* __restrict__ att_enc,
        const float* __restrict__ att_dec, long long ld_dec,
        const float* __restrict__ w_full, const float* __restrict__ b_full,
        const float* __restrict__ fbeta_pre, long long ld_fb,
        float* __restrict__ alpha, long long ld_alpha, float* __restrict__ gated,
        const int* __restrict__ slot_img, const int* __restrict__ n_slots, const int* __restrict__ row_off,
        unsigned short* __restrict__ gated_x3, int x3_nseg) {
    extern __shared__ __align__(16) float sm[];
    // slot = the live beams of one image: state rows (att_dec / fbeta / gated) row_off[slot] + j, or slot*k + j without a
    // row map; img = the image whose features the slot decodes (slot == img without a slot map).  alpha rows are
    // addressed by IMAGE (img*k + j): the caller back-tracks them per image.
    const int slot = blockIdx.x;
    if (n_slots && slot >= n_slots[0]) return;
    const int img = slot_img ? slot_img[slot] : slot;
    const int kl = k_live ? min(k_live[slot], K) : min(k, K);
    if (kl <= 0) return;
    const int Pp = (P + 3) & ~3;
    float* s_dec = sm;                 // K * A
    float* s_wf = sm + K * A;          // A
    float* s_e = s_wf + A;             // K * Pp
    const long long r0 = row_off ? (long long)row_off[slot] : (long long)slot * k, ra = (long long)img * k;
    for (int i = threadIdx.x; i < kl * A; i += blockDim.x) s_dec[i] = att_dec[(r0 + i / A) * ld_dec + (i % A)];
    for (int a = threadIdx.x; a < A; a += blockDim.x) s_wf[a] = w_full[a];
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    const float bfull = b_full ? b_full[0] : 0.f;
    const int A4 = A >> 2;
    const float* ae = att_enc + (long long)img * P * A;
    // GROUPED_ROWS pixel rows per warp iteration: a lane loads the same float4 column q of all of them, so one shared-memory
    // read of att_dec[j][q] / w_full[q] feeds GROUPED_ROWS rows (the score phase is shared-memory-bound otherwise).  Per row
    // the summation order (q = lane, lane + 32, ...; x, y, z, w) is that of the per-row kernel: bit-identical scores.
    constexpr int GROUPED_ROWS = 4;
    for (int p0 = warp; p0 < P; p0 += GROUPED_ROWS * nwarp) {
        float acc[GROUPED_ROWS][K];
#pragma unroll
        for (int u = 0; u < GROUPED_ROWS; ++u)
#pragma unroll
            for (int j = 0; j < K; ++j) acc[u][j] = 0.f;
        for (int q = lane; q < A4; q += 32) {
            float4 xs[GROUPED_ROWS];
#pragma unroll
            for (int u = 0; u < GROUPED_ROWS; ++u) {
                const int p = p0 + u * nwarp;                        // warp-uniform
                xs[u] = (p < P) ? ld_stream_f4(ae + (long long)p * A + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            const float4 w = *reinterpret_cast<const float4*>(s_wf + 4 * q);
#pragma unroll
            for (int j = 0; j < K; ++j) {
                if (j < kl) {
                    const float4 d = *reinterpret_cast<const float4*>(s_dec + j * A + 4 * q);
#pragma unroll
                    for (int u = 0; u < GROUPED_ROWS; ++u) {
                        const float4 x = xs[u];
                        acc[u][j] = fmaf(fmaxf(x.x + d.x, 0.f), w.x, acc[u][j]);
                        acc[u][j] = fmaf(fmaxf(x.y + d.y, 0.f), w.y, acc[u][j]);
                        acc[u][j] = fmaf(fmaxf(x.z + d.z, 0.f), w.z, acc[u][j]);
                        acc[u][j] = fmaf(fmaxf(x.w + d.w, 0.f), w.w, acc[u][j]);
                    }
                }
            }
        }
#pragma unroll
        for (int u = 0; u < GROUPED_ROWS; ++u) {
            const int p = p0 + u * nwarp;
            if (p < P) {
#pragma unroll
                for (int j = 0; j < K; ++j) {
                    if (j < kl) {
                        const float v = warp_sum(acc[u][j]);
                        if (lane == 0) s_e[j * Pp + p] = v + bfull;
                    }
                }
            }
        }
    }
    __syncthreads();
    // softmax over pixels: warp j handles row j (kl <= K <= 8 = number of warps)
    for (int j = warp; j < kl; j += nwarp) {
        float* e = s_e + j * Pp;
        float m = -INFINITY;
        for (int p = lane; p < P; p += 32) m = fmaxf(m, e[p]);
        m = warp_max(m);
        float sum = 0.f;
        for (int p = lane; p < P; p += 32) { const float ex = expf(e[p] - m); e[p] = ex; sum += ex; }
        sum = warp_sum(sum);
        float* out = alpha + (ra + j) * ld_alpha;
        for (int p = lane; p < P; p += 32) { const float al = e[p] / sum; e[p] = al; out[p] = al; }
    }
    __syncthreads();
    // weighted sums for all live rows: each enc row is loaded once and feeds kl accumulators
    const float* eb = enc + (long long)img * P * C;
    for (int c = threadIdx.x * 4; c < C; c += blockDim.x * 4) {
        float4 acc[K];
#pragma unroll
        for (int j = 0; j < K; ++j) acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        int p = 0;
        for (; p + 8 <= P; p += 8) {                                  // 8 independent 128-bit loads in flight per thread
            float4 x[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) x[u] = ld_stream_f4(eb + (long long)(p + u) * C + c);
#pragma unroll
            for (int j = 0; j < K; ++j) {
                if (j < kl) {
                    // p is a multiple of 8 and Pp of 4: two 128-bit broadcast reads serve the 8 rows (same order of adds)
                    const float4 a0 = *reinterpret_cast<const float4*>(s_e + j * Pp + p);
                    const float4 a1 = *reinterpret_cast<const float4*>(s_e + j * Pp + p + 4);
                    const float al8[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        acc[j].x = fmaf(al8[u], x[u].x, acc[j].x); acc[j].y = fmaf(al8[u], x[u].y, acc[j].y);
                        acc[j].z = fmaf(al8[u], x[u].z, acc[j].z); acc[j].w = fmaf(al8[u], x[u].w, acc[j].w);
                    }
                }
            }
        }
        for (; p < P; ++p) {
            const float4 x = ld_stream_f4(eb + (long long)p * C + c);
#pragma unroll
            for (int j = 0; j < K; ++j) {
                if (j < kl) {
                    const float al = s_e[j * Pp + p];
                    acc[j].x = fmaf(al, x.x, acc[j].x); acc[j].y = fmaf(al, x.y, acc[j].y);
                    acc[j].z = fmaf(al, x.z, acc[j].z); acc[j].w = fmaf(al, x.w, acc[j].w);
                }
            }
        }
#pragma unroll
        for (int j = 0; j < K; ++j) {
            if (j < kl) {
                const float4 f = *reinterpret_cast<const float4*>(fbeta_pre + (r0 + j) * ld_fb + c);
                const float4 g = make_float4(sigmoidf_(f.x), sigmoidf_(f.y), sigmoidf_(f.z), sigmoidf_(f.w));
                const float4 o = make_float4(g.x * acc[j].x, g.y * acc[j].y, g.z * acc[j].z, g.w * acc[j].w);
                if (gated) *reinterpret_cast<float4*>(gated + (r0 + j) * C + c) = o;
                if (gated_x3) {
                    // fp32-grade tensor-core tier: emit the 3-term bf16 split of the row right here, in the A-operand layout of
                    // the next contraction ([a1 | a1 | a2 | a1 | a3 | a2] along K, segment length C; gemm_tc.cu) — the separate
                    // split pass over the (rows, C) activation disappears
                    const float xs[4] = {o.x, o.y, o.z, o.w};
                    unsigned short t[3][4];
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const __nv_bfloat16 b1 = __float2bfloat16_rn(xs[q]);
                        const float r1 = xs[q] - __bfloat162float(b1);
                        const __nv_bfloat16 b2 = __float2bfloat16_rn(r1);
                        const __nv_bfloat16 b3 = __float2bfloat16_rn(r1 - __bfloat162float(b2));
                        t[0][q] = __bfloat16_as_ushort(b1); t[1][q] = __bfloat16_as_ushort(b2); t[2][q] = __bfloat16_as_ushort(b3);
                    }
                    unsigned short* dst = gated_x3 + (r0 + j) * x3_nseg * (long long)C + c;
                    const int pat[6] = {0, 0, 1, 0, 2, 1};
#pragma unroll
                    for (int sg = 0; sg < 6; ++sg) {
                        if (sg >= x3_nseg) break;
                        const unsigned short* tt = t[x3_nseg == 3 ? sg : pat[sg]];
                        *reinterpret_cast<uint2*>(dst + (long long)sg * C) =
                            make_uint2((unsigned)tt[0] | ((unsigned)tt[1] << 16), (unsigned)tt[2] | ((unsigned)tt[3] << 16));
                    }
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Grouped forward, RING variant (the one caption generation runs when the shapes allow): persistent CTAs, two per SM, walk
// the live slots (slot = blockIdx.x, += gridDim.x); a single producer thread per CTA streams each image's att_enc (P x A) and
// enc (P x C) tiles through a shared-memory ring with 1-D bulk async copies (cp.async.bulk -> mbarrier complete_tx), eight
// consumer warps compute from shared memory.  Bytes in flight (3 x 32 KB per CTA) no longer cost registers, the producer keeps
// fetching across the latency-bound pieces of an image (att_dec staging, softmax, epilogue) and across images, there is no
// partial last wave of 2 MB work units, and the two CTAs of an SM drift apart so that the issue-bound score phase of one
// overlaps the HBM-bound weighted sums of the other.  Per row the arithmetic is that of att_step_fwd_grouped_kernel in the
// same order (lane partition q = lane, lane + 32, ... of the score dot, warp-shuffle tree, ascending pixel order of the
// weighted sum), so alphas / gated rows are bit-identical to it (tested).
//   ring slot = RING_ROWS1 (16) pixel rows of att_enc, or RING_ROWS2 (4) pixel rows of enc, each one contiguous copy
//   score phase: warp w owns rows w and w + 8 of a slot => one shared-memory read of att_dec[j] / w_full feeds two pixel rows
//   weighted sum: thread t owns channels 4t..4t+3 and 1024+4t..1024+4t+3 (C <= 2048), one slot = 4 pixels per iteration
// smem: 3 x 32 KB ring + K*A (att_dec) + A (w_full) + K*Ppad (scores / alpha) floats + 6 mbarriers.
// ------------------------------------------------------------------------------------------------
#ifndef ICD_RING_SLOTS
#define ICD_RING_SLOTS 3
#endif
constexpr int RING_SLOT_BYTES = 32768, RING_SLOTS = ICD_RING_SLOTS, RING_CONS_WARPS = 8, RING_ROWS1 = 16, RING_ROWS2 = 4;
constexpr int RING_CONS = RING_CONS_WARPS * 32, RING_THREADS = RING_CONS + 32;

__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void ring_consumer_sync() { asm volatile("bar.sync 1, %0;" :: "n"(RING_CONS) : "memory"); }

__device__ __forceinline__ void ring_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok = 0, spins = 0;
    while (true) {
        asm volatile("{\n\t.reg .pred p;\n\t"
                     "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                     "selp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        if (ok) break;
        if (++spins > (1u << 24)) __trap();          // a protocol bug must fault, never hang the GPU
    }
}

struct RingArgs {
    int P, C, A, Pp, n1, n2;
    const float* att_dec; long long ld_dec;
    const float* fbeta_pre; long long ld_fb;
    float* alpha; long long ld_alpha;
    float* gated; unsigned short* gated_x3; int x3_nseg;
    float bfull;
};

// One image with KL live beams (compile-time: the beam loops are fully unrolled, no per-beam branches in the inner loops —
// the kernel is issue-bound at five beams, every instruction that is not an FADD / FMNMX / FFMA of the two sums counts).
template <int KL>
__device__ __forceinline__ void ring_image(const RingArgs& g, unsigned char* ring_raw, float* s_dec, float* s_wf, float* s_e,
                                           uint32_t full0, uint32_t empty0, uint32_t& it, long long r0, long long ra) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int A = g.A, C = g.C, P = g.P, Pp = g.Pp, A4 = A >> 2;
    for (int i = tid; i < KL * A4; i += RING_CONS) {
        const int j = i / A4, q = i - j * A4;
        *reinterpret_cast<float4*>(s_dec + j * A + 4 * q) = *reinterpret_cast<const float4*>(g.att_dec + (r0 + j) * g.ld_dec + 4 * q);
    }
    ring_consumer_sync();            // s_dec / s_wf staged; everyone has left the previous image's weighted sums (s_e is free)
    // ---- scores: relu(att_enc + att_dec) . w_full, one ring slot (16 pixel rows) per iteration
    for (int gi = 0; gi < g.n1; ++gi, ++it) {
        const uint32_t s = it % RING_SLOTS;
        ring_wait(full0 + 8 * s, (it / RING_SLOTS) & 1);
        const int pa = gi * RING_ROWS1 + warp, pb = pa + RING_CONS_WARPS;
        if (pa < P) {
            const bool vb = pb < P;
            const float* xa = reinterpret_cast<const float*>(ring_raw + (size_t)s * RING_SLOT_BYTES) + warp * A;
            const float* xb = vb ? xa + RING_CONS_WARPS * A : xa;         // row past P: recompute row a, result dropped
            float acc[2][KL];
#pragma unroll
            for (int j = 0; j < KL; ++j) acc[0][j] = acc[1][j] = 0.f;
            for (int q = lane; q < A4; q += 32) {
                const float4 x0 = *reinterpret_cast<const float4*>(xa + 4 * q);
                const float4 x1 = *reinterpret_cast<const float4*>(xb + 4 * q);
                const float4 w = *reinterpret_cast<const float4*>(s_wf + 4 * q);
#pragma unroll
                for (int j = 0; j < KL; ++j) {
                    const float4 d = *reinterpret_cast<const float4*>(s_dec + j * A + 4 * q);
                    acc[0][j] = fmaf(fmaxf(x0.x + d.x, 0.f), w.x, acc[0][j]);
                    acc[1][j] = fmaf(fmaxf(x1.x + d.x, 0.f), w.x, acc[1][j]);
                    acc[0][j] = fmaf(fmaxf(x0.y + d.y, 0.f), w.y, acc[0][j]);
                    acc[1][j] = fmaf(fmaxf(x1.y + d.y, 0.f), w.y, acc[1][j]);
                    acc[0][j] = fmaf(fmaxf(x0.z + d.z, 0.f), w.z, acc[0][j]);
                    acc[1][j] = fmaf(fmaxf(x1.z + d.z, 0.f), w.z, acc[1][j]);
                    acc[0][j] = fmaf(fmaxf(x0.w + d.w, 0.f), w.w, acc[0][j]);
                    acc[1][j] = fmaf(fmaxf(x1.w + d.w, 0.f), w.w, acc[1][j]);
                }
            }
#pragma unroll
            for (int j = 0; j < KL; ++j) {
                const float v0 = warp_sum(acc[0][j]);
                const float v1 = warp_sum(acc[1][j]);
                if (lane == 0) {
                    s_e[j * Pp + pa] = v0 + g.bfull;
                    if (vb) s_e[j * Pp + pb] = v1 + g.bfull;
                }
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(empty0 + 8 * s);
    }
    ring_consumer_sync();
    // ---- softmax over pixels: warp j handles row j (KL <= 8 warps)
    if (warp < KL) {
        float* e = s_e + warp * Pp;
        float m = -INFINITY;
        for (int p = lane; p < P; p += 32) m = fmaxf(m, e[p]);
        m = warp_max(m);
        float sum = 0.f;
        for (int p = lane; p < P; p += 32) { const float ex = expf(e[p] - m); e[p] = ex; sum += ex; }
        sum = warp_sum(sum);
        float* out = g.alpha + (ra + warp) * g.ld_alpha;
        for (int p = lane; p < P; p += 32) { const float al = e[p] / sum; e[p] = al; out[p] = al; }
    }
    ring_consumer_sync();
    // ---- weighted sums: one ring slot = 4 pixel rows of enc per iteration, thread owns channels c .. c+3 and c+1024 .. c+1027
    const int c = tid * 4;
    const bool act0 = c < C, act1 = c + RING_CONS * 4 < C;
    const int c1off = act1 ? RING_CONS * 4 : 0;              // no second column: re-read the first, result dropped
    float4 acc[2][KL];
#pragma unroll
    for (int j = 0; j < KL; ++j) acc[0][j] = acc[1][j] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int i = 0; i < g.n2; ++i, ++it) {
        const uint32_t s = it % RING_SLOTS;
        ring_wait(full0 + 8 * s, (it / RING_SLOTS) & 1);
        if (act0) {
            const int rows = min(RING_ROWS2, P - i * RING_ROWS2);
            const float* xs = reinterpret_cast<const float*>(ring_raw + (size_t)s * RING_SLOT_BYTES) + c;
            if (rows == RING_ROWS2) {
                float4 x[2][RING_ROWS2];
#pragma unroll
                for (int u = 0; u < RING_ROWS2; ++u) {
                    x[0][u] = *reinterpret_cast<const float4*>(xs + (size_t)u * C);
                    x[1][u] = *reinterpret_cast<const float4*>(xs + (size_t)u * C + c1off);
                }
#pragma unroll
                for (int j = 0; j < KL; ++j) {
                    const float4 a4 = *reinterpret_cast<const float4*>(s_e + j * Pp + i * RING_ROWS2);
                    const float al[RING_ROWS2] = {a4.x, a4.y, a4.z, a4.w};
#pragma unroll
                    for (int u = 0; u < RING_ROWS2; ++u) {
#pragma unroll
                        for (int h = 0; h < 2; ++h) {
                            acc[h][j].x = fmaf(al[u], x[h][u].x, acc[h][j].x); acc[h][j].y = fmaf(al[u], x[h][u].y, acc[h][j].y);
                            acc[h][j].z = fmaf(al[u], x[h][u].z, acc[h][j].z); acc[h][j].w = fmaf(al[u], x[h][u].w, acc[h][j].w);
                        }
                    }
                }
            } else {
                for (int u = 0; u < rows; ++u) {                      // last slot of a P that is not a multiple of 4
                    const float4 x0 = *reinterpret_cast<const float4*>(xs + (size_t)u * C);
                    const float4 x1 = *reinterpret_cast<const float4*>(xs + (size_t)u * C + c1off);
#pragma unroll
                    for (int j = 0; j < KL; ++j) {
                        const float al = s_e[j * Pp + i * RING_ROWS2 + u];
                        acc[0][j].x = fmaf(al, x0.x, acc[0][j].x); acc[0][j].y = fmaf(al, x0.y, acc[0][j].y);
                        acc[0][j].z = fmaf(al, x0.z, acc[0][j].z); acc[0][j].w = fmaf(al, x0.w, acc[0][j].w);
                        acc[1][j].x = fmaf(al, x1.x, acc[1][j].x); acc[1][j].y = fmaf(al, x1.y, acc[1][j].y);
                        acc[1][j].z = fmaf(al, x1.z, acc[1][j].z); acc[1][j].w = fmaf(al, x1.w, acc[1][j].w);
                    }
                }
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(empty0 + 8 * s);
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int ch = c + h * RING_CONS * 4;
        if (ch >= C) continue;
#pragma unroll
        for (int j = 0; j < KL; ++j) {
            const float4 f = *reinterpret_cast<const float4*>(g.fbeta_pre + (r0 + j) * g.ld_fb + ch);
            const float4 gt = make_float4(sigmoidf_(f.x), sigmoidf_(f.y), sigmoidf_(f.z), sigmoidf_(f.w));
            const float4 o = make_float4(gt.x * acc[h][j].x, gt.y * acc[h][j].y, gt.z * acc[h][j].z, gt.w * acc[h][j].w);
            if (g.gated) *reinterpret_cast<float4*>(g.gated + (r0 + j) * C + ch) = o;
            if (g.gated_x3) {                // 3-term bf16 split in the A-operand layout of the gate contraction (see the kernel above)
                const float xs[4] = {o.x, o.y, o.z, o.w};
                unsigned short t[3][4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const __nv_bfloat16 b1 = __float2bfloat16_rn(xs[q]);
                    const float r1 = xs[q] - __bfloat162float(b1);
                    const __nv_bfloat16 b2 = __float2bfloat16_rn(r1);
                    const __nv_bfloat16 b3 = __float2bfloat16_rn(r1 - __bfloat162float(b2));
                    t[0][q] = __bfloat16_as_ushort(b1); t[1][q] = __bfloat16_as_ushort(b2); t[2][q] = __bfloat16_as_ushort(b3);
                }
                unsigned short* dst = g.gated_x3 + (r0 + j) * g.x3_nseg * (long long)C + ch;
                const int pat[6] = {0, 0, 1, 0, 2, 1};
#pragma unroll
                for (int sg = 0; sg < 6; ++sg) {
                    if (sg >= g.x3_nseg) break;
                    const unsigned short* tt = t[g.x3_nseg == 3 ? sg : pat[sg]];
                    *reinterpret_cast<uint2*>(dst + (long long)sg * C) =
                        make_uint2((unsigned)tt[0] | ((unsigned)tt[1] << 16), (unsigned)tt[2] | ((unsigned)tt[3] << 16));
                }
            }
        }
    }
}

template <int K>
__global__ void __launch_bounds__(RING_THREADS, (K <= 5 ? 2 : 1)) att_step_fwd_grouped_ring_kernel(
        int n_img, int k, int P, int C, int A, const int* __restrict__ k_live,
        const float* __restrict__ enc, const float* __restrict__ att_enc,
        const float* __restrict__ att_dec, long long ld_dec,
        const float* __restrict__ w_full, const float* __restrict__ b_full,
        const float* __restrict__ fbeta_pre, long long ld_fb,
        float* __restrict__ alpha, long long ld_alpha, float* __restrict__ gated,
        const int* __restrict__ slot_img, const int* __restrict__ n_slots, const int* __restrict__ row_off,
        unsigned short* __restrict__ gated_x3, int* __restrict__ ticket, int stagger_ns_per_beam, int x3_nseg) {
    extern __shared__ __align__(128) unsigned char ring_raw[];
    const int Pp = (P + 3) & ~3;
    float* s_dec = reinterpret_cast<float*>(ring_raw + (size_t)RING_SLOTS * RING_SLOT_BYTES);   // K * A
    float* s_wf = s_dec + K * A;                                                                  // A
    float* s_e = s_wf + A;                                                                        // K * Pp
    const uint32_t ring0 = smem_u32(ring_raw);
    const uint32_t full0 = smem_u32(s_e + K * Pp), empty0 = full0 + 8 * RING_SLOTS;
    volatile int* s_slot = reinterpret_cast<volatile int*>(s_e + K * Pp) + 4 * RING_SLOTS;   // RING_SLOTS ints behind the 2 * RING_SLOTS mbarriers
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        for (int i = 0; i < RING_SLOTS; ++i) { mbar_init(full0 + 8 * i, 1); mbar_init(empty0 + 8 * i, RING_CONS_WARPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int nsl = n_slots ? min(n_slots[0], n_img) : n_img;
    const int n1 = (P + RING_ROWS1 - 1) / RING_ROWS1, n2 = (P + RING_ROWS2 - 1) / RING_ROWS2;

    if (warp == RING_CONS_WARPS) {
        // ---------------------------------------------------------------- producer: one thread, runs ahead of the consumers
        // Work distribution: with a ticket counter the CTAs draw their slots dynamically (no tail of uneven image counts, and
        // the late start of the second CTA per SM costs nothing); the slot id travels to the consumers in s_slot[ring stage of the image's first tile],
        // published before the arrive on the image's first ring stage.  -1 = no more work (a stage without bytes).
        if (lane != 0) return;
        uint32_t it = 0;
        for (int n_done = 0;; ++n_done) {
            const int slot = ticket ? atomicAdd(ticket, 1) : (int)blockIdx.x + n_done * (int)gridDim.x;
            const uint32_t s0 = it % RING_SLOTS, n0 = it / RING_SLOTS;
            if (n0 > 0) mbar_wait_backoff(empty0 + 8 * s0, (n0 - 1) & 1);
            const bool valid = slot < nsl;
            const int kl = !valid ? 0 : (k_live ? min(k_live[slot], K) : min(k, K));
            s_slot[s0] = valid ? slot : -1;
            if (kl <= 0) {                                            // end of work, or a slot without live beams: an empty stage
                mbar_arrive(full0 + 8 * s0);
                ++it;
                if (!valid) break;
                continue;
            }
            const int img = slot_img ? slot_img[slot] : slot;
            const float* ae = att_enc + (long long)img * P * A;
            const float* eb = enc + (long long)img * P * C;
            for (int i = 0; i < n1 + n2; ++i, ++it) {
                const uint32_t s = it % RING_SLOTS, n = it / RING_SLOTS;
                if (i > 0 && n > 0) mbar_wait_backoff(empty0 + 8 * s, (n - 1) & 1);
                const float* src;
                uint32_t bytes;
                if (i < n1) {
                    src = ae + (long long)i * RING_ROWS1 * A;
                    bytes = (uint32_t)min(RING_ROWS1, P - i * RING_ROWS1) * (uint32_t)A * 4u;
                } else {
                    const int i2 = i - n1;
                    src = eb + (long long)i2 * RING_ROWS2 * C;
                    bytes = (uint32_t)min(RING_ROWS2, P - i2 * RING_ROWS2) * (uint32_t)C * 4u;
                }
                mbar_arrive_expect_tx(full0 + 8 * s, bytes);
                bulk_g2s(ring0 + s * RING_SLOT_BYTES, src, bytes, full0 + 8 * s);
            }
        }
        return;
    }

    // -------------------------------------------------------------------- consumers: 8 warps
    RingArgs g;
    g.P = P; g.C = C; g.A = A; g.Pp = Pp; g.n1 = n1; g.n2 = n2;
    g.att_dec = att_dec; g.ld_dec = ld_dec; g.fbeta_pre = fbeta_pre; g.ld_fb = ld_fb;
    g.alpha = alpha; g.ld_alpha = ld_alpha; g.gated = gated; g.gated_x3 = gated_x3; g.x3_nseg = x3_nseg;
    g.bfull = b_full ? b_full[0] : 0.f;
    for (int a = tid; a < A; a += RING_CONS) s_wf[a] = w_full[a];
    uint32_t it = 0;
    for (int n_done = 0;; ++n_done) {
        const uint32_t s0 = it % RING_SLOTS;
        ring_wait(full0 + 8 * s0, (it / RING_SLOTS) & 1);             // the image's first stage (or an empty stage): s_slot is valid
        const int slot = s_slot[s0];          // read before this stage is released: the producer cannot overwrite it
        if (slot < 0) break;
        const int kl = k_live ? min(k_live[slot], K) : min(k, K);
        if (kl <= 0) {                                                // empty stage of a slot without live beams
            __syncwarp();
            if (lane == 0) mbar_arrive(empty0 + 8 * s0);
            ++it;
            continue;
        }
        // Every image costs the same, so all CTAs would walk through the issue-bound score phase and the HBM-bound weighted
        // sums in lockstep (HBM idle, then oversubscribed).  The second CTA of every SM starts its first image half an image
        // late: the two halves of the grid then run in anti-phase.  Free with the ticket counter (late CTAs draw fewer slots).
        if (n_done == 0 && stagger_ns_per_beam > 0 && blockIdx.x >= ICD_NUM_SMS && 2 * kl > K) {      // few live beams: HBM-bound in both phases
            unsigned long long t0, t1;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
            const unsigned long long wait_ns = (unsigned long long)stagger_ns_per_beam * (unsigned)kl;
            do { __nanosleep(256); asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1)); } while (t1 - t0 < wait_ns);
        }
        const int img = slot_img ? slot_img[slot] : slot;
        const long long r0 = row_off ? (long long)row_off[slot] : (long long)slot * k, ra = (long long)img * k;
#define ICD_RING_CASE(KL) case KL: if constexpr (KL <= K) ring_image<KL>(g, ring_raw, s_dec, s_wf, s_e, full0, empty0, it, r0, ra); break
        switch (kl) {
            ICD_RING_CASE(1); ICD_RING_CASE(2); ICD_RING_CASE(3); ICD_RING_CASE(4);
            ICD_RING_CASE(5); ICD_RING_CASE(6); ICD_RING_CASE(7); ICD_RING_CASE(8);
        }
#undef ICD_RING_CASE
    }
}

// ------------------------------------------------------------------------------------------------
// weighted pixel sum + gate.  grid = (ceil(C/256), rows), block = 256 = 4 pixel groups x 64 float4 lanes.
// alpha == NULL  => plain mean over pixels (init_hidden_state, models/attention.py:161).
// out_row_ptr != NULL (captions that share images): CTA row r is image r, and its result is written to the output rows
// out_rows[out_row_ptr[r] .. out_row_ptr[r+1]) instead of row r (the pixel mean computed once per image, gathered to rows).
// ------------------------------------------------------------------------------------------------
constexpr int WS_LANES = 64, WS_GROUPS = 4, WS_UNROLL = 7;

__global__ void __launch_bounds__(256) weighted_pixel_sum_kernel(
        int P, int C, const int* __restrict__ img_index, const float* __restrict__ enc,
        const float* __restrict__ alpha, long long ld_alpha,
        const float* __restrict__ fbeta_pre, long long ld_fb,
        float* __restrict__ awe_raw, float* __restrict__ gate, float* __restrict__ gated,
        const int* __restrict__ out_row_ptr, const int* __restrict__ out_rows) {
    extern __shared__ __align__(16) float sm[];
    float* s_alpha = sm;                                                  // P (padded to mult. of 4)
    float4* s_part = reinterpret_cast<float4*>(sm + ((P + 3) & ~3));      // (WS_GROUPS-1) * WS_LANES float4
    const int r = blockIdx.y;
    const int img = img_index ? img_index[r] : r;
    const int lane = threadIdx.x & (WS_LANES - 1), grp = threadIdx.x / WS_LANES;
    const int c = blockIdx.x * (WS_LANES * 4) + lane * 4;
    if (alpha) {
        const float* al = alpha + (long long)r * ld_alpha;
        for (int p = threadIdx.x; p < P; p += blockDim.x) s_alpha[p] = al[p];
    } else {
        for (int p = threadIdx.x; p < P; p += blockDim.x) s_alpha[p] = 1.f;
    }
    __syncthreads();
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c < C) {
        const float* base = enc + (long long)img * P * C + c;
        int p = grp;
        for (; p + (WS_UNROLL - 1) * WS_GROUPS < P; p += WS_UNROLL * WS_GROUPS) {
            float4 x[WS_UNROLL];
#pragma unroll
            for (int u = 0; u < WS_UNROLL; ++u) x[u] = ld_stream_f4(base + (long long)(p + u * WS_GROUPS) * C);
#pragma unroll
            for (int u = 0; u < WS_UNROLL; ++u) {
                const float a = s_alpha[p + u * WS_GROUPS];
                acc.x = fmaf(a, x[u].x, acc.x); acc.y = fmaf(a, x[u].y, acc.y);
                acc.z = fmaf(a, x[u].z, acc.z); acc.w = fmaf(a, x[u].w, acc.w);
            }
        }
        for (; p < P; p += WS_GROUPS) {
            const float4 x = ld_stream_f4(base + (long long)p * C);
            const float a = s_alpha[p];
            acc.x = fmaf(a, x.x, acc.x); acc.y = fmaf(a, x.y, acc.y);
            acc.z = fmaf(a, x.z, acc.z); acc.w = fmaf(a, x.w, acc.w);
        }
    }
    if (grp > 0) s_part[(grp - 1) * WS_LANES + lane] = acc;
    __syncthreads();
    if (grp == 0 && c < C) {
#pragma unroll
        for (int g = 0; g < WS_GROUPS - 1; ++g) {
            const float4 o = s_part[g * WS_LANES + lane];
            acc.x += o.x; acc.y += o.y; acc.z += o.z; acc.w += o.w;
        }
        if (!alpha) { const float inv = (float)P; acc.x /= inv; acc.y /= inv; acc.z /= inv; acc.w /= inv; }
        const int k0 = out_row_ptr ? out_row_ptr[r] : r, k1 = out_row_ptr ? out_row_ptr[r + 1] : r + 1;
        for (int k = k0; k < k1; ++k) {
            const int ro = out_row_ptr ? out_rows[k] : r;
            const long long o = (long long)ro * C + c;
            if (awe_raw) *reinterpret_cast<float4*>(awe_raw + o) = acc;
            if (fbeta_pre) {
                const float4 f = *reinterpret_cast<const float4*>(fbeta_pre + (long long)ro * ld_fb + c);
                const float4 g = make_float4(sigmoidf_(f.x), sigmoidf_(f.y), sigmoidf_(f.z), sigmoidf_(f.w));
                if (gate) *reinterpret_cast<float4*>(gate + o) = g;
                if (gated) *reinterpret_cast<float4*>(gated + o) =
                        make_float4(g.x * acc.x, g.y * acc.y, g.z * acc.z, g.w * acc.w);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// step backward.  grid = rows, block = 256.  smem: C + 3*P + A + 40 floats + 2*... see launcher.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) att_step_bwd_kernel(
        int P, int C, int A, const int* __restrict__ img_index,
        const float* __restrict__ enc, const float* __restrict__ att_enc,
        const float* __restrict__ att_dec, long long ld_dec, const float* __restrict__ w_full,
        const float* __restrict__ alpha, long long ld_alpha,
        const float* __restrict__ d_alpha_ext, long long ld_dalpha,
        const float* __restrict__ gate, const float* __restrict__ awe_raw, const float* __restrict__ d_gated,
        float* __restrict__ d_att_dec, long long ld_ddec,
        float* __restrict__ d_fbeta_pre, long long ld_dfb,
        float* __restrict__ d_e, long long ld_de, float* __restrict__ d_awe_out) {
    extern __shared__ __align__(16) float sm[];
    float* s_dawe = sm;                       // C
    float* s_dec = s_dawe + C;                // A
    float* s_alpha = s_dec + A;               // P
    float* s_de = s_alpha + ((P + 3) & ~3);   // P   (d_alpha, then d_e)
    float* s_red = s_de + ((P + 3) & ~3);     // 40
    float* s_part = s_red + 40;               // A   (second pixel-group partial of d_att_dec)
    const int r = blockIdx.x;
    const int img = img_index ? img_index[r] : r;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;

    // (A) gate backward, elementwise over C
    {
        const long long o = (long long)r * C;
        for (int c = threadIdx.x * 4; c < C; c += blockDim.x * 4) {
            const float4 dg = *reinterpret_cast<const float4*>(d_gated + o + c);
            const float4 g = *reinterpret_cast<const float4*>(gate + o + c);
            const float4 aw = *reinterpret_cast<const float4*>(awe_raw + o + c);
            const float4 da = make_float4(dg.x * g.x, dg.y * g.y, dg.z * g.z, dg.w * g.w);
            *reinterpret_cast<float4*>(s_dawe + c) = da;
            if (d_awe_out) *reinterpret_cast<float4*>(d_awe_out + o + c) = da;     // kept for the encoder gradient
            const float4 df = make_float4(dg.x * aw.x * g.x * (1.f - g.x), dg.y * aw.y * g.y * (1.f - g.y),
                                          dg.z * aw.z * g.z * (1.f - g.z), dg.w * aw.w * g.w * (1.f - g.w));
            *reinterpret_cast<float4*>(d_fbeta_pre + (long long)r * ld_dfb + c) = df;
        }
        const float* dec = att_dec + (long long)r * ld_dec;
        for (int a = threadIdx.x; a < A; a += blockDim.x) s_dec[a] = dec[a];
        const float* al = alpha + (long long)r * ld_alpha;
        for (int p = threadIdx.x; p < P; p += blockDim.x) s_alpha[p] = al[p];
    }
    __syncthreads();

    // (B) d_alpha[p] = <d_awe, enc[r,p,:]>   warp per pixel row, 8 x 128-bit loads in flight per lane
    {
        const float* eb = enc + (long long)img * P * C;
        const int C4 = C >> 2;
        for (int p = warp; p < P; p += nwarp) {
            const float* row = eb + (long long)p * C;
            float acc = 0.f;
            int j = lane;
            for (; j + 7 * 32 < C4; j += 8 * 32) {
                float4 x[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) x[u] = ld_stream_f4(row + 4 * (j + u * 32));
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const float4 d = *reinterpret_cast<const float4*>(s_dawe + 4 * (j + u * 32));
                    acc = fmaf(x[u].x, d.x, acc); acc = fmaf(x[u].y, d.y, acc);
                    acc = fmaf(x[u].z, d.z, acc); acc = fmaf(x[u].w, d.w, acc);
                }
            }
            for (; j < C4; j += 32) {
                const float4 x = ld_stream_f4(row + 4 * j);
                const float4 d = *reinterpret_cast<const float4*>(s_dawe + 4 * j);
                acc = fmaf(x.x, d.x, acc); acc = fmaf(x.y, d.y, acc);
                acc = fmaf(x.z, d.z, acc); acc = fmaf(x.w, d.w, acc);
            }
            acc = warp_sum(acc);
            if (lane == 0) {
                if (d_alpha_ext) acc += d_alpha_ext[(long long)r * ld_dalpha + p];
                s_de[p] = acc;
            }
        }
    }
    __syncthreads();

    // (C) softmax backward, centred:  d_e = alpha * (d_alpha - sum_q alpha_q d_alpha_q)
    {
        float part = 0.f;
        for (int p = threadIdx.x; p < P; p += blockDim.x) part = fmaf(s_alpha[p], s_de[p], part);
        const float dot = block_sum(part, s_red);
        float* out = d_e + (long long)r * ld_de;
        for (int p = threadIdx.x; p < P; p += blockDim.x) {
            const float v = s_alpha[p] * (s_de[p] - dot);
            s_de[p] = v;
            out[p] = v;
        }
    }
    __syncthreads();

    // (D) d_att_dec[a] = w_full[a] * sum_p d_e[p] * [att_enc[p,a] + att_dec[a] > 0]
    {
        const float* ab = att_enc + (long long)img * P * A;
        const int A4 = A >> 2;
        const int half = blockDim.x >> 1;                 // two pixel groups
        const int grp = threadIdx.x / half, t = threadIdx.x % half;
        for (int j0 = 0; j0 < A4; j0 += half) {
            const int j = j0 + t;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            if (j < A4) {
                const float4 d = *reinterpret_cast<const float4*>(s_dec + 4 * j);
                int p = grp;
                for (; p + 6 * 2 < P; p += 7 * 2) {
                    float4 x[7];
#pragma unroll
                    for (int u = 0; u < 7; ++u) x[u] = ld_stream_f4(ab + (long long)(p + 2 * u) * A + 4 * j);
#pragma unroll
                    for (int u = 0; u < 7; ++u) {
                        const float de = s_de[p + 2 * u];
                        acc.x += (x[u].x + d.x > 0.f) ? de : 0.f;
                        acc.y += (x[u].y + d.y > 0.f) ? de : 0.f;
                        acc.z += (x[u].z + d.z > 0.f) ? de : 0.f;
                        acc.w += (x[u].w + d.w > 0.f) ? de : 0.f;
                    }
                }
                for (; p < P; p += 2) {
                    const float4 x = ld_stream_f4(ab + (long long)p * A + 4 * j);
                    const float de = s_de[p];
                    acc.x += (x.x + d.x > 0.f) ? de : 0.f;
                    acc.y += (x.y + d.y > 0.f) ? de : 0.f;
                    acc.z += (x.z + d.z > 0.f) ? de : 0.f;
                    acc.w += (x.w + d.w > 0.f) ? de : 0.f;
                }
            }
            if (grp == 1 && j < A4) *reinterpret_cast<float4*>(s_part + 4 * j) = acc;
            __syncthreads();
            if (grp == 0 && j < A4) {
                const float4 o = *reinterpret_cast<const float4*>(s_part + 4 * j);
                const float4 w = *reinterpret_cast<const float4*>(w_full + 4 * j);
                float4 res = make_float4((acc.x + o.x) * w.x, (acc.y + o.y) * w.y,
                                         (acc.z + o.z) * w.z, (acc.w + o.w) * w.w);
                *reinterpret_cast<float4*>(d_att_dec + (long long)r * ld_ddec + 4 * j) = res;
            }
            __syncthreads();
        }
    }
}

// ------------------------------------------------------------------------------------------------
// After the loop: d_att_enc + full_att / enc_att-bias parameter gradients.
//   d_att_enc[b,p,a] = w_full[a] * sum_t d_e[b,t,p] * [att_enc[b,p,a] + att_dec[t,b,a] > 0]
// grid = (ceil(P/PB), B), block = A/4 threads (each 4 consecutive a), 4 pixels per pass so that one 128-bit
// shared-memory read of att_dec[t, a..a+3] feeds 16 updates.  smem: T*A (att_dec) + T*PB (d_e).
// partial[(b*gridDim.x + chunk)*(2A+4)] = { d_w_full[A], colsum_p d_att_enc[A] (-> d enc_att.bias), sum d_e, 0,0,0 }.
// ------------------------------------------------------------------------------------------------
constexpr int PROJ_PB = 28;

__device__ __forceinline__ void att_proj_bwd_body(int B, int T, int P, int A,
                                    const int* __restrict__ row_len,   // [B] number of active steps of row b
                                    const float* __restrict__ att_enc, const float* __restrict__ att_dec_all,
                                    long long ld_dec, const float* __restrict__ w_full,
                                    const float* __restrict__ d_e, float* __restrict__ d_att_enc,
                                    float* __restrict__ partial) {
    extern __shared__ __align__(16) float sm[];
    const int b = blockIdx.y, p0 = blockIdx.x * PROJ_PB;
    const int np = min(PROJ_PB, P - p0);
    const int Tb = row_len[b];
    float* s_dec = sm;                  // Tb * A
    float* s_de = sm + (size_t)T * A;   // Tb * PROJ_PB
    float* s_red = s_de + (size_t)T * PROJ_PB;   // 40
    for (int i = threadIdx.x; i < Tb * (A >> 2); i += blockDim.x) {
        const int t = i / (A >> 2), a4 = (i % (A >> 2)) * 4;
        *reinterpret_cast<float4*>(s_dec + (size_t)t * A + a4) =
            *reinterpret_cast<const float4*>(att_dec_all + ((long long)t * B + b) * ld_dec + a4);
    }
    float de_sum = 0.f;
    for (int i = threadIdx.x; i < Tb * PROJ_PB; i += blockDim.x) {
        const int t = i / PROJ_PB, pp = i % PROJ_PB;
        const float v = (pp < np) ? d_e[((long long)b * T + t) * P + p0 + pp] : 0.f;
        s_de[i] = v;
        de_sum += v;
    }
    __syncthreads();
    const int a = threadIdx.x * 4;
    float4 wacc = make_float4(0.f, 0.f, 0.f, 0.f), bacc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (a < A) {
        const float4 w = *reinterpret_cast<const float4*>(w_full + a);
        for (int pq = 0; pq < np; pq += 4) {                          // PROJ_PB % 4 == 0; rows >= np carry d_e = 0
            float x[4][4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int pp = min(pq + u, np - 1);
                const float4 raw = ld_stream_f4(att_enc + ((long long)b * P + p0 + pp) * A + a);
                x[u][0] = raw.x; x[u][1] = raw.y; x[u][2] = raw.z; x[u][3] = raw.w;
            }
            float acc[4][4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int i = 0; i < 4; ++i) acc[u][i] = 0.f;
            for (int t = 0; t < Tb; ++t) {
                const float4 de4 = *reinterpret_cast<const float4*>(s_de + t * PROJ_PB + pq);
                const float4 d = *reinterpret_cast<const float4*>(s_dec + (size_t)t * A + a);
                const float de[4] = {de4.x, de4.y, de4.z, de4.w};
                const float dd[4] = {d.x, d.y, d.z, d.w};
                float wl[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int u = 0; u < 4; ++u) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const float sv = x[u][i] + dd[i];
                        acc[u][i] += (sv > 0.f) ? de[u] : 0.f;
                        wl[i] = fmaf(de[u], fmaxf(sv, 0.f), wl[i]);
                    }
                }
                wacc.x += wl[0]; wacc.y += wl[1]; wacc.z += wl[2]; wacc.w += wl[3];
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (pq + u >= np) break;
                const long long o = ((long long)b * P + p0 + pq + u) * A + a;
                const float4 r = make_float4(acc[u][0] * w.x, acc[u][1] * w.y, acc[u][2] * w.z, acc[u][3] * w.w);
                bacc.x += r.x; bacc.y += r.y; bacc.z += r.z; bacc.w += r.w;
                *reinterpret_cast<float4*>(d_att_enc + o) = r;
            }
        }
    }
    float* mine = partial + ((long long)b * gridDim.x + blockIdx.x) * (2 * A + 4);
    if (a < A) { *reinterpret_cast<float4*>(mine + a) = wacc; *reinterpret_cast<float4*>(mine + A + a) = bacc; }
    const float tot = block_sum(de_sum, s_red);
    if (threadIdx.x == 0) { mine[2 * A] = tot; mine[2 * A + 1] = 0.f; mine[2 * A + 2] = 0.f; mine[2 * A + 3] = 0.f; }
}
__global__ void att_proj_bwd_kernel(int B, int T, int P, int A,
                                    const int* __restrict__ row_len,   // [B] number of active steps of row b
                                    const float* __restrict__ att_enc, const float* __restrict__ att_dec_all,
                                    long long ld_dec, const float* __restrict__ w_full,
                                    const float* __restrict__ d_e, float* __restrict__ d_att_enc,
                                    float* __restrict__ partial) {
    att_proj_bwd_body(B, T, P, A, row_len, att_enc, att_dec_all, ld_dec, w_full, d_e, d_att_enc, partial);
}
// blocks of more than 512 threads (A > 2048): the kernel above uses more than 64 registers, so 1024 threads would not fit the 64K
// registers of an SM; this instantiation caps them at 64
__global__ void __launch_bounds__(1024) att_proj_bwd_kernel_wide(int B, int T, int P, int A,
                                    const int* __restrict__ row_len,   // [B] number of active steps of row b
                                    const float* __restrict__ att_enc, const float* __restrict__ att_dec_all,
                                    long long ld_dec, const float* __restrict__ w_full,
                                    const float* __restrict__ d_e, float* __restrict__ d_att_enc,
                                    float* __restrict__ partial) {
    att_proj_bwd_body(B, T, P, A, row_len, att_enc, att_dec_all, ld_dec, w_full, d_e, d_att_enc, partial);
}

// Captions that share images: the same sums per IMAGE i over the (row, step) pairs of its rows,
//   d_att_enc[i,p,a] = w_full[a] * sum_{r in rows(i)} sum_{t < len_r} d_e[r,t,p] * [att_enc[i,p,a] + att_dec[t,r,a] > 0],
// formed directly (no per-row (B,P,A) tensor).  grid = (ceil(P/PROJ_IMG_PB), n_img), block = A/4 threads; a thread owns 4
// channels of the CTA's 4 pixels and keeps their sums in registers while the (row, step) pairs of the image pass through shared
// memory, PROJ_IMG_KC steps of one row at a time: rows in CSR order (ascending), then steps in order — deterministic.
// partial[(i*gridDim.x + chunk)*(2A+4)] as above.  smem: PROJ_IMG_KC*(A + PROJ_IMG_PB) + 40 floats.
constexpr int PROJ_IMG_PB = 4, PROJ_IMG_KC = 32;
__global__ void __launch_bounds__(1024) att_proj_bwd_img_kernel(int B, int T, int P, int A, const int* __restrict__ row_len,
                                        const int* __restrict__ row_ptr, const int* __restrict__ rows,
                                        const float* __restrict__ att_enc, const float* __restrict__ att_dec_all,
                                        long long ld_dec, const float* __restrict__ w_full,
                                        const float* __restrict__ d_e, float* __restrict__ d_att_enc,
                                        float* __restrict__ partial) {
    extern __shared__ __align__(16) float sm[];
    const int i = blockIdx.y, p0 = blockIdx.x * PROJ_IMG_PB;
    const int np = min(PROJ_IMG_PB, P - p0);
    float* s_dec = sm;                                   // PROJ_IMG_KC * A
    float* s_de = sm + (size_t)PROJ_IMG_KC * A;          // PROJ_IMG_KC * PROJ_IMG_PB
    float* s_red = s_de + PROJ_IMG_KC * PROJ_IMG_PB;     // 40
    const int a = threadIdx.x * 4;
    float x[4][4], acc[4][4];
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int c = 0; c < 4; ++c) { x[u][c] = 0.f; acc[u][c] = 0.f; }
    if (a < A) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const float4 raw = ld_stream_f4(att_enc + ((long long)i * P + p0 + min(u, np - 1)) * A + a);
            x[u][0] = raw.x; x[u][1] = raw.y; x[u][2] = raw.z; x[u][3] = raw.w;
        }
    }
    float4 wacc = make_float4(0.f, 0.f, 0.f, 0.f);
    float de_sum = 0.f;
    for (int k = row_ptr[i]; k < row_ptr[i + 1]; ++k) {
        const int b = rows[k], Tb = row_len[b];
        for (int t0 = 0; t0 < Tb; t0 += PROJ_IMG_KC) {
            const int nt = min(PROJ_IMG_KC, Tb - t0);
            __syncthreads();                             // the previous round is consumed
            for (int j = threadIdx.x; j < nt * (A >> 2); j += blockDim.x) {
                const int t = j / (A >> 2), a4 = (j % (A >> 2)) * 4;
                *reinterpret_cast<float4*>(s_dec + (size_t)t * A + a4) =
                    *reinterpret_cast<const float4*>(att_dec_all + ((long long)(t0 + t) * B + b) * ld_dec + a4);
            }
            for (int j = threadIdx.x; j < nt * PROJ_IMG_PB; j += blockDim.x) {
                const int t = j / PROJ_IMG_PB, pp = j % PROJ_IMG_PB;
                const float v = (pp < np) ? d_e[((long long)b * T + t0 + t) * P + p0 + pp] : 0.f;
                s_de[j] = v;
                de_sum += v;
            }
            __syncthreads();
            if (a < A) {
                for (int t = 0; t < nt; ++t) {
                    const float4 de4 = *reinterpret_cast<const float4*>(s_de + t * PROJ_IMG_PB);
                    const float4 d = *reinterpret_cast<const float4*>(s_dec + (size_t)t * A + a);
                    const float de[4] = {de4.x, de4.y, de4.z, de4.w};
                    const float dd[4] = {d.x, d.y, d.z, d.w};
                    float wl[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            const float sv = x[u][c] + dd[c];
                            acc[u][c] += (sv > 0.f) ? de[u] : 0.f;
                            wl[c] = fmaf(de[u], fmaxf(sv, 0.f), wl[c]);
                        }
                    }
                    wacc.x += wl[0]; wacc.y += wl[1]; wacc.z += wl[2]; wacc.w += wl[3];
                }
            }
        }
    }
    float4 bacc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (a < A) {
        const float4 w = *reinterpret_cast<const float4*>(w_full + a);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (u >= np) break;
            const long long o = ((long long)i * P + p0 + u) * A + a;
            const float4 r = make_float4(acc[u][0] * w.x, acc[u][1] * w.y, acc[u][2] * w.z, acc[u][3] * w.w);
            bacc.x += r.x; bacc.y += r.y; bacc.z += r.z; bacc.w += r.w;
            *reinterpret_cast<float4*>(d_att_enc + o) = r;
        }
    }
    float* mine = partial + ((long long)i * gridDim.x + blockIdx.x) * (2 * A + 4);
    if (a < A) { *reinterpret_cast<float4*>(mine + a) = wacc; *reinterpret_cast<float4*>(mine + A + a) = bacc; }
    const float tot = block_sum(de_sum, s_red);
    if (threadIdx.x == 0) { mine[2 * A] = tot; mine[2 * A + 1] = 0.f; mine[2 * A + 2] = 0.f; mine[2 * A + 3] = 0.f; }
}

struct BtPack { int v[ICD_MAX_STEPS]; };
__global__ void row_len_from_pack_kernel(int B, int T, const BtPack bt, int* __restrict__ row_len) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    int n = 0;
    for (int t = 0; t < T; ++t) n += (b < bt.v[t]) ? 1 : 0;
    row_len[b] = n;
}

}  // namespace

int icd_weighted_pixel_sum(int rows, int P, int C, const int32_t* img_index, const float* enc,
                           const float* alpha, int64_t ld_alpha, const float* fbeta_pre, int64_t ld_fb,
                           float* awe_raw, float* gate, float* gated, cudaStream_t s,
                           const int32_t* out_row_ptr, const int32_t* out_rows) {
    if (rows == 0) return 0;
    ICD_CHECK_ARG(C % 4 == 0, "attention: C=%d must be a multiple of 4", C);
    ICD_CHECK_ARG(!fbeta_pre || ld_fb % 4 == 0, "attention: ld_fb must be a multiple of 4");
    ICD_CHECK_ARG(rows <= 65535, "attention: rows=%d exceeds gridDim.y", rows);
    dim3 grid((C + WS_LANES * 4 - 1) / (WS_LANES * 4), rows);
    const size_t smem = (((P + 3) & ~3) + (WS_GROUPS - 1) * WS_LANES * 4) * sizeof(float);
    weighted_pixel_sum_kernel<<<grid, 256, smem, s>>>(P, C, img_index, enc, alpha, ld_alpha, fbeta_pre, ld_fb,
                                                      awe_raw, gate, gated, out_row_ptr, out_rows);
    ICD_LAUNCH_CHECK();
    return 0;
}

extern "C" int icd_attention_step_fwd(int rows, int P, int C, int A, const int32_t* img_index,
                                      const float* enc, const float* att_enc,
                                      const float* att_dec, int64_t ld_dec,
                                      const float* w_full, const float* b_full,
                                      const float* fbeta_pre, int64_t ld_fb,
                                      float* alpha, int64_t ld_alpha,
                                      float* awe_raw, float* gate, float* gated, void* stream) {
    cudaStream_t s = icd_stream(stream);
    if (rows == 0) return 0;
    ICD_CHECK_ARG(rows > 0 && P > 0 && C > 0 && A > 0, "attention_step_fwd: bad dims");
    ICD_CHECK_ARG(A % 4 == 0 && C % 4 == 0, "attention_step_fwd: A=%d and C=%d must be multiples of 4", A, C);
    ICD_CHECK_ARG(ld_dec % 4 == 0, "attention_step_fwd: ld_dec must be a multiple of 4");
    ICD_CHECK_ARG(!fbeta_pre || ld_fb % 4 == 0, "attention_step_fwd: ld_fb must be a multiple of 4");
    const size_t smem = (2 * (size_t)A + ((P + 3) & ~3) + 40) * sizeof(float);
    ICD_CHECK_ARG(smem <= 200 * 1024, "attention_step_fwd: A/P too large for shared memory");
    {
        static size_t configured = 48 * 1024;
        if (smem > configured) {
            ICD_CUDA(cudaFuncSetAttribute(att_step_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            configured = smem;
        }
    }
    icd_prof_mark_begin(0, rows, s);
    att_step_fwd_kernel<<<rows, 256, smem, s>>>(P, C, A, img_index, enc, att_enc, att_dec, ld_dec, w_full, b_full,
                                                 fbeta_pre, ld_fb, alpha, ld_alpha, awe_raw, gate, gated);
    icd_prof_mark_end(0, s);
    ICD_LAUNCH_CHECK();
    return 0;
}

extern "C" int icd_attention_step_bwd(int rows, int P, int C, int A,
                                      const float* enc, const float* att_enc,
                                      const float* att_dec, int64_t ld_dec, const float* w_full,
                                      const float* alpha, int64_t ld_alpha,
                                      const float* d_alpha_ext, int64_t ld_dalpha,
                                      const float* gate, const float* awe_raw, const float* d_gated,
                                      float* d_att_dec, int64_t ld_ddec,
                                      float* d_fbeta_pre, int64_t ld_dfb,
                                      float* d_e, int64_t ld_de, float* d_awe_out, void* stream) {
    return icd_attention_step_bwd_idx(rows, P, C, A, nullptr, enc, att_enc, att_dec, ld_dec, w_full, alpha, ld_alpha, d_alpha_ext,
                                      ld_dalpha, gate, awe_raw, d_gated, d_att_dec, ld_ddec, d_fbeta_pre, ld_dfb, d_e, ld_de,
                                      d_awe_out, stream);
}

int icd_attention_step_bwd_idx(int rows, int P, int C, int A, const int32_t* img_index,
                                      const float* enc, const float* att_enc,
                                      const float* att_dec, int64_t ld_dec, const float* w_full,
                                      const float* alpha, int64_t ld_alpha,
                                      const float* d_alpha_ext, int64_t ld_dalpha,
                                      const float* gate, const float* awe_raw, const float* d_gated,
                                      float* d_att_dec, int64_t ld_ddec,
                                      float* d_fbeta_pre, int64_t ld_dfb,
                                      float* d_e, int64_t ld_de, float* d_awe_out, void* stream) {
    cudaStream_t s = icd_stream(stream);
    if (rows == 0) return 0;
    ICD_CHECK_ARG(A % 4 == 0 && C % 4 == 0, "attention_step_bwd: A and C must be multiples of 4");
    ICD_CHECK_ARG(ld_dec % 4 == 0 && ld_ddec % 4 == 0 && ld_dfb % 4 == 0, "attention_step_bwd: row strides must be multiples of 4");
    const size_t smem = ((size_t)C + 2 * (size_t)A + 2 * ((P + 3) & ~3) + 40) * sizeof(float);
    ICD_CHECK_ARG(smem <= 200 * 1024, "attention_step_bwd: dims too large for shared memory");
    {
        static size_t configured = 48 * 1024;
        if (smem > configured) {
            ICD_CUDA(cudaFuncSetAttribute(att_step_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            configured = smem;
        }
    }
    icd_prof_mark_begin(1, rows, s);
    att_step_bwd_kernel<<<rows, 256, smem, s>>>(P, C, A, (const int*)img_index, enc, att_enc, att_dec, ld_dec, w_full, alpha, ld_alpha,
                                                 d_alpha_ext, ld_dalpha, gate, awe_raw, d_gated,
                                                 d_att_dec, ld_ddec, d_fbeta_pre, ld_dfb, d_e, ld_de, d_awe_out);
    icd_prof_mark_end(1, s);
    ICD_LAUNCH_CHECK();
    return 0;
}

extern "C" int64_t icd_attention_proj_bwd_ws_floats(int B, int P, int A) {
    const int64_t chunks = (P + PROJ_PB - 1) / PROJ_PB;
    // per-CTA partials (d_w_full[A] | d_b_enc[A] | sum d_e + pad) + [B] int row lengths (4-byte words at the end)
    // + A floats for the att_dec part of d_w_full (bf16 tier, icd_attention_proj_bwd_bf16_ex)
    return (int64_t)B * chunks * (2 * A + 4) + B + 8 + 49 * (int64_t)A;      // 49 = 1 + COLDOT_CHUNKS (attention_step_bf16.cu)
}

extern "C" int64_t icd_attention_proj_bwd_ws_floats_indexed(int B, int n_img, int P, int A) {
    // per-CTA partials of the per-image pass (its chunks are PROJ_IMG_PB = 4 pixels; the bf16 pass uses 8 and needs fewer)
    // + [B] row lengths + the att_dec part of d_w_full, as above
    const int64_t chunks = (P + PROJ_IMG_PB - 1) / PROJ_IMG_PB;
    return (int64_t)n_img * chunks * (2 * A + 4) + B + 8 + 49 * (int64_t)A;
}

// the row-length vector of both per-image passes sits behind their partials (n_img * chunks rows of 2A+4 floats)
int icd_attention_proj_bwd_indexed(int B, int n_img, int T, int P, int A, const int32_t* bt_host, const int32_t* row_ptr,
                                   const int32_t* rows, const float* att_enc, const float* att_dec_all, int64_t ld_dec,
                                   const float* w_full, const float* d_e, float* d_att_enc, float* d_w_full, float* d_b_full,
                                   float* d_b_enc, float* partial, cudaStream_t s) {
    ICD_CHECK_ARG(T > 0 && T <= ICD_MAX_STEPS, "attention_proj_bwd: T=%d out of range", T);
    ICD_CHECK_ARG(A % 4 == 0 && A / 4 <= 1024, "attention_proj_bwd: A=%d unsupported", A);
    ICD_CHECK_ARG(ld_dec % 4 == 0, "attention_proj_bwd: ld_dec must be a multiple of 4");
    ICD_CHECK_ARG(n_img > 0 && n_img <= 65535, "attention_proj_bwd: n_img=%d out of range", n_img);
    const int chunks = (P + PROJ_IMG_PB - 1) / PROJ_IMG_PB;
    const int W = 2 * A + 4;
    int* row_len = reinterpret_cast<int*>(partial + (int64_t)n_img * chunks * W);
    BtPack pack;
    for (int t = 0; t < ICD_MAX_STEPS; ++t) pack.v[t] = t < T ? bt_host[t] : 0;
    row_len_from_pack_kernel<<<(B + 127) / 128, 128, 0, s>>>(B, T, pack, row_len);
    ICD_LAUNCH_CHECK();
    const size_t smem = ((size_t)PROJ_IMG_KC * (A + PROJ_IMG_PB) + 40) * sizeof(float);
    ICD_CHECK_ARG(smem <= 220 * 1024, "attention_proj_bwd: A too large for shared memory");
    static size_t configured = 48 * 1024;
    if (smem > configured) {
        ICD_CUDA(cudaFuncSetAttribute(att_proj_bwd_img_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = smem;
    }
    const int threads = ((A / 4 + 31) / 32) * 32;
    att_proj_bwd_img_kernel<<<dim3(chunks, n_img), threads, smem, s>>>(B, T, P, A, row_len, row_ptr, rows, att_enc, att_dec_all,
                                                                        ld_dec, w_full, d_e, d_att_enc, partial);
    ICD_LAUNCH_CHECK();
    ICD_TRY(icd_colsum(partial, W, (int64_t)n_img * chunks, A, nullptr, d_w_full, s));
    if (d_b_enc) ICD_TRY(icd_colsum(partial + A, W, (int64_t)n_img * chunks, A, nullptr, d_b_enc, s));
    ICD_TRY(icd_colsum(partial + 2 * A, W, (int64_t)n_img * chunks, 1, nullptr, d_b_full, s));
    return 0;
}

extern "C" int icd_attention_proj_bwd(int B, int T, int P, int A, const int32_t* bt_host,
                                      const float* att_enc, const float* att_dec_all, int64_t ld_dec,
                                      const float* w_full, const float* d_e,
                                      float* d_att_enc, float* d_w_full, float* d_b_full, float* d_b_enc,
                                      float* partial, void* stream) {
    cudaStream_t s = icd_stream(stream);
    ICD_CHECK_ARG(T > 0 && T <= ICD_MAX_STEPS, "attention_proj_bwd: T=%d out of range", T);
    ICD_CHECK_ARG(A % 4 == 0 && A / 4 <= 1024, "attention_proj_bwd: A=%d unsupported", A);
    ICD_CHECK_ARG(ld_dec % 4 == 0, "attention_proj_bwd: ld_dec must be a multiple of 4");
    ICD_CHECK_ARG(B <= 65535, "attention_proj_bwd: B too large");
    const int chunks = (P + PROJ_PB - 1) / PROJ_PB;
    const int W = 2 * A + 4;
    int* row_len = reinterpret_cast<int*>(partial + (int64_t)B * chunks * W);
    BtPack pack;
    for (int t = 0; t < ICD_MAX_STEPS; ++t) pack.v[t] = t < T ? bt_host[t] : 0;
    row_len_from_pack_kernel<<<(B + 127) / 128, 128, 0, s>>>(B, T, pack, row_len);
    ICD_LAUNCH_CHECK();
    const size_t smem = ((size_t)T * A + (size_t)T * PROJ_PB + 40) * sizeof(float);
    ICD_CHECK_ARG(smem <= 220 * 1024, "attention_proj_bwd: T*A too large for shared memory");
    {
        static size_t configured = 48 * 1024;
        if (smem > configured) {
            ICD_CUDA(cudaFuncSetAttribute(att_proj_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            ICD_CUDA(cudaFuncSetAttribute(att_proj_bwd_kernel_wide, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            configured = smem;
        }
    }
    int threads = ((A / 4 + 31) / 32) * 32;
    dim3 grid(chunks, B);
    if (threads > 512)
        att_proj_bwd_kernel_wide<<<grid, threads, smem, s>>>(B, T, P, A, row_len, att_enc, att_dec_all, ld_dec, w_full,
                                                               d_e, d_att_enc, partial);
    else
        att_proj_bwd_kernel<<<grid, threads, smem, s>>>(B, T, P, A, row_len, att_enc, att_dec_all, ld_dec, w_full,
                                                              d_e, d_att_enc, partial);
    ICD_LAUNCH_CHECK();
    // reduce the per-CTA partials: [0,A) -> d_w_full, [A,2A) -> d enc_att.bias, column 2A -> d_b_full
    ICD_TRY(icd_colsum(partial, W, (int64_t)B * chunks, A, nullptr, d_w_full, s));
    if (d_b_enc) ICD_TRY(icd_colsum(partial + A, W, (int64_t)B * chunks, A, nullptr, d_b_enc, s));
    ICD_TRY(icd_colsum(partial + 2 * A, W, (int64_t)B * chunks, 1, nullptr, d_b_full, s));
    return 0;
}

// Caption-generation variant (internal): rows img*k + j, j < k_live[img], of image img are served by one CTA.
template <int K>
static int launch_grouped(int n_img, int k, int P, int C, int A, const int* k_live, const float* enc, const float* att_enc,
                          const float* att_dec, int64_t ld_dec, const float* w_full, const float* b_full,
                          const float* fbeta_pre, int64_t ld_fb, float* alpha, int64_t ld_alpha, float* gated,
                          const int* slot_img, const int* n_slots, const int* row_off, cudaStream_t s, void* gated_x3, int* ticket, int x3_nseg) {
    const size_t smem = ((size_t)K * A + A + (size_t)K * ((P + 3) & ~3)) * sizeof(float);
    // ring variant (persistent CTAs, bulk-async shared-memory ring): needs one ring slot to hold 14 att_enc rows / 4 enc rows,
    // 16-byte aligned streams, and the ring + the staged rows within the 227 KB of one SM.  ICD_BEAM_ATT_RING=0 keeps the
    // register-staged kernel (A/B runs, equivalence test).
    {
        const char* ring_env = getenv("ICD_BEAM_ATT_RING");      // read per call: the equivalence test toggles it
        const bool ring_off = ring_env && atoi(ring_env) == 0;
        const size_t ring_smem = (size_t)RING_SLOTS * RING_SLOT_BYTES + smem + 2 * 8 * RING_SLOTS + 16;
        const bool aligned = ((reinterpret_cast<uintptr_t>(enc) | reinterpret_cast<uintptr_t>(att_enc) |
                               reinterpret_cast<uintptr_t>(att_dec) | reinterpret_cast<uintptr_t>(fbeta_pre)) & 15) == 0;
        if (!ring_off && aligned && (size_t)RING_ROWS1 * A * 4 <= RING_SLOT_BYTES && (size_t)RING_ROWS2 * C * 4 <= RING_SLOT_BYTES &&
            C <= RING_CONS * 8 && ring_smem <= 227 * 1024) {
            static size_t ring_configured = 0;
            if (ring_smem > ring_configured) {
                ICD_CUDA(cudaFuncSetAttribute(att_step_fwd_grouped_ring_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                              (int)ring_smem));
                ring_configured = ring_smem;
            }
            const int per_sm = (ring_smem + 1024) * 2 <= 228 * 1024 ? 2 : 1;
            // anti-phase start of the second CTA per SM: only with dynamic slot tickets (else the late CTAs would finish late)
            const char* stag_env = getenv("ICD_RING_STAGGER_NS");
            const int stagger = (ticket && per_sm == 2 && n_img > ICD_NUM_SMS && k > 1) ? (stag_env ? atoi(stag_env) : 10000) : 0;
            att_step_fwd_grouped_ring_kernel<K><<<std::min(n_img, per_sm * ICD_NUM_SMS), RING_THREADS, ring_smem, s>>>(
                n_img, k, P, C, A, k_live, enc, att_enc, att_dec, ld_dec, w_full, b_full, fbeta_pre, ld_fb, alpha, ld_alpha, gated,
                slot_img, n_slots, row_off, reinterpret_cast<unsigned short*>(gated_x3), ticket, stagger, x3_nseg);
            ICD_LAUNCH_CHECK();
            return 0;
        }
    }
    ICD_CHECK_ARG(smem <= 200 * 1024, "attention_step_fwd_grouped: K*A too large for shared memory");
    static size_t configured = 48 * 1024;
    if (smem > configured) {
        ICD_CUDA(cudaFuncSetAttribute(att_step_fwd_grouped_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = smem;
    }
    att_step_fwd_grouped_kernel<K><<<n_img, 256, smem, s>>>(k, P, C, A, k_live, enc, att_enc, att_dec, ld_dec, w_full, b_full,
                                                            fbeta_pre, ld_fb, alpha, ld_alpha, gated, slot_img, n_slots, row_off,
                                                            reinterpret_cast<unsigned short*>(gated_x3), x3_nseg);
    ICD_LAUNCH_CHECK();
    return 0;
}

int icd_attention_step_fwd_grouped(int n_img, int k, int P, int C, int A, const int* k_live, const float* enc,
                                   const float* att_enc, const float* att_dec, int64_t ld_dec, const float* w_full,
                                   const float* b_full, const float* fbeta_pre, int64_t ld_fb, float* alpha,
                                   int64_t ld_alpha, float* gated, const int* slot_img, const int* n_slots, const int* row_off,
                                   cudaStream_t s, void* gated_x3, int* ticket, int x3_nseg) {
    if (n_img == 0) return 0;
    ICD_CHECK_ARG(!gated_x3 || C % 8 == 0, "attention_step_fwd_grouped: the fused 3-term split needs C % 8 == 0");
    ICD_CHECK_ARG(k >= 1 && k <= 8, "attention_step_fwd_grouped: k=%d (1..8)", k);
    ICD_CHECK_ARG(A % 4 == 0 && C % 4 == 0 && ld_dec % 4 == 0 && ld_fb % 4 == 0, "attention_step_fwd_grouped: misaligned dims");
#define ICD_GROUPED(KK) return launch_grouped<KK>(n_img, k, P, C, A, k_live, enc, att_enc, att_dec, ld_dec, w_full, b_full, \
                                                  fbeta_pre, ld_fb, alpha, ld_alpha, gated, slot_img, n_slots, row_off, s, gated_x3, ticket, x3_nseg)
    switch (k) {
        case 1: ICD_GROUPED(1);
        case 2: ICD_GROUPED(2);
        case 3: ICD_GROUPED(3);
        case 4: ICD_GROUPED(4);
        case 5: ICD_GROUPED(5);
        case 6: ICD_GROUPED(6);
        default: ICD_GROUPED(8);
    }
#undef ICD_GROUPED
}

// ------------------------------------------------------------------------------------------------
// Encoder gradient, attention + initial-state part (models/attention.py:59-60 and :161):
//   d_enc[b,p,c] = sum_{t < len_b} alpha[b,t,p] * d_awe[t,b,c]  +  d_mean[b,c] / P          (written, not accumulated)
// The enc_att part, d_att_enc W_e, is added afterwards by a contraction with beta = 1.
// grid = (ceil(C/1024), B), block = 256 threads x 4 channels; d_awe of up to 32 steps lives in registers, alphas in smem.
// row_ptr != NULL (captions that share images): CTA row i is image i and d_enc[i] is the sum of the above over the rows
// rows[row_ptr[i] .. row_ptr[i+1]), added in that order (an image without rows gets zeros).
// ------------------------------------------------------------------------------------------------
namespace {
constexpr int EG_TCH = 32;
__global__ void __launch_bounds__(256, 1) enc_grad_kernel(int B, int T, int P, int C, const int* __restrict__ row_len,
                                                          const int* __restrict__ row_ptr, const int* __restrict__ rows,
                                                          const float* __restrict__ alphas,      // (B,T,P)
                                                          const float* __restrict__ d_awe_all,   // (T,B,C)
                                                          const float* __restrict__ d_mean,      // (B,C) or NULL
                                                          float* __restrict__ d_enc) {           // (B,P,C)
    extern __shared__ __align__(16) float sm[];     // EG_TCH * P alphas of the current step chunk
    const int img = blockIdx.y;
    const int c = blockIdx.x * 1024 + threadIdx.x * 4;
    const float invP = 1.f / (float)P;
    const int k0 = row_ptr ? row_ptr[img] : img, k1 = row_ptr ? row_ptr[img + 1] : img + 1;
    if (k0 == k1 && c < C)
        for (int p = 0; p < P; ++p) *reinterpret_cast<float4*>(d_enc + ((long long)img * P + p) * C + c) = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int k = k0; k < k1; ++k) {
        const int b = row_ptr ? rows[k] : img;
        const int Tb = row_len ? row_len[b] : T;
        for (int t0 = 0; t0 < max(Tb, 1); t0 += EG_TCH) {
            const int nt = min(EG_TCH, Tb - t0);
            __syncthreads();
            for (int j = threadIdx.x; j < max(nt, 0) * P; j += blockDim.x)
                sm[j] = alphas[((long long)b * T + t0 + j / P) * P + (j % P)];
            __syncthreads();
            if (c >= C) continue;
            float4 da[EG_TCH];
#pragma unroll
            for (int u = 0; u < EG_TCH; ++u)
                da[u] = (u < nt) ? *reinterpret_cast<const float4*>(d_awe_all + ((long long)(t0 + u) * B + b) * C + c)
                                 : make_float4(0.f, 0.f, 0.f, 0.f);
            float4 base = make_float4(0.f, 0.f, 0.f, 0.f);
            if (t0 == 0 && d_mean) {
                const float4 m = *reinterpret_cast<const float4*>(d_mean + (long long)b * C + c);
                base = make_float4(m.x * invP, m.y * invP, m.z * invP, m.w * invP);
            }
            for (int p = 0; p < P; ++p) {
                float4 acc = base;
                float* o = d_enc + ((long long)img * P + p) * C + c;
                if (t0 > 0) acc = *reinterpret_cast<const float4*>(o);
                else if (k > k0) {                                    // a later row of the image: add to the rows before it
                    const float4 prev = *reinterpret_cast<const float4*>(o);
                    acc = make_float4(prev.x + base.x, prev.y + base.y, prev.z + base.z, prev.w + base.w);
                }
#pragma unroll
                for (int u = 0; u < EG_TCH; ++u) {
                    if (u < nt) {
                        const float al = sm[u * P + p];
                        acc.x = fmaf(al, da[u].x, acc.x); acc.y = fmaf(al, da[u].y, acc.y);
                        acc.z = fmaf(al, da[u].z, acc.z); acc.w = fmaf(al, da[u].w, acc.w);
                    }
                }
                *reinterpret_cast<float4*>(o) = acc;
            }
        }
    }
}
}  // namespace

extern "C" int icd_attention_enc_grad(int B, int T, int P, int C, const int32_t* bt_host,
                                      const float* alphas, const float* d_awe_all, const float* d_mean,
                                      float* d_enc, int32_t* row_len_ws, void* stream) {
    return icd_attention_enc_grad_indexed(B, B, T, P, C, bt_host, nullptr, nullptr, alphas, d_awe_all, d_mean, d_enc, row_len_ws,
                                          icd_stream(stream));
}

int icd_attention_enc_grad_indexed(int B, int n_img, int T, int P, int C, const int32_t* bt_host, const int32_t* row_ptr,
                                   const int32_t* rows, const float* alphas, const float* d_awe_all, const float* d_mean,
                                   float* d_enc, int32_t* row_len_ws, cudaStream_t s) {
    ICD_CHECK_ARG(B > 0 && T > 0 && T <= ICD_MAX_STEPS && C % 4 == 0 && B <= 65535, "attention_enc_grad: bad dims");
    ICD_CHECK_ARG(n_img > 0 && n_img <= 65535 && (row_ptr != nullptr || n_img == B), "attention_enc_grad: bad image count");
    ICD_CHECK_ARG(alphas && d_awe_all && d_enc, "attention_enc_grad: null argument");
    int* row_len = nullptr;
    if (bt_host) {
        ICD_CHECK_ARG(row_len_ws != nullptr, "attention_enc_grad: row_len_ws (B ints) required with bt_host");
        BtPack pack;
        for (int t = 0; t < ICD_MAX_STEPS; ++t) pack.v[t] = t < T ? bt_host[t] : 0;
        row_len_from_pack_kernel<<<(B + 127) / 128, 128, 0, s>>>(B, T, pack, row_len_ws);
        ICD_LAUNCH_CHECK();
        row_len = row_len_ws;
    }
    const size_t smem = (size_t)EG_TCH * P * sizeof(float);
    ICD_CHECK_ARG(smem <= 200 * 1024, "attention_enc_grad: P too large");
    static size_t configured = 48 * 1024;
    if (smem > configured) {
        ICD_CUDA(cudaFuncSetAttribute(enc_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = smem;
    }
    dim3 grid((C + 1023) / 1024, n_img);
    enc_grad_kernel<<<grid, 256, smem, s>>>(B, T, P, C, row_len, (const int*)row_ptr, (const int*)rows, alphas, d_awe_all, d_mean, d_enc);
    ICD_LAUNCH_CHECK();
    return 0;
}
