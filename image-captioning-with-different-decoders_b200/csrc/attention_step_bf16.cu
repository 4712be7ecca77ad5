// Fused additive-attention step kernels for bf16-STORED features (the tensor-core tier; BASELINE.json configs[2] allows
// the 14x14x2048 features and their enc_att projection to be stored in bf16).  Arithmetic is fp32 throughout; only the
// two big HBM streams — enc (P x C) and att_enc (P x A) per image — are read as bf16, halving the bytes of the
// HBM-bound step: 196*2048*2 + 196*512*2 + small = 1 022 736 B per (image, step) forward (SURVEY.md 8d).
// Same math and same reference lines as attention_step.cu (models/attention.py:55-60, 270-271).
#include "common.cuh"
#include <stdlib.h>
#include <cuda_bf16.h>

namespace {

__device__ __forceinline__ uint4 ld_stream_u4(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ uint2 ld_stream_u2(const void* p) {
    uint2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}
// 8 packed bf16 -> 8 floats (element 2i in the low half of word i)
__device__ __forceinline__ void unpack8(const uint4& v, float (&f)[8]) {
    f[0] = __uint_as_float(v.x << 16); f[1] = __uint_as_float(v.x & 0xffff0000u);
    f[2] = __uint_as_float(v.y << 16); f[3] = __uint_as_float(v.y & 0xffff0000u);
    f[4] = __uint_as_float(v.z << 16); f[5] = __uint_as_float(v.z & 0xffff0000u);
    f[6] = __uint_as_float(v.w << 16); f[7] = __uint_as_float(v.w & 0xffff0000u);
}
__device__ __forceinline__ uint32_t pack2(float a, float b) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&h);
}

// m16n8k16 bf16 x bf16 -> fp32 warp MMA (legacy tensor path; used here as a batched matrix-vector product: the k index of
// A and B may be ANY consistent permutation of the contraction index, which lets A fragments come straight from 128-bit
// global loads of row-major bf16 features with no shuffles or shared-memory transposes)
__device__ __forceinline__ void mma_bf16_16816(float& d0, float& d1, float& d2, float& d3,
                                               uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d0), "+f"(d1), "+f"(d2), "+f"(d3) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// ------------------------------------------------------------------------------------------------
// forward: one kernel per decode step, grid = rows, block = 256.
// ------------------------------------------------------------------------------------------------
constexpr int FW16_ROWS = 4;      // pixel rows per warp iteration in the score phase
constexpr int FW16_UNROLL = 8;    // pixel rows in flight per thread in the weighted-sum phase
// rows per launch at or below which a row is shared by 4 / 2 CTAs (att_step_fwd_bf16_split_kernel); fitted on att_bench.py
constexpr int ICD_ATT_FWD_SPLIT4_ROWS = 48;      // 16-32 rows: 35 -> 27 us; 100 rows: two CTAs per row are better (33 us vs 34)
constexpr int ICD_ATT_FWD_SPLIT2_ROWS = 222;     // = 1.5 x 148 (three CTAs per SM when shared by two): 200 rows 45.7 -> 43.5 us, 256 rows lose
// rows per launch at or below which the backward runs EVERY row as two half-row CTAs (its row-balance machinery, see the kernel)
constexpr int ICD_ATT_BWD_SPLIT_ALL_ROWS = 222;  // 32 rows 43 -> 34 us, 148 rows 46 -> 37, 200 rows 51.5 -> 44; 256 rows: no gain

// phases 1 + 2 of the forward step for ONE row: scores e_p = w_full . relu(att_enc[p, :] + att_dec) + b_full over the row's pixels
// (att_enc streamed once), softmax over the pixels; alpha is left in s_e and, when `out` is given, written to global memory.
template <bool HAS_OUT,      // true: `out` is known to be non-null (no test in the whole-row kernel)
          int ROWS = FW16_ROWS, int JU = 1>   // pixel rows per warp iteration x 16-byte chunks per lane in flight (the few-rows kernels, which
                                              // have the register file of an SM almost to themselves, keep 16 loads in flight per lane)
__device__ __forceinline__ void fwd16_scores_softmax(int P, int A, const __nv_bfloat16* ae,
                                                     const float* b_full, float* s_dec, float* s_wf, float* s_e,
                                                     float* s_red, float* out) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    const float bfull = b_full ? b_full[0] : 0.f;
    const int A8 = A >> 3;
    // phase 1: scores; ROWS pixel rows per warp iteration, 16 B per lane per row chunk
    for (int p0 = warp; p0 < P; p0 += ROWS * nwarp) {
        float acc[ROWS];
#pragma unroll
        for (int u = 0; u < ROWS; ++u) acc[u] = 0.f;
        for (int j0 = lane; j0 < A8; j0 += 32 * JU) {
            uint4 x[JU][ROWS];
#pragma unroll
            for (int ju = 0; ju < JU; ++ju) {
                const int j = j0 + 32 * ju;
#pragma unroll
                for (int u = 0; u < ROWS; ++u) {
                    const int p = p0 + u * nwarp;                 // warp-uniform: rows past P are not loaded at all
                    x[ju][u] = (p < P && (JU == 1 || j < A8)) ? ld_stream_u4(ae + (long long)p * A + 8 * j) : make_uint4(0u, 0u, 0u, 0u);
                }
            }
#pragma unroll
            for (int ju = 0; ju < JU; ++ju) {
                const int j = j0 + 32 * ju;
                if (JU > 1 && j >= A8) break;                     // (the chunks of a lane are added in the same order for every JU)
                const float4 d0 = *reinterpret_cast<const float4*>(s_dec + 8 * j);
                const float4 d1 = *reinterpret_cast<const float4*>(s_dec + 8 * j + 4);
                const float4 w0 = *reinterpret_cast<const float4*>(s_wf + 8 * j);
                const float4 w1 = *reinterpret_cast<const float4*>(s_wf + 8 * j + 4);
                const float dd[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
                const float ww[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
                for (int u = 0; u < ROWS; ++u) {
                    float f[8];
                    unpack8(x[ju][u], f);
#pragma unroll
                    for (int i = 0; i < 8; ++i) acc[u] = fmaf(fmaxf(f[i] + dd[i], 0.f), ww[i], acc[u]);
                }
            }
        }
#pragma unroll
        for (int u = 0; u < ROWS; ++u) {
            const float v = warp_sum(acc[u]);
            const int p = p0 + u * nwarp;
            if (lane == 0 && p < P) s_e[p] = v + bfull;
        }
    }
    __syncthreads();
    // phase 2: softmax over pixels
    float m = -INFINITY;
    for (int p = threadIdx.x; p < P; p += blockDim.x) m = fmaxf(m, s_e[p]);
    m = block_max(m, s_red);
    float sum = 0.f;
    for (int p = threadIdx.x; p < P; p += blockDim.x) { const float ex = expf(s_e[p] - m); s_e[p] = ex; sum += ex; }
    sum = block_sum(sum, s_red);
    if (HAS_OUT || out) {
        for (int p = threadIdx.x; p < P; p += blockDim.x) { const float al = s_e[p] / sum; s_e[p] = al; out[p] = al; }
    } else {
        for (int p = threadIdx.x; p < P; p += blockDim.x) s_e[p] = s_e[p] / sum;
    }
    __syncthreads();
}

__global__ void __launch_bounds__(256, 4) att_step_fwd_bf16_kernel(
        int P, int C, int A, const int* __restrict__ img_index,
        const __nv_bfloat16* __restrict__ enc, const __nv_bfloat16* __restrict__ att_enc,
        const float* __restrict__ att_dec, long long ld_dec,
        const float* __restrict__ w_full, const float* __restrict__ b_full,
        const float* __restrict__ fbeta_pre, long long ld_fb,
        float* __restrict__ alpha, long long ld_alpha,
        float* __restrict__ awe_raw, float* __restrict__ gate, float* __restrict__ gated,
        __nv_bfloat16* __restrict__ gated16) {
    extern __shared__ __align__(16) float sm[];
    float* s_dec = sm;
    float* s_wf = sm + A;
    float* s_e = sm + 2 * A;
    float* s_red = s_e + ((P + 3) & ~3);
    const int r = blockIdx.x;
    pdl_trigger();
    pdl_wait();
    const int img = img_index ? img_index[r] : r;
    const __nv_bfloat16* ae = att_enc + (long long)img * P * A;
    const float* dec = att_dec + (long long)r * ld_dec;
    for (int a = threadIdx.x; a < A; a += blockDim.x) { s_dec[a] = dec[a]; s_wf[a] = w_full[a]; }
    __syncthreads();
    fwd16_scores_softmax<true>(P, A, ae, b_full, s_dec, s_wf, s_e, s_red, alpha + (long long)r * ld_alpha);
    // phase 3: alpha-weighted sum; thread owns 8 consecutive channels (16 B), FW16_UNROLL pixel rows in flight
    const __nv_bfloat16* eb = enc + (long long)img * P * C;
    for (int c = threadIdx.x * 8; c < C; c += blockDim.x * 8) {
        float acc[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] = 0.f;
        int p = 0;
        for (; p + FW16_UNROLL <= P; p += FW16_UNROLL) {
            uint4 x[FW16_UNROLL];
#pragma unroll
            for (int u = 0; u < FW16_UNROLL; ++u) x[u] = ld_stream_u4(eb + (long long)(p + u) * C + c);
#pragma unroll
            for (int u = 0; u < FW16_UNROLL; ++u) {
                const float al = s_e[p + u];
                float f[8];
                unpack8(x[u], f);
#pragma unroll
                for (int i = 0; i < 8; ++i) acc[i] = fmaf(al, f[i], acc[i]);
            }
        }
        for (; p < P; ++p) {
            const uint4 x = ld_stream_u4(eb + (long long)p * C + c);
            const float al = s_e[p];
            float f[8];
            unpack8(x, f);
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[i] = fmaf(al, f[i], acc[i]);
        }
        const long long o = (long long)r * C + c;
        if (awe_raw) {
            *reinterpret_cast<float4*>(awe_raw + o) = make_float4(acc[0], acc[1], acc[2], acc[3]);
            *reinterpret_cast<float4*>(awe_raw + o + 4) = make_float4(acc[4], acc[5], acc[6], acc[7]);
        }
        if (fbeta_pre) {
            const float4 f0 = *reinterpret_cast<const float4*>(fbeta_pre + (long long)r * ld_fb + c);
            const float4 f1 = *reinterpret_cast<const float4*>(fbeta_pre + (long long)r * ld_fb + c + 4);
            const float g[8] = {sigmoidf_(f0.x), sigmoidf_(f0.y), sigmoidf_(f0.z), sigmoidf_(f0.w),
                                sigmoidf_(f1.x), sigmoidf_(f1.y), sigmoidf_(f1.z), sigmoidf_(f1.w)};
            float gd[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) gd[i] = g[i] * acc[i];
            if (gate) {
                *reinterpret_cast<float4*>(gate + o) = make_float4(g[0], g[1], g[2], g[3]);
                *reinterpret_cast<float4*>(gate + o + 4) = make_float4(g[4], g[5], g[6], g[7]);
            }
            if (gated) {
                *reinterpret_cast<float4*>(gated + o) = make_float4(gd[0], gd[1], gd[2], gd[3]);
                *reinterpret_cast<float4*>(gated + o + 4) = make_float4(gd[4], gd[5], gd[6], gd[7]);
            }
            if (gated16) {
                uint4 pk = make_uint4(pack2(gd[0], gd[1]), pack2(gd[2], gd[3]), pack2(gd[4], gd[5]), pack2(gd[6], gd[7]));
                *reinterpret_cast<uint4*>(gated16 + o) = pk;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// forward, FEW rows per launch (ragged batches late in the caption, small batches): a row is shared by S = 8 / CH CTAs so that a launch
// of fewer rows than the GPU has CTA slots still keeps every SM streaming.  CTA (r, s) forms ALL scores of row r (the S readers of the
// row's att_enc, 20 % of its bytes, meet in L2) and the weighted sum of channels [s C / S, (s + 1) C / S); a thread owns CH consecutive
// channels and keeps FW16_UNROLL * S pixel rows in flight (the same bytes per thread as the whole-row kernel).  Every output element is
// formed by the same operations in the same order as in the whole-row kernel: the results are bit-identical (tested).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned ld_stream_u1(const void* p) {
    unsigned r;
    asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}
template <int CH> struct StreamChunk;
template <> struct StreamChunk<4> {
    uint2 v;
    __device__ __forceinline__ void load(const void* p) { v = ld_stream_u2(p); }
    __device__ __forceinline__ void unpack(float (&f)[4]) const {
        f[0] = __uint_as_float(v.x << 16); f[1] = __uint_as_float(v.x & 0xffff0000u);
        f[2] = __uint_as_float(v.y << 16); f[3] = __uint_as_float(v.y & 0xffff0000u);
    }
};
template <> struct StreamChunk<2> {
    unsigned v;
    __device__ __forceinline__ void load(const void* p) { v = ld_stream_u1(p); }
    __device__ __forceinline__ void unpack(float (&f)[2]) const {
        f[0] = __uint_as_float(v << 16); f[1] = __uint_as_float(v & 0xffff0000u);
    }
};

template <int CH, bool DEEP>   // DEEP (at most two CTAs per SM: <= 148 rows shared by two, <= 48 by four): 128 registers, 16 score-phase loads
                               // per lane in flight instead of 4 — a launch of few rows is bound by the chain of dependent load batches
__global__ void __launch_bounds__(256, DEEP ? 2 : 4) att_step_fwd_bf16_split_kernel(
        int P, int C, int A, const int* __restrict__ img_index,
        const __nv_bfloat16* __restrict__ enc, const __nv_bfloat16* __restrict__ att_enc,
        const float* __restrict__ att_dec, long long ld_dec,
        const float* __restrict__ w_full, const float* __restrict__ b_full,
        const float* __restrict__ fbeta_pre, long long ld_fb,
        float* __restrict__ alpha, long long ld_alpha,
        float* __restrict__ awe_raw, float* __restrict__ gate, float* __restrict__ gated,
        __nv_bfloat16* __restrict__ gated16) {
    constexpr int S = 8 / CH;
    constexpr int UN = FW16_UNROLL * S;
    extern __shared__ __align__(16) float sm[];
    float* s_dec = sm;
    float* s_wf = sm + A;
    float* s_e = sm + 2 * A;
    float* s_red = s_e + ((P + 3) & ~3);
    const int r = blockIdx.x / S, part = blockIdx.x % S;
    pdl_trigger();
    pdl_wait();
    const int img = img_index ? img_index[r] : r;
    const __nv_bfloat16* ae = att_enc + (long long)img * P * A;
    const float* dec = att_dec + (long long)r * ld_dec;
    for (int a = threadIdx.x; a < A; a += blockDim.x) { s_dec[a] = dec[a]; s_wf[a] = w_full[a]; }
    __syncthreads();
    fwd16_scores_softmax<false, DEEP ? 8 : FW16_ROWS, DEEP ? 2 : 1>(P, A, ae, b_full, s_dec, s_wf, s_e, s_red,
                                                                     part == 0 ? alpha + (long long)r * ld_alpha : nullptr);
    // phase 3: this CTA's channel range, CH channels per thread
    const __nv_bfloat16* eb = enc + (long long)img * P * C;
    const int cw = C / S;                                         // C % 8 == 0: cw is a multiple of CH
    for (int c = part * cw + threadIdx.x * CH; c < (part + 1) * cw; c += blockDim.x * CH) {
        float acc[CH];
#pragma unroll
        for (int i = 0; i < CH; ++i) acc[i] = 0.f;
        int p = 0;
        for (; p + UN <= P; p += UN) {
            StreamChunk<CH> x[UN];
#pragma unroll
            for (int u = 0; u < UN; ++u) x[u].load(eb + (long long)(p + u) * C + c);
#pragma unroll
            for (int u = 0; u < UN; ++u) {
                const float al = s_e[p + u];
                float f[CH];
                x[u].unpack(f);
#pragma unroll
                for (int i = 0; i < CH; ++i) acc[i] = fmaf(al, f[i], acc[i]);
            }
        }
        if (!DEEP) {                                              // (at 64 registers a second batched block costs the main loop its batching)
            for (; p < P; ++p) {
                StreamChunk<CH> x;
                x.load(eb + (long long)p * C + c);
                const float al = s_e[p];
                float f[CH];
                x.unpack(f);
#pragma unroll
                for (int i = 0; i < CH; ++i) acc[i] = fmaf(al, f[i], acc[i]);
            }
        } else if (p < P) {                                       // the remaining pixel rows as ONE batch of loads (not one round trip each)
            StreamChunk<CH> x[UN];
#pragma unroll
            for (int u = 0; u < UN; ++u)
                if (p + u < P) x[u].load(eb + (long long)(p + u) * C + c);
#pragma unroll
            for (int u = 0; u < UN; ++u) {
                if (p + u < P) {
                    const float al = s_e[p + u];
                    float f[CH];
                    x[u].unpack(f);
#pragma unroll
                    for (int i = 0; i < CH; ++i) acc[i] = fmaf(al, f[i], acc[i]);
                }
            }
        }
        const long long o = (long long)r * C + c;
        if (awe_raw) {
#pragma unroll
            for (int i = 0; i < CH; i += 2) *reinterpret_cast<float2*>(awe_raw + o + i) = make_float2(acc[i], acc[i + 1]);
        }
        if (fbeta_pre) {
            float g[CH], gd[CH];
#pragma unroll
            for (int i = 0; i < CH; i += 2) {
                const float2 f = *reinterpret_cast<const float2*>(fbeta_pre + (long long)r * ld_fb + c + i);
                g[i] = sigmoidf_(f.x);
                g[i + 1] = sigmoidf_(f.y);
            }
#pragma unroll
            for (int i = 0; i < CH; ++i) gd[i] = g[i] * acc[i];
#pragma unroll
            for (int i = 0; i < CH; i += 2) {
                if (gate) *reinterpret_cast<float2*>(gate + o + i) = make_float2(g[i], g[i + 1]);
                if (gated) *reinterpret_cast<float2*>(gated + o + i) = make_float2(gd[i], gd[i + 1]);
                if (gated16) *reinterpret_cast<uint32_t*>(gated16 + o + i) = pack2(gd[i], gd[i + 1]);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// backward: grid = rows, block = 256.  smem: C + 2*A + 2*Ppad + 40 + 3*8*(A/8) floats
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned smem_addr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ unsigned mapa_shared(unsigned addr, unsigned rank) {
    unsigned r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void st_shared_cluster_f32(unsigned addr, float v) {
    asm volatile("st.shared::cluster.f32 [%0], %1;" :: "r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ void cluster_barrier() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

template <bool DEEP>     // DEEP (launches of at most two CTAs per SM: few rows, every row shared by two CTAs): 128 registers, twice the loads
                         // in flight in the two streaming phases — such a launch is bound by its chain of dependent load batches.
                         // Same operations in the same order as the 64-register instantiation: bit-identical (tested).
__global__ void __launch_bounds__(256, DEEP ? 2 : 4) att_step_bwd_bf16_kernel(
        int P, int C, int A, const int* __restrict__ img_index,
        const __nv_bfloat16* __restrict__ enc, const __nv_bfloat16* __restrict__ att_enc,
        const float* __restrict__ att_dec, long long ld_dec, const float* __restrict__ w_full,
        const float* __restrict__ alpha, long long ld_alpha,
        const float* __restrict__ d_alpha_ext, long long ld_dalpha,
        const float* __restrict__ gate, const float* __restrict__ awe_raw, const float* __restrict__ d_gated,
        float* __restrict__ d_att_dec, long long ld_ddec,
        float* __restrict__ d_fbeta_pre, long long ld_dfb,
        float* __restrict__ d_e, long long ld_de,
        __nv_bfloat16* __restrict__ dz16, long long ld_dz16, float* __restrict__ d_awe_out, int use_mma,
        int n_whole /* < 0: plain launch, one CTA per row; >= 0: launched as 2-CTA clusters, the first n_whole CTAs take whole rows */) {
    extern __shared__ __align__(16) float sm[];
    float* s_dawe = sm;                       // C
    float* s_dec = s_dawe + C;                // A
    float* s_alpha = s_dec + A;               // Ppad
    float* s_de = s_alpha + ((P + 3) & ~3);   // Ppad
    float* s_red = s_de + ((P + 3) & ~3);     // 40
    float* s_part = s_red + 40;               // 3 * A
    float* s_pb = s_part + 3 * A;             // nwarp * Pp16   (tensor-core path: per-warp partial d_alpha)
    __nv_bfloat16* s_hl = reinterpret_cast<__nv_bfloat16*>(s_pb + (blockDim.x >> 5) * (((P + 15) >> 4) << 4));   // 3 * C bf16
    float* s_xch = reinterpret_cast<float*>(s_hl + 3 * C);      // A floats (split rows: rank 1's d_att_dec partial lands here on rank 0)
    // Row balance.  This kernel's throughput per SM saturates at ~43 GB/s, its fair share of HBM, so a launch is as slow as its
    // busiest SM: 512 rows put 4 CTAs on 68 SMs and 3 on the other 80 and take 93.9 us where 592 rows take 98.2
    // (profiles/r02_att_rows_per_launch.txt).  When the row count is not a multiple of the SM count, the launcher therefore runs
    // the LAST few rows as TWO half-row CTAs each (a 2-CTA cluster: pixels [0, p_split) / [p_split, P) in the two streaming
    // phases; the softmax-backward dot product and the d_att_dec partial sums meet through distributed shared memory) so that
    // whole rows + half rows fill every SM's four CTA slots evenly in ONE wave.  (Splitting every row is slower: cluster barriers
    // and a second wave cost more than the balance gains — profiles/r02_experiments.md.)
    int r = blockIdx.x, hrank = 0;
    bool split = false;
    if (n_whole >= 0 && (int)blockIdx.x >= n_whole) {
        split = true;
        r = n_whole + (((int)blockIdx.x - n_whole) >> 1);
        hrank = ((int)blockIdx.x - n_whole) & 1;
    }
    const int p_split = min(P, (((P >> 1) + 8) >> 4) << 4);
    const int p_lo = (split && hrank) ? p_split : 0, p_hi = (split && !hrank) ? p_split : P;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    pdl_trigger();
    pdl_wait();
    const int img = img_index ? img_index[r] : r;

    // (A) gate backward (elementwise over C)
    {
        const long long o = (long long)r * C;
        for (int c = threadIdx.x * 4; c < C; c += blockDim.x * 4) {
            const float4 dg = *reinterpret_cast<const float4*>(d_gated + o + c);
            const float4 g = *reinterpret_cast<const float4*>(gate + o + c);
            const float4 aw = *reinterpret_cast<const float4*>(awe_raw + o + c);
            const float4 da = make_float4(dg.x * g.x, dg.y * g.y, dg.z * g.z, dg.w * g.w);
            *reinterpret_cast<float4*>(s_dawe + c) = da;                           // both CTAs of a split row need all of d_awe
            if (split && ((c * 2 >= C) ? 1 : 0) != hrank) continue;                // ... but each output element has one owner
            if (d_awe_out) *reinterpret_cast<float4*>(d_awe_out + o + c) = da;     // kept for the encoder gradient
            const float4 df = make_float4(dg.x * aw.x * g.x * (1.f - g.x), dg.y * aw.y * g.y * (1.f - g.y),
                                          dg.z * aw.z * g.z * (1.f - g.z), dg.w * aw.w * g.w * (1.f - g.w));
            *reinterpret_cast<float4*>(d_fbeta_pre + (long long)r * ld_dfb + c) = df;
            if (dz16) {
                uint2 pk = make_uint2(pack2(df.x, df.y), pack2(df.z, df.w));
                *reinterpret_cast<uint2*>(dz16 + (long long)r * ld_dz16 + A + c) = pk;
            }
        }
        const float* dec = att_dec + (long long)r * ld_dec;
        for (int a = threadIdx.x; a < A; a += blockDim.x) s_dec[a] = dec[a];
        const float* al = alpha + (long long)r * ld_alpha;
        for (int p = threadIdx.x; p < P; p += blockDim.x) s_alpha[p] = al[p];
    }
    __syncthreads();

    // (B) d_alpha[p] = <d_awe, enc[r,p,:]>
    if (use_mma) {
        // Tensor-core path.  d_awe (fp32) is split into three bf16 terms (24 mantissa bits: hi, mid, lo = columns n = 0, 1, 2
        // of the B operand), enc rows are the A operand: D[16 pixels x 8] += A[16 pixels x 16 ch] * B[16 ch x 8].
        // Warp w owns the channel strip [w*CW, (w+1)*CW) of every pixel row; lane (g = lane/4, t = lane%4) loads 16 B
        // (channels 8t..8t+7 of a 32-channel block) of rows g and g+8 of the pixel block: those two 128-bit loads are
        // the A fragments of two MMAs (k-slots 2t,2t+1 <-> channels 8t+0,1; 2t+8,2t+9 <-> 8t+2,3; second MMA: 8t+4..7).
        // ~5 instructions per KB of features instead of ~38 for the unpack + FMA loop.
        __nv_bfloat16* s_h0 = s_hl; __nv_bfloat16* s_h1 = s_hl + C; __nv_bfloat16* s_h2 = s_hl + 2 * C;
        for (int c = threadIdx.x; c < C; c += blockDim.x) {
            const float v = s_dawe[c];
            const __nv_bfloat16 h0 = __float2bfloat16_rn(v);
            const float r1 = v - __bfloat162float(h0);
            const __nv_bfloat16 h1 = __float2bfloat16_rn(r1);
            s_h0[c] = h0; s_h1[c] = h1; s_h2[c] = __float2bfloat16_rn(r1 - __bfloat162float(h1));
        }
        __syncthreads();
        const int g = lane >> 2, t = lane & 3;
        const int CW = C / nwarp, NB = CW >> 5;
        const int cb0 = warp * CW;
        const int Pp16 = ((P + 15) >> 4) << 4;
        const __nv_bfloat16* eb = enc + (long long)img * P * C + cb0 + 8 * t;
        const __nv_bfloat16* bsrc = (g < 3) ? (s_hl + g * C + cb0 + 8 * t) : s_hl;
        for (int pb = p_lo >> 4; pb < ((p_hi + 15) >> 4); ++pb) {
            const int p0 = pb * 16 + g, p1 = p0 + 8;
            const __nv_bfloat16* rowA = eb + (long long)min(p0, P - 1) * C;
            const __nv_bfloat16* rowB = eb + (long long)min(p1, P - 1) * C;
            float d0 = 0.f, d1 = 0.f, d2 = 0.f, d3 = 0.f;
            constexpr int UB = DEEP ? 8 : 4;
            for (int nb0 = 0; nb0 < NB; nb0 += UB) {
                uint4 xa[UB], xb[UB];
#pragma unroll
                for (int u = 0; u < UB; ++u) {
                    if (nb0 + u < NB) {                           // rows past P (last pixel block) are zero, not re-read
                        xa[u] = (p0 < P) ? ld_stream_u4(rowA + 32 * (nb0 + u)) : make_uint4(0u, 0u, 0u, 0u);
                        xb[u] = (p1 < P) ? ld_stream_u4(rowB + 32 * (nb0 + u)) : make_uint4(0u, 0u, 0u, 0u);
                    }
                }
#pragma unroll
                for (int u = 0; u < UB; ++u) {
                    if (nb0 + u < NB) {
                        uint4 bq = make_uint4(0u, 0u, 0u, 0u);
                        if (g < 3) bq = *reinterpret_cast<const uint4*>(bsrc + 32 * (nb0 + u));
                        mma_bf16_16816(d0, d1, d2, d3, xa[u].x, xb[u].x, xa[u].y, xb[u].y, bq.x, bq.y);
                        mma_bf16_16816(d0, d1, d2, d3, xa[u].z, xb[u].z, xa[u].w, xb[u].w, bq.z, bq.w);
                    }
                }
            }
            // D columns 0,1 (hi, mid) sit on the t == 0 lane of each quad, column 2 (lo) on the t == 1 lane
            float s0 = (t == 0) ? d0 + d1 : ((t == 1) ? d0 : 0.f);
            float s1 = (t == 0) ? d2 + d3 : ((t == 1) ? d2 : 0.f);
            s0 += __shfl_xor_sync(0xffffffffu, s0, 1); s1 += __shfl_xor_sync(0xffffffffu, s1, 1);
            if (t == 0) {
                if (p0 < P) s_pb[warp * Pp16 + p0] = s0;
                if (p1 < P) s_pb[warp * Pp16 + p1] = s1;
            }
        }
        __syncthreads();
        for (int p = p_lo + threadIdx.x; p < p_hi; p += blockDim.x) {
            float acc = 0.f;
            for (int w = 0; w < nwarp; ++w) acc += s_pb[w * Pp16 + p];
            if (d_alpha_ext) acc += d_alpha_ext[(long long)r * ld_dalpha + p];
            s_de[p] = acc;
        }
    } else {
        const __nv_bfloat16* eb = enc + (long long)img * P * C;
        const int C8 = C >> 3;
        for (int p = p_lo + warp; p < p_hi; p += nwarp) {
            const __nv_bfloat16* row = eb + (long long)p * C;
            float acc = 0.f;
            int j = lane;
            for (; j + 7 * 32 < C8; j += 8 * 32) {
                uint4 x[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) x[u] = ld_stream_u4(row + 8 * (j + u * 32));
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    float f[8];
                    unpack8(x[u], f);
                    const float4 d0 = *reinterpret_cast<const float4*>(s_dawe + 8 * (j + u * 32));
                    const float4 d1 = *reinterpret_cast<const float4*>(s_dawe + 8 * (j + u * 32) + 4);
                    acc = fmaf(f[0], d0.x, acc); acc = fmaf(f[1], d0.y, acc); acc = fmaf(f[2], d0.z, acc); acc = fmaf(f[3], d0.w, acc);
                    acc = fmaf(f[4], d1.x, acc); acc = fmaf(f[5], d1.y, acc); acc = fmaf(f[6], d1.z, acc); acc = fmaf(f[7], d1.w, acc);
                }
            }
            for (; j < C8; j += 32) {
                const uint4 x = ld_stream_u4(row + 8 * j);
                float f[8];
                unpack8(x, f);
                const float4 d0 = *reinterpret_cast<const float4*>(s_dawe + 8 * j);
                const float4 d1 = *reinterpret_cast<const float4*>(s_dawe + 8 * j + 4);
                acc = fmaf(f[0], d0.x, acc); acc = fmaf(f[1], d0.y, acc); acc = fmaf(f[2], d0.z, acc); acc = fmaf(f[3], d0.w, acc);
                acc = fmaf(f[4], d1.x, acc); acc = fmaf(f[5], d1.y, acc); acc = fmaf(f[6], d1.z, acc); acc = fmaf(f[7], d1.w, acc);
            }
            acc = warp_sum(acc);
            if (lane == 0) {
                if (d_alpha_ext) acc += d_alpha_ext[(long long)r * ld_dalpha + p];
                s_de[p] = acc;
            }
        }
    }
    __syncthreads();

    // (C) softmax backward, centred
    {
        float part = 0.f;
        for (int p = p_lo + threadIdx.x; p < p_hi; p += blockDim.x) part = fmaf(s_alpha[p], s_de[p], part);
        float dot = block_sum(part, s_red);
        if (split) {                                  // the other half's share of sum_p alpha_p d_alpha_p, through its shared memory
            if (threadIdx.x == 0) {
                s_red[34 + hrank] = dot;
                st_shared_cluster_f32(mapa_shared(smem_addr(s_red + 34 + hrank), (unsigned)(hrank ^ 1)), dot);
            }
            cluster_barrier();
            dot = s_red[34] + s_red[35];              // rank 0's share first on both sides: identical, deterministic
        }
        float* out = d_e + (long long)r * ld_de;
        for (int p = p_lo + threadIdx.x; p < p_hi; p += blockDim.x) {
            const float v = s_alpha[p] * (s_de[p] - dot);
            s_de[p] = v;
            out[p] = v;
        }
    }
    __syncthreads();

    // (D) d_att_dec[a] = w_full[a] * sum_p d_e[p] * [att_enc[p,a] + att_dec[a] > 0]
    //     thread = (pixel group g of 4, 8-channel column j); loops over column chunks of 64 * 8 channels
    {
        const __nv_bfloat16* ab = att_enc + (long long)img * P * A;
        const int A8 = A >> 3;
        const int grp = threadIdx.x >> 6, t = threadIdx.x & 63;
        for (int j0 = 0; j0 < A8; j0 += 64) {
            const int j = j0 + t;
            float acc[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[i] = 0.f;
            if (j < A8) {
                const float4 d0 = *reinterpret_cast<const float4*>(s_dec + 8 * j);
                const float4 d1 = *reinterpret_cast<const float4*>(s_dec + 8 * j + 4);
                const float dd[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
                int p = p_lo + grp;
                constexpr int UD = DEEP ? 13 : 7;                 // (a half row = 24-25 pixels per group: two batches of <= 13)
                for (; DEEP ? (p < p_hi) : (p + (UD - 1) * 4 < p_hi); p += UD * 4) {
                    uint4 x[UD];
#pragma unroll
                    for (int u = 0; u < UD; ++u)
                        if (!DEEP || p + 4 * u < p_hi) x[u] = ld_stream_u4(ab + (long long)(p + 4 * u) * A + 8 * j);
#pragma unroll
                    for (int u = 0; u < UD; ++u) {
                        if (!DEEP || p + 4 * u < p_hi) {
                            const float de = s_de[p + 4 * u];
                            float f[8];
                            unpack8(x[u], f);
#pragma unroll
                            for (int i = 0; i < 8; ++i) acc[i] += (f[i] + dd[i] > 0.f) ? de : 0.f;
                        }
                    }
                }
                for (; p < p_hi; p += 4) {
                    const uint4 x = ld_stream_u4(ab + (long long)p * A + 8 * j);
                    const float de = s_de[p];
                    float f[8];
                    unpack8(x, f);
#pragma unroll
                    for (int i = 0; i < 8; ++i) acc[i] += (f[i] + dd[i] > 0.f) ? de : 0.f;
                }
            }
            if (grp > 0 && j < A8) {
                float* dst = s_part + (size_t)(grp - 1) * A + 8 * j;
                *reinterpret_cast<float4*>(dst) = make_float4(acc[0], acc[1], acc[2], acc[3]);
                *reinterpret_cast<float4*>(dst + 4) = make_float4(acc[4], acc[5], acc[6], acc[7]);
            }
            __syncthreads();
            if (split) {
                // rank 1 hands the sum over ITS pixels to rank 0 (its own exchange buffer), which finishes the row
                if (hrank == 1 && grp == 0 && j < A8) {
                    const unsigned dst = mapa_shared(smem_addr(s_xch + 8 * j), 0u);
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        st_shared_cluster_f32(dst + 4 * i, acc[i] + s_part[8 * j + i] + s_part[A + 8 * j + i] + s_part[2 * A + 8 * j + i]);
                }
                cluster_barrier();
                if (hrank == 1) continue;
            }
            if (grp == 0 && j < A8) {
                float res[8];
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    res[i] = (acc[i] + s_part[8 * j + i] + s_part[A + 8 * j + i] + s_part[2 * A + 8 * j + i] +
                              (split ? s_xch[8 * j + i] : 0.f)) * w_full[8 * j + i];
                float* o = d_att_dec + (long long)r * ld_ddec + 8 * j;
                *reinterpret_cast<float4*>(o) = make_float4(res[0], res[1], res[2], res[3]);
                *reinterpret_cast<float4*>(o + 4) = make_float4(res[4], res[5], res[6], res[7]);
                if (dz16) {
                    uint4 pk = make_uint4(pack2(res[0], res[1]), pack2(res[2], res[3]), pack2(res[4], res[5]), pack2(res[6], res[7]));
                    *reinterpret_cast<uint4*>(dz16 + (long long)r * ld_dz16 + 8 * j) = pk;
                }
            }
            __syncthreads();
        }
    }
}

// ------------------------------------------------------------------------------------------------
// after the loop: d_att_enc + full_att / enc_att-bias parameter gradients, att_enc stored as bf16.
//   d_att_enc[b,p,a] = w_full[a] * sum_t d_e[b,t,p] * [att_enc[b,p,a] + att_dec[t,b,a] > 0]
// grid = (ceil(P/PROJ_PB), B), block = 2 x A/4 threads (each 4 consecutive a; the halves alternate over groups of 4 pixels), 4 pixels per pass so that one 128-bit
// shared-memory read of att_dec[t, a..a+3] feeds 16 updates.  smem: T*A (att_dec) + T*PROJ_PB (d_e).
// Outputs: d_att_enc fp32 and / or bf16 (either may be NULL: the bf16 tier only needs the bf16 copy, which is the
// MN-major A operand of the enc_att weight-gradient contraction) and per-CTA partials
//   partial[(b*gridDim.x + chunk)*(2A+4)] = { d_w_full[A], colsum_p d_att_enc[A] (-> d enc_att.bias), sum d_e, 0,0,0 }.
// ------------------------------------------------------------------------------------------------
constexpr int PROJ_PB = 28;
constexpr float PROJ_W_MIN = 1e-18f;       // below this |w_full[a]| the split form of d_w_full is not used (see the kernel)

// out[blockIdx.y][n] = sum over the rows of chunk blockIdx.y of X[m*ldx + n] * Y[m*ldy + n]   (deterministic; block (32,32) like
// colsum_kernel; the chunks are added by a colsum pass afterwards)
constexpr int COLDOT_CHUNKS = 48;
__global__ void coldot_kernel(const float* __restrict__ X, long long ldx, const float* __restrict__ Y, long long ldy,
                              long long M_all, int N, float* __restrict__ out_all) {
    pdl_trigger();
    pdl_wait();
    __shared__ float s[32][33];
    const int n = blockIdx.x * 32 + threadIdx.x;
    const long long per = (M_all + gridDim.y - 1) / gridDim.y, m_lo = per * blockIdx.y;
    const long long M = min(M_all, m_lo + per);
    float* out = out_all + (long long)blockIdx.y * N;
    float acc = 0.f;
    if (n < N) {
        long long m = m_lo + threadIdx.y;
        for (; m + 96 < M; m += 128) {                       // four rows in flight per thread
            const float x0 = X[m * ldx + n], x1 = X[(m + 32) * ldx + n], x2 = X[(m + 64) * ldx + n], x3 = X[(m + 96) * ldx + n];
            const float y0 = Y[m * ldy + n], y1 = Y[(m + 32) * ldy + n], y2 = Y[(m + 64) * ldy + n], y3 = Y[(m + 96) * ldy + n];
            acc = fmaf(x0, y0, acc); acc = fmaf(x1, y1, acc); acc = fmaf(x2, y2, acc); acc = fmaf(x3, y3, acc);
        }
        for (; m < M; m += 32) acc = fmaf(X[m * ldx + n], Y[m * ldy + n], acc);
    }
    s[threadIdx.y][threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.y == 0 && n < N) {
        float t = 0.f;
#pragma unroll
        for (int y = 0; y < 32; ++y) t += s[y][threadIdx.x];
        out[n] = t;
    }
}
// d_w_full[a] += t2[a] / w_full[a], t2[a] = sum_{t,b} att_dec[t,b,a] * d_att_dec[t,b,a]: since d_att_dec = w_full * sum_p mask * d_e,
// this is the part of  sum d_e * relu(att_enc + att_dec)  that multiplies att_dec.  Skipped when the projection kernel did not
// split (same predicate).  One CTA.
__global__ void proj_wfull_finish_kernel(int A, const float* __restrict__ w_full, const float* __restrict__ t2,
                                         float* __restrict__ d_w_full) {
    pdl_trigger();
    pdl_wait();
    int bad = 0;
    for (int a4 = threadIdx.x * 4; a4 < A; a4 += blockDim.x * 4) {
        const float4 w = *reinterpret_cast<const float4*>(w_full + a4);
        bad |= (fabsf(w.x) < PROJ_W_MIN) | (fabsf(w.y) < PROJ_W_MIN) | (fabsf(w.z) < PROJ_W_MIN) | (fabsf(w.w) < PROJ_W_MIN);
    }
    if (__syncthreads_or(bad)) return;
    for (int a = threadIdx.x; a < A; a += blockDim.x) d_w_full[a] += t2[a] / w_full[a];
}

// 1.0f where a > b, else 0.0f, as ONE instruction (FSET.BF): with the FFMA that consumes it the masked accumulation
// `acc += (a > b) ? v : 0` is two instructions, one per pipe (ALU + FMA) — FSETP + FSEL + FADD puts two of three on the
// half-rate ALU pipe.  fma(1, v, acc) and fma(0, v, acc) round exactly like acc + v and acc (v finite).
__device__ __forceinline__ float gt_mask(float a, float b) {
    float m;
    asm("set.gt.f32.f32 %0, %1, %2;" : "=f"(m) : "f"(a), "f"(b));
    return m;
}

__device__ __forceinline__ void att_proj_bwd_bf16_body(int B, int T, int P, int A, const int* __restrict__ row_len,
                                         const __nv_bfloat16* __restrict__ att_enc,
                                         const float* __restrict__ att_dec_all, long long ld_dec,
                                         const float* __restrict__ w_full, const float* __restrict__ d_e,
                                         float* __restrict__ d_att_enc, __nv_bfloat16* __restrict__ d_att_enc16,
                                         float* __restrict__ partial, int split_wfull) {
    pdl_trigger();
    pdl_wait();
    extern __shared__ __align__(16) float sm[];
    const int b = blockIdx.y, p0 = blockIdx.x * PROJ_PB;
    const int np = min(PROJ_PB, P - p0);
    const int Tb = row_len[b];
    float* s_dec = sm;
    float* s_de = sm + (size_t)T * A;
    float* s_red = s_de + (size_t)T * PROJ_PB;
    // split_wfull (see proj_wfull_finish_kernel): the inner loop only forms the masked sums S = sum_t [att_enc + att_dec_t > 0] d_e_t
    // — with the NEGATED att_dec staged in shared memory that is one compare and one predicated add per (pixel, channel, step)
    // instead of add / compare / add / max / fma — and d_w_full = sum att_enc * S here + (sum_t att_dec_t * d_att_dec_t) / w
    // later.  Needs every |w_full[a]| to be a sane divisor: the predicate is evaluated identically here and in the finish kernel.
    bool fast = false;
    if (split_wfull) {
        int bad = 0;
        for (int a4 = threadIdx.x * 4; a4 < A; a4 += blockDim.x * 4) {
            const float4 w = *reinterpret_cast<const float4*>(w_full + a4);
            bad |= (fabsf(w.x) < PROJ_W_MIN) | (fabsf(w.y) < PROJ_W_MIN) | (fabsf(w.z) < PROJ_W_MIN) | (fabsf(w.w) < PROJ_W_MIN);
        }
        fast = __syncthreads_or(bad) == 0;
    }
    const float sgn = fast ? -1.f : 1.f;
    for (int i = threadIdx.x; i < Tb * (A >> 2); i += blockDim.x) {
        const int t = i / (A >> 2), a4 = (i % (A >> 2)) * 4;
        const float4 v = *reinterpret_cast<const float4*>(att_dec_all + ((long long)t * B + b) * ld_dec + a4);
        *reinterpret_cast<float4*>(s_dec + (size_t)t * A + a4) = make_float4(sgn * v.x, sgn * v.y, sgn * v.z, sgn * v.w);
    }
    float de_sum = 0.f;
    for (int i = threadIdx.x; i < Tb * PROJ_PB; i += blockDim.x) {
        const int t = i / PROJ_PB, pp = i % PROJ_PB;
        const float v = (pp < np) ? d_e[((long long)b * T + t) * P + p0 + pp] : 0.f;
        s_de[i] = v;
        de_sum += v;
    }
    __syncthreads();
    // two thread halves share the staged att_dec / d_e and take alternate groups of 4 pixels (twice the warps per byte of
    // shared memory: the loop is latency-bound at 4 warps per scheduler)
    const int th = blockDim.x >> 1, half = threadIdx.x / th;
    const int a = (threadIdx.x - half * th) * 4;
    float4 wacc = make_float4(0.f, 0.f, 0.f, 0.f), bacc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (a < A) {
        const float4 w = *reinterpret_cast<const float4*>(w_full + a);
        for (int pq = half * 4; pq < np; pq += 8) {                   // PROJ_PB is a multiple of 4; rows >= np carry d_e = 0
            float x[4][4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int pp = min(pq + u, np - 1);
                const uint2 raw = ld_stream_u2(att_enc + ((long long)b * P + p0 + pp) * A + a);
                x[u][0] = __uint_as_float(raw.x << 16); x[u][1] = __uint_as_float(raw.x & 0xffff0000u);
                x[u][2] = __uint_as_float(raw.y << 16); x[u][3] = __uint_as_float(raw.y & 0xffff0000u);
            }
            float acc[4][4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int i = 0; i < 4; ++i) acc[u][i] = 0.f;
            if (fast) {
                for (int t = 0; t < Tb; ++t) {
                    const float4 de4 = *reinterpret_cast<const float4*>(s_de + t * PROJ_PB + pq);
                    const float4 d = *reinterpret_cast<const float4*>(s_dec + (size_t)t * A + a);     // -att_dec[t]
                    const float de[4] = {de4.x, de4.y, de4.z, de4.w};
                    const float nd[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
                    for (int u = 0; u < 4; ++u)
#pragma unroll
                        for (int i = 0; i < 4; ++i)
                            acc[u][i] = fmaf(gt_mask(x[u][i], nd[i]), de[u], acc[u][i]);   // x + att_dec > 0  <=>  x > -att_dec (exactly, in fp32)
                }
                float wl[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int u = 0; u < 4; ++u)
#pragma unroll
                    for (int i = 0; i < 4; ++i) wl[i] = fmaf(x[u][i], acc[u][i], wl[i]);    // rows past np carry S = 0
                wacc.x += wl[0]; wacc.y += wl[1]; wacc.z += wl[2]; wacc.w += wl[3];
            } else
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
                if (d_att_enc) *reinterpret_cast<float4*>(d_att_enc + o) = r;
                if (d_att_enc16) *reinterpret_cast<uint2*>(d_att_enc16 + o) = make_uint2(pack2(r.x, r.y), pack2(r.z, r.w));
            }
        }
    }
    float* mine = partial + ((long long)b * gridDim.x + blockIdx.x) * (2 * A + 4);
    __syncthreads();                                                  // everyone is done with s_dec: reuse it to add the halves
    if (half == 1 && a < A) { *reinterpret_cast<float4*>(s_dec + a) = wacc; *reinterpret_cast<float4*>(s_dec + A + a) = bacc; }
    __syncthreads();
    if (half == 0 && a < A) {
        const float4 w1 = *reinterpret_cast<const float4*>(s_dec + a), b1 = *reinterpret_cast<const float4*>(s_dec + A + a);
        *reinterpret_cast<float4*>(mine + a) = make_float4(wacc.x + w1.x, wacc.y + w1.y, wacc.z + w1.z, wacc.w + w1.w);
        *reinterpret_cast<float4*>(mine + A + a) = make_float4(bacc.x + b1.x, bacc.y + b1.y, bacc.z + b1.z, bacc.w + b1.w);
    }
    const float tot = block_sum(de_sum, s_red);
    if (threadIdx.x == 0) { mine[2 * A] = tot; mine[2 * A + 1] = 0.f; mine[2 * A + 2] = 0.f; mine[2 * A + 3] = 0.f; }
}
__global__ void att_proj_bwd_bf16_kernel(int B, int T, int P, int A, const int* __restrict__ row_len,
                                         const __nv_bfloat16* __restrict__ att_enc,
                                         const float* __restrict__ att_dec_all, long long ld_dec,
                                         const float* __restrict__ w_full, const float* __restrict__ d_e,
                                         float* __restrict__ d_att_enc, __nv_bfloat16* __restrict__ d_att_enc16,
                                         float* __restrict__ partial, int split_wfull) {
    att_proj_bwd_bf16_body(B, T, P, A, row_len, att_enc, att_dec_all, ld_dec, w_full, d_e, d_att_enc, d_att_enc16, partial, split_wfull);
}
// blocks of more than 512 threads (two halves of A/4 > 256 threads, up to A = 2048): the kernel above uses more than 64 registers, so
// 1024 threads would not fit the 64K registers of an SM; this instantiation caps them at 64
__global__ void __launch_bounds__(1024) att_proj_bwd_bf16_kernel_wide(int B, int T, int P, int A, const int* __restrict__ row_len,
                                         const __nv_bfloat16* __restrict__ att_enc,
                                         const float* __restrict__ att_dec_all, long long ld_dec,
                                         const float* __restrict__ w_full, const float* __restrict__ d_e,
                                         float* __restrict__ d_att_enc, __nv_bfloat16* __restrict__ d_att_enc16,
                                         float* __restrict__ partial, int split_wfull) {
    att_proj_bwd_bf16_body(B, T, P, A, row_len, att_enc, att_dec_all, ld_dec, w_full, d_e, d_att_enc, d_att_enc16, partial, split_wfull);
}

// Captions that share images: the same pass per IMAGE i over the (row, step) pairs of its rows (rows in CSR order, then steps):
//   d_att_enc[i,p,a] = w_full[a] * sum_{r in rows(i)} sum_{t < len_r} d_e[r,t,p] * [att_enc[i,p,a] + att_dec[t,r,a] > 0]
// grid = (ceil(P/PROJ_IMG16_PB), n_img), block = 2 x A/4 threads: each half owns 4 of the CTA's 8 pixels, a thread 4 channels,
// and the 16 masked sums stay in registers while the pairs pass through shared memory PROJ_IMG16_KC steps of one row at a
// time — no per-row (B,P,A) tensor, a fixed summation order.  The split form of d_w_full and its fallback are those above.
// ------------------------------------------------------------------------------------------------
constexpr int PROJ_IMG16_PB = 8, PROJ_IMG16_KC = 32;
__global__ void __launch_bounds__(1024) att_proj_bwd_img_bf16_kernel(int B, int T, int P, int A, const int* __restrict__ row_len,
                                         const int* __restrict__ row_ptr, const int* __restrict__ rows,
                                         const __nv_bfloat16* __restrict__ att_enc,
                                         const float* __restrict__ att_dec_all, long long ld_dec,
                                         const float* __restrict__ w_full, const float* __restrict__ d_e,
                                         __nv_bfloat16* __restrict__ d_att_enc16, float* __restrict__ partial, int split_wfull) {
    pdl_trigger();
    pdl_wait();
    extern __shared__ __align__(16) float sm[];
    const int i = blockIdx.y, p0 = blockIdx.x * PROJ_IMG16_PB;
    const int np = min(PROJ_IMG16_PB, P - p0);
    float* s_dec = sm;                                        // PROJ_IMG16_KC * A
    float* s_de = sm + (size_t)PROJ_IMG16_KC * A;             // PROJ_IMG16_KC * PROJ_IMG16_PB
    float* s_red = s_de + PROJ_IMG16_KC * PROJ_IMG16_PB;      // 40
    bool fast = false;
    if (split_wfull) {
        int bad = 0;
        for (int a4 = threadIdx.x * 4; a4 < A; a4 += blockDim.x * 4) {
            const float4 w = *reinterpret_cast<const float4*>(w_full + a4);
            bad |= (fabsf(w.x) < PROJ_W_MIN) | (fabsf(w.y) < PROJ_W_MIN) | (fabsf(w.z) < PROJ_W_MIN) | (fabsf(w.w) < PROJ_W_MIN);
        }
        fast = __syncthreads_or(bad) == 0;
    }
    const float sgn = fast ? -1.f : 1.f;
    const int th = blockDim.x >> 1, half = threadIdx.x / th;
    const int a = (threadIdx.x - half * th) * 4, pq = half * 4;
    float x[4][4], acc[4][4];
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int c = 0; c < 4; ++c) { x[u][c] = 0.f; acc[u][c] = 0.f; }
    if (a < A) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const uint2 raw = ld_stream_u2(att_enc + ((long long)i * P + p0 + min(pq + u, np - 1)) * A + a);
            x[u][0] = __uint_as_float(raw.x << 16); x[u][1] = __uint_as_float(raw.x & 0xffff0000u);
            x[u][2] = __uint_as_float(raw.y << 16); x[u][3] = __uint_as_float(raw.y & 0xffff0000u);
        }
    }
    float4 wacc = make_float4(0.f, 0.f, 0.f, 0.f);
    float de_sum = 0.f;
    for (int k = row_ptr[i]; k < row_ptr[i + 1]; ++k) {
        const int b = rows[k], Tb = row_len[b];
        for (int t0 = 0; t0 < Tb; t0 += PROJ_IMG16_KC) {
            const int nt = min(PROJ_IMG16_KC, Tb - t0);
            __syncthreads();                                  // the previous round is consumed
            for (int j = threadIdx.x; j < nt * (A >> 2); j += blockDim.x) {
                const int t = j / (A >> 2), a4 = (j % (A >> 2)) * 4;
                const float4 v = *reinterpret_cast<const float4*>(att_dec_all + ((long long)(t0 + t) * B + b) * ld_dec + a4);
                *reinterpret_cast<float4*>(s_dec + (size_t)t * A + a4) = make_float4(sgn * v.x, sgn * v.y, sgn * v.z, sgn * v.w);
            }
            for (int j = threadIdx.x; j < nt * PROJ_IMG16_PB; j += blockDim.x) {
                const int t = j / PROJ_IMG16_PB, pp = j % PROJ_IMG16_PB;
                const float v = (pp < np) ? d_e[((long long)b * T + t0 + t) * P + p0 + pp] : 0.f;
                s_de[j] = v;
                de_sum += v;
            }
            __syncthreads();
            if (a >= A) continue;
            if (fast) {
                for (int t = 0; t < nt; ++t) {
                    const float4 de4 = *reinterpret_cast<const float4*>(s_de + t * PROJ_IMG16_PB + pq);
                    const float4 d = *reinterpret_cast<const float4*>(s_dec + (size_t)t * A + a);     // -att_dec[t]
                    const float de[4] = {de4.x, de4.y, de4.z, de4.w};
                    const float nd[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
                    for (int u = 0; u < 4; ++u)
#pragma unroll
                        for (int c = 0; c < 4; ++c) acc[u][c] = fmaf(gt_mask(x[u][c], nd[c]), de[u], acc[u][c]);
                }
            } else {
                for (int t = 0; t < nt; ++t) {
                    const float4 de4 = *reinterpret_cast<const float4*>(s_de + t * PROJ_IMG16_PB + pq);
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
        if (fast) {
            float wl[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int c = 0; c < 4; ++c) wl[c] = fmaf(x[u][c], acc[u][c], wl[c]);    // pixels past np carry S = 0
            wacc = make_float4(wl[0], wl[1], wl[2], wl[3]);
        }
        const float4 w = *reinterpret_cast<const float4*>(w_full + a);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (pq + u >= np) break;
            const long long o = ((long long)i * P + p0 + pq + u) * A + a;
            const float4 r = make_float4(acc[u][0] * w.x, acc[u][1] * w.y, acc[u][2] * w.z, acc[u][3] * w.w);
            bacc.x += r.x; bacc.y += r.y; bacc.z += r.z; bacc.w += r.w;
            *reinterpret_cast<uint2*>(d_att_enc16 + o) = make_uint2(pack2(r.x, r.y), pack2(r.z, r.w));
        }
    }
    float* mine = partial + ((long long)i * gridDim.x + blockIdx.x) * (2 * A + 4);
    __syncthreads();                                          // everyone is done with s_dec: reuse it to add the halves
    if (half == 1 && a < A) { *reinterpret_cast<float4*>(s_dec + a) = wacc; *reinterpret_cast<float4*>(s_dec + A + a) = bacc; }
    __syncthreads();
    if (half == 0 && a < A) {
        const float4 w1 = *reinterpret_cast<const float4*>(s_dec + a), b1 = *reinterpret_cast<const float4*>(s_dec + A + a);
        *reinterpret_cast<float4*>(mine + a) = make_float4(wacc.x + w1.x, wacc.y + w1.y, wacc.z + w1.z, wacc.w + w1.w);
        *reinterpret_cast<float4*>(mine + A + a) = make_float4(bacc.x + b1.x, bacc.y + b1.y, bacc.z + b1.z, bacc.w + b1.w);
    }
    const float tot = block_sum(de_sum, s_red);
    if (threadIdx.x == 0) { mine[2 * A] = tot; mine[2 * A + 1] = 0.f; mine[2 * A + 2] = 0.f; mine[2 * A + 3] = 0.f; }
}

// ------------------------------------------------------------------------------------------------
// fp32 features -> bf16 features + pixel mean in ONE pass over encoder_out (models/attention.py:161 mean(dim=1)).
// grid = (ceil(C/256), B), block = 256 = 4 pixel groups x 64 float4 lanes.
// ------------------------------------------------------------------------------------------------
// row_ptr != NULL (captions that share images): CTA row b is image b, its mean goes to rows[row_ptr[b] .. row_ptr[b+1]).
__device__ __forceinline__ void mean_rows(int b, const int* row_ptr, int& k0, int& k1) {
    k0 = row_ptr ? row_ptr[b] : b;
    k1 = row_ptr ? row_ptr[b + 1] : b + 1;
}
__global__ void __launch_bounds__(256) convert_features_kernel(int P, int C, const float* __restrict__ enc,
                                                               __nv_bfloat16* __restrict__ enc16,
                                                               float* __restrict__ mean, __nv_bfloat16* __restrict__ mean16,
                                                               const int* __restrict__ row_ptr, const int* __restrict__ rows) {
    pdl_trigger();
    pdl_wait();
    __shared__ float4 s_part[3 * 64];
    const int b = blockIdx.y;
    const int lane = threadIdx.x & 63, grp = threadIdx.x >> 6;
    const int c = blockIdx.x * 256 + lane * 4;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c < C) {
        const float* base = enc + (long long)b * P * C + c;
        __nv_bfloat16* ob = enc16 + (long long)b * P * C + c;
        int p = grp;
        for (; p + 6 * 4 < P; p += 7 * 4) {
            float4 x[7];
#pragma unroll
            for (int u = 0; u < 7; ++u) x[u] = ld_stream_f4(base + (long long)(p + 4 * u) * C);
#pragma unroll
            for (int u = 0; u < 7; ++u) {
                acc.x += x[u].x; acc.y += x[u].y; acc.z += x[u].z; acc.w += x[u].w;
                *reinterpret_cast<uint2*>(ob + (long long)(p + 4 * u) * C) = make_uint2(pack2(x[u].x, x[u].y), pack2(x[u].z, x[u].w));
            }
        }
        for (; p < P; p += 4) {
            const float4 x = ld_stream_f4(base + (long long)p * C);
            acc.x += x.x; acc.y += x.y; acc.z += x.z; acc.w += x.w;
            *reinterpret_cast<uint2*>(ob + (long long)p * C) = make_uint2(pack2(x.x, x.y), pack2(x.z, x.w));
        }
    }
    if (grp > 0) s_part[(grp - 1) * 64 + lane] = acc;
    __syncthreads();
    if (grp == 0 && c < C) {
#pragma unroll
        for (int g = 0; g < 3; ++g) { const float4 o = s_part[g * 64 + lane]; acc.x += o.x; acc.y += o.y; acc.z += o.z; acc.w += o.w; }
        const float inv = (float)P;
        acc.x /= inv; acc.y /= inv; acc.z /= inv; acc.w /= inv;
        int k0, k1;
        mean_rows(b, row_ptr, k0, k1);
        for (int k = k0; k < k1; ++k) {
            const long long o = (long long)(row_ptr ? rows[k] : b) * C + c;
            if (mean) *reinterpret_cast<float4*>(mean + o) = acc;
            if (mean16) *reinterpret_cast<uint2*>(mean16 + o) = make_uint2(pack2(acc.x, acc.y), pack2(acc.z, acc.w));
        }
    }
}

struct BtPack { int v[ICD_MAX_STEPS]; };
__global__ void row_len_from_pack_kernel16(int B, int T, const BtPack bt, int* __restrict__ row_len) {
    pdl_trigger();
    pdl_wait();
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    int n = 0;
    for (int t = 0; t < T; ++t) n += (b < bt.v[t]) ? 1 : 0;
    row_len[b] = n;
}

// pixel mean of bf16-stored features (models/attention.py:161) when the caller hands the features over in bf16.
// grid = (ceil(C/512), B), block = 256 = 4 pixel groups x 64 lanes of 8 channels (16 B).
__global__ void __launch_bounds__(256) feature_mean_bf16_kernel(int P, int C, const __nv_bfloat16* __restrict__ enc16,
                                                                float* __restrict__ mean, __nv_bfloat16* __restrict__ mean16,
                                                                const int* __restrict__ row_ptr, const int* __restrict__ rows) {
    pdl_trigger();
    pdl_wait();
    __shared__ float s_part[3 * 64 * 8];
    const int b = blockIdx.y;
    const int lane = threadIdx.x & 63, grp = threadIdx.x >> 6;
    const int c = blockIdx.x * 512 + lane * 8;
    float acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.f;
    if (c < C) {
        const __nv_bfloat16* base = enc16 + (long long)b * P * C + c;
        int p = grp;
        for (; p + 6 * 4 < P; p += 7 * 4) {
            uint4 x[7];
#pragma unroll
            for (int u = 0; u < 7; ++u) x[u] = ld_stream_u4(base + (long long)(p + 4 * u) * C);
#pragma unroll
            for (int u = 0; u < 7; ++u) {
                float f[8];
                unpack8(x[u], f);
#pragma unroll
                for (int i = 0; i < 8; ++i) acc[i] += f[i];
            }
        }
        for (; p < P; p += 4) {
            const uint4 x = ld_stream_u4(base + (long long)p * C);
            float f[8];
            unpack8(x, f);
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[i] += f[i];
        }
    }
    if (grp > 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) s_part[((grp - 1) * 64 + lane) * 8 + i] = acc[i];
    }
    __syncthreads();
    if (grp == 0 && c < C) {
        const float inv = (float)P;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            acc[i] += s_part[(0 * 64 + lane) * 8 + i] + s_part[(1 * 64 + lane) * 8 + i] + s_part[(2 * 64 + lane) * 8 + i];
            acc[i] /= inv;
        }
        int k0, k1;
        mean_rows(b, row_ptr, k0, k1);
        for (int k = k0; k < k1; ++k) {
            const long long o = (long long)(row_ptr ? rows[k] : b) * C + c;
            if (mean) {
                *reinterpret_cast<float4*>(mean + o) = make_float4(acc[0], acc[1], acc[2], acc[3]);
                *reinterpret_cast<float4*>(mean + o + 4) = make_float4(acc[4], acc[5], acc[6], acc[7]);
            }
            if (mean16)
                *reinterpret_cast<uint4*>(mean16 + o) = make_uint4(pack2(acc[0], acc[1]), pack2(acc[2], acc[3]),
                                                                   pack2(acc[4], acc[5]), pack2(acc[6], acc[7]));
        }
    }
}

}  // namespace

// ---- launch forms (pure host logic, also exported for the CPU tests: icd_attention_step_launch_plan_bf16) ---------------
struct AttLaunchPlan {
    int per_row;        // CTAs per row of the rows that are shared (1: none are)
    int shared_rows;    // rows that run shared (forward: 0 or all; backward: the last n_split rows)
    int grid;           // CTAs of the launch
    int deep;           // 1: the 128-register instantiation (at most two CTAs per SM)
};

// forward: few rows per launch (ragged batches late in the caption, small batches) -> 2 or 4 CTAs per row (channel split, bit-identical
// results) so that the launch still fills the CTA slots of the GPU.  ICD_ATT_FWD_SPLIT = 1 | 2 | 4 forces a variant (tests, tools).
static AttLaunchPlan att_fwd16_plan(int rows, size_t smem) {
    const char* fsplit_e = getenv("ICD_ATT_FWD_SPLIT");
    const int split_env = fsplit_e ? atoi(fsplit_e) : 0;
    int nsplit = split_env == 1 || split_env == 2 || split_env == 4 ? split_env
                 : (rows <= ICD_ATT_FWD_SPLIT4_ROWS ? 4 : rows <= ICD_ATT_FWD_SPLIT2_ROWS ? 2 : 1);
    if (smem > 48 * 1024) nsplit = 1;          // (only the whole-row kernel is configured for large shared memory)
    AttLaunchPlan pl;
    pl.per_row = nsplit;
    pl.shared_rows = nsplit > 1 ? rows : 0;
    pl.grid = rows * nsplit;
    pl.deep = (nsplit > 1 && rows * nsplit <= 2 * ICD_NUM_SMS) ? 1 : 0;
    return pl;
}

static AttLaunchPlan att_bwd16_plan(int rows, int P, size_t smem) {
    // row balance (see the kernel): with up to 4 CTAs on each of the 148 SMs, a launch of `rows` CTAs whose last wave is partly
    // filled runs its last n_split rows as two half-row CTAs each, so that every SM gets the same number of CTAs: rows + n_split = a
    // multiple of the SM count.  Only when the rows are not already balanced and the split part stays a minority.
    const char* split_e = getenv("ICD_ATT_BWD_SPLIT");     // 0: never, 2: every row (tests), else: the balance rule
    const bool split_env = !split_e || split_e[0] != '0';
    int n_split = 0;
    // few rows per launch (ragged batches late in the caption, small batches): EVERY row as two half-row CTAs, twice the CTAs
    // streaming.  ICD_ATT_BWD_SPLIT_ROWS overrides the row count at or below which that happens (tools/att_bench.py fits it).
    const char* few_e = getenv("ICD_ATT_BWD_SPLIT_ROWS");
    const int few_rows = few_e ? atoi(few_e) : ICD_ATT_BWD_SPLIT_ALL_ROWS;
    if (split_e && split_e[0] == '2' && P >= 32) n_split = rows;
    else if (split_env && P >= 32 && rows <= few_rows) n_split = rows;
    else if (split_env && P >= 32) {
        const int rem = rows % ICD_NUM_SMS;                 // rows beyond an equal number per SM
        if (rem) n_split = ICD_NUM_SMS - rem;               // e.g. 512 rows: 80 split rows -> 432 + 160 CTAs = 4 per SM
        // the split part must stay a minority; where it would not, the minimal form: only the `rem` rows beyond an equal number L per SM
        // run as halves (2 rem <= 148 half-row CTAs), so that no SM carries more than L + 1/2 rows instead of L + 1 (320 rows: 69 -> 60 us)
        if (n_split > rows / 4) n_split = (rem <= ICD_NUM_SMS / 2 && rows > ICD_NUM_SMS) ? rem : 0;
        if ((rows - n_split) & 1) n_split += (n_split < rows) ? 1 : -1;          // the whole rows must pair up (2-CTA clusters)
        if (n_split < 0 || n_split > rows) n_split = 0;
    }
    AttLaunchPlan pl;
    pl.per_row = n_split > 0 ? 2 : 1;
    pl.shared_rows = n_split;
    pl.grid = rows + n_split;
    const char* deep_e = getenv("ICD_ATT_BWD_DEEP");         // 0: never the 128-register instantiation (A/B and test hook)
    pl.deep = (n_split == rows && rows > 0 && 2 * rows <= 2 * ICD_NUM_SMS && smem <= 100 * 1024 && !(deep_e && deep_e[0] == '0')) ? 1 : 0;
    return pl;
}

static size_t att_fwd16_smem(int P, int A) { return (2 * (size_t)A + ((P + 3) & ~3) + 40) * sizeof(float); }
static size_t att_bwd16_smem(int P, int C, int A) {
    return ((size_t)C + 5 * (size_t)A + 2 * ((P + 3) & ~3) + 40 + 8 * (((P + 15) >> 4) << 4)) * sizeof(float) + 3 * (size_t)C * 2;
}

extern "C" int icd_attention_step_launch_plan_bf16(int direction, int rows, int P, int C, int A, int32_t* out4) {
    ICD_CHECK_ARG(out4 && rows >= 0 && P > 0 && C > 0 && A > 0 && (direction == 0 || direction == 1), "attention_step_launch_plan_bf16: bad arguments");
    const AttLaunchPlan pl = direction == 0 ? att_fwd16_plan(rows, att_fwd16_smem(P, A)) : att_bwd16_plan(rows, P, att_bwd16_smem(P, C, A));
    out4[0] = pl.per_row; out4[1] = pl.shared_rows; out4[2] = pl.grid; out4[3] = pl.deep;
    return 0;
}

extern "C" int icd_attention_step_fwd_bf16(int rows, int P, int C, int A, const int32_t* img_index,
                                           const void* enc16, const void* att_enc16,
                                           const float* att_dec, int64_t ld_dec,
                                           const float* w_full, const float* b_full,
                                           const float* fbeta_pre, int64_t ld_fb,
                                           float* alpha, int64_t ld_alpha,
                                           float* awe_raw, float* gate, float* gated, void* gated16, void* stream) {
    cudaStream_t s = icd_stream(stream);
    if (rows == 0) return 0;
    ICD_CHECK_ARG(rows > 0 && P > 0, "attention_step_fwd_bf16: bad dims");
    ICD_CHECK_ARG(A % 8 == 0 && C % 8 == 0, "attention_step_fwd_bf16: A=%d and C=%d must be multiples of 8", A, C);
    ICD_CHECK_ARG(ld_dec % 4 == 0 && (!fbeta_pre || ld_fb % 4 == 0), "attention_step_fwd_bf16: row strides must be multiples of 4");
    const size_t smem = att_fwd16_smem(P, A);
    ICD_CHECK_ARG(smem <= 200 * 1024, "attention_step_fwd_bf16: A/P too large for shared memory");
    static size_t configured = 48 * 1024;
    if (smem > configured) {
        ICD_CUDA(cudaFuncSetAttribute(att_step_fwd_bf16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = smem;
    }
    const AttLaunchPlan plan = att_fwd16_plan(rows, smem);
    const int nsplit = plan.per_row;
    icd_prof_mark_begin(0, rows, s);
#define ICD_FWD16_ARGS P, C, A, (const int*)img_index, reinterpret_cast<const __nv_bfloat16*>(enc16),                      \
                       reinterpret_cast<const __nv_bfloat16*>(att_enc16), att_dec, (long long)ld_dec, w_full, b_full, fbeta_pre, \
                       (long long)ld_fb, alpha, (long long)ld_alpha, awe_raw, gate, gated, reinterpret_cast<__nv_bfloat16*>(gated16)
    if (nsplit == 4 && plan.deep)
        ICD_CUDA(icd_launch_pdl(ICD_PDL_ATT_FWD, att_step_fwd_bf16_split_kernel<2, true>, dim3(rows * 4), dim3(256), smem, s, ICD_FWD16_ARGS));
    else if (nsplit == 4)
        ICD_CUDA(icd_launch_pdl(ICD_PDL_ATT_FWD, att_step_fwd_bf16_split_kernel<2, false>, dim3(rows * 4), dim3(256), smem, s, ICD_FWD16_ARGS));
    else if (nsplit == 2 && plan.deep)
        ICD_CUDA(icd_launch_pdl(ICD_PDL_ATT_FWD, att_step_fwd_bf16_split_kernel<4, true>, dim3(rows * 2), dim3(256), smem, s, ICD_FWD16_ARGS));
    else if (nsplit == 2)
        ICD_CUDA(icd_launch_pdl(ICD_PDL_ATT_FWD, att_step_fwd_bf16_split_kernel<4, false>, dim3(rows * 2), dim3(256), smem, s, ICD_FWD16_ARGS));
    else
        ICD_CUDA(icd_launch_pdl(ICD_PDL_ATT_FWD, att_step_fwd_bf16_kernel, dim3(rows), dim3(256), smem, s, ICD_FWD16_ARGS));
#undef ICD_FWD16_ARGS
    icd_prof_mark_end(0, s);
    ICD_LAUNCH_CHECK();
    return 0;
}

extern "C" int icd_attention_step_bwd_bf16(int rows, int P, int C, int A,
                                           const void* enc16, const void* att_enc16,
                                           const float* att_dec, int64_t ld_dec, const float* w_full,
                                           const float* alpha, int64_t ld_alpha,
                                           const float* d_alpha_ext, int64_t ld_dalpha,
                                           const float* gate, const float* awe_raw, const float* d_gated,
                                           float* d_att_dec, int64_t ld_ddec,
                                           float* d_fbeta_pre, int64_t ld_dfb,
                                           float* d_e, int64_t ld_de,
                                           void* dz16, int64_t ld_dz16, float* d_awe_out, void* stream) {
    return icd_attention_step_bwd_bf16_idx(rows, P, C, A, nullptr, enc16, att_enc16, att_dec, ld_dec, w_full, alpha, ld_alpha,
                                           d_alpha_ext, ld_dalpha, gate, awe_raw, d_gated, d_att_dec, ld_ddec, d_fbeta_pre, ld_dfb,
                                           d_e, ld_de, dz16, ld_dz16, d_awe_out, stream);
}

int icd_attention_step_bwd_bf16_idx(int rows, int P, int C, int A, const int32_t* img_index,
                                    const void* enc16, const void* att_enc16,
                                    const float* att_dec, int64_t ld_dec, const float* w_full,
                                    const float* alpha, int64_t ld_alpha,
                                    const float* d_alpha_ext, int64_t ld_dalpha,
                                    const float* gate, const float* awe_raw, const float* d_gated,
                                    float* d_att_dec, int64_t ld_ddec,
                                    float* d_fbeta_pre, int64_t ld_dfb,
                                    float* d_e, int64_t ld_de,
                                    void* dz16, int64_t ld_dz16, float* d_awe_out, void* stream) {
    cudaStream_t s = icd_stream(stream);
    if (rows == 0) return 0;
    ICD_CHECK_ARG(A % 8 == 0 && C % 8 == 0, "attention_step_bwd_bf16: A and C must be multiples of 8");
    ICD_CHECK_ARG(ld_dec % 4 == 0 && ld_ddec % 4 == 0 && ld_dfb % 4 == 0 && (!dz16 || ld_dz16 % 8 == 0),
                  "attention_step_bwd_bf16: row strides misaligned");
    // tensor-core d_alpha path: 8 warps x channel strips of whole 32-channel blocks
    const int use_mma = (C % 256 == 0) ? 1 : 0;
    const size_t smem = att_bwd16_smem(P, C, A);
    ICD_CHECK_ARG(smem <= 200 * 1024, "attention_step_bwd_bf16: dims too large for shared memory");
    static size_t configured = 48 * 1024;
    if (smem > configured) {
        ICD_CUDA(cudaFuncSetAttribute(att_step_bwd_bf16_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ICD_CUDA(cudaFuncSetAttribute(att_step_bwd_bf16_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = smem;
    }
    const AttLaunchPlan plan = att_bwd16_plan(rows, P, smem);
    const int n_split = plan.shared_rows;
    icd_prof_mark_begin(1, rows, s);
#define ICD_BWD16_ARGS P, C, A, (const int*)img_index, reinterpret_cast<const __nv_bfloat16*>(enc16), reinterpret_cast<const __nv_bfloat16*>(att_enc16),           \
                       att_dec, (long long)ld_dec, w_full, alpha, (long long)ld_alpha, d_alpha_ext, (long long)ld_dalpha,                   \
                       gate, awe_raw, d_gated, d_att_dec, (long long)ld_ddec, d_fbeta_pre, (long long)ld_dfb,                               \
                       d_e, (long long)ld_de, reinterpret_cast<__nv_bfloat16*>(dz16), (long long)ld_dz16, d_awe_out, use_mma
    if (plan.deep)
        ICD_CUDA(icd_launch_pdl_cluster(ICD_PDL_ATT_BWD, att_step_bwd_bf16_kernel<true>, dim3(2 * rows), dim3(256), smem, s, 2u,
                                        ICD_BWD16_ARGS, 0));
    else if (n_split > 0)
        ICD_CUDA(icd_launch_pdl_cluster(ICD_PDL_ATT_BWD, att_step_bwd_bf16_kernel<false>, dim3(rows + n_split), dim3(256), smem, s, 2u, P, C, A,
                            (const int*)img_index, reinterpret_cast<const __nv_bfloat16*>(enc16), reinterpret_cast<const __nv_bfloat16*>(att_enc16),
                            att_dec, (long long)ld_dec, w_full, alpha, (long long)ld_alpha, d_alpha_ext, (long long)ld_dalpha,
                            gate, awe_raw, d_gated, d_att_dec, (long long)ld_ddec, d_fbeta_pre, (long long)ld_dfb,
                            d_e, (long long)ld_de, reinterpret_cast<__nv_bfloat16*>(dz16), (long long)ld_dz16, d_awe_out,
                            use_mma, rows - n_split));
    else
        ICD_CUDA(icd_launch_pdl(ICD_PDL_ATT_BWD, att_step_bwd_bf16_kernel<false>, dim3(rows), dim3(256), smem, s, P, C, A,
                            (const int*)img_index, reinterpret_cast<const __nv_bfloat16*>(enc16), reinterpret_cast<const __nv_bfloat16*>(att_enc16),
                            att_dec, (long long)ld_dec, w_full, alpha, (long long)ld_alpha, d_alpha_ext, (long long)ld_dalpha,
                            gate, awe_raw, d_gated, d_att_dec, (long long)ld_ddec, d_fbeta_pre, (long long)ld_dfb,
                            d_e, (long long)ld_de, reinterpret_cast<__nv_bfloat16*>(dz16), (long long)ld_dz16, d_awe_out,
                            use_mma, -1));
#undef ICD_BWD16_ARGS
    icd_prof_mark_end(1, s);
    ICD_LAUNCH_CHECK();
    return 0;
}

extern "C" int icd_attention_proj_bwd_bf16(int B, int T, int P, int A, const int32_t* bt_host,
                                           const void* att_enc16, const float* att_dec_all, int64_t ld_dec,
                                           const float* w_full, const float* d_e,
                                           float* d_att_enc, void* d_att_enc16, float* d_w_full, float* d_b_full,
                                           float* d_b_enc, float* partial, void* stream) {
    return icd_attention_proj_bwd_bf16_ex(B, T, P, A, bt_host, att_enc16, att_dec_all, ld_dec, w_full, d_e, d_att_enc, d_att_enc16,
                                          d_w_full, d_b_full, d_b_enc, partial, nullptr, 0, stream);
}

// d_att_dec_all != NULL: the (T*B, A) gradient w.r.t. att_dec that the per-step backward kernels wrote (rows of inactive
// (t, b) zero, as att_dec_all's): enables the split form of d_w_full (see att_proj_bwd_bf16_kernel).
extern "C" int icd_attention_proj_bwd_bf16_ex(int B, int T, int P, int A, const int32_t* bt_host,
                                              const void* att_enc16, const float* att_dec_all, int64_t ld_dec,
                                              const float* w_full, const float* d_e,
                                              float* d_att_enc, void* d_att_enc16, float* d_w_full, float* d_b_full,
                                              float* d_b_enc, float* partial, const float* d_att_dec_all, int64_t ld_ddec,
                                              void* stream) {
    cudaStream_t s = icd_stream(stream);
    ICD_CHECK_ARG(T > 0 && T <= ICD_MAX_STEPS, "attention_proj_bwd_bf16: T=%d out of range", T);
    ICD_CHECK_ARG(A % 4 == 0 && A / 4 <= 512, "attention_proj_bwd_bf16: A=%d unsupported", A);
    ICD_CHECK_ARG(ld_dec % 4 == 0, "attention_proj_bwd_bf16: ld_dec must be a multiple of 4");
    ICD_CHECK_ARG(B <= 65535, "attention_proj_bwd_bf16: B too large");
    const int chunks = (P + PROJ_PB - 1) / PROJ_PB;
    const int W = 2 * A + 4;
    int* row_len = reinterpret_cast<int*>(partial + (int64_t)B * chunks * W);
    BtPack pack;
    for (int t = 0; t < ICD_MAX_STEPS; ++t) pack.v[t] = t < T ? bt_host[t] : 0;
    ICD_CUDA(icd_launch_pdl(ICD_PDL_POINTWISE, row_len_from_pack_kernel16, dim3((unsigned)((B + 127) / 128)), dim3(128), (size_t)0, s, B, T, pack, row_len));
    ICD_LAUNCH_CHECK();
    // (the first 2*A floats are reused to add the two thread halves' partials: at least 2 rows of att_dec are allocated)
    const size_t smem = ((size_t)(T > 2 ? T : 2) * A + (size_t)T * PROJ_PB + 40) * sizeof(float);
    ICD_CHECK_ARG(smem <= 220 * 1024, "attention_proj_bwd_bf16: T*A too large for shared memory");
    static size_t configured = 48 * 1024;
    if (smem > configured) {
        ICD_CUDA(cudaFuncSetAttribute(att_proj_bwd_bf16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ICD_CUDA(cudaFuncSetAttribute(att_proj_bwd_bf16_kernel_wide, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = smem;
    }
    const int threads = 2 * (((A / 4 + 31) / 32) * 32);              // two halves, see the kernel
    dim3 grid(chunks, B);
    ICD_CUDA(icd_launch_pdl(ICD_PDL_POINTWISE, threads > 512 ? att_proj_bwd_bf16_kernel_wide : att_proj_bwd_bf16_kernel, grid,
                            dim3((unsigned)threads), smem, s, B, T, P, A, (const int*)row_len,
                            reinterpret_cast<const __nv_bfloat16*>(att_enc16), att_dec_all, ld_dec, w_full, d_e, d_att_enc,
                            reinterpret_cast<__nv_bfloat16*>(d_att_enc16), partial, d_att_dec_all ? 1 : 0));
    ICD_LAUNCH_CHECK();
    ICD_TRY(icd_colsum(partial, W, (int64_t)B * chunks, A, nullptr, d_w_full, s));
    if (d_att_dec_all) {
        float* t2 = partial + (int64_t)B * chunks * W + B + 8;       // (1 + COLDOT_CHUNKS) * A floats behind the row lengths
        float* t2_parts = t2 + A;
        ICD_CUDA(icd_launch_pdl(ICD_PDL_POINTWISE, coldot_kernel, dim3((A + 31) / 32, COLDOT_CHUNKS), dim3(32, 32), (size_t)0, s, att_dec_all,
                                (long long)ld_dec, d_att_dec_all, (long long)ld_ddec, (long long)T * B, A, t2_parts));
        ICD_LAUNCH_CHECK();
        ICD_TRY(icd_colsum(t2_parts, A, COLDOT_CHUNKS, A, nullptr, t2, s));
        ICD_CUDA(icd_launch_pdl(ICD_PDL_POINTWISE, proj_wfull_finish_kernel, dim3(1), dim3(256), (size_t)0, s, A, w_full, (const float*)t2, d_w_full));
        ICD_LAUNCH_CHECK();
    }
    if (d_b_enc) ICD_TRY(icd_colsum(partial + A, W, (int64_t)B * chunks, A, nullptr, d_b_enc, s));
    ICD_TRY(icd_colsum(partial + 2 * A, W, (int64_t)B * chunks, 1, nullptr, d_b_full, s));
    return 0;
}

// per-image pass (see att_proj_bwd_img_bf16_kernel); partial: icd_attention_proj_bwd_ws_floats_indexed floats, whose layout
// (per-image partials, then B row lengths, then the (1 + COLDOT_CHUNKS) * A floats of the split d_w_full) is that of the
// per-row pass with n_img * ceil(P / PROJ_IMG16_PB) partial rows
int icd_attention_proj_bwd_bf16_indexed(int B, int n_img, int T, int P, int A, const int32_t* bt_host, const int32_t* row_ptr,
                                        const int32_t* rows, const void* att_enc16, const float* att_dec_all, int64_t ld_dec,
                                        const float* w_full, const float* d_e, void* d_att_enc16, float* d_w_full,
                                        float* d_b_full, float* d_b_enc, float* partial, const float* d_att_dec_all,
                                        int64_t ld_ddec, cudaStream_t s) {
    ICD_CHECK_ARG(T > 0 && T <= ICD_MAX_STEPS, "attention_proj_bwd_bf16: T=%d out of range", T);
    ICD_CHECK_ARG(A % 4 == 0 && A / 4 <= 512, "attention_proj_bwd_bf16: A=%d unsupported", A);
    ICD_CHECK_ARG(ld_dec % 4 == 0, "attention_proj_bwd_bf16: ld_dec must be a multiple of 4");
    ICD_CHECK_ARG(n_img > 0 && n_img <= 65535, "attention_proj_bwd_bf16: n_img=%d out of range", n_img);
    const int chunks = (P + PROJ_IMG16_PB - 1) / PROJ_IMG16_PB;
    const int W = 2 * A + 4;
    const int64_t nparts = (int64_t)n_img * chunks;
    int* row_len = reinterpret_cast<int*>(partial + nparts * W);
    BtPack pack;
    for (int t = 0; t < ICD_MAX_STEPS; ++t) pack.v[t] = t < T ? bt_host[t] : 0;
    ICD_CUDA(icd_launch_pdl(ICD_PDL_POINTWISE, row_len_from_pack_kernel16, dim3((unsigned)((B + 127) / 128)), dim3(128), (size_t)0, s, B, T, pack, row_len));
    ICD_LAUNCH_CHECK();
    const size_t smem = ((size_t)PROJ_IMG16_KC * (A + PROJ_IMG16_PB) + 40) * sizeof(float);
    ICD_CHECK_ARG(smem <= 220 * 1024, "attention_proj_bwd_bf16: A too large for shared memory");
    static size_t configured = 48 * 1024;
    if (smem > configured) {
        ICD_CUDA(cudaFuncSetAttribute(att_proj_bwd_img_bf16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = smem;
    }
    const int threads = 2 * (((A / 4 + 31) / 32) * 32);
    ICD_CUDA(icd_launch_pdl(ICD_PDL_POINTWISE, att_proj_bwd_img_bf16_kernel, dim3(chunks, n_img), dim3((unsigned)threads), smem, s,
                            B, T, P, A, (const int*)row_len, (const int*)row_ptr, (const int*)rows,
                            reinterpret_cast<const __nv_bfloat16*>(att_enc16), att_dec_all, (long long)ld_dec, w_full, d_e,
                            reinterpret_cast<__nv_bfloat16*>(d_att_enc16), partial, d_att_dec_all ? 1 : 0));
    ICD_LAUNCH_CHECK();
    ICD_TRY(icd_colsum(partial, W, nparts, A, nullptr, d_w_full, s));
    if (d_att_dec_all) {
        float* t2 = partial + nparts * W + B + 8;
        float* t2_parts = t2 + A;
        ICD_CUDA(icd_launch_pdl(ICD_PDL_POINTWISE, coldot_kernel, dim3((A + 31) / 32, COLDOT_CHUNKS), dim3(32, 32), (size_t)0, s, att_dec_all,
                                (long long)ld_dec, d_att_dec_all, (long long)ld_ddec, (long long)T * B, A, t2_parts));
        ICD_LAUNCH_CHECK();
        ICD_TRY(icd_colsum(t2_parts, A, COLDOT_CHUNKS, A, nullptr, t2, s));
        ICD_CUDA(icd_launch_pdl(ICD_PDL_POINTWISE, proj_wfull_finish_kernel, dim3(1), dim3(256), (size_t)0, s, A, w_full, (const float*)t2, d_w_full));
        ICD_LAUNCH_CHECK();
    }
    if (d_b_enc) ICD_TRY(icd_colsum(partial + A, W, nparts, A, nullptr, d_b_enc, s));
    ICD_TRY(icd_colsum(partial + 2 * A, W, nparts, 1, nullptr, d_b_full, s));
    return 0;
}

int icd_convert_features_bf16(int B, int P, int C, const float* enc, void* enc16, float* mean, void* mean16, cudaStream_t s,
                              const int32_t* row_ptr, const int32_t* rows) {
    ICD_CHECK_ARG(C % 4 == 0 && B <= 65535, "convert_features: C=%d must be a multiple of 4, B <= 65535", C);
    dim3 grid((C + 255) / 256, B);
    ICD_CUDA(icd_launch_pdl(ICD_PDL_POINTWISE, convert_features_kernel, grid, dim3(256), (size_t)0, s, P, C, enc,
                            reinterpret_cast<__nv_bfloat16*>(enc16), mean, reinterpret_cast<__nv_bfloat16*>(mean16),
                            (const int*)row_ptr, (const int*)rows));
    ICD_LAUNCH_CHECK();
    return 0;
}

int icd_feature_mean_bf16(int B, int P, int C, const void* enc16, float* mean, void* mean16, cudaStream_t s,
                          const int32_t* row_ptr, const int32_t* rows) {
    ICD_CHECK_ARG(C % 8 == 0 && B <= 65535, "feature_mean_bf16: C=%d must be a multiple of 8, B <= 65535", C);
    dim3 grid((C + 511) / 512, B);
    ICD_CUDA(icd_launch_pdl(ICD_PDL_POINTWISE, feature_mean_bf16_kernel, grid, dim3(256), (size_t)0, s, P, C,
                            reinterpret_cast<const __nv_bfloat16*>(enc16), mean, reinterpret_cast<__nv_bfloat16*>(mean16),
                            (const int*)row_ptr, (const int*)rows));
    ICD_LAUNCH_CHECK();
    return 0;
}
