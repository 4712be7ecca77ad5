// Small fused pointwise / reduction kernels around the contractions:
//   LSTMCell gate math fwd/bwd (torch.nn.LSTMCell semantics, gate order i,f,g,o — models/attention.py:277-278,
//   models/baseline.py:106) with the nn.Dropout keep-mask of models/attention.py:279 fused into the h store,
//   masked column sums (bias gradients), embedding gather / scatter-add (models/attention.py:247),
//   Philox keep-mask generation, clamp+Adam (train_utils.py:2-12, models/attention.py:423-428),
//   row-wise cross-entropy forward+backward (models/attention.py:411).
#include "common.cuh"
#include <cuda_bf16.h>
#include <cstdlib>

namespace {

__global__ void lstm_pointwise_fwd_kernel(int rows, int D, const float* __restrict__ gates_pre,
                                          const float* __restrict__ c_prev, float* __restrict__ gates_act,
                                          float* __restrict__ c_new, float* __restrict__ h_new,
                                          float* __restrict__ hdrop, long long hdrop_row_stride,
                                          const unsigned char* __restrict__ mask, float scale,
                                          __nv_bfloat16* __restrict__ h16, __nv_bfloat16* __restrict__ hdrop16,
                                          const int* __restrict__ m_live) {
    pdl_trigger();
    pdl_wait();
    if (m_live) rows = min(rows, max(*m_live, 0));        // device-side row count (beam search: live rows only)
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)rows * D) return;
    const int r = (int)(idx / D), d = (int)(idx % D);
    const float* g = gates_pre + (long long)r * 4 * D;
    const float i = sigmoidf_(g[d]);
    const float f = sigmoidf_(g[D + d]);
    const float gg = tanhf(g[2 * D + d]);
    const float o = sigmoidf_(g[3 * D + d]);
    const float c = f * c_prev[idx] + i * gg;
    const float h = o * tanhf(c);
    if (gates_act) {
        float* ga = gates_act + (long long)r * 4 * D;
        ga[d] = i; ga[D + d] = f; ga[2 * D + d] = gg; ga[3 * D + d] = o;
    }
    c_new[idx] = c;
    h_new[idx] = h;
    if (hdrop) {
        float hd = h;
        if (mask) hd = mask[idx] ? h * scale : 0.f;
        hdrop[(long long)r * hdrop_row_stride + d] = hd;
        if (hdrop16) hdrop16[(long long)r * hdrop_row_stride + d] = __float2bfloat16_rn(hd);
    }
    if (h16) h16[idx] = __float2bfloat16_rn(h);
}

__global__ void lstm_pointwise_bwd_kernel(int rows, int D, const float* __restrict__ dh_in,
                                          const float* __restrict__ d_hdrop, long long hdrop_row_stride,
                                          const unsigned char* __restrict__ mask, float scale,
                                          float* __restrict__ dc_inout, const float* __restrict__ gates_act,
                                          const float* __restrict__ c_prev, const float* __restrict__ c_new,
                                          float* __restrict__ dgates_pre, long long ld_dg,
                                          __nv_bfloat16* __restrict__ dg16, long long ld_dg16,
                                          const float* __restrict__ dh_parts, int n_parts, int parts_rows) {
    pdl_trigger();
    pdl_wait();
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)rows * D) return;
    const int r = (int)(idx / D), d = (int)(idx % D);
    const float* ga = gates_act + (long long)r * 4 * D;
    const float i = ga[d], f = ga[D + d], g = ga[2 * D + d], o = ga[3 * D + d];
    float dh;
    if (n_parts > 0 && r < parts_rows) {       // deferred split-K: sum the K-slice planes of the dh contraction here
        dh = 0.f;
        const long long stride = (long long)parts_rows * D;
        for (int sp = 0; sp < n_parts; ++sp) dh += dh_parts[sp * stride + idx];
    } else dh = dh_in ? dh_in[idx] : 0.f;
    if (d_hdrop) {
        float u = d_hdrop[(long long)r * hdrop_row_stride + d];
        if (mask) u = mask[idx] ? u * scale : 0.f;
        dh += u;
    }
    const float tc = tanhf(c_new[idx]);
    const float d_o = dh * tc;
    const float dc = dc_inout[idx] + dh * o * (1.f - tc * tc);
    const float d_i = dc * g, d_g = dc * i, d_f = dc * c_prev[idx];
    dc_inout[idx] = dc * f;
    float* dg = dgates_pre + (long long)r * ld_dg;
    const float p_i = d_i * i * (1.f - i), p_f = d_f * f * (1.f - f), p_g = d_g * (1.f - g * g), p_o = d_o * o * (1.f - o);
    dg[d] = p_i; dg[D + d] = p_f; dg[2 * D + d] = p_g; dg[3 * D + d] = p_o;
    if (dg16) {
        __nv_bfloat16* q = dg16 + (long long)r * ld_dg16;
        q[d] = __float2bfloat16_rn(p_i); q[D + d] = __float2bfloat16_rn(p_f);
        q[2 * D + d] = __float2bfloat16_rn(p_g); q[3 * D + d] = __float2bfloat16_rn(p_o);
    }
}

// The same adjoint, four hidden units per thread (128-bit loads / stores, 64-bit bf16 stores), element arithmetic identical to
// the scalar kernel above (results are bit-identical).  Operands that the FORWARD pass produced (gate activations, cell
// states, keep mask) are fetched BEFORE griddepcontrol.wait, so their latency hides behind the tail of the dh contraction in
// front of this launch.  Everything the backward itself writes is read after the wait: dh and dc (dc by the previous adjoint,
// which in the baseline decoder's chain may still be running when this grid becomes resident) and the vocabulary-layer
// gradient — at the first time step its contraction is only a few early-launched kernels upstream and may still be running
// (see pdl_trigger in common.cuh).
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void st4_bf16(__nv_bfloat16* p, float4 v) {
    __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
    uint2 w;
    w.x = *reinterpret_cast<unsigned*>(&lo); w.y = *reinterpret_cast<unsigned*>(&hi);
    *reinterpret_cast<uint2*>(p) = w;
}

__global__ void __launch_bounds__(128) lstm_pointwise_bwd_vec4_kernel(
        int rows, int D, const float* __restrict__ dh_in, const float* __restrict__ d_hdrop, long long hdrop_row_stride,
        const unsigned char* __restrict__ mask, float scale, float* __restrict__ dc_inout,
        const float* __restrict__ gates_act, const float* __restrict__ c_prev, const float* __restrict__ c_new,
        float* __restrict__ dgates_pre, long long ld_dg, __nv_bfloat16* __restrict__ dg16, long long ld_dg16,
        const float* __restrict__ dh_parts, int n_parts, int parts_rows) {
    pdl_trigger();
    const int D4 = D >> 2;
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = q < (long long)rows * D4;
    int r = 0, d = 0;
    long long idx = 0;
    float4 gi, gf, gg, go, cn, cp, u;
    gi = gf = gg = go = cn = cp = u = make_float4(0.f, 0.f, 0.f, 0.f);
    uchar4 m = make_uchar4(1, 1, 1, 1);
    if (live) {
        r = (int)(q / D4); d = (int)(q % D4) * 4;
        idx = (long long)r * D + d;
        const float* ga = gates_act + (long long)r * 4 * D + d;
        gi = ld4(ga); gf = ld4(ga + D); gg = ld4(ga + 2 * D); go = ld4(ga + 3 * D);
        cn = ld4(c_new + idx); cp = ld4(c_prev + idx);
        if (d_hdrop && mask) m = *reinterpret_cast<const uchar4*>(mask + idx);
    }
    pdl_wait();
    if (!live) return;
    if (d_hdrop) {
        u = ld4(d_hdrop + (long long)r * hdrop_row_stride + d);
        if (mask) {
            u.x = m.x ? u.x * scale : 0.f; u.y = m.y ? u.y * scale : 0.f;
            u.z = m.z ? u.z * scale : 0.f; u.w = m.w ? u.w * scale : 0.f;
        }
    }
    float4 dh;
    if (n_parts > 0 && r < parts_rows) {       // deferred split-K: sum the K-slice planes of the dh contraction here
        dh = make_float4(0.f, 0.f, 0.f, 0.f);
        const long long stride = (long long)parts_rows * D;
        for (int sp = 0; sp < n_parts; ++sp) {
            const float4 p = ld4(dh_parts + sp * stride + idx);
            dh.x += p.x; dh.y += p.y; dh.z += p.z; dh.w += p.w;
        }
    } else dh = dh_in ? ld4(dh_in + idx) : make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 dc_old = ld4(dc_inout + idx);
    float4 pi, pf, pg, po, dcn;
#define ICD_ADJ(X)                                                                                                    \
    {                                                                                                                 \
        const float i = gi.X, f = gf.X, g = gg.X, o = go.X;                                                           \
        float dhx = dh.X;                                                                                             \
        if (d_hdrop) dhx += u.X;                                                                                      \
        const float tc = tanhf(cn.X);                                                                                 \
        const float d_o = dhx * tc;                                                                                   \
        const float dc = dc_old.X + dhx * o * (1.f - tc * tc);                                                        \
        const float d_i = dc * g, d_g = dc * i, d_f = dc * cp.X;                                                      \
        dcn.X = dc * f;                                                                                               \
        pi.X = d_i * i * (1.f - i); pf.X = d_f * f * (1.f - f); pg.X = d_g * (1.f - g * g); po.X = d_o * o * (1.f - o); \
    }
    ICD_ADJ(x) ICD_ADJ(y) ICD_ADJ(z) ICD_ADJ(w)
#undef ICD_ADJ
    st4(dc_inout + idx, dcn);
    float* dg = dgates_pre + (long long)r * ld_dg + d;
    st4(dg, pi); st4(dg + D, pf); st4(dg + 2 * D, pg); st4(dg + 3 * D, po);
    if (dg16) {
        __nv_bfloat16* q16 = dg16 + (long long)r * ld_dg16 + d;
        st4_bf16(q16, pi); st4_bf16(q16 + D, pf); st4_bf16(q16 + 2 * D, pg); st4_bf16(q16 + 3 * D, po);
    }
}

// out[n] = sum_m mask[m] * X[m*ld + n].  block (32,32): x -> column, y -> row phase.  deterministic.
__global__ void colsum_kernel(const float* __restrict__ X, long long ld, long long M, int N,
                              const unsigned char* __restrict__ row_mask, float* __restrict__ out) {
    pdl_trigger();
    pdl_wait();
    __shared__ float s[32][33];
    const int n = blockIdx.x * 32 + threadIdx.x;
    float acc = 0.f;
    if (n < N) {
        for (long long m = threadIdx.y; m < M; m += 32)
            if (!row_mask || row_mask[m]) acc += X[m * ld + n];
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

// partial[chunk][n] = sum over the rows of `chunk` of mask[m] * X16[m*ld + n]   (bf16 source, fp32 accumulate).
// grid = (ceil(N/1024), chunks), block = 128 threads x 8 columns; 8 rows in flight per thread with 128-bit loads when the
// rows are 16-byte aligned (vec), element loads otherwise; masked rows are not read.  Rows are added in index order.
constexpr int COLSUM16_ROWS = 128;          // rows per chunk (partial row); also the workspace contract below
__global__ void __launch_bounds__(128) colsum_bf16_partial_kernel(const __nv_bfloat16* __restrict__ X, long long ld,
                                                                  long long M, int N, int rows_per_chunk,
                                                                  const unsigned char* __restrict__ row_mask,
                                                                  float* __restrict__ partial, int vec) {
    pdl_trigger();
    pdl_wait();
    const int n = blockIdx.x * 1024 + threadIdx.x * 8;
    if (n >= N) return;
    const long long m0 = (long long)blockIdx.y * rows_per_chunk;
    const long long m1 = min(M, m0 + rows_per_chunk);
    const int nc = min(8, N - n);                          // valid columns of this thread
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    auto load_row = [&](long long m) -> uint4 {
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (row_mask && !row_mask[m]) return v;            // masked row: contributes +0, not read
        const __nv_bfloat16* p = X + m * ld + n;
        if (vec && nc == 8) return *reinterpret_cast<const uint4*>(p);
        unsigned short e[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) e[j] = (j < nc) ? *reinterpret_cast<const unsigned short*>(p + j) : (unsigned short)0;
        v.x = e[0] | ((uint32_t)e[1] << 16); v.y = e[2] | ((uint32_t)e[3] << 16);
        v.z = e[4] | ((uint32_t)e[5] << 16); v.w = e[6] | ((uint32_t)e[7] << 16);
        return v;
    };
    auto add_row = [&](const uint4& v) {
        acc[0] += __uint_as_float(v.x << 16); acc[1] += __uint_as_float(v.x & 0xffff0000u);
        acc[2] += __uint_as_float(v.y << 16); acc[3] += __uint_as_float(v.y & 0xffff0000u);
        acc[4] += __uint_as_float(v.z << 16); acc[5] += __uint_as_float(v.z & 0xffff0000u);
        acc[6] += __uint_as_float(v.w << 16); acc[7] += __uint_as_float(v.w & 0xffff0000u);
    };
    long long m = m0;
    for (; m + 7 < m1; m += 8) {
        uint4 v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = load_row(m + u);
#pragma unroll
        for (int u = 0; u < 8; ++u) add_row(v[u]);
    }
    for (; m < m1; ++m) add_row(load_row(m));
    float* o = partial + (long long)blockIdx.y * N + n;
#pragma unroll
    for (int j = 0; j < 8; ++j) if (j < nc) o[j] = acc[j];
}

template <typename TT>
__global__ void embed_gather_kernel(const TT* __restrict__ table, const long long* __restrict__ captions,
                                    int B, int L, int T, int E, int V, float* __restrict__ out) {
    pdl_trigger();
    pdl_wait();
    const int row = blockIdx.x;                  // row = t*B + b
    const int t = row / B, b = row % B;
    const long long tok = captions[(long long)b * L + t];
    if (tok < 0 || tok >= V) __trap();           // nn.Embedding raises on an out-of-range id; never read outside the table
    const TT* src = table + tok * E;
    float* dst = out + (long long)row * E;
    for (int e = threadIdx.x; e < E; e += blockDim.x) dst[e] = (float)src[e];
}

struct BtPack { int v[ICD_MAX_STEPS]; };

template <typename TT>
__global__ void embed_scatter_add_kernel(TT* __restrict__ d_table, const long long* __restrict__ captions,
                                         int B, int L, int T, int E, const BtPack bt,
                                         const float* __restrict__ d_x) {
    const int row = blockIdx.x;
    const int t = row / B, b = row % B;
    if (b >= bt.v[t]) return;
    const long long tok = captions[(long long)b * L + t];
    TT* dst = d_table + tok * E;
    const float* src = d_x + (long long)row * E;
    for (int e = threadIdx.x; e < E; e += blockDim.x) atomicAdd(dst + e, (TT)src[e]);
}

// ---- deterministic embedding gradient: sort the (token, row) pairs, then one CTA per token adds its rows in row order -------
// (the atomic variant above accumulates in arrival order: run-to-run different in the last bits, and slow in fp64)
constexpr int EMB_SORT_N = 16384;                   // keys per chunk: 128 KB of shared memory
constexpr unsigned long long EMB_KEY_NONE = ~0ull;

// chunk c sorts rows [c * EMB_SORT_N, ...) of the (T, B) row space by (token id, row index): key = token << 32 | row; rows
// that are inactive at their step (b >= batch_size_t) get the sentinel and sink to the end.  Bitonic network in shared memory.
__global__ void __launch_bounds__(1024) embed_sort_kernel(const long long* __restrict__ captions, int B, int L, int T, int V,
                                                           const BtPack bt, int n_sort, unsigned long long* __restrict__ keys) {
    extern __shared__ unsigned long long s_key[];
    const long long base = (long long)blockIdx.x * EMB_SORT_N;
    const long long N = (long long)T * B;
    for (int i = threadIdx.x; i < n_sort; i += blockDim.x) {
        const long long r = base + i;
        unsigned long long key = EMB_KEY_NONE;
        if (r < N) {
            const int t = (int)(r / B), b = (int)(r % B);
            if (b < bt.v[t]) {
                const long long tok = captions[(long long)b * L + t];
                if (tok < 0 || tok >= V) __trap();
                key = ((unsigned long long)tok << 32) | (unsigned long long)(unsigned int)r;
            }
        }
        s_key[i] = key;
    }
    __syncthreads();
    for (int k = 2; k <= n_sort; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < n_sort; i += blockDim.x) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const unsigned long long a = s_key[i], b2 = s_key[ixj];
                    const bool asc = (i & k) == 0;
                    if ((a > b2) == asc) { s_key[i] = b2; s_key[ixj] = a; }
                }
            }
            __syncthreads();
        }
    }
    for (int i = threadIdx.x; i < n_sort; i += blockDim.x) keys[base + i] = s_key[i];
}

// one CTA (8 warps) per sorted position; only segment heads (first occurrence of a token in the chunk) work.  Warp w adds the
// segment's rows head + w, head + w + 8, ... in ascending order (lanes own columns e = lane, lane + 32, ...: every row is one
// coalesced read), then the eight partial sums are added in warp order — a FIXED association, so the result is deterministic —
// and accumulated into the table row (chunks are launched one after the other: no two CTAs touch a table row concurrently).
constexpr int EMB_MAX_E = 1024;                     // columns per table row the register accumulators cover (E <= 1024)
template <typename TT>
__global__ void __launch_bounds__(256) embed_segment_reduce_kernel(const unsigned long long* __restrict__ keys, int n_sort,
                                                                    const float* __restrict__ d_x, TT* __restrict__ d_table, int E) {
    extern __shared__ unsigned char s_raw[];
    TT* s_part = reinterpret_cast<TT*>(s_raw);                           // [8 warps][E]
    const int i = blockIdx.x;
    const unsigned long long key = keys[i];
    if (key == EMB_KEY_NONE) return;
    const unsigned int tok = (unsigned int)(key >> 32);
    if (i > 0 && (unsigned int)(keys[i - 1] >> 32) == tok) return;
    int end = i + 1;
    while (end < n_sort && keys[end] != EMB_KEY_NONE && (unsigned int)(keys[end] >> 32) == tok) ++end;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int NE = EMB_MAX_E / 32;
    TT acc[NE];
#pragma unroll
    for (int q = 0; q < NE; ++q) acc[q] = (TT)0;
    for (int j = i + warp; j < end; j += 8) {
        const float* src = d_x + (long long)(unsigned int)(keys[j] & 0xffffffffull) * E;
#pragma unroll
        for (int q = 0; q < NE; ++q) { const int e = lane + 32 * q; if (e < E) acc[q] += (TT)src[e]; }
    }
#pragma unroll
    for (int q = 0; q < NE; ++q) { const int e = lane + 32 * q; if (e < E) s_part[(size_t)warp * E + e] = acc[q]; }
    __syncthreads();
    TT* dst = d_table + (long long)tok * E;
    for (int e = threadIdx.x; e < E; e += blockDim.x) {
        TT t = s_part[e];
#pragma unroll
        for (int w = 1; w < 8; ++w) t += s_part[(size_t)w * E + e];
        dst[e] += t;
    }
}

__global__ void dropout_mask_kernel(unsigned char* __restrict__ out, long long n, float p,
                                    unsigned long long seed, unsigned long long offset) {
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // one thread -> 4 outputs
    if (q * 4 >= n) return;
    const unsigned long long ctr = offset + (unsigned long long)q;
    uint32_t c[4] = {(uint32_t)ctr, (uint32_t)(ctr >> 32), 0u, 0u};
    philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));          // common.cuh
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const long long i = q * 4 + j;
        if (i < n) {
            const float u = (float)(c[j] >> 8) * (1.0f / 16777216.0f);   // [0,1)
            out[i] = (u >= p) ? 1 : 0;
        }
    }
}

__global__ void clip_adam_kernel(float* __restrict__ param, const float* __restrict__ grad,
                                 float* __restrict__ m, float* __restrict__ v, long long n,
                                 float grad_scale, float clip, float lr, float b1, float b2, float eps,
                                 float bias_c1, float bias_c2_sqrt) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x) {
        float g = grad[i] * grad_scale;
        g = fminf(fmaxf(g, -clip), clip);                         // train_utils.py:12 clamp_(-c, c)
        const float mi = b1 * m[i] + (1.f - b1) * g;              // torch.optim.Adam (single-tensor form)
        const float vi = b2 * v[i] + (1.f - b2) * g * g;
        m[i] = mi; v[i] = vi;
        const float denom = sqrtf(vi) / bias_c2_sqrt + eps;
        param[i] -= (lr / bias_c1) * (mi / denom);
    }
}

// Row-wise softmax cross-entropy.  Forward: grid = R rows, block = 256: row_loss[r] = lse - logit[target] (0 for ignored
// rows), lse[r] saved.  Backward: one CTA per row again, pure streaming: d = (exp(x - lse) - onehot) * scale with
// scale = inv_count * upstream[0] read from device memory; optional bf16 copy (row stride ld16, tail columns zeroed).
__device__ __forceinline__ void online_add(float& m, float& s, float x) {       // running (max, sum exp(x - max))
    const float mn = fmaxf(m, x);
    s = s * __expf(m - mn) + __expf(x - mn);
    m = mn;
}
__device__ __forceinline__ void online_merge(float& m, float& s, float m2, float s2) {
    const float mn = fmaxf(m, m2);
    const float a = (m == -INFINITY) ? 0.f : s * __expf(m - mn);
    const float b = (m2 == -INFINITY) ? 0.f : s2 * __expf(m2 - mn);
    s = a + b; m = mn;
}

// d(loss)/d(logit) of one element: (exp(x - lse) - onehot) * scale.  ONE definition for the streaming backward kernel and the
// one-pass kernel, so their bf16 gradients agree bit for bit (exp through ex2.approx: 2^-22 relative, far inside every tier's bar).
__device__ __forceinline__ float ce_grad(float x, bool is_target, float lse, float scale) {
    return (__expf(x - lse) - (is_target ? 1.f : 0.f)) * scale;
}

// Running (max, sum exp) of one row over a 256-thread CTA, before the cross-thread merge: scalar head up to the row's first
// 16-byte boundary (rows of V = 9490 floats start 8-byte aligned on odd r), scalar tail, 128-bit body.  CE_U body loads of a thread are issued
// before the first one is consumed.  (Measured on the 12288 x 9490 logits: more loads per thread lose more through the lower
// occupancy than they gain — 3 at eight CTAs per SM for the streaming kernel, 5 at five CTAs per SM for the kernel that parks the row.)  PARK: the row is also copied to shared memory (sx[v] = x[v]).  One definition for
// cross_entropy_fwd_kernel and the one-pass kernel: their log-sum-exp agrees bit for bit.
template <bool PARK, int CE_U>
__device__ __forceinline__ void ce_row_stats(const float* __restrict__ x, int V, int head, int V4, float* sx, float& m, float& s) {
    if ((int)threadIdx.x < head) { const float v = x[threadIdx.x]; if (PARK) sx[threadIdx.x] = v; online_add(m, s, v); }
    for (int v = head + 4 * V4 + threadIdx.x; v < V; v += 256) { const float t = x[v]; if (PARK) sx[v] = t; online_add(m, s, t); }
    const float* xb = x + head;
    for (int j0 = threadIdx.x; j0 < V4; j0 += CE_U * 256) {
        float4 v[CE_U];
#pragma unroll
        for (int u = 0; u < CE_U; ++u)
            if (j0 + u * 256 < V4) v[u] = ld_stream_f4(xb + 4 * (j0 + u * 256));
#pragma unroll
        for (int u = 0; u < CE_U; ++u) {
            if (j0 + u * 256 < V4) {
                if (PARK) *reinterpret_cast<float4*>(sx + head + 4 * (j0 + u * 256)) = v[u];
                const float mx = fmaxf(fmaxf(v[u].x, v[u].y), fmaxf(v[u].z, v[u].w)), mn = fmaxf(m, mx);
                s = s * __expf(m - mn) + __expf(v[u].x - mn) + __expf(v[u].y - mn) + __expf(v[u].z - mn) + __expf(v[u].w - mn);
                m = mn;
            }
        }
    }
}

// single pass over the row: online log-sum-exp, 128-bit loads (scalar head / tail around the 16-byte aligned body)
__global__ void __launch_bounds__(256, 8) cross_entropy_fwd_kernel(int V, const float* __restrict__ logits,
                                                                const long long* __restrict__ targets,
                                                                float* __restrict__ row_loss, float* __restrict__ lse_out) {
    __shared__ float s_m[8], s_s[8];
    const long long r = blockIdx.x;
    const float* x = logits + r * V;
    const long long tgt = targets[r];
    if (tgt < 0) {
        if (threadIdx.x == 0) { row_loss[r] = 0.f; lse_out[r] = 0.f; }
        return;
    }
    if (tgt >= V) __trap();                          // nn.CrossEntropyLoss raises on a class index >= V; never read outside the row
    float m = -INFINITY, s = 0.f;
    const int head = min(V, (int)((4 - ((reinterpret_cast<uintptr_t>(x) >> 2) & 3)) & 3));      // see ce_row_stats
    const int V4 = (V - head) >> 2;
    ce_row_stats<false, 3>(x, V, head, V4, nullptr, m, s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, s, o);
        online_merge(m, s, m2, s2);
    }
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) { s_m[w] = m; s_s[w] = s; }
    __syncthreads();
    if (threadIdx.x == 0) {
        float M = s_m[0], S = s_s[0];
        for (int i = 1; i < 8; ++i) online_merge(M, S, s_m[i], s_s[i]);
        const float lse = M + logf(S);
        row_loss[r] = lse - x[tgt];
        lse_out[r] = lse;
    }
}

// Forward AND gradient in one pass over the logits (training fast path of the bf16 tier): the row is parked in shared memory
// while its log-sum-exp is formed (exactly as cross_entropy_fwd_kernel does), then the bf16 gradient
// (exp(x - lse) - onehot) * inv_count is written from the parked copy — every logit is read from HBM once instead of twice.
// The upstream gradient of the loss is applied afterwards (scale_bf16_by_device_scalar_kernel: a no-op when it is 1).
// WEIGHTED: the gradient of row r is also scaled by weights[r] (scale = inv_count * w_r; row_loss stays unweighted).
template <bool WEIGHTED>
__global__ void __launch_bounds__(256, 5) cross_entropy_fwd_grad16_kernel(int V, const float* __restrict__ logits,
                                                                       const long long* __restrict__ targets, float inv_count,
                                                                       float* __restrict__ row_loss, float* __restrict__ lse_out,
                                                                       __nv_bfloat16* __restrict__ d16, long long ld16,
                                                                       const float* __restrict__ weights) {
    extern __shared__ __align__(16) float s_x[];     // V floats (+ reduction scratch behind them)
    float* s_m = s_x + ((V + 3) & ~3) + 4;           // behind the row and its alignment pad (see sx below)
    float* s_s = s_m + 8;
    const long long r = blockIdx.x;
    const float* x = logits + r * V;
    const long long tgt = targets[r];
    __nv_bfloat16* d16r = d16 + r * ld16;
    if (tgt >= V) __trap();
    if (tgt < 0) {                                   // ignored row: loss 0, zero gradient row (16-byte aligned, ld16 % 8 == 0)
        if (threadIdx.x == 0) { row_loss[r] = 0.f; lse_out[r] = 0.f; }
        uint4* z = reinterpret_cast<uint4*>(d16r);
        for (int v = threadIdx.x; v < (int)(ld16 >> 3); v += blockDim.x) z[v] = make_uint4(0u, 0u, 0u, 0u);
        return;
    }
    float m = -INFINITY, s = 0.f;
    const int head = min(V, (int)((4 - ((reinterpret_cast<uintptr_t>(x) >> 2) & 3)) & 3));
    const int V4 = (V - head) >> 2;
    // the shared copy keeps the row's own alignment phase: element v lives at s_x[v + pad], pad = (4 - head) & 3, so that the
    // 128-bit body is 16-byte aligned on both sides
    const int pad = (4 - head) & 3;
    float* sx = s_x + pad;
    ce_row_stats<true, 5>(x, V, head, V4, sx, m, s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, s, o);
        online_merge(m, s, m2, s2);
    }
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) { s_m[w] = m; s_s[w] = s; }
    __syncthreads();                                  // also: the parked row is complete
    float M = s_m[0], S = s_s[0];
    for (int i = 1; i < 8; ++i) online_merge(M, S, s_m[i], s_s[i]);      // every thread, same order as cross_entropy_fwd_kernel
    const float lse = M + logf(S);
    if (threadIdx.x == 0) { row_loss[r] = lse - sx[tgt]; lse_out[r] = lse; }
    // gradient, 8 columns (16 bytes of bf16) per thread and pass; the parked row is read back with 64-bit accesses when its
    // alignment phase allows (pad even: every row of an even-V matrix)
    const int V8 = V >> 3, itgt = (int)tgt;
    const bool pair_ok = (pad & 1) == 0;
    float scale = inv_count;
    if (WEIGHTED) scale *= weights[r];
    for (int q = threadIdx.x; q < (int)(ld16 >> 3); q += 256) {
        float xv[8];
        const int v0 = 8 * q;
        if (q < V8 && pair_ok) {
#pragma unroll
            for (int h = 0; h < 4; ++h) { const float2 t = *reinterpret_cast<const float2*>(sx + v0 + 2 * h); xv[2 * h] = t.x; xv[2 * h + 1] = t.y; }
        } else {
#pragma unroll
            for (int h = 0; h < 8; ++h) xv[h] = (v0 + h < V) ? sx[v0 + h] : 0.f;
        }
        float g[8];
#pragma unroll
        for (int h = 0; h < 8; ++h) g[h] = ce_grad(xv[h], v0 + h == itgt, lse, scale);
        if (q >= V8) {
#pragma unroll
            for (int h = 0; h < 8; ++h) if (v0 + h >= V) g[h] = 0.f;                    // pad columns of the bf16 row
        }
        uint32_t pk[4];
#pragma unroll
        for (int h = 0; h < 4; ++h) { const __nv_bfloat162 t = __floats2bfloat162_rn(g[2 * h], g[2 * h + 1]); pk[h] = *reinterpret_cast<const uint32_t*>(&t); }
        *reinterpret_cast<uint4*>(d16r + v0) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    }
}

// x[i] *= *scale for a bf16 buffer — unless *scale == 1 (the usual upstream gradient of a loss): then nothing is touched
__global__ void __launch_bounds__(256) scale_bf16_by_device_scalar_kernel(__nv_bfloat16* __restrict__ x, long long n8,
                                                                          const float* __restrict__ scale) {
    const float g = scale[0];
    if (g == 1.f) return;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n8; i += (long long)gridDim.x * 256) {
        uint4 v = reinterpret_cast<uint4*>(x)[i];
        uint32_t* w = reinterpret_cast<uint32_t*>(&v);
#pragma unroll
        for (int h = 0; h < 4; ++h) {
            const float lo = __uint_as_float(w[h] << 16) * g, hi = __uint_as_float(w[h] & 0xffff0000u) * g;
            const __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
            w[h] = *reinterpret_cast<const uint32_t*>(&t);
        }
        reinterpret_cast<uint4*>(x)[i] = v;
    }
}

// WEIGHTED: the gradient of row r is also scaled by weights[r] (scale = (inv_count * upstream) * w_r, so w = 1 gives the
// unweighted bits); a row of weight 0 is still written, as zeros.
template <bool WEIGHTED>
__global__ void __launch_bounds__(256) cross_entropy_bwd_kernel(int V, const float* __restrict__ logits,
                                                                const long long* __restrict__ targets,
                                                                const float* __restrict__ lse_in,
                                                                const float* __restrict__ upstream, float inv_count,
                                                                float* __restrict__ d_logits,
                                                                __nv_bfloat16* __restrict__ d16, long long ld16,
                                                                const float* __restrict__ weights) {
    const long long r = blockIdx.x;
    const float* x = logits + r * V;
    const long long tgt = targets[r];
    float* dx = d_logits ? d_logits + r * V : nullptr;
    __nv_bfloat16* d16r = d16 ? d16 + r * ld16 : nullptr;
    if (tgt >= V) __trap();
    if (d16r) for (int v = V + threadIdx.x; v < ld16; v += blockDim.x) d16r[v] = __float2bfloat16_rn(0.f);
    if (tgt < 0) {                                   // ignored row: zeros (the bf16 row is 16-byte aligned, ld16 % 8 == 0)
        if (dx) for (int v = threadIdx.x; v < V; v += blockDim.x) dx[v] = 0.f;
        if (d16r) {
            uint4* z = reinterpret_cast<uint4*>(d16r);
            for (int v = threadIdx.x; v < (int)(ld16 >> 3); v += blockDim.x) z[v] = make_uint4(0u, 0u, 0u, 0u);
        }
        return;
    }
    const float lse = lse_in[r];
    float scale = inv_count * (upstream ? upstream[0] : 1.f);
    if (WEIGHTED) scale *= weights[r];
    // scalar head up to the row's first 16-byte boundary, 128-bit body with four loads in flight per thread, scalar tail
    // (the fp32 gradient rows share the alignment of the logit rows when both buffers are 16-byte aligned)
    const int itgt = (int)tgt;
    auto grad = [&](float xv, int v) { return ce_grad(xv, v == itgt, lse, scale); };
    auto emit1 = [&](int v) {
        const float g = grad(x[v], v);
        if (dx) dx[v] = g;
        if (d16r) d16r[v] = __float2bfloat16_rn(g);
    };
    const int head = min(V, (int)((4 - ((reinterpret_cast<uintptr_t>(x) >> 2) & 3)) & 3));
    const int V4 = (V - head) >> 2;
    if ((int)threadIdx.x < head) emit1(threadIdx.x);
    for (int v = head + 4 * V4 + threadIdx.x; v < V; v += 256) emit1(v);
    const bool dx_vec = dx && ((reinterpret_cast<uintptr_t>(dx + head) & 15) == 0);
    auto emit4 = [&](int jj, float4 xv) {
        const int v = head + 4 * jj;
        const float4 g = make_float4(grad(xv.x, v), grad(xv.y, v + 1), grad(xv.z, v + 2), grad(xv.w, v + 3));
        if (dx) {
            if (dx_vec) *reinterpret_cast<float4*>(dx + v) = g;
            else { dx[v] = g.x; dx[v + 1] = g.y; dx[v + 2] = g.z; dx[v + 3] = g.w; }
        }
        if (d16r) {
            const __nv_bfloat162 lo = __floats2bfloat162_rn(g.x, g.y), hi = __floats2bfloat162_rn(g.z, g.w);
            if ((v & 3) == 0) {                                        // 8-byte aligned in the bf16 row
                uint2 pk; pk.x = *reinterpret_cast<const uint32_t*>(&lo); pk.y = *reinterpret_cast<const uint32_t*>(&hi);
                *reinterpret_cast<uint2*>(d16r + v) = pk;
            } else if ((v & 1) == 0) {
                *reinterpret_cast<__nv_bfloat162*>(d16r + v) = lo; *reinterpret_cast<__nv_bfloat162*>(d16r + v + 2) = hi;
            } else {
                d16r[v] = __low2bfloat16(lo); d16r[v + 1] = __high2bfloat16(lo); d16r[v + 2] = __low2bfloat16(hi); d16r[v + 3] = __high2bfloat16(hi);
            }
        }
    };
    const float* xb = x + head;
    int j = threadIdx.x;
    for (; j + 3 * 256 < V4; j += 4 * 256) {
        float4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = ld_stream_f4(xb + 4 * (j + u * 256));
#pragma unroll
        for (int u = 0; u < 4; ++u) emit4(j + u * 256, v[u]);
    }
    for (; j < V4; j += 256) emit4(j, ld_stream_f4(xb + 4 * j));
}

}  // namespace

int icd_lstm_pointwise_fwd(int rows, int D, const float* gates_pre, const float* c_prev,
                           float* gates_act, float* c_new, float* h_new,
                           float* hdrop, int64_t hdrop_row_stride, const uint8_t* mask, float scale,
                           cudaStream_t s, void* h16, void* hdrop16, const int* m_live) {
    if (rows == 0) return 0;
    const long long n = (long long)rows * D;
    ICD_CUDA(icd_launch_pdl(ICD_PDL_POINTWISE, lstm_pointwise_fwd_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), (size_t)0, s, rows, D,
                            gates_pre, c_prev, gates_act, c_new, h_new, hdrop, (long long)hdrop_row_stride,
                            (const unsigned char*)mask, scale, (__nv_bfloat16*)h16, (__nv_bfloat16*)hdrop16, m_live));
    ICD_LAUNCH_CHECK();
    return 0;
}

int icd_lstm_pointwise_bwd(int rows, int D, const float* dh_in, const float* d_hdrop, int64_t hdrop_row_stride,
                           const uint8_t* mask, float scale, float* dc_inout,
                           const float* gates_act, const float* c_prev, const float* c_new,
                           float* dgates_pre, int64_t ld_dg, cudaStream_t s, void* dg16, int64_t ld_dg16,
                           const float* dh_parts, int n_parts, int parts_rows) {
    if (rows == 0) return 0;
    const long long n = (long long)rows * D;
    auto al = [](const void* p, uintptr_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; };
    const bool scalar_only = getenv("ICD_LSTM_BWD_SCALAR") != nullptr;        // test hook: the one-unit-per-thread kernel
    const bool vec4 = !scalar_only && D % 4 == 0 && ld_dg % 4 == 0 && hdrop_row_stride % 4 == 0 && (!dg16 || ld_dg16 % 4 == 0) &&
                      al(dh_in, 16) && al(d_hdrop, 16) && al(mask, 4) && al(dc_inout, 16) && al(gates_act, 16) && al(c_prev, 16) &&
                      al(c_new, 16) && al(dgates_pre, 16) && al(dg16, 8) && al(dh_parts, 16);
    if (vec4) {
        ICD_CUDA(icd_launch_pdl(ICD_PDL_POINTWISE, lstm_pointwise_bwd_vec4_kernel, dim3((unsigned)((n / 4 + 127) / 128)), dim3(128), (size_t)0,
                                s, rows, D, dh_in, d_hdrop, (long long)hdrop_row_stride, (const unsigned char*)mask, scale, dc_inout,
                                gates_act, c_prev, c_new, dgates_pre, (long long)ld_dg, (__nv_bfloat16*)dg16, (long long)ld_dg16,
                                dh_parts, n_parts, parts_rows));
        ICD_LAUNCH_CHECK();
        return 0;
    }
    ICD_CUDA(icd_launch_pdl(ICD_PDL_POINTWISE, lstm_pointwise_bwd_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), (size_t)0, s, rows, D,
                            dh_in, d_hdrop, (long long)hdrop_row_stride, (const unsigned char*)mask, scale, dc_inout, gates_act,
                            c_prev, c_new, dgates_pre, (long long)ld_dg, (__nv_bfloat16*)dg16, (long long)ld_dg16,
                            dh_parts, n_parts, parts_rows));
    ICD_LAUNCH_CHECK();
    return 0;
}

int icd_colsum(const float* X, int64_t ld, int64_t M, int N, const uint8_t* row_mask, float* out, cudaStream_t s) {
    if (N == 0) return 0;
    ICD_CUDA(icd_launch_pdl(ICD_PDL_POINTWISE, colsum_kernel, dim3((unsigned)((N + 31) / 32)), dim3(32, 32), (size_t)0, s, X, (long long)ld,
                            (long long)M, N, (const unsigned char*)row_mask, out));
    ICD_LAUNCH_CHECK();
    return 0;
}

int64_t icd_colsum_bf16_ws_floats(int64_t M, int N) {
    const int64_t chunks = (M + COLSUM16_ROWS - 1) / COLSUM16_ROWS;
    return chunks * N;
}

// out[n] = sum_m mask[m] * X16[m*ld + n] over a tall bf16 matrix; deterministic (fixed chunking, fixed order).
int icd_colsum_bf16(const void* X16, int64_t ld, int64_t M, int N, const uint8_t* row_mask, float* out, float* ws,
                    cudaStream_t s) {
    if (N == 0) return 0;
    ICD_CHECK_ARG(ld % 2 == 0, "colsum_bf16: ld must be even");
    const int rows_per_chunk = COLSUM16_ROWS;
    const int chunks = (int)((M + rows_per_chunk - 1) / rows_per_chunk);
    ICD_CHECK_ARG(chunks <= 65535, "colsum_bf16: too many rows");
    const int vec = (ld % 8 == 0) && ((reinterpret_cast<uintptr_t>(X16) & 15) == 0);
    dim3 grid((N + 1023) / 1024, chunks);
    ICD_CUDA(icd_launch_pdl(ICD_PDL_POINTWISE, colsum_bf16_partial_kernel, grid, dim3(128), (size_t)0, s,
                            reinterpret_cast<const __nv_bfloat16*>(X16), (long long)ld, (long long)M, N, rows_per_chunk,
                            (const unsigned char*)row_mask, ws, vec));
    ICD_LAUNCH_CHECK();
    return icd_colsum(ws, N, chunks, N, nullptr, out, s);
}

int icd_embed_gather(const void* table, int is_f64, const int64_t* captions, int B, int L, int T, int E, int V,
                     float* out, cudaStream_t s) {
    if (B * T == 0) return 0;
    if (is_f64) ICD_CUDA(icd_launch_pdl(ICD_PDL_POINTWISE, embed_gather_kernel<double>, dim3((unsigned)(B * T)), dim3(128), (size_t)0, s,
                                        (const double*)table, (const long long*)captions, B, L, T, E, V, out));
    else        ICD_CUDA(icd_launch_pdl(ICD_PDL_POINTWISE, embed_gather_kernel<float>, dim3((unsigned)(B * T)), dim3(128), (size_t)0, s,
                                        (const float*)table, (const long long*)captions, B, L, T, E, V, out));
    ICD_LAUNCH_CHECK();
    return 0;
}

int64_t icd_embed_scatter_ws_bytes(int B, int T) {
    const int64_t N = (int64_t)B * T;
    const int64_t chunks = (N + EMB_SORT_N - 1) / EMB_SORT_N;
    int64_t n_sort = EMB_SORT_N;
    if (chunks == 1) { n_sort = 32; while (n_sort < N) n_sort <<= 1; }        // one chunk: the next power of two is enough
    return chunks * n_sort * (int64_t)sizeof(unsigned long long);
}

int icd_embed_scatter_add(void* d_table, int is_f64, const int64_t* captions, int B, int L, int T, int E, int V,
                          const int32_t* bt_host, const float* d_x, cudaStream_t s, void* ws, int64_t ws_bytes) {
    if (B * T == 0) return 0;
    ICD_CHECK_ARG(T <= ICD_MAX_STEPS, "embed_scatter_add: T too large");
    BtPack pack;
    for (int t = 0; t < ICD_MAX_STEPS; ++t) pack.v[t] = t < T ? bt_host[t] : 0;
    static const bool atomic_mode = [] { const char* e = getenv("ICD_EMBED_ATOMIC"); return e && e[0] == '1'; }();
    if (!atomic_mode && ws && ws_bytes >= icd_embed_scatter_ws_bytes(B, T) && E <= EMB_MAX_E) {
        // deterministic path: sort (token, row) per chunk of 16384 rows, then segment sums in row order, chunk after chunk
        const long long N = (long long)B * T;
        const int chunks = (int)((N + EMB_SORT_N - 1) / EMB_SORT_N);
        int n_sort = EMB_SORT_N;
        if (chunks == 1) { n_sort = 32; while (n_sort < N) n_sort <<= 1; }
        const size_t smem = (size_t)n_sort * sizeof(unsigned long long);
        static size_t configured = 48 * 1024;
        if (smem > configured) {
            ICD_CUDA(cudaFuncSetAttribute(embed_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            configured = smem;
        }
        unsigned long long* keys = reinterpret_cast<unsigned long long*>(ws);
        embed_sort_kernel<<<chunks, 1024, smem, s>>>((const long long*)captions, B, L, T, V, pack, n_sort, keys);
        ICD_LAUNCH_CHECK();
        for (int c = 0; c < chunks; ++c) {
            const unsigned long long* kc = keys + (size_t)c * EMB_SORT_N;
            const size_t rs = (size_t)8 * E * (is_f64 ? sizeof(double) : sizeof(float));      // <= 64 KB: opted in below
            static size_t red_configured[2] = {48 * 1024, 48 * 1024};
            if (rs > red_configured[is_f64 ? 1 : 0]) {
                if (is_f64) ICD_CUDA(cudaFuncSetAttribute(embed_segment_reduce_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rs));
                else        ICD_CUDA(cudaFuncSetAttribute(embed_segment_reduce_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rs));
                red_configured[is_f64 ? 1 : 0] = rs;
            }
            if (is_f64) embed_segment_reduce_kernel<double><<<n_sort, 256, rs, s>>>(kc, n_sort, d_x, (double*)d_table, E);
            else        embed_segment_reduce_kernel<float><<<n_sort, 256, rs, s>>>(kc, n_sort, d_x, (float*)d_table, E);
            ICD_LAUNCH_CHECK();
        }
        return 0;
    }
    if (is_f64) embed_scatter_add_kernel<double><<<B * T, 128, 0, s>>>((double*)d_table, (const long long*)captions, B, L, T, E, pack, d_x);
    else        embed_scatter_add_kernel<float><<<B * T, 128, 0, s>>>((float*)d_table, (const long long*)captions, B, L, T, E, pack, d_x);
    ICD_LAUNCH_CHECK();
    return 0;
}

extern "C" int icd_dropout_mask(uint8_t* out, int64_t n, float p, uint64_t seed, uint64_t offset, void* stream) {
    if (n <= 0) return 0;
    const long long q = (n + 3) / 4;
    dropout_mask_kernel<<<(unsigned)((q + 255) / 256), 256, 0, icd_stream(stream)>>>(out, n, p, seed, offset);
    ICD_LAUNCH_CHECK();
    return 0;
}

extern "C" int icd_clip_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq,
                                  int64_t n, float grad_scale, float grad_clip, float lr, float beta1, float beta2,
                                  float eps, int32_t step, void* stream) {
    if (n <= 0) return 0;
    ICD_CHECK_ARG(step >= 1, "clip_adam_step: step must be >= 1");
    const double bc1 = 1.0 - pow((double)beta1, (double)step);
    const double bc2 = 1.0 - pow((double)beta2, (double)step);
    long long blocks = (n + 255) / 256;
    if (blocks > ICD_NUM_SMS * 16) blocks = ICD_NUM_SMS * 16;
    clip_adam_kernel<<<(unsigned)blocks, 256, 0, icd_stream(stream)>>>(param, grad, exp_avg, exp_avg_sq, n,
                                                                       grad_scale, grad_clip, lr, beta1, beta2, eps,
                                                                       (float)bc1, (float)sqrt(bc2));
    ICD_LAUNCH_CHECK();
    return 0;
}

extern "C" int icd_cross_entropy_fwd(int64_t R, int V, const float* logits, const int64_t* targets,
                                     float* row_loss, float* lse, void* stream) {
    if (R <= 0) return 0;
    ICD_CHECK_ARG(row_loss && lse, "cross_entropy_fwd: row_loss and lse are required");
    cross_entropy_fwd_kernel<<<(unsigned)R, 256, 0, icd_stream(stream)>>>(V, logits, (const long long*)targets, row_loss, lse);
    ICD_LAUNCH_CHECK();
    return 0;
}

template <bool WEIGHTED>
static int cross_entropy_fwd_grad16(int64_t R, int V, const float* logits, const int64_t* targets, float inv_count,
                                    const float* weights, float* row_loss, float* lse, void* d_logits16, int64_t ld16,
                                    void* stream) {
    ICD_CHECK_ARG(!WEIGHTED || weights, "weighted_cross_entropy_fwd_grad16: weights is null");
    if (R <= 0) return 0;
    ICD_CHECK_ARG(row_loss && lse && d_logits16, "cross_entropy_fwd_grad16: null output");
    ICD_CHECK_ARG(ld16 % 8 == 0 && ld16 >= V && (reinterpret_cast<uintptr_t>(d_logits16) & 15) == 0,
                  "cross_entropy_fwd_grad16: ld16=%lld must be a multiple of 8 and >= V, the gradient 16-byte aligned", (long long)ld16);
    const size_t smem = ((size_t)((V + 3) & ~3) + 4 + 16) * sizeof(float);
    ICD_CHECK_ARG(smem <= 200 * 1024, "cross_entropy_fwd_grad16: V=%d does not fit in shared memory (use the two-kernel path)", V);
    static size_t configured = 48 * 1024;
    if (smem > configured) {
        ICD_CUDA(cudaFuncSetAttribute(cross_entropy_fwd_grad16_kernel<WEIGHTED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = smem;
    }
    cross_entropy_fwd_grad16_kernel<WEIGHTED><<<(unsigned)R, 256, smem, icd_stream(stream)>>>(
        V, logits, (const long long*)targets, inv_count, row_loss, lse, (__nv_bfloat16*)d_logits16, ld16, weights);
    ICD_LAUNCH_CHECK();
    return 0;
}

extern "C" int icd_cross_entropy_fwd_grad16(int64_t R, int V, const float* logits, const int64_t* targets, float inv_count,
                                            float* row_loss, float* lse, void* d_logits16, int64_t ld16, void* stream) {
    return cross_entropy_fwd_grad16<false>(R, V, logits, targets, inv_count, nullptr, row_loss, lse, d_logits16, ld16, stream);
}

extern "C" int icd_weighted_cross_entropy_fwd_grad16(int64_t R, int V, const float* logits, const int64_t* targets,
                                                     float inv_count, const float* weights, float* row_loss, float* lse,
                                                     void* d_logits16, int64_t ld16, void* stream) {
    return cross_entropy_fwd_grad16<true>(R, V, logits, targets, inv_count, weights, row_loss, lse, d_logits16, ld16, stream);
}

extern "C" int icd_scale_bf16_by_device_scalar(void* x16, int64_t n, const float* scale, void* stream) {
    if (n <= 0) return 0;
    ICD_CHECK_ARG(n % 8 == 0 && (reinterpret_cast<uintptr_t>(x16) & 15) == 0 && scale, "scale_bf16: n %% 8 and 16-byte alignment required");
    long long blocks = (n / 8 + 255) / 256;
    if (blocks > ICD_NUM_SMS * 16) blocks = ICD_NUM_SMS * 16;
    scale_bf16_by_device_scalar_kernel<<<(unsigned)blocks, 256, 0, icd_stream(stream)>>>((__nv_bfloat16*)x16, (long long)(n / 8), scale);
    ICD_LAUNCH_CHECK();
    return 0;
}

template <bool WEIGHTED>
static int cross_entropy_bwd(int64_t R, int V, const float* logits, const int64_t* targets, const float* lse,
                             const float* upstream, float inv_count, const float* weights, float* d_logits, void* d_logits16,
                             int64_t ld16, void* stream) {
    ICD_CHECK_ARG(!WEIGHTED || weights, "weighted_cross_entropy_bwd: weights is null");
    if (R <= 0) return 0;
    ICD_CHECK_ARG(!d_logits16 || (ld16 % 8 == 0 && ld16 >= V), "cross_entropy_bwd: ld16=%lld must be a multiple of 8 and >= V", (long long)ld16);
    cross_entropy_bwd_kernel<WEIGHTED><<<(unsigned)R, 256, 0, icd_stream(stream)>>>(
        V, logits, (const long long*)targets, lse, upstream, inv_count, d_logits, (__nv_bfloat16*)d_logits16, ld16, weights);
    ICD_LAUNCH_CHECK();
    return 0;
}

extern "C" int icd_cross_entropy_bwd(int64_t R, int V, const float* logits, const int64_t* targets, const float* lse,
                                     const float* upstream, float inv_count, float* d_logits, void* d_logits16,
                                     int64_t ld16, void* stream) {
    return cross_entropy_bwd<false>(R, V, logits, targets, lse, upstream, inv_count, nullptr, d_logits, d_logits16, ld16, stream);
}

extern "C" int icd_weighted_cross_entropy_bwd(int64_t R, int V, const float* logits, const int64_t* targets, const float* lse,
                                              const float* upstream, float inv_count, const float* weights, float* d_logits,
                                              void* d_logits16, int64_t ld16, void* stream) {
    return cross_entropy_bwd<true>(R, V, logits, targets, lse, upstream, inv_count, weights, d_logits, d_logits16, ld16, stream);
}

// ---- doubly stochastic attention regulariser (models/attention.py:413-414) -------------------------------------------
namespace {
__global__ void __launch_bounds__(256) alpha_reg_fwd_kernel(int T, int P, long long BP, const float* __restrict__ alphas,
                                                            float alpha_c, float inv_bp, float* __restrict__ resid,
                                                            float* __restrict__ partial) {
    __shared__ float s_red[40];
    const long long i = (long long)blockIdx.x * 256 + threadIdx.x;           // i = b*P + p
    float sq = 0.f;
    if (i < BP) {
        const long long b = i / P; const int p = (int)(i % P);
        const float* a = alphas + b * T * P + p;
        float s = 0.f;
        for (int t = 0; t < T; ++t) s += a[(long long)t * P];                // t = 0, 1, ...: torch's sum(dim=1) order per (b,p)
        const float r = alpha_c - s;
        resid[i] = r;
        sq = r * r * inv_bp;
    }
    const float tot = block_sum(sq, s_red);
    if (threadIdx.x == 0) partial[blockIdx.x] = tot;
}
__global__ void __launch_bounds__(256) alpha_reg_bwd_kernel(int T, int P, long long BP, const float* __restrict__ resid,
                                                            const float* __restrict__ upstream, float scale,
                                                            float* __restrict__ d_alphas) {
    const long long n = BP * T;
    const float g = scale * (upstream ? upstream[0] : 1.f);
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
        const long long b = i / ((long long)T * P); const int p = (int)(i % P);
        d_alphas[i] = g * resid[b * P + p];
    }
}
}  // namespace

extern "C" int icd_alpha_regulariser_fwd(int B, int T, int P, const float* alphas, float alpha_c, float* resid,
                                         float* partial, float* reg, void* stream) {
    ICD_CHECK_ARG(B > 0 && T > 0 && P > 0, "alpha_regulariser_fwd: empty shape");
    ICD_CHECK_ARG(alphas && resid && partial && reg, "alpha_regulariser_fwd: null pointer");
    cudaStream_t s = icd_stream(stream);
    const long long BP = (long long)B * P;
    const unsigned blocks = (unsigned)((BP + 255) / 256);
    alpha_reg_fwd_kernel<<<blocks, 256, 0, s>>>(T, P, BP, alphas, alpha_c, 1.f / (float)BP, resid, partial);
    ICD_LAUNCH_CHECK();
    return icd_colsum(partial, 1, (int64_t)blocks, 1, nullptr, reg, s);
}

extern "C" int icd_alpha_regulariser_bwd(int B, int T, int P, const float* resid, const float* upstream, float* d_alphas,
                                         void* stream) {
    ICD_CHECK_ARG(B > 0 && T > 0 && P > 0, "alpha_regulariser_bwd: empty shape");
    ICD_CHECK_ARG(resid && d_alphas, "alpha_regulariser_bwd: null pointer");
    const long long BP = (long long)B * P, n = BP * T;
    long long blocks = (n + 255) / 256;
    if (blocks > ICD_NUM_SMS * 16) blocks = ICD_NUM_SMS * 16;
    alpha_reg_bwd_kernel<<<(unsigned)blocks, 256, 0, icd_stream(stream)>>>(T, P, BP, resid, upstream, -2.f / (float)BP, d_alphas);
    ICD_LAUNCH_CHECK();
    return 0;
}
