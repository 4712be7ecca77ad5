// Shared helpers for libicd_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include "../../include/icd_b200.h"

#ifndef ICD_NUM_SMS
#define ICD_NUM_SMS 148          // B200: 2 dies x 74 SMs
#endif

void icd_set_error(const char* fmt, ...);

#define ICD_CHECK_ARG(cond, ...)                         \
    do { if (!(cond)) { icd_set_error(__VA_ARGS__); return -1; } } while (0)

#define ICD_CUDA(call)                                                                 \
    do { cudaError_t e_ = (call); if (e_ != cudaSuccess) {                             \
        icd_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
        (void)cudaGetLastError();   /* consumed: a refused launch is not reported again by a later call */ \
        return (int)e_; } } while (0)

extern long long g_icd_launches;      // api.cu: kernels launched by this library (bench.py reports it)
#define ICD_LAUNCH_CHECK()  do { ++g_icd_launches; ICD_CUDA(cudaGetLastError()); } while (0)

#define ICD_TRY(call) do { int r_ = (call); if (r_ != 0) return r_; } while (0)

static inline cudaStream_t icd_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

#ifdef __CUDACC__
// kernel classes for the programmatic-dependent-launch policy (bit index into icd_pdl_mask())
enum { ICD_PDL_GEMM = 0, ICD_PDL_ATT_FWD = 1, ICD_PDL_ATT_BWD = 2, ICD_PDL_POINTWISE = 3, ICD_PDL_REDUCE = 4,
       ICD_PDL_GEMM_LATE = 5 };      // a contraction that does NOT release its dependents early (they start when its last CTA exits)
void icd_gemm_next_feeds_attention();   // api.cu: the next contraction of this thread is followed by an attention-step launch
int icd_gemm_take_late_hint();          // api.cu: consumes the hint (1 once, then 0)
unsigned icd_pdl_mask();             // api.cu: which classes may start early (env ICD_PDL_MASK overrides the default)
unsigned icd_pdl_allowed(int cls);   // api.cu: 1 if a launch of class `cls` may start early behind the previous launch

// launch with the programmatic-stream-serialization attribute (see pdl_trigger / pdl_wait below)
template <typename... KArgs, typename... Args>
static inline cudaError_t icd_launch_pdl(int cls, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s,
                                         Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = icd_pdl_allowed(cls);
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
// the same, as thread-block clusters of `cluster_x` CTAs (grid.x must be a multiple of cluster_x)
template <typename... KArgs, typename... Args>
static inline cudaError_t icd_launch_pdl_cluster(int cls, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                                                 cudaStream_t s, unsigned cluster_x, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = icd_pdl_allowed(cls);
    attr[1].id = cudaLaunchAttributeClusterDimension;
    attr[1].val.clusterDim.x = cluster_x; attr[1].val.clusterDim.y = 1; attr[1].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 2;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
#endif

// ---- device helpers -------------------------------------------------------------------------
__device__ __forceinline__ float4 ld_stream_f4(const float* p) {
    // streaming 128-bit load: read-only path, do not allocate in L1 (each byte is used once per CTA)
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}

__device__ __forceinline__ float2 ld_stream_f2(const float2* p) {
    float2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
    return r;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// block-wide reductions for blockDim.x <= 1024 (multiple of 32); scratch: >= 33 floats of smem.
__device__ __forceinline__ float block_sum(float v, float* scratch) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_sum(v);
    __syncthreads();                 // protect scratch reuse
    if (lane == 0) scratch[w] = v;
    __syncthreads();
    float r = (threadIdx.x < nw) ? scratch[threadIdx.x] : 0.f;
    if (w == 0) { r = warp_sum(r); if (lane == 0) scratch[32] = r; }
    __syncthreads();
    return scratch[32];
}
__device__ __forceinline__ float block_max(float v, float* scratch) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_max(v);
    __syncthreads();
    if (lane == 0) scratch[w] = v;
    __syncthreads();
    float r = (threadIdx.x < nw) ? scratch[threadIdx.x] : -INFINITY;
    if (w == 0) { r = warp_max(r); if (lane == 0) scratch[32] = r; }
    __syncthreads();
    return scratch[32];
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

// Philox4x32-10 counter-based generator (Salmon et al. 2011): ten rounds on the counter c under the key (k0, k1), in place.
// Dropout's keep masks (pointwise.cu) and the caption sampler's Gumbel noise (sample.cu) draw from it.
__device__ __forceinline__ void philox4x32_10(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
        c[0] = hi1 ^ c[1] ^ k0; c[1] = lo1; c[2] = hi0 ^ c[3] ^ k1; c[3] = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}

// ---- programmatic dependent launch (PDL) ----------------------------------------------------------------
// The kernels of the per-time-step chain (contraction -> attention step -> contraction -> LSTM gate math) are short and
// strictly dependent; launched with cudaLaunchAttributeProgrammaticStreamSerialization the next kernel's CTAs become
// resident, run their prologue (barrier init, TMEM allocation, tensor-map prefetch) and then block in pdl_wait() until
// the previous grid has completed and flushed — launch latency and prologue leave the critical path.  Every kernel of
// the chain executes pdl_trigger() at its top and pdl_wait() before its first dependent global access (reads of
// upstream results AND writes: a buffer the previous kernel still reads must not be overwritten early).  Because every
// kernel triggers at its top, the part of a grid before pdl_wait() may overlap ANY earlier kernel of the unbroken chain of
// early-launched kernels, not only the one in front of it: before the wait, read only what was complete when the chain
// started (e.g. forward activations in a backward pass).
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// attention-step profiling hooks (api.cu)
void icd_prof_mark_begin(int dir, int rows, cudaStream_t s);
void icd_prof_mark_end(int dir, cudaStream_t s);

// ---- internal (non-exported) launchers shared between translation units -----------------------
int icd_colsum(const float* X, int64_t ld, int64_t M, int N, const uint8_t* row_mask, float* out, cudaStream_t s);
int64_t icd_colsum_bf16_ws_floats(int64_t M, int N);
int icd_colsum_bf16(const void* X16, int64_t ld, int64_t M, int N, const uint8_t* row_mask, float* out, float* ws,
                    cudaStream_t s);
int icd_embed_gather(const void* table, int is_f64, const int64_t* captions, int B, int L, int T, int E, int V,
                     float* out /* (T,B,E) */, cudaStream_t s);
// d_table (V,E) += rows of d_x scattered by token id.  With a workspace of icd_embed_scatter_ws_bytes(B, T) bytes the sum
// is DETERMINISTIC (rows sorted by (token, row), one CTA per token adds them in row order); without it (or with
// ICD_EMBED_ATOMIC=1) atomics accumulate in arrival order.
int64_t icd_embed_scatter_ws_bytes(int B, int T);
int icd_embed_scatter_add(void* d_table, int is_f64, const int64_t* captions, int B, int L, int T, int E, int V,
                          const int32_t* bt_host, const float* d_x /* (T,B,E) */, cudaStream_t s,
                          void* ws = nullptr, int64_t ws_bytes = 0);
int icd_lstm_pointwise_fwd(int rows, int D, const float* gates_pre, const float* c_prev,
                           float* gates_act, float* c_new, float* h_new,
                           float* hdrop, int64_t hdrop_row_stride, const uint8_t* mask, float scale,
                           cudaStream_t s, void* h16 = nullptr, void* hdrop16 = nullptr,
                           const int* m_live = nullptr /* optional device-side row count */);
int icd_lstm_pointwise_bwd(int rows, int D, const float* dh_in, const float* d_hdrop, int64_t hdrop_row_stride,
                           const uint8_t* mask, float scale, float* dc_inout,
                           const float* gates_act, const float* c_prev, const float* c_new,
                           float* dgates_pre, int64_t ld_dg, cudaStream_t s, void* dg16 = nullptr, int64_t ld_dg16 = 0,
                           const float* dh_parts = nullptr, int n_parts = 0, int parts_rows = 0);   // deferred split-K planes of dh
int icd_weighted_pixel_sum(int rows, int P, int C, const int32_t* img_index, const float* enc,
                           const float* alpha, int64_t ld_alpha, const float* fbeta_pre, int64_t ld_fb,
                           float* awe_raw, float* gate, float* gated, cudaStream_t s,
                           const int32_t* out_row_ptr = nullptr, const int32_t* out_rows = nullptr);
// ---- captions that share images (icd_att_index_t): the step backward with an image index, and the per-image reductions ----
int icd_attention_step_bwd_idx(int rows, int P, int C, int A, const int32_t* img_index, const float* enc, const float* att_enc,
                               const float* att_dec, int64_t ld_dec, const float* w_full, const float* alpha, int64_t ld_alpha,
                               const float* d_alpha_ext, int64_t ld_dalpha, const float* gate, const float* awe_raw,
                               const float* d_gated, float* d_att_dec, int64_t ld_ddec, float* d_fbeta_pre, int64_t ld_dfb,
                               float* d_e, int64_t ld_de, float* d_awe_out, void* stream);
int icd_attention_step_bwd_bf16_idx(int rows, int P, int C, int A, const int32_t* img_index, const void* enc16,
                                    const void* att_enc16, const float* att_dec, int64_t ld_dec, const float* w_full,
                                    const float* alpha, int64_t ld_alpha, const float* d_alpha_ext, int64_t ld_dalpha,
                                    const float* gate, const float* awe_raw, const float* d_gated, float* d_att_dec,
                                    int64_t ld_ddec, float* d_fbeta_pre, int64_t ld_dfb, float* d_e, int64_t ld_de,
                                    void* dz16, int64_t ld_dz16, float* d_awe_out, void* stream);
int icd_attention_proj_bwd_indexed(int B, int n_img, int T, int P, int A, const int32_t* bt_host, const int32_t* row_ptr,
                                   const int32_t* rows, const float* att_enc, const float* att_dec_all, int64_t ld_dec,
                                   const float* w_full, const float* d_e, float* d_att_enc, float* d_w_full, float* d_b_full,
                                   float* d_b_enc, float* partial, cudaStream_t s);
int icd_attention_proj_bwd_bf16_indexed(int B, int n_img, int T, int P, int A, const int32_t* bt_host, const int32_t* row_ptr,
                                        const int32_t* rows, const void* att_enc16, const float* att_dec_all, int64_t ld_dec,
                                        const float* w_full, const float* d_e, void* d_att_enc16, float* d_w_full,
                                        float* d_b_full, float* d_b_enc, float* partial, const float* d_att_dec_all,
                                        int64_t ld_ddec, cudaStream_t s);
int icd_attention_enc_grad_indexed(int B, int n_img, int T, int P, int C, const int32_t* bt_host, const int32_t* row_ptr,
                                   const int32_t* rows, const float* alphas, const float* d_awe_all, const float* d_mean,
                                   float* d_enc, int32_t* row_len_ws, cudaStream_t s);
int icd_attention_step_fwd_grouped(int n_img, int k, int P, int C, int A, const int* k_live, const float* enc,
                                   const float* att_enc, const float* att_dec, int64_t ld_dec, const float* w_full,
                                   const float* b_full, const float* fbeta_pre, int64_t ld_fb, float* alpha,
                                   int64_t ld_alpha, float* gated, const int* slot_img /* slot -> image, or NULL */,
                                   const int* n_slots /* device: live slots, or NULL */,
                                   const int* row_off /* slot -> first state row, or NULL (slot*k) */, cudaStream_t s,
                                   void* gated_x3 = nullptr /* optional: 3-term bf16 split of gated, rows of 6*C (gemm_tc.cu A layout) */,
                                   int* ticket = nullptr /* optional: ONE zeroed device int per launch: the ring kernel's CTAs draw slots dynamically */,
                                   int x3_nseg = 6 /* layout of gated_x3: 6 K-concatenated segments, or 3 stored planes (gemm_tc.cuh) */);
void icd_gemm_simple_set_ws(void* ws, int64_t bytes);
// ICD_PREC_FP32X3: the 3-term bf16 split of an operand that stays constant during one entry-point call (a weight matrix read by
// every step of the time loop) is made ONCE and kept in a cache region at the tail of the caller's arena.  Only operands whose
// base pointer was marked are cached (activation buffers are rewritten in place between steps); the cache dies with the scope.
void icd_x3_cache_begin(void* mem, int64_t bytes);
void icd_x3_cache_end();
void icd_x3_cache_mark(const float* base);
void* icd_x3_cache_lookup(const float* p, int64_t stride, int mn, int K, int mn_major, int seg, int which, int64_t bytes, bool* fresh);
inline int64_t icd_x3_split_bytes(int64_t mn, int64_t K) {          // == the operand regions of icd_gemm_x3_ws_bytes
    const int64_t b = ((mn + 7) / 8 * 8) * 6 * ((K + 7) / 8 * 8) * 2;
    return (b + 255) / 256 * 256;
}
struct IcdSimpleWsScope {          // RAII: workspace for icd_gemm_simple's tensor-core tiers during one entry-point call
    IcdSimpleWsScope(void* ws, int64_t bytes, int64_t cache_bytes = 0) {
        if (cache_bytes > 0 && ws && bytes > cache_bytes) {
            icd_gemm_simple_set_ws(ws, bytes - cache_bytes);
            icd_x3_cache_begin(reinterpret_cast<char*>(ws) + (bytes - cache_bytes), cache_bytes);
        } else
            icd_gemm_simple_set_ws(ws, bytes);
    }
    ~IcdSimpleWsScope() { icd_gemm_simple_set_ws(nullptr, 0); icd_x3_cache_end(); }
};
int icd_gemm_simple(int prec, const float* A, int64_t sam, int64_t sak, const float* B, int64_t sbn, int64_t sbk,
                    float* C, int64_t ldc, int M, int N, int K, const float* bias1, const float* bias2,
                    const float* add1, int64_t ld1, const float* add2, int64_t ld2, const uint8_t* row_mask,
                    float beta, cudaStream_t s, int flags = 0);
