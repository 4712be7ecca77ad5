// K8 — the recurrent part of the baseline LSTM decoder (nn.LSTM, models/baseline.py:106) as ONE persistent kernel per
// direction, driven by a grid barrier instead of a launch chain (SURVEY.md 2.3 row `baseline.py:106`, 7.1 step 6).
//
// Forward, step t:   gates = h_{t-1} W_hh^T + xg_t   (xg = x W_ih^T + b_ih + b_hh, hoisted over all steps by the caller)
//                    i,f,g,o -> c_t = f c_{t-1} + i g,  h_t = o tanh(c_t)          (gate order i,f,g,o)
// Backward, step t:  dh_t = dg_{t+1} W_hh + d_hout_t ;  LSTM cell adjoint -> dg_t, dc_{t-1}
//
// Decomposition (weight-stationary — it pays here because the per-step activation is only B x H):
//   * the grid is H/4 CTAs: forward, 4 hidden units = 16 gate columns each; backward, clusters of 4 CTAs own 16 hidden units and
//     each rank contracts a quarter of the 4H-long K dimension (partial sums exchanged through distributed shared memory);
//     a CTA keeps ITS slice of W_hh (16 rows of the B operand x K, bf16, 128B-swizzled K-major UMMA tiles) in shared memory
//     for all L steps — converted from the fp32 weight once, by the kernel itself;
//   * per step the whole CTA grid streams the same small A operand (h_{t-1} or dg_{t+1}, bf16, B x K) through a TMA ring and
//     issues tcgen05.mma (M = 128 rows per tile, N = 16, K = 16 per instruction) into a TMEM accumulator;
//   * the epilogue warps read the accumulator (tcgen05.ld), apply the LSTM cell math for their row and write the new state —
//     including the bf16 copy that is the NEXT step's A operand — straight to global memory;
//   * steps are separated by a grid-wide barrier (one atomic counter; cooperative launch guarantees co-residency), with the
//     generic->async proxy fences the TMA reads of freshly written rows require.
// No per-step launches, no gates_pre round trip, no separate gate-math kernel.
#include "common.cuh"
#include "gemm_tc.cuh"
#include "tc_common.cuh"
#include <cstdlib>

namespace {

constexpr int LP_THREADS = 192;           // warp 0: TMA producer + grid barrier, warp 1: TMEM alloc + MMA issue, warps 2-5: epilogue
constexpr int LP_BM = 128;
constexpr int LP_N = 16;                  // accumulator columns per CTA
constexpr int LP_A_BYTES = LP_BM * TC_BK * 2;       // 16 KB per stage
constexpr int LP_W_KB_BYTES = LP_N * TC_BK * 2;     // 2 KB of the resident weight slice per k-block
constexpr int LP_TMEM_COLS = 64;          // up to 4 row tiles of 16 columns
constexpr int LP_MAX_MT = LP_TMEM_COLS / LP_N;
// cute::UMMA::InstrDescriptor: c F32, a/b BF16, both K-major, N = 16, M = 128
constexpr uint32_t LP_IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(LP_N >> 3) << 17) | ((uint32_t)(LP_BM >> 4) << 24);

struct LstmSeqArgs {
    int B, L, H, K, nkb, stages;
    const float* w_hh;                    // (4H, H) fp32
    // forward
    const float* xg;                      // (L,B,4H)
    float* gates_act;                     // (L,B,4H)
    float* c_all;                         // (L+1,B,H)
    float* h_all;                         // (L+1,B,H)
    float* hout;                          // (B,L,H)
    __nv_bfloat16* h16;                   // ((L+1)*B, H): row block t = h_t, the A operand of step t
    __nv_bfloat16* hout16;                // (B*L, H)
    // backward
    const float* d_hout;                  // (B,L,H)
    float* dc;                            // (B,H) running cell-state gradient (zero on entry)
    float* dg;                            // (L,B,4H)
    __nv_bfloat16* dg16;                  // (L*B, 4H): row block t = dg_t, the A operand of step t-1
    unsigned int* bar;                    // grid barrier counter (zero on entry)
};

__device__ __forceinline__ void tc_ld_32x32b_x16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 "
                 "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ uint32_t lp_mapa(uint32_t addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// byte offset of element (n, k) of the resident weight slice: k-blocks of 16 rows x 128 B, 8-row swizzle atoms of 1024 B,
// 16-byte chunk index XOR row-in-atom (the SWIZZLE_128B pattern the UMMA descriptor expects of a K-major tile)
__device__ __forceinline__ uint32_t w_slice_off(int n, int k) {
    const int kb = k >> 6, kk = k & 63;
    return (uint32_t)(kb * LP_W_KB_BYTES + (n >> 3) * 1024 + (n & 7) * 128 + (((kk >> 3) ^ (n & 7)) << 4) + (kk & 7) * 2);
}

__device__ __forceinline__ void grid_arrive(unsigned int* bar) {
    __threadfence();
    atomicAdd(bar, 1u);
}
__device__ __forceinline__ void grid_wait(const unsigned int* bar, unsigned int target) {
    unsigned int v;
    unsigned long long spins = 0;
    while (true) {
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(bar) : "memory");
        if (v >= target) break;
        if (++spins > (1ull << 26)) __trap();          // a lost CTA must fault, never hang the GPU
    }
    __threadfence();
}

__device__ __forceinline__ uint2 pack4_bf16(float a, float b, float c, float d) {
    const __nv_bfloat162 lo = __floats2bfloat162_rn(a, b), hi = __floats2bfloat162_rn(c, d);
    uint2 pk;
    pk.x = *reinterpret_cast<const uint32_t*>(&lo); pk.y = *reinterpret_cast<const uint32_t*>(&hi);
    return pk;
}

struct Cell4 { float4 a, b, c, d, e, f, g, h; };          // the per-row operands of one 4-unit LSTM cell update

// operands of the forward cell update of (row, units u0..u0+3) at step t: xg_i, xg_f, xg_g, xg_o, c_{t-1}
__device__ __forceinline__ void cell_fwd_load(const LstmSeqArgs& p, int t, int row, int u0, Cell4& o) {
    const size_t g_off = ((size_t)t * p.B + row) * 4 * p.H + u0;
    o.a = *reinterpret_cast<const float4*>(p.xg + g_off);
    o.b = *reinterpret_cast<const float4*>(p.xg + g_off + p.H);
    o.c = *reinterpret_cast<const float4*>(p.xg + g_off + 2 * p.H);
    o.d = *reinterpret_cast<const float4*>(p.xg + g_off + 3 * p.H);
    o.e = *reinterpret_cast<const float4*>(p.c_all + ((size_t)t * p.B + row) * p.H + u0);
}
// hh: h_{t-1} W_hh^T for the 4 units, [gate][unit]
__device__ __forceinline__ void cell_fwd_apply(const LstmSeqArgs& p, int t, int row, int u0, const Cell4& o, const float (&hh)[16]) {
    const int H = p.H, B = p.B, L = p.L;
    const size_t g_off = ((size_t)t * B + row) * 4 * H + u0;
    const size_t s_off = (size_t)row * H + u0;
    const size_t BH = (size_t)B * H;
    const float xi_[4] = {o.a.x, o.a.y, o.a.z, o.a.w}, xf_[4] = {o.b.x, o.b.y, o.b.z, o.b.w};
    const float xc_[4] = {o.c.x, o.c.y, o.c.z, o.c.w}, xo_[4] = {o.d.x, o.d.y, o.d.z, o.d.w};
    const float cp_[4] = {o.e.x, o.e.y, o.e.z, o.e.w};
    float gi[4], gf[4], gg[4], go[4], cn[4], hn[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        gi[u] = sigmoidf_(hh[u] + xi_[u]);
        gf[u] = sigmoidf_(hh[4 + u] + xf_[u]);
        gg[u] = tanhf(hh[8 + u] + xc_[u]);
        go[u] = sigmoidf_(hh[12 + u] + xo_[u]);
        cn[u] = gf[u] * cp_[u] + gi[u] * gg[u];
        hn[u] = go[u] * tanhf(cn[u]);
    }
    *reinterpret_cast<float4*>(p.gates_act + g_off) = make_float4(gi[0], gi[1], gi[2], gi[3]);
    *reinterpret_cast<float4*>(p.gates_act + g_off + H) = make_float4(gf[0], gf[1], gf[2], gf[3]);
    *reinterpret_cast<float4*>(p.gates_act + g_off + 2 * H) = make_float4(gg[0], gg[1], gg[2], gg[3]);
    *reinterpret_cast<float4*>(p.gates_act + g_off + 3 * H) = make_float4(go[0], go[1], go[2], go[3]);
    *reinterpret_cast<float4*>(p.c_all + (size_t)(t + 1) * BH + s_off) = make_float4(cn[0], cn[1], cn[2], cn[3]);
    const float4 h4 = make_float4(hn[0], hn[1], hn[2], hn[3]);
    *reinterpret_cast<float4*>(p.h_all + (size_t)(t + 1) * BH + s_off) = h4;
    const uint2 hb = pack4_bf16(hn[0], hn[1], hn[2], hn[3]);
    *reinterpret_cast<uint2*>(p.h16 + (size_t)(t + 1) * BH + s_off) = hb;                    // next step's A operand
    const size_t o_off = ((size_t)row * L + t) * H + u0;
    *reinterpret_cast<float4*>(p.hout + o_off) = h4;
    if (p.hout16) *reinterpret_cast<uint2*>(p.hout16 + o_off) = hb;
}
// operands of the backward cell update: d_hout, gates i f g o, c_{t-1}, c_t, dc
__device__ __forceinline__ void cell_bwd_load(const LstmSeqArgs& p, int t, int row, int u0, Cell4& o) {
    const size_t g_off = ((size_t)t * p.B + row) * 4 * p.H + u0;
    const size_t s_off = (size_t)row * p.H + u0;
    const size_t BH = (size_t)p.B * p.H;
    o.a = *reinterpret_cast<const float4*>(p.d_hout + ((size_t)row * p.L + t) * p.H + u0);
    o.b = *reinterpret_cast<const float4*>(p.gates_act + g_off);
    o.c = *reinterpret_cast<const float4*>(p.gates_act + g_off + p.H);
    o.d = *reinterpret_cast<const float4*>(p.gates_act + g_off + 2 * p.H);
    o.e = *reinterpret_cast<const float4*>(p.gates_act + g_off + 3 * p.H);
    o.f = *reinterpret_cast<const float4*>(p.c_all + (size_t)t * BH + s_off);
    o.g = *reinterpret_cast<const float4*>(p.c_all + (size_t)(t + 1) * BH + s_off);
    o.h = *reinterpret_cast<const float4*>(p.dc + s_off);
}
__device__ __forceinline__ void cell_bwd_apply(const LstmSeqArgs& p, int t, int row, int u0, const Cell4& o, const float (&dhh)[4]) {
    const int H = p.H;
    const size_t g_off = ((size_t)t * p.B + row) * 4 * H + u0;
    const size_t s_off = (size_t)row * H + u0;
    const float dh_[4] = {dhh[0] + o.a.x, dhh[1] + o.a.y, dhh[2] + o.a.z, dhh[3] + o.a.w};
    const float i_[4] = {o.b.x, o.b.y, o.b.z, o.b.w}, f_[4] = {o.c.x, o.c.y, o.c.z, o.c.w};
    const float g_[4] = {o.d.x, o.d.y, o.d.z, o.d.w}, o_[4] = {o.e.x, o.e.y, o.e.z, o.e.w};
    const float cp_[4] = {o.f.x, o.f.y, o.f.z, o.f.w}, cn_[4] = {o.g.x, o.g.y, o.g.z, o.g.w};
    const float dc_[4] = {o.h.x, o.h.y, o.h.z, o.h.w};
    float pi[4], pf[4], pg[4], po[4], dcn[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const float tc = tanhf(cn_[u]);
        const float d_o = dh_[u] * tc;
        const float dc = dc_[u] + dh_[u] * o_[u] * (1.f - tc * tc);
        const float d_i = dc * g_[u], d_g = dc * i_[u], d_f = dc * cp_[u];
        dcn[u] = dc * f_[u];
        pi[u] = d_i * i_[u] * (1.f - i_[u]); pf[u] = d_f * f_[u] * (1.f - f_[u]);
        pg[u] = d_g * (1.f - g_[u] * g_[u]); po[u] = d_o * o_[u] * (1.f - o_[u]);
    }
    *reinterpret_cast<float4*>(p.dc + s_off) = make_float4(dcn[0], dcn[1], dcn[2], dcn[3]);
    *reinterpret_cast<float4*>(p.dg + g_off) = make_float4(pi[0], pi[1], pi[2], pi[3]);
    *reinterpret_cast<float4*>(p.dg + g_off + H) = make_float4(pf[0], pf[1], pf[2], pf[3]);
    *reinterpret_cast<float4*>(p.dg + g_off + 2 * H) = make_float4(pg[0], pg[1], pg[2], pg[3]);
    *reinterpret_cast<float4*>(p.dg + g_off + 3 * H) = make_float4(po[0], po[1], po[2], po[3]);
    *reinterpret_cast<uint2*>(p.dg16 + g_off) = pack4_bf16(pi[0], pi[1], pi[2], pi[3]);      // next step's A operand
    *reinterpret_cast<uint2*>(p.dg16 + g_off + H) = pack4_bf16(pf[0], pf[1], pf[2], pf[3]);
    *reinterpret_cast<uint2*>(p.dg16 + g_off + 2 * H) = pack4_bf16(pg[0], pg[1], pg[2], pg[3]);
    *reinterpret_cast<uint2*>(p.dg16 + g_off + 3 * H) = pack4_bf16(po[0], po[1], po[2], po[3]);
}

// BWD = 0: forward recurrence.  CTA c owns hidden units [4c, 4c+4): accumulator column n = gate * 4 + unit, K = H.
// BWD = 1: backward recurrence.  Clusters of 4 CTAs: cluster i accumulates dh for hidden units [16i, 16i+16) (column n = unit);
//          CTA rank q of the cluster contracts the K-slice [qH, (q+1)H) of dg (= gate q) — a quarter of the operand stream per
//          SM — then the four partial sums are exchanged through distributed shared memory (rank q sends columns 4j..4j+3 to
//          rank j) and rank j finishes units [16i + 4j, 16i + 4j + 4): summed in rank order, so the result is deterministic.
template <int BWD>
__global__ void __launch_bounds__(LP_THREADS, 1)
lstm_seq_kernel(const __grid_constant__ CUtensorMap tmA, const LstmSeqArgs p) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* gbase = smem_raw + (base - smem_u32(smem_raw));
    const int S = p.stages;
    const uint32_t sA = base;                                          // S stages x 16 KB
    const uint32_t sW = base + (uint32_t)S * LP_A_BYTES;               // nkb x 2 KB, resident
    uint8_t* gW = gbase + (size_t)S * LP_A_BYTES;
    const uint32_t bars = sW + (uint32_t)p.nkb * LP_W_KB_BYTES;
    const uint32_t full0 = bars, empty0 = bars + 8 * S, tfull = bars + 16 * S, tempty = tfull + 8;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(gW + (size_t)p.nkb * LP_W_KB_BYTES + 16 * S + 16);
    const uint32_t sRed = bars + 256;                                  // BWD: [MT][4 source ranks][128 rows] float4
    float4* gRed = reinterpret_cast<float4*>(gW + (size_t)p.nkb * LP_W_KB_BYTES + 256);

    const int warp = (int)uniform_u32(threadIdx.x >> 5), lane = threadIdx.x & 31;
    const int B = p.B, L = p.L, H = p.H, K = p.K;
    const int MT = (B + LP_BM - 1) / LP_BM;
    const uint32_t crank = BWD ? cluster_ctarank() : 0u;
    const int unit0 = BWD ? (int)(blockIdx.x / 4) * 16 : (int)blockIdx.x * 4;      // first unit of the accumulator columns
    const int k0 = BWD ? (int)crank * K : 0;                                       // first column of this CTA's K-slice of A
    const int my_u0 = BWD ? unit0 + 4 * (int)crank : unit0;                        // the 4 units this CTA finishes
    const unsigned int NC = gridDim.x;

    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" :: "l"(&tmA) : "memory");
        for (int i = 0; i < S; ++i) { mbar_init(full0 + 8 * i, 1); mbar_init(empty0 + 8 * i, 1); }
        mbar_init(tfull, 1); mbar_init(tempty, 4);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     :: "r"(smem_u32(tmem_slot)), "r"((uint32_t)LP_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    // resident weight slice, fp32 -> bf16, written in the swizzled UMMA layout (zero beyond K)
    {
        const int Kpad = p.nkb * TC_BK;
        for (int idx = threadIdx.x; idx < LP_N * Kpad; idx += LP_THREADS) {
            int n, k;
            float v = 0.f;
            if (!BWD) {                                    // B(n, k) = W_hh[gate * H + unit0 + u][k],  n = gate * 4 + u
                n = idx / Kpad; k = idx % Kpad;
                if (k < K) v = p.w_hh[(size_t)((n >> 2) * H + unit0 + (n & 3)) * H + k];
            } else {                                       // B(n, k) = W_hh[k0 + k][unit0 + n]   (dh = dg W_hh)
                k = idx / LP_N; n = idx % LP_N;
                if (k < K) v = p.w_hh[(size_t)(k0 + k) * H + unit0 + n];
            }
            *reinterpret_cast<__nv_bfloat16*>(gW + w_slice_off(n, k)) = __float2bfloat16_rn(v);
        }
    }
    fence_proxy_async_smem();                              // generic-proxy smem writes -> visible to the tensor core (async proxy)
    tc_fence_before();
    __syncthreads();
    if (BWD) cluster_sync_all();                           // peers' shared memory is live before any remote store targets it
    tc_fence_after();
    const uint32_t tmem_base = uniform_u32(*tmem_slot);

    int stage = 0; uint32_t phase = 0;                     // A ring (producer and MMA warps keep their own copies)
    uint32_t acc_phase = 0;                                // accumulator hand-off (MMA and epilogue warps)

    for (int it = 0; it < L; ++it) {
        const int t = BWD ? (L - 1 - it) : it;
        const bool has_gemm = it > 0;                      // forward: h_0 = 0; backward: no dh flows in from beyond the last step
        const int a_row0 = (BWD ? (t + 1) : t) * B;        // first row of this step's A operand (h_t resp. dg_{t+1})
        Cell4 ops;                                         // epilogue warps: cell operands of the first row tile, fetched early
        if (warp == 0) {
            // =================================== TMA producer + grid barrier ===================================
            // (whole warp in uniform control flow, one elected lane issues: tc_common.cuh elect_one)
            if (has_gemm) {
                if (lane == 0) grid_wait(p.bar, NC * (unsigned int)it);   // every CTA has published its rows of iteration it-1
                __syncwarp();
                fence_proxy_async_all();                       // ... and the async proxy (TMA) may now read them
                for (int mt = 0; mt < MT; ++mt)
                    for (int kb = 0; kb < p.nkb; ++kb) {
                        mbar_wait(empty0 + 8 * stage, phase ^ 1);
                        if (elect_one()) {
                            mbar_arrive_expect_tx(full0 + 8 * stage, LP_A_BYTES);
                            tma_load_2d(sA + stage * LP_A_BYTES, &tmA, k0 + kb * TC_BK, a_row0 + mt * LP_BM, full0 + 8 * stage);
                        }
                        __syncwarp();
                        if (++stage == S) { stage = 0; phase ^= 1; }
                    }
            }
        } else if (warp == 1) {
            // =================================== MMA issuer ===================================
            if (has_gemm) {
                mbar_wait(tempty, acc_phase ^ 1);          // the epilogue has drained the previous step's accumulator
                tc_fence_after();
                for (int mt = 0; mt < MT; ++mt)
                    for (int kb = 0; kb < p.nkb; ++kb) {
                        mbar_wait(full0 + 8 * stage, phase);
                        tc_fence_after();
                        if (elect_one()) {
                            const uint64_t adesc = make_smem_desc(sA + stage * LP_A_BYTES, 0);
                            const uint64_t bdesc = make_smem_desc(sW + kb * LP_W_KB_BYTES, 0);
#pragma unroll
                            for (int k = 0; k < TC_BK / 16; ++k)
                                tc_mma_f16(tmem_base + (uint32_t)(mt * LP_N), adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k),
                                           LP_IDESC, (kb > 0 || k > 0) ? 1u : 0u);
                            tc_commit(empty0 + 8 * stage);
                            if (mt == MT - 1 && kb == p.nkb - 1) tc_commit(tfull);
                        }
                        __syncwarp();
                        if (++stage == S) { stage = 0; phase ^= 1; }
                    }
                acc_phase ^= 1;
            }
        } else {
            // =================================== epilogue: LSTM cell math, warps 2..5 ===================================
            const int q = warp & 3;                        // TMEM lane quarter this warp may access
            const int r0 = q * 32 + lane;                  // row inside a 128-row tile
            if (r0 < B) {                                  // fetched while the contraction runs
                if (BWD) cell_bwd_load(p, t, r0, my_u0, ops); else cell_fwd_load(p, t, r0, my_u0, ops);
            }
            if (has_gemm) {
                mbar_wait(tfull, acc_phase);
                tc_fence_after();
                acc_phase ^= 1;
            }
            if (!BWD) {
                for (int mt = 0; mt < MT; ++mt) {
                    const int row = mt * LP_BM + r0;
                    float hh[16];
                    if (has_gemm) {
                        uint32_t v[16];
                        tc_ld_32x32b_x16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(mt * LP_N), v);
                        tc_wait_ld();
#pragma unroll
                        for (int j = 0; j < 16; ++j) hh[j] = __uint_as_float(v[j]);
                    } else {
#pragma unroll
                        for (int j = 0; j < 16; ++j) hh[j] = 0.f;
                    }
                    if (has_gemm && mt == MT - 1) {        // all TMEM reads of this warp are done: hand the accumulator back
                        tc_fence_before();
                        if (lane == 0) mbar_arrive(tempty);
                    }
                    if (row >= B) continue;
                    if (mt > 0) cell_fwd_load(p, t, row, my_u0, ops);
                    cell_fwd_apply(p, t, row, my_u0, ops, hh);
                }
            } else {
                if (has_gemm) {
                    // partial sums of this K-slice -> the rank that finishes each group of 4 units (distributed shared memory)
                    for (int mt = 0; mt < MT; ++mt) {
                        uint32_t v[16];
                        tc_ld_32x32b_x16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(mt * LP_N), v);
                        tc_wait_ld();
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const uint32_t local = sRed + (uint32_t)(((mt * 4 + (int)crank) * LP_BM + r0) * 16);
                            const uint32_t remote = lp_mapa(local, (uint32_t)j);
                            asm volatile("st.shared::cluster.v4.b32 [%0], {%1, %2, %3, %4};"
                                         :: "r"(remote), "r"(v[4 * j]), "r"(v[4 * j + 1]), "r"(v[4 * j + 2]), "r"(v[4 * j + 3]) : "memory");
                        }
                    }
                    tc_fence_before();
                    if (lane == 0) mbar_arrive(tempty);
                }
            }
        }
        if (BWD) {
            __syncwarp();
            if (has_gemm) cluster_sync_all();              // every rank's partial sums have landed (release / acquire)
            if (warp >= 2) {
                const int q = warp & 3, r0 = q * 32 + lane;
                for (int mt = 0; mt < MT; ++mt) {
                    const int row = mt * LP_BM + r0;
                    if (row >= B) continue;
                    float dhh[4] = {0.f, 0.f, 0.f, 0.f};
                    if (has_gemm) {
#pragma unroll
                        for (int src = 0; src < 4; ++src) {                       // fixed order: deterministic
                            const float4 x = gRed[(mt * 4 + src) * LP_BM + r0];
                            dhh[0] += x.x; dhh[1] += x.y; dhh[2] += x.z; dhh[3] += x.w;
                        }
                    }
                    if (mt > 0) cell_bwd_load(p, t, row, my_u0, ops);
                    cell_bwd_apply(p, t, row, my_u0, ops, dhh);
                }
            }
        }
        if (warp >= 2) fence_proxy_async_all();            // the rows just written are read by other CTAs' TMA in the next step
        __syncthreads();
        if (threadIdx.x == 0 && it + 1 < L) grid_arrive(p.bar);
    }

    tc_fence_before();
    __syncthreads();
    if (BWD) cluster_sync_all();                           // no rank exits while a peer could still address its shared memory
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"((uint32_t)LP_TMEM_COLS) : "memory");
    }
}

int plan_smem(int nkb, int red_bytes, int* stages) {
    // resident weight slice + barriers (+ the backward's exchange buffer) + as many 16 KB A stages as fit (2..8)
    const int fixed = 1024 + nkb * LP_W_KB_BYTES + 256 + red_bytes;
    int s = (200 * 1024 - fixed) / LP_A_BYTES;
    if (s > 8) s = 8;
    *stages = s;
    return fixed + s * LP_A_BYTES;
}

int g_bwd_launch_mode = 0;      // 0 = not launched yet, 1 = cooperative + cluster launch accepted, 2 = plain cluster launch

bool persistent_enabled() {
    static const bool on = [] { const char* e = getenv("ICD_LSTM_PERSISTENT"); return !(e && e[0] == '0'); }();
    return on;
}

// dynamic shared memory of one CTA for B rows and hidden size H (the backward adds the DSMEM exchange buffer); 0 if fewer
// than 2 A stages fit beside the resident weight slice
int seq_smem(int BWD, int B, int H, int* stages) {
    const int MT = (B + LP_BM - 1) / LP_BM;
    const int smem = plan_smem((H + TC_BK - 1) / TC_BK, BWD ? MT * 4 * LP_BM * 16 : 0, stages);
    return *stages >= 2 ? smem : 0;
}

// raise the kernel's dynamic-shared-memory limit to at least smem (never lowers it: other shapes may be in flight)
template <int BWD>
cudaError_t ensure_smem_attr(int smem) {
    static int smem_set = 0;
    if (smem_set >= smem) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(lstm_seq_kernel<BWD>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess) smem_set = smem;
    return e;
}

// the pure shape rules: whole 16-unit groups, one forward CTA per SM at most, every row tile's accumulator in the TMEM
// allocation, at least 2 A stages beside the resident weight slice
bool shape_ok(int B, int L, int H) {
    if (B < 1 || L < 1 || H < 16 || H % 16 != 0) return false;
    if (H / 4 > ICD_NUM_SMS) return false;
    if ((B + LP_BM - 1) / LP_BM > LP_MAX_MT) return false;
    int st;
    return seq_smem(1, B, H, &st) > 0;
}

// Co-residency, read from the occupancy calculator at the shared memory each direction launches with: the forward grid
// (H/4 CTAs) needs blocks-per-SM x SMs >= H/4, the backward (H/16 clusters of 4) needs as many co-resident 4-CTA clusters.
// Clusters cannot span GPCs, so the second answer is not implied by the first.  Launches nothing.
// -> 0 and the two capacities, or -1 if a query failed (its error is consumed).
int query_residency(int B, int H, int* fwd_ctas, int* bwd_clusters) {
    *fwd_ctas = 0; *bwd_clusters = 0;
    int st, dev = 0, sms = 0, per_sm = 0;
    const int smem_f = seq_smem(0, B, H, &st), smem_b = seq_smem(1, B, H, &st);
    if (!smem_f || !smem_b) return 0;
    bool ok = cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess &&
              ensure_smem_attr<0>(smem_f) == cudaSuccess && ensure_smem_attr<1>(smem_b) == cudaSuccess &&
              cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, lstm_seq_kernel<0>, LP_THREADS, (size_t)smem_f) == cudaSuccess;
    if (ok) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(H / 4); cfg.blockDim = dim3(LP_THREADS); cfg.dynamicSmemBytes = (size_t)smem_b;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = 4; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        ok = cudaOccupancyMaxActiveClusters(bwd_clusters, lstm_seq_kernel<1>, &cfg) == cudaSuccess;
    }
    if (!ok) { (void)cudaGetLastError(); *bwd_clusters = 0; return -1; }
    *fwd_ctas = per_sm * sms;
    return 0;
}

// 1 if both grids of (B, H) are co-resident; cached per shape class (row tiles, H): the answer depends on nothing else.
// A failed query refuses the shape.
bool resident(int B, int H) {
    static signed char cache[LP_MAX_MT + 1][ICD_NUM_SMS / 4 + 1] = {};     // 0 unknown, 1 fits, -1 refused
    signed char& c = cache[(B + LP_BM - 1) / LP_BM][H / 16];
    if (c == 0) {
        int f, b;
        c = (query_residency(B, H, &f, &b) == 0 && f >= H / 4 && b >= H / 16) ? 1 : -1;
    }
    return c == 1;
}

// A16: the bf16 activation stack [a_rows][a_cols] the per-step A operands are cut from (a.K = this CTA's contraction length)
template <int BWD>
int launch_seq(const LstmSeqArgs& a0, const __nv_bfloat16* A16, int a_rows, int a_cols, cudaStream_t s) {
    LstmSeqArgs a = a0;
    a.nkb = (a.K + TC_BK - 1) / TC_BK;
    const int smem = seq_smem(BWD, a.B, a.H, &a.stages);
    ICD_CHECK_ARG(smem > 0, "lstm_seq: hidden size %d too large for the resident weight slice", a.H);
    CUtensorMap tmA;
    ICD_TRY(make_tmap(&tmA, A16, a_cols, a_rows, a_cols, LP_BM, 0));
    ICD_CUDA(ensure_smem_attr<BWD>(smem));
    ICD_CUDA(cudaMemsetAsync(a.bar, 0, sizeof(unsigned int), s));
    const int grid = a.H / 4;                              // forward: 4 units per CTA; backward: 16 units per 4-CTA cluster
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(LP_THREADS); cfg.dynamicSmemBytes = (size_t)smem; cfg.stream = s;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeCooperative;           // every CTA co-resident, or the launch fails: the grid barrier cannot hang
    attr[0].val.cooperative = 1;
    attr[1].id = cudaLaunchAttributeClusterDimension;
    attr[1].val.clusterDim.x = 4; attr[1].val.clusterDim.y = 1; attr[1].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = BWD ? 2 : 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, lstm_seq_kernel<BWD>, tmA, a);
    if (BWD && e == cudaSuccess) g_bwd_launch_mode = 1;
    if (e != cudaSuccess && BWD && resident(a.B, a.H)) {
        // a driver that refuses cooperative + cluster launches: the occupancy query said every cluster of this grid is
        // co-resident on an idle device, so the grid barrier completes once the stream's earlier work has drained; the
        // barrier's spin limit turns a violation into a fault, not a hang
        (void)cudaGetLastError();
        cfg.attrs = attr + 1; cfg.numAttrs = 1;
        e = cudaLaunchKernelEx(&cfg, lstm_seq_kernel<BWD>, tmA, a);
        if (e == cudaSuccess) g_bwd_launch_mode = 2;
    }
    ICD_CUDA(e);
    ICD_LAUNCH_CHECK();
    return 0;
}

}  // namespace

// 1 if the persistent kernels cover this shape (else the caller keeps its launch chain): the pure shape rules first, then
// co-residency of both directions' grids as the occupancy calculator reports it for this device (the grid barrier needs
// every CTA resident at once).
int icd_lstm_seq_persistent_ok(int B, int L, int H) {
    if (!persistent_enabled()) return 0;
    return shape_ok(B, L, H) && resident(B, H) ? 1 : 0;
}

int icd_lstm_seq_fwd_persistent(int B, int L, int H, const float* w_hh, const float* xg, float* gates_act, float* c_all,
                                float* h_all, float* hout, void* h16, void* hout16, unsigned int* bar, cudaStream_t s) {
    ICD_CHECK_ARG(icd_lstm_seq_persistent_ok(B, L, H), "lstm_seq_fwd: shape B=%d L=%d H=%d not covered by the persistent kernel", B, L, H);
    LstmSeqArgs a = {};
    a.B = B; a.L = L; a.H = H; a.K = H; a.w_hh = w_hh; a.xg = xg; a.gates_act = gates_act; a.c_all = c_all; a.h_all = h_all;
    a.hout = hout; a.h16 = reinterpret_cast<__nv_bfloat16*>(h16); a.hout16 = reinterpret_cast<__nv_bfloat16*>(hout16); a.bar = bar;
    return launch_seq<0>(a, a.h16, (L + 1) * B, H, s);
}

int icd_lstm_seq_bwd_persistent(int B, int L, int H, const float* w_hh, const float* d_hout, const float* gates_act,
                                const float* c_all, float* dc, float* dg, void* dg16, unsigned int* bar, cudaStream_t s) {
    ICD_CHECK_ARG(icd_lstm_seq_persistent_ok(B, L, H), "lstm_seq_bwd: shape B=%d L=%d H=%d not covered by the persistent kernel", B, L, H);
    LstmSeqArgs a = {};
    a.B = B; a.L = L; a.H = H; a.K = H; a.w_hh = w_hh; a.d_hout = d_hout;      // K: one rank's slice of the 4H-long contraction
    a.gates_act = const_cast<float*>(gates_act);
    a.c_all = const_cast<float*>(c_all); a.dc = dc; a.dg = dg; a.dg16 = reinterpret_cast<__nv_bfloat16*>(dg16); a.bar = bar;
    return launch_seq<1>(a, a.dg16, L * B, 4 * H, s);
}

// ---- C ABI (include/icd_b200.h): the LSTM recurrence on its own, for callers that hoist the input contraction themselves ----
extern "C" int icd_lstm_seq_supported(int B, int L, int H) { return icd_lstm_seq_persistent_ok(B, L, H); }
extern "C" int icd_lstm_seq_shape_ok(int B, int L, int H) { return shape_ok(B, L, H) ? 1 : 0; }
extern "C" int icd_lstm_seq_residency(int B, int H, int* fwd_ctas, int* bwd_clusters) {
    ICD_CHECK_ARG(fwd_ctas && bwd_clusters, "lstm_seq_residency: null output");
    ICD_CHECK_ARG(shape_ok(B, 1, H), "lstm_seq_residency: shape B=%d H=%d fails the shape rules", B, H);
    ICD_CHECK_ARG(query_residency(B, H, fwd_ctas, bwd_clusters) == 0, "lstm_seq_residency: occupancy query failed");
    return 0;
}
extern "C" int icd_lstm_seq_bwd_launch_mode(void) { return g_bwd_launch_mode; }

extern "C" int icd_lstm_seq_fwd(int B, int L, int H, const float* w_hh, const float* xg, float* gates_act, float* c_all,
                                float* h_all, float* hout, void* h16, void* hout16, void* barrier_ws, void* stream) {
    cudaStream_t s = icd_stream(stream);
    const size_t BH = (size_t)B * H;
    ICD_CUDA(cudaMemsetAsync(c_all, 0, sizeof(float) * BH, s));                    // zero (h0, c0): nn.LSTM default state
    ICD_CUDA(cudaMemsetAsync(h_all, 0, sizeof(float) * BH, s));
    ICD_CUDA(cudaMemsetAsync(h16, 0, 2 * BH, s));
    return icd_lstm_seq_fwd_persistent(B, L, H, w_hh, xg, gates_act, c_all, h_all, hout, h16, hout16,
                                       reinterpret_cast<unsigned int*>(barrier_ws), s);
}

extern "C" int icd_lstm_seq_bwd(int B, int L, int H, const float* w_hh, const float* d_hout, const float* gates_act,
                                const float* c_all, float* dc_ws, float* dg, void* dg16, void* barrier_ws, void* stream) {
    cudaStream_t s = icd_stream(stream);
    ICD_CUDA(cudaMemsetAsync(dc_ws, 0, sizeof(float) * (size_t)B * H, s));
    return icd_lstm_seq_bwd_persistent(B, L, H, w_hh, d_hout, gates_act, c_all, dc_ws, dg, dg16,
                                       reinterpret_cast<unsigned int*>(barrier_ws), s);
}
