// Version / error plumbing of the C ABI (include/icd_b200.h).
#include "common.cuh"
#include <string.h>

static thread_local char g_err[512] = "";

void icd_set_error(const char* fmt, ...) {
    va_list ap; va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

long long g_icd_launches = 0;

// ---- attention-step profiling: cudaEvent pairs recorded on the launching stream ---------------------
namespace {
constexpr int PROF_MAX = 8192;
struct ProfRec { cudaEvent_t a, b; int dir, rows; };
int g_prof_stride = 0;               // 0 = off; n = every n-th attention launch of each direction is timed
int g_prof_seen[2] = {0, 0};
}  // namespace

// Which kernel classes are launched with the programmatic-stream-serialization attribute (bit = ICD_PDL_* class).
unsigned icd_pdl_mask() {
    static const unsigned mask = [] {
        const char* e = getenv("ICD_PDL_MASK");
        // default: contractions, LSTM gate math and split-K reductions start early; the attention-step kernels do NOT —
        // their CTAs would be placed while the previous contraction still holds part of the SMs, and the uneven placement
        // costs the HBM-bound kernel 15-60 us per launch (measured: tools/e2e_diag.py, DESIGN.md)
        return e ? (unsigned)strtoul(e, nullptr, 0) : ((1u << ICD_PDL_GEMM) | (1u << ICD_PDL_POINTWISE) | (1u << ICD_PDL_REDUCE));
    }();
    return mask;
}
// ... and behind which predecessor classes (env ICD_PDL_PRED_MASK); tracks the previous launch of this thread
unsigned icd_pdl_allowed(int cls) {
    static const unsigned pred_mask = [] {
        const char* e = getenv("ICD_PDL_PRED_MASK");
        return e ? (unsigned)strtoul(e, nullptr, 0) : 0xffffffffu;
    }();
    static thread_local int last_cls = -1;
    unsigned ok = ((icd_pdl_mask() >> cls) & 1u) && (last_cls < 0 || ((pred_mask >> last_cls) & 1u));
    if (cls == ICD_PDL_GEMM_LATE) ok = (icd_pdl_mask() >> ICD_PDL_GEMM) & 1u;
    // an attention-step grid may be STAGED behind a contraction that keeps its dependents back until its last CTA has exited:
    // every SM is free when the grid is placed (no uneven placement), and the launch latency hides behind the contraction
    if ((cls == ICD_PDL_ATT_FWD || cls == ICD_PDL_ATT_BWD) && last_cls == ICD_PDL_GEMM_LATE) ok = 1u;
    last_cls = cls;
    return ok;
}

namespace { thread_local int g_late_hint = 0; }
void icd_gemm_next_feeds_attention() {
    static const bool on = [] { const char* e = getenv("ICD_PDL_LATE"); return !e || e[0] != '0'; }();
    g_late_hint = on ? 1 : 0;
}
int icd_gemm_take_late_hint() { const int h = g_late_hint; g_late_hint = 0; return h; }

namespace {
ProfRec g_prof[PROF_MAX];
int g_prof_n = 0, g_prof_created = 0;
bool g_prof_open = false;
}

void icd_prof_mark_begin(int dir, int rows, cudaStream_t s) {
    g_prof_open = false;
    if (g_prof_stride <= 0 || g_prof_n >= PROF_MAX) return;
    if (g_prof_seen[dir & 1]++ % g_prof_stride != 0) return;
    if (g_prof_n >= g_prof_created) {
        if (cudaEventCreate(&g_prof[g_prof_n].a) != cudaSuccess || cudaEventCreate(&g_prof[g_prof_n].b) != cudaSuccess) return;
        g_prof_created = g_prof_n + 1;
    }
    g_prof[g_prof_n].dir = dir; g_prof[g_prof_n].rows = rows;
    cudaEventRecord(g_prof[g_prof_n].a, s);
    g_prof_open = true;
}

void icd_prof_mark_end(int dir, cudaStream_t s) {
    (void)dir;
    if (!g_prof_open) return;
    cudaEventRecord(g_prof[g_prof_n].b, s);
    ++g_prof_n;
    g_prof_open = false;
}

extern "C" {
int64_t icd_launch_count(void) { return (int64_t)g_icd_launches; }

int icd_prof_enable(int on) {
    g_prof_stride = on > 0 ? on : 0; g_prof_seen[0] = g_prof_seen[1] = 0;
    if (!on) g_prof_n = 0;
    return 0;
}

int icd_prof_collect(double* fwd_ms, int64_t* fwd_launches, int64_t* fwd_rows,
                     double* bwd_ms, int64_t* bwd_launches, int64_t* bwd_rows) {
    double ms[2] = {0, 0}; int64_t n[2] = {0, 0}, rows[2] = {0, 0};
    for (int i = 0; i < g_prof_n; ++i) {
        cudaError_t e = cudaEventSynchronize(g_prof[i].b);
        if (e != cudaSuccess) { icd_set_error("prof_collect: %s", cudaGetErrorString(e)); g_prof_n = 0; return (int)e; }
        float t = 0.f;
        e = cudaEventElapsedTime(&t, g_prof[i].a, g_prof[i].b);
        if (e != cudaSuccess) { icd_set_error("prof_collect: %s", cudaGetErrorString(e)); g_prof_n = 0; return (int)e; }
        ms[g_prof[i].dir] += t; n[g_prof[i].dir] += 1; rows[g_prof[i].dir] += g_prof[i].rows;
    }
    g_prof_n = 0;
    if (fwd_ms) *fwd_ms = ms[0]; if (fwd_launches) *fwd_launches = n[0]; if (fwd_rows) *fwd_rows = rows[0];
    if (bwd_ms) *bwd_ms = ms[1]; if (bwd_launches) *bwd_launches = n[1]; if (bwd_rows) *bwd_rows = rows[1];
    return 0;
}

int icd_version(void) { return ICD_B200_ABI_VERSION; }
const char* icd_last_error_string(void) { return g_err; }
int icd_sizeof_att_desc(void) { return (int)sizeof(icd_att_desc_t); }
int icd_sizeof_base_desc(void) { return (int)sizeof(icd_base_desc_t); }
int icd_sizeof_beam_desc(void) { return (int)sizeof(icd_beam_desc_t); }
int icd_sizeof_base_beam_desc(void) { return (int)sizeof(icd_base_beam_desc_t); }
int icd_sizeof_sample_desc(void) { return (int)sizeof(icd_sample_desc_t); }
int icd_sizeof_base_sample_desc(void) { return (int)sizeof(icd_base_sample_desc_t); }
int icd_sizeof_att_index(void) { return (int)sizeof(icd_att_index_t); }
}
