// capi.cu -- error plumbing and the per-stage device timers of the C-ABI (include/imsegm_b200.h)
#include "common.cuh"
#include <stdarg.h>
#include <vector>

static thread_local char g_err[512] = "";
long long g_isb_launches = 0;

void isb_set_error(const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char* isb_last_error(void) { return g_err; }
extern "C" int isb_abi_version(void) { return 6; }  // 6: predict_proba of a given mixture model (isb_gmm_predict); 5: banded Leung-Malik statistics (accumulate / finish), tcgen05 issue-rate probe; 4: tcgen05 operand layout (w_tc), UMMA self-test, graph replay accounting, segment median
extern "C" long long isb_launch_count(void) { return g_isb_launches; }
extern "C" int isb_note_graph_replay(long long n_kernels) { g_isb_launches += n_kernels; return ISB_OK; }

// ---- stage timers: CUDA events recorded on the launching stream around a kernel (or a family of kernels) ----
struct ProfRec { cudaEvent_t a, b; int id; };
static int g_prof_on = 0;
static std::vector<ProfRec> g_recs;
static std::vector<cudaEvent_t> g_free;

static cudaEvent_t prof_event()
{
    if (!g_free.empty()) { cudaEvent_t e = g_free.back(); g_free.pop_back(); return e; }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}

int isb_prof_begin(int id, cudaStream_t st)
{
    if (!g_prof_on) return -1;
    ProfRec r; r.a = prof_event(); r.b = prof_event(); r.id = id;
    cudaEventRecord(r.a, st);
    g_recs.push_back(r);
    return (int)g_recs.size() - 1;
}

void isb_prof_end(int handle, cudaStream_t st)
{
    if (handle < 0 || handle >= (int)g_recs.size()) return;
    cudaEventRecord(g_recs[handle].b, st);
}

extern "C" int isb_profile_enable(int on)
{
    g_prof_on = on;
    return ISB_OK;
}

extern "C" int isb_profile_stage_count(void) { return ISB_PROF_COUNT; }

extern "C" const char* isb_profile_stage_name(int id)
{
    static const char* names[ISB_PROF_COUNT] = { "slic_prepare", "slic_assign", "slic_update", "slic_finalize_bin", "slic_connectivity",
                                                 "segment_stats", "adjacency", "gc_energies", "alpha_expansion", "gather", "gmm", "lm_texture" };
    return (id >= 0 && id < ISB_PROF_COUNT) ? names[id] : "";
}

extern "C" int isb_profile_collect(double* ms_out, long long* count_out)
{
    for (int i = 0; i < ISB_PROF_COUNT; ++i) { ms_out[i] = 0.0; count_out[i] = 0; }
    for (auto& r : g_recs) {
        cudaError_t e = cudaEventSynchronize(r.b);
        float ms = 0.f;
        if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, r.a, r.b);
        if (e != cudaSuccess) { isb_set_error("profile collect: %s", cudaGetErrorString(e)); return ISB_ERR_CUDA; }
        ms_out[r.id] += ms;
        count_out[r.id] += 1;
        g_free.push_back(r.a);
        g_free.push_back(r.b);
    }
    g_recs.clear();
    return ISB_OK;
}
