// Library-level state of libbdetr: error text, compute mode, launch counter.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <mutex>
#include "kernels.cuh"

namespace bdetr {
static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};
static std::atomic<int> g_mode{BDETR_MODE_FP32};
static std::atomic<int> g_attn_f16{0};       // BDETR_MODE_FP16 = tensor-core mode + fp16 attention operands
static std::atomic<int> g_pdl{1};
bool pdl_enabled() { return g_pdl.load(std::memory_order_relaxed) != 0; }

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
static thread_local int t_mode_override = -1;
int current_mode() { return t_mode_override >= 0 ? t_mode_override : g_mode.load(std::memory_order_relaxed); }
ModeScope::ModeScope(int mode) : saved(t_mode_override) { t_mode_override = mode; }
ModeScope::~ModeScope() { t_mode_override = saved; }
bool attention_f16_enabled() { return g_attn_f16.load(std::memory_order_relaxed) != 0; }

// ---- auxiliary stream pool (per device) ---------------------------------------------------------------------
static std::atomic<int> g_conc{1};
bool concurrency_enabled() { return g_conc.load(std::memory_order_relaxed) != 0; }
constexpr int AUX_GROUPS = 32, AUX_PER_GROUP = 3, AUX_STREAMS = AUX_GROUPS * AUX_PER_GROUP, MAX_DEVICES = 16;
static std::atomic<int> g_defer{0};
struct AuxPool {
    int pending[AUX_GROUPS] = {0};      // per group: aux streams with deferred (not yet joined) work
    bool ready = false;
    cudaStream_t st[AUX_STREAMS];
    cudaEvent_t fork_ev[AUX_STREAMS], join_ev[AUX_STREAMS];
    cudaStream_t owner[AUX_GROUPS];      // caller stream each group of three auxiliary streams is bound to
    int owners = 0, next = 0;
};
static AuxPool g_pools[MAX_DEVICES];
static std::mutex g_pool_mu;

static AuxPool *pool_for_current_device()
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MAX_DEVICES) return nullptr;
    AuxPool &p = g_pools[dev];
    std::lock_guard<std::mutex> lk(g_pool_mu);
    if (!p.ready) {
        for (int i = 0; i < AUX_STREAMS; ++i) {
            if (cudaStreamCreateWithFlags(&p.st[i], cudaStreamNonBlocking) != cudaSuccess) return nullptr;
            if (cudaEventCreateWithFlags(&p.fork_ev[i], cudaEventDisableTiming) != cudaSuccess) return nullptr;
            if (cudaEventCreateWithFlags(&p.join_ev[i], cudaEventDisableTiming) != cudaSuccess) return nullptr;
        }
        p.ready = true;
    }
    return &p;
}

Branches::Branches(cudaStream_t main_stream) : main(main_stream), base(0), used(0), rc(BDETR_OK), on(concurrency_enabled()), shared(false)
{
    if (!on) return;
    AuxPool *p = pool_for_current_device();
    if (!p) { on = false; return; }
    // Each caller stream gets its own group of auxiliary streams, so entry points issued from different caller
    // streams (the model runs encoder / decoder / head chains side by side) never queue behind each other.
    std::lock_guard<std::mutex> lk(g_pool_mu);
    int g = -1;
    for (int i = 0; i < p->owners; ++i) if (p->owner[i] == main_stream) { g = i; break; }
    if (g < 0) {
        if (p->owners < AUX_GROUPS) { g = p->owners++; }
        else { g = p->next; p->next = (p->next + 1) % AUX_GROUPS; shared = true; }       // more caller streams than groups: share
        if (!shared) p->owner[g] = main_stream;
    }
    base = g * AUX_PER_GROUP;
}

cudaStream_t Branches::fork(int i)
{
    if (!on) return main;
    AuxPool *p = pool_for_current_device();
    const int k = base + i;
    if (cudaEventRecord(p->fork_ev[k], main) != cudaSuccess || cudaStreamWaitEvent(p->st[k], p->fork_ev[k], 0) != cudaSuccess) {
        set_error("Branches::fork: %s", cudaGetErrorString(cudaGetLastError()));
        rc = BDETR_E_CUDA;
        return main;
    }
    used |= 1 << i;
    return p->st[k];
}

// Parameter-gradient side chains (weight gradients, bias / positional gradients) are only consumed at the end of the
// step (optimizer / gradient all-reduce).  With bdetr_set_deferred_join(1) an entry point does not wait for them before
// it returns: they keep running on their auxiliary streams and the CALLER orders its stream after them with
// bdetr_join(stream) before it reads the gradients.  Everything else is joined inside the call as usual.
int Branches::join_deferrable()
{
    if (!on) return rc;
    if (g_defer.load(std::memory_order_relaxed) == 0 || shared) return join();      // (a shared group cannot track deferred work per caller)
    AuxPool *p = pool_for_current_device();
    std::lock_guard<std::mutex> lk(g_pool_mu);
    p->pending[base / AUX_PER_GROUP] |= used;
    used = 0;
    return rc;
}

int join_pending(cudaStream_t main_stream, cudaStream_t waiter)
{
    if (!concurrency_enabled()) return BDETR_OK;
    AuxPool *p = pool_for_current_device();
    if (!p) return BDETR_OK;
    int g = -1, mask = 0;
    {
        std::lock_guard<std::mutex> lk(g_pool_mu);
        for (int i = 0; i < p->owners; ++i) if (p->owner[i] == main_stream) { g = i; break; }
        if (g < 0) return BDETR_OK;
        mask = p->pending[g];
        p->pending[g] = 0;
    }
    for (int i = 0; i < AUX_PER_GROUP; ++i) {
        if (!(mask & (1 << i))) continue;
        const int k = g * AUX_PER_GROUP + i;
        if (cudaEventRecord(p->join_ev[k], p->st[k]) != cudaSuccess || cudaStreamWaitEvent(waiter, p->join_ev[k], 0) != cudaSuccess) {
            set_error("bdetr_join: %s", cudaGetErrorString(cudaGetLastError()));
            return BDETR_E_CUDA;
        }
    }
    return BDETR_OK;
}

int Branches::join()
{
    if (!on) return rc;
    AuxPool *p = pool_for_current_device();
    for (int i = 0; i < 3; ++i) {
        if (!(used & (1 << i))) continue;
        const int k = base + i;
        if (cudaEventRecord(p->join_ev[k], p->st[k]) != cudaSuccess || cudaStreamWaitEvent(main, p->join_ev[k], 0) != cudaSuccess) {
            set_error("Branches::join: %s", cudaGetErrorString(cudaGetLastError()));
            rc = BDETR_E_CUDA;
        }
    }
    used = 0;
    return rc;
}
}  // namespace bdetr

extern "C" __attribute__((visibility("default"))) int bdetr_set_concurrency(int on) { bdetr::g_conc.store(on ? 1 : 0); return BDETR_OK; }
extern "C" __attribute__((visibility("default"))) int bdetr_get_concurrency(void) { return bdetr::g_conc.load(); }
extern "C" __attribute__((visibility("default"))) int bdetr_set_deferred_join(int on) { bdetr::g_defer.store(on ? 1 : 0); return BDETR_OK; }
extern "C" __attribute__((visibility("default"))) int bdetr_join(void *stream) { return bdetr::join_pending(reinterpret_cast<cudaStream_t>(stream), reinterpret_cast<cudaStream_t>(stream)); }
extern "C" __attribute__((visibility("default"))) int bdetr_join_into(void *stream, void *waiter) { return bdetr::join_pending(reinterpret_cast<cudaStream_t>(stream), reinterpret_cast<cudaStream_t>(waiter)); }
extern "C" __attribute__((visibility("default"))) int bdetr_version(void) { return 105; }
extern "C" __attribute__((visibility("default"))) const char *bdetr_last_error(void) { return bdetr::g_err; }
extern "C" __attribute__((visibility("default"))) int bdetr_set_mode(int mode)
{
    if (mode != BDETR_MODE_FP32 && mode != BDETR_MODE_TF32 && mode != BDETR_MODE_FP16) {
        bdetr::set_error("bdetr_set_mode: unknown mode %d", mode);
        return BDETR_E_UNSUPPORTED;
    }
    // internally the fp16 mode IS the tensor-core mode (every `mode == TF32` dispatch holds) plus the operand switch
    bdetr::g_mode.store(mode == BDETR_MODE_FP16 ? BDETR_MODE_TF32 : mode);
    bdetr::g_attn_f16.store(mode == BDETR_MODE_FP16 ? 1 : 0);
    return BDETR_OK;
}
extern "C" __attribute__((visibility("default"))) int bdetr_get_mode(void) { return bdetr::g_attn_f16.load() ? BDETR_MODE_FP16 : bdetr::g_mode.load(); }
extern "C" __attribute__((visibility("default"))) long long bdetr_launch_count(void) { return bdetr::g_launches.load(); }
extern "C" __attribute__((visibility("default"))) void bdetr_reset_launch_count(void) { bdetr::g_launches.store(0); }
extern "C" __attribute__((visibility("default"))) int bdetr_set_pdl(int on) { bdetr::g_pdl.store(on ? 1 : 0); return BDETR_OK; }
extern "C" __attribute__((visibility("default"))) int bdetr_get_pdl(void) { return bdetr::g_pdl.load(); }
