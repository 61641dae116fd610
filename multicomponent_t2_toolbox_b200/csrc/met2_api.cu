// met2_api.cu — error state, launch accounting, test hooks and diagnostics of the C ABI (include/met2.h).
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>

#include "met2_host.h"

namespace met2 {

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

int set_error(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(MET2_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
    return MET2_OK;
}

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

int sm_count() {
    // per-device table: a host thread that drives several GPUs (pipeline.MultiGpuFit) alternates devices on every call,
    // and cudaGetDeviceProperties costs milliseconds (measured: 3.2 ms per met2_fa_fit / met2_t2_fit call with a
    // one-entry cache, 0.1 ms with the table)
    static std::atomic<int> table[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 0;
    if (dev >= 0 && dev < 64) {
        const int c = table[dev].load(std::memory_order_relaxed);
        if (c > 0) return c;
    }
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
    if (dev >= 0 && dev < 64) table[dev].store(n, std::memory_order_relaxed);
    return n;
}

Overrides read_overrides() {
    Overrides o;
    const char* ev = getenv("MET2_T2_WARPS");
    o.t2_warps = ev ? atoi(ev) : 0;
    ev = getenv("MET2_T2_TILE");
    o.t2_tile = ev ? atoi(ev) : 0;
    ev = getenv("MET2_LCURVE_SWITCH");
    o.lcurve_switch_set = ev != nullptr;
    o.lcurve_switch = ev ? atof(ev) : 0.0;
    ev = getenv("MET2_FA_SEARCH");
    o.fa_search_warp = ev && ev[0] == 'w';
    ev = getenv("MET2_FA_THREAD_PCAP");
    o.fa_thread_pcap_set = ev != nullptr;
    o.fa_thread_pcap = ev ? atoi(ev) : 0;
    return o;
}

}  // namespace met2

extern "C" const char* met2_last_error(void) { return met2::g_err; }
extern "C" int met2_version(void) { return MET2_VERSION; }
extern "C" int met2_echo_rank(int small) { return small ? MET2_ECHO_RANK_SMALL : MET2_ECHO_RANK; }
extern "C" int64_t met2_launch_count(void) { return (int64_t)met2::g_launches.load(); }
