// Process-level entry points of the C ABI: error state, device check.
#include "mms_common.cuh"
#include <string.h>

namespace mms {

static thread_local char g_error[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
    set_error("%s failed: %s (%s:%d)", what, cudaGetErrorString(e), file, line);
    return MMS_E_CUDA;
}

}  // namespace mms

using namespace mms;

extern "C" int mms_version(void) { return 104; }

extern "C" const char* mms_last_error(void) { return g_error; }

extern "C" int mms_init(int device) {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        set_error("no CUDA device is visible (%s); libmms_b200 has no CPU fallback", cudaGetErrorString(e));
        return MMS_E_ARCH;
    }
    MMS_REQUIRE(device >= 0 && device < count, "device %d outside [0,%d)", device, count);
    cudaDeviceProp prop;
    MMS_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        set_error("device %d is sm_%d%d; libmms_b200 is built for sm_100a (B200) only and has no fallback", device, prop.major,
                  prop.minor);
        return MMS_E_ARCH;
    }
    MMS_CUDA(cudaSetDevice(device));
    return MMS_OK;
}

// ---- launch counter + opt-in per-kernel event timer -------------------------------------------
#include <atomic>
#include <map>
#include <string>
#include <vector>

namespace mms {

static std::atomic<long long> g_launches{0};
static bool g_prof_on = false;
struct ProfRec { const char* name; cudaEvent_t a, b; };
static std::vector<ProfRec> g_recs;
static thread_local cudaStream_t tl_stream = nullptr;
static thread_local cudaEvent_t tl_begin = nullptr;

// ---- in-graph timeline (diagnostic, mms_timeline_enable): every launch is bracketed by two one-thread kernels that write
// %globaltimer into a device buffer, on the launch's own stream.  Unlike the event profile above this also works under
// CUDA-graph capture (the stamps become graph nodes and every replay overwrites the buffer), so it shows what the kernels
// of the main chain and of the side streams cost WHILE they overlap.  The stamps add ~2 launches of latency per kernel:
// read overlaps and relative stretch from it, not absolute step times.
constexpr int TL_MAX = 1024;
static bool g_tl_on = false;
static unsigned long long* g_tl_buf = nullptr;          // [TL_MAX][2] start / end, device
struct TlRec { const char* name; cudaStream_t stream; };
static std::vector<TlRec> g_tl_recs;
static thread_local int tl_idx = -1;

__global__ void timeline_stamp_kernel(unsigned long long* slot) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    *slot = t;
}

void prof_begin(cudaStream_t st) {
    tl_stream = st;
    if (g_tl_on) {
        tl_idx = -1;
        if ((int)g_tl_recs.size() < TL_MAX) {
            tl_idx = (int)g_tl_recs.size();
            g_tl_recs.push_back({"?", st});
            timeline_stamp_kernel<<<1, 1, 0, st>>>(g_tl_buf + 2 * tl_idx);
        }
    }
    if (!g_prof_on) return;
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) return;
    if (cudaEventCreate(&tl_begin) != cudaSuccess) { tl_begin = nullptr; return; }
    cudaEventRecord(tl_begin, st);
}

void prof_end(const char* name) {
    g_launches.fetch_add(1, std::memory_order_relaxed);
    if (g_tl_on && tl_idx >= 0) {
        g_tl_recs[tl_idx].name = name;
        timeline_stamp_kernel<<<1, 1, 0, tl_stream>>>(g_tl_buf + 2 * tl_idx + 1);
        tl_idx = -1;
    }
    if (!g_prof_on || !tl_begin) return;
    ProfRec r;
    r.name = name;
    r.a = tl_begin;
    tl_begin = nullptr;
    if (cudaEventCreate(&r.b) != cudaSuccess) { cudaEventDestroy(r.a); return; }
    cudaEventRecord(r.b, tl_stream);
    g_recs.push_back(r);
}

}  // namespace mms

// ---- run-time switches ------------------------------------------------------------------------
#include <mutex>
#include <stdlib.h>

namespace mms {

static std::mutex g_opt_mu;
struct OptVal { bool set; int v; };
static std::map<std::string, OptVal> g_opt;     // explicit settings and cached environment reads (set = false: neither)

int option_get(const char* name, int dflt) {
    std::lock_guard<std::mutex> lk(g_opt_mu);
    auto it = g_opt.find(name);
    if (it == g_opt.end()) {
        OptVal o = {false, 0};
        const std::string env = std::string("MMS_") + name;
        if (const char* e = getenv(env.c_str())) { if (e[0]) { o.set = true; o.v = atoi(e); } }
        it = g_opt.emplace(name, o).first;
    }
    return it->second.set ? it->second.v : dflt;      // the default belongs to the caller and is never cached
}

}  // namespace mms

extern "C" int mms_set_option(const char* name, int32_t value) {
    MMS_REQUIRE(name && name[0], "set_option: empty name");
    std::lock_guard<std::mutex> lk(g_opt_mu);
    g_opt[name] = OptVal{true, value};
    return MMS_OK;
}

extern "C" int mms_clear_option(const char* name) {
    MMS_REQUIRE(name && name[0], "clear_option: empty name");
    std::lock_guard<std::mutex> lk(g_opt_mu);
    g_opt[name] = OptVal{false, 0};               // back to the built-in default (the environment is not re-read)
    return MMS_OK;
}

extern "C" int32_t mms_get_option(const char* name, int32_t dflt) {
    if (!name || !name[0]) return dflt;
    return option_get(name, dflt);
}

extern "C" int64_t mms_launch_count(void) { return (int64_t)g_launches.load(); }

extern "C" int mms_profile_enable(int32_t on) {
    for (auto& r : g_recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    g_recs.clear();
    g_prof_on = on != 0;
    return MMS_OK;
}

extern "C" int mms_timeline_enable(int32_t on) {
    g_tl_recs.clear();
    if (on && !g_tl_buf) MMS_CUDA(cudaMalloc(&g_tl_buf, sizeof(unsigned long long) * 2 * TL_MAX));      // diagnostic only
    if (on) MMS_CUDA(cudaMemset(g_tl_buf, 0, sizeof(unsigned long long) * 2 * TL_MAX));
    g_tl_on = on != 0;
    return MMS_OK;
}

extern "C" int mms_timeline_report(char* buf_host, int64_t buf_bytes) {
    MMS_REQUIRE(buf_host && buf_bytes > 0, "timeline_report: bad buffer");
    MMS_REQUIRE(g_tl_buf, "timeline_report: mms_timeline_enable(1) was never called");
    MMS_CUDA(cudaDeviceSynchronize());
    const size_t n = g_tl_recs.size();
    std::vector<unsigned long long> t(2 * n + 2);
    if (n) MMS_CUDA(cudaMemcpy(t.data(), g_tl_buf, sizeof(unsigned long long) * 2 * n, cudaMemcpyDeviceToHost));
    unsigned long long t0 = ~0ull;
    for (size_t i = 0; i < n; ++i)
        if (t[2 * i] && t[2 * i] < t0) t0 = t[2 * i];
    std::map<cudaStream_t, int> sid;
    std::string out;
    char line[256];
    for (size_t i = 0; i < n; ++i) {
        if (!t[2 * i] || !t[2 * i + 1]) continue;                  // recorded but not executed (yet)
        auto it = sid.find(g_tl_recs[i].stream);
        if (it == sid.end()) it = sid.emplace(g_tl_recs[i].stream, (int)sid.size()).first;
        snprintf(line, sizeof(line), "%s %d %llu %llu\n", g_tl_recs[i].name, it->second, t[2 * i] - t0, t[2 * i + 1] - t0);
        out += line;
    }
    if ((int64_t)out.size() + 1 > buf_bytes) out.resize(buf_bytes - 1);
    memcpy(buf_host, out.c_str(), out.size() + 1);
    return MMS_OK;
}

extern "C" int mms_profile_report(char* buf_host, int64_t buf_bytes) {
    MMS_REQUIRE(buf_host && buf_bytes > 0, "profile_report: bad buffer");
    MMS_CUDA(cudaDeviceSynchronize());
    std::map<std::string, std::pair<long long, double>> agg;
    std::vector<std::string> order;
    for (auto& r : g_recs) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, r.a, r.b) != cudaSuccess) continue;
        auto it = agg.find(r.name);
        if (it == agg.end()) { agg[r.name] = {1, (double)ms}; order.push_back(r.name); }
        else { it->second.first += 1; it->second.second += ms; }
    }
    std::string out;
    char line[256];
    for (auto& n : order) {
        snprintf(line, sizeof(line), "%s %lld %.6f\n", n.c_str(), agg[n].first, agg[n].second);
        out += line;
    }
    if ((int64_t)out.size() + 1 > buf_bytes) out.resize(buf_bytes - 1);
    memcpy(buf_host, out.c_str(), out.size() + 1);
    return MMS_OK;
}
