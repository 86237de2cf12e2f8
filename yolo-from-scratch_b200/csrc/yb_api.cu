// yb_api.cu — library-wide plumbing: thread-local error text, launch counter, device query.
#include <atomic>
#include <cstdarg>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>
#include "yb_common.cuh"

namespace yb {

static thread_local char g_err[512] = "";
static std::atomic<unsigned long long> g_launches{0};

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

void count_launch(int n) { g_launches.fetch_add((unsigned long long)n, std::memory_order_relaxed); }

int sm_count() {
    static thread_local int cached_dev = -1, cached = 148;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (dev != cached_dev) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) {
            cached = n;
            cached_dev = dev;
        }
    }
    return cached;
}

struct TimingRec { const char* name; cudaEvent_t a, b; };
static std::mutex g_tmu;
static std::vector<TimingRec> g_trecs;
static std::atomic<int> g_timing{0};

KernelScope::KernelScope(const char* name, cudaStream_t st) : name_(name), st_(st), a_(nullptr), b_(nullptr), on_(false) {
    if (!g_timing.load(std::memory_order_relaxed)) return;
    if (cudaEventCreate(&a_) != cudaSuccess || cudaEventCreate(&b_) != cudaSuccess) return;
    on_ = cudaEventRecord(a_, st_) == cudaSuccess;
}
KernelScope::~KernelScope() {
    if (!on_) return;
    cudaEventRecord(b_, st_);
    std::lock_guard<std::mutex> lk(g_tmu);
    g_trecs.push_back({name_, a_, b_});
}

}  // namespace yb

extern "C" void yb_timing_enable(int on) { yb::g_timing.store(on ? 1 : 0); }

// Synchronises the recorded events and writes "name count total_ms\n" lines into buf.
extern "C" int yb_timing_collect(char* buf, size_t n) {
    using namespace yb;
    std::lock_guard<std::mutex> lk(g_tmu);
    std::map<std::string, std::pair<int, double>> agg;
    std::vector<std::string> order;
    for (auto& r : g_trecs) {
        float ms = 0.f;
        cudaEventSynchronize(r.b);
        cudaEventElapsedTime(&ms, r.a, r.b);
        cudaEventDestroy(r.a);
        cudaEventDestroy(r.b);
        if (!agg.count(r.name)) order.push_back(r.name);
        auto& e = agg[r.name];
        e.first += 1;
        e.second += ms;
    }
    g_trecs.clear();
    std::string out;
    for (auto& k : order) {
        char line[256];
        snprintf(line, sizeof(line), "%s %d %.6f\n", k.c_str(), agg[k].first, agg[k].second);
        out += line;
    }
    if (buf && n) {
        strncpy(buf, out.c_str(), n - 1);
        buf[n - 1] = 0;
    }
    return (int)out.size();
}

extern "C" int yb_version(void) { return 102; }
extern "C" const char* yb_last_error(void) { return yb::g_err; }
extern "C" unsigned long long yb_launch_count(void) { return yb::g_launches.load(); }
