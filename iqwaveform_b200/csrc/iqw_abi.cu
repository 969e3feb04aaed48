// iqw_abi.cu -- version / error plumbing of the C-ABI (include/iqw_b200.h) and the per-device caches.
#include <mutex>
#include <vector>
#include <string>
#include <map>
#include <tuple>
#include <atomic>
#include <cstring>
#include "iqw_common.cuh"

namespace iqw {

char* last_error_buffer() {
    static thread_local char buf[512] = "";
    return buf;
}

int device_sm_count(int* sms) {
    static std::mutex m;
    static int cache[64] = {0};
    int dev = 0;
    IQW_CUDA_OK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(m);
    if (dev < 64 && cache[dev]) { *sms = cache[dev]; return IQW_OK; }
    int n = 0;
    IQW_CUDA_OK(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
    if (dev < 64) cache[dev] = n;
    *sms = n;
    return IQW_OK;
}

static std::mutex g_table_mutex;
static std::map<std::tuple<int, int, int>, float2*> g_tables;   // (device, kind, param) -> table

int device_table(TableKind kind, int param, size_t count, void (*init)(float2*, int, cudaStream_t), cudaStream_t stream,
                 const float2** out) {
    int dev = 0;
    IQW_CUDA_OK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(g_table_mutex);
    const auto key = std::make_tuple(dev, (int)kind, param);
    auto it = g_tables.find(key);
    if (it == g_tables.end()) {
        float2* d = nullptr;
        IQW_CUDA_OK(cudaMalloc(&d, sizeof(float2) * count));
        init(d, param, stream);
        IQW_CUDA_OK(cudaGetLastError());
        IQW_CUDA_OK(cudaStreamSynchronize(stream));
        it = g_tables.emplace(key, d).first;
    }
    *out = it->second;
    return IQW_OK;
}

static std::atomic<int> g_prof_level{0};
static std::mutex g_prof_mutex;
struct ProfRec { const char* name; int launches; cudaEvent_t a, b; };
static std::vector<ProfRec> g_prof;

int profile_level() { return g_prof_level.load(std::memory_order_relaxed); }
// at most kProfCap open records: a caller that leaves profiling on without ever reading the report
// gets the oldest scopes only, and the events of the dropped ones are released at once
static constexpr size_t kProfCap = 1 << 16;
void profile_push(const char* name, int launches, cudaEvent_t a, cudaEvent_t b) {
    std::lock_guard<std::mutex> lock(g_prof_mutex);
    if (g_prof.size() >= kProfCap) { cudaEventDestroy(a); cudaEventDestroy(b); return; }
    g_prof.push_back({name, launches, a, b});
}

}  // namespace iqw

extern "C" int iqw_abi_version(void) { return IQW_ABI_VERSION; }
extern "C" const char* iqw_last_error(void) { return iqw::last_error_buffer(); }

extern "C" int iqw_profile_enable(int level) { iqw::g_prof_level.store(level < 0 ? 0 : level > 2 ? 2 : level); return IQW_OK; }

extern "C" int iqw_profile_reset(void) {
    std::lock_guard<std::mutex> lock(iqw::g_prof_mutex);
    for (auto& r : iqw::g_prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    iqw::g_prof.clear();
    return IQW_OK;
}

// one line per kernel name: "<name> <launches> <total_ms>\n"; call after synchronising the stream
extern "C" int iqw_profile_report(char* buf, size_t cap) {
    std::lock_guard<std::mutex> lock(iqw::g_prof_mutex);
    std::map<std::string, std::pair<long, double>> agg;
    for (auto& r : iqw::g_prof) {
        float ms = 0.f;
        cudaError_t e = cudaEventElapsedTime(&ms, r.a, r.b);
        if (e != cudaSuccess) return iqw::fail(IQW_ERR_CUDA, "profile: %s", cudaGetErrorString(e));
        auto& x = agg[r.name];
        x.first += r.launches;
        x.second += ms;
    }
    std::string out;
    for (auto& kv : agg) {
        char line[256];
        snprintf(line, sizeof line, "%s %ld %.6f\n", kv.first.c_str(), kv.second.first, kv.second.second);
        out += line;
    }
    if (out.size() + 1 > cap) return iqw::fail(IQW_ERR_INVALID, "profile buffer too small");
    memcpy(buf, out.c_str(), out.size() + 1);
    return IQW_OK;
}
