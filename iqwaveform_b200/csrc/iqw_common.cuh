// iqw_common.cuh -- error and launch plumbing and small device helpers shared by the kernels.
#pragma once
#include <cuda_runtime.h>
#include <cstdarg>
#include <cstdio>
#include <cstdint>
#include <type_traits>
#include "../../include/iqw_b200.h"

namespace iqw {

char* last_error_buffer();   // thread-local, defined in iqw_abi.cu

inline int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(last_error_buffer(), 512, fmt, ap);
    va_end(ap);
    return code;
}

#define IQW_CUDA_OK(expr)                                                                   \
    do {                                                                                    \
        cudaError_t _e = (expr);                                                            \
        if (_e != cudaSuccess)                                                              \
            return ::iqw::fail(IQW_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,                \
                               cudaGetErrorString(_e), __FILE__, __LINE__);                 \
    } while (0)

int device_sm_count(int* sms);

// log2(v) when v is a power of two, -1 otherwise (so a result < 1 rejects every v that is not a power of two >= 2)
inline int log2_exact(long long v) {
    if (v < 1 || (v & (v - 1))) return -1;
    int l = 0;
    while ((1ll << l) < v) ++l;
    return l;
}

// Turns the runtime value v into a template argument: f(std::integral_constant<int, v>{}) when LO <= v <= HI,
// fallback() otherwise.  Only the kernels that f names for LO..HI are instantiated.
template <int LO, int HI, class F, class G>
int dispatch(int v, F&& f, G&& fallback) {
    if constexpr (LO > HI) return fallback();
    else return v == LO ? f(std::integral_constant<int, LO>{}) : dispatch<LO + 1, HI>(v, f, fallback);
}

// Number of CTAs of `kern` that are resident at once (SMs x CTAs per SM) with `threads` threads and `smem` bytes of
// dynamic shared memory, after raising the kernel's dynamic shared-memory limit to `smem`.
template <class Kernel>
int resident_ctas(Kernel kern, int threads, size_t smem, const char* name, long long* ctas) {
    IQW_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int sms = 0, per_sm = 0;
    if (int rc = device_sm_count(&sms)) return rc;
    IQW_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem));
    if (per_sm < 1)
        return fail(IQW_ERR_CUDA, "%s (%d threads, %zu bytes of shared memory) does not fit on an SM", name, threads, smem);
    *ctas = (long long)sms * per_sm;
    return IQW_OK;
}

// Immutable float2 tables on the current device, built on first use: `init` launches the kernel that fills the
// `count` entries of the table (kind, param) on `stream`; the stream is synchronised once, so that the table is
// visible to every later stream.  `init` must not call device_table.
enum TableKind { kFftTwiddles, kTwoPassTwiddles, kThreePassTwiddles, kStepTwiddles, kPfbRotation };
int device_table(TableKind kind, int param, size_t count, void (*init)(float2* table, int param, cudaStream_t stream),
                 cudaStream_t stream, const float2** out);

// Every compute entry point launches on the device that OWNS its buffers, whatever device is current
// in the calling thread (a tensor on cuda:1 while cuda:0 is current would otherwise be launched on the
// wrong device, with a foreign stream and a twiddle table of the other device).  The previous device
// is restored on return.  Costs one cudaPointerGetAttributes (~0.3 us) per call.
struct DeviceGuard {
    int prev = -1;
    bool switched = false;
    explicit DeviceGuard(const void* p) {
        if (!p) return;
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return; }
        if (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged) return;
        if (cudaGetDevice(&prev) != cudaSuccess) return;
        if (at.device != prev && cudaSetDevice(at.device) == cudaSuccess) switched = true;
    }
    ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
};

// Optional kernel timing (off by default): a launch site is wrapped in a scope that records a CUDA
// event before and after it ON THE LAUNCHING STREAM.  Level 1 (what bench.py runs its timed region
// under) times the heavy kernels one by one and the trains of small follow-up kernels as one scope
// each -- ~12 events per persistence-spectrum step instead of ~46, which cost 2 % of the step;
// level 2 times every launch (probes).  A scope carries the number of launches it covers.
int profile_level();
inline bool profile_enabled() { return profile_level() >= 1; }
void profile_push(const char* name, int launches, cudaEvent_t a, cudaEvent_t b);
struct ProfScope {
    const char* name; cudaStream_t s; int n; cudaEvent_t a = nullptr, b = nullptr;
    ProfScope(const char* nm, cudaStream_t st, int launches, bool on) : name(nm), s(st), n(launches) {
        if (on) { cudaEventCreate(&a); cudaEventCreate(&b); cudaEventRecord(a, s); }
    }
    ~ProfScope() { if (a) { cudaEventRecord(b, s); profile_push(name, n, a, b); } }
};
#define IQW_CAT2(a, b) a##b
#define IQW_CAT(a, b) IQW_CAT2(a, b)
// one heavy launch: timed at every level
#define IQW_PROFILE(name, stream) ::iqw::ProfScope IQW_CAT(_prof_, __LINE__)(name, stream, 1, ::iqw::profile_level() >= 1)
// one small launch inside a train: timed at level 2 only
#define IQW_PROFILE_FINE(name, stream) ::iqw::ProfScope IQW_CAT(_prof_, __LINE__)(name, stream, 1, ::iqw::profile_level() >= 2)
// a train of n small launches as one scope: timed at level 1 only (level 2 times its members)
#define IQW_PROFILE_TRAIN(name, stream, n) ::iqw::ProfScope IQW_CAT(_prof_, __LINE__)(name, stream, n, ::iqw::profile_level() == 1)

// order-preserving map float32 -> uint32 (total order: -nan < -inf < ... < -0 < +0 < ... < +inf < nan)
__host__ __device__ __forceinline__ uint32_t float_to_key(float f) {
#if defined(__CUDA_ARCH__)
    uint32_t b = __float_as_uint(f);
#else
    union { float f; uint32_t u; } c; c.f = f; uint32_t b = c.u;
#endif
    return b ^ ((b & 0x80000000u) ? 0xFFFFFFFFu : 0x80000000u);
}
__host__ __device__ __forceinline__ float key_to_float(uint32_t k) {
    uint32_t b = k ^ ((k & 0x80000000u) ? 0x80000000u : 0xFFFFFFFFu);
#if defined(__CUDA_ARCH__)
    return __uint_as_float(b);
#else
    union { float f; uint32_t u; } c; c.u = b; return c.f;
#endif
}

// 10*log10(|p| + eps) in float32 (power_analysis.py:199-204: abs, += eps, log10, *= 10).
// log10 is ONE `lg2.approx.ftz` times log10(2).  Measured over every exponent of the normal range
// (tools/exp/lg2_accuracy.cu, 2^24 random arguments): the result is within one ulp of log2(v) -- 2.1e-7 for
// |log2| < 1, 7.8e-6 at log2 = -111 -- i.e. at most 2.3e-5 dB at -334 dB and 1e-5 dB around +-100 dB, inside the
// 5e-5 dB parity bound, at a fifth of the instructions of log10f.  (Rounds 1 and 2 split v = m * 2^e and took
// lg2 of the mantissa alone: five more instructions per value for half an ulp.)  Zero, denormal, infinite and
// NaN arguments take log10f so that -inf / nan come out exactly as the reference's.
static __device__ __noinline__ float power_to_dB_slow(float v) { return 10.0f * log10f(v); }

// the two halves of power_to_dB for kernels that convert many values per thread: a branch-free fast
// path that is right whenever dB_fast_ok(v), so that the (rare) other arguments can be patched later
__device__ __forceinline__ bool dB_fast_ok(float v) { return __float_as_uint(v) - 0x00800000u < 0x7F000000u; }
__device__ __forceinline__ float power_to_dB_fast(float v /* = |p| + eps */, bool& ok) {
    ok = dB_fast_ok(v);
    float l;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(v));
    return l * 3.01029995663981195f;
}

__device__ __forceinline__ float power_to_dB(float p, float eps) {
    const float v = fabsf(p) + eps;
    if (dB_fast_ok(v)) {                          // normal, finite, positive
        float l;
        asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(v));
        return l * 3.01029995663981195f;
    }
    return power_to_dB_slow(v);                   // rare: out of line keeps the hot loops small
}

}  // namespace iqw
