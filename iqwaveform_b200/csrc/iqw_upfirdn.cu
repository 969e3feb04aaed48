// iqw_upfirdn.cu -- kernel 6: polyphase FIR filter / rational resampler (scipy.signal.upfirdn semantics,
// zero padding), complex64 samples, real or complex fp32 taps.
//
//   y[n] = sum_{j < Lp} hp[p][j] * x[i0 - j],   t = n*down, p = t mod up, i0 = t div up,
//   hp[p][j] = h[p + j*up] (the host's polyphase table, zero-padded), Lp = ceil(L / up).
//
// Outputs n = s + k*U (U = up/g, D = down/g, g = gcd) share the phase p_s = (s*down) mod up and read
// i0 = k*D + i0_s, i0_s = (s*down) div up < D.  Two thread mappings, chosen by iqw_upfirdn_c64 from
// (up, down, L) alone (DESIGN.md "Kernel 6"):
//
//   upfirdn_slide_kernel  (U <= 8 and the tile fits in shared memory: decimators, interpolators, plain
//     filters).  A CTA owns KT = 128*R consecutive k of one channel for every phase class s.  Its input
//     span is staged into shared memory DE-INTERLEAVED by D (stream rho holds samples rho, rho+D, ...), so
//     that the R outputs of a thread, which step the input by D, read consecutive words of one stream.
//     Taps are walked residue by residue (j = r + c*D): tap c+1 of output m reads what tap c of output m-1
//     read, so a thread keeps a sliding window of R samples in registers and loads ONE new sample (plus
//     one warp-uniform broadcast tap) per R packed FMAs.  R = 7 is odd, which makes the lane stride of
//     those loads conflict-free for any D.  Results go through shared memory for coalesced stores.
//   upfirdn_phase_kernel  (everything else, e.g. 147/160).  Lanes span phase classes; a thread owns R
//     outputs of one phase (stepping k) and, for Lp <= 32 real / 16 complex taps, holds that phase's taps
//     in registers.  Neighbouring lanes read neighbouring samples, through L1 (ld.global.nc).
//
// Every output is one accumulator summed in an order fixed by (up, down, L) -- never by the tile, the
// CTA or the caller's x_first / out_first -- so time shards concatenate to the single-call bits.
#include "iqw_common.cuh"
#include "fft_core.cuh"

namespace iqw {

namespace {

constexpr int kSlideR = 7;                     // outputs per thread (odd: conflict-free window loads)
constexpr int kSlideThreads = 128;
constexpr int kSlideKT = kSlideR * kSlideThreads;
constexpr int kSlideMaxU = 8;
constexpr size_t kSmemBudget = 200 * 1024;
constexpr int kPhaseR = 4;
constexpr int kPhaseThreads = 128;
constexpr int kRegTapsReal = 32;
constexpr int kRegTapsComplex = 16;
constexpr long long kMaxTableFloats = 32768;   // 128 KB: 16384 real or 8192 complex taps for any up

struct UpfirdnArgs {
    const float2* x;
    long long n_in, x_stride, x_first;
    const void* taps;            // polyphase table, rows p < n_rows, Lp entries each
    int n_rows, lp, up, down, U, D;
    long long out_first, n_out, out_stride;
    long long k_min;             // k of the first tile
    float2* out;
};

template <bool CPLX> struct Tap;
template <> struct Tap<false> {
    using T = float;
    static __device__ __forceinline__ float2 fma(float2 x, float h, float2 acc) { return cfma_rs(x, h, acc); }
    static __device__ __forceinline__ float zero() { return 0.f; }
};
template <> struct Tap<true> {
    using T = float2;
    static __device__ __forceinline__ float2 fma(float2 x, float2 h, float2 acc) { return cfma(x, h, acc); }
    static __device__ __forceinline__ float2 zero() { return make_float2(0.f, 0.f); }
};

__device__ __forceinline__ float2 load_x(const float2* x, long long i, long long n) {
    return (i >= 0 && i < n) ? __ldg(x + i) : make_float2(0.f, 0.f);
}

// shared memory of the slide kernel, in bytes: de-interleaved span + output tile + the U used tap rows
__host__ __device__ inline int slide_qs(int lp, int D) { return (kSlideKT + (lp - 1 + D - 1) / D + 1) | 1; }
inline size_t slide_smem(int lp, int U, int D, bool cplx) {
    return sizeof(float2) * ((size_t)D * slide_qs(lp, D) + (size_t)kSlideKT * U) +
           (cplx ? sizeof(float2) : sizeof(float)) * (size_t)U * lp;
}

template <bool CPLX>
__global__ void __launch_bounds__(kSlideThreads) upfirdn_slide_kernel(const UpfirdnArgs a) {
    using T = typename Tap<CPLX>::T;
    constexpr int R = kSlideR, KT = kSlideKT;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int D = a.D, U = a.U, Lp = a.lp;
    const int QS = slide_qs(Lp, D);
    float2* X = reinterpret_cast<float2*>(smem_raw);             // [D][QS]
    float2* Y = X + (size_t)D * QS;                               // [KT][U]
    T* H = reinterpret_cast<T*>(Y + (size_t)KT * U);              // [U][Lp]
    const int tid = threadIdx.x;
    const long long ch = blockIdx.y;
    const long long kA = a.k_min + (long long)blockIdx.x * KT;
    const float2* x = a.x + ch * a.x_stride;

    // the U tap rows this CTA uses (row p_s of the table, zero when p_s >= n_rows)
    const T* taps = reinterpret_cast<const T*>(a.taps);
    for (int e = tid; e < U * Lp; e += kSlideThreads) {
        const int s = e / Lp, j = e - s * Lp;
        const int p = (int)(((long long)s * a.down) % a.up);
        H[e] = p < a.n_rows ? taps[(size_t)p * Lp + j] : Tap<CPLX>::zero();
    }
    // span [S0, S0 + Ls): every sample an output of the tile reads, stream rho = i mod D, word i div D
    const long long S0 = kA * D - (Lp - 1) - a.x_first;
    const int Ls = KT * D + Lp - 1;
    {
        int q = tid / D, rho = tid - (tid / D) * D;
        const int qstep = kSlideThreads / D, rstep = kSlideThreads - qstep * D;
        for (int i = tid; i < Ls; i += kSlideThreads) {
            X[rho * QS + q] = load_x(x, S0 + i, a.n_in);
            q += qstep;
            rho += rstep;
            if (rho >= D) { rho -= D; ++q; }
        }
    }
    __syncthreads();

    const int nres = D < Lp ? D : Lp;
    for (int s = 0; s < U; ++s) {
        const int i0s = (int)(((long long)s * a.down) / a.up);
        const T* h = H + s * Lp;
        float2 acc[R];
#pragma unroll
        for (int m = 0; m < R; ++m) acc[m] = make_float2(0.f, 0.f);
        for (int r = 0; r < nres; ++r) {
            // output m of this thread, tap j = r + c*D reads stream rho, word tid*R + qb + m - c
            const int e = i0s + Lp - 1 - r;
            const int qb = e / D, rho = e - qb * D;
            const float2* xs = X + rho * QS + tid * R + qb;
            const int Cr = (Lp - r + D - 1) / D;
            float2 b[R];                          // window: w[m] at tap c is b[(m - c) mod R]
#pragma unroll
            for (int m = 0; m < R; ++m) b[m] = xs[m];
            // tap c: every output takes it with its window sample, then the window slides by one
            auto step = [&](int c, int u) {
                const T hv = h[r + c * D];
#pragma unroll
                for (int m = 0; m < R; ++m) acc[m] = Tap<CPLX>::fma(b[(m - u + R) % R], hv, acc[m]);
                if (c + 1 < Cr) b[R - 1 - u] = xs[-(c + 1)];
            };
            // whole blocks of R taps carry no branch between their steps, so the tap and window loads of
            // later steps are issued ahead of the FMAs of earlier ones; the tail is the same sum, guarded
            int c0 = 0;
            for (; c0 + R <= Cr; c0 += R) {
#pragma unroll
                for (int u = 0; u < R; ++u) step(c0 + u, u);
            }
#pragma unroll
            for (int u = 0; u < R - 1; ++u) {
                if (c0 + u >= Cr) break;
                step(c0 + u, u);
            }
        }
#pragma unroll
        for (int m = 0; m < R; ++m) Y[(tid * R + m) * U + s] = acc[m];
    }
    __syncthreads();

    // coalesced store of outputs [kA*U, (kA+KT)*U) that fall inside [out_first, out_first + n_out)
    float2* out = a.out + ch * a.out_stride;
    const long long n0 = kA * U - a.out_first;
    for (int e = tid; e < KT * U; e += kSlideThreads) {
        const long long n = n0 + e;
        if (n >= 0 && n < a.n_out) __stcs(out + n, Y[e]);
    }
}

template <bool CPLX, bool REGS>
__global__ void __launch_bounds__(kPhaseThreads) upfirdn_phase_kernel(const UpfirdnArgs a, long long n_items) {
    using T = typename Tap<CPLX>::T;
    constexpr int R = kPhaseR;
    constexpr int NREG = REGS ? (CPLX ? kRegTapsComplex : kRegTapsReal) : 1;
    const long long it = (long long)blockIdx.x * kPhaseThreads + threadIdx.x;
    if (it >= n_items) return;
    const long long ch = blockIdx.y;
    const int s = (int)(it % a.U);
    const long long k0 = a.k_min + (it / a.U) * R;
    const int p = (int)(((long long)s * a.down) % a.up);
    const long long i0s = ((long long)s * a.down) / a.up;
    const int Lp = a.lp;
    const float2* x = a.x + ch * a.x_stride;
    float2* out = a.out + ch * a.out_stride;
    const T* h = reinterpret_cast<const T*>(a.taps) + (size_t)p * Lp;
    const bool live = p < a.n_rows;

    T hr[NREG];
    if constexpr (REGS) {
#pragma unroll
        for (int j = 0; j < NREG; ++j) hr[j] = (live && j < Lp) ? __ldg(h + j) : Tap<CPLX>::zero();
    }
    float2 acc[R];
    long long base[R];
    bool inside = true;
#pragma unroll
    for (int m = 0; m < R; ++m) {
        acc[m] = make_float2(0.f, 0.f);
        base[m] = (k0 + m) * a.D + i0s - a.x_first;      // buffer index of tap 0
        inside &= base[m] - (Lp - 1) >= 0 && base[m] < a.n_in;
    }
    // the same sum in both branches; the first skips the bounds test when every read is inside the buffer
    auto run = [&](auto ld) {
        if constexpr (REGS) {
#pragma unroll
            for (int j = 0; j < NREG; ++j) {
                if (j >= Lp) break;
#pragma unroll
                for (int m = 0; m < R; ++m) acc[m] = Tap<CPLX>::fma(ld(base[m] - j), hr[j], acc[m]);
            }
        } else {
            for (int j = 0; j < Lp; ++j) {
                const T hv = __ldg(h + j);
#pragma unroll
                for (int m = 0; m < R; ++m) acc[m] = Tap<CPLX>::fma(ld(base[m] - j), hv, acc[m]);
            }
        }
    };
    if (live) {
        if (inside) run([&](long long i) { return __ldg(x + i); });
        else run([&](long long i) { return load_x(x, i, a.n_in); });
    }
#pragma unroll
    for (int m = 0; m < R; ++m) {
        const long long n = s + (k0 + m) * a.U - a.out_first;
        if (n >= 0 && n < a.n_out) __stcs(out + n, acc[m]);
    }
}

long long gcd_ll(long long a, long long b) {
    while (b) { const long long t = a % b; a = b; b = t; }
    return a;
}

long long floor_div(long long a, long long b) { return a >= 0 ? a / b : -((-a + b - 1) / b); }

template <bool CPLX>
int launch_upfirdn(UpfirdnArgs a, int n_channels, cudaStream_t stream) {
    const long long k_first = floor_div(a.out_first, a.U);
    const long long k_last = floor_div(a.out_first + a.n_out - 1, a.U);
    a.k_min = k_first;
    const size_t smem = slide_smem(a.lp, a.U, a.D, CPLX);
    if (a.U <= kSlideMaxU && smem <= kSmemBudget) {
        auto kern = upfirdn_slide_kernel<CPLX>;
        IQW_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const long long tiles = (k_last - k_first) / kSlideKT + 1;
        if (tiles > 0x7FFFFFFFLL) return fail(IQW_ERR_UNSUPPORTED, "upfirdn: %lld output tiles", tiles);
        { IQW_PROFILE("upfirdn_slide_kernel", stream);
          kern<<<dim3((unsigned)tiles, (unsigned)n_channels), kSlideThreads, smem, stream>>>(a); }
    } else {
        const long long n_items = a.U * ((k_last - k_first) / kPhaseR + 1);
        const long long blocks = (n_items + kPhaseThreads - 1) / kPhaseThreads;
        if (blocks > 0x7FFFFFFFLL) return fail(IQW_ERR_UNSUPPORTED, "upfirdn: %lld blocks", blocks);
        const dim3 grid((unsigned)blocks, (unsigned)n_channels);
        IQW_PROFILE("upfirdn_phase_kernel", stream);
        if (a.lp <= (CPLX ? kRegTapsComplex : kRegTapsReal))
            upfirdn_phase_kernel<CPLX, true><<<grid, kPhaseThreads, 0, stream>>>(a, n_items);
        else
            upfirdn_phase_kernel<CPLX, false><<<grid, kPhaseThreads, 0, stream>>>(a, n_items);
    }
    IQW_CUDA_OK(cudaGetLastError());
    return IQW_OK;
}

}  // namespace

}  // namespace iqw

extern "C" int iqw_upfirdn_c64(const void* d_x, int64_t n_channels, int64_t n_in, int64_t x_channel_stride,
                               int64_t x_first, const void* d_taps, int32_t taps_complex, int32_t n_taps, int32_t up,
                               int32_t down, int64_t out_first, int64_t n_out, void* d_out,
                               int64_t out_channel_stride, void* stream) {
    using namespace iqw;
    if (n_taps < 1 || up < 1 || down < 1)
        return fail(IQW_ERR_INVALID, "upfirdn: need n_taps >= 1, up >= 1, down >= 1 (got %d, %d, %d)", n_taps, up, down);
    if (n_channels < 0 || n_in < 0 || n_out < 0 || out_first < 0)
        return fail(IQW_ERR_INVALID, "upfirdn: negative size");
    if (n_channels == 0 || n_out == 0) return IQW_OK;
    if (!d_taps || !d_out || (n_in > 0 && !d_x)) return fail(IQW_ERR_INVALID, "upfirdn: null pointer");
    if (n_channels > 65535) return fail(IQW_ERR_UNSUPPORTED, "upfirdn: more than 65535 channels");
    if (n_channels > 1 && (x_channel_stride < n_in || out_channel_stride < n_out))
        return fail(IQW_ERR_INVALID, "upfirdn: channel stride shorter than a channel");
    const int lp = (n_taps + up - 1) / up;
    const int rows = up < n_taps ? up : n_taps;
    if ((long long)rows * lp * (taps_complex ? 2 : 1) > kMaxTableFloats)
        return fail(IQW_ERR_UNSUPPORTED, "upfirdn: polyphase table of %d x %d %s taps exceeds %lld floats", rows, lp,
                    taps_complex ? "complex" : "real", kMaxTableFloats);
    DeviceGuard guard(d_out);
    const long long g = gcd_ll(up, down);
    UpfirdnArgs a{};
    a.x = reinterpret_cast<const float2*>(d_x);
    a.n_in = n_in;
    a.x_stride = x_channel_stride;
    a.x_first = x_first;
    a.taps = d_taps;
    a.n_rows = rows;
    a.lp = lp;
    a.up = up;
    a.down = down;
    a.U = (int)(up / g);
    a.D = (int)(down / g);
    a.out_first = out_first;
    a.n_out = n_out;
    a.out_stride = out_channel_stride;
    a.out = reinterpret_cast<float2*>(d_out);
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    return taps_complex ? launch_upfirdn<true>(a, (int)n_channels, s) : launch_upfirdn<false>(a, (int)n_channels, s);
}
