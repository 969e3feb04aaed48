// iqw_stft_bluestein.cu -- kernel 1 for frame lengths that are NOT a power of two.
//
// The reference derives nfft = round(fs / resolution) (fourier.py:1250-1255) and hands any length to
// scipy.fft / cuFFT (fourier.py:200-218).  Here such a frame is transformed with Bluestein's chirp-z
// identity  n k = (n^2 + k^2 - (k - n)^2) / 2 :
//     X[k] = conj(ch[k]) * sum_n (c[n] x[n] conj(ch[n])) * ch[k - n],      ch[m] = exp(i pi m^2 / N)
// i.e. a circular convolution of length M = 2^p >= 2N - 1, evaluated with the power-of-two machinery of
// kernel 1 WITHOUT leaving the CTA: gather x window x chirp -> M-point FFT (fft_core.cuh passes in
// registers and shared memory) -> multiply by the precomputed spectrum of the chirp filter -> M-point
// inverse FFT (conj . FFT . conj, the renaming trick of ola_kernel) -> chirp -> {complex | |X|^2 | dB} ->
// band trim.  One read of the samples, one write of the result, like the power-of-two kernel; the price
// is two transforms of 2-4x the frame length.  Tables (host, float64, cached per window / N):
//   pre[n]  = c[n] * exp(-i pi n^2 / N)   n < N     (c = the frame coefficients of iqw_stft_c64's window)
//   bh[k]   = FFT_M(wrapped ch)[k] / M              (the 1/M of the inverse transform folded in)
//   post[k] = exp(-i pi k^2 / N)          k < N
// Built for even N with 2N - 1 <= 8192 (N <= 4096); longer frames take the composed path of
// iqw_bluestein_* below through the large-nfft kernels.
#include "iqw_stft.cuh"

namespace iqw {

struct BlueArgs {
    const float2* x;
    long long x_ch_stride;
    int n_channels;
    const float2 *pre, *bh, *post;
    int n;                      // frame length N
    long long hop, n_frames;
    float eps;
    int bin_lo, bin_hi;
    void* out;
    long long out_ch_stride;
    const float2* twiddle;
    long long n_groups, groups_per_ch;
};

template <int LOG2M, int MODE>
__global__ void __launch_bounds__(StftCfg<LOG2M>::THREADS, StftCfg<LOG2M>::MIN_BLOCKS)
bluestein_kernel(const BlueArgs a) {
    using C = StftCfg<LOG2M>;
    constexpr int M = C::N, E = C::E, TPF = C::TPF, FPC = C::FPC;
    constexpr int R0 = plan_radix(LOG2M, 0);
    constexpr int RL = plan_radix(LOG2M, C::NP - 1);

    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* tw = reinterpret_cast<float2*>(smem_raw);
    float2* bufs = tw + C::TW_ALLOC;
    for (int i = threadIdx.x; i < C::TW; i += C::THREADS) tw[i] = a.twiddle[i];
    __syncthreads();

    const int slot = threadIdx.x / TPF;
    const int ltid = threadIdx.x % TPF;
    const long long per = (a.n_groups + gridDim.x - 1) / gridDim.x;
    const long long g_begin = per * blockIdx.x;
    const long long g_end = g_begin + per < a.n_groups ? g_begin + per : a.n_groups;
    const int nbins = a.bin_hi - a.bin_lo;
    int par = 0;
    long long c = g_begin / a.groups_per_ch;
    long long gc = g_begin - c * a.groups_per_ch;

    for (long long g = g_begin; g < g_end; ++g) {
        const long long frame = gc * FPC + slot;
        const bool valid = frame < a.n_frames;
        const long long c_cur = c;
        if (++gc == a.groups_per_ch) { gc = 0; ++c; }

        // a[n] = x[n] * pre[n] for n < N, zero up to M
        float2 v[E];
        {
            const float2* src = a.x + c_cur * a.x_ch_stride + frame * a.hop;
#pragma unroll
            for (int q = 0; q < E / R0; ++q)
#pragma unroll
                for (int r = 0; r < R0; ++r) {
                    const int n = (ltid + q * TPF) + r * (M / R0);
                    float2 z = make_float2(0.f, 0.f);
                    if (valid && n < a.n) z = cmul(__ldg(src + n), __ldg(a.pre + n));
                    v[q * R0 + r] = z;
                }
        }
        PassLoop<LOG2M, 0>::run(v, bufs, tw, nullptr, ltid, slot, par);

        // spectrum of the convolution, conjugated and renamed into the load order of the next transform
        float2 u[E];
#pragma unroll
        for (int q = 0; q < E / RL; ++q)
#pragma unroll
            for (int r = 0; r < RL; ++r) {
                const int j = q + r * (E / RL);
                const int k = ltid + j * TPF;
                const float2 p = cmul(v[q * RL + r], __ldg(a.bh + k));
                u[(j % (E / R0)) * R0 + j / (E / R0)] = make_float2(p.x, -p.y);
            }
        PassLoop<LOG2M, 0>::run(u, bufs, tw, nullptr, ltid, slot, par);

        if (valid) {
            const long long row = c_cur * a.out_ch_stride + frame * (long long)nbins - a.bin_lo;
#pragma unroll
            for (int q = 0; q < E / RL; ++q)
#pragma unroll
                for (int r = 0; r < RL; ++r) {
                    const int k = ltid + (q + r * (E / RL)) * TPF;
                    if (k >= a.bin_lo && k < a.bin_hi) {        // (bin_hi <= N)
                        const float2 cz = u[q * RL + r];        // conj of the convolution value
                        if constexpr (MODE == IQW_STFT_COMPLEX) {
                            const float2 X = cmul(make_float2(cz.x, -cz.y), __ldg(a.post + k));
                            __stcs(reinterpret_cast<float2*>(a.out) + row + k, X);
                        } else {
                            float p = cz.x * cz.x + cz.y * cz.y;        // |post[k]| = 1
                            if constexpr (MODE == IQW_STFT_DB) p = power_to_dB(p, a.eps);
                            __stcs(reinterpret_cast<float*>(a.out) + row + k, p);
                        }
                    }
                }
        }
    }
}

template <int LOG2M, int MODE>
static int launch_blue_mode(BlueArgs a, cudaStream_t stream) {
    using C = StftCfg<LOG2M>;
    auto kern = bluestein_kernel<LOG2M, MODE>;
    if (int rc = get_twiddles(LOG2M, stream, &a.twiddle)) return rc;
    long long grid = 0;
    if (int rc = resident_ctas(kern, C::THREADS, C::SMEM, "bluestein kernel", &grid)) return rc;
    a.groups_per_ch = (a.n_frames + C::FPC - 1) / C::FPC;
    a.n_groups = a.groups_per_ch * a.n_channels;
    if (grid > a.n_groups) grid = a.n_groups;
    { IQW_PROFILE("stft_bluestein_kernel", stream); kern<<<(unsigned)grid, C::THREADS, C::SMEM, stream>>>(a); }
    IQW_CUDA_OK(cudaGetLastError());
    return IQW_OK;
}

// ---- composed path for longer frames: three elementwise kernels around two calls of the large FFT ----
// a[f][m] = x[f*hop + m] * pre[m] (m < N), 0 (N <= m < M)
__global__ void blue_pre_kernel(const float2* __restrict__ x, long long hop, const float2* __restrict__ pre, int n, int m,
                                long long n_frames, float2* __restrict__ out) {
    const long long total = n_frames * m;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long f = i / m;
        const int k = (int)(i - f * m);
        out[i] = k < n ? cmul(__ldg(x + f * hop + k), __ldg(pre + k)) : make_float2(0.f, 0.f);
    }
}
// in place: a[f][k] = conj(a[f][k] * bh[k])
__global__ void blue_mul_kernel(float2* __restrict__ a, const float2* __restrict__ bh, int m, long long n_frames) {
    const long long total = n_frames * m;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const float2 p = cmul(a[i], __ldg(bh + (int)(i % m)));
        a[i] = make_float2(p.x, -p.y);
    }
}
// X[f][k] = post[k] * conj(a[f][k]), k in [bin_lo, bin_hi)
template <int MODE>
__global__ void blue_post_kernel(const float2* __restrict__ a, const float2* __restrict__ post, int m, long long n_frames,
                                 int bin_lo, int bin_hi, float eps, void* __restrict__ out) {
    const int nb = bin_hi - bin_lo;
    const long long total = n_frames * nb;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long f = i / nb;
        const int k = bin_lo + (int)(i - f * nb);
        const float2 cz = a[f * m + k];
        if constexpr (MODE == IQW_STFT_COMPLEX) {
            reinterpret_cast<float2*>(out)[i] = cmul(make_float2(cz.x, -cz.y), __ldg(post + k));
        } else {
            float p = cz.x * cz.x + cz.y * cz.y;
            if constexpr (MODE == IQW_STFT_DB) p = power_to_dB(p, eps);
            reinterpret_cast<float*>(out)[i] = p;
        }
    }
}

}  // namespace iqw

using namespace iqw;

extern "C" int iqw_stft_bluestein_c64(const void* d_x, int64_t n_channels, int64_t n_samples, int64_t x_channel_stride,
                                      const void* d_pre, const void* d_bh, const void* d_post, int32_t nfft, int32_t m,
                                      int64_t hop, int64_t n_frames, int32_t mode, float eps, int32_t bin_lo,
                                      int32_t bin_hi, void* d_out, int64_t out_channel_stride, void* stream) {
    iqw::DeviceGuard _dev_guard(d_x);
    if (!d_x || !d_pre || !d_bh || !d_post || !d_out) return fail(IQW_ERR_INVALID, "null pointer argument");
    if (nfft < 2) return fail(IQW_ERR_INVALID, "nfft=%d", nfft);
    const int log2m = log2_exact(m);
    if (log2m < 1 || m < 2 * nfft - 1) return fail(IQW_ERR_INVALID, "m=%d must be a power of two >= 2*nfft - 1", m);
    if (log2m < 4 || log2m > 13)
        return fail(IQW_ERR_UNSUPPORTED, "iqw_stft_bluestein_c64: convolution length %d outside 16..8192 (nfft <= 4096)", m);
    if (hop < 1) return fail(IQW_ERR_INVALID, "hop=%lld must be >= 1", (long long)hop);
    if (n_channels < 0 || n_frames < 0) return fail(IQW_ERR_INVALID, "negative size");
    if (n_channels == 0 || n_frames == 0) return IQW_OK;
    if ((n_frames - 1) * hop + nfft > n_samples)
        return fail(IQW_ERR_INVALID, "n_frames=%lld does not fit in n_samples=%lld", (long long)n_frames, (long long)n_samples);
    if (bin_lo < 0 || bin_hi > nfft || bin_lo >= bin_hi) return fail(IQW_ERR_INVALID, "bad bin range [%d, %d)", bin_lo, bin_hi);
    if (n_channels > 0x7fffffff) return fail(IQW_ERR_INVALID, "too many channels");
    BlueArgs a{};
    a.x = static_cast<const float2*>(d_x);
    a.x_ch_stride = x_channel_stride;
    a.n_channels = (int)n_channels;
    a.pre = static_cast<const float2*>(d_pre);
    a.bh = static_cast<const float2*>(d_bh);
    a.post = static_cast<const float2*>(d_post);
    a.n = nfft;
    a.hop = hop;
    a.n_frames = n_frames;
    a.eps = eps;
    a.bin_lo = bin_lo;
    a.bin_hi = bin_hi;
    a.out = d_out;
    a.out_ch_stride = out_channel_stride;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    return dispatch<4, 13>(
        log2m, [&](auto L) { return dispatch_stft_mode(mode, [&](auto M) { return launch_blue_mode<L, M>(a, s); }); },
        [&] { return fail(IQW_ERR_UNSUPPORTED, "m=%d", m); });
}

// the three elementwise steps of the composed path (python drives the two FFT calls between them)
extern "C" int iqw_bluestein_pre_c64(const void* d_x, int64_t hop, const void* d_pre, int32_t nfft, int32_t m,
                                     int64_t n_frames, void* d_a, void* stream) {
    iqw::DeviceGuard _dev_guard(d_x);
    if (!d_x || !d_pre || !d_a || nfft < 1 || m < nfft || n_frames < 0 || hop < 1) return fail(IQW_ERR_INVALID, "bad argument");
    if (n_frames == 0) return IQW_OK;
    int sms = 0;
    if (int rc = device_sm_count(&sms)) return rc;
    blue_pre_kernel<<<sms * 8, 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const float2*>(d_x), hop, static_cast<const float2*>(d_pre), nfft, m, n_frames, static_cast<float2*>(d_a));
    IQW_CUDA_OK(cudaGetLastError());
    return IQW_OK;
}

extern "C" int iqw_bluestein_mul_c64(void* d_a, const void* d_bh, int32_t m, int64_t n_frames, void* stream) {
    iqw::DeviceGuard _dev_guard(d_a);
    if (!d_a || !d_bh || m < 1 || n_frames < 0) return fail(IQW_ERR_INVALID, "bad argument");
    if (n_frames == 0) return IQW_OK;
    int sms = 0;
    if (int rc = device_sm_count(&sms)) return rc;
    blue_mul_kernel<<<sms * 8, 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<float2*>(d_a),
                                                                         static_cast<const float2*>(d_bh), m, n_frames);
    IQW_CUDA_OK(cudaGetLastError());
    return IQW_OK;
}

extern "C" int iqw_bluestein_post_c64(const void* d_a, const void* d_post, int32_t m, int64_t n_frames, int32_t mode,
                                      float eps, int32_t bin_lo, int32_t bin_hi, void* d_out, void* stream) {
    iqw::DeviceGuard _dev_guard(d_a);
    if (!d_a || !d_post || !d_out || m < 1 || n_frames < 0 || bin_lo < 0 || bin_hi > m || bin_lo >= bin_hi)
        return fail(IQW_ERR_INVALID, "bad argument");
    if (n_frames == 0) return IQW_OK;
    int sms = 0;
    if (int rc = device_sm_count(&sms)) return rc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const float2* a = static_cast<const float2*>(d_a);
    const float2* post = static_cast<const float2*>(d_post);
    return dispatch_stft_mode(mode, [&](auto M) -> int {
        blue_post_kernel<M><<<sms * 8, 256, 0, s>>>(a, post, m, n_frames, bin_lo, bin_hi, eps, d_out);
        IQW_CUDA_OK(cudaGetLastError());
        return IQW_OK;
    });
}
