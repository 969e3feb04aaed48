// iqw_istft.cu -- kernel 4: fused inverse STFT: band mask -> inverse FFT -> (-1)^n -> overlap-add.
//
// One pass over the frames replaces the reference's four materialising steps
// (/root/reference/src/iqwaveform/):
//   fourier.py:710-723   zero_stft_by_freq (two strided fills of the STFT, ola_filter only)
//   fourier.py:1075-1080 ifft of every frame (scipy.fft / cuFFT), 1/nfft inside
//   fourier.py:1084-1092 multiply by the (-1)^n 'rect' window that undoes the baked-in fft shift
//   fourier.py:584-649   _unstack_stft_windows: nfft/hop strided passes that add the frames up
//
// Work decomposition: the geometry of kernel 1 (a frame slot = TPF = nfft/E threads, E values per
// thread in registers, exchanges through padded ping-pong shared memory).  A slot walks a
// contiguous range of frames of one channel IN ORDER.  After the last FFT pass thread `ltid` holds
// the samples ltid + j*TPF (j = 0..E-1) of its frame; with hop = nfft/R = (E/R)*TPF the sample
// that overlaps it in the next frame is held BY THE SAME THREAD (j shifted by E/R), so the
// overlap-add is a register shift: acc[j] + y[j], the first E/R sums are complete and are stored
// (coalesced, TPF consecutive float2 per j), the rest slide down.  A range starts R-1 frames early
// to build up its accumulator (redundant work (R-1)/range, ~1 %).
//
// Bound: HBM, 8*R bytes read + 8 written per output sample (24 B at 50 % overlap).
// Sums run in frame order; the reference adds the frames of one residue class (m mod R) after the
// other -- identical for R <= 2 (two terms commute), last-bit different for R >= 4.
#include "iqw_stft.cuh"

namespace iqw {

struct IstftArgs {
    const float2* y;
    long long y_ch_stride;
    int n_channels;
    long long n_frames;
    int bin_lo, bin_hi;
    long long y_row;          // bins stored per frame: N, or bin_hi - bin_lo when only the band is stored
    int y_off;                // bin index of the first stored bin (0, or bin_lo)
    const float2* gain;       // optional per-bin complex gain (frequency-domain FIR), or null
    float scale;              // factor applied to every output sample after the overlap-add
    int natural;              // != 0: bins in natural (unshifted) order, no (-1)^n on the samples (plain ifft)
    float2* out;
    long long out_ch_stride;
    const float2* twiddle;
    long long streams_per_ch, frames_per_stream;
};

template <int LOG2N, int LOG2R, bool MASK, bool GAIN>
__global__ void __launch_bounds__(StftCfg<LOG2N>::THREADS, StftCfg<LOG2N>::MIN_BLOCKS)
istft_kernel(const IstftArgs a) {
    using C = StftCfg<LOG2N>;
    constexpr int N = C::N, E = C::E, TPF = C::TPF, FPC = C::FPC;
    constexpr int R0 = plan_radix(LOG2N, 0);
    constexpr int RL = plan_radix(LOG2N, C::NP - 1);
    constexpr int R = 1 << LOG2R;
    constexpr int H = E / R;              // values per thread that complete with every frame
    constexpr int A = E - H;              // values carried to the next frame
    constexpr long long HOP = N / R;
    static_assert(R <= E, "hop must be a multiple of nfft / E");

    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* tw = reinterpret_cast<float2*>(smem_raw);
    float2* bufs = tw + C::TW_ALLOC;
    for (int i = threadIdx.x; i < C::TW; i += C::THREADS) tw[i] = a.twiddle[i];
    __syncthreads();

    const int slot = threadIdx.x / TPF;
    const int ltid = threadIdx.x % TPF;
    const long long sid = (long long)blockIdx.x * FPC + slot;
    // every slot of the CTA runs the same number of iterations (the inter-pass barriers may span
    // several slots): a slot without work, warm-up frames before frame 0 and the short last range
    // transform zeros and store nothing
    const bool live = sid < a.streams_per_ch * a.n_channels;
    const long long c = live ? sid / a.streams_per_ch : 0;
    const long long f0 = live ? (sid - c * a.streams_per_ch) * a.frames_per_stream : 0;
    const long long f1 = !live ? 0 : f0 + a.frames_per_stream < a.n_frames ? f0 + a.frames_per_stream : a.n_frames;

    const float2* src = a.y + c * a.y_ch_stride + ltid;
    float2* dst = a.out + c * a.out_ch_stride + ltid;
    // conj(FFT(conj(Y))) / N, and the (-1)^n of sample n = ltid + j*TPF
    const float s_even = 1.0f / (float)N, s_odd = ((TPF & 1) && !a.natural) ? -s_even : s_even;
    const float sg = ((ltid & 1) && !a.natural) ? -1.0f : 1.0f;

    float2 acc[A > 0 ? A : 1];
#pragma unroll
    for (int j = 0; j < (A > 0 ? A : 1); ++j) acc[j] = make_float2(0.f, 0.f);
    int par = 0;

    // software pipeline: the bins of the NEXT frame are loaded while the current one is transformed
    float2 nx[E];
    auto prefetch = [&](long long m) {
        if (m >= 0 && m < f1) {
            const float2* fr = src + m * a.y_row - a.y_off;
#pragma unroll
            for (int q = 0; q < E / R0; ++q)
#pragma unroll
                for (int r = 0; r < R0; ++r) {
                    const int k = (ltid + q * TPF) + r * (N / R0);
                    if (!MASK || (k >= a.bin_lo && k < a.bin_hi))
                        nx[q * R0 + r] = __ldcs(fr + q * TPF + r * (N / R0));
                    else
                        nx[q * R0 + r] = make_float2(0.f, 0.f);      // outside the stored / kept band
                }
        } else {
#pragma unroll
            for (int e = 0; e < E; ++e) nx[e] = make_float2(0.f, 0.f);
        }
    };
    prefetch(f0 - (R - 1));

#pragma unroll 1
    for (long long m = f0 - (R - 1); m < f0 + a.frames_per_stream; ++m) {
        float2 v[E];
#pragma unroll
        for (int q = 0; q < E / R0; ++q)
#pragma unroll
            for (int r = 0; r < R0; ++r) {
                float2 z = nx[q * R0 + r];
                if (GAIN) z = cmul(z, __ldg(a.gain + (ltid + q * TPF) + r * (N / R0)));
                v[q * R0 + r] = make_float2(z.x, -z.y);
            }
        prefetch(m + 1);

        PassLoop<LOG2N, 0>::run(v, bufs, tw, nullptr, ltid, slot, par);

        // y[j]: sample ltid + j*TPF of this frame; v[q*RL + r] is position j = q + r*(E/RL)
        float2 s[E];
#pragma unroll
        for (int q = 0; q < E / RL; ++q)
#pragma unroll
            for (int r = 0; r < RL; ++r) {
                const int j = q + r * (E / RL);
                const float sc = sg * ((j & 1) ? s_odd : s_even);
                const float2 X = v[q * RL + r];
                s[j] = make_float2(X.x * sc, -X.y * sc);
            }
#pragma unroll
        for (int j = 0; j < A; ++j) s[j] = make_float2(acc[j].x + s[j].x, acc[j].y + s[j].y);
        if (m >= f0 && m < f1) {
            float2* o = dst + m * HOP;
            const float g = a.scale;
#pragma unroll
            for (int j = 0; j < H; ++j) __stcs(o + j * TPF, make_float2(s[j].x * g, s[j].y * g));
            if (m == a.n_frames - 1) {      // the tail of the last frame: noverlap more samples
#pragma unroll
                for (int j = 0; j < A; ++j) __stcs(o + (j + H) * TPF, make_float2(s[j + H].x * g, s[j + H].y * g));
            }
        }
#pragma unroll
        for (int j = 0; j < A; ++j) acc[j] = s[j + H];
    }
}

// ---- ola_filter in one kernel: frame gather * window -> FFT -> band mask -> inverse FFT ->
// overlap-add.  The STFT never exists in memory: 8 B read + 8 B written per sample instead of the
// 48 B of the stft + istft chain (and the ~150 B of the reference's materialising steps).  The
// forward passes leave bin ltid + j*TPF in register slot (j % (E/RL))*RL + j/(E/RL); the inverse
// passes want it in slot (j % (E/R0))*R0 + j/(E/R0): a compile-time renaming, no data moves.
struct OlaArgs {
    const float2* x;
    long long n_samples, x_ch_stride;
    int n_channels;
    const float* window;
    long long n_frames;
    int bin_lo, bin_hi;
    float2* out;
    long long out_ch_stride;
    const float2* twiddle;
    long long streams_per_ch, frames_per_stream;
};

template <int LOG2N, int LOG2R>
__global__ void __launch_bounds__(StftCfg<LOG2N>::THREADS, StftCfg<LOG2N>::MIN_BLOCKS)
ola_kernel(const OlaArgs a) {
    using C = StftCfg<LOG2N>;
    constexpr int N = C::N, E = C::E, TPF = C::TPF, FPC = C::FPC;
    constexpr int R0 = plan_radix(LOG2N, 0);
    constexpr int RL = plan_radix(LOG2N, C::NP - 1);
    constexpr int R = 1 << LOG2R;
    constexpr int H = E / R, A = E - H;
    constexpr long long HOP = N / R;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* tw = reinterpret_cast<float2*>(smem_raw);
    float2* bufs = tw + C::TW_ALLOC;
    for (int i = threadIdx.x; i < C::TW; i += C::THREADS) tw[i] = a.twiddle[i];
    __syncthreads();

    const int slot = threadIdx.x / TPF;
    const int ltid = threadIdx.x % TPF;
    const long long sid = (long long)blockIdx.x * FPC + slot;
    const bool live = sid < a.streams_per_ch * a.n_channels;
    const long long c = live ? sid / a.streams_per_ch : 0;
    const long long f0 = live ? (sid - c * a.streams_per_ch) * a.frames_per_stream : 0;
    const long long f1 = !live ? 0 : f0 + a.frames_per_stream < a.n_frames ? f0 + a.frames_per_stream : a.n_frames;

    // window coefficient of sample ltid + j*TPF, in the register order of the forward loads
    float w[E];
#pragma unroll
    for (int q = 0; q < E / R0; ++q)
#pragma unroll
        for (int r = 0; r < R0; ++r) w[q * R0 + r] = __ldg(a.window + (ltid + q * TPF) + r * (N / R0));

    const float2* src = a.x + c * a.x_ch_stride + ltid;
    float2* dst = a.out + c * a.out_ch_stride + ltid;
    const float s_even = 1.0f / (float)N, s_odd = (TPF & 1) ? -s_even : s_even;
    const float sg = (ltid & 1) ? -1.0f : 1.0f;

    float2 acc[A > 0 ? A : 1];
#pragma unroll
    for (int j = 0; j < (A > 0 ? A : 1); ++j) acc[j] = make_float2(0.f, 0.f);
    int par = 0;

    // software pipeline: the samples of the NEXT frame are loaded while the current one is processed
    float2 nx[E];
    auto prefetch = [&](long long m) {
        if (m >= 0 && m < f1) {
            const float2* fr = src + m * HOP;
#pragma unroll
            for (int q = 0; q < E / R0; ++q)
#pragma unroll
                for (int r = 0; r < R0; ++r) nx[q * R0 + r] = __ldg(fr + q * TPF + r * (N / R0));
        } else {
#pragma unroll
            for (int e = 0; e < E; ++e) nx[e] = make_float2(0.f, 0.f);
        }
    };
    prefetch(f0 - (R - 1));

#pragma unroll 1
    for (long long m = f0 - (R - 1); m < f0 + a.frames_per_stream; ++m) {
        float2 v[E];
#pragma unroll
        for (int e = 0; e < E; ++e) v[e] = cscale(nx[e], w[e]);
        prefetch(m + 1);
        PassLoop<LOG2N, 0>::run(v, bufs, tw, nullptr, ltid, slot, par);

        // band mask, conjugate, and rename into the load order of the inverse transform
        float2 u[E];
#pragma unroll
        for (int q = 0; q < E / RL; ++q)
#pragma unroll
            for (int r = 0; r < RL; ++r) {
                const int j = q + r * (E / RL);
                const int k = ltid + j * TPF;
                float2 X = v[q * RL + r];
                if (k < a.bin_lo || k >= a.bin_hi) X = make_float2(0.f, 0.f);
                u[(j % (E / R0)) * R0 + j / (E / R0)] = make_float2(X.x, -X.y);
            }
        // (the inverse transform continues the ping-pong parity of the exchange buffers: the
        // buffer its first exchange writes was last read before the forward transform's last barrier)
        PassLoop<LOG2N, 0>::run(u, bufs, tw, nullptr, ltid, slot, par);

        float2 s[E];
#pragma unroll
        for (int q = 0; q < E / RL; ++q)
#pragma unroll
            for (int r = 0; r < RL; ++r) {
                const int j = q + r * (E / RL);
                const float sc = sg * ((j & 1) ? s_odd : s_even);
                const float2 X = u[q * RL + r];
                s[j] = make_float2(X.x * sc, -X.y * sc);
            }
#pragma unroll
        for (int j = 0; j < A; ++j) s[j] = make_float2(acc[j].x + s[j].x, acc[j].y + s[j].y);
        if (m >= f0 && m < f1) {
            float2* o = dst + m * HOP;
#pragma unroll
            for (int j = 0; j < H; ++j) __stcs(o + j * TPF, s[j]);
            if (m == a.n_frames - 1) {
#pragma unroll
                for (int j = 0; j < A; ++j) __stcs(o + (j + H) * TPF, s[j + H]);
            }
        }
#pragma unroll
        for (int j = 0; j < A; ++j) acc[j] = s[j + H];
    }
}

template <int LOG2N, int LOG2R>
static int launch_ola_r(OlaArgs a, cudaStream_t stream) {
    if constexpr ((1 << LOG2R) > plan_elems(LOG2N)) {
        return fail(IQW_ERR_UNSUPPORTED, "ola: nfft/hop = %d is larger than %d for nfft = %d", 1 << LOG2R,
                    plan_elems(LOG2N), 1 << LOG2N);
    } else {
        using C = StftCfg<LOG2N>;
        auto kern = ola_kernel<LOG2N, LOG2R>;
        long long ctas = 0;
        if (int rc = resident_ctas(kern, C::THREADS, C::SMEM, "ola kernel", &ctas)) return rc;
        constexpr int R = 1 << LOG2R;
        long long streams = ctas * C::FPC;
        long long per_ch = streams / a.n_channels > 0 ? streams / a.n_channels : 1;
        const long long most = (a.n_frames + 16 * R - 1) / (16 * R);
        if (per_ch > most) per_ch = most;
        a.streams_per_ch = per_ch;
        a.frames_per_stream = (a.n_frames + per_ch - 1) / per_ch;
        const long long grid = (per_ch * a.n_channels + C::FPC - 1) / C::FPC;
        { IQW_PROFILE("ola_kernel", stream); kern<<<(unsigned)grid, C::THREADS, C::SMEM, stream>>>(a); }
        IQW_CUDA_OK(cudaGetLastError());
        return IQW_OK;
    }
}

template <int LOG2N, int LOG2R, bool MASK, bool GAIN>
static int launch_istft_r(IstftArgs a, cudaStream_t stream) {
    using C = StftCfg<LOG2N>;
    auto kern = istft_kernel<LOG2N, LOG2R, MASK, GAIN>;
    long long ctas = 0;
    if (int rc = resident_ctas(kern, C::THREADS, C::SMEM, "istft kernel", &ctas)) return rc;
    constexpr int R = 1 << LOG2R;
    // one frame range ("stream") per slot of the resident grid, but ranges of at least 16*R frames
    // so that the R-1 warm-up frames of a range stay a few per cent
    long long streams = ctas * C::FPC;
    long long per_ch = streams / a.n_channels > 0 ? streams / a.n_channels : 1;
    const long long most = (a.n_frames + 16 * R - 1) / (16 * R);
    if (per_ch > most) per_ch = most;
    a.streams_per_ch = per_ch;
    a.frames_per_stream = (a.n_frames + per_ch - 1) / per_ch;
    const long long total = per_ch * a.n_channels;
    const long long grid = (total + C::FPC - 1) / C::FPC;
    { IQW_PROFILE("istft_kernel", stream); kern<<<(unsigned)grid, C::THREADS, C::SMEM, stream>>>(a); }
    IQW_CUDA_OK(cudaGetLastError());
    return IQW_OK;
}

template <int LOG2N, int LOG2R>
static int launch_istft_m(const IstftArgs& a, cudaStream_t s) {
    if constexpr ((1 << LOG2R) > plan_elems(LOG2N)) {
        return fail(IQW_ERR_UNSUPPORTED, "istft: nfft/hop = %d is larger than %d for nfft = %d", 1 << LOG2R,
                    plan_elems(LOG2N), 1 << LOG2N);
    } else {
        const bool full = a.bin_lo == 0 && a.bin_hi == (1 << LOG2N);
        if (a.gain) return full ? launch_istft_r<LOG2N, LOG2R, false, true>(a, s) : launch_istft_r<LOG2N, LOG2R, true, true>(a, s);
        return full ? launch_istft_r<LOG2N, LOG2R, false, false>(a, s) : launch_istft_r<LOG2N, LOG2R, true, false>(a, s);
    }
}

}  // namespace iqw

using namespace iqw;

static int istft_entry(const void* d_y, int64_t n_channels, int64_t n_frames, int64_t y_channel_stride,
                       int32_t nfft, int64_t hop, int32_t bin_lo, int32_t bin_hi, int32_t y_bins,
                       const void* d_bin_gain, float scale, int natural, void* d_out,
                       int64_t out_channel_stride, void* stream) {
    if (!d_y || !d_out) return fail(IQW_ERR_INVALID, "null pointer argument");
    const int log2n = log2_exact(nfft);
    if (log2n < 1) return fail(IQW_ERR_UNSUPPORTED, "nfft=%d: only powers of two are built", nfft);
    if (log2n < 4 || log2n > 13)
        return fail(IQW_ERR_UNSUPPORTED, "istft: nfft=%d outside the built range 16..8192", nfft);
    const int log2r = hop >= 1 && hop <= nfft && nfft % hop == 0 ? log2_exact(nfft / hop) : -1;
    if (log2r < 0) return fail(IQW_ERR_UNSUPPORTED, "istft: hop=%lld: nfft/hop must be 1, 2, 4, 8 or 16", (long long)hop);
    if (n_channels < 1 || n_frames < 1) return fail(IQW_ERR_INVALID, "istft: need at least one channel and one frame");
    if (bin_lo < 0 || bin_hi > nfft || bin_lo > bin_hi) return fail(IQW_ERR_INVALID, "istft: bad bin range");
    if (y_bins != nfft && y_bins != bin_hi - bin_lo)
        return fail(IQW_ERR_INVALID, "istft: y_bins must be nfft (whole frames stored) or bin_hi - bin_lo (band only)");
    if (y_bins < 1) return fail(IQW_ERR_INVALID, "istft: empty band");
    if (y_channel_stride < n_frames * y_bins || out_channel_stride < n_frames * hop + (nfft - hop))
        return fail(IQW_ERR_INVALID, "istft: channel stride smaller than a channel");
    cudaStream_t s = (cudaStream_t)stream;
    IstftArgs a;
    a.y = (const float2*)d_y; a.y_ch_stride = y_channel_stride; a.n_channels = (int)n_channels;
    a.n_frames = n_frames; a.bin_lo = bin_lo; a.bin_hi = bin_hi;
    a.y_row = y_bins; a.y_off = y_bins == nfft ? 0 : bin_lo;
    a.gain = (const float2*)d_bin_gain; a.scale = scale; a.natural = natural;
    a.out = (float2*)d_out; a.out_ch_stride = out_channel_stride;
    a.streams_per_ch = a.frames_per_stream = 0;
    if (int rc = get_twiddles(log2n, s, &a.twiddle)) return rc;
    return dispatch<4, 13>(
        log2n,
        [&](auto L) {
            return dispatch<0, 4>(log2r, [&](auto R) { return launch_istft_m<L, R>(a, s); }, [&] {
                return fail(IQW_ERR_UNSUPPORTED, "istft: nfft/hop = %d: only 1, 2, 4, 8, 16 are built", 1 << log2r);
            });
        },
        [&] { return fail(IQW_ERR_UNSUPPORTED, "istft: nfft=%d", nfft); });
}

extern "C" int iqw_istft_c64(const void* d_y, int64_t n_channels, int64_t n_frames, int64_t y_channel_stride,
                             int32_t nfft, int64_t hop, int32_t bin_lo, int32_t bin_hi, int32_t y_bins,
                             const void* d_bin_gain, float scale, void* d_out, int64_t out_channel_stride,
                             void* stream) {
    iqw::DeviceGuard _dev_guard(d_y);
    return istft_entry(d_y, n_channels, n_frames, y_channel_stride, nfft, hop, bin_lo, bin_hi, y_bins,
                       d_bin_gain, scale, 0, d_out, out_channel_stride, stream);
}

// plain batched inverse DFT (1/nfft normalised, natural bin order in, natural sample order out):
// kernel 4 with hop = nfft (nothing to overlap-add) and without the (-1)^n of the baked-in shift
extern "C" int iqw_ifft_c64(const void* d_y, int64_t n_rows, int32_t nfft, void* d_out, void* stream) {
    iqw::DeviceGuard _dev_guard(d_y);
    if (n_rows < 1) return fail(IQW_ERR_INVALID, "ifft: need at least one row");
    return istft_entry(d_y, 1, n_rows, n_rows * (int64_t)nfft, nfft, nfft, 0, nfft, nfft, nullptr, 1.0f, 1,
                       d_out, n_rows * (int64_t)nfft, stream);
}

extern "C" int iqw_ola_filter_c64(const void* d_x, int64_t n_channels, int64_t n_samples, int64_t x_channel_stride,
                                  const float* d_window, int32_t nfft, int64_t hop, int64_t n_frames,
                                  int32_t bin_lo, int32_t bin_hi, void* d_out, int64_t out_channel_stride,
                                  void* stream) {
    iqw::DeviceGuard _dev_guard(d_x);
    if (!d_x || !d_out || !d_window) return fail(IQW_ERR_INVALID, "null pointer argument");
    const int log2n = log2_exact(nfft);
    if (log2n < 1) return fail(IQW_ERR_UNSUPPORTED, "nfft=%d: only powers of two are built", nfft);
    if (log2n < 4 || log2n > 13)
        return fail(IQW_ERR_UNSUPPORTED, "ola_filter: nfft=%d outside the built range 16..8192", nfft);
    const int log2r = hop >= 1 && hop <= nfft && nfft % hop == 0 ? log2_exact(nfft / hop) : -1;
    if (log2r < 0)
        return fail(IQW_ERR_UNSUPPORTED, "ola_filter: hop=%lld: nfft/hop must be 1, 2, 4, 8 or 16", (long long)hop);
    if (n_channels < 1 || n_frames < 1) return fail(IQW_ERR_INVALID, "ola_filter: need at least one channel and one frame");
    if ((n_frames - 1) * hop + nfft > n_samples) return fail(IQW_ERR_INVALID, "ola_filter: frames run past the samples");
    if (bin_lo < 0 || bin_hi > nfft || bin_lo > bin_hi) return fail(IQW_ERR_INVALID, "ola_filter: bad bin range");
    if (x_channel_stride < n_samples || out_channel_stride < n_frames * hop + (nfft - hop))
        return fail(IQW_ERR_INVALID, "ola_filter: channel stride smaller than a channel");
    cudaStream_t s = (cudaStream_t)stream;
    OlaArgs a;
    a.x = (const float2*)d_x; a.n_samples = n_samples; a.x_ch_stride = x_channel_stride; a.n_channels = (int)n_channels;
    a.window = d_window; a.n_frames = n_frames; a.bin_lo = bin_lo; a.bin_hi = bin_hi;
    a.out = (float2*)d_out; a.out_ch_stride = out_channel_stride;
    a.streams_per_ch = a.frames_per_stream = 0;
    if (int rc = get_twiddles(log2n, s, &a.twiddle)) return rc;
    return dispatch<4, 13>(
        log2n,
        [&](auto L) {
            return dispatch<0, 4>(log2r, [&](auto R) { return launch_ola_r<L, R>(a, s); }, [&] {
                return fail(IQW_ERR_UNSUPPORTED, "ola: nfft/hop = %d: only 1, 2, 4, 8, 16 are built", 1 << log2r);
            });
        },
        [&] { return fail(IQW_ERR_UNSUPPORTED, "ola_filter: nfft=%d", nfft); });
}
