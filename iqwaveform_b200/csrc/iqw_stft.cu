// iqw_stft.cu -- kernel 1: fused overlapped-frame gather * window -> FFT -> |X|^2 / dB -> trim.
//
// One pass over the samples replaces the reference's five materialising steps
// (/root/reference/src/iqwaveform/):
//   fourier.py:568-581   sliding_window_view + multiply   (writes (T, nfft) complex64)
//   fourier.py:1044      fft (scipy.fft / cuFFT), in place
//   power_analysis.py:254-255   abs, square                (writes (T, nfft) float32)
//   power_analysis.py:199-204   abs, += eps, log10, *= 10  (4 passes)
//   fourier.py:1295      band slice
//
// Work decomposition: a CTA owns FPC frame slots of TPF = nfft/E threads each; thread `ltid` of a
// slot holds E = 16 (8 for nfft 32/64) complex values in registers.  A persistent grid walks a
// contiguous range of frame groups per CTA so that the overlapped half of consecutive frames is
// re-read from L1/L2, never from HBM.  Between passes the values are exchanged through padded
// ping-pong shared-memory buffers; the per-pass twiddle tables live in shared memory, laid out
// [r][i] so that a warp reads consecutive entries.
#include "iqw_stft.cuh"

namespace iqw {

// FULLBAND: every bin is stored (bin_lo == 0, bin_hi == nfft), so the per-bin range checks vanish
// MODE == kStftReduce: the 48-64 accumulator registers per thread leave room for one CTA per SM only
// (measured on the plain kernel: one CTA per SM costs 6 %), but no spectrogram is written at all
template <int LOG2N, int MODE, bool FULLBAND>
__global__ void __launch_bounds__(StftCfg<LOG2N>::THREADS, MODE == kStftReduce ? 1 : StftCfg<LOG2N>::MIN_BLOCKS)
stft_kernel(const StftArgs a) {
    using C = StftCfg<LOG2N>;
    constexpr int N = C::N, E = C::E, TPF = C::TPF, FPC = C::FPC;
    constexpr int R0 = plan_radix(LOG2N, 0);
    constexpr int RL = plan_radix(LOG2N, C::NP - 1);

    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* tw = reinterpret_cast<float2*>(smem_raw);
    float2* bufs = tw + C::TW_ALLOC;

    for (int i = threadIdx.x; i < C::TW; i += C::THREADS) tw[i] = a.twiddle[i];

    const int slot = threadIdx.x / TPF;
    const int ltid = threadIdx.x % TPF;

    // window coefficients of the samples this thread loads, kept in registers for every frame
    float w[E];
#pragma unroll
    for (int q = 0; q < E / R0; ++q)
#pragma unroll
        for (int r = 0; r < R0; ++r) w[q * R0 + r] = __ldg(a.window + (ltid + q * TPF) + r * (N / R0));

    __syncthreads();

    // contiguous range of frame groups for this CTA
    const long long per = (a.n_groups + gridDim.x - 1) / gridDim.x;
    const long long g_begin = per * blockIdx.x;
    const long long g_end = g_begin + per < a.n_groups ? g_begin + per : a.n_groups;
    const int nbins = a.bin_hi - a.bin_lo;
    int par = 0;

    // running statistics of the bins this thread owns (kStftReduce): max, min and a two-level sum (the
    // inner sum runs over 32 frames, the outer over the inner sums, so that thousands of frames add up
    // with the rounding error of a few dozen additions)
    constexpr int EA = MODE == kStftReduce ? E : 1;
    float acc_mx[EA], acc_mn[EA], acc_s[EA], acc_big[EA];
#pragma unroll
    for (int e = 0; e < EA; ++e) { acc_mx[e] = -INFINITY; acc_mn[e] = INFINITY; acc_s[e] = 0.f; acc_big[e] = 0.f; }
    int acc_n = 0;

    // (channel, frame group) of g_begin, then advanced incrementally: no 64-bit divisions in the loop
    long long c_nx = g_begin / a.groups_per_ch;
    long long gc_nx = g_begin - c_nx * a.groups_per_ch;

    // software pipeline: the samples of the NEXT frame group are loaded into registers while the
    // current one is transformed (they are only multiplied by the window when their turn comes)
    float2 nx[E];
    auto prefetch = [&](long long g) {
        const long long frame = gc_nx * FPC + slot;
        if (g < g_end && frame < a.n_frames) {
            const float2* src = a.x + c_nx * a.x_ch_stride + frame * a.hop + ltid;
#pragma unroll
            for (int q = 0; q < E / R0; ++q)
#pragma unroll
                for (int r = 0; r < R0; ++r) nx[q * R0 + r] = __ldg(src + q * TPF + r * (N / R0));
        }       // (a slot past the last frame keeps stale values: its results are never stored)
    };
#pragma unroll
    for (int e = 0; e < E; ++e) nx[e] = make_float2(0.f, 0.f);
    prefetch(g_begin);

    for (long long g = g_begin; g < g_end; ++g) {
        const long long c = c_nx;
        const long long frame = gc_nx * FPC + slot;
        const bool valid = frame < a.n_frames;
        if (++gc_nx == a.groups_per_ch) { gc_nx = 0; ++c_nx; }

        float2 v[E];
#pragma unroll
        for (int e = 0; e < E; ++e) v[e] = cscale(nx[e], w[e]);
        prefetch(g + 1);

        PassLoop<LOG2N, 0>::run(v, bufs, tw, nullptr, ltid, slot, par);

        if constexpr (MODE == kStftReduce) {
            if (valid) {
                float p[E];
#pragma unroll
                for (int e = 0; e < E; ++e) p[e] = v[e].x * v[e].x + v[e].y * v[e].y;
                if (a.reduce_flags & 1) {
#pragma unroll
                    for (int e = 0; e < E; ++e) { acc_mx[e] = fmaxf(acc_mx[e], p[e]); acc_mn[e] = fminf(acc_mn[e], p[e]); }
                }
                if (a.reduce_flags & 2) {
                    if (a.reduce_dB) {
                        // branch-free dB of the 16 values (independent MUFU chains); an argument that needs
                        // log10f (zero, denormal, inf, nan) is rare and patched behind one branch per frame
                        bool all_ok = true;
                        float d[E];
#pragma unroll
                        for (int e = 0; e < E; ++e) {
                            bool ok;
                            d[e] = power_to_dB_fast(fabsf(p[e]) + a.eps, ok);
                            all_ok &= ok;
                        }
                        if (!all_ok) {
#pragma unroll
                            for (int e = 0; e < E; ++e)
                                if (!dB_fast_ok(fabsf(p[e]) + a.eps)) d[e] = power_to_dB_slow(fabsf(p[e]) + a.eps);
                        }
#pragma unroll
                        for (int e = 0; e < E; ++e) acc_s[e] += d[e];
                    } else {
#pragma unroll
                        for (int e = 0; e < E; ++e) acc_s[e] += p[e];
                    }
                    if (++acc_n == 32) {
                        acc_n = 0;
#pragma unroll
                        for (int e = 0; e < E; ++e) { acc_big[e] += acc_s[e]; acc_s[e] = 0.f; }
                    }
                }
            }
        } else if (valid) {
            const long long row = c * a.out_ch_stride + frame * (long long)nbins - a.bin_lo;
#pragma unroll
            for (int q = 0; q < E / RL; ++q)
#pragma unroll
                for (int r = 0; r < RL; ++r) {
                    const int k = (ltid + q * TPF) + r * (N / RL);
                    if (FULLBAND || (k >= a.bin_lo && k < a.bin_hi)) {
                        const float2 X = v[q * RL + r];
                        if constexpr (MODE == IQW_STFT_COMPLEX) {
                            __stcs(reinterpret_cast<float2*>(a.out) + row + k, X);
                        } else {
                            float p = X.x * X.x + X.y * X.y;
                            if constexpr (MODE == IQW_STFT_DB) p = power_to_dB(p, a.eps);
                            __stcs(reinterpret_cast<float*>(a.out) + row + k, p);
                        }
                    }
                }
        }
        // no trailing barrier needed: the ping-pong parity keeps an exchange buffer from being
        // rewritten before every thread has passed the barrier that follows its last read
        if constexpr (C::NP == 1) { /* no shared memory exchange at all */ }
    }
    if constexpr (MODE == kStftReduce) {
        // one partial row per frame slot of the grid (slots that saw no frame write the neutral elements)
        const long long part = ((long long)blockIdx.x * FPC + slot) * N;
#pragma unroll
        for (int q = 0; q < E / RL; ++q)
#pragma unroll
            for (int r = 0; r < RL; ++r) {
                const int k = (ltid + q * TPF) + r * (N / RL);
                const int e = q * RL + r;
                a.part_max[part + k] = acc_mx[e];
                a.part_min[part + k] = acc_mn[e];
                a.part_sum[part + k] = (double)acc_big[e] + (double)acc_s[e];
            }
    }
}

// max / min / sum over the partial rows of one channel, then the named statistics of the request
// (fourier.py:1322-1325: np.max / np.min / np.mean over the time axis of the (dB) spectrogram).  dB is
// monotone, so max and min are taken on the power and converted once.
struct ReducePlan { int n_stats; int kind[16]; };
__global__ void stft_reduce_combine_kernel(const float* __restrict__ pmax, const float* __restrict__ pmin,
                                           const double* __restrict__ psum, int n_parts, int nfft, int bin_lo,
                                           int bin_hi, long long n_frames, ReducePlan st, int to_dB, float eps,
                                           float* __restrict__ out /* [n_stats][bin_hi - bin_lo] */) {
    const int k = bin_lo + blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= bin_hi) return;
    float mx = -INFINITY, mn = INFINITY;
    double sum = 0.0;
    for (int p = 0; p < n_parts; ++p) {
        mx = fmaxf(mx, pmax[(long long)p * nfft + k]);
        mn = fminf(mn, pmin[(long long)p * nfft + k]);
        sum += psum[(long long)p * nfft + k];
    }
    const int nb = bin_hi - bin_lo;
    for (int t = 0; t < st.n_stats; ++t) {
        float r;
        if (st.kind[t] == IQW_STAT_MEAN) r = (float)(sum / (double)n_frames);
        else if (st.kind[t] == IQW_STAT_MAX) r = to_dB ? power_to_dB(mx, eps) : mx;
        else r = to_dB ? power_to_dB(mn, eps) : mn;
        out[(long long)t * nb + (k - bin_lo)] = r;
    }
}

// ---------------------------------------------------------------------------------------------
// twiddle tables: one immutable table per (device, log2 nfft), built on first use in float64
// ---------------------------------------------------------------------------------------------
__global__ void twiddle_init_kernel(float2* tw, int log2n) {
    const int np = plan_passes(log2n);
    for (int p = 1; p < np; ++p) {
        const int R = plan_radix(log2n, p), Ns = plan_ns(log2n, p), off = plan_tw_offset(log2n, p);
        const int count = (R - 1) * Ns;
        for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < count; e += gridDim.x * blockDim.x) {
            const int r = e / Ns + 1, i = e % Ns;
            double s, c;
            sincospi(-2.0 * (double)(r * i) / (double)(Ns * R), &s, &c);
            tw[off + e] = make_float2((float)c, (float)s);
        }
    }
}

int get_twiddles(int log2n, cudaStream_t stream, const float2** out) {
    return device_table(kFftTwiddles, log2n, plan_tw_size(log2n) + 16,
                        [](float2* d, int log2n, cudaStream_t s) { twiddle_init_kernel<<<8, 256, 0, s>>>(d, log2n); },
                        stream, out);
}

template <int LOG2N, int MODE, bool FULLBAND>
static int launch_stft_band(StftArgs a, cudaStream_t stream) {
    using C = StftCfg<LOG2N>;
    auto kern = stft_kernel<LOG2N, MODE, FULLBAND>;
    long long grid = 0;
    if (int rc = resident_ctas(kern, C::THREADS, C::SMEM, "stft kernel", &grid)) return rc;
    a.groups_per_ch = (a.n_frames + C::FPC - 1) / C::FPC;
    a.n_groups = a.groups_per_ch * a.n_channels;
    if (grid > a.n_groups) grid = a.n_groups;
    { IQW_PROFILE("stft_kernel", stream); kern<<<(unsigned)grid, C::THREADS, C::SMEM, stream>>>(a); }
    IQW_CUDA_OK(cudaGetLastError());
    return IQW_OK;
}

template <int LOG2N, int MODE>
static int launch_stft(const StftArgs& a, cudaStream_t stream) {
    if (a.bin_lo == 0 && a.bin_hi == (1 << LOG2N)) return launch_stft_band<LOG2N, MODE, true>(a, stream);
    return launch_stft_band<LOG2N, MODE, false>(a, stream);
}

template <int LOG2N>
static int launch_stft_reduce(StftArgs a, const ReducePlan& st, float* out, void* ws, size_t ws_bytes, cudaStream_t stream) {
    using C = StftCfg<LOG2N>;
    auto kern = stft_kernel<LOG2N, kStftReduce, true>;
    long long grid = 0;
    if (int rc = resident_ctas(kern, C::THREADS, C::SMEM, "stft reduce kernel", &grid)) return rc;
    a.n_channels = 1;
    a.groups_per_ch = (a.n_frames + C::FPC - 1) / C::FPC;
    a.n_groups = a.groups_per_ch;
    if (grid > a.n_groups) grid = a.n_groups;
    const long long n_parts = grid * C::FPC;
    const size_t need = (size_t)n_parts * C::N * (2 * sizeof(float) + sizeof(double));
    if (!ws || ws_bytes < need) return fail(IQW_ERR_WORKSPACE, "stft reduce workspace %zu bytes < required %zu", ws_bytes, need);
    a.part_sum = static_cast<double*>(ws);
    a.part_max = reinterpret_cast<float*>(a.part_sum + n_parts * C::N);
    a.part_min = a.part_max + n_parts * C::N;
    { IQW_PROFILE("stft_reduce_kernel", stream); kern<<<(unsigned)grid, C::THREADS, C::SMEM, stream>>>(a); }
    IQW_CUDA_OK(cudaGetLastError());
    const int nb = a.bin_hi - a.bin_lo;
    { IQW_PROFILE_FINE("stft_reduce_combine", stream);
      stft_reduce_combine_kernel<<<(nb + 127) / 128, 128, 0, stream>>>(a.part_max, a.part_min, a.part_sum, (int)n_parts, C::N,
                                                                       a.bin_lo, a.bin_hi, a.n_frames, st, a.reduce_dB, a.eps, out); }
    IQW_CUDA_OK(cudaGetLastError());
    return IQW_OK;
}

// nfft 1024 / 2048 / 4096 with at most two of {max, min, sum}: the warp-specialised two-pass kernel (iqw_stft2p.cu)
static int launch_stft_reduce_two_pass(StftArgs a, int log2n, const ReducePlan& st, float* out, void* ws, size_t ws_bytes,
                                       cudaStream_t stream, bool* done) {
    *done = false;
    if (stft_variant() == 1 || log2n < 10 || log2n > 12) return IQW_OK;
    int flags = 0;
    for (int t = 0; t < st.n_stats; ++t)
        flags |= st.kind[t] == IQW_STAT_MAX ? 1 : st.kind[t] == IQW_STAT_MIN ? 2 : 4;
    int sms = 0;
    if (int rc = device_sm_count(&sms)) return rc;
    const long long N = 1ll << log2n;
    const size_t need = (size_t)sms * N * (2 * sizeof(float) + sizeof(double));
    if (!ws || ws_bytes < need) return fail(IQW_ERR_WORKSPACE, "stft reduce workspace %zu bytes < required %zu", ws_bytes, need);
    a.n_channels = 1;
    a.part_sum = static_cast<double*>(ws);
    a.part_max = reinterpret_cast<float*>(a.part_sum + (size_t)sms * N);
    a.part_min = a.part_max + (size_t)sms * N;
    long long n_parts = 0;
    const int rc = launch_stft_two_pass_reduce(a, log2n, flags, &n_parts, stream);
    if (rc == IQW_ERR_UNSUPPORTED) return IQW_OK;
    if (rc) return rc;
    const int nb = a.bin_hi - a.bin_lo;
    const int convert = a.reduce_dB;
    { IQW_PROFILE_FINE("stft_reduce_combine", stream);
      stft_reduce_combine_kernel<<<(nb + 127) / 128, 128, 0, stream>>>(a.part_max, a.part_min, a.part_sum, (int)n_parts, (int)N,
                                                                       a.bin_lo, a.bin_hi, a.n_frames, st, convert, a.eps, out); }
    IQW_CUDA_OK(cudaGetLastError());
    *done = true;
    return IQW_OK;
}

}  // namespace iqw

using namespace iqw;

// partial rows: at most (SMs * 2 CTAs) * 16 frame slots, 16 bytes per bin each
extern "C" size_t iqw_stft_reduce_workspace_bytes(int32_t nfft) {
    if (nfft < 16 || nfft > 8192 || (nfft & (nfft - 1))) return 0;
    int sms = 0;
    if (device_sm_count(&sms) != IQW_OK) sms = 160;
    return (size_t)sms * 2 * 16 * (size_t)nfft * 16;
}

extern "C" int iqw_stft_reduce_c64(const void* d_x, int64_t n_channels, int64_t n_samples, int64_t x_channel_stride,
                                   const float* d_window, int32_t nfft, int64_t hop, int64_t n_frames, int32_t to_dB,
                                   float eps, int32_t bin_lo, int32_t bin_hi, const iqw_stat* stats, int32_t n_stats,
                                   float* d_out, void* d_workspace, size_t workspace_bytes, void* stream) {
    iqw::DeviceGuard _dev_guard(d_x);
    if (!d_x || !d_window || !d_out || !stats) return fail(IQW_ERR_INVALID, "null pointer argument");
    const int log2n = log2_exact(nfft);
    if (log2n < 4 || log2n > 13)
        return fail(IQW_ERR_UNSUPPORTED, "iqw_stft_reduce_c64: nfft=%d: powers of two from 16 to 8192 are built", nfft);
    if (hop < 1 || n_channels < 1 || n_frames < 1) return fail(IQW_ERR_INVALID, "need hop, n_channels, n_frames >= 1");
    if ((n_frames - 1) * hop + nfft > n_samples)
        return fail(IQW_ERR_INVALID, "n_frames=%lld does not fit in n_samples=%lld", (long long)n_frames, (long long)n_samples);
    if (bin_lo < 0 || bin_hi > nfft || bin_lo >= bin_hi) return fail(IQW_ERR_INVALID, "bad bin range [%d, %d)", bin_lo, bin_hi);
    if (n_stats < 1 || n_stats > 16) return fail(IQW_ERR_INVALID, "1 <= n_stats <= 16");
    ReducePlan st{};
    st.n_stats = n_stats;
    for (int t = 0; t < n_stats; ++t) {
        if (stats[t].kind != IQW_STAT_MEAN && stats[t].kind != IQW_STAT_MAX && stats[t].kind != IQW_STAT_MIN)
            return fail(IQW_ERR_UNSUPPORTED, "iqw_stft_reduce_c64 takes mean / max / min only (order statistics need the spectrogram)");
        st.kind[t] = stats[t].kind;
    }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int nb = bin_hi - bin_lo;
    for (int64_t c = 0; c < n_channels; ++c) {
        StftArgs a{};
        a.x = static_cast<const float2*>(d_x) + c * x_channel_stride;
        a.n_samples = n_samples;
        a.x_ch_stride = x_channel_stride;
        a.window = d_window;
        a.hop = hop;
        a.n_frames = n_frames;
        a.eps = eps;
        a.bin_lo = bin_lo;
        a.bin_hi = bin_hi;
        a.reduce_dB = to_dB ? 1 : 0;
        for (int t = 0; t < n_stats; ++t) a.reduce_flags |= stats[t].kind == IQW_STAT_MEAN ? 2 : 1;
        if (int rc = get_twiddles(log2n, s, &a.twiddle)) return rc;
        float* out = d_out + c * (int64_t)n_stats * nb;
        bool done = false;
        if (int rc2 = launch_stft_reduce_two_pass(a, log2n, st, out, d_workspace, workspace_bytes, s, &done)) return rc2;
        if (done) continue;
        const int rc = dispatch<4, 13>(
            log2n, [&](auto L) { return launch_stft_reduce<L>(a, st, out, d_workspace, workspace_bytes, s); },
            [] { return IQW_ERR_UNSUPPORTED; });
        if (rc) return rc;
    }
    return IQW_OK;
}

extern "C" size_t iqw_stft_workspace_bytes(int32_t nfft, int64_t n_channels, int64_t n_frames) {
    const int log2n = log2_exact(nfft);
    if (log2n < 1) return 0;
    // the four-step path's scratch (also the fallback for unaligned captures) or the cluster kernels' exchange
    // scratch, whichever is larger
    const size_t four_step = stft_large_workspace_bytes(log2n, n_channels, n_frames);
    const size_t cluster = stft_three_pass_scratch_bytes(log2n, n_channels, n_frames);
    return four_step > cluster ? four_step : cluster;
}

extern "C" int iqw_stft_c64(const void* d_x, int64_t n_channels, int64_t n_samples,
                            int64_t x_channel_stride, const float* d_window, int32_t nfft,
                            int64_t hop, int64_t n_frames, int32_t mode, float eps, int32_t bin_lo,
                            int32_t bin_hi, void* d_out, int64_t out_channel_stride, void* d_workspace,
                            size_t workspace_bytes, void* stream) {
    iqw::DeviceGuard _dev_guard(d_x);
    if (!d_x || !d_window || !d_out) return fail(IQW_ERR_INVALID, "null pointer argument");
    const int log2n = log2_exact(nfft);
    if (log2n < 1) return fail(IQW_ERR_UNSUPPORTED, "nfft=%d: only powers of two are built", nfft);
    if (log2n < 4 || log2n > 16)
        return fail(IQW_ERR_UNSUPPORTED, "nfft=%d outside the built range 16..65536", nfft);
    if (hop < 1) return fail(IQW_ERR_INVALID, "hop=%lld must be >= 1", (long long)hop);
    if (n_channels < 0 || n_frames < 0) return fail(IQW_ERR_INVALID, "negative size");
    if (n_channels == 0 || n_frames == 0) return IQW_OK;
    if ((n_frames - 1) * hop + nfft > n_samples)
        return fail(IQW_ERR_INVALID, "n_frames=%lld does not fit in n_samples=%lld",
                    (long long)n_frames, (long long)n_samples);
    if (bin_lo < 0 || bin_hi > nfft || bin_lo >= bin_hi)
        return fail(IQW_ERR_INVALID, "bad bin range [%d, %d)", bin_lo, bin_hi);
    if (x_channel_stride < n_samples && n_channels > 1)
        return fail(IQW_ERR_INVALID, "x_channel_stride smaller than n_samples");
    if (out_channel_stride < n_frames * (int64_t)(bin_hi - bin_lo) && n_channels > 1)
        return fail(IQW_ERR_INVALID, "out_channel_stride too small");
    if (n_channels > 0x7fffffff) return fail(IQW_ERR_INVALID, "too many channels");

    cudaStream_t s = static_cast<cudaStream_t>(stream);
    StftArgs a{};
    a.x = static_cast<const float2*>(d_x);
    a.n_samples = n_samples;
    a.x_ch_stride = x_channel_stride;
    a.n_channels = (int)n_channels;
    a.window = d_window;
    a.hop = hop;
    a.n_frames = n_frames;
    a.eps = eps;
    a.bin_lo = bin_lo;
    a.bin_hi = bin_hi;
    a.out = d_out;
    a.out_ch_stride = out_channel_stride;
    // nfft 8192 / 16384: the one-pass kernel with the frame in one CTA's shared memory.  nfft 32768 / 65536: the
    // cluster variant of that kernel is built and correct but measured no faster than the four-step path
    // (18 % / 15 % against 19 % of the HBM peak: its exchanges, through DSMEM or through the L2, are not overlapped
    // with arithmetic at one frame per cluster), so it runs only on request (variant 3)
    if (stft_variant() != 1 && stft_three_pass_cluster_ok(a, log2n) &&
        (log2n < 15 || (stft_variant() == 3 && d_workspace && workspace_bytes >= stft_three_pass_scratch_bytes(log2n, 1, 1))))
        return launch_stft_three_pass_cluster(a, log2n, mode, d_workspace, workspace_bytes, s);
    if (log2n > 13) return launch_stft_large(a, log2n, mode, d_workspace, workspace_bytes, s);
    if (stft_two_pass_wanted(log2n)) return launch_stft_two_pass(a, log2n, mode, s);
    if (int rc = get_twiddles(log2n, s, &a.twiddle)) return rc;
    return dispatch<4, 13>(
        log2n, [&](auto L) { return dispatch_stft_mode(mode, [&](auto M) { return launch_stft<L, M>(a, s); }); },
        [&] { return fail(IQW_ERR_UNSUPPORTED, "nfft=%d", nfft); });
}
