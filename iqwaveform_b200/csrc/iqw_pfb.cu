// iqw_pfb.cu -- kernel 8: polyphase filter-bank (WOLA) analysis channelizer of complex64 rows: K adjacent
// channels of complex baseband IQ, each filtered by an L-tap real prototype h, one frame every `hop` samples.
//
//   y[m, k] = sum_{n < L} h[n] * x[m*hop + n] * W_K^((k - K/2) * (m*hop + n)),   W_K = exp(-2 pi i / K)
//
// With h zero-padded to P*K taps (P = ceil(L / K)) and K even this factors exactly into
//   u_m[r]  = (-1)^r * sum_{p < P} h[r + p*K] * x[m*hop + r + p*K]        (the fold)
//   Y_m     = FFT_K(u_m)
//   y[m, k] = Y_m[k] * W_K^(((k - K/2) * (m*hop mod K)) mod K)            (the rotation)
// since (-1)^(p*K) = 1 and W_K^((k - K/2) * p*K) = 1.  The host folds the sign into the tap table,
// taps[p*K + r] = (-1)^r * h[r + p*K] (python: _plan.pfb_taps).  The rotation references the phase to absolute
// sample time, so each column is "mix channel k to baseband, filter, keep every hop-th sample"; it is an
// integer index into a per-device table of W_K^j, and the identity when hop is a multiple of K.
//
// Geometry of kernels 4 and 7 (StftCfg / PassLoop): a frame slot of TPF = K/E threads holds E values per
// thread in registers; thread ltid folds the branches r = ltid + q*TPF + j*(K/R0) that the first FFT pass
// reads, one fused multiply-add (FFMA2) per tap and branch, the P segments in order p = 0, 1, ..., P-1.  A CTA
// walks a contiguous range of groups of FPC consecutive frames of one channel.  Each input sample belongs to
// L/hop frames; the slots of a group read overlapping spans at the same time and consecutive groups of a CTA
// re-read the span of the last ones, so those re-reads hit L1 (ld.global.nc) or, where the span outgrows it,
// L2, which holds every CTA's span many times over.  The taps are read through L1 too.
//
// Determinism: a frame's arithmetic depends only on its L samples, the taps and its global index m, never on
// where a call starts (frame_first), so time shards concatenate to the bits of one call.
#include "iqw_stft.cuh"

namespace iqw {

struct PfbArgs {
    const float2* x;
    long long x_ch_stride;
    long long x0;                  // buffer index of the first sample of local frame 0
    const float* taps;             // (P, K) folded, sign-applied taps, zero past L
    int n_taps, n_seg;             // L, P
    long long hop;
    long long frame_first;         // global index of local frame 0 (the rotation uses the global m*hop)
    long long n_frames;
    float2* out;                   // (n_channels, n_frames, K)
    long long out_ch_stride;
    const float2* twiddle;
    const float2* rot;             // W_K^j, j < K
    int n_channels;
    long long groups_per_ch, n_groups;
};

template <int LOG2N>
__global__ void __launch_bounds__(StftCfg<LOG2N>::THREADS, StftCfg<LOG2N>::MIN_BLOCKS)
pfb_kernel(const PfbArgs a) {
    using C = StftCfg<LOG2N>;
    constexpr int N = C::N, E = C::E, TPF = C::TPF, FPC = C::FPC;
    constexpr int R0 = plan_radix(LOG2N, 0);
    constexpr int RL = plan_radix(LOG2N, C::NP - 1);

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
    // taps of the last segment: its branches at or past this index are the zero padding, whose samples may
    // lie past the end of the buffer and are not read
    const int last_len = a.n_taps - (a.n_seg - 1) * N;
    const float* hp = a.taps + ltid;
    int par = 0;

    // every slot of the CTA runs the same number of iterations (the inter-pass barriers may span several
    // slots); a slot past the last frame transforms zeros and stores nothing
#pragma unroll 1
    for (long long g = g_begin; g < g_end; ++g) {
        const long long c = g / a.groups_per_ch;
        const long long frame = (g - c * a.groups_per_ch) * FPC + slot;
        const bool valid = frame < a.n_frames;

        float2 v[E];
#pragma unroll
        for (int e = 0; e < E; ++e) v[e] = make_float2(0.f, 0.f);
        if (valid) {
            const float2* src = a.x + c * a.x_ch_stride + a.x0 + frame * a.hop + ltid;
#pragma unroll 1
            for (int p = 0; p < a.n_seg - 1; ++p) {
                const float2* s = src + (long long)p * N;
                const float* h = hp + p * N;
#pragma unroll
                for (int q = 0; q < E / R0; ++q)
#pragma unroll
                    for (int r = 0; r < R0; ++r) {
                        const int o = q * TPF + r * (N / R0);
                        v[q * R0 + r] = cfma_rs(__ldg(s + o), __ldg(h + o), v[q * R0 + r]);
                    }
            }
            const int p = a.n_seg - 1;
            const float2* s = src + (long long)p * N;
            const float* h = hp + p * N;
#pragma unroll
            for (int q = 0; q < E / R0; ++q)
#pragma unroll
                for (int r = 0; r < R0; ++r) {
                    const int o = q * TPF + r * (N / R0);
                    if (ltid + o < last_len) v[q * R0 + r] = cfma_rs(__ldg(s + o), __ldg(h + o), v[q * R0 + r]);
                }
        }

        PassLoop<LOG2N, 0>::run(v, bufs, tw, nullptr, ltid, slot, par);

        if (valid) {
            // bin k = ltid + q*TPF + r*(K/RL) is in v[q*RL + r]
            const int sh = (int)(((a.frame_first + frame) * a.hop) & (N - 1));     // m*hop mod K
            float2* dst = a.out + c * a.out_ch_stride + frame * N;
#pragma unroll
            for (int q = 0; q < E / RL; ++q)
#pragma unroll
                for (int r = 0; r < RL; ++r) {
                    const int k = ltid + q * TPF + r * (N / RL);
                    float2 X = v[q * RL + r];
                    if (sh) X = cmul(X, __ldg(a.rot + (((k - N / 2) * sh) & (N - 1))));
                    __stcs(dst + k, X);
                }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// rotation table W_K^j = exp(-2 pi i j / K), j < K: one immutable table per (device, log2 K), built on first
// use in float64 and rounded once
// ---------------------------------------------------------------------------------------------
__global__ void pfb_rot_init_kernel(float2* rot, int n) {
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
        double s, c;
        sincospi(-2.0 * (double)j / (double)n, &s, &c);
        rot[j] = make_float2((float)c, (float)s);
    }
}

template <int LOG2N>
static int launch_pfb(PfbArgs a, cudaStream_t stream) {
    using C = StftCfg<LOG2N>;
    auto kern = pfb_kernel<LOG2N>;
    long long grid = 0;
    if (int rc = resident_ctas(kern, C::THREADS, C::SMEM, "pfb kernel", &grid)) return rc;
    a.groups_per_ch = (a.n_frames + C::FPC - 1) / C::FPC;
    a.n_groups = a.groups_per_ch * a.n_channels;
    if (grid > a.n_groups) grid = a.n_groups;
    { IQW_PROFILE("pfb_kernel", stream); kern<<<(unsigned)grid, C::THREADS, C::SMEM, stream>>>(a); }
    IQW_CUDA_OK(cudaGetLastError());
    return IQW_OK;
}

}  // namespace iqw

extern "C" int iqw_pfb_channelize_c64(const void* d_x, int64_t n_channels, int64_t n_in, int64_t x_channel_stride,
                                      int64_t x_first, const void* d_taps, int32_t n_taps, int32_t nfft, int32_t hop,
                                      int64_t frame_first, int64_t n_frames, void* d_out, int64_t out_channel_stride,
                                      void* stream) {
    using namespace iqw;
    const int log2n = log2_exact(nfft);
    if (log2n < 1) return fail(IQW_ERR_UNSUPPORTED, "pfb_channelize: nfft=%d: only powers of two are built", nfft);
    if (log2n < 4 || log2n > 13)
        return fail(IQW_ERR_UNSUPPORTED, "pfb_channelize: nfft=%d outside the built range 16..8192", nfft);
    if (n_taps < 1) return fail(IQW_ERR_INVALID, "pfb_channelize: n_taps=%d: need at least one tap", n_taps);
    const int n_seg = (n_taps + nfft - 1) / nfft;
    if (n_taps > 32768 || n_seg > 16)
        return fail(IQW_ERR_UNSUPPORTED, "pfb_channelize: %d taps = %d segments of nfft=%d: at most 16 segments and "
                    "32768 taps are built", n_taps, n_seg, nfft);
    if (hop < 1 || hop > nfft) return fail(IQW_ERR_INVALID, "pfb_channelize: hop=%d outside [1, nfft=%d]", hop, nfft);
    if (n_channels < 0 || n_in < 0 || n_frames < 0 || frame_first < 0 || x_first < 0)
        return fail(IQW_ERR_INVALID, "pfb_channelize: negative size or index");
    if (n_channels == 0 || n_frames == 0) return IQW_OK;
    const long long x0 = frame_first * (long long)hop - x_first;
    if (x0 < 0 || x0 + (n_frames - 1) * (long long)hop + n_taps > n_in)
        return fail(IQW_ERR_INVALID, "pfb_channelize: frames [%lld, %lld) read samples outside the buffer [%lld, %lld)",
                    (long long)frame_first, (long long)(frame_first + n_frames), (long long)x_first,
                    (long long)(x_first + n_in));
    if (!d_x || !d_taps || !d_out) return fail(IQW_ERR_INVALID, "pfb_channelize: null pointer");
    if (n_channels > 1 && (x_channel_stride < n_in || out_channel_stride < n_frames * nfft))
        return fail(IQW_ERR_INVALID, "pfb_channelize: channel stride shorter than a channel");
    if (n_channels > 0x7FFFFFFF) return fail(IQW_ERR_UNSUPPORTED, "pfb_channelize: %lld channels", (long long)n_channels);
    DeviceGuard guard(d_out);
    PfbArgs a{};
    a.x = reinterpret_cast<const float2*>(d_x);
    a.x_ch_stride = x_channel_stride;
    a.x0 = x0;
    a.taps = reinterpret_cast<const float*>(d_taps);
    a.n_taps = n_taps;
    a.n_seg = n_seg;
    a.hop = hop;
    a.frame_first = frame_first;
    a.n_frames = n_frames;
    a.out = reinterpret_cast<float2*>(d_out);
    a.out_ch_stride = out_channel_stride;
    a.n_channels = (int)n_channels;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    if (int rc = get_twiddles(log2n, s, &a.twiddle)) return rc;
    if (int rc = device_table(kPfbRotation, log2n, (size_t)1 << log2n,
                              [](float2* d, int log2n, cudaStream_t s) { pfb_rot_init_kernel<<<8, 256, 0, s>>>(d, 1 << log2n); },
                              s, &a.rot))
        return rc;
    return dispatch<4, 13>(log2n, [&](auto L) { return launch_pfb<L>(a, s); },
                           [&] { return fail(IQW_ERR_UNSUPPORTED, "pfb_channelize: nfft=%d", nfft); });
}

// =============================================================================================
// kernel 9: polyphase synthesis bank, the adjoint of kernel 8 with a synthesis prototype g (Lg taps):
//
//   xr[t] = sum_m sum_k g[t - m*hop] * y[m, k] * W_K^(-(k - K/2) * t),   0 <= t - m*hop < Lg
//
// factored exactly (K even) into
//   Y'_m[k] = y[m, k] * conj(W_K^(((k - K/2) * (m*hop mod K)) mod K))       (unrotate, kernel 8's table)
//   u_m     = K * IFFT_K(Y'_m) = conj(FFT_K(conj(Y'_m)))                      (no 1/K)
//   xr[t]   = sum_m gs[t - m*hop] * u_m[(t - m*hop) mod K],  m ascending       (unfold)
// with gs = _plan.pfb_taps(g, K), the table kernel 8 folds with ((-1)^r applied).  Two kernels: the first
// writes u to a caller-owned workspace, the second sums each output from the frames that cover it.  Both
// depend only on y[m], the global m and the taps, never on where a call starts, so time shards concatenate
// to the bits of one call at any hop.
// =============================================================================================
namespace iqw {

struct PfbUnrotateArgs {
    const float2* y;               // (n_channels, n_frames, K) frames, channel stride y_ch_stride
    long long y_ch_stride;
    long long frame_first;         // global index of local frame 0
    long long n_frames;
    long long hop;
    float2* u;                     // (n_channels, n_frames, K), contiguous
    const float2* twiddle;
    const float2* rot;             // W_K^j, j < K (conjugated at the point of use)
    int n_channels;
    long long groups_per_ch, n_groups;
};

// u_m = conj(FFT_K(conj(y_m * conj(W)))) = conj(FFT_K(conj(y_m) * W)): the unrotation and the first conjugate
// are one complex multiply per bin
template <int LOG2N>
__global__ void __launch_bounds__(StftCfg<LOG2N>::THREADS, StftCfg<LOG2N>::MIN_BLOCKS)
pfb_unrotate_ifft_kernel(const PfbUnrotateArgs a) {
    using C = StftCfg<LOG2N>;
    constexpr int N = C::N, E = C::E, TPF = C::TPF, FPC = C::FPC;
    constexpr int R0 = plan_radix(LOG2N, 0);
    constexpr int RL = plan_radix(LOG2N, C::NP - 1);

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
    int par = 0;

    // every slot of the CTA runs the same number of iterations (the inter-pass barriers may span several
    // slots); a slot past the last frame transforms zeros and stores nothing
#pragma unroll 1
    for (long long g = g_begin; g < g_end; ++g) {
        const long long c = g / a.groups_per_ch;
        const long long frame = (g - c * a.groups_per_ch) * FPC + slot;
        const bool valid = frame < a.n_frames;

        float2 v[E];
        if (valid) {
            // bin k = ltid + q*TPF + r*(K/R0) goes to v[q*R0 + r], the order the first pass reads
            const int sh = (int)(((a.frame_first + frame) * a.hop) & (N - 1));     // m*hop mod K
            const float2* src = a.y + c * a.y_ch_stride + frame * N;
#pragma unroll
            for (int q = 0; q < E / R0; ++q)
#pragma unroll
                for (int r = 0; r < R0; ++r) {
                    const int k = ltid + q * TPF + r * (N / R0);
                    const float2 Y = __ldcs(src + k);
                    const float2 Yc = make_float2(Y.x, -Y.y);
                    v[q * R0 + r] = sh ? cmul(Yc, __ldg(a.rot + (((k - N / 2) * sh) & (N - 1)))) : Yc;
                }
        } else {
#pragma unroll
            for (int e = 0; e < E; ++e) v[e] = make_float2(0.f, 0.f);
        }

        PassLoop<LOG2N, 0>::run(v, bufs, tw, nullptr, ltid, slot, par);

        if (valid) {
            // sample j = ltid + q*TPF + r*(K/RL) is in v[q*RL + r]
            float2* dst = a.u + (c * a.n_frames + frame) * N;
#pragma unroll
            for (int q = 0; q < E / RL; ++q)
#pragma unroll
                for (int r = 0; r < RL; ++r) {
                    const float2 X = v[q * RL + r];
                    dst[ltid + q * TPF + r * (N / RL)] = make_float2(X.x, -X.y);
                }
        }
    }
}

struct PfbUnfoldArgs {
    const float2* u;               // (n_channels, n_frames, K) from pfb_unrotate_ifft_kernel
    long long frame_first, n_frames, n_frames_total;
    const float* taps;             // gs, (P, K) folded, sign-applied, zero past Lg
    int n_taps;
    int log2n;
    int hop;
    long long out_first, n_out;
    float2* out;                   // (n_channels, n_out), channel stride out_ch_stride
    long long out_ch_stride;
    long long tiles_per_ch, n_tiles;
};

constexpr int kUnfoldThreads = 256;

// one output per thread: a CTA takes a tile of kUnfoldThreads consecutive outputs of one channel, so the lanes
// of a warp read consecutive taps and consecutive samples of each frame they share
__global__ void __launch_bounds__(kUnfoldThreads) pfb_unfold_kernel(const PfbUnfoldArgs a) {
    const int K = 1 << a.log2n;
    const long long hop = a.hop;
#pragma unroll 1
    for (long long tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        const long long c = tile / a.tiles_per_ch;
        const long long j0 = (tile - c * a.tiles_per_ch) * kUnfoldThreads;
        const long long j = j0 + threadIdx.x;
        if (j >= a.n_out) continue;
        const long long t0 = a.out_first + j0;
        const long long m0 = t0 / hop;                                   // one 64-bit division per tile
        const int d = (int)(t0 - m0 * hop) + threadIdx.x;
        const long long t = t0 + threadIdx.x;
        long long m_hi = m0 + d / a.hop;                                  // floor(t / hop)
        if (m_hi > a.n_frames_total - 1) m_hi = a.n_frames_total - 1;
        const long long n_hi = t - m_hi * hop;                           // smallest tap index of t
        float2 acc = make_float2(0.f, 0.f);
        if (n_hi < a.n_taps) {
            long long m = m_hi - (a.n_taps - 1 - n_hi) / hop;
            if (m < 0) m = 0;
            long long n = t - m * hop;
            const float2* up = a.u + (c * a.n_frames + (m - a.frame_first)) * K;
#pragma unroll 4
            for (; m <= m_hi; ++m, n -= hop, up += K)
                acc = cfma_rs(__ldg(up + (n & (K - 1))), __ldg(a.taps + n), acc);
        }
        __stcs(a.out + c * a.out_ch_stride + j, acc);
    }
}

template <int LOG2N>
static int launch_pfb_unrotate(PfbUnrotateArgs a, cudaStream_t stream) {
    using C = StftCfg<LOG2N>;
    auto kern = pfb_unrotate_ifft_kernel<LOG2N>;
    long long grid = 0;
    if (int rc = resident_ctas(kern, C::THREADS, C::SMEM, "pfb unrotate-ifft kernel", &grid)) return rc;
    a.groups_per_ch = (a.n_frames + C::FPC - 1) / C::FPC;
    a.n_groups = a.groups_per_ch * a.n_channels;
    if (grid > a.n_groups) grid = a.n_groups;
    { IQW_PROFILE("pfb_unrotate_ifft_kernel", stream); kern<<<(unsigned)grid, C::THREADS, C::SMEM, stream>>>(a); }
    IQW_CUDA_OK(cudaGetLastError());
    return IQW_OK;
}

static int launch_pfb_unfold(PfbUnfoldArgs a, long long n_channels, cudaStream_t stream) {
    long long grid = 0;
    if (int rc = resident_ctas(pfb_unfold_kernel, kUnfoldThreads, 0, "pfb unfold kernel", &grid)) return rc;
    a.tiles_per_ch = (a.n_out + kUnfoldThreads - 1) / kUnfoldThreads;
    a.n_tiles = a.tiles_per_ch * n_channels;
    if (grid > a.n_tiles) grid = a.n_tiles;
    { IQW_PROFILE("pfb_unfold_kernel", stream); pfb_unfold_kernel<<<(unsigned)grid, kUnfoldThreads, 0, stream>>>(a); }
    IQW_CUDA_OK(cudaGetLastError());
    return IQW_OK;
}

}  // namespace iqw

extern "C" size_t iqw_pfb_synthesize_workspace_bytes(int64_t n_channels, int64_t n_frames, int32_t nfft) {
    if (n_channels < 0 || n_frames < 0 || nfft < 0) return 0;
    return (size_t)n_channels * (size_t)n_frames * (size_t)nfft * sizeof(float2);
}

extern "C" int iqw_pfb_synthesize_c64(const void* d_y, int64_t n_channels, int64_t n_frames, int64_t y_channel_stride,
                                      int64_t frame_first, int64_t n_frames_total, const void* d_taps, int32_t n_taps,
                                      int32_t nfft, int32_t hop, int64_t out_first, int64_t n_out, void* d_out,
                                      int64_t out_channel_stride, void* d_workspace, size_t workspace_bytes,
                                      void* stream) {
    using namespace iqw;
    const int log2n = log2_exact(nfft);
    if (log2n < 1) return fail(IQW_ERR_UNSUPPORTED, "pfb_synthesize: nfft=%d: only powers of two are built", nfft);
    if (log2n < 4 || log2n > 13)
        return fail(IQW_ERR_UNSUPPORTED, "pfb_synthesize: nfft=%d outside the built range 16..8192", nfft);
    if (n_taps < 1) return fail(IQW_ERR_INVALID, "pfb_synthesize: n_taps=%d: need at least one tap", n_taps);
    const int n_seg = (n_taps + nfft - 1) / nfft;
    if (n_taps > 32768 || n_seg > 16)
        return fail(IQW_ERR_UNSUPPORTED, "pfb_synthesize: %d taps = %d segments of nfft=%d: at most 16 segments and "
                    "32768 taps are built", n_taps, n_seg, nfft);
    if (hop < 1 || hop > nfft) return fail(IQW_ERR_INVALID, "pfb_synthesize: hop=%d outside [1, nfft=%d]", hop, nfft);
    if (n_channels < 0 || n_frames < 0 || n_out < 0 || frame_first < 0 || out_first < 0 || n_frames_total < 1)
        return fail(IQW_ERR_INVALID, "pfb_synthesize: negative size or index, or no frames");
    if (n_channels == 0 || n_out == 0) return IQW_OK;
    const long long total_out = (n_frames_total - 1) * (long long)hop + n_taps;
    if (out_first + n_out > total_out)
        return fail(IQW_ERR_INVALID, "pfb_synthesize: outputs [%lld, %lld) past the %lld samples of %lld frames",
                    (long long)out_first, (long long)(out_first + n_out), total_out, (long long)n_frames_total);
    // frames that cover the outputs: [max(0, ceil((o0 - Lg + 1) / hop)), min(T, floor((o1 - 1) / hop) + 1))
    const long long lo_num = out_first - n_taps + 1;
    const long long f_lo = lo_num <= 0 ? 0 : (lo_num + hop - 1) / hop;
    long long f_hi = (out_first + n_out - 1) / hop + 1;
    if (f_hi > n_frames_total) f_hi = n_frames_total;
    if (frame_first + n_frames > n_frames_total ||
        (f_lo < f_hi && (f_lo < frame_first || f_hi > frame_first + n_frames)))
        return fail(IQW_ERR_INVALID, "pfb_synthesize: outputs [%lld, %lld) need frames [%lld, %lld), the call holds "
                    "frames [%lld, %lld) of %lld", (long long)out_first, (long long)(out_first + n_out), f_lo, f_hi,
                    (long long)frame_first, (long long)(frame_first + n_frames), (long long)n_frames_total);
    if (!d_taps || !d_out || (n_frames > 0 && (!d_y || !d_workspace)))
        return fail(IQW_ERR_INVALID, "pfb_synthesize: null pointer");
    if (n_channels > 1 && (y_channel_stride < n_frames * nfft || out_channel_stride < n_out))
        return fail(IQW_ERR_INVALID, "pfb_synthesize: channel stride shorter than a channel");
    if (workspace_bytes < iqw_pfb_synthesize_workspace_bytes(n_channels, n_frames, nfft))
        return fail(IQW_ERR_INVALID, "pfb_synthesize: workspace of %zu bytes, need %zu", workspace_bytes,
                    iqw_pfb_synthesize_workspace_bytes(n_channels, n_frames, nfft));
    if (n_channels > 0x7FFFFFFF) return fail(IQW_ERR_UNSUPPORTED, "pfb_synthesize: %lld channels", (long long)n_channels);
    DeviceGuard guard(d_out);
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    if (n_frames > 0) {
        PfbUnrotateArgs a{};
        a.y = reinterpret_cast<const float2*>(d_y);
        a.y_ch_stride = y_channel_stride;
        a.frame_first = frame_first;
        a.n_frames = n_frames;
        a.hop = hop;
        a.u = reinterpret_cast<float2*>(d_workspace);
        a.n_channels = (int)n_channels;
        if (int rc = get_twiddles(log2n, s, &a.twiddle)) return rc;
        if (int rc = device_table(kPfbRotation, log2n, (size_t)1 << log2n,
                                  [](float2* d, int log2n, cudaStream_t s) { pfb_rot_init_kernel<<<8, 256, 0, s>>>(d, 1 << log2n); },
                                  s, &a.rot))
            return rc;
        if (int rc = dispatch<4, 13>(log2n, [&](auto L) { return launch_pfb_unrotate<L>(a, s); },
                                     [&] { return fail(IQW_ERR_UNSUPPORTED, "pfb_synthesize: nfft=%d", nfft); }))
            return rc;
    }
    PfbUnfoldArgs b{};
    b.u = reinterpret_cast<const float2*>(d_workspace);
    b.frame_first = frame_first;
    b.n_frames = n_frames;
    b.n_frames_total = n_frames_total;
    b.taps = reinterpret_cast<const float*>(d_taps);
    b.n_taps = n_taps;
    b.log2n = log2n;
    b.hop = hop;
    b.out_first = out_first;
    b.n_out = n_out;
    b.out = reinterpret_cast<float2*>(d_out);
    b.out_ch_stride = out_channel_stride;
    return launch_pfb_unfold(b, n_channels, s);
}
