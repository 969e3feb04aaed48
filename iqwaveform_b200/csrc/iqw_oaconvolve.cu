// iqw_oaconvolve.cu -- kernel 7: FFT convolution of complex64 rows with an M-tap filter by overlap-save
// (scipy.signal.oaconvolve output windows), one kernel per call.
//
//   y[n] = sum_{k < M} h[k] * x[n - k],   n in [out_first, out_first + n_out) of the full convolution
//
// Blocks of nfft input samples step by hop = nfft - D (D = nfft/R, the discard, D >= M - 1).  Block b
// reads the global samples [b*hop - D, b*hop - D + nfft) (zero outside the buffer), runs the forward FFT
// (natural order, no window), multiplies bin k by H[k] = fft(h, nfft)[k] / nfft (the host's float64
// spectrum rounded once), runs the inverse FFT and keeps samples D .. nfft-1: there the circular
// convolution equals the linear one, and they are the outputs [b*hop, b*hop + hop).
//
// Geometry of kernel 4's ola_kernel (iqw_istft.cu): a frame slot of TPF = nfft/E threads holds E values
// per thread in registers and walks a contiguous range of blocks of one channel, the next block's samples
// prefetched into registers while the current one is transformed.  After the inverse transform thread
// ltid holds samples ltid + j*TPF; D = (E/R)*TPF, so the kept samples are j >= E/R -- TPF consecutive
// float2 per j, coalesced stores.  Only blocks that touch a buffer edge take the predicated loads /
// stores.
//
// Determinism: blocks are anchored at global full-convolution index 0, whatever out_first and x_first
// are, and a block's arithmetic depends only on its nfft input samples and H.  So a 'same' / 'valid'
// window is a bitwise crop of 'full', and time shards that hold every in-range sample of each block
// they touch (D samples of halo before their first output) concatenate to the bits of one call.
#include "iqw_stft.cuh"

namespace iqw {

struct OaconvArgs {
    const float2* x;
    long long n_in, x_ch_stride, x_first;  // x[0] is global sample x_first
    const float2* hspec;                   // (1 | n_channels, nfft) spectrum rows
    long long h_ch_stride;                 // 0: one spectrum for every channel
    long long out_first, n_out, out_ch_stride;
    float2* out;
    const float2* twiddle;
    int n_channels;
    long long b_first, n_blocks;           // global index of the first block, blocks per channel
    long long streams_per_ch, blocks_per_stream;
};

template <int LOG2N, int LOG2R>
__global__ void __launch_bounds__(StftCfg<LOG2N>::THREADS, StftCfg<LOG2N>::MIN_BLOCKS)
oaconvolve_kernel(const OaconvArgs a) {
    using C = StftCfg<LOG2N>;
    constexpr int N = C::N, E = C::E, TPF = C::TPF, FPC = C::FPC;
    constexpr int R0 = plan_radix(LOG2N, 0);
    constexpr int RL = plan_radix(LOG2N, C::NP - 1);
    constexpr int R = 1 << LOG2R;
    constexpr int K = E / R;                  // register index of the first kept sample
    constexpr long long D = N / R, HOP = N - N / R;
    static_assert(R <= E, "the discard must be a multiple of nfft / E");

    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* tw = reinterpret_cast<float2*>(smem_raw);
    float2* bufs = tw + C::TW_ALLOC;
    for (int i = threadIdx.x; i < C::TW; i += C::THREADS) tw[i] = a.twiddle[i];
    __syncthreads();

    const int slot = threadIdx.x / TPF;
    const int ltid = threadIdx.x % TPF;
    const long long sid = (long long)blockIdx.x * FPC + slot;
    // every slot of the CTA runs the same number of iterations (the inter-pass barriers may span
    // several slots); a slot without work transforms zeros and stores nothing
    const bool live = sid < a.streams_per_ch * a.n_channels;
    const long long c = live ? sid / a.streams_per_ch : 0;
    const long long r0 = live ? (sid - c * a.streams_per_ch) * a.blocks_per_stream : 0;
    const long long r1 = !live ? 0 : r0 + a.blocks_per_stream < a.n_blocks ? r0 + a.blocks_per_stream : a.n_blocks;

    // H[k] of bin k = ltid + j*TPF, in the register order the forward transform leaves the bins in
    const float2* hs = a.hspec + c * a.h_ch_stride + ltid;
    const float2* src = a.x + c * a.x_ch_stride;
    float2* dst = a.out + c * a.out_ch_stride;

    // software pipeline: the samples of the NEXT block are loaded while the current one is transformed
    float2 nx[E];
    auto prefetch = [&](long long rb) {
        if (rb < r1) {
            const long long i0 = (a.b_first + rb) * HOP - D - a.x_first;    // buffer index of sample 0
            if (i0 >= 0 && i0 + N <= a.n_in) {
                const float2* fr = src + i0 + ltid;
#pragma unroll
                for (int q = 0; q < E / R0; ++q)
#pragma unroll
                    for (int r = 0; r < R0; ++r) nx[q * R0 + r] = __ldg(fr + q * TPF + r * (N / R0));
            } else {                                   // a block at an edge of the buffer
#pragma unroll
                for (int q = 0; q < E / R0; ++q)
#pragma unroll
                    for (int r = 0; r < R0; ++r) {
                        const long long i = i0 + ltid + q * TPF + r * (N / R0);
                        nx[q * R0 + r] = (unsigned long long)i < (unsigned long long)a.n_in ? __ldg(src + i)
                                                                                           : make_float2(0.f, 0.f);
                    }
            }
        } else {
#pragma unroll
            for (int e = 0; e < E; ++e) nx[e] = make_float2(0.f, 0.f);
        }
    };
    prefetch(r0);
    int par = 0;

#pragma unroll 1
    for (long long rb = r0; rb < r0 + a.blocks_per_stream; ++rb) {
        float2 v[E];
#pragma unroll
        for (int e = 0; e < E; ++e) v[e] = nx[e];
        prefetch(rb + 1);
        PassLoop<LOG2N, 0>::run(v, bufs, tw, nullptr, ltid, slot, par);

        // times H, conjugated (inverse = conj(FFT(conj(.)))), renamed into the load order of the inverse
        float2 u[E];
#pragma unroll
        for (int q = 0; q < E / RL; ++q)
#pragma unroll
            for (int r = 0; r < RL; ++r) {
                const int j = q + r * (E / RL);
                const float2 X = cmul(v[q * RL + r], __ldg(hs + j * TPF));
                u[(j % (E / R0)) * R0 + j / (E / R0)] = make_float2(X.x, -X.y);
            }
        PassLoop<LOG2N, 0>::run(u, bufs, tw, nullptr, ltid, slot, par);

        if (rb < r1) {
            // kept sample ltid + j*TPF (j >= K) is output b*hop + ltid + (j - K)*TPF
            const long long o0 = (a.b_first + rb) * HOP - a.out_first;     // buffer index of kept sample 0
            const bool inside = o0 >= 0 && o0 + HOP <= a.n_out;
#pragma unroll
            for (int q = 0; q < E / RL; ++q)
#pragma unroll
                for (int r = 0; r < RL; ++r) {
                    const int j = q + r * (E / RL);
                    if (j < K) continue;
                    const float2 X = u[q * RL + r];
                    const long long i = o0 + ltid + (j - K) * TPF;
                    if (inside || (unsigned long long)i < (unsigned long long)a.n_out)
                        __stcs(dst + i, make_float2(X.x, -X.y));
                }
        }
    }
}

// the (nfft, nfft/discard) pairs oaconvolve_plan (_plan.py) picks for 1..4097 taps; other pairs are not
// instantiated (IQW_ERR_UNSUPPORTED): fewer kernels to build, and every built one runs without spills
constexpr bool oaconvolve_built(int log2n, int log2r) {
    return (log2n == 4 && log2r >= 2) || (log2n >= 5 && log2n <= 6 && log2r == 2) ||
           (log2n >= 8 && log2n <= 12 && log2r == 3) || (log2n == 13 && log2r >= 1 && log2r <= 3);
}

template <int LOG2N, int LOG2R>
static int launch_oaconvolve_r(OaconvArgs a, cudaStream_t stream) {
    if constexpr (!oaconvolve_built(LOG2N, LOG2R)) {
        return fail(IQW_ERR_UNSUPPORTED, "oaconvolve: nfft = %d with nfft/discard = %d is not built "
                    "(see oaconvolve_plan)", 1 << LOG2N, 1 << LOG2R);
    } else {
        using C = StftCfg<LOG2N>;
        auto kern = oaconvolve_kernel<LOG2N, LOG2R>;
        long long ctas = 0;
        if (int rc = resident_ctas(kern, C::THREADS, C::SMEM, "oaconvolve kernel", &ctas)) return rc;
        // one block range per slot of the resident grid, of at least 4 blocks so that the first,
        // unhidden load of a range stays a small part of it
        const long long streams = ctas * C::FPC;
        long long per_ch = streams / a.n_channels > 0 ? streams / a.n_channels : 1;
        const long long most = (a.n_blocks + 3) / 4;
        if (per_ch > most) per_ch = most;
        a.streams_per_ch = per_ch;
        a.blocks_per_stream = (a.n_blocks + per_ch - 1) / per_ch;
        const long long grid = (per_ch * a.n_channels + C::FPC - 1) / C::FPC;
        if (grid > 0x7FFFFFFFLL) return fail(IQW_ERR_UNSUPPORTED, "oaconvolve: %lld CTAs", grid);
        { IQW_PROFILE("oaconvolve_kernel", stream); kern<<<(unsigned)grid, C::THREADS, C::SMEM, stream>>>(a); }
        IQW_CUDA_OK(cudaGetLastError());
        return IQW_OK;
    }
}

}  // namespace iqw

extern "C" int iqw_oaconvolve_c64(const void* d_x, int64_t n_channels, int64_t n_in, int64_t x_channel_stride,
                                  int64_t x_first, const void* d_hspec, int64_t hspec_channel_stride,
                                  int32_t n_taps, int32_t nfft, int32_t discard, int64_t out_first, int64_t n_out,
                                  void* d_out, int64_t out_channel_stride, void* stream) {
    using namespace iqw;
    const int log2n = log2_exact(nfft);
    if (log2n < 1) return fail(IQW_ERR_UNSUPPORTED, "oaconvolve: nfft=%d: only powers of two are built", nfft);
    if (log2n < 4 || log2n > 13)
        return fail(IQW_ERR_UNSUPPORTED, "oaconvolve: nfft=%d outside the built range 16..8192", nfft);
    const int log2r = discard >= 1 && discard < nfft && nfft % discard == 0 ? log2_exact(nfft / discard) : -1;
    if (log2r < 0 || log2r > 4)
        return fail(IQW_ERR_UNSUPPORTED, "oaconvolve: discard=%d: nfft/discard must be 2, 4, 8 or 16", discard);
    if (n_taps < 1 || discard < n_taps - 1)
        return fail(IQW_ERR_INVALID, "oaconvolve: need 1 <= n_taps <= discard + 1 (n_taps %d, discard %d)", n_taps,
                    discard);
    if (hspec_channel_stride != 0 && hspec_channel_stride != nfft)
        return fail(IQW_ERR_INVALID, "oaconvolve: hspec_channel_stride must be 0 or nfft");
    if (n_channels < 0 || n_in < 0 || n_out < 0 || out_first < 0)
        return fail(IQW_ERR_INVALID, "oaconvolve: negative size");
    if (n_channels == 0 || n_out == 0) return IQW_OK;
    if (!d_hspec || !d_out || (n_in > 0 && !d_x)) return fail(IQW_ERR_INVALID, "oaconvolve: null pointer");
    if (n_channels > 1 && (x_channel_stride < n_in || out_channel_stride < n_out))
        return fail(IQW_ERR_INVALID, "oaconvolve: channel stride shorter than a channel");
    DeviceGuard guard(d_out);
    const long long hop = nfft - discard;
    OaconvArgs a{};
    a.x = reinterpret_cast<const float2*>(d_x);
    a.n_in = n_in;
    a.x_ch_stride = x_channel_stride;
    a.x_first = x_first;
    a.hspec = reinterpret_cast<const float2*>(d_hspec);
    a.h_ch_stride = hspec_channel_stride;
    a.out_first = out_first;
    a.n_out = n_out;
    a.out_ch_stride = out_channel_stride;
    a.out = reinterpret_cast<float2*>(d_out);
    a.n_channels = (int)n_channels;
    a.b_first = out_first / hop;
    a.n_blocks = (out_first + n_out - 1) / hop - a.b_first + 1;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    if (int rc = get_twiddles(log2n, s, &a.twiddle)) return rc;
    return dispatch<4, 13>(
        log2n,
        [&](auto L) {
            return dispatch<1, 4>(log2r, [&](auto R) { return launch_oaconvolve_r<L, R>(a, s); }, [&] {
                return fail(IQW_ERR_UNSUPPORTED, "oaconvolve: nfft/discard = %d: only 2, 4, 8, 16 are built", 1 << log2r);
            });
        },
        [&] { return fail(IQW_ERR_UNSUPPORTED, "oaconvolve: nfft=%d", nfft); });
}
