// iqw_stft_large.cu -- kernel 1 for frames that do not fit one CTA's shared memory:
// nfft = 2^14 .. 2^16 (128 .. 512 KB of complex64 per frame) as a four-step FFT in two kernels.
//
// Same reference steps as iqw_stft.cu (/root/reference/src/iqwaveform/fourier.py:568-581 gather *
// window, fourier.py:1044 fft, power_analysis.py:254-255 / 199-204 power / dB, fourier.py:1295 band
// slice); only the FFT is factored:  N = N1 * N2 with N2 = 256,  n = n1*N2 + n2,  k = k1 + N1*k2,
//
//     X[k1 + N1*k2] = sum_n2  W_N2^(n2 k2) * { W_N^(n2 k1) * sum_n1 w[n] x[n] W_N1^(n1 k1) }
//
//   columns_kernel : per frame and n2, the length-N1 transform over n1 (input stride N2).  The 16
//                    lanes of a half-warp own 16 adjacent n2, so every global access is a full
//                    128-byte line; the transforms of a CTA are interleaved element by element in
//                    shared memory (fft_pass STRIDE layout).  Multiplies by W_N^(n2 k1) and writes
//                    the scratch S[frame][k1][n2] (complex64, caller's workspace).
//   rows_kernel    : per frame and k1, the length-256 transform over n2 (contiguous in S), then
//                    |X|^2 / dB / band trim.  Output bin k = k1 + N1*k2 is strided, so the 16 rows of
//                    a CTA go through a shared-memory tile and leave as 64/128-byte segments.
// The scratch is written and read once (16*nfft/hop bytes per sample of extra HBM traffic); frames
// are processed in chunks so that it never exceeds the scratch cap.
#include <algorithm>
#include <atomic>
#include "iqw_stft.cuh"

namespace iqw {

constexpr int kLog2N2 = 8;
constexpr int kN2 = 1 << kLog2N2;
constexpr int kCols = 16;                         // n2 per CTA of columns_kernel / k1 per CTA of rows_kernel
static std::atomic<size_t> g_scratch_cap{1ull << 30};         // bytes of scratch per chunk of frames (iqw_debug_set_stft_scratch_cap)

struct LargeArgs {
    StftArgs a;
    const float2* step_a;       // W_N1^e, e < N1   ( = W_N^(256 e) )
    const float2* step_b;       // W_N^e,  e < 256
    float2* scratch;
    long long gf0, gf1;         // flattened (channel, frame) range of this chunk
    int mode;
};

__device__ __forceinline__ float2 cmul_d(float2 a, float2 b) { return cmul(a, b); }

// ---------------------------------------------------------------------------------------------
// columns
// ---------------------------------------------------------------------------------------------
template <int L1>
struct ColCfg {
    static constexpr int N1 = 1 << L1;
    static constexpr int E = plan_elems(L1);
    static constexpr int TPF = N1 / E;
    static constexpr int THREADS = kCols * TPF;
    static constexpr int NP = plan_passes(L1);
    static constexpr int TW = plan_tw_size(L1);
    static constexpr int TW_ALLOC = (TW + 15) & ~15;
    static constexpr size_t SMEM = sizeof(float2) * ((size_t)TW_ALLOC + 2 * (size_t)N1 * kCols + N1 + kN2);
};

template <int L1, int P>
struct ColPasses {
    static __device__ __forceinline__ void run(float2* v, float2* bufs, const float2* tw, const float2* t,
                                               int ltid, int col, int& par) {
        using C = ColCfg<L1>;
        constexpr bool LAST = (P == C::NP - 1);
        float2* wr = bufs + (size_t)par * C::N1 * kCols + col;
        const float2* rd = bufs + (size_t)(par ^ 1) * C::N1 * kCols + col;
        fft_pass<L1, P, kCols>(v, rd, wr, t, ltid);
        if constexpr (!LAST) {
            float2 tn[C::E];
            load_twiddles<L1, P + 1>(tn, tw, ltid);
            __syncthreads();
            par ^= 1;
            ColPasses<L1, P + 1>::run(v, bufs, tw, tn, ltid, col, par);
        }
    }
};

template <int L1>
__global__ void __launch_bounds__(ColCfg<L1>::THREADS)
columns_kernel(const LargeArgs g) {
    using C = ColCfg<L1>;
    constexpr int N1 = C::N1, E = C::E, TPF = C::TPF;
    constexpr int R0 = plan_radix(L1, 0), RL = plan_radix(L1, C::NP - 1);
    constexpr long long N = (long long)N1 * kN2;
    const StftArgs& a = g.a;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* tw = reinterpret_cast<float2*>(smem_raw);
    float2* bufs = tw + C::TW_ALLOC;
    float2* sa = bufs + 2 * N1 * kCols;
    float2* sb = sa + N1;
    for (int i = threadIdx.x; i < C::TW; i += C::THREADS) tw[i] = a.twiddle[i];
    for (int i = threadIdx.x; i < N1; i += C::THREADS) sa[i] = g.step_a[i];
    for (int i = threadIdx.x; i < kN2; i += C::THREADS) sb[i] = g.step_b[i];
    __syncthreads();

    const int col = threadIdx.x % kCols;
    const int ltid = threadIdx.x / kCols;
    constexpr int TILES = kN2 / kCols;
    const long long n_items = (g.gf1 - g.gf0) * TILES;
    const long long per = (n_items + gridDim.x - 1) / gridDim.x;
    const long long it0 = per * blockIdx.x;
    const long long it1 = it0 + per < n_items ? it0 + per : n_items;
    int par = 0;

    // software pipeline: samples and window of the next item are loaded while this one is transformed
    float2 nx[E];
    float nw[E];
    auto prefetch = [&](long long it) {
        if (it < it1) {
            const long long gf = g.gf0 + it / TILES;
            const int n2 = (int)(it % TILES) * kCols + col;
            const long long c = gf / a.n_frames, frame = gf - c * a.n_frames;
            const float2* src = a.x + c * a.x_ch_stride + frame * a.hop + n2;
            const float* win = a.window + n2;
#pragma unroll
            for (int q = 0; q < E / R0; ++q)
#pragma unroll
                for (int r = 0; r < R0; ++r) {
                    const int n1 = (ltid + q * TPF) + r * (N1 / R0);
                    nx[q * R0 + r] = __ldg(src + (long long)n1 * kN2);
                    nw[q * R0 + r] = __ldg(win + n1 * kN2);
                }
        }
    };
    prefetch(it0);

    for (long long it = it0; it < it1; ++it) {
        const long long gf = g.gf0 + it / TILES;
        const int n2 = (int)(it % TILES) * kCols + col;

        float2 v[E];
#pragma unroll
        for (int e = 0; e < E; ++e) v[e] = cscale(nx[e], nw[e]);
        prefetch(it + 1);
        ColPasses<L1, 0>::run(v, bufs, tw, nullptr, ltid, col, par);

        float2* dst = g.scratch + (gf - g.gf0) * N + n2;
#pragma unroll
        for (int q = 0; q < E / RL; ++q)
#pragma unroll
            for (int r = 0; r < RL; ++r) {
                const int k1 = (ltid + q * TPF) + r * (N1 / RL);
                const int e = n2 * k1;                       // < N: W_N^e = W_N1^(e >> 8) * W_N^(e & 255)
                const float2 t = cmul_d(sa[e >> kLog2N2], sb[e & (kN2 - 1)]);
                dst[(long long)k1 * kN2] = cmul_d(v[q * RL + r], t);
            }
    }
}

// ---------------------------------------------------------------------------------------------
// rows: 16 length-256 transforms per CTA (16 threads x 16 elements each), transposed store
// ---------------------------------------------------------------------------------------------
constexpr int kRowE = plan_elems(kLog2N2);            // 16
constexpr int kRowTPF = kN2 / kRowE;                  // 16
constexpr int kRowThreads = kCols * kRowTPF;          // 256
constexpr int kRowNP = plan_passes(kLog2N2);          // 2
constexpr int kRowTW = plan_tw_size(kLog2N2);
constexpr int kRowTWAlloc = (kRowTW + 15) & ~15;
constexpr int kRowPad = padded_size(kN2);
constexpr int kTilePitch = kCols + 1;
constexpr size_t kRowSmem = sizeof(float2) * ((size_t)kRowTWAlloc + 2 * (size_t)kCols * kRowPad + (size_t)kN2 * kTilePitch);

template <int P>
struct RowPasses {
    static __device__ __forceinline__ void run(float2* v, float2* bufs, const float2* tw, const float2* t,
                                               int ltid, int slot, int& par) {
        constexpr bool LAST = (P == kRowNP - 1);
        float2* wr = bufs + ((size_t)par * kCols + slot) * kRowPad;
        const float2* rd = bufs + ((size_t)(par ^ 1) * kCols + slot) * kRowPad;
        fft_pass<kLog2N2, P>(v, rd, wr, t, ltid);
        if constexpr (!LAST) {
            float2 tn[kRowE];
            load_twiddles<kLog2N2, P + 1>(tn, tw, ltid);
            static_assert(kRowTPF <= 32 && 32 % kRowTPF == 0, "a row transform lives inside one warp");
            __syncwarp();
            par ^= 1;
            RowPasses<P + 1>::run(v, bufs, tw, tn, ltid, slot, par);
        }
    }
};

template <int MODE>
__global__ void __launch_bounds__(kRowThreads)
rows_kernel(const LargeArgs g, int log2n1) {
    const StftArgs& a = g.a;
    const int N1 = 1 << log2n1;
    const long long N = (long long)N1 * kN2;
    constexpr int R0 = plan_radix(kLog2N2, 0), RL = plan_radix(kLog2N2, kRowNP - 1);
    static_assert(kRowE == R0 && kRowE == RL, "one butterfly per thread and pass");

    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* tw = reinterpret_cast<float2*>(smem_raw);
    float2* bufs = tw + kRowTWAlloc;
    float2* tile = bufs + 2 * kCols * kRowPad;          // [k2][kTilePitch]; float2 or float entries
    for (int i = threadIdx.x; i < kRowTW; i += kRowThreads) tw[i] = a.twiddle[i];
    __syncthreads();

    const int slot = threadIdx.x / kRowTPF;             // row (k1) within the tile
    const int ltid = threadIdx.x % kRowTPF;
    const int tiles = N1 / kCols;                       // power of two
    const int tile_shift = log2n1 - 4;
    const long long n_items = (g.gf1 - g.gf0) * tiles;
    const long long per = (n_items + gridDim.x - 1) / gridDim.x;
    const long long it0 = per * blockIdx.x;
    const long long it1 = it0 + per < n_items ? it0 + per : n_items;
    const int nbins = a.bin_hi - a.bin_lo;
    int par = 0;

    // software pipeline: the rows of the next item are loaded while this one is transformed
    float2 nx[kRowE];
    auto prefetch = [&](long long it) {
        if (it < it1) {
            const long long gf = g.gf0 + (it >> tile_shift);
            const int k1_0 = (int)(it & (tiles - 1)) * kCols;
            const float2* src = g.scratch + (gf - g.gf0) * N + (long long)(k1_0 + slot) * kN2 + ltid;
#pragma unroll
            for (int r = 0; r < R0; ++r) nx[r] = __ldcs(src + r * (kN2 / R0));
        }
    };
    prefetch(it0);

    for (long long it = it0; it < it1; ++it) {
        const long long gf = g.gf0 + (it >> tile_shift);
        const int k1_0 = (int)(it & (tiles - 1)) * kCols;
        const long long c = gf / a.n_frames, frame = gf - c * a.n_frames;

        float2 v[kRowE];
#pragma unroll
        for (int r = 0; r < R0; ++r) v[r] = nx[r];
        prefetch(it + 1);
        RowPasses<0>::run(v, bufs, tw, nullptr, ltid, slot, par);

        // tile[k2][slot] <- result of bin k2 = ltid + r*16; then rows of 16 adjacent k leave together
#pragma unroll
        for (int r = 0; r < RL; ++r) {
            const int k2 = ltid + r * (kN2 / RL);
            const float2 X = v[r];
            if constexpr (MODE == IQW_STFT_COMPLEX) {
                tile[k2 * kTilePitch + slot] = X;
            } else {
                float p = X.x * X.x + X.y * X.y;
                if constexpr (MODE == IQW_STFT_DB) p = power_to_dB(p, a.eps);
                reinterpret_cast<float*>(tile)[k2 * kTilePitch + slot] = p;
            }
        }
        __syncthreads();
        const long long row = c * a.out_ch_stride + frame * (long long)nbins - a.bin_lo;
        const int kk = threadIdx.x % kCols;
#pragma unroll 4
        for (int k2 = threadIdx.x / kCols; k2 < kN2; k2 += kRowThreads / kCols) {
            const int k = k1_0 + kk + N1 * k2;
            if (k >= a.bin_lo && k < a.bin_hi) {
                if constexpr (MODE == IQW_STFT_COMPLEX)
                    __stcs(reinterpret_cast<float2*>(a.out) + row + k, tile[k2 * kTilePitch + kk]);
                else
                    __stcs(reinterpret_cast<float*>(a.out) + row + k,
                           reinterpret_cast<const float*>(tile)[k2 * kTilePitch + kk]);
            }
        }
        __syncthreads();        // the tile is rewritten by the next item
    }
}

// ---------------------------------------------------------------------------------------------
// step twiddles W_N1^e (e < N1) and W_N^e (e < 256), per (device, log2 n), float64 -> float32
// ---------------------------------------------------------------------------------------------
__global__ void step_twiddle_kernel(float2* ta, float2* tb, int n1, long long n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    double s, c;
    if (i < n1) {
        sincospi(-2.0 * (double)i / (double)n1, &s, &c);
        ta[i] = make_float2((float)c, (float)s);
    }
    if (i < kN2) {
        sincospi(-2.0 * (double)i / (double)n, &s, &c);
        tb[i] = make_float2((float)c, (float)s);
    }
}

static int get_step_twiddles(int log2n, cudaStream_t stream, const float2** ta, const float2** tb) {
    const int n1 = 1 << (log2n - kLog2N2);
    auto init = [](float2* d, int log2n, cudaStream_t s) {
        const int n1 = 1 << (log2n - kLog2N2);
        step_twiddle_kernel<<<(std::max(n1, kN2) + 255) / 256, 256, 0, s>>>(d, d + n1, n1, 1ll << log2n);
    };
    if (int rc = device_table(kStepTwiddles, log2n, n1 + kN2, init, stream, ta)) return rc;
    *tb = *ta + n1;
    return IQW_OK;
}

size_t stft_large_workspace_bytes(int log2n, long long n_channels, long long n_frames) {
    if (log2n < 14 || log2n > 16 || n_channels < 1 || n_frames < 1) return 0;
    const size_t frame_bytes = sizeof(float2) << log2n;
    const size_t all = frame_bytes * (size_t)n_channels * (size_t)n_frames;
    const size_t cap_bytes = g_scratch_cap.load();
    const size_t cap = cap_bytes / frame_bytes * frame_bytes > 0 ? cap_bytes / frame_bytes * frame_bytes : frame_bytes;
    return all < cap ? all : cap;
}

template <int L1>
static int launch_columns(const LargeArgs& g, cudaStream_t s) {
    using C = ColCfg<L1>;
    auto kern = columns_kernel<L1>;
    long long grid = 0;
    if (int rc = resident_ctas(kern, C::THREADS, C::SMEM, "columns kernel", &grid)) return rc;
    const long long items = (g.gf1 - g.gf0) * (kN2 / kCols);
    if (grid > items) grid = items;
    { IQW_PROFILE("stft_columns", s); kern<<<(unsigned)grid, C::THREADS, C::SMEM, s>>>(g); }
    IQW_CUDA_OK(cudaGetLastError());
    return IQW_OK;
}

template <int MODE>
static int launch_rows(const LargeArgs& g, int log2n1, cudaStream_t s) {
    auto kern = rows_kernel<MODE>;
    long long grid = 0;
    if (int rc = resident_ctas(kern, kRowThreads, kRowSmem, "rows kernel", &grid)) return rc;
    const long long items = (g.gf1 - g.gf0) * ((1 << log2n1) / kCols);
    if (grid > items) grid = items;
    { IQW_PROFILE("stft_rows", s); kern<<<(unsigned)grid, kRowThreads, kRowSmem, s>>>(g, log2n1); }
    IQW_CUDA_OK(cudaGetLastError());
    return IQW_OK;
}

int launch_stft_large(const StftArgs& a, int log2n, int mode, void* workspace, size_t workspace_bytes,
                      cudaStream_t stream) {
    const int log2n1 = log2n - kLog2N2;
    const size_t frame_bytes = sizeof(float2) << log2n;
    if (!workspace || workspace_bytes < frame_bytes)
        return fail(IQW_ERR_WORKSPACE, "nfft=%d needs a workspace of at least %zu bytes (iqw_stft_workspace_bytes)",
                    1 << log2n, frame_bytes);
    if (((uintptr_t)workspace & 15) != 0) return fail(IQW_ERR_INVALID, "workspace not 16-byte aligned");

    LargeArgs g{};
    g.a = a;
    g.mode = mode;
    g.scratch = static_cast<float2*>(workspace);
    if (int rc = get_step_twiddles(log2n, stream, &g.step_a, &g.step_b)) return rc;
    const float2 *tw_cols = nullptr, *tw_rows = nullptr;
    if (int rc = get_twiddles(log2n1, stream, &tw_cols)) return rc;
    if (int rc = get_twiddles(kLog2N2, stream, &tw_rows)) return rc;

    const long long total = (long long)a.n_channels * a.n_frames;
    long long chunk = (long long)(workspace_bytes / frame_bytes);
    if (chunk > total) chunk = total;
    for (long long gf0 = 0; gf0 < total; gf0 += chunk) {
        g.gf0 = gf0;
        g.gf1 = gf0 + chunk < total ? gf0 + chunk : total;
        g.a.twiddle = tw_cols;
        if (int rc = dispatch<6, 8>(log2n1, [&](auto L1) { return launch_columns<L1>(g, stream); },
                                    [&] { return fail(IQW_ERR_UNSUPPORTED, "nfft=%d", 1 << log2n); }))
            return rc;
        g.a.twiddle = tw_rows;
        if (int rc = dispatch_stft_mode(mode, [&](auto M) { return launch_rows<M>(g, log2n1, stream); })) return rc;
    }
    return IQW_OK;
}

}  // namespace iqw

extern "C" int iqw_debug_set_stft_scratch_cap(size_t bytes) {
    iqw::g_scratch_cap = bytes;
    return IQW_OK;
}
