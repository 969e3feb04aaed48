// iqw_stft2p.cu -- kernel 1, two-pass variant for nfft 1024 / 2048 / 4096 (the headline sizes).
//
// Same contract as stft_kernel (iqw_stft.cu): fused overlapped-frame gather * window -> FFT ->
// {complex | |X|^2 | dB} -> band trim, replacing fourier.py:568-581 + 1044 + power_analysis.py:254-255 +
// 199-204 + fourier.py:1295 of the reference in one pass over the samples.
//
// Why a second geometry.  With 16 values per thread a 4096-point frame needs three radix-16 passes and
// TWO exchanges through shared memory; ncu showed that kernel bound by the L1/shared-memory data pipe
// (73 % busy: 2000 wavefronts per frame, 1590 of them shared-memory exchanges and twiddle reads), not by
// HBM (42 %).  Here a thread holds 64 values (32 for nfft 1024), N = RA x RB with RA, RB in {32, 64}, so a
// frame is TWO register-resident radix-32/64 passes and ONE exchange: ~1100 wavefronts per frame.
//   pass A  butterfly jA = ltid (RB of them): elements x[jA + r*RB], r < RA, windowed; writes row jA of
//           the RB x RA exchange matrix M (Stockham, Ns = 1) with 128-bit stores
//   pass B  butterfly jB = ltid + q*TPF (RA of them, E/RB per thread): reads column jB of M, multiplies by
//           W_N^(r*jB), radix-RB DFT; output r' is bin jB + r'*RA (natural order, coalesced stores)
// A frame slot is TPF = RB threads: ONE warp for nfft 1024 / 2048 (the exchange needs only __syncwarp), two
// warps for 4096 (a 64-thread named barrier).  Slots are independent: each walks its own contiguous range
// of frames, so the overlapped half of consecutive frames is re-read from L2 a few microseconds after its
// first use.  Rows of M are padded by two elements (a row is an odd number of 16-byte units), which makes
// both the 128-bit row stores and the 64-bit column loads conflict-free.
#include <atomic>
#include "iqw_stft.cuh"

#ifndef IQW_P2_SLOTS12
#define IQW_P2_SLOTS12 6
#endif
#ifndef IQW_P2_SLOTS11
#define IQW_P2_SLOTS11 12
#endif

namespace iqw {

template <int LOG2N, bool STAGED = true>
struct P2Cfg {
    static constexpr int N = 1 << LOG2N;
    static constexpr int RA = LOG2N >= 11 ? 64 : 32;
    static constexpr int RB = N / RA;                  // 32 (1024), 32 (2048), 64 (4096)
    static constexpr int E = RA;                       // values per thread
    static constexpr int TPF = N / E;                  // threads per frame slot == RB
    static constexpr int NB = E / RB;                  // pass-B butterflies per thread
    // frame slots per CTA: 12 warps (168 registers per thread; a warp count that is a multiple of the 4
    // schedulers) for the staged kernels at nfft 2048 / 4096, 8 warps (up to 255 registers) otherwise
    static constexpr int SLOTS = LOG2N == 12 ? (STAGED ? IQW_P2_SLOTS12 : 4) : LOG2N == 11 ? (STAGED ? IQW_P2_SLOTS11 : 8) : 8;
    static constexpr int THREADS = SLOTS * TPF;        // 256 or 384
    static constexpr int MIN_BLOCKS = LOG2N == 10 ? 2 : 1;
    static constexpr int ROW = RA + 2;                 // padded row of M, float2 units
    static constexpr int BUF = RB * ROW;               // one slot's exchange matrix
    // pass-B twiddles W_N^(r*jB), r = 8a + b, factored as A_a * B_b: rows A_1 .. A_(RB/8-1) = W_N^(8a*jB), then
    // rows B_1 .. B_7 = W_N^(b*jB), each RA entries long (7 KB at nfft 4096 instead of 32 KB for all RB - 1 rows;
    // 14 shared-memory loads per butterfly instead of 63, the products are computed)
    static constexpr int NA8 = RB / 8;
    static constexpr int TW_ROWS = (NA8 - 1) + 7;
    static constexpr int TW = TW_ROWS * RA;
    static constexpr size_t SMEM = sizeof(float2) * ((size_t)TW + (size_t)SLOTS * BUF);
    static_assert(RA >= RB && RA * RB == N && TPF == RB && TPF % 32 == 0, "geometry");
    static_assert((ROW * sizeof(float2)) % 16 == 0 && ((ROW * sizeof(float2)) / 16) % 2 == 1, "row padding");
};

__device__ __forceinline__ float2 ldg_stream(const float2* p) {
    float2 v;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p));
    return v;
}

// ---- mbarrier / bulk-copy (TMA) plumbing, raw PTX ---------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// one contiguous span of global memory -> shared memory, completion counted in bytes on `bar`
__device__ __forceinline__ void bulk_load(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// STAGED: the frame's samples are staged by ONE bulk copy (TMA) per frame into the slot's exchange buffer
// while the previous frame's second pass and epilogue run -- the buffer is idle exactly then -- so pass A
// reads shared memory instead of waiting for HBM / L2 with only two warps per scheduler to hide it.
template <int LOG2N, int MODE, bool FULLBAND, bool STAGED>
__global__ void __launch_bounds__(P2Cfg<LOG2N, STAGED>::THREADS, P2Cfg<LOG2N, STAGED>::MIN_BLOCKS)
stft2p_kernel(const StftArgs a) {
    using C = P2Cfg<LOG2N, STAGED>;
    constexpr int RA = C::RA, RB = C::RB, E = C::E, TPF = C::TPF, NB = C::NB, ROW = C::ROW;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* tw = reinterpret_cast<float2*>(smem_raw);
    __shared__ __align__(8) uint64_t full_bar[C::SLOTS];
    for (int i = threadIdx.x; i < C::TW; i += C::THREADS) tw[i] = a.twiddle[i];
    if constexpr (STAGED) {
        if (threadIdx.x < C::SLOTS) mbar_init(&full_bar[threadIdx.x], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        fence_proxy_async();
    }
    __syncthreads();

    const int slot = threadIdx.x / TPF;
    const int ltid = threadIdx.x % TPF;
    float2* buf = tw + C::TW + (size_t)slot * C::BUF;
    constexpr uint32_t kFrameBytes = (uint32_t)(C::N * sizeof(float2));
    static_assert(!STAGED || C::BUF >= C::N, "the exchange buffer doubles as the staging buffer");

    auto slot_sync = [&]() {
        if constexpr (TPF == 32) __syncwarp();
        else asm volatile("bar.sync %0, %1;" ::"r"(slot + 1), "n"(TPF) : "memory");
    };

    // contiguous range of (channel, frame) items for this slot
    const long long total = (long long)a.n_channels * a.n_frames;
    const long long n_slots = (long long)gridDim.x * C::SLOTS;
    const long long per = (total + n_slots - 1) / n_slots;
    const long long sg = (long long)blockIdx.x * C::SLOTS + slot;
    long long f = sg * per;
    const long long f_end = f + per < total ? f + per : total;
    if (f >= f_end) return;                      // (slots own whole warps and their own barrier id)
    long long c = f / a.n_frames;
    long long frame = f - c * a.n_frames;
    const int nbins = a.bin_hi - a.bin_lo;
    const float* wp = a.window + ltid;
    uint32_t parity = 0;
    if constexpr (STAGED) {
        if (ltid == 0) {
            mbar_expect_tx(&full_bar[slot], kFrameBytes);
            bulk_load(buf, a.x + c * a.x_ch_stride + frame * a.hop, kFrameBytes, &full_bar[slot]);
        }
    }

    for (; f < f_end; ++f) {
        float2 v[E];
        {
            // the window multiply rides on the first radix-2 stage of the butterfly (bfly_big_scaled)
            float w[RA];
#pragma unroll
            for (int r = 0; r < RA; ++r) w[r] = __ldg(wp + r * RB);
            if constexpr (STAGED) {
                mbar_wait(&full_bar[slot], parity);
                parity ^= 1;
#pragma unroll
                for (int r = 0; r < RA; ++r) v[r] = buf[ltid + r * RB];
            } else {
                const float2* src = a.x + c * a.x_ch_stride + frame * a.hop + ltid;
#pragma unroll
                for (int r = 0; r < RA; ++r) v[r] = ldg_stream(src + r * RB);
            }
            bfly_big_scaled<RA>(v, w);
        }

        slot_sync();                             // every thread of the slot has read the previous frame's M
        {
            float4* row = reinterpret_cast<float4*>(buf + ltid * ROW);
#pragma unroll
            for (int k = 0; k < RA; k += 2) row[k / 2] = make_float4(v[k].x, v[k].y, v[k + 1].x, v[k + 1].y);
        }
        slot_sync();

#pragma unroll
        for (int q = 0; q < NB; ++q) {
            const int jB = ltid + q * TPF;
            float2* u = v + q * RB;
#pragma unroll
            for (int r = 0; r < RB; ++r) u[r] = buf[r * ROW + jB];
        }
        // (channel, frame) of the next item
        const long long c_cur = c, frame_cur = frame;
        if (++frame == a.n_frames) { frame = 0; ++c; }
        if constexpr (STAGED) {
            slot_sync();                         // M has been read by every thread: the buffer is free
            if (ltid == 0 && f + 1 < f_end) {
                fence_proxy_async();             // generic-proxy reads above before the async-proxy writes
                mbar_expect_tx(&full_bar[slot], kFrameBytes);
                bulk_load(buf, a.x + c * a.x_ch_stride + frame * a.hop, kFrameBytes, &full_bar[slot]);
            }
        }
#pragma unroll
        for (int q = 0; q < NB; ++q) {
            const int jB = ltid + q * TPF;
            float2* u = v + q * RB;
            // pass-B twiddles A_k * B_b, products formed per first-stage butterfly and fused into it
            float2 A[C::NA8], B[8];
            A[0] = make_float2(1.f, 0.f);
            B[0] = make_float2(1.f, 0.f);
#pragma unroll
            for (int k = 1; k < C::NA8; ++k) A[k] = tw[(k - 1) * RA + jB];
#pragma unroll
            for (int b = 1; b < 8; ++b) B[b] = tw[(C::NA8 - 1 + b - 1) * RA + jB];
            bfly_big_twiddled<RB>(u, A, B);
        }

        const long long row0 = c_cur * a.out_ch_stride + frame_cur * (long long)nbins - a.bin_lo;
        if constexpr (MODE == IQW_STFT_DB) {
            // branch-free dB of all the thread's bins first (64 independent MUFU chains); the rare argument
            // that needs log10f (zero, denormal, inf, nan) is patched afterwards behind ONE branch per frame
            // (|X|^2 + eps is a normal float, or inf / nan which lg2 passes on like log10f, whenever eps is a normal
            // float: then nothing needs checking)
            if (a.eps >= 1.17549435e-38f) {
#pragma unroll
                for (int i = 0; i < E; ++i) {
                    bool ok;
                    v[i].x = power_to_dB_fast(v[i].x * v[i].x + v[i].y * v[i].y + a.eps, ok);
                }
            } else {
                bool all_ok = true;
#pragma unroll
                for (int i = 0; i < E; ++i) {
                    const float arg = fabsf(v[i].x * v[i].x + v[i].y * v[i].y) + a.eps;
                    bool ok;
                    const float d = power_to_dB_fast(arg, ok);
                    all_ok &= ok;
                    v[i] = make_float2(d, arg);
                }
                if (!all_ok) {
#pragma unroll
                    for (int i = 0; i < E; ++i)
                        if (!dB_fast_ok(v[i].y)) v[i].x = power_to_dB_slow(v[i].y);
                }
            }
        }
#pragma unroll
        for (int q = 0; q < NB; ++q)
#pragma unroll
            for (int r = 0; r < RB; ++r) {
                const int k = ltid + q * TPF + r * RA;
                if (FULLBAND || (k >= a.bin_lo && k < a.bin_hi)) {
                    const float2 X = v[q * RB + r];
                    if constexpr (MODE == IQW_STFT_COMPLEX) {
                        __stcs(reinterpret_cast<float2*>(a.out) + row0 + k, X);
                    } else if constexpr (MODE == IQW_STFT_DB) {
                        __stcs(reinterpret_cast<float*>(a.out) + row0 + k, X.x);
                    } else {
                        __stcs(reinterpret_cast<float*>(a.out) + row0 + k, X.x * X.x + X.y * X.y);
                    }
                }
            }
    }
}

// W_N^(r*jB) tables of the two-pass kernels, one immutable table per (device, log2 nfft)
__global__ void twiddle2p_init_kernel(float2* tw, int n, int ra, int rb) {
    const int na8 = rb / 8;
    const int count = (na8 - 1 + 7) * ra;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < count; e += gridDim.x * blockDim.x) {
        const int row = e / ra, j = e % ra;
        const int r = row < na8 - 1 ? 8 * (row + 1) : row - (na8 - 1) + 1;      // A rows: r = 8a, B rows: r = b
        double s, c;
        sincospi(-2.0 * (double)(r * j) / (double)n, &s, &c);
        tw[e] = make_float2((float)c, (float)s);
    }
}

template <int LOG2N>
static int get_twiddles2p(cudaStream_t stream, const float2** out) {
    return device_table(kTwoPassTwiddles, LOG2N, P2Cfg<LOG2N, true>::TW,
                        [](float2* d, int, cudaStream_t s) {
                            using C = P2Cfg<LOG2N, true>;
                            twiddle2p_init_kernel<<<16, 256, 0, s>>>(d, C::N, C::RA, C::RB);
                        },
                        stream, out);
}

template <int LOG2N, int MODE, bool FULLBAND, bool STAGED>
static int launch2p_staged(StftArgs a, cudaStream_t stream) {
    using C = P2Cfg<LOG2N, STAGED>;
    auto kern = stft2p_kernel<LOG2N, MODE, FULLBAND, STAGED>;
    if (int rc = get_twiddles2p<LOG2N>(stream, &a.twiddle)) return rc;
    long long grid = 0;
    if (int rc = resident_ctas(kern, C::THREADS, C::SMEM, "two-pass stft kernel", &grid)) return rc;
    const long long total = (long long)a.n_channels * a.n_frames;
    const long long need = (total + C::SLOTS - 1) / C::SLOTS;
    if (grid > need) grid = need;
    { IQW_PROFILE("stft_kernel", stream); kern<<<(unsigned)grid, C::THREADS, C::SMEM, stream>>>(a); }
    IQW_CUDA_OK(cudaGetLastError());
    return IQW_OK;
}

static std::atomic<int> g_stft_variant{0};   // 0 = auto, 1 = three-pass, 2 = two-pass with global loads, 3 = two-pass staged

// a bulk copy needs 16-byte aligned source addresses: every frame start of every channel
static bool frames_16B_aligned(const StftArgs& a) {
    return (reinterpret_cast<uintptr_t>(a.x) % 16 == 0) && (a.hop % 2 == 0) && (a.n_channels == 1 || a.x_ch_stride % 2 == 0);
}

template <int LOG2N, int MODE, bool FULLBAND>
static int launch2p_band(const StftArgs& a, cudaStream_t stream) {
    if (g_stft_variant.load() != 2 && frames_16B_aligned(a)) return launch2p_staged<LOG2N, MODE, FULLBAND, true>(a, stream);
    return launch2p_staged<LOG2N, MODE, FULLBAND, false>(a, stream);
}

template <int LOG2N>
static int launch2p(const StftArgs& a, int mode, cudaStream_t s) {
    const bool full = a.bin_lo == 0 && a.bin_hi == (1 << LOG2N);
    return dispatch_stft_mode(mode, [&](auto M) {
        return full ? launch2p_band<LOG2N, M, true>(a, s) : launch2p_band<LOG2N, M, false>(a, s);
    });
}

// ---------------------------------------------------------------------------------------------------
// Reducible statistics fused into the two-pass kernel (iqw_stft_reduce_c64 at nfft 1024 / 2048 / 4096):
// WARP SPECIALISATION.  A thread of the transform holds 64 values and has no registers left for 64 + 64
// running statistics, so the CTA carries a second role: PS producer slots run the two-pass transform
// exactly as stft2p_kernel does and, instead of storing |X|^2 to HBM, hand each frame to a consumer group
// through a per-slot power tile in shared memory (N floats) guarded by a full / empty mbarrier pair; the CT
// consumer threads own the bins k = ct + CT*i of EVERY frame of the CTA and keep their running max / min / sum
// in registers (two of the three: 128 registers).  Sums are flushed every 64 frames into a float64 partial row
// in global memory (two-level summation); max / min leave at the end.  Four consumer warps (a thread owns 32 / 16 / 8
// bins at nfft 4096 / 2048 / 1024) keep up with the eight producer warps; all three statistics fit their registers and
// the logarithms of a mean of dB values run there, beside the FMA-bound transform of the producers.  stft_reduce_combine_kernel
// (iqw_stft.cu) then combines the per-CTA rows.  Nothing is written per frame: 8 B/sample of HBM traffic.
// ---------------------------------------------------------------------------------------------------
static __device__ __noinline__ float power_to_dB_outlined(float p, float eps) { return power_to_dB(p, eps); }

#ifndef IQW_RED_FLUSH
#define IQW_RED_FLUSH 64
#endif
template <int LOG2N>
struct P2RCfg {
    using B = P2Cfg<LOG2N, true>;
    static constexpr int PS = LOG2N == 12 ? 4 : 8;                 // producer slots (8 producer warps)
    static constexpr int CT = 128;                                 // consumer threads: four warps keep up with eight producer warps
    static constexpr int BPT = B::N / CT;                          // bins per consumer thread: 32 / 16 / 8
    static constexpr int PTHREADS = PS * B::TPF;                   // 256
    static constexpr int THREADS = PTHREADS + CT;                  // 384: 12 warps, 168 registers per thread
    static constexpr size_t SMEM = sizeof(float2) * ((size_t)B::TW + (size_t)PS * B::BUF) + sizeof(float) * (size_t)PS * B::N;
};

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// FLAGS: bit 0 = max, bit 1 = min, bit 2 = sum (of dB values when a.reduce_dB)
template <int LOG2N, int FLAGS, bool STAGED>
__global__ void __launch_bounds__(P2RCfg<LOG2N>::THREADS, 1)
stft2p_reduce_kernel(const StftArgs a) {
    using C = P2Cfg<LOG2N, true>;
    using R = P2RCfg<LOG2N>;
    constexpr int RA = C::RA, RB = C::RB, E = C::E, TPF = C::TPF, NB = C::NB, ROW = C::ROW, N = C::N;
    constexpr int PS = R::PS, CT = R::CT, BPT = R::BPT;
    constexpr bool WMAX = (FLAGS & 1) != 0, WMIN = (FLAGS & 2) != 0, WSUM = (FLAGS & 4) != 0;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* tw = reinterpret_cast<float2*>(smem_raw);
    float* ptiles = reinterpret_cast<float*>(tw + C::TW + (size_t)PS * C::BUF);
    __shared__ __align__(8) uint64_t in_bar[PS], full_bar[PS], empty_bar[PS];
    for (int i = threadIdx.x; i < C::TW; i += R::THREADS) tw[i] = a.twiddle[i];
    if (threadIdx.x < PS) {
        mbar_init(&in_bar[threadIdx.x], 1);
        mbar_init(&full_bar[threadIdx.x], TPF);
        mbar_init(&empty_bar[threadIdx.x], CT);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    fence_proxy_async();
    __syncthreads();

    // frame range of every producer slot (the consumers need all of them)
    const long long total = a.n_frames;                                   // one channel per launch
    const long long n_slots = (long long)gridDim.x * PS;
    const long long per = (total + n_slots - 1) / n_slots;
    auto slot_begin = [&](int sl) { return ((long long)blockIdx.x * PS + sl) * per; };
    auto slot_end = [&](int sl) { const long long b = slot_begin(sl) + per; return b < total ? b : total; };

    if (threadIdx.x >= R::PTHREADS) {
        // ------------------------------ consumer ------------------------------
        const int ct = threadIdx.x - R::PTHREADS;
        float mx[WMAX ? BPT : 1], mn[WMIN ? BPT : 1], sm[WSUM ? BPT : 1];
#pragma unroll
        for (int i = 0; i < BPT; ++i) {
            if (WMAX) mx[i] = -INFINITY;
            if (WMIN) mn[i] = INFINITY;
            if (WSUM) sm[i] = 0.f;
        }
        const long long part = (long long)blockIdx.x * N;
        if (WSUM) {
#pragma unroll
            for (int i = 0; i < BPT; ++i) a.part_sum[part + ct + CT * i] = 0.0;
        }
        long long cnt[PS], most = 0;
#pragma unroll
        for (int sl = 0; sl < PS; ++sl) {
            cnt[sl] = slot_end(sl) - slot_begin(sl);
            if (cnt[sl] < 0) cnt[sl] = 0;
            most = cnt[sl] > most ? cnt[sl] : most;
        }
        // slots take consecutive frame ranges of (almost) equal length: slot sl has a frame in iteration `it` iff
        // it < cnt[sl], and the counts do not increase with sl
        long long cnt_min = cnt[PS - 1];
        int since = 0;
        // |X|^2 >= 0, so |X|^2 + eps is a normal float whenever eps is one
        const bool direct_lg2 = a.reduce_dB && a.eps >= 1.17549435e-38f;
        const float sum_scale = direct_lg2 ? 3.01029995663981195f : 1.f;
        for (long long it = 0; it < most; ++it) {
            int live = PS;          // slots with a frame in this iteration
            if (it >= cnt_min) {
                live = 0;
#pragma unroll
                for (int sl = 0; sl < PS; ++sl) live += it < cnt[sl] ? 1 : 0;
            }
#pragma unroll 1
            for (int sl = 0; sl < live; ++sl) {
                mbar_wait(&full_bar[sl], (uint32_t)(it & 1));
                const float* pt = ptiles + sl * N + ct;
                // the tile is taken 16 values at a time (reading all 32 first and handing the tile back earlier was
                // measured: more live registers, 5.4 against 5.1 ms at nfft 4096)
                constexpr int QB = BPT < 16 ? BPT : 16;
#pragma unroll
                for (int h = 0; h < BPT; h += QB) {
                    float p[QB];
#pragma unroll
                    for (int j = 0; j < QB; ++j) p[j] = pt[CT * (h + j)];
                    if (h + QB >= BPT) mbar_arrive(&empty_bar[sl]);       // last read issued: the tile may be overwritten
#pragma unroll
                    for (int j = 0; j < QB; ++j) {
                        if (WMAX) mx[h + j] = fmaxf(mx[h + j], p[j]);
                        if (WMIN) mn[h + j] = fminf(mn[h + j], p[j]);
                    }
                    if (WSUM) {
                        if (a.reduce_dB && direct_lg2) {
                            // p + eps is a normal float (or inf / nan, which lg2 passes on as numpy does): ONE lg2 per value,
                            // summed in log2 units and scaled when the sum is flushed -- three instructions per value.  (The
                            // split into exponent and mantissa that the spectrogram epilogue uses keeps every single value
                            // within 5e-5 dB; a mean over frames does not need that, lg2.approx is within 2^-22 relative.)
#pragma unroll
                            for (int j = 0; j < QB; ++j) {
                                float l;
                                asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(p[j] + a.eps));
                                sm[h + j] += l;
                            }
                        } else if (a.reduce_dB) {
                            // eps is zero or denormal (not what the persistence spectrum passes): the checked logarithm,
                            // out of line -- the consumers' loop must stay small, the instruction cache is shared with
                            // the producers' transform
#pragma unroll
                            for (int j = 0; j < QB; ++j) sm[h + j] += power_to_dB_outlined(p[j], a.eps);
                        } else {
#pragma unroll
                            for (int j = 0; j < QB; ++j) sm[h + j] += p[j];
                        }
                    }
                }
                if (WSUM) {
                    if (++since == IQW_RED_FLUSH) {                       // two-level summation
                        since = 0;
#pragma unroll
                        for (int i = 0; i < BPT; ++i) { a.part_sum[part + ct + CT * i] += (double)(sm[i] * sum_scale); sm[i] = 0.f; }
                    }
                }
            }
        }
#pragma unroll
        for (int i = 0; i < BPT; ++i) {
            const long long k = part + ct + CT * i;
            a.part_max[k] = WMAX ? mx[i] : -INFINITY;
            a.part_min[k] = WMIN ? mn[i] : INFINITY;
            if (WSUM) a.part_sum[k] += (double)(sm[i] * sum_scale);
            else a.part_sum[k] = 0.0;
        }
        return;
    }

    // ------------------------------ producers: the two-pass transform of stft2p_kernel ------------------------------
    const int slot = threadIdx.x / TPF;
    const int ltid = threadIdx.x % TPF;
    float2* buf = tw + C::TW + (size_t)slot * C::BUF;
    float* ptile = ptiles + slot * N;
    constexpr uint32_t kFrameBytes = (uint32_t)(N * sizeof(float2));
    auto slot_sync = [&]() {
        if constexpr (TPF == 32) __syncwarp();
        else asm volatile("bar.sync %0, %1;" ::"r"(slot + 1), "n"(TPF) : "memory");
    };
    long long frame = slot_begin(slot);
    const long long f_end = slot_end(slot);
    if (frame >= f_end) return;
    const float* wp = a.window + ltid;
    uint32_t parity = 0;
    if constexpr (STAGED) {
        if (ltid == 0) {
            mbar_expect_tx(&in_bar[slot], kFrameBytes);
            bulk_load(buf, a.x + frame * a.hop, kFrameBytes, &in_bar[slot]);
        }
    }
    for (long long it = 0; frame < f_end; ++frame, ++it) {
        float2 v[E];
        {
            float w[RA];
#pragma unroll
            for (int r = 0; r < RA; ++r) w[r] = __ldg(wp + r * RB);
            if constexpr (STAGED) {
                mbar_wait(&in_bar[slot], parity);
                parity ^= 1;
#pragma unroll
                for (int r = 0; r < RA; ++r) v[r] = buf[ltid + r * RB];
            } else {
                const float2* src = a.x + frame * a.hop + ltid;
#pragma unroll
                for (int r = 0; r < RA; ++r) v[r] = ldg_stream(src + r * RB);
            }
            bfly_big_scaled<RA>(v, w);
        }
        slot_sync();
        {
            float4* row = reinterpret_cast<float4*>(buf + ltid * ROW);
#pragma unroll
            for (int k = 0; k < RA; k += 2) row[k / 2] = make_float4(v[k].x, v[k].y, v[k + 1].x, v[k + 1].y);
        }
        slot_sync();
#pragma unroll
        for (int q = 0; q < NB; ++q) {
            const int jB = ltid + q * TPF;
            float2* u = v + q * RB;
#pragma unroll
            for (int r = 0; r < RB; ++r) u[r] = buf[r * ROW + jB];
        }
        if constexpr (STAGED) {
            slot_sync();
            if (ltid == 0 && frame + 1 < f_end) {
                fence_proxy_async();
                mbar_expect_tx(&in_bar[slot], kFrameBytes);
                bulk_load(buf, a.x + (frame + 1) * a.hop, kFrameBytes, &in_bar[slot]);
            }
        }
#pragma unroll
        for (int q = 0; q < NB; ++q) {
            const int jB = ltid + q * TPF;
            float2* u = v + q * RB;
            float2 A[C::NA8], B[8];
            A[0] = make_float2(1.f, 0.f);
            B[0] = make_float2(1.f, 0.f);
#pragma unroll
            for (int k = 1; k < C::NA8; ++k) A[k] = tw[(k - 1) * RA + jB];
#pragma unroll
            for (int b = 1; b < 8; ++b) B[b] = tw[(C::NA8 - 1 + b - 1) * RA + jB];
            bfly_big_twiddled<RB>(u, A, B);
        }
        // the frame's power
#pragma unroll
        for (int i = 0; i < E; ++i) v[i].x = v[i].x * v[i].x + v[i].y * v[i].y;
        // hand it to the consumers (wait until they have taken the previous frame of this slot)
        if (it > 0) mbar_wait(&empty_bar[slot], (uint32_t)((it - 1) & 1));
#pragma unroll
        for (int q = 0; q < NB; ++q)
#pragma unroll
            for (int r = 0; r < RB; ++r) ptile[ltid + q * TPF + r * RA] = v[q * RB + r].x;
        mbar_arrive(&full_bar[slot]);
    }
}

template <int LOG2N, int FLAGS>
static int launch2p_reduce_flags(StftArgs a, long long* n_parts, cudaStream_t stream) {
    using R = P2RCfg<LOG2N>;
    const bool staged = g_stft_variant.load() != 2 && frames_16B_aligned(a);
    if (int rc = get_twiddles2p<LOG2N>(stream, &a.twiddle)) return rc;
    int sms = 0;
    if (int rc = device_sm_count(&sms)) return rc;
    long long grid = sms;
    const long long need = (a.n_frames + R::PS - 1) / R::PS;
    if (grid > need) grid = need;
    *n_parts = grid;
    if (staged) {
        auto kern = stft2p_reduce_kernel<LOG2N, FLAGS, true>;
        IQW_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)R::SMEM));
        IQW_PROFILE("stft_reduce_kernel", stream);
        kern<<<(unsigned)grid, R::THREADS, R::SMEM, stream>>>(a);
    } else {
        auto kern = stft2p_reduce_kernel<LOG2N, FLAGS, false>;
        IQW_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)R::SMEM));
        IQW_PROFILE("stft_reduce_kernel", stream);
        kern<<<(unsigned)grid, R::THREADS, R::SMEM, stream>>>(a);
    }
    IQW_CUDA_OK(cudaGetLastError());
    return IQW_OK;
}

// flags: bit 0 max, bit 1 min, bit 2 sum; returns IQW_ERR_UNSUPPORTED, without an error message, for an nfft or
// flags that are not built here (the caller then takes the three-pass kernel)
int launch_stft_two_pass_reduce(const StftArgs& a, int log2n, int flags, long long* n_parts, cudaStream_t stream) {
    auto unsupported = [] { return IQW_ERR_UNSUPPORTED; };
    return dispatch<10, 12>(log2n, [&](auto L) {
        return dispatch<1, 7>(flags, [&](auto F) { return launch2p_reduce_flags<L, F>(a, n_parts, stream); }, unsupported);
    }, unsupported);
}

int stft_variant() { return g_stft_variant.load(); }

bool stft_two_pass_wanted(int log2n) {
    if (log2n < 10 || log2n > 12) return false;
    return g_stft_variant.load() != 1;
}

int launch_stft_two_pass(const StftArgs& a, int log2n, int mode, cudaStream_t stream) {
    return dispatch<10, 12>(log2n, [&](auto L) { return launch2p<L>(a, mode, stream); },
                            [&] { return fail(IQW_ERR_UNSUPPORTED, "two-pass stft: nfft=%d", 1 << log2n); });
}

}  // namespace iqw

extern "C" int iqw_debug_set_stft_variant(int variant) {
    if (variant < 0 || variant > 3)
        return iqw::fail(IQW_ERR_INVALID, "variant must be 0 (auto), 1 (three-pass), 2 (two-pass, global loads) or 3 (two-pass, staged)");
    iqw::g_stft_variant.store(variant);
    return IQW_OK;
}
