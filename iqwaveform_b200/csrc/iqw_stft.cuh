// iqw_stft.cuh -- pieces of the STFT kernels shared by iqw_stft.cu (nfft <= 8192, one CTA per frame
// group) and iqw_stft_large.cu (nfft 16384..65536, two-kernel four-step).
#pragma once
#include "iqw_common.cuh"
#include "fft_core.cuh"

namespace iqw {

struct StftArgs {
    const float2* x;
    long long n_samples, x_ch_stride;
    int n_channels;
    const float* window;
    const float2* twiddle;
    long long hop, n_frames;
    float eps;
    int bin_lo, bin_hi;
    void* out;
    long long out_ch_stride;
    long long n_groups;        // n_channels * groups_per_channel
    long long groups_per_ch;   // ceil(n_frames / FPC)
    // MODE == kStftReduce (iqw_stft_reduce_c64): nothing is stored per frame; every frame slot keeps the
    // running max / min / sum over its frames of each bin it owns and writes one partial row at the end
    float* part_max;           // [n_parts][nfft]
    float* part_min;
    double* part_sum;          // sum of the power, or of its dB when reduce_dB
    int reduce_dB;
    int reduce_flags;          // bit 0: max / min wanted, bit 1: sum wanted
    float2* xscratch;          // cluster kernels (nfft 32768 / 65536): per-cluster exchange scratch in global memory
};

constexpr int kStftReduce = 3;   // internal mode of stft_kernel, next to IQW_STFT_COMPLEX / POWER / DB

// f(std::integral_constant<int, mode>{}) for the output modes IQW_STFT_COMPLEX / POWER / DB
template <class F>
int dispatch_stft_mode(int mode, F&& f) {
    return dispatch<IQW_STFT_COMPLEX, IQW_STFT_DB>(mode, f, [&] { return fail(IQW_ERR_INVALID, "unknown stft mode %d", mode); });
}

// geometry of the in-CTA FFT (shared by the forward kernel, iqw_stft.cu, and the inverse one,
// iqw_istft.cu)
template <int LOG2N>
struct StftCfg {
    static constexpr int N = 1 << LOG2N;
    static constexpr int E = plan_elems(LOG2N);
    static constexpr int TPF = N / E;                           // threads per frame
    static constexpr int THREADS = TPF >= 256 ? TPF : 256;
    static constexpr int FPC = THREADS / TPF;                   // frames per CTA iteration
    static constexpr int NP = plan_passes(LOG2N);
    static constexpr int TW = plan_tw_size(LOG2N);
    static constexpr int TW_ALLOC = (TW + 15) & ~15;
    static constexpr int PADN = padded_size(N);
    static constexpr int NBUF = NP > 1 ? 2 : 0;
    static constexpr size_t SMEM = sizeof(float2) * ((size_t)TW_ALLOC + (size_t)NBUF * FPC * PADN);
    // CTAs per SM we aim for (register budget = 65536 / (THREADS * MIN_BLOCKS))
    static constexpr int MIN_BLOCKS = THREADS >= 512 ? 1 : 2;
};

template <int LOG2N, int P>
struct PassLoop {
    // runs passes P..NP-1; `par` selects the ping-pong buffer the NEXT exchange writes.  The
    // twiddles of pass P+1 are fetched before the barrier that separates it from pass P.
    static __device__ __forceinline__ void run(float2* v, float2* bufs, const float2* tw, const float2* t,
                                               int ltid, int slot, int& par) {
        using C = StftCfg<LOG2N>;
        constexpr bool LAST = (P == C::NP - 1);
        float2* wr = bufs + ((size_t)par * C::FPC + slot) * C::PADN;
        const float2* rd = bufs + ((size_t)(par ^ 1) * C::FPC + slot) * C::PADN;
        fft_pass<LOG2N, P>(v, rd, wr, t, ltid);
        if constexpr (!LAST) {
            constexpr int E = plan_elems(LOG2N);
            float2 tn[E];
            load_twiddles<LOG2N, P + 1>(tn, tw, ltid);
            // only the threads of this frame slot exchange data: a named barrier per slot when a
            // slot is made of whole warps, a warp barrier when it fits in one warp, the CTA barrier otherwise
            if constexpr (C::TPF <= 32)
                __syncwarp();                       // the slot lives inside one warp
            else if constexpr (C::FPC > 1 && C::TPF % 32 == 0)
                asm volatile("bar.sync %0, %1;" ::"r"(slot + 1), "n"(C::TPF) : "memory");
            else
                __syncthreads();
            par ^= 1;
            PassLoop<LOG2N, P + 1>::run(v, bufs, tw, tn, ltid, slot, par);
        }
    }
};

// immutable per-(device, log2 n) twiddle table of the in-CTA FFT (built on first use)
int get_twiddles(int log2n, cudaStream_t stream, const float2** out);

// nfft 1024 / 2048 / 4096, two-pass geometry (iqw_stft2p.cu)
bool stft_two_pass_wanted(int log2n);
int launch_stft_two_pass(const StftArgs& a, int log2n, int mode, cudaStream_t stream);

// reducible statistics fused into the two-pass kernel (warp-specialised; iqw_stft2p.cu).  flags: bit 0 max, bit 1 min,
// bit 2 sum; IQW_ERR_UNSUPPORTED (no error message) outside nfft 1024..4096 and flags 1..7.  Leaves *n_parts partial rows in a.part_max / min / sum.
int launch_stft_two_pass_reduce(const StftArgs& a, int log2n, int flags, long long* n_parts, cudaStream_t stream);

// nfft 8192 .. 65536 in one pass: frame in (distributed) shared memory, cluster of 1 / 1 / 2 / 4 CTAs (iqw_stft3p.cu)
bool stft_three_pass_cluster_ok(const StftArgs& a, int log2n);
size_t stft_three_pass_scratch_bytes(int log2n, long long n_channels, long long n_frames);
int launch_stft_three_pass_cluster(const StftArgs& a, int log2n, int mode, void* workspace, size_t workspace_bytes,
                                   cudaStream_t stream);
int stft_variant();      // iqw_debug_set_stft_variant

// nfft = 2^14 .. 2^16 (iqw_stft_large.cu)
size_t stft_large_workspace_bytes(int log2n, long long n_channels, long long n_frames);
int launch_stft_large(const StftArgs& a, int log2n, int mode, void* workspace, size_t workspace_bytes,
                      cudaStream_t stream);

}  // namespace iqw
