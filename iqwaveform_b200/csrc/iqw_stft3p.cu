// iqw_stft3p.cu -- kernel 1 for nfft 8192 .. 65536: ONE pass over the samples, the frame held in (distributed)
// shared memory, staged by bulk copies (TMA), exchanged across a thread-block cluster where it exceeds a CTA.
//
// Replaces, for these sizes, the two-kernel four-step path through an HBM scratch (iqw_stft_large.cu: 3.5x the
// algorithmic traffic, 19 % of the HBM peak at nfft 65536) and the three-pass kernel at nfft 8192 (38 %).  Same
// contract as iqw_stft_c64's other kernels (fourier.py:568-581 + 1044 + power_analysis.py:254-255, 199-204 +
// fourier.py:1295 of the reference in one pass).
//
// Geometry: N = 64 x 64 x R3 (R3 = N/4096 = 2, 4, 8, 16), 64 values per thread, a frame slot is TPF = N/64
// threads: 128 (nfft 8192, three slots per CTA), 256 (16384, one CTA), 512 / 1024 (32768 / 65536: a CLUSTER of
// 2 / 4 CTAs of 256 threads).  Stockham decimation in time:
//   pass A  radix 64, butterfly jA = t:   x[jA + r*TPF] * window, r < 64            -> index 64*jA + k
//   pass B  radix 64, butterfly jB = t:   in[jB + r*TPF] * W_4096^(r*(jB mod 64))   -> index (jB/64)*4096 + (jB mod 64) + 64*r
//   pass C  radix R3, butterflies jC = t + q*TPF (q < 64/R3): in[jC + r*4096] * W_N^(r*jC) -> bin jC + r*4096
// Exchange 1 (A -> B): thread jA owns the 64 consecutive elements 64*jA .. 64*jA+63, read by the 64 threads
// jB = 64*(jA mod R3) + k at r = jA div R3: it writes ONE padded 66-element segment with 128-bit stores and the
// readers read conflict-free / coalesced.  Exchange 2 (B -> C) is an R3 x R3 block transpose among the R3 threads
// that share jB mod 64, in a [slot][thread] layout.
//   * one CTA per frame (nfft 8192, 16384): both exchanges go through the CTA's shared memory (five barriers per
//     frame: a named barrier per slot / the CTA barrier).  The buffer is idle from the last read of exchange 2 to
//     the first write of exchange 1 of the next frame: exactly then the next frame is staged into it by ONE bulk
//     copy (cp.async.bulk, completion on an mbarrier) while pass C and the epilogue run.
//   * a cluster per frame (32768: 2 CTAs, 65536: 4 CTAs): the exchanges go through a per-cluster scratch in
//     global memory that never leaves the L2 (1 MB per cluster), ordered by TWO barrier.cluster (release / acquire)
//     per frame; shared memory only stages the samples (64 bulk copies of the 256 consecutive samples
//     x[r*TPF + 256*rank ..] per CTA) and is free again as soon as pass A has read them, so the next frame streams
//     in during the whole transform.  MEASURED AND REJECTED for this exchange: distributed shared memory
//     (st.shared::cluster into the readers' CTA): 20 % / 15 % of the HBM peak at nfft 32768 / 65536 with 256
//     threads per CTA, 17 % / 13 % with three 128-thread CTAs per SM -- remote shared-memory stores sustain only
//     ~20 B/clk per SM, an order of magnitude below the L2 path.
#include "iqw_stft.cuh"

namespace iqw {

template <int LOG2N>
struct P3Cfg {
    static constexpr int N = 1 << LOG2N;
    static constexpr int R3 = N / 4096;                  // radix of the third pass
    static constexpr int TPF = N / 64;                   // threads per frame
    static constexpr int TPC = TPF < 256 ? TPF : 256;    // threads of one frame inside one CTA
    static constexpr int NC = TPF / TPC;                 // CTAs per frame (cluster size): 1, 2, 4, 8
#ifndef IQW_P3_SLOTS13
#define IQW_P3_SLOTS13 3
#endif
    static constexpr int SLOTS = NC == 1 ? (TPC == 128 ? IQW_P3_SLOTS13 : 1) : 1;    // frame slots per CTA
    static constexpr int THREADS = SLOTS * TPC;          // 384, or 128 with three CTAs per SM
    static constexpr int MIN_BLOCKS = (NC > 1 && TPC == 128) ? 3 : 1;
    static constexpr int HL = R3 / NC;                   // groups of 64 threads per CTA and slot (2 or 4)
    static constexpr int SEG = 66;                       // padded 64-element segment (odd number of 16-byte units)
    static constexpr int BUF = TPC * SEG;                // float2 per slot and CTA
    static constexpr int TW = 14 * 64;                   // pass-B twiddles, factored (see iqw_stft2p.cu)
    static constexpr size_t SMEM = sizeof(float2) * ((size_t)TW + (size_t)SLOTS * BUF);
    // per-cluster exchange scratch in global memory (NC > 1): region 1 = TPF padded segments, region 2 = [64][TPF]
    static constexpr size_t X1 = (size_t)TPF * SEG, X2 = (size_t)64 * TPF;
    static constexpr size_t SCRATCH_BYTES = NC > 1 ? sizeof(float2) * (X1 + X2) : 0;
    static_assert(TPC == 64 * HL && R3 >= 2 && R3 <= 16, "geometry");
};

__device__ __forceinline__ uint32_t s3_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t s3_cluster_rank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void s3_mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(s3_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void s3_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(s3_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void s3_mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT3_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE3_%=;\n\t"
        "bra WAIT3_%=;\n\t"
        "DONE3_%=:\n\t}" ::"r"(s3_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void s3_bulk_load(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(s3_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(s3_u32(bar))
                 : "memory");
}

template <int LOG2N, int MODE>
__global__ void __launch_bounds__(P3Cfg<LOG2N>::THREADS, P3Cfg<LOG2N>::MIN_BLOCKS)
stft3p_kernel(const StftArgs a) {
    using C = P3Cfg<LOG2N>;
    constexpr int N = C::N, R3 = C::R3, TPF = C::TPF, NC = C::NC, TPC = C::TPC, HL = C::HL, SEG = C::SEG;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* tw = reinterpret_cast<float2*>(smem_raw);
    __shared__ __align__(8) uint64_t full_bar[C::SLOTS];
    for (int i = threadIdx.x; i < C::TW; i += C::THREADS) tw[i] = a.twiddle[i];
    if (threadIdx.x < C::SLOTS) s3_mbar_init(&full_bar[threadIdx.x], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();

    const int slot = threadIdx.x / TPC;
    const int lt = threadIdx.x % TPC;                    // thread of the slot inside this CTA
    const uint32_t crank = NC > 1 ? s3_cluster_rank() : 0u;
    const int gt = (int)crank * TPC + lt;                // thread of the frame: butterfly index of every pass
    const int l = lt & 63, hl = lt >> 6;                 // jB = 64*h + l with h = crank*HL + hl
    const int h = (int)crank * HL + hl;
    float2* buf = tw + C::TW + (size_t)slot * C::BUF;

    auto slot_sync = [&]() {              // one CTA per frame: the frame's threads
        if constexpr (C::SLOTS == 1) {
            __syncthreads();
        } else {
            asm volatile("bar.sync %0, %1;" ::"r"(slot + 1), "n"(TPC) : "memory");
        }
    };

    // pass-C twiddle bases W_N^(r*gt), r = 1 .. R3-1, once per kernel in float64
    float2 base[R3];
#pragma unroll
    for (int r = 1; r < R3; ++r) {
        double s, c;
        sincospi(-2.0 * (double)(r * gt) / (double)N, &s, &c);
        base[r] = make_float2((float)c, (float)s);
    }

    // contiguous range of (channel, frame) items for this slot (of this cluster)
    const long long total = (long long)a.n_channels * a.n_frames;
    const long long n_units = (long long)(gridDim.x / NC) * C::SLOTS;
    const long long per = (total + n_units - 1) / n_units;
    const long long sg = (long long)(blockIdx.x / NC) * C::SLOTS + slot;
    long long f = sg * per;
    const long long f_end = f + per < total ? f + per : total;
    if (f >= f_end) return;                              // the whole slot (all its CTAs) leaves together
    long long c = f / a.n_frames;
    long long frame = f - c * a.n_frames;
    const int nbins = a.bin_hi - a.bin_lo;
    const float* wp = a.window + gt;
    uint32_t parity = 0;

    // this CTA's samples of a frame: chunk r = x[r*TPF + crank*TPC .. + TPC), r < 64, at buf[r*TPC ..]
    auto stage = [&](const float2* fr) {
        if constexpr (NC == 1) {
            if (lt == 0) {
                s3_mbar_expect_tx(&full_bar[slot], (uint32_t)(N * sizeof(float2)));
                s3_bulk_load(buf, fr, (uint32_t)(N * sizeof(float2)), &full_bar[slot]);
            }
        } else {
            if (lt < 32) {
                if (lt == 0) s3_mbar_expect_tx(&full_bar[slot], (uint32_t)(64 * TPC * sizeof(float2)));
                __syncwarp();
#pragma unroll
                for (int r = lt; r < 64; r += 32)
                    s3_bulk_load(buf + r * TPC, fr + (long long)r * TPF + crank * TPC, (uint32_t)(TPC * sizeof(float2)),
                                 &full_bar[slot]);
            }
        }
    };
    stage(a.x + c * a.x_ch_stride + frame * a.hop);

    // (NC > 1) exchange scratch of this cluster in global memory
    float2* x1 = nullptr;
    float2* x2 = nullptr;
    if constexpr (NC > 1) {
        x1 = a.xscratch + (size_t)(blockIdx.x / NC) * (C::X1 + C::X2);
        x2 = x1 + C::X1;
    }
    auto cluster_sync = [&]() {
        asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
    };

    for (; f < f_end; ++f) {
        float2 v[64];
        {
            float w[64];
#pragma unroll
            for (int r = 0; r < 64; ++r) w[r] = __ldg(wp + r * TPF);
            s3_mbar_wait(&full_bar[slot], parity);
            parity ^= 1;
#pragma unroll
            for (int r = 0; r < 64; ++r) v[r] = buf[r * TPC + lt];
            bfly_big_scaled<64>(v, w);                   // window fused into the first radix-2 stage; v[k] = element 64*gt + k
        }
        const long long c_cur = c, frame_cur = frame;
        if (++frame == a.n_frames) { frame = 0; ++c; }
        if constexpr (NC > 1) {
            // shared memory only stages the samples: free as soon as every thread of the CTA has read its own
            __syncthreads();
            if (f + 1 < f_end) {
                if (lt < 32) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                stage(a.x + c * a.x_ch_stride + frame * a.hop);
            }
        }

        if constexpr (NC == 1) {
            slot_sync();                                 // 1: every thread of the frame has read its samples
            // segment gt is read by jB = 64*(gt mod R3) + k at r = gt / R3: local segment (gt / R3)*HL + gt mod R3
            float4* row = reinterpret_cast<float4*>(buf + ((gt / R3) * HL + (gt % R3)) * SEG);
#pragma unroll
            for (int k = 0; k < 64; k += 2) row[k / 2] = make_float4(v[k].x, v[k].y, v[k + 1].x, v[k + 1].y);
            slot_sync();                                 // 2
#pragma unroll
            for (int r = 0; r < 64; ++r) v[r] = buf[(r * HL + hl) * SEG + l];
            slot_sync();                                 // 3: exchange 1 has been read everywhere
        } else {
            float4* row = reinterpret_cast<float4*>(x1 + (size_t)gt * SEG);
#pragma unroll
            for (int k = 0; k < 64; k += 2) __stcg(row + k / 2, make_float4(v[k].x, v[k].y, v[k + 1].x, v[k + 1].y));
            cluster_sync();                              // exchange 1 written by every CTA of the frame
#pragma unroll
            for (int r = 0; r < 64; ++r) v[r] = __ldcg(x1 + (size_t)(r * R3 + h) * SEG + l);
        }

        // pass B: W_4096^(r*l), r = 8k + b, factored A_k * B_b (table of the two-pass kernel at nfft 4096), the
        // products formed per first-stage butterfly and fused into it
        {
            float2 A[8], B[8];
            A[0] = make_float2(1.f, 0.f);
            B[0] = make_float2(1.f, 0.f);
#pragma unroll
            for (int k = 1; k < 8; ++k) A[k] = tw[(k - 1) * 64 + l];
#pragma unroll
            for (int b = 1; b < 8; ++b) B[b] = tw[(7 + b - 1) * 64 + l];
            bfly_big_twiddled<64>(v, A, B);              // v[r] = element h*4096 + l + 64*r
        }

        // exchange 2: element r goes to thread 64*(r mod R3) + l of the frame, slot (r / R3)*R3 + h
        if constexpr (NC == 1) {
#pragma unroll
            for (int r = 0; r < 64; ++r) buf[((r / R3) * R3 + h) * TPC + 64 * (r % R3) + l] = v[r];
            slot_sync();                                 // 4
#pragma unroll
            for (int s = 0; s < 64; ++s) v[s] = buf[s * TPC + lt];
            slot_sync();                                 // 5: the buffer is free: stage the next frame into it
            if (f + 1 < f_end) {
                if (lt < 32) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                stage(a.x + c * a.x_ch_stride + frame * a.hop);
            }
        } else {
#pragma unroll
            for (int r = 0; r < 64; ++r) __stcg(x2 + (size_t)((r / R3) * R3 + h) * TPF + 64 * (r % R3) + l, v[r]);
            cluster_sync();                              // exchange 2 written; every CTA has also read exchange 1
#pragma unroll
            for (int s = 0; s < 64; ++s) v[s] = __ldcg(x2 + (size_t)s * TPF + gt);
            // (the next frame's exchange 1 is written only after this CTA's next barrier-free stretch; a peer
            // may overwrite region 1 now -- everyone has read it -- and region 2 only after the next
            // cluster_sync, which this CTA reaches after the loads above have returned)
        }

        // pass C: butterfly q takes v[q*R3 + r], r < R3, times W_N^(r*(gt + q*TPF)) = base[r] * W_64^(r*q)
#pragma unroll
        for (int q = 0; q < 64 / R3; ++q) {
#pragma unroll
            for (int r = 1; r < R3; ++r) {
                const float2 t = q == 0 ? base[r] : mul_w64(base[r], (r * q) & 63);
                v[q * R3 + r] = cmul(v[q * R3 + r], t);
            }
            bfly<R3, 1>(v + q * R3);                    // v[q*R3 + r] = bin gt + q*TPF + r*4096
        }

        const long long row0 = c_cur * a.out_ch_stride + frame_cur * (long long)nbins - a.bin_lo;
        if constexpr (MODE == IQW_STFT_DB) {
            bool all_ok = true;
#pragma unroll
            for (int i = 0; i < 64; ++i) {
                const float arg = fabsf(v[i].x * v[i].x + v[i].y * v[i].y) + a.eps;
                bool ok;
                const float d = power_to_dB_fast(arg, ok);
                all_ok &= ok;
                v[i] = make_float2(d, arg);
            }
            if (!all_ok) {
#pragma unroll
                for (int i = 0; i < 64; ++i)
                    if (!dB_fast_ok(v[i].y)) v[i].x = power_to_dB_slow(v[i].y);
            }
        }
#pragma unroll
        for (int q = 0; q < 64 / R3; ++q)
#pragma unroll
            for (int r = 0; r < R3; ++r) {
                const int k = gt + q * TPF + r * 4096;
                if (k >= a.bin_lo && k < a.bin_hi) {
                    const float2 X = v[q * R3 + r];
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
    if constexpr (NC > 1) cluster_sync();                // no CTA of a cluster leaves while a peer still runs
}

// pass-B twiddle table: rows A_1..A_7 = W_4096^(8k*l), rows B_1..B_7 = W_4096^(b*l), l < 64
__global__ void twiddle3p_init_kernel(float2* tw) {
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < 14 * 64; e += gridDim.x * blockDim.x) {
        const int row = e / 64, j = e % 64;
        const int r = row < 7 ? 8 * (row + 1) : row - 7 + 1;
        double s, c;
        sincospi(-2.0 * (double)(r * j) / 4096.0, &s, &c);
        tw[e] = make_float2((float)c, (float)s);
    }
}

template <int LOG2N, int MODE>
static int launch3p_mode(StftArgs a, void* ws, size_t ws_bytes, cudaStream_t stream) {
    using C = P3Cfg<LOG2N>;
    auto kern = stft3p_kernel<LOG2N, MODE>;
    if (int rc = device_table(kThreePassTwiddles, 0, 14 * 64,
                              [](float2* d, int, cudaStream_t s) { twiddle3p_init_kernel<<<4, 256, 0, s>>>(d); }, stream,
                              &a.twiddle))
        return rc;
    IQW_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM));
    int sms = 0;
    if (int rc = device_sm_count(&sms)) return rc;
    const long long total = (long long)a.n_channels * a.n_frames;
    cudaLaunchConfig_t cfg{};
    cfg.blockDim = dim3(C::THREADS);
    cfg.dynamicSmemBytes = C::SMEM;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = C::NC;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    long long clusters = (long long)sms * C::MIN_BLOCKS / C::NC;
    if constexpr (C::NC > 1) {
        cfg.gridDim = dim3((unsigned)(clusters * C::NC));
        int max_clusters = 0;
        IQW_CUDA_OK(cudaOccupancyMaxActiveClusters(&max_clusters, kern, &cfg));
        if (max_clusters < 1) return fail(IQW_ERR_CUDA, "stft nfft=%d: no cluster of %d CTAs fits", C::N, C::NC);
        if (clusters > max_clusters) clusters = max_clusters;
    }
    const long long need = (total + C::SLOTS - 1) / C::SLOTS;
    if (clusters > need) clusters = need;
    if constexpr (C::NC > 1) {
        // exchange scratch: as many clusters as the caller's workspace covers (it stays in the L2)
        const long long fit = (long long)(ws ? ws_bytes / C::SCRATCH_BYTES : 0);
        if (fit < 1) return fail(IQW_ERR_WORKSPACE, "stft nfft=%d: workspace %zu bytes < %zu for one cluster", C::N, ws_bytes, C::SCRATCH_BYTES);
        if (clusters > fit) clusters = fit;
        a.xscratch = static_cast<float2*>(ws);
    }
    cfg.gridDim = dim3((unsigned)(clusters * C::NC));
    { IQW_PROFILE("stft_kernel", stream); IQW_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, a)); }
    IQW_CUDA_OK(cudaGetLastError());
    return IQW_OK;
}

// a bulk copy needs 16-byte aligned source addresses: every frame start of every channel
bool stft_three_pass_cluster_ok(const StftArgs& a, int log2n) {
    if (log2n < 13 || log2n > 16) return false;
    return (reinterpret_cast<uintptr_t>(a.x) % 16 == 0) && (a.hop % 2 == 0) && (a.n_channels == 1 || a.x_ch_stride % 2 == 0);
}

// bytes of exchange scratch the cluster kernels want (nfft 32768 / 65536): one region pair per resident cluster
size_t stft_three_pass_scratch_bytes(int log2n, long long n_channels, long long n_frames) {
    if (log2n < 15 || log2n > 16 || n_channels < 1 || n_frames < 1) return 0;
    int sms = 0;
    if (device_sm_count(&sms) != IQW_OK) sms = 160;
    const long long nc = log2n == 15 ? P3Cfg<15>::NC : P3Cfg<16>::NC;
    long long clusters = sms / nc;
    if (clusters > n_channels * n_frames) clusters = n_channels * n_frames;
    return (size_t)clusters * (log2n == 15 ? P3Cfg<15>::SCRATCH_BYTES : P3Cfg<16>::SCRATCH_BYTES);
}

int launch_stft_three_pass_cluster(const StftArgs& a, int log2n, int mode, void* ws, size_t ws_bytes, cudaStream_t stream) {
    return dispatch<13, 16>(
        log2n,
        [&](auto L) { return dispatch_stft_mode(mode, [&](auto M) { return launch3p_mode<L, M>(a, ws, ws_bytes, stream); }); },
        [&] { return fail(IQW_ERR_UNSUPPORTED, "cluster stft: nfft=%d", 1 << log2n); });
}

}  // namespace iqw
