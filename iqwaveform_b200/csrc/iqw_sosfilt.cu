// iqw_sosfilt.cu -- kernel 10: IIR filtering of complex64 rows by a cascade of S <= 16 second-order sections in
// direct form II transposed (scipy.signal.sosfilt semantics), real fp32 coefficients.
//
// The cascade is one linear system of 2S states z = (z1_0, z2_0, z1_1, ...) (scipy's zi order):
// z[n+1] = A z[n] + B x[n].  A row is cut into chunks of L samples and groups of G chunks (one CTA), all anchored
// at sample 0, and groups into carry blocks of H groups.  L, G and H depend on S alone (iqw_sosfilt_geometry), so every
// output is a function of its row alone: a row alone or in a batch, and time shards on group boundaries, give
// the same bits.
//
//   sosfilt_chunk_kernel<S, false> (states) one thread per chunk runs the fp32 cascade over its chunk from a zero state and keeps
//     the final state b_c (complex64, to the workspace); the CTA folds its G states t <- P t + b_c in float64,
//     P = A^L, into the zero-state final state b_g of the group.
//   sos_fold_kernel x 3    the carry, in float64: (a) each carry block folds its H group states with A^(LG),
//     (b) one fold per row over the blocks with A^(LGH) from zi gives each block's start state, (c) each block
//     expands its groups' start states s_g from it.  Anchored at sample 0 at every level.
//   sosfilt_chunk_kernel<S, true> (apply) the CTA expands its chunks' start states s_c from s_g and the b_c in the same order as
//     (c), rounds them to complex64, and each thread re-runs the cascade over its chunk from s_c and writes y;
//     the thread that owns the row's last sample writes zf.
//
// x is read twice and y written once (24 B/sample).  A thread's chunk is staged through shared memory in tiles
// of T samples per chunk, loaded with 8-byte cp.async so that a warp reads whole 128-byte lines.  The
// coefficients are kernel parameters (constant bank), so the 4S state floats are the only per-sample registers.
#include "iqw_common.cuh"

namespace iqw {

namespace {

constexpr int kMaxSections = 16;
constexpr int kG = 128;              // chunks per group = threads per CTA of the chunk kernels
constexpr int kT = 16;               // samples per chunk and tile
constexpr int kH = 64;               // groups per carry block
constexpr int kPitch = kT + 1;       // tile row pitch in float2: conflict-free per-thread reads
constexpr int kFoldThreads = 64;     // 4S workers of a fold: one per (state, re/im)

__host__ __device__ constexpr int chunk_len(int S) { return S <= 8 ? 512 : 1024; }

struct SosCoef {
    float c[kMaxSections][5];        // b0, b1, b2, -a1, -a2 of each section (a0 == 1)
};

// one sample through the cascade: y = b0 u + z1, z1 = b1 u - a1 y + z2, z2 = b2 u - a2 y
template <int S>
__device__ __forceinline__ float2 cascade(const SosCoef& k, float2 (&z)[2 * S], float2 u) {
#pragma unroll
    for (int s = 0; s < S; ++s) {
        const float b0 = k.c[s][0], b1 = k.c[s][1], b2 = k.c[s][2], na1 = k.c[s][3], na2 = k.c[s][4];
        float2 y, z1, z2;
        y.x = fmaf(b0, u.x, z[2 * s].x);
        y.y = fmaf(b0, u.y, z[2 * s].y);
        z1.x = fmaf(na1, y.x, fmaf(b1, u.x, z[2 * s + 1].x));
        z1.y = fmaf(na1, y.y, fmaf(b1, u.y, z[2 * s + 1].y));
        z2.x = fmaf(na2, y.x, b2 * u.x);
        z2.y = fmaf(na2, y.y, b2 * u.y);
        z[2 * s] = z1;
        z[2 * s + 1] = z2;
        u = y;
    }
    return u;
}

// t <- P t + b_k for k < count, in float64, by the first 4S threads of the block (one per state and re/im
// part); every thread of the block must call it.  Pt: P transposed in shared memory, Pt[j][i] = P[i][j].
// tb: 2 x (re, im) x 2S doubles; the caller puts the start state in tb[0] and synchronises.  load(k, i, part)
// returns component (i, part) of b_k; store(k, i, part, v) receives the state before item k.  Returns the
// final state's slot.  The sum of each component is b + P[i][even j] t + P[i][odd j] t, in ascending j.
template <int S, class Load, class Store>
__device__ const double* fold(const double* Pt, double* tb, long long count, Load load, Store store) {
    constexpr int N = 2 * S;
    const int w = threadIdx.x, i = w % N, part = w / N;
    const bool worker = w < 2 * N;
    for (long long k = 0; k < count; ++k) {
        const double* t = tb + (k & 1) * 2 * N + part * N;
        if (worker) {
            const double b = load(k, i, part);
            store(k, i, part, t[i]);
            double a0 = b, a1 = 0.0;
#pragma unroll
            for (int j = 0; j < N; j += 2) {
                a0 = fma(Pt[j * N + i], t[j], a0);
                a1 = fma(Pt[(j + 1) * N + i], t[j + 1], a1);
            }
            tb[((k + 1) & 1) * 2 * N + part * N + i] = a0 + a1;
        }
        __syncthreads();
    }
    return tb + (count & 1) * 2 * N;
}

template <int S>
__device__ void load_transposed(const double* P, double* Pt) {
    constexpr int N = 2 * S;
    for (int e = threadIdx.x; e < N * N; e += blockDim.x) Pt[(e % N) * N + e / N] = P[e];
}

__device__ __forceinline__ void cp_async8(void* smem, const void* gmem, bool valid) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(s), "l"(gmem), "r"(valid ? 8 : 0) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

struct ChunkArgs {
    const float2* x;
    long long n, x_stride;          // samples per row (of this call), row pitch
    const double* P;                // A^L, row-major 2S x 2S
    float2* chunk_states;           // [rows][groups * G][2S]: b_c (states pass), read by the apply pass
    double2* group_states;          // [rows][groups][2S]: b_g out (states), s_g in (apply)
    long long groups;               // groups per row
    float2* y;                      // apply: [rows][y_stride]
    long long y_stride;
    float2* zf;                     // apply: [rows][2S] or null
};

template <int S>
__host__ __device__ constexpr size_t chunk_smem() {
    constexpr size_t tiles = sizeof(float2) * 2 * kG * kPitch;
    constexpr size_t states = sizeof(float2) * kG * 2 * S;
    return (tiles > states ? tiles : states) + sizeof(double) * (4 * S * S + 8 * S);
}

// One CTA = one group of G chunks of L samples; thread c owns chunk c.  APPLY = false: the states pass;
// APPLY = true: the apply pass.  Both run the same per-chunk loop, so a chunk's recursion is the same code in
// both passes.
template <int S, bool APPLY>
__global__ void __launch_bounds__(kG, 4) sosfilt_chunk_kernel(const SosCoef k, const ChunkArgs a) {
    constexpr int N = 2 * S, L = chunk_len(S);
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* tile = reinterpret_cast<float2*>(smem_raw);                     // [2][G][kPitch], or
    float2* cs = tile;                                                      // [G][2S] chunk states
    double* Pt = reinterpret_cast<double*>(smem_raw + (chunk_smem<S>() - sizeof(double) * (4 * S * S + 8 * S)));
    double* tb = Pt + N * N;
    const int tid = threadIdx.x;
    const long long row = blockIdx.y, grp = blockIdx.x;
    const float2* x = a.x + row * a.x_stride;
    const long long g0 = grp * (long long)kG * L;          // first sample of the group
    const long long c0 = g0 + (long long)tid * L;          // first sample of this thread's chunk
    float2* cs_row = a.chunk_states + (row * a.groups + grp) * (long long)kG * N;
    double2* gs = a.group_states + (row * a.groups + grp) * N;

    float2 z[N];
    if constexpr (APPLY) {
        // expand the chunk start states from s_g: t <- P t + b_c in chunk order, state before chunk c to cs[c]
        load_transposed<S>(a.P, Pt);
        for (int e = tid; e < kG * N; e += kG) cs[e] = cs_row[e];
        if (tid < 2 * N) tb[tid] = tid < N ? gs[tid].x : gs[tid - N].y;
        __syncthreads();
        fold<S>(Pt, tb, kG,
                [&](long long c, int i, int part) { return (double)(part ? cs[c * N + i].y : cs[c * N + i].x); },
                [&](long long c, int i, int part, double v) {
                    float* p = reinterpret_cast<float*>(&cs[c * N + i]);
                    p[part] = __double2float_rn(v);
                });
#pragma unroll
        for (int j = 0; j < N; ++j) z[j] = cs[tid * N + j];
        __syncthreads();                                    // cs aliases the tiles
    } else {
#pragma unroll
        for (int j = 0; j < N; ++j) z[j] = make_float2(0.f, 0.f);
    }

    // tile j of every chunk: samples [c0 + j*T, c0 + (j+1)*T); element e of a tile is chunk e / T, sample e % T
    auto issue = [&](int j, int buf) {
#pragma unroll
        for (int r = 0; r < kT; ++r) {
            const int e = tid + r * kG, c = e / kT, o = e % kT;
            const long long i = g0 + (long long)c * L + (long long)j * kT + o;
            cp_async8(tile + (buf * kG + c) * kPitch + o, x + (i < a.n ? i : 0), i < a.n);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    issue(0, 0);
    for (int j = 0; j < L / kT; ++j) {
        const int buf = j & 1;
        cp_async_wait_all();
        __syncthreads();
        if (j + 1 < L / kT) issue(j + 1, buf ^ 1);
        float2* t = tile + (buf * kG + tid) * kPitch;
        const long long s0 = c0 + (long long)j * kT;
        if (s0 + kT <= a.n) {
#pragma unroll
            for (int o = 0; o < kT; ++o) {
                const float2 v = cascade<S>(k, z, t[o]);
                if constexpr (APPLY) t[o] = v;
            }
        } else {
            // the row ends inside this tile: the same recursion, stopped at the last sample
            for (int o = 0; o < kT && s0 + o < a.n; ++o) {
                const float2 v = cascade<S>(k, z, t[o]);
                if constexpr (APPLY) t[o] = v;
            }
        }
        if constexpr (APPLY) {
            __syncthreads();
            float2* y = a.y + row * a.y_stride;
#pragma unroll
            for (int r = 0; r < kT; ++r) {
                const int e = tid + r * kG, c = e / kT, o = e % kT;
                const long long i = g0 + (long long)c * L + (long long)j * kT + o;
                if (i < a.n) __stcs(y + i, tile[(buf * kG + c) * kPitch + o]);
            }
        }
    }

    if constexpr (APPLY) {
        if (a.zf && c0 <= a.n - 1 && a.n - 1 < c0 + L) {
#pragma unroll
            for (int j = 0; j < N; ++j) a.zf[row * N + j] = z[j];
        }
    } else {
        // b_c to shared memory (aliasing the tiles) and the workspace, then the group's fold from zero
        __syncthreads();
#pragma unroll
        for (int j = 0; j < N; ++j) cs[tid * N + j] = z[j];
        load_transposed<S>(a.P, Pt);
        if (tid < 2 * N) tb[tid] = 0.0;
        __syncthreads();
        for (int e = tid; e < kG * N; e += kG) cs_row[e] = cs[e];
        const double* t = fold<S>(Pt, tb, kG,
                                  [&](long long c, int i, int part) {
                                      return (double)(part ? cs[c * N + i].y : cs[c * N + i].x);
                                  },
                                  [](long long, int, int, double) {});
        if (tid < N) gs[tid] = make_double2(t[tid], t[N + tid]);
    }
}

struct FoldArgs {
    const double2* in;              // [rows][in_stride]: the items b_k of each row
    long long in_stride, count, seg;    // items per row, items per segment (one CTA each)
    const double* P;                // 2S x 2S, row-major
    const double2* init64;          // [rows][segments][2S] start states, or
    const float2* init32;           // [rows][2S] (one segment per row), or zero when both are null
    double2* out;                   // every: [rows][out_stride] state before each item; else [rows][segments]
    long long out_stride;
    int every;
};

// one fold per (segment of a.seg items, row): grid (segments, rows), kFoldThreads threads
template <int S>
__global__ void __launch_bounds__(kFoldThreads) sos_fold_kernel(const FoldArgs a) {
    constexpr int N = 2 * S;
    __shared__ double Pt[N * N];
    __shared__ double tb[4 * N];
    const long long row = blockIdx.y, seg = blockIdx.x, first = seg * a.seg;
    const long long count = (a.count - first < a.seg) ? a.count - first : a.seg;
    const long long segs = gridDim.x;
    load_transposed<S>(a.P, Pt);
    const int tid = threadIdx.x;
    if (tid < 2 * N) {
        const int i = tid % N, part = tid / N;
        double v = 0.0;
        if (a.init64) { const double2 s = a.init64[(row * segs + seg) * N + i]; v = part ? s.y : s.x; }
        else if (a.init32) { const float2 s = a.init32[row * N + i]; v = part ? s.y : s.x; }
        tb[tid] = v;
    }
    __syncthreads();
    const double2* in = a.in + row * a.in_stride + first * N;
    double* out = reinterpret_cast<double*>(a.out + row * a.out_stride + (a.every ? first * N : seg * N));
    const double* t = fold<S>(Pt, tb, count,
                              [&](long long k, int i, int part) {
                                  const double2 b = in[k * N + i];
                                  return part ? b.y : b.x;
                              },
                              [&](long long k, int i, int part, double v) {
                                  if (a.every) out[2 * (k * N + i) + part] = v;
                              });
    if (!a.every && tid < 2 * N) out[2 * (tid % N) + tid / N] = t[tid];
}

struct Geometry {
    int L, G, H;
    long long groups, blocks;       // per row
};
Geometry geometry(int S, long long n) {
    Geometry g{chunk_len(S), kG, kH, 0, 0};
    const long long span = (long long)g.L * g.G;
    g.groups = (n + span - 1) / span;
    g.blocks = (g.groups + kH - 1) / kH;
    return g;
}

size_t chunk_states_bytes(long long rows, long long groups, int S) { return sizeof(float2) * rows * groups * kG * 2 * S; }
size_t group_states_bytes(long long rows, long long groups, int S) { return sizeof(double2) * rows * groups * 2 * S; }
size_t carry_bytes(long long rows, long long groups, int S) {
    return sizeof(double2) * rows * ((groups + kH - 1) / kH) * 2 * S;
}

int check_sos(const float* h_sos, int S, SosCoef* k) {
    if (S < 1 || S > kMaxSections)
        return fail(IQW_ERR_UNSUPPORTED, "sosfilt: %d sections (1..%d are built)", S, kMaxSections);
    if (!h_sos) return fail(IQW_ERR_INVALID, "sosfilt: null sos");
    *k = SosCoef{};
    for (int s = 0; s < S; ++s) {
        const float* r = h_sos + 6 * s;
        if (r[3] != 1.0f) return fail(IQW_ERR_INVALID, "sosfilt: sos[%d, 3] is %g, should be 1", s, (double)r[3]);
        k->c[s][0] = r[0];
        k->c[s][1] = r[1];
        k->c[s][2] = r[2];
        k->c[s][3] = -r[4];
        k->c[s][4] = -r[5];
    }
    return IQW_OK;
}

int check_rows(const char* what, long long rows, long long n, long long stride, const void* p) {
    if (rows < 0 || n < 0) return fail(IQW_ERR_INVALID, "sosfilt: negative size");
    if (rows > 65535) return fail(IQW_ERR_UNSUPPORTED, "sosfilt: more than 65535 rows");
    if (rows > 0 && n > 0 && !p) return fail(IQW_ERR_INVALID, "sosfilt: null %s", what);
    if (rows > 1 && stride < n) return fail(IQW_ERR_INVALID, "sosfilt: %s row stride %lld shorter than a row of %lld",
                                            what, stride, n);
    return IQW_OK;
}

template <bool APPLY>
int launch_chunks(int S, const SosCoef& k, const ChunkArgs& a, long long rows, cudaStream_t stream) {
    return dispatch<1, kMaxSections>(S, [&](auto sc) -> int {
        constexpr int SC = decltype(sc)::value;
        auto kern = sosfilt_chunk_kernel<SC, APPLY>;
        constexpr size_t smem = chunk_smem<SC>();
        IQW_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        if (a.groups > 0x7FFFFFFFLL) return fail(IQW_ERR_UNSUPPORTED, "sosfilt: %lld groups per row", a.groups);
        {
            IQW_PROFILE(APPLY ? "sosfilt_apply_kernel" : "sosfilt_states_kernel", stream);
            kern<<<dim3((unsigned)a.groups, (unsigned)rows), kG, smem, stream>>>(k, a);
        }
        IQW_CUDA_OK(cudaGetLastError());
        return IQW_OK;
    }, [] { return IQW_ERR_UNSUPPORTED; });
}

int launch_carry(int S, double2* g, long long rows, long long groups, const float2* zi, const double* powers,
                 double2* blocks, cudaStream_t stream) {
    return dispatch<1, kMaxSections>(S, [&](auto sc) -> int {
        constexpr int SC = decltype(sc)::value, N = 2 * SC;
        const long long nb = (groups + kH - 1) / kH;
        if (nb > 0x7FFFFFFFLL) return fail(IQW_ERR_UNSUPPORTED, "sosfilt: %lld carry blocks per row", nb);
        IQW_PROFILE_TRAIN("sosfilt_carry", stream, 3);
        FoldArgs f{};
        // (a) each block of H groups folds its zero-state finals with A^(LG)
        f = FoldArgs{g, groups * N, groups, kH, powers + N * N, nullptr, nullptr, blocks, nb * N, 0};
        { IQW_PROFILE_FINE("sosfilt_carry_blocks", stream);
          sos_fold_kernel<SC><<<dim3((unsigned)nb, (unsigned)rows), kFoldThreads, 0, stream>>>(f); }
        // (b) per row over the blocks with A^(LGH) from zi: each block's start state, in place
        f = FoldArgs{blocks, nb * N, nb, nb, powers + 2 * N * N, nullptr, zi, blocks, nb * N, 1};
        { IQW_PROFILE_FINE("sosfilt_carry_rows", stream);
          sos_fold_kernel<SC><<<dim3(1, (unsigned)rows), kFoldThreads, 0, stream>>>(f); }
        // (c) each block expands its groups' start states with A^(LG), in place
        f = FoldArgs{g, groups * N, groups, kH, powers + N * N, blocks, nullptr, g, groups * N, 1};
        { IQW_PROFILE_FINE("sosfilt_carry_groups", stream);
          sos_fold_kernel<SC><<<dim3((unsigned)nb, (unsigned)rows), kFoldThreads, 0, stream>>>(f); }
        IQW_CUDA_OK(cudaGetLastError());
        return IQW_OK;
    }, [] { return IQW_ERR_UNSUPPORTED; });
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace

}  // namespace iqw

extern "C" int iqw_sosfilt_geometry(int32_t n_sections, int32_t* out3) {
    using namespace iqw;
    if (n_sections < 1 || n_sections > kMaxSections)
        return fail(IQW_ERR_UNSUPPORTED, "sosfilt: %d sections (1..%d are built)", n_sections, kMaxSections);
    if (!out3) return fail(IQW_ERR_INVALID, "sosfilt: null output");
    out3[0] = chunk_len(n_sections);
    out3[1] = kG;
    out3[2] = kH;
    return IQW_OK;
}

extern "C" size_t iqw_sosfilt_workspace_bytes(int64_t n_rows, int64_t n_samples, int32_t n_sections) {
    using namespace iqw;
    if (n_rows < 0 || n_samples < 0 || n_sections < 1 || n_sections > kMaxSections) return 0;
    const Geometry g = geometry(n_sections, n_samples);
    return chunk_states_bytes(n_rows, g.groups, n_sections) + group_states_bytes(n_rows, g.groups, n_sections) +
           carry_bytes(n_rows, g.groups, n_sections);
}

extern "C" size_t iqw_sosfilt_carry_workspace_bytes(int64_t n_rows, int64_t n_groups, int32_t n_sections) {
    using namespace iqw;
    if (n_rows < 0 || n_groups < 0 || n_sections < 1 || n_sections > kMaxSections) return 0;
    return carry_bytes(n_rows, n_groups, n_sections);
}

extern "C" int iqw_sosfilt_states_c64(const void* d_x, int64_t n_rows, int64_t n_samples, int64_t x_row_stride,
                                      const float* h_sos, int32_t n_sections, const void* d_powers,
                                      void* d_group_states, void* d_workspace, size_t workspace_bytes, void* stream) {
    using namespace iqw;
    SosCoef k;
    if (int rc = check_sos(h_sos, n_sections, &k)) return rc;
    if (int rc = check_rows("x", n_rows, n_samples, x_row_stride, d_x)) return rc;
    if (n_rows == 0 || n_samples == 0) return IQW_OK;
    const Geometry g = geometry(n_sections, n_samples);
    if (!d_powers || !d_group_states || !d_workspace) return fail(IQW_ERR_INVALID, "sosfilt: null pointer");
    if (!aligned16(d_group_states) || !aligned16(d_workspace) || (reinterpret_cast<uintptr_t>(d_powers) & 7))
        return fail(IQW_ERR_INVALID, "sosfilt: misaligned powers, group states or workspace");
    if (workspace_bytes < chunk_states_bytes(n_rows, g.groups, n_sections))
        return fail(IQW_ERR_WORKSPACE, "sosfilt: workspace of %zu bytes, need %zu", workspace_bytes,
                    chunk_states_bytes(n_rows, g.groups, n_sections));
    DeviceGuard guard(d_x);
    ChunkArgs a{};
    a.x = reinterpret_cast<const float2*>(d_x);
    a.n = n_samples;
    a.x_stride = n_rows > 1 ? x_row_stride : n_samples;
    a.P = reinterpret_cast<const double*>(d_powers);
    a.chunk_states = reinterpret_cast<float2*>(d_workspace);
    a.group_states = reinterpret_cast<double2*>(d_group_states);
    a.groups = g.groups;
    return launch_chunks<false>(n_sections, k, a, n_rows, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int iqw_sosfilt_carry_c64(void* d_group_states, int64_t n_rows, int64_t n_groups, const void* d_zi,
                                     int32_t n_sections, const void* d_powers, void* d_workspace,
                                     size_t workspace_bytes, void* stream) {
    using namespace iqw;
    if (n_sections < 1 || n_sections > kMaxSections)
        return fail(IQW_ERR_UNSUPPORTED, "sosfilt: %d sections (1..%d are built)", n_sections, kMaxSections);
    if (n_rows < 0 || n_groups < 0) return fail(IQW_ERR_INVALID, "sosfilt: negative size");
    if (n_rows > 65535) return fail(IQW_ERR_UNSUPPORTED, "sosfilt: more than 65535 rows");
    if (n_rows == 0 || n_groups == 0) return IQW_OK;
    if (!d_group_states || !d_powers || !d_workspace) return fail(IQW_ERR_INVALID, "sosfilt: null pointer");
    if (!aligned16(d_group_states) || !aligned16(d_workspace) || (reinterpret_cast<uintptr_t>(d_powers) & 7) ||
        (reinterpret_cast<uintptr_t>(d_zi) & 7))
        return fail(IQW_ERR_INVALID, "sosfilt: misaligned powers, zi, group states or workspace");
    if (workspace_bytes < carry_bytes(n_rows, n_groups, n_sections))
        return fail(IQW_ERR_WORKSPACE, "sosfilt: carry workspace of %zu bytes, need %zu", workspace_bytes,
                    carry_bytes(n_rows, n_groups, n_sections));
    DeviceGuard guard(d_group_states);
    return launch_carry(n_sections, reinterpret_cast<double2*>(d_group_states), n_rows, n_groups,
                        reinterpret_cast<const float2*>(d_zi), reinterpret_cast<const double*>(d_powers),
                        reinterpret_cast<double2*>(d_workspace), reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int iqw_sosfilt_apply_c64(const void* d_x, int64_t n_rows, int64_t n_samples, int64_t x_row_stride,
                                     const float* h_sos, int32_t n_sections, const void* d_powers,
                                     const void* d_group_states, const void* d_workspace, size_t workspace_bytes,
                                     void* d_y, int64_t y_row_stride, void* d_zf, void* stream) {
    using namespace iqw;
    SosCoef k;
    if (int rc = check_sos(h_sos, n_sections, &k)) return rc;
    if (int rc = check_rows("x", n_rows, n_samples, x_row_stride, d_x)) return rc;
    if (int rc = check_rows("y", n_rows, n_samples, y_row_stride, d_y)) return rc;
    if (n_rows == 0 || n_samples == 0) return IQW_OK;
    const Geometry g = geometry(n_sections, n_samples);
    if (!d_powers || !d_group_states || !d_workspace) return fail(IQW_ERR_INVALID, "sosfilt: null pointer");
    if (!aligned16(d_group_states) || !aligned16(d_workspace) || (reinterpret_cast<uintptr_t>(d_powers) & 7) ||
        (reinterpret_cast<uintptr_t>(d_zf) & 7))
        return fail(IQW_ERR_INVALID, "sosfilt: misaligned powers, zf, group states or workspace");
    if (workspace_bytes < chunk_states_bytes(n_rows, g.groups, n_sections))
        return fail(IQW_ERR_WORKSPACE, "sosfilt: workspace of %zu bytes, need %zu", workspace_bytes,
                    chunk_states_bytes(n_rows, g.groups, n_sections));
    DeviceGuard guard(d_y);
    ChunkArgs a{};
    a.x = reinterpret_cast<const float2*>(d_x);
    a.n = n_samples;
    a.x_stride = n_rows > 1 ? x_row_stride : n_samples;
    a.P = reinterpret_cast<const double*>(d_powers);
    a.chunk_states = reinterpret_cast<float2*>(const_cast<void*>(d_workspace));
    a.group_states = reinterpret_cast<double2*>(const_cast<void*>(d_group_states));
    a.groups = g.groups;
    a.y = reinterpret_cast<float2*>(d_y);
    a.y_stride = n_rows > 1 ? y_row_stride : n_samples;
    a.zf = reinterpret_cast<float2*>(d_zf);
    return launch_chunks<true>(n_sections, k, a, n_rows, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int iqw_sosfilt_c64(const void* d_x, int64_t n_rows, int64_t n_samples, int64_t x_row_stride,
                               const float* h_sos, int32_t n_sections, const void* d_powers, const void* d_zi,
                               void* d_y, int64_t y_row_stride, void* d_zf, void* d_workspace, size_t workspace_bytes,
                               void* stream) {
    using namespace iqw;
    SosCoef k;
    if (int rc = check_sos(h_sos, n_sections, &k)) return rc;
    if (int rc = check_rows("x", n_rows, n_samples, x_row_stride, d_x)) return rc;
    if (n_rows == 0 || n_samples == 0) return IQW_OK;
    if (workspace_bytes < iqw_sosfilt_workspace_bytes(n_rows, n_samples, n_sections))
        return fail(IQW_ERR_WORKSPACE, "sosfilt: workspace of %zu bytes, need %zu", workspace_bytes,
                    iqw_sosfilt_workspace_bytes(n_rows, n_samples, n_sections));
    if (!d_workspace || !aligned16(d_workspace)) return fail(IQW_ERR_INVALID, "sosfilt: null or misaligned workspace");
    // the three passes through the entry points the time shards use: [group states][carry blocks][chunk states]
    const Geometry g = geometry(n_sections, n_samples);
    unsigned char* ws = reinterpret_cast<unsigned char*>(d_workspace);
    void* gs = ws;
    void* blocks = ws + group_states_bytes(n_rows, g.groups, n_sections);
    void* chunks = ws + group_states_bytes(n_rows, g.groups, n_sections) + carry_bytes(n_rows, g.groups, n_sections);
    const size_t chunk_bytes = chunk_states_bytes(n_rows, g.groups, n_sections);
    if (int rc = iqw_sosfilt_states_c64(d_x, n_rows, n_samples, x_row_stride, h_sos, n_sections, d_powers, gs, chunks,
                                        chunk_bytes, stream))
        return rc;
    if (int rc = iqw_sosfilt_carry_c64(gs, n_rows, g.groups, d_zi, n_sections, d_powers, blocks,
                                       carry_bytes(n_rows, g.groups, n_sections), stream))
        return rc;
    return iqw_sosfilt_apply_c64(d_x, n_rows, n_samples, x_row_stride, h_sos, n_sections, d_powers, gs, chunks,
                                 chunk_bytes, d_y, y_row_stride, d_zf, stream);
}
