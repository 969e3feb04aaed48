// iqw_stats.cu -- kernel 2: statistics over the time axis of a (rows, cols) float32 matrix:
// exact order statistics (+ numpy 'linear' lerp), mean, max, min -- per column.
//
// Replaces /root/reference/src/iqwaveform/fourier.py:1311-1325 (np.quantile with float32 q and
// the named ufuncs over the time axis; 73 % of the reference's CPU time is ndarray.partition)
// and the in-place powtodB at fourier.py:1298-1299.
//
// Exact selection without sorting and without atomics in the hot loop.  The matrix is frame-major
// (a row = one frame, written coalesced by kernel 1), so a THREAD OWNS A COLUMN: lanes of a warp
// read 32 adjacent columns of one row (128 B, coalesced) and every thread streams down the time
// axis keeping PRIVATE counters in shared memory, laid out [bucket][thread] so that bank == lane
// (conflict free, no atomics).  The m <= 8 distinct target ranks of a call are located level by
// level; per column the state is a short ordered list of disjoint key INTERVALS, each known to
// contain a contiguous group of the target ranks, with the exact number of keys below it:
//
// EXACT PIPELINE (rows < 16384; every pass reads all rows):
//   range   : min/max key of ~2k rows per column  -> bucket map of that column
//   L0      : 256-bucket histogram of every element (bucket 0 / 255 catch keys outside the range
//             seen by `range`, so counts are exact whatever it missed)
//   scan0   : per column, group the target ranks by bucket -> intervals
//   R (x 7) : 32 sub-buckets per pending interval, all intervals in one pass; the scan that follows
//             splits each interval by sub-bucket.  Kernels exit at once when nothing is pending;
//             7 levels always suffice (32 key bits / 5 bits per level)
//   collect : keys inside the final intervals -> candidate lists (<= CAP each)
//   resolve : bitonic sort of the candidates in shared memory -> key of every target rank
//   finalize: dB, numpy lerp, mean/max/min, store
//
// LONG COLUMNS (rows >= 16384): ONE full read of the matrix instead of four.
//   A. sample_brackets : a stratified, jittered ROW SAMPLE (<= 8192 rows) of two columns per CTA is
//      staged in shared memory; a two-level histogram (2048 bins, then 256 sub-bins around each
//      wanted sample rank) gives, per group of target ranks, a key BRACKET [lo, hi] that holds the
//      group's ranks unless the sample was > 5 sigma off (a miss costs time, never exactness)
//   B. bracket_pass    : the single pass over ALL rows.  A thread owns a column and keeps the
//      brackets in registers; per bracket it counts the keys below it and appends the keys inside
//      it to a private candidate list (~15 % of the elements in total), + exact min / max / sum
//   C. scan_brackets   : per column, the exact counts say which bracket (or, after a miss or a list
//      overflow, which gap) holds each rank -> SELECT intervals (candidates are in the lists) or,
//      rarely, generic intervals that the exact pipeline above refines from the matrix
//   D. select          : one CTA per column histograms its candidate lists (2048 bins per bracket),
//      collects the few keys in the target bins and ranks them -> key of every target rank
//   E. refine / collect / resolve of the exact pipeline run only for what is still open (they exit
//      at once otherwise), then finalize.
// The result is exact for ANY sample: brackets only decide which keys are set aside.
//
// Keys are the order-preserving uint32 image of the float (iqw_common.cuh float_to_key), so the
// selection is exact for any input, ties and signed zeros included.  NaNs sort above +inf.
#include <cmath>
#include <atomic>
#include <cooperative_groups.h>
#include "iqw_common.cuh"

namespace iqw {

constexpr int kMaxRanks = 8;       // distinct target ranks (and therefore intervals) per call
constexpr int kMaxStats = 32;      // output rows per call
constexpr int kNB0 = 256;          // level-0 buckets
constexpr int kNSub = 32;          // sub-buckets per interval and refinement level
constexpr int kCap = 2048;         // candidates kept per (column, interval)
constexpr int kRefineLevels = 7;   // 32 key bits / 5 bits per level
constexpr int kBX = 128;           // columns (= threads) per CTA in the streaming passes
#ifndef IQW_UNROLL
#define IQW_UNROLL 8
#endif
constexpr int kUnroll = IQW_UNROLL;         // rows in flight per thread
constexpr long long kSampleMinRows = 16384;   // below this the exact pipeline reads all rows
constexpr int kSampleRows = 8192;  // rows of the sample staged in shared memory (per column)
#ifndef IQW_SAMPLE_COLS
#define IQW_SAMPLE_COLS 2
#endif
constexpr int kSampleCols = IQW_SAMPLE_COLS;     // columns per CTA of sample_brackets
constexpr int kMaxGroups = 8;      // rank groups (brackets) per call on the sampled path
constexpr int kSelBins = 2048;     // level-1 bins of sample_brackets and select
constexpr int kSubBins = 256;      // level-2 sub-bins of sample_brackets
#ifndef IQW_SEL_BUF
#define IQW_SEL_BUF 2048
#endif
#ifndef IQW_SEL_THREADS
#define IQW_SEL_THREADS 512
#endif
#ifndef IQW_SEL_MINBLOCKS
#define IQW_SEL_MINBLOCKS 3
#endif
constexpr int kSelBuf = IQW_SEL_BUF;      // keys ranked in shared memory at the end of select
constexpr int kSelThreads = IQW_SEL_THREADS;
constexpr int kMaxSplits = 512;    // row splits of the bracket pass (select stages their counts)
#ifndef IQW_BP_CTAS_PER_SM
#define IQW_BP_CTAS_PER_SM 64
#endif
constexpr long long kBracketCtas = 148 * IQW_BP_CTAS_PER_SM;   // CTAs the bracket pass aims at (a few waves)
#ifndef IQW_MIN_ROWS_PER_SPLIT
#define IQW_MIN_ROWS_PER_SPLIT 512
#endif
constexpr long long kMinRowsPerSplit = IQW_MIN_ROWS_PER_SPLIT;

enum IvStatus : uint32_t { IV_REFINE = 0, IV_COLLECT = 1, IV_RESOLVED = 2, IV_SELECT = 3 };

struct RankPlan {                  // same for every column: depends only on the row count
    int n_ranks;
    unsigned int rank[kMaxRanks];  // ascending, distinct
};

struct StatPlan {
    int n_stats;
    int kind[kMaxStats];
    int ia[kMaxStats], ib[kMaxStats];   // indices into RankPlan::rank
    float gamma[kMaxStats];
};

// which sample order statistics bracket which group of full-matrix ranks, and how many candidate
// keys each bracket may set aside per (row split, column)
struct BracketPlan {
    int n_groups;
    int n_sranks;
    unsigned int srank[2 * kMaxGroups];          // ascending, distinct sample ranks
    int s_lo[kMaxGroups], s_hi[kMaxGroups];      // indices into srank, -1 = open end of key space
    unsigned int cap_sum;                        // keys a (row split, column) candidate list holds
};

// the row sample of sample_brackets: one pseudo-random row out of every `step` consecutive rows
// (a stratified sample; the jitter defeats periodic captures)
struct RowMap {
    long long n;       // rows visited
    long long step;
    uint32_t seed;
};
__device__ __forceinline__ long long map_row(const RowMap& m, long long i) {
    uint32_t h = (uint32_t)i * 2654435761u + m.seed;
    h ^= h >> 15; h *= 2246822519u; h ^= h >> 13;
    // the jitter inside the stratum: high word of h * step (uniform in [0, step), one multiply instead of a division)
    return i * m.step + (long long)__umulhi(h, (uint32_t)m.step);
}

// per-pipeline state, carved from the caller's workspace
struct Work {
    uint32_t* range_lo;   // [cols]
    uint32_t* range_hi;   // [cols]
    uint32_t* kmin;       // [cols]
    uint32_t* kmax;       // [cols]
    double* dsum;         // [cols]
    uint32_t* hist0;      // [cols][256]
    uint32_t* n_iv;       // [cols]
    uint32_t* iv_klo;     // [cols][8]  first key of the interval
    uint32_t* iv_khi;     // [cols][8]  last key
    uint32_t* iv_shift;   // [cols][8]  sub-bucket shift (REFINE) / bracket slot (SELECT)
    uint32_t* iv_below;   // [cols][8]  number of keys < klo in the column
    uint32_t* iv_status;  // [cols][8]
    uint32_t* iv_first;   // [cols][8]  first target-rank index inside
    uint32_t* iv_nr;      // [cols][8]  number of target ranks inside
    uint32_t* iv_cnt;     // [cols][8]  number of keys inside (checked against what is collected)
    uint32_t* r_key;      // [cols][8]  key of each target rank once known (0xFFFFFFFF = NaN until then)
    uint32_t* hist1;      // [cols][8][32]
    uint32_t* cursor;     // [cols][8]
    uint32_t* cand;       // [cols][8][kCap]
    uint32_t* pending;    // [0] intervals in IV_REFINE, [1] intervals in IV_COLLECT; diagnostics:
                          // [2] ranks found in a gap (bracket missed), [3] brackets of overflowed
                          // columns, [4] SELECT intervals handed on as COLLECT, [5] as REFINE,
                          // [6] inconsistent candidate lists, [7] SELECT intervals
    // long-column path
    uint32_t* bk_lo;      // [cols][kMaxGroups] bracket bounds (empty slot: lo > hi)
    uint32_t* bk_hi;
    uint32_t* t_below;    // [cols][kMaxGroups] keys below each bracket, all rows
    uint32_t* t_cnt;      // [cols][kMaxGroups] keys in the bracket's region (bracket + the gap after it), from scan_brackets
    uint32_t* t_gap_hi;   // [cols][kMaxGroups] last key of that gap
    uint32_t* t_ovf;      // [cols] != 0: some candidate list of the column overflowed
    uint32_t* s_cnt;      // [splits][cols] keys in each candidate list
    uint32_t* lists;      // [splits][cols][cap_sum] candidate keys (of all brackets, unordered)
    size_t zero_bytes;    // leading bytes that must be zero before a pipeline starts
    size_t ff_bytes;      // bytes after them that must be 0xFF
};

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// long-column layout: splits == 0 carves the exact pipeline only
static size_t carve_work(void* base, int64_t cols, int64_t splits, int64_t cap_sum, Work* w) {
    size_t off = 0;
    auto take = [&](size_t bytes) {
        void* p = base ? static_cast<char*>(base) + off : nullptr;
        off = align_up(off + bytes, 256);
        return p;
    };
    const size_t c = (size_t)cols, m = kMaxRanks, g = kMaxGroups;
    Work t{};
    // --- zero-initialised region first ---
    t.range_hi = (uint32_t*)take(4 * c);
    t.kmax = (uint32_t*)take(4 * c);
    t.dsum = (double*)take(8 * c);
    t.hist0 = (uint32_t*)take(4 * c * kNB0);
    t.hist1 = (uint32_t*)take(4 * c * m * kNSub);
    t.cursor = (uint32_t*)take(4 * c * m);
    t.n_iv = (uint32_t*)take(4 * c);
    t.pending = (uint32_t*)take(256);
    if (splits > 0) {
        t.t_below = (uint32_t*)take(4 * c * g);
        t.t_cnt = (uint32_t*)take(4 * c * g);
        t.t_ovf = (uint32_t*)take(4 * c);
    }
    t.zero_bytes = off;
    // --- 0xFF-initialised ---
    t.range_lo = (uint32_t*)take(4 * c);
    t.kmin = (uint32_t*)take(4 * c);
    t.r_key = (uint32_t*)take(4 * c * m);
    t.ff_bytes = off - t.zero_bytes;
    // --- written before read ---
    t.iv_klo = (uint32_t*)take(4 * c * m);
    t.iv_khi = (uint32_t*)take(4 * c * m);
    t.iv_shift = (uint32_t*)take(4 * c * m);
    t.iv_below = (uint32_t*)take(4 * c * m);
    t.iv_status = (uint32_t*)take(4 * c * m);
    t.iv_first = (uint32_t*)take(4 * c * m);
    t.iv_nr = (uint32_t*)take(4 * c * m);
    t.iv_cnt = (uint32_t*)take(4 * c * m);
    t.cand = (uint32_t*)take(4 * c * m * kCap);
    if (splits > 0) {
        t.bk_lo = (uint32_t*)take(4 * c * g);
        t.bk_hi = (uint32_t*)take(4 * c * g);
        t.t_gap_hi = (uint32_t*)take(4 * c * g);
        t.s_cnt = (uint32_t*)take(4 * (size_t)splits * c);
        t.lists = (uint32_t*)take(4 * (size_t)splits * c * (size_t)cap_sum);
    }
    if (w) *w = t;
    return off;
}

// ---------------------------------------------------------------------------------------------
// streaming skeleton: thread `col` visits rows i0..i1, kUnroll loads in flight
// ---------------------------------------------------------------------------------------------
template <typename F>
__device__ __forceinline__ void stream_column(const float* __restrict__ p, long long cols,
                                              long long col, long long i0, long long i1, F&& visit) {
    long long i = i0;
    const float* src = p + i0 * cols + col;
    for (; i + kUnroll <= i1; i += kUnroll, src += (long long)kUnroll * cols) {
        float f[kUnroll];
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) f[u] = __ldcs(src + (long long)u * cols);
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) visit(f[u]);
    }
    for (; i < i1; ++i, src += cols) visit(__ldcs(src));
}

// ---------------------------------------------------------------------------------------------
// range: min / max key over ~2k of the rows
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBX)
range_kernel(const float* __restrict__ p, long long cols, long long rows, long long stride, Work w) {
    const long long col = (long long)blockIdx.x * kBX + threadIdx.x;
    if (col >= cols) return;
    uint32_t lo = 0xFFFFFFFFu, hi = 0u;
    for (long long i = (long long)blockIdx.y * stride; i < rows; i += stride * gridDim.y) {
        const uint32_t k = float_to_key(__ldg(p + i * cols + col));
        lo = min(lo, k);
        hi = max(hi, k);
    }
    atomicMin(w.range_lo + col, lo);
    atomicMax(w.range_hi + col, hi);
}

// bucket map of level 0: 0 = below the range, 255 = above, 1..254 inside
__device__ __forceinline__ uint32_t l0_shift(uint32_t lo, uint32_t hi) {
    const uint32_t span = hi - lo;
    uint32_t s = 0;
    while ((span >> s) >= (uint32_t)(kNB0 - 2)) ++s;
    return s;
}
__device__ __forceinline__ uint32_t l0_bucket(uint32_t k, uint32_t lo, uint32_t hi, uint32_t s) {
    if (k < lo) return 0;
    if (k > hi) return kNB0 - 1;
    return 1 + ((k - lo) >> s);
}

// exact min / max / sum of a column (named statistics), shared by L0 and the bracket pass
template <bool WANT_MINMAX, bool WANT_SUM, bool TO_DB>
struct Named {
    uint32_t kmin = 0xFFFFFFFFu, kmax = 0u;
    double dsum = 0.0;
    float part = 0.f;
    int n_part = 0;
    __device__ __forceinline__ void add(float f, uint32_t k, float eps) {
        if (WANT_MINMAX) {
            kmin = min(kmin, k);
            kmax = max(kmax, k);
        }
        if (WANT_SUM) {
            part += TO_DB ? power_to_dB(f, eps) : f;
            if (++n_part == 8) { dsum += (double)part; part = 0.f; n_part = 0; }
        }
    }
    __device__ __forceinline__ void flush(const Work& w, long long col) {
        if (WANT_MINMAX) {
            atomicMin(w.kmin + col, kmin);
            atomicMax(w.kmax + col, kmax);
        }
        if (WANT_SUM) atomicAdd(w.dsum + col, dsum + (double)part);
    }
};

// ---------------------------------------------------------------------------------------------
// L0: private 256-bucket histogram per column + named statistics
// ---------------------------------------------------------------------------------------------
template <bool WANT_SUM, bool TO_DB>
__global__ void __launch_bounds__(kBX)
l0_kernel(const float* __restrict__ p, long long cols, long long rows, long long rows_per_split,
          float eps, Work w) {
    extern __shared__ uint16_t hist[];   // [kNB0][kBX]
    for (int i = threadIdx.x; i < kNB0 * kBX; i += kBX) hist[i] = 0;
    __syncthreads();

    const long long col = (long long)blockIdx.x * kBX + threadIdx.x;
    if (col >= cols) return;
    const uint32_t lo = w.range_lo[col], hi = w.range_hi[col];
    const uint32_t s = l0_shift(lo, hi);
    uint16_t* h = hist + threadIdx.x;
    const long long i0 = (long long)blockIdx.y * rows_per_split;
    const long long i1 = min(rows, i0 + rows_per_split);
    Named<true, WANT_SUM, TO_DB> named;

    auto visit = [&](float f) {
        const uint32_t k = float_to_key(f);
        named.add(f, k, eps);
        h[l0_bucket(k, lo, hi, s) * kBX] += 1;
    };
    stream_column(p, cols, col, i0, i1, visit);

    uint32_t* g = w.hist0 + col * kNB0;
    for (int b = 0; b < kNB0; ++b) {
        const uint32_t c = h[b * kBX];
        if (c) atomicAdd(g + b, c);
    }
    named.flush(w, col);
}

// ---------------------------------------------------------------------------------------------
// interval bookkeeping (one thread per column, sequential)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t ceil_log2_u64(unsigned long long v) {
    uint32_t l = 0;
    while ((1ull << l) < v) ++l;
    return l;
}

struct IvList {
    uint32_t n;
    uint32_t klo[kMaxRanks], khi[kMaxRanks], shift[kMaxRanks], below[kMaxRanks],
        status[kMaxRanks], first[kMaxRanks], nr[kMaxRanks], cnt[kMaxRanks];
};

// append the interval [klo, klo + span) holding `cnt` keys, `below` keys under it, and target
// ranks [first, first + nr).  `single` = every key in it equals `key_exact`.
__device__ void iv_append(IvList& L, const Work& w, long long col, uint32_t klo,
                          unsigned long long span, uint32_t below, uint32_t cnt, uint32_t first,
                          uint32_t nr, bool single, uint32_t key_exact) {
    const uint32_t i = L.n++;
    const unsigned long long last = (unsigned long long)klo + span - 1ull;
    L.klo[i] = klo;
    L.khi[i] = last > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)last;
    L.below[i] = below;
    L.first[i] = first;
    L.nr[i] = nr;
    L.cnt[i] = cnt;
    L.shift[i] = 0;
    if (single || span == 1ull) {
        L.status[i] = IV_RESOLVED;
        for (uint32_t q = 0; q < nr; ++q) w.r_key[col * kMaxRanks + first + q] = single ? key_exact : klo;
    } else if (cnt <= (uint32_t)kCap) {
        L.status[i] = IV_COLLECT;
        atomicAdd(w.pending + 1, 1u);
    } else {
        L.status[i] = IV_REFINE;
        const uint32_t l = ceil_log2_u64(span);
        L.shift[i] = l > 5 ? l - 5 : 0;
        atomicAdd(w.pending, 1u);
    }
}

__device__ void iv_store(const IvList& L, const Work& w, long long col) {
    w.n_iv[col] = L.n;
    for (uint32_t i = 0; i < L.n; ++i) {
        const long long x = col * kMaxRanks + i;
        w.iv_klo[x] = L.klo[i];
        w.iv_khi[x] = L.khi[i];
        w.iv_shift[x] = L.shift[i];
        w.iv_below[x] = L.below[i];
        w.iv_status[x] = L.status[i];
        w.iv_first[x] = L.first[i];
        w.iv_nr[x] = L.nr[i];
        w.iv_cnt[x] = L.cnt[i];
    }
}

__device__ void iv_load(IvList& L, const Work& w, long long col) {
    L.n = w.n_iv[col];
    for (uint32_t i = 0; i < L.n; ++i) {
        const long long x = col * kMaxRanks + i;
        L.klo[i] = w.iv_klo[x]; L.khi[i] = w.iv_khi[x]; L.shift[i] = w.iv_shift[x];
        L.below[i] = w.iv_below[x]; L.status[i] = w.iv_status[x];
        L.first[i] = w.iv_first[x]; L.nr[i] = w.iv_nr[x]; L.cnt[i] = w.iv_cnt[x];
    }
}

// split the interval O[v] by its sub-bucket counts h[0..kNSub) (zeroed on the way), `cum` = number
// of keys below the first sub-bucket on entry, advanced past the interval on exit
__device__ void split_by_subbuckets(IvList& L, const IvList& O, uint32_t v, uint32_t* h,
                                    const RankPlan& rp, uint32_t& i, uint32_t& cum, const Work& w,
                                    long long col) {
    const uint32_t sh = O.shift[v];
    const uint32_t i_end = O.first[v] + O.nr[v];
    for (int b = 0; b < kNSub; ++b) {
        const uint32_t c = h[b];
        h[b] = 0;
        const uint32_t next = cum + c;
        if (i < i_end && rp.rank[i] < next) {
            const uint32_t first = i;
            while (i < i_end && rp.rank[i] < next) ++i;
            // the sub-bucket is clamped to its parent: keys above the parent's last key were NOT
            // counted in c (they belong to the gap / interval that follows)
            const uint32_t klo = O.klo[v] + ((uint32_t)b << sh);
            unsigned long long span = 1ull << sh;
            const unsigned long long room = (unsigned long long)O.khi[v] - klo + 1ull;
            if (span > room) span = room;
            iv_append(L, w, col, klo, span, cum, c, first, i - first, sh == 0, klo);
        }
        cum = next;
    }
}

__global__ void scan0_kernel(long long cols, RankPlan rp, Work w) {
    const long long col = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= cols) return;
    const uint32_t lo = w.range_lo[col], hi = w.range_hi[col];
    const uint32_t s0 = l0_shift(lo, hi);
    const uint32_t* h = w.hist0 + col * kNB0;

    IvList L;
    L.n = 0;
    uint32_t cum = 0;
    int i = 0;
    for (int b = 0; b < kNB0 && i < rp.n_ranks; ++b) {
        const uint32_t c = h[b];
        const uint32_t next = cum + c;
        if (rp.rank[i] < next) {
            const int first = i;
            while (i < rp.n_ranks && rp.rank[i] < next) ++i;
            const unsigned long long start =
                b == 0 ? 0ull
                       : b == kNB0 - 1 ? (unsigned long long)hi + 1ull
                                       : (unsigned long long)lo + ((unsigned long long)(b - 1) << s0);
            unsigned long long end =
                b == 0 ? (unsigned long long)lo
                       : b == kNB0 - 1 ? 0x100000000ull
                                       : (unsigned long long)lo + ((unsigned long long)b << s0);
            // keys above `hi` were counted in the last bucket, not in the interior bucket that
            // straddles hi
            if (b >= 1 && b <= kNB0 - 2 && end > (unsigned long long)hi + 1ull) end = (unsigned long long)hi + 1ull;
            const bool interior = b >= 1 && b <= kNB0 - 2;
            iv_append(L, w, col, (uint32_t)start, end - start, cum, c, (uint32_t)first,
                      (uint32_t)(i - first), interior && s0 == 0, lo + (uint32_t)(b - 1));
        }
        cum = next;
    }
    iv_store(L, w, col);
}

__device__ void scan_refine_body(long long col, long long cols, const RankPlan& rp, const Work& w) {
    if (col >= cols) return;
    IvList O, L;
    iv_load(O, w, col);
    bool any = false;
    for (uint32_t v = 0; v < O.n; ++v) any |= O.status[v] == IV_REFINE;
    if (!any) return;
    L.n = 0;
    for (uint32_t v = 0; v < O.n; ++v) {
        if (O.status[v] != IV_REFINE) {
            const uint32_t i = L.n++;
            L.klo[i] = O.klo[v]; L.khi[i] = O.khi[v]; L.shift[i] = O.shift[v]; L.below[i] = O.below[v];
            L.status[i] = O.status[v]; L.first[i] = O.first[v]; L.nr[i] = O.nr[v]; L.cnt[i] = O.cnt[v];
            continue;
        }
        atomicSub(w.pending, 1u);
        uint32_t cum = O.below[v], i = O.first[v];
        split_by_subbuckets(L, O, v, w.hist1 + (col * kMaxRanks + v) * kNSub, rp, i, cum, w, col);
    }
    iv_store(L, w, col);
}

__global__ void scan_refine_kernel(long long cols, RankPlan rp, Work w) {
    if (*w.pending == 0) return;
    scan_refine_body((long long)blockIdx.x * blockDim.x + threadIdx.x, cols, rp, w);
}

// after the bracket pass (long-column path): the number of keys below every bracket is known, the number
// INSIDE is not (select_kernel counts it from the lists).  Regions in key order: the gap below the first
// bracket, then per bracket the bracket TOGETHER WITH the gap that follows it.  Every target rank is located
// in its region.  A rank in the region of a bracket whose lists did not overflow becomes a SELECT interval
// (select_kernel moves it on to the gap if it lies beyond the bracket's keys); anything else becomes a
// generic interval that the exact pipeline refines.
__global__ void scan_brackets_kernel(long long cols, long long rows, RankPlan rp, int n_groups,
                                     Work w) {
    const long long col = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= cols) return;
    IvList L;
    L.n = 0;
    uint32_t i = 0;
    const uint32_t nrk = (uint32_t)rp.n_ranks;
    const uint32_t ovf = w.t_ovf[col];
    bool first_live = true;
    for (int g = 0; g < n_groups && i < nrk; ++g) {
        const uint32_t lo = w.bk_lo[col * kMaxGroups + g], hi = w.bk_hi[col * kMaxGroups + g];
        if (lo > hi) continue;                                     // slot merged into an earlier one
        const uint32_t below = w.t_below[col * kMaxGroups + g];
        // the region ends where the next live bracket starts
        unsigned long long next_lo = 0x100000000ull;
        uint32_t next_below = (uint32_t)rows;
        for (int h = g + 1; h < n_groups; ++h) {
            const uint32_t l2 = w.bk_lo[col * kMaxGroups + h];
            if (l2 <= w.bk_hi[col * kMaxGroups + h]) { next_lo = l2; next_below = w.t_below[col * kMaxGroups + h]; break; }
        }
        if (first_live && rp.rank[i] < below) {                    // ranks below the first bracket
            const uint32_t first = i;
            while (i < nrk && rp.rank[i] < below) ++i;
            atomicAdd(w.pending + 2, i - first);
            iv_append(L, w, col, 0u, (unsigned long long)lo, 0u, below, first, i - first, false, 0u);
        }
        first_live = false;
        if (i < nrk && rp.rank[i] < next_below) {
            const uint32_t first = i;
            while (i < nrk && rp.rank[i] < next_below) ++i;
            const uint32_t region = next_below - below;
            if (ovf) {
                atomicAdd(w.pending + 3, 1u);
                iv_append(L, w, col, lo, next_lo - lo, below, region, first, i - first, false, 0u);
            } else {
                const uint32_t v = L.n++;
                L.klo[v] = lo; L.khi[v] = hi; L.below[v] = below; L.cnt[v] = region;
                L.first[v] = first; L.nr[v] = i - first;
                L.shift[v] = (uint32_t)g; L.status[v] = IV_SELECT;
                w.t_cnt[col * kMaxGroups + g] = region;
                w.t_gap_hi[col * kMaxGroups + g] = (uint32_t)(next_lo - 1ull);
                atomicAdd(w.pending + 7, 1u);
            }
        }
    }
    if (i < nrk) {                                                 // no live bracket at all
        atomicAdd(w.pending + 2, nrk - i);
        iv_append(L, w, col, 0u, 0x100000000ull, 0u, (uint32_t)rows, i, nrk - i, false, 0u);
    }
    iv_store(L, w, col);
}

// ---------------------------------------------------------------------------------------------
// interval lookup shared by refine / bracket / collect: intervals are disjoint and ordered by key;
// the candidate of key k is the LAST interval with klo <= k.  Bounds live in registers.
// ---------------------------------------------------------------------------------------------
template <int M>
struct IvRegs {
    uint32_t klo[M], khi[M], shift[M];
    uint32_t n;
    __device__ __forceinline__ void load(const Work& w, long long col, bool live, uint32_t want_status,
                                         int& active) {
        n = live ? w.n_iv[col] : 0;
#pragma unroll
        for (int v = 0; v < M; ++v) {
            // unused / not-wanted entries keep their klo (the lookup needs the ordering) but carry
            // shift = 0x80000000, which every consumer treats as "reject"
            klo[v] = 0xFFFFFFFFu; khi[v] = 0u; shift[v] = 0x80000000u;
            if ((uint32_t)v < n) {
                const long long x = col * kMaxRanks + v;
                klo[v] = w.iv_klo[x];
                if (w.iv_status[x] == want_status) {
                    khi[v] = w.iv_khi[x];
                    shift[v] = w.iv_shift[x];
                    active = 1;
                }
            }
        }
    }
    // returns interval index or -1; sets (kl, kh, sh) of that interval
    __device__ __forceinline__ int find(uint32_t k, uint32_t& kl, uint32_t& kh, uint32_t& sh) const {
        int v = -1;
        kl = 0; kh = 0; sh = 0x80000000u;
#pragma unroll
        for (int q = 0; q < M; ++q) {
            const bool ge = k >= klo[q];
            v = ge ? q : v;
            kl = ge ? klo[q] : kl;
            kh = ge ? khi[q] : kh;
            sh = ge ? shift[q] : sh;
        }
        return v;
    }
};

// refine: 32 sub-buckets per pending interval, private counters [interval*32+sub][thread]
template <int M>
__device__ __forceinline__ void refine_body(unsigned bx, unsigned by, unsigned gdx, const float* __restrict__ p, long long cols,
                                            long long rows, long long rows_per_split, const Work& w, uint16_t* hist /* [M*32][kBX] */) {
    const int t = threadIdx.x;
    const long long col_tiles = (cols + kBX - 1) / kBX;
    const long long i0 = (long long)by * rows_per_split;
    const long long i1 = min(rows, i0 + rows_per_split);
    // a CTA owns the row range of `by` and walks column tiles bx, + gdx, ...;
    // tiles without a pending interval cost one look at their interval lists.  (After the long
    // path only a few tiles are ever pending, so its launch uses few tile slots and many row
    // splits: the whole GPU then works on the one tile that needs it.)
    for (long long tile = bx; tile < col_tiles; tile += gdx) {
        const long long col = tile * kBX + t;
        int active = 0;
        IvRegs<M> iv;
        iv.load(w, col, col < cols, IV_REFINE, active);
        if (!__syncthreads_or(active)) continue;
        for (int i = t; i < M * kNSub * kBX; i += kBX) hist[i] = 0;
        __syncthreads();
        if (active) {
            auto visit = [&](float f) {
                const uint32_t k = float_to_key(f);
                uint32_t kl, kh, sh;
                const int v = iv.find(k, kl, kh, sh);
                if (v >= 0 && k <= kh && sh < 32u) hist[(v * kNSub + ((k - kl) >> sh)) * kBX + t] += 1;
            };
            stream_column(p, cols, col, i0, i1, visit);

            uint32_t* g = w.hist1 + col * (kMaxRanks * kNSub);
#pragma unroll
            for (int v = 0; v < M; ++v) {
                if (iv.shift[v] >= 32u) continue;
                for (int b = 0; b < kNSub; ++b) {
                    const uint32_t c = hist[(v * kNSub + b) * kBX + t];
                    if (c) atomicAdd(g + v * kNSub + b, c);
                }
            }
        }
        __syncthreads();        // the private counters are zeroed again for the next tile
    }
}

// refine: 32 sub-buckets per pending interval, private counters [interval*32+sub][thread]
template <int M>
__global__ void __launch_bounds__(kBX)
refine_kernel(const float* __restrict__ p, long long cols, long long rows, long long rows_per_split,
              Work w) {
    if (*w.pending == 0) return;
    extern __shared__ uint16_t hist[];   // [M*32][kBX]
    refine_body<M>(blockIdx.x, blockIdx.y, gridDim.x, p, cols, rows, rows_per_split, w, hist);
}

// bracket pass (long-column path): the ONE read of all rows.  A thread owns a column; its M
// brackets and 2M counters live in registers.  Per bracket it counts the keys >= lo and the keys
// inside [lo, hi] (which give the keys below and inside the bracket), and every key inside ANY
// bracket is appended to the thread's private candidate list of this row split (brackets are
// disjoint, so the key itself says which bracket it belongs to): no atomics, no shared memory.
// A full list keeps counting; the overflow is flagged and the column is refined from the matrix.
//
// The per-element body is inline PTX (bracket_visit.inc, 4M + 7 instructions for M brackets).
// RAW mode compares the raw float bits as signed integers instead of order-preserving keys, which
// is exact when every bracket bound is a non-negative float or an open end (always the case for
// power spectra) and saves the key conversion; the lists then hold raw bits.  Flag pending[8],
// set by sample_brackets when it sees a negative bound, selects the mode for the whole call.
#include "bracket_visit.inc"

// generic (M = 8) body in C++
template <bool RAW, int M>
__device__ __forceinline__ void bracket_visit_generic(uint32_t v, float (&nge)[M], float (&nin)[M],
                                                      uint32_t& slot, const uint32_t (&lo)[M],
                                                      const uint32_t (&hi)[M], uint32_t base) {
    bool inside = false;
#pragma unroll
    for (int g = 0; g < M; ++g) {
        const bool ge = RAW ? (int32_t)v >= (int32_t)lo[g] : v >= lo[g];
        const bool in = ge && (RAW ? (int32_t)v <= (int32_t)hi[g] : v <= hi[g]);
        nge[g] += ge ? 1.f : 0.f;
        nin[g] += in ? 1.f : 0.f;
        inside |= in;
    }
    if (inside) {
        asm volatile("st.shared.u32 [%0], %1;" :: "r"(base + 4 * slot), "r"(v) : "memory");
        slot += 1;
    }
}

// Candidate appends go through a per-thread staging buffer of kStage keys in shared memory.  After
// every kUnroll rows, a buffer holding >= 32 keys is drained: the whole warp writes its first 32
// keys as ONE aligned 128-byte line of the owner's list, and the owner moves the (< kUnroll) keys
// that are left to the front.  (Appending with scattered 4-byte stores costs ~9 ps each chip-wide
// -- partial-sector writes -- which was 60 % of this kernel's time; tools/exp/exp_colstream.cu.)
constexpr int kLine = 32;                       // keys per 128-byte line
constexpr int kStage = kLine + kUnroll;         // most keys a buffer can hold between drains
constexpr int kStagePitch = kStage + 1;         // odd pitch: a warp reads one buffer conflict-free

template <int M, int NAMED /* bit 0: min/max, bit 1: sum, bit 2: sum of dB */, bool RAW>
__device__ __forceinline__ void bracket_pass_body(const float* __restrict__ p, long long cols, long long col,
                                                  bool live_col, long long i0, long long i1, float eps,
                                                  const BracketPlan& bp, const Work& w, uint32_t* stage) {
    uint32_t lo[M], hi[M];
    float n_ge[M], n_in[M];      // float counters: exact (rows per split < 2^24), FMA-pipe adds
#pragma unroll
    for (int g = 0; g < M; ++g) {
        // a thread past the last column streams the last column but owns empty brackets
        lo[g] = (live_col ? w.bk_lo[col * kMaxGroups + g] : 0xFFFFFFFFu) ^ (RAW ? 0x80000000u : 0u);
        hi[g] = (live_col ? w.bk_hi[col * kMaxGroups + g] : 0u) ^ (RAW ? 0x80000000u : 0u);
        n_ge[g] = 0.f; n_in[g] = 0.f;
    }
    const uint32_t cap = bp.cap_sum;                    // multiple of kLine
    const int lane = threadIdx.x & 31;
    uint32_t* my_stage = stage + threadIdx.x * kStagePitch;
    const uint32_t* warp_stage = stage + (threadIdx.x - lane) * kStagePitch;
    const uint32_t stage_addr = (uint32_t)__cvta_generic_to_shared(my_stage);
    uint32_t slot = 0;                                  // keys in the staging buffer
    uint32_t n_lines = 0;                               // lines this thread's list received so far
    // list of lane 0's column in this row split; lists of adjacent columns are `cap` keys apart.
    // (computed from the unclamped thread index: a thread past the last column never appends)
    uint32_t* warp_list = w.lists + ((long long)blockIdx.y * cols + (long long)blockIdx.x * kBX +
                                     (threadIdx.x - lane)) * (long long)cap;
    Named<(NAMED & 1) != 0, (NAMED & 2) != 0, (NAMED & 4) != 0> named;

    auto drain = [&](bool ready) {
        unsigned m = __ballot_sync(0xFFFFFFFFu, ready);
        __syncwarp();                       // the owners' appends are visible to the warp
        while (m) {
            const int src = __ffs(m) - 1;
            m &= m - 1;
            const uint32_t start = __shfl_sync(0xFFFFFFFFu, n_lines, src) * kLine;
            if (start + kLine <= cap)
                warp_list[(uint32_t)src * cap + start + lane] = warp_stage[src * kStagePitch + lane];
        }
        __syncwarp();                       // buffers are read before their owners touch them again
        if (ready) {
            // move the (< kUnroll) keys behind the line to the front: independent loads first
            const uint32_t left = slot - kLine;
            uint32_t t[kUnroll];
#pragma unroll
            for (int j = 0; j < kUnroll; ++j) t[j] = my_stage[kLine + j];
#pragma unroll
            for (int j = 0; j < kUnroll; ++j)
                if ((uint32_t)j < left) my_stage[j] = t[j];
            slot -= kLine;
            ++n_lines;
        }
    };
    auto visit = [&](float f) {
        const uint32_t bits = __float_as_uint(f);
        if (NAMED) named.add(f, float_to_key(f), eps);
        const uint32_t v = RAW ? bits : float_to_key(f);
        if constexpr (M <= 4) bracket_visit<RAW>(v, n_ge, n_in, slot, lo, hi, stage_addr);
        else bracket_visit_generic<RAW, M>(v, n_ge, n_in, slot, lo, hi, stage_addr);
    };
    // rows i0..i1 of this column; software-pipelined with two register buffers: the loads of the
    // next kUnroll rows are in flight while the current ones are classified
    const float* src = p + i0 * cols + col;
    long long i = i0;
    float fa[kUnroll], fb[kUnroll];
    auto load_block = [&](float (&f)[kUnroll]) {
#pragma unroll
        for (int u = 0; u < kUnroll; ++u, src += cols) f[u] = __ldcs(src);
    };
    auto visit_block = [&](float (&f)[kUnroll]) {
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) visit(f[u]);
        const bool ready = slot >= kLine;
        if (__any_sync(0xFFFFFFFFu, ready)) drain(ready);
    };
    if (i + kUnroll <= i1) load_block(fa);
#pragma unroll 1
    while (i + kUnroll <= i1) {
        if (i + 2 * kUnroll <= i1) load_block(fb);
        visit_block(fa);
        i += kUnroll;
        if (i + kUnroll > i1) break;
        if (i + 2 * kUnroll <= i1) load_block(fa);
        visit_block(fb);
        i += kUnroll;
    }
#pragma unroll 1
    for (; i < i1; ++i, src += cols) {      // < kUnroll rows: the buffer cannot overflow
        visit(__ldcs(src));
    }
    {
        const bool ready = slot >= kLine;
        if (__any_sync(0xFFFFFFFFu, ready)) drain(ready);
    }
    // what is left (< 32 keys per thread)
    const uint32_t rem_mine = slot;
    __syncwarp();
    for (int s = 0; s < 32; ++s) {
        const uint32_t rem = __shfl_sync(0xFFFFFFFFu, rem_mine, s);
        const uint32_t start = __shfl_sync(0xFFFFFFFFu, n_lines, s) * kLine;
        if ((uint32_t)lane < rem && start + kLine <= cap)
            warp_list[(uint32_t)s * cap + start + lane] = warp_stage[s * kStagePitch + lane];
    }
    if (!live_col) return;

    const uint32_t n = (uint32_t)(i1 > i0 ? i1 - i0 : 0);
#pragma unroll
    for (int g = 0; g < M; ++g) {
        const bool live = RAW ? (int32_t)lo[g] <= (int32_t)hi[g] : lo[g] <= hi[g];
        if (g < bp.n_groups && live) {
            const uint32_t ge = (uint32_t)n_ge[g];
            if (n - ge) atomicAdd(w.t_below + col * kMaxGroups + g, n - ge);
        }
    }
    const uint32_t n_list = n_lines * kLine + rem_mine;
    w.s_cnt[(long long)blockIdx.y * cols + col] = min(n_list, cap);
    if (n_list > cap) atomicOr(w.t_ovf + col, 1u);
    named.flush(w, col);
}

// RAW mode for M <= 4 brackets: difference form of the per-key body (bracket_visit_diff, 3M + 4 instructions)
// and a 32-key staging RING per thread which its OWNER drains, 16 keys (64 bytes, two full sectors) at a time
// with four 128-bit loads and stores: no warp-wide step, nothing is moved inside the buffer.  The keys
// INSIDE each bracket are not counted here: select_kernel counts them when it histograms the lists.
constexpr int kRing = 32;                       // keys per thread: one chunk being filled, one being drained
constexpr int kChunk = 16;                      // keys per drain
#ifndef IQW_BP_UNROLL
#define IQW_BP_UNROLL 12
#endif
constexpr int kBpUnroll = IQW_BP_UNROLL;        // rows per block of the difference-form body (two blocks in flight):
                                                // 8 / 12 / 16 rows measured 1.74 / 1.68 / 1.68 ms (61 / 72 / 87 registers)
static_assert(kChunk - 1 + kBpUnroll < kRing, "the ring holds what a block can append before it is drained");

template <int M, int NAMED>
__device__ __forceinline__ void bracket_pass_body_diff(const float* __restrict__ p, long long cols, long long col,
                                                       bool live_col, long long i0, long long i1, float eps,
                                                       const BracketPlan& bp, const Work& w, uint32_t* stage) {
    uint32_t lo[M], wd[M];       // raw-bit low bound (open low end: 0) and width hi - lo + 1 (empty slot: 0)
    uint32_t nlt[M];             // keys below lo[g]
#pragma unroll
    for (int g = 0; g < M; ++g) {
        const uint32_t klo = live_col ? w.bk_lo[col * kMaxGroups + g] : 0xFFFFFFFFu;
        const uint32_t khi = live_col ? w.bk_hi[col * kMaxGroups + g] : 0u;
        lo[g] = 0u; wd[g] = 0u; nlt[g] = 0u;
        if (klo <= khi) {
            // RAW mode: klo is 0 (open) or the key of a float > +0, khi the key of a float >= +0 or 0xFFFFFFFF
            lo[g] = klo < 0x80000000u ? 0u : klo ^ 0x80000000u;
            wd[g] = (khi ^ 0x80000000u) - lo[g] + 1u;
        }
    }
    const uint32_t cap = bp.cap_sum;                    // multiple of kLine, hence of kChunk
    uint32_t* my_stage = stage + threadIdx.x * kRing;
    const uint32_t stage_addr = (uint32_t)__cvta_generic_to_shared(my_stage);    // 128-byte aligned
    uint32_t p4 = 0;                                    // bytes appended so far (4 per key)
    uint32_t n_chunks = 0;                              // chunks taken out of the ring so far
    // this thread's list in this row split (a thread past the last column never appends: its brackets are empty)
    uint32_t* my_list = w.lists + ((long long)blockIdx.y * cols + col) * (long long)cap;
    Named<(NAMED & 1) != 0, (NAMED & 2) != 0, (NAMED & 4) != 0> named;

    auto drain = [&](uint32_t at_least) {
        if (p4 - n_chunks * (4u * kChunk) >= 4u * at_least) {
            const uint4* q = reinterpret_cast<const uint4*>(my_stage + ((n_chunks & 1u) << 4));
            const uint4 q0 = q[0], q1 = q[1], q2 = q[2], q3 = q[3];
            if ((n_chunks + 1u) * kChunk <= cap) {      // a full list keeps counting; the column is flagged below
                uint4* d = reinterpret_cast<uint4*>(my_list + n_chunks * kChunk);
                d[0] = q0; d[1] = q1; d[2] = q2; d[3] = q3;
            }
            ++n_chunks;
        }
    };
    auto visit = [&](float f) {
        if (NAMED) named.add(f, float_to_key(f), eps);
        bracket_visit_diff(__float_as_uint(f), nlt, p4, lo, wd, stage_addr);
    };
    const float* src = p + i0 * cols + col;
    long long i = i0;
    float fa[kBpUnroll], fb[kBpUnroll];
    auto load_block = [&](float (&f)[kBpUnroll]) {
#pragma unroll
        for (int u = 0; u < kBpUnroll; ++u, src += cols) f[u] = __ldcs(src);
    };
    auto visit_block = [&](float (&f)[kBpUnroll]) {
#pragma unroll
        for (int u = 0; u < kBpUnroll; ++u) visit(f[u]);
        drain(kChunk);          // at most kChunk - 1 + kBpUnroll < kRing keys are ever in the ring
    };
    if (i + kBpUnroll <= i1) load_block(fa);
#pragma unroll 1
    while (i + kBpUnroll <= i1) {
        if (i + 2 * kBpUnroll <= i1) load_block(fb);
        visit_block(fa);
        i += kBpUnroll;
        if (i + kBpUnroll > i1) break;
        if (i + 2 * kBpUnroll <= i1) load_block(fa);
        visit_block(fb);
        i += kBpUnroll;
    }
#pragma unroll 1
    for (; i < i1; ++i, src += cols) {      // < kBpUnroll rows: the ring cannot overflow
        visit(__ldcs(src));
    }
    drain(kChunk);
    const uint32_t n_list = p4 >> 2;
    drain(1u);                              // what is left (< kChunk keys) goes out as one more chunk
    if (!live_col) return;

#pragma unroll
    for (int g = 0; g < M; ++g)
        if (g < bp.n_groups && wd[g] != 0u && nlt[g]) atomicAdd(w.t_below + col * kMaxGroups + g, nlt[g]);
    w.s_cnt[(long long)blockIdx.y * cols + col] = min(n_list, cap);
    if (n_list > cap) atomicOr(w.t_ovf + col, 1u);
    named.flush(w, col);
}

// (no minimum-blocks bound: ptxas settles at 61 registers = 8 CTAs per SM by itself, and its schedule with an explicit
// bound of 8 measured 1.92 instead of 1.74 ms)
template <int M, int NAMED>
__global__ void __launch_bounds__(kBX)
bracket_pass_kernel(const float* __restrict__ p, long long cols, long long rows,
                    long long rows_per_split, float eps, BracketPlan bp, Work w) {
    static_assert(kRing <= kStagePitch, "the staging area serves both bodies");
    __shared__ __align__(128) uint32_t stage[kBX * kStagePitch];
    long long col = (long long)blockIdx.x * kBX + threadIdx.x;
    const bool live_col = col < cols;
    if (!live_col) col = cols - 1;          // keep the warp whole: it flushes rings cooperatively
    const long long i0 = (long long)blockIdx.y * rows_per_split;
    const long long i1 = min(rows, i0 + rows_per_split);
    if (w.pending[8] == 0) {
        if constexpr (M <= 4) bracket_pass_body_diff<M, NAMED>(p, cols, col, live_col, i0, i1, eps, bp, w, stage);
        else bracket_pass_body<M, NAMED, true>(p, cols, col, live_col, i0, i1, eps, bp, w, stage);
    } else {
        bracket_pass_body<M, NAMED, false>(p, cols, col, live_col, i0, i1, eps, bp, w, stage);
    }
}

template <int M>
__device__ __forceinline__ void collect_body(unsigned bx, unsigned by, unsigned gdx, const float* __restrict__ p,
                                             long long cols, long long rows, long long rows_per_split, const Work& w) {
    const long long col_tiles = (cols + kBX - 1) / kBX;
    const long long i0 = (long long)by * rows_per_split;
    const long long i1 = min(rows, i0 + rows_per_split);
    for (long long tile = bx; tile < col_tiles; tile += gdx) {     // see refine_body
        const long long col = tile * kBX + threadIdx.x;
        int active = 0;
        IvRegs<M> iv;
        iv.load(w, col, col < cols, IV_COLLECT, active);
        if (!__syncthreads_or(active)) continue;
        if (!active) continue;
        auto visit = [&](float f) {
            const uint32_t k = float_to_key(f);
            uint32_t kl, kh, sh;
            const int v = iv.find(k, kl, kh, sh);
            if (v >= 0 && k <= kh && sh < 32u) {
                const long long x = col * kMaxRanks + v;
                const uint32_t pos = atomicAdd(w.cursor + x, 1u);
                if (pos < (uint32_t)kCap) w.cand[x * kCap + pos] = k;
            }
        };
        stream_column(p, cols, col, i0, i1, visit);
    }
}

template <int M>
__global__ void __launch_bounds__(kBX)
collect_kernel(const float* __restrict__ p, long long cols, long long rows, long long rows_per_split,
               Work w) {
    if (w.pending[1] == 0) return;
    collect_body<M>(blockIdx.x, blockIdx.y, gridDim.x, p, cols, rows, rows_per_split, w);
}

// ---------------------------------------------------------------------------------------------
// resolve: one CTA per column; sort each COLLECT interval's candidates -> key of every rank
// ---------------------------------------------------------------------------------------------
constexpr int kResolveThreads = 256;

// (any block size: the tail kernel calls it with kBX threads)
__device__ void resolve_body(long long col, const RankPlan& rp, const Work& w, uint32_t* keys /* [kCap] shared */) {
    const int t = threadIdx.x, nt = blockDim.x;
    const uint32_t n_iv = w.n_iv[col];
    for (uint32_t v = 0; v < n_iv; ++v) {
        const long long x = col * kMaxRanks + v;
        if (w.iv_status[x] != IV_COLLECT) continue;     // RESOLVED ranks are already in r_key
        // invariant: the collect pass found exactly the keys the histograms counted; if not, the
        // ranks of this interval are poisoned (NaN) instead of silently wrong
        const bool sane = w.cursor[x] == w.iv_cnt[x] && w.cursor[x] <= (uint32_t)kCap;
        const uint32_t n = min(w.cursor[x], (uint32_t)kCap);
        int m = 1;
        while (m < (int)n) m <<= 1;
        __syncthreads();
        for (int i = t; i < m; i += nt)
            keys[i] = i < (int)n ? w.cand[x * kCap + i] : 0xFFFFFFFFu;
        __syncthreads();
        for (int k = 2; k <= m; k <<= 1)
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int i = t; i < m; i += nt) {
                    const int ixj = i ^ j;
                    if (ixj > i) {
                        const uint32_t a = keys[i], b = keys[ixj];
                        const bool up = (i & k) == 0;
                        if ((a > b) == up) { keys[i] = b; keys[ixj] = a; }
                    }
                }
                __syncthreads();
            }
        const uint32_t first = w.iv_first[x], nr = w.iv_nr[x], below = w.iv_below[x];
        if ((uint32_t)t < nr) {
            const uint32_t pos = rp.rank[first + t] - below;
            w.r_key[col * kMaxRanks + first + t] = (sane && pos < n) ? keys[pos] : 0xFFFFFFFFu;
        }
    }
}

__global__ void __launch_bounds__(kResolveThreads)
resolve_kernel(long long cols, RankPlan rp, Work w) {
    __shared__ uint32_t keys[kCap];
    if (w.pending[1] == 0) return;
    resolve_body(blockIdx.x, rp, w, keys);
}

// ---------------------------------------------------------------------------------------------
// long-column path, step A: row sample -> brackets.  One CTA stages the sampled keys of
// kSampleCols adjacent columns in shared memory and locates the wanted SAMPLE ranks with a
// two-level histogram; the bracket bounds are bin edges (a little wider than the sample order
// statistics, never narrower), which is all the bracket pass needs.
// ---------------------------------------------------------------------------------------------
#ifndef IQW_SAMPLE_THREADS
#define IQW_SAMPLE_THREADS 512
#endif
constexpr int kSampleThreads = IQW_SAMPLE_THREADS;
constexpr int kSR = 2 * kMaxGroups;   // sample ranks per column
constexpr size_t kSampleSmem =
    sizeof(uint32_t) * ((size_t)kSampleCols * kSampleRows + (size_t)kSampleCols * kSR * kSubBins) +
    (size_t)kSampleCols * kSelBins;            // + one byte per level-1 bin: which level-2 histogram it feeds
static_assert(kSampleCols * kSR * kSubBins >= kSampleCols * kSelBins, "level-1 bins reuse the level-2 area");

__device__ __forceinline__ uint32_t sel_shift(uint32_t span, uint32_t bins) {
    uint32_t s = 0;
    while ((span >> s) >= bins) ++s;
    return s;
}

__global__ void __launch_bounds__(kSampleThreads)
sample_brackets_kernel(const float* __restrict__ p, long long cols, RowMap rm, BracketPlan bp, Work w) {
    extern __shared__ uint32_t smem_u32[];
    uint32_t* keys = smem_u32;                                   // [kSampleCols][kSampleRows]
    uint32_t* hist = keys + kSampleCols * kSampleRows;           // level 1: [kSampleCols][kSelBins]
                                                                 // level 2: [kSampleCols][kSR][kSubBins]
    unsigned char* slot_of_bin = reinterpret_cast<unsigned char*>(hist + kSampleCols * kSR * kSubBins);
    __shared__ uint32_t s_min[kSampleCols], s_max[kSampleCols];
    __shared__ uint32_t s_bin[kSampleCols][kSR], s_below[kSampleCols][kSR], s_slot[kSampleCols][kSR];
    __shared__ uint32_t s_elo[kSampleCols][kSR], s_ehi[kSampleCols][kSR];

    const int t = threadIdx.x;
    const long long c0 = (long long)blockIdx.x * kSampleCols;
    const int S = (int)rm.n;
    const int nsr = bp.n_sranks;
    if (t < kSampleCols) { s_min[t] = 0xFFFFFFFFu; s_max[t] = 0u; }
    for (int i = t; i < kSampleCols * kSelBins; i += kSampleThreads) hist[i] = 0;
    __syncthreads();

    // ---- stage the sample, min / max per column ----
    uint32_t mn[kSampleCols], mx[kSampleCols];
#pragma unroll
    for (int c = 0; c < kSampleCols; ++c) { mn[c] = 0xFFFFFFFFu; mx[c] = 0u; }
#ifndef IQW_SAMPLE_U
#define IQW_SAMPLE_U 4
#endif
    constexpr int U = IQW_SAMPLE_U;            // rows in flight per thread
    for (int i0 = 0; i0 < S; i0 += kSampleThreads * U) {
        float v[U][kSampleCols];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = i0 + u * kSampleThreads + t;
            if (i < S) {
                const float* src = p + map_row(rm, i) * cols + c0;
#pragma unroll
                for (int c = 0; c < kSampleCols; ++c) v[u][c] = (c0 + c < cols) ? __ldg(src + c) : 0.f;
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = i0 + u * kSampleThreads + t;
            if (i < S) {
#pragma unroll
                for (int c = 0; c < kSampleCols; ++c) {
                    const uint32_t k = float_to_key(v[u][c]);
                    keys[c * kSampleRows + i] = k;
                    mn[c] = min(mn[c], k);
                    mx[c] = max(mx[c], k);
                }
            }
        }
    }
#pragma unroll
    for (int c = 0; c < kSampleCols; ++c) {
        mn[c] = __reduce_min_sync(0xFFFFFFFFu, mn[c]);
        mx[c] = __reduce_max_sync(0xFFFFFFFFu, mx[c]);
        if ((t & 31) == 0) { atomicMin(&s_min[c], mn[c]); atomicMax(&s_max[c], mx[c]); }
    }
    __syncthreads();

    // ---- level 1: kSelBins bins over [min, max] ----
    uint32_t kmin[kSampleCols], sh1[kSampleCols];
#pragma unroll
    for (int c = 0; c < kSampleCols; ++c) {
        kmin[c] = s_min[c];
        sh1[c] = sel_shift(s_max[c] - s_min[c], kSelBins);
    }
    for (int i = t; i < S; i += kSampleThreads) {
#pragma unroll
        for (int c = 0; c < kSampleCols; ++c)
            if (c0 + c < cols) atomicAdd(&hist[c * kSelBins + ((keys[c * kSampleRows + i] - kmin[c]) >> sh1[c])], 1u);
    }
    __syncthreads();
    {   // WPC warps scan a column (all sixteen warps work: two warps walking 64 bins per lane kept the other
        // fourteen at the barrier for a fifth of the kernel's time); a lane owns PER consecutive bins
        constexpr int WPC = kSampleThreads / 32 / kSampleCols;     // warps per column
        constexpr int PER = kSelBins / (32 * WPC);
        static_assert(kSelBins % (32 * WPC) == 0, "bins divide among the lanes of a column's warps");
        __shared__ uint32_t s_wtot[kSampleCols][WPC];
        const int c = (t >> 5) / WPC, wi = (t >> 5) % WPC, lane = t & 31;
        const bool live = c0 + c < cols;
        const uint32_t* h = hist + c * kSelBins + (wi * 32 + lane) * PER;
        uint32_t sum = 0;
        if (live)
            for (int b = 0; b < PER; ++b) sum += h[b];
        uint32_t inc = sum;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t o = __shfl_up_sync(0xFFFFFFFFu, inc, d);
            if (lane >= d) inc += o;
        }
        if (lane == 31) s_wtot[c][wi] = inc;
        __syncthreads();
        if (live) {
            uint32_t cum = inc - sum;
            for (int q = 0; q < wi; ++q) cum += s_wtot[c][q];
            int j = 0;
            while (j < nsr && bp.srank[j] < cum) ++j;
            for (int b = 0; b < PER && j < nsr; ++b) {
                const uint32_t hb = h[b];
                while (j < nsr && bp.srank[j] < cum + hb) {
                    s_bin[c][j] = (uint32_t)((wi * 32 + lane) * PER + b);
                    s_below[c][j] = cum;
                    ++j;
                }
                cum += hb;
            }
        }
    }
    __syncthreads();
    if (t < kSampleCols) {      // sample ranks that share a level-1 bin share a level-2 histogram
        for (int j = 0; j < nsr; ++j)
            s_slot[t][j] = (j > 0 && s_bin[t][j] == s_bin[t][j - 1]) ? s_slot[t][j - 1] : (uint32_t)j;
    }
    for (int i = t; i < kSampleCols * kSR * kSubBins; i += kSampleThreads) hist[i] = 0;
    for (int i = t; i < kSampleCols * kSelBins / 4; i += kSampleThreads)
        reinterpret_cast<uint32_t*>(slot_of_bin)[i] = 0xFFFFFFFFu;
    __syncthreads();
    // level-1 bin -> the level-2 histogram it feeds (0xFF: none), so that the level-2 sweep is one
    // byte lookup per key instead of a walk over the sample ranks
    if (t < kSampleCols && c0 + t < cols) {
        for (int j = nsr - 1; j >= 0; --j)              // descending: the first rank of a bin wins
            if (s_bin[t][j] < (uint32_t)kSelBins) slot_of_bin[t * kSelBins + s_bin[t][j]] = (unsigned char)s_slot[t][j];
    }
    __syncthreads();

    // ---- level 2: kSubBins sub-bins inside each wanted bin ----
    for (int i = t; i < S; i += kSampleThreads) {
#pragma unroll
        for (int c = 0; c < kSampleCols; ++c) {
            if (c0 + c >= cols) continue;
            const uint32_t d = keys[c * kSampleRows + i] - kmin[c];
            const uint32_t b = d >> sh1[c];
            const uint32_t sh2 = sh1[c] > 8 ? sh1[c] - 8 : 0;
            const uint32_t j = slot_of_bin[c * kSelBins + b];
            if (j != 0xFFu) atomicAdd(&hist[(c * kSR + j) * kSubBins + ((d - (b << sh1[c])) >> sh2)], 1u);
        }
    }
    __syncthreads();
    // one warp per (column, sample rank): sub-bin holding the rank -> key edges
    for (int task = t >> 5; task < kSampleCols * nsr; task += kSampleThreads / 32) {
        const int c = task / nsr, j = task % nsr, lane = t & 31;
        if (c0 + c >= cols) continue;
        constexpr int PER = kSubBins / 32;
        const uint32_t* h = hist + (c * kSR + (int)s_slot[c][j]) * kSubBins + lane * PER;
        uint32_t sum = 0;
        for (int b = 0; b < PER; ++b) sum += h[b];
        uint32_t inc = sum;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t o = __shfl_up_sync(0xFFFFFFFFu, inc, d);
            if (lane >= d) inc += o;
        }
        uint32_t cum = inc - sum;
        const uint32_t pos = bp.srank[j] - s_below[c][j];
        if (pos >= cum && pos < cum + sum) {
            int b = 0;
            while (pos >= cum + h[b]) { cum += h[b]; ++b; }
            const uint32_t sh2 = sh1[c] > 8 ? sh1[c] - 8 : 0;
            const unsigned long long e0 = (unsigned long long)kmin[c] +
                                          ((unsigned long long)s_bin[c][j] << sh1[c]) +
                                          ((unsigned long long)(lane * PER + b) << sh2);
            const unsigned long long e1 = e0 + (1ull << sh2) - 1ull;
            s_elo[c][j] = (uint32_t)e0;
            s_ehi[c][j] = e1 > (unsigned long long)s_max[c] ? s_max[c] : (uint32_t)e1;
        }
    }
    __syncthreads();

    // ---- brackets: a group that reaches into its predecessor is merged into it ----
    if (t < kSampleCols && c0 + t < cols) {
        const long long col = c0 + t;
        int last = -1;
        uint32_t last_hi = 0u;                                     // upper bound of slot `last` (kept in a register)
        bool not_raw = false;
        for (int g = 0; g < kMaxGroups; ++g) {
            uint32_t lo = 0xFFFFFFFFu, hi = 0u;                    // empty slot
            if (g < bp.n_groups) {
                lo = bp.s_lo[g] < 0 ? 0u : s_elo[t][bp.s_lo[g]];
                hi = bp.s_hi[g] < 0 ? 0xFFFFFFFFu : s_ehi[t][bp.s_hi[g]];
                if (hi < lo) hi = lo;
                if (last >= 0 && lo <= last_hi) {
                    if (hi > last_hi) { last_hi = hi; w.bk_hi[col * kMaxGroups + last] = hi; }
                    lo = 0xFFFFFFFFu; hi = 0u;
                } else {
                    last = g; last_hi = hi;
                }
            }
            w.bk_lo[col * kMaxGroups + g] = lo;
            w.bk_hi[col * kMaxGroups + g] = hi;
            // a bound that is a negative float (other than the open low end) rules out RAW mode, and so does a low
            // bound of exactly +0 (key 0x80000000): RAW mode clamps negative values to +0, which must stay below
            // every closed low bound
            not_raw |= lo <= hi && ((lo != 0u && lo <= 0x80000000u) || hi < 0x80000000u);
        }
        if (not_raw) atomicOr(w.pending + 8, 1u);
    }
}

// ---------------------------------------------------------------------------------------------
// long-column path, step D: one CTA per column ranks the candidate lists of its SELECT intervals.
// Each sweep reads every list of the column once (a warp per row split, 8 loads in flight per
// lane).  Sweep 1 histograms the keys (kSelBins bins per bracket); a warp per bracket then finds
// the bins holding its first and last rank and either
//   * collects the keys of those bins in a second sweep (a few dozen) and ranks them by counting,
//   * reads the answer off the histogram when bins are single keys,
//   * descends into the one bin holding all its ranks (heavy ties) and histograms again, or
//   * (ranks in different, crowded bins) hands a much narrower generic interval to the exact
//     pipeline.
// ---------------------------------------------------------------------------------------------
enum SelMode : uint32_t { SEL_IDLE = 0, SEL_HIST = 1, SEL_COLLECT = 2 };

template <int M>
__global__ void __launch_bounds__(kSelThreads, IQW_SEL_MINBLOCKS)
select_kernel(long long cols, int splits, RankPlan rp, BracketPlan bp, Work w) {
    extern __shared__ uint32_t smem_u32[];
    uint32_t* hist = smem_u32;                         // [M][kSelBins]
    uint32_t* buf = hist + M * kSelBins;               // [M][kSelBuf]
    uint32_t* cnts = buf + M * kSelBuf;                // [splits]
    __shared__ uint32_t s_a[M], s_b[M], s_sh[M], s_below[M], s_first[M], s_nr[M], s_iv[M];
    __shared__ uint32_t s_bf[M], s_bl[M], s_cb[M], s_n[M], s_mode[M];
    // ranks of a bracket's region that lie beyond the bracket's keys move on to the gap after it
    __shared__ uint32_t s_region[M], s_gap_hi[M], s_out_first[M], s_out_nr[M], s_out_below[M], s_out_cnt[M], s_keep[M];
    __shared__ int s_any, s_rebuild;
    // lookup of the sweeps: the live brackets in key order.  A key k can only belong to entry
    // #{i >= 1 : k > s_thr[i]}, s_thr[i] = first key of entry i, minus one; unused thresholds are 0xFFFFFFFF
    // (never exceeded), so that unused entries are never looked at.
    __shared__ uint4 s_tbl[M + 1];          // x: first key, y: last key - first key, z: shift (sweep 1), w: offset / tag
    __shared__ uint32_t s_thr[M + 1];

    const long long col = blockIdx.x;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    constexpr int NW = kSelThreads / 32;
    if (t < M) { s_mode[t] = SEL_IDLE; s_iv[t] = 0xFFFFFFFFu; s_n[t] = 0; s_a[t] = 0xFFFFFFFFu; s_b[t] = 0; s_sh[t] = 0;
                 s_out_nr[t] = 0; s_keep[t] = 1; }
    if (t == 0) { s_any = 0; s_rebuild = 0; }
    __syncthreads();
    // one thread per interval of the column (their loads overlap; thread 0 alone walked several dependent load
    // rounds per interval), the list lengths of the sweeps in the same round
    if (t < kMaxRanks && (uint32_t)t < w.n_iv[col]) {
        const long long x = col * kMaxRanks + t;
        const uint32_t status = w.iv_status[x], g = w.iv_shift[x];
        const uint32_t klo = w.iv_klo[x], khi = w.iv_khi[x], below = w.iv_below[x], first = w.iv_first[x], nr = w.iv_nr[x];
        if (status == IV_SELECT && g < (uint32_t)M) {
            s_iv[g] = (uint32_t)t;
            s_a[g] = klo; s_b[g] = khi;
            s_sh[g] = sel_shift(khi - klo, kSelBins);
            s_below[g] = below; s_first[g] = first; s_nr[g] = nr;
            s_region[g] = w.t_cnt[col * kMaxGroups + g]; s_gap_hi[g] = w.t_gap_hi[col * kMaxGroups + g];
            s_mode[g] = SEL_HIST;
            s_any = 1;
        }
    }
    for (int i = t; i < splits; i += kSelThreads) cnts[i] = w.s_cnt[(long long)i * cols + col];
    __syncthreads();
    if (!s_any) return;

    const uint32_t cap_sum = bp.cap_sum;
    const bool raw = w.pending[8] == 0;     // lists hold raw float bits (bracket pass RAW mode)
    // One warp per row split.  A lane reads FOUR consecutive keys with one 128-bit load (the lists are 128-byte
    // aligned and a whole number of 16-key chunks long, so the load stays inside the list); two loads per lane
    // are in flight, which covers the ~200 keys of a config-3 list in one round.  visit(key, live): keys past the
    // end of the list are visited with live = false instead of branching around them.  `keep` = true leaves the
    // lists in L2 for the second sweep (the lists of the CTAs in flight, ~110 MB, fit the 126 MB L2).
    const uint32_t key_or = raw ? 0x80000000u : 0u, key_and = raw ? 0x7FFFFFFFu : 0u;
    auto key_of = [&](uint32_t v) {        // raw float bits -> order-preserving key (identity in key mode)
        return v ^ ((((uint32_t)((int32_t)v >> 31)) & key_and) | key_or);
    };
    auto sweep = [&](bool keep, auto&& visit) {
        const size_t stride = (size_t)cols * cap_sum;                       // keys between row splits
        const uint32_t* src = w.lists + (size_t)col * cap_sum + (size_t)warp * stride + 4 * lane;
        auto load = [&](const uint32_t* q) {
            return keep ? __ldcg(reinterpret_cast<const uint4*>(q)) : __ldcs(reinterpret_cast<const uint4*>(q));
        };
        auto visit4 = [&](const uint4& q, uint32_t i, uint32_t n) {
            visit(key_of(q.x), i < n);
            visit(key_of(q.y), i + 1 < n);
            visit(key_of(q.z), i + 2 < n);
            visit(key_of(q.w), i + 3 < n);
        };
#pragma unroll 1
        for (int sp = warp; sp < splits; sp += NW, src += stride * NW) {
            const uint32_t n = cnts[sp];
#pragma unroll 1
            for (uint32_t i0 = 4u * lane; i0 < n; i0 += 256u) {
                const uint4 q0 = load(src + (i0 - 4u * lane));
                const bool two = i0 + 128u < n;
                uint4 q1 = make_uint4(0u, 0u, 0u, 0u);
                if (two) q1 = load(src + (i0 - 4u * lane) + 128u);
                visit4(q0, i0, n);
                if (two) visit4(q1, i0 + 128u, n);
            }
        }
    };

    for (int level = 0; level < 4; ++level) {
        // ---- histogram sweep over the brackets in SEL_HIST ----
        for (int i = t; i < M * kSelBins; i += kSelThreads) hist[i] = 0;
        if (t == 0) {
            int n = 0;
            for (int g = 0; g < M; ++g) {       // brackets are in key order
                if (s_mode[g] != SEL_HIST) continue;
                s_tbl[n] = make_uint4(s_a[g], s_b[g] - s_a[g], s_sh[g], (uint32_t)(g * kSelBins));
                s_thr[n] = s_a[g] - 1u;
                ++n;
            }
            for (; n < M + 1; ++n) {
                s_tbl[n] = make_uint4(0u, 0u, 0u, 0u);
                s_thr[n] = 0xFFFFFFFFu;
            }
        }
        __syncthreads();
        {   // The brackets are disjoint, so a key feeds at most one histogram: three compares against the
            // first keys of the live brackets pick the table entry, one 128-bit shared load fetches its
            // parameters and ONE shared atomic follows (testing every bracket in turn cost 33 instructions
            // per key, this costs about 15).
            uint32_t thr[M];
#pragma unroll
            for (int i = 0; i < M; ++i) thr[i] = s_thr[i + 1];
            sweep(true, [&](uint32_t k, bool live) {
                uint32_t j = 0;
#pragma unroll
                for (int i = 0; i + 1 < M; ++i) j += k > thr[i] ? 1u : 0u;
                const uint4 e = s_tbl[j];
                const uint32_t d = k - e.x;
                if (live && d <= e.y) atomicAdd(&hist[e.w + (d >> e.z)], 1u);
            });
        }
        __syncthreads();

        // ---- a warp per bracket: where are its ranks? ----
        for (int g = warp; g < M; g += NW) {
            if (s_mode[g] != SEL_HIST) continue;
            constexpr int PER = kSelBins / 32;
            const uint32_t* h = hist + g * kSelBins + lane * PER;
            uint32_t sum = 0;
            for (int b = 0; b < PER; ++b) sum += h[b];
            uint32_t inc = sum;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t o = __shfl_up_sync(0xFFFFFFFFu, inc, d);
                if (lane >= d) inc += o;
            }
            const uint32_t total = __shfl_sync(0xFFFFFFFFu, inc, 31);
            const uint32_t pre = inc - sum;
            const long long x = col * kMaxRanks + s_iv[g];
            const uint32_t first = s_first[g], below = s_below[g], sh = s_sh[g];
            uint32_t nr = s_nr[g];
            __syncwarp();
            if (level == 0) {
                // `total` is the number of keys inside the bracket: the ranks beyond them are in the gap that
                // follows (the bracket missed them); they become a generic interval when the list is rebuilt
                uint32_t nin = 0;
                while (nin < nr && rp.rank[first + nin] - below < total) ++nin;
                if (lane == 0) {
                    w.iv_cnt[x] = total;
                    if (nin < nr) {
                        s_out_first[g] = first + nin; s_out_nr[g] = nr - nin;
                        s_out_below[g] = below + total; s_out_cnt[g] = s_region[g] - total;
                        s_nr[g] = nin; w.iv_nr[x] = nin;
                        s_rebuild = 1;
                        if (nin == 0) { s_keep[g] = 0; s_mode[g] = SEL_IDLE; }
                    }
                }
                nr = nin;
                __syncwarp();
                if (nr == 0) continue;
            }
            const uint32_t pos_f = rp.rank[first] - below;
            const uint32_t pos_l = rp.rank[first + nr - 1] - below;
            const bool sane = pos_l < total;
            if (sane && sh == 0) {
                // bins are single keys: every rank reads its key off the histogram
                for (uint32_t q = 0; q < nr; ++q) {
                    const uint32_t pos = rp.rank[first + q] - below;
                    if (pos >= pre && pos < pre + sum) {
                        uint32_t cum = pre; int b = 0;
                        while (pos >= cum + h[b]) { cum += h[b]; ++b; }
                        w.r_key[col * kMaxRanks + first + q] = s_a[g] + (uint32_t)(lane * PER + b);
                    }
                }
            } else if (sane) {
                if (pos_f >= pre && pos_f < pre + sum) {
                    uint32_t cum = pre; int b = 0;
                    while (pos_f >= cum + h[b]) { cum += h[b]; ++b; }
                    s_bf[g] = (uint32_t)(lane * PER + b); s_cb[g] = cum;
                }
                if (pos_l >= pre && pos_l < pre + sum) {
                    uint32_t cum = pre; int b = 0;
                    while (pos_l >= cum + h[b]) { cum += h[b]; ++b; }
                    s_bl[g] = (uint32_t)(lane * PER + b); s_n[g] = cum + h[b];   // keys up to and incl. bin bl
                }
            }
            __syncwarp();
            if (lane == 0) {
                if (!sane) {
                    s_mode[g] = SEL_IDLE;          // inconsistent lists: ranks stay poisoned (NaN)
                    atomicAdd(w.pending + 6, 1u);
                } else if (sh == 0) {
                    s_mode[g] = SEL_IDLE;
                    w.iv_status[x] = IV_RESOLVED;
                } else {
                    const uint32_t n_mid = s_n[g] - s_cb[g];
                    const uint32_t klo = s_a[g] + (s_bf[g] << sh);
                    unsigned long long last = (unsigned long long)s_a[g] + (((unsigned long long)s_bl[g] + 1ull) << sh) - 1ull;
                    if (last > (unsigned long long)s_b[g]) last = s_b[g];
                    if (n_mid <= (uint32_t)kSelBuf) {
                        s_mode[g] = SEL_COLLECT;
                        s_n[g] = 0;
                    } else if (s_bf[g] == s_bl[g] && level < 3) {
                        // all ranks in one crowded bin: histogram that bin next
                        s_a[g] = klo; s_b[g] = (uint32_t)last;
                        s_below[g] = below + s_cb[g];
                        s_sh[g] = sel_shift((uint32_t)last - klo, kSelBins);
                    } else {
                        // ranks in different crowded bins: generic interval for the exact pipeline
                        s_mode[g] = SEL_IDLE;
                        w.iv_klo[x] = klo; w.iv_khi[x] = (uint32_t)last;
                        w.iv_below[x] = below + s_cb[g];
                        w.iv_cnt[x] = n_mid;
                        if (n_mid <= (uint32_t)kCap) {
                            w.iv_status[x] = IV_COLLECT; w.iv_shift[x] = 0;
                            atomicAdd(w.pending + 1, 1u);
                            atomicAdd(w.pending + 4, 1u);
                        } else {
                            const uint32_t l = ceil_log2_u64(last - klo + 1ull);
                            w.iv_status[x] = IV_REFINE; w.iv_shift[x] = l > 5 ? l - 5 : 0;
                            atomicAdd(w.pending, 1u);
                            atomicAdd(w.pending + 5, 1u);
                        }
                    }
                }
            }
        }
        __syncthreads();
        bool again = false;
#pragma unroll
        for (int g = 0; g < M; ++g) again |= s_mode[g] == SEL_HIST;
        if (!again) break;
    }
    bool any_collect = false;
#pragma unroll
    for (int g = 0; g < M; ++g) {
        any_collect |= s_mode[g] == SEL_COLLECT;
        if (s_mode[g] == SEL_HIST && t == 0) atomicAdd(w.pending + 6, 1u);   // cannot happen (4 levels >= 32 bits)
    }
    // the interval list of the column with the gap intervals of missed ranks inserted in key order
    auto rebuild = [&]() {
        __syncthreads();
        if (t != 0 || !s_rebuild) return;
        IvList O, L;
        iv_load(O, w, col);
        L.n = 0;
        for (uint32_t v = 0; v < O.n; ++v) {
            int g = -1;
            for (int q = 0; q < M; ++q) if (s_iv[q] == v) g = q;
            if (g < 0 || s_keep[g]) {
                const uint32_t i = L.n++;
                L.klo[i] = O.klo[v]; L.khi[i] = O.khi[v]; L.shift[i] = O.shift[v]; L.below[i] = O.below[v];
                L.status[i] = O.status[v]; L.first[i] = O.first[v]; L.nr[i] = O.nr[v]; L.cnt[i] = O.cnt[v];
            }
            if (g >= 0 && s_out_nr[g]) {
                atomicAdd(w.pending + 2, s_out_nr[g]);
                const unsigned long long glo = (unsigned long long)w.bk_hi[col * kMaxGroups + g] + 1ull;
                iv_append(L, w, col, (uint32_t)glo, (unsigned long long)s_gap_hi[g] + 1ull - glo, s_out_below[g],
                          s_out_cnt[g], s_out_first[g], s_out_nr[g], false, 0u);
            }
        }
        iv_store(L, w, col);
    };
    if (!any_collect) { rebuild(); return; }

    // ---- second sweep: the keys of the target bins ----
    __syncthreads();
    if (t == 0) {                          // the same lookup over the target bins of the collecting brackets
        int n = 0;
        for (int g = 0; g < M; ++g) {
            if (s_mode[g] != SEL_COLLECT) continue;
            const uint32_t sh = s_sh[g];
            const uint32_t lo = s_a[g] + (s_bf[g] << sh);
            unsigned long long hi = (unsigned long long)s_a[g] + (((unsigned long long)s_bl[g] + 1ull) << sh) - 1ull;
            if (hi > (unsigned long long)s_b[g]) hi = s_b[g];
            s_tbl[n] = make_uint4(lo, (uint32_t)hi - lo, 0u, (uint32_t)g);
            s_thr[n] = lo - 1u;
            ++n;
        }
        for (; n < M + 1; ++n) {
            s_tbl[n] = make_uint4(0u, 0u, 0u, 0u);
            s_thr[n] = 0xFFFFFFFFu;
        }
    }
    __syncthreads();
    {
        uint32_t thr[M];
#pragma unroll
        for (int i = 0; i < M; ++i) thr[i] = s_thr[i + 1];
        sweep(false, [&](uint32_t k, bool live) {
            uint32_t j = 0;
#pragma unroll
            for (int i = 0; i + 1 < M; ++i) j += k > thr[i] ? 1u : 0u;
            const uint4 e = s_tbl[j];
            if (live && k - e.x <= e.y) {
                const uint32_t pos = atomicAdd(&s_n[e.w], 1u);
                if (pos < (uint32_t)kSelBuf) buf[e.w * kSelBuf + pos] = k;
            }
        });
    }
    __syncthreads();

    // ---- rank by counting: key e answers position q iff less(e) <= q < less(e) + equal(e) ----
    for (int g = 0; g < M; ++g) {
        if (s_mode[g] != SEL_COLLECT) continue;
        const uint32_t n = min(s_n[g], (uint32_t)kSelBuf);
        const uint32_t* bk = buf + g * kSelBuf;
        for (uint32_t e = t; e < n; e += kSelThreads) {
            const uint32_t ke = bk[e];
            uint32_t less = 0, eq = 0;
            for (uint32_t o = 0; o < n; ++o) {
                const uint32_t ko = bk[o];
                less += ko < ke ? 1u : 0u;
                eq += ko == ke ? 1u : 0u;
            }
            for (uint32_t q = 0; q < s_nr[g]; ++q) {
                const uint32_t pos = rp.rank[s_first[g] + q] - s_below[g] - s_cb[g];
                if (pos >= less && pos < less + eq) w.r_key[col * kMaxRanks + s_first[g] + q] = ke;
            }
        }
        if (t == 0) w.iv_status[col * kMaxRanks + s_iv[g]] = IV_RESOLVED;
    }
    rebuild();
}

// final rows: dB, numpy lerp, named statistics
__device__ __forceinline__ void finalize_body(long long col, long long rows, long long cols, const StatPlan& st, int to_dB,
                                              float eps, const Work& w, float* __restrict__ out /* [n_stats][cols] */) {
    if (col >= cols) return;
    auto xf = [&](uint32_t key) {
        const float v = key_to_float(key);
        return to_dB ? power_to_dB(v, eps) : v;
    };
    for (int t = 0; t < st.n_stats; ++t) {
        float r;
        const int kind = st.kind[t];
        if (kind == IQW_STAT_MEAN) {
            r = (float)(w.dsum[col] / (double)rows);
        } else if (kind == IQW_STAT_MAX) {
            r = xf(w.kmax[col]);
        } else if (kind == IQW_STAT_MIN) {
            r = xf(w.kmin[col]);
        } else {
            const float a = xf(w.r_key[col * kMaxRanks + st.ia[t]]);
            const float b = xf(w.r_key[col * kMaxRanks + st.ib[t]]);
            if (kind == IQW_STAT_MEDIAN) {
                r = __fmul_rn(__fadd_rn(a, b), 0.5f);
            } else if (kind == IQW_STAT_ORDER) {
                r = a;      // no arithmetic: +-inf stay what they are (a lerp would give inf - inf)
            } else {
                // numpy _lerp: a + (b-a)*g, or b - (b-a)*(1-g) where g >= 0.5; no fused ops
                const float g = st.gamma[t];
                const float d = __fsub_rn(b, a);
                r = g >= 0.5f ? __fsub_rn(b, __fmul_rn(d, __fsub_rn(1.0f, g)))
                              : __fadd_rn(a, __fmul_rn(d, g));
            }
        }
        out[(long long)t * cols + col] = r;
    }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------

__global__ void finalize_kernel(long long rows, long long cols, StatPlan st, int to_dB, float eps,
                                Work w, float* __restrict__ out /* [n_stats][cols] */) {
    finalize_body((long long)blockIdx.x * blockDim.x + threadIdx.x, rows, cols, st, to_dB, eps, w, out);
}

// ---------------------------------------------------------------------------------------------
// long-column path, everything after select in ONE cooperative launch: what select could not settle
// from the candidate lists (missed brackets, overflowed lists, heavy ties; about one call in a hundred)
// goes through the interval pipeline -- 7 x (refine, scan), collect, resolve -- with grid-wide barriers
// between the steps, then the result rows are written.  When nothing is open the kernel goes straight to
// the result rows: one launch where a train of 17 kernels used to exit one after the other (0.08 ms per
// call, a seventh of the whole configs[0] call).  Every condition that guards a barrier is read from
// memory while nobody writes it, so all CTAs take the same path.
// ---------------------------------------------------------------------------------------------
struct TailArgs {
    const float* p;
    long long rows, cols;
    unsigned gx, gy;              // virtual grid of the refine / collect steps (tile slots x row splits)
    long long rows_per_split;
    RankPlan rp;
    StatPlan st;
    int to_dB;
    float eps;
    Work w;
    float* out;
};

template <int M>
__global__ void __launch_bounds__(kBX)
tail_kernel(TailArgs a) {
    extern __shared__ __align__(16) unsigned char tail_smem[];
    cooperative_groups::grid_group grid = cooperative_groups::this_grid();
    const Work& w = a.w;
    const unsigned nvb = a.gx * a.gy;
    const unsigned cblocks = (unsigned)((a.cols + kBX - 1) / kBX);
    if ((w.pending[0] | w.pending[1]) != 0u) {          // select (the previous kernel) wrote them
        for (int level = 0; level < kRefineLevels; ++level) {
            const bool open = *w.pending != 0u;         // stable until the scan step below
            // (virtual block vb = tile slot * row splits + row split: the row splits of a pending tile spread over ALL CTAs)
            if (open)
                for (unsigned vb = blockIdx.x; vb < nvb; vb += gridDim.x)
                    refine_body<M>(vb / a.gy, vb % a.gy, a.gx, a.p, a.cols, a.rows, a.rows_per_split, w,
                                   reinterpret_cast<uint16_t*>(tail_smem));
            grid.sync();
            if (open)
                for (unsigned vb = blockIdx.x; vb < cblocks; vb += gridDim.x)
                    scan_refine_body((long long)vb * kBX + threadIdx.x, a.cols, a.rp, w);
            grid.sync();
        }
        if (w.pending[1] != 0u) {                       // nobody writes it after the last scan step
            for (unsigned vb = blockIdx.x; vb < nvb; vb += gridDim.x)
                collect_body<M>(vb / a.gy, vb % a.gy, a.gx, a.p, a.cols, a.rows, a.rows_per_split, w);
            grid.sync();
            for (long long col = blockIdx.x; col < a.cols; col += gridDim.x) {
                resolve_body(col, a.rp, w, reinterpret_cast<uint32_t*>(tail_smem));
                __syncthreads();
            }
        }
        grid.sync();
    }
    for (unsigned vb = blockIdx.x; vb < cblocks; vb += gridDim.x)
        finalize_body((long long)vb * kBX + threadIdx.x, a.rows, a.cols, a.st, a.to_dB, a.eps, w, a.out);
}

static int build_plans(const iqw_stat* stats, int n_stats, int64_t rows, RankPlan* rp, StatPlan* st,
                       bool* want_sum) {
    st->n_stats = n_stats;
    *want_sum = false;
    int64_t ranks[2 * kMaxStats];
    int nr = 0;
    for (int i = 0; i < n_stats; ++i) {
        const iqw_stat& s = stats[i];
        st->kind[i] = s.kind;
        st->gamma[i] = s.gamma;
        st->ia[i] = st->ib[i] = 0;
        if (s.kind < 0 || s.kind > IQW_STAT_ORDER)
            return fail(IQW_ERR_INVALID, "statistic %d: unknown kind %d", i, s.kind);
        if (s.kind == IQW_STAT_MEAN) *want_sum = true;
        if (s.kind == IQW_STAT_QUANTILE || s.kind == IQW_STAT_MEDIAN || s.kind == IQW_STAT_ORDER) {
            const int64_t lo = s.kind == IQW_STAT_MEDIAN ? (rows - 1) / 2 : s.rank_lo;
            const int64_t hi = s.kind == IQW_STAT_MEDIAN ? rows / 2 : s.kind == IQW_STAT_ORDER ? s.rank_lo : s.rank_hi;
            if (lo < 0 || hi < lo || hi >= rows)
                return fail(IQW_ERR_INVALID, "statistic %d: ranks (%lld, %lld) outside [0, %lld)", i,
                            (long long)lo, (long long)hi, (long long)rows);
            ranks[nr++] = lo;
            ranks[nr++] = hi;
        }
    }
    for (int i = 1; i < nr; ++i)
        for (int j = i; j > 0 && ranks[j] < ranks[j - 1]; --j) {
            int64_t tmp = ranks[j]; ranks[j] = ranks[j - 1]; ranks[j - 1] = tmp;
        }
    int nu = 0;
    for (int i = 0; i < nr; ++i)
        if (nu == 0 || ranks[i] != ranks[nu - 1]) ranks[nu++] = ranks[i];
    if (nu > kMaxRanks)
        return fail(IQW_ERR_UNSUPPORTED,
                    "%d distinct order statistics requested; at most %d per call (split the request)",
                    nu, kMaxRanks);
    rp->n_ranks = nu;
    for (int i = 0; i < nu; ++i) rp->rank[i] = (unsigned)ranks[i];
    for (int i = 0; i < n_stats; ++i) {
        const iqw_stat& s = stats[i];
        if (s.kind != IQW_STAT_QUANTILE && s.kind != IQW_STAT_MEDIAN && s.kind != IQW_STAT_ORDER) continue;
        const int64_t lo = s.kind == IQW_STAT_MEDIAN ? (rows - 1) / 2 : s.rank_lo;
        const int64_t hi = s.kind == IQW_STAT_MEDIAN ? rows / 2 : s.kind == IQW_STAT_ORDER ? s.rank_lo : s.rank_hi;
        for (int k = 0; k < nu; ++k) {
            if (ranks[k] == lo) st->ia[i] = k;
            if (ranks[k] == hi) st->ib[i] = k;
        }
    }
    return IQW_OK;
}

// long-column plan: row splits of the bracket pass, the row sample, and per group of target
// ranks the two SAMPLE ranks (margin-sigma away) whose keys bracket it.
static std::atomic<double> g_margin_sigmas{5.0};   // iqw_debug_set_sample_margin; 5 sigma: ~1 % of config-3 calls refine one column
static std::atomic<int> g_margin_extra{2};
static std::atomic<long long> g_sample_min_rows{kSampleMinRows};   // iqw_debug_set_sample_min_rows
constexpr long long kSampleRowsMin = 2048;
static std::atomic<long long> g_sample_share{8};                  // iqw_debug_set_sample_min_rows(-share)

struct LongPlan {
    long long splits, rows_per_split;
    RowMap sample;
    BracketPlan bp;
};

static void plan_long_shape(int64_t rows, int64_t cols, LongPlan* lp) {
    const long long col_tiles = (cols + kBX - 1) / kBX;
    long long splits = kBracketCtas / col_tiles;
    if (splits < 1) splits = 1;
    if (splits > kMaxSplits) splits = kMaxSplits;
    long long rps = (rows + splits - 1) / splits;
    if (rps < kMinRowsPerSplit) rps = kMinRowsPerSplit;
    // rps <= rows / 512 + 1 < 2^23 + 1 for rows < 2^32: the bracket pass counts rows in floats
    lp->rows_per_split = rps;
    lp->splits = (rows + rps - 1) / rps;
    // sample size: kSampleRows for long columns; shorter ones take rows / kSampleShare (at least kSampleRowsMin),
    // because the sample pass costs as much per sampled row as the bracket pass per row and twice-wider brackets
    // hardly matter when the whole matrix is small
    long long want = rows / g_sample_share.load();
    if (want < kSampleRowsMin) want = kSampleRowsMin;
    if (want > kSampleRows) want = kSampleRows;
    long long step = (rows + want - 1) / want;
    if (step < 2) step = 2;
    lp->sample = RowMap{rows / step, step, 0x9E3779B9u};
}

// widest bracket the default margins produce, in sample ranks (q = 1/2, one statistic's two ranks)
static long long max_group_width(long long srows) {
    return 2 * ((long long)std::ceil(6.0 * std::sqrt((double)srows * 0.25)) + 2) + 3;
}

// candidate-list budget per (row split, column), in keys, for `n_groups` brackets
static long long cap_budget(const LongPlan& lp, int n_groups) {
    double f = (double)n_groups * (double)(max_group_width(lp.sample.n) + 2) / (double)lp.sample.n;
    if (f > 1.0) f = 1.0;
    const long long cap = (long long)std::ceil(1.5 * (double)lp.rows_per_split * f) + 32ll * n_groups;
    return (cap + kLine - 1) / kLine * kLine;            // whole 128-byte lines
}

// Returns false when the sampled path does not apply (too many groups).
static bool build_long_plan(const RankPlan& rp, int64_t rows, int64_t cols, int n_stats, LongPlan* lp) {
    plan_long_shape(rows, cols, lp);
    const long long srows = lp->sample.n;
    const double f = (double)srows / (double)rows;
    auto margin = [&](double r) {
        const double q = r / (double)rows;
        return (int64_t)std::ceil(g_margin_sigmas.load() * std::sqrt((double)srows * q * (1.0 - q))) + g_margin_extra.load();
    };
    int64_t lo[kMaxRanks], hi[kMaxRanks];
    int ng = 0;
    for (int i = 0; i < rp.n_ranks; ++i) {
        const int64_t a = (int64_t)std::floor(rp.rank[i] * f) - margin(rp.rank[i]);
        const int64_t b = (int64_t)std::ceil(rp.rank[i] * f) + margin(rp.rank[i]);
        if (ng > 0 && a <= hi[ng - 1]) {               // overlaps the previous group: same bracket
            hi[ng - 1] = b > hi[ng - 1] ? b : hi[ng - 1];
        } else {
            lo[ng] = a; hi[ng] = b; ++ng;
        }
    }
    if (ng > kMaxGroups || ng > n_stats) return false;
    BracketPlan& bp = lp->bp;
    bp = BracketPlan{};
    bp.n_groups = ng;
    int64_t sr[2 * kMaxGroups];
    int ns = 0;
    for (int g = 0; g < ng; ++g) {
        const bool open_lo = lo[g] <= 0, open_hi = hi[g] >= srows - 1;
        bp.s_lo[g] = open_lo ? -1 : ns;
        if (!open_lo) sr[ns++] = lo[g];
        bp.s_hi[g] = open_hi ? -1 : ns;
        if (!open_hi) sr[ns++] = hi[g];
    }
    // sample ranks are ascending by construction (groups are disjoint); equal neighbours are legal
    bp.n_sranks = ns;
    for (int i = 0; i < ns; ++i) bp.srank[i] = (unsigned)sr[i];
    // candidate capacity per (row split, column): 1.5 x the expected share of the brackets plus
    // slack, within the budget the workspace was sized for
    double share = 0.0;
    for (int g = 0; g < ng; ++g) {
        const int64_t a = lo[g] < 0 ? 0 : lo[g], b = hi[g] > srows - 1 ? srows - 1 : hi[g];
        share += (double)(b - a + 3) / (double)srows;
    }
    if (share > 1.0) share = 1.0;
    long long cap = (long long)std::ceil(1.5 * (double)lp->rows_per_split * share) + 32ll * ng;
    const long long budget = cap_budget(*lp, n_stats < kMaxGroups ? n_stats : kMaxGroups);
    if (cap > budget) cap = budget;
    bp.cap_sum = (unsigned)(cap / kLine * kLine);       // whole 128-byte lines
    if (bp.cap_sum == 0) bp.cap_sum = kLine;
    return true;
}

struct Grid {
    dim3 grid;
    long long rows_per_split;
};

// grid of the streaming passes: tile slots (at most `max_slots` column tiles; a CTA walks the tiles of its slot) x
// row splits, enough CTAs to fill the machine `ctas_per_sm` times, < 65536 rows per split (uint16 counters)
static int plan_grid(long long n_rows, long long col_tiles, long long max_slots, int ctas_per_sm, int sms, Grid* g) {
    const long long slots = col_tiles < max_slots ? col_tiles : max_slots;
    long long splits = ((long long)ctas_per_sm * sms + slots - 1) / slots;
    if (splits < 1) splits = 1;
    long long rps = (n_rows + splits - 1) / splits;
    if (rps > 65535) rps = 65535;
    if (rps < 4 * kUnroll) rps = 4 * kUnroll;
    splits = (n_rows + rps - 1) / rps;
    if (splits > 65535) return fail(IQW_ERR_UNSUPPORTED, "too many rows for the split grid");
    g->grid = dim3((unsigned)slots, (unsigned)splits);
    g->rows_per_split = rps;
    return IQW_OK;
}

// the interval train: 7 x (refine, scan), collect, resolve; each kernel exits at once when nothing is open
template <int M>
static int launch_interval_train(const Grid& g, cudaStream_t s, const float* p, long long rows, long long cols,
                                 const RankPlan& rp, const Work& w, unsigned cblocks, unsigned cthreads) {
    static const char* const refine_names[kRefineLevels] = {"stats_refine_1", "stats_refine_2", "stats_refine_3",
                                                            "stats_refine_4", "stats_refine_5", "stats_refine_6",
                                                            "stats_refine_7"};
    const size_t smem = sizeof(uint16_t) * M * kNSub * kBX;
    cudaFuncSetAttribute(refine_kernel<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    for (int level = 0; level < kRefineLevels; ++level) {
        { IQW_PROFILE_FINE(refine_names[level], s);
          refine_kernel<M><<<g.grid, kBX, smem, s>>>(p, cols, rows, g.rows_per_split, w); }
        { IQW_PROFILE_FINE("stats_scan", s);
          scan_refine_kernel<<<cblocks, cthreads, 0, s>>>(cols, rp, w); }
    }
    { IQW_PROFILE_FINE("stats_collect", s);
      collect_kernel<M><<<g.grid, kBX, 0, s>>>(p, cols, rows, g.rows_per_split, w); }
    { IQW_PROFILE_FINE("stats_resolve", s);
      resolve_kernel<<<(unsigned)cols, kResolveThreads, 0, s>>>(cols, rp, w); }
    return IQW_OK;
}

template <int M>
static int launch_bracket_pass(cudaStream_t s, const float* p, long long cols, long long rows,
                               const LongPlan& lp, bool want_minmax, bool want_sum, bool to_dB, float eps,
                               const Work& w) {
    const dim3 grid((unsigned)((cols + kBX - 1) / kBX), (unsigned)lp.splits);
    IQW_PROFILE("stats_bracket_pass", s);
#define IQW_BP(N) bracket_pass_kernel<M, N><<<grid, kBX, 0, s>>>(p, cols, rows, lp.rows_per_split, eps, lp.bp, w)
    const int named = (want_minmax ? 1 : 0) | (want_sum ? 2 : 0) | (want_sum && to_dB ? 4 : 0);
    switch (named) {
        case 0: IQW_BP(0); break;
        case 1: IQW_BP(1); break;
        case 2: IQW_BP(2); break;
        case 3: IQW_BP(3); break;
        case 6: IQW_BP(6); break;
        default: IQW_BP(7); break;
    }
#undef IQW_BP
    return IQW_OK;
}

// grid of the cooperative tail kernel: every CTA must be resident (a few per SM are plenty: its common case is
// one pass over the result rows)
template <int M>
static int launch_tail(cudaStream_t s, const TailArgs& a, int sms) {
    constexpr size_t smem_refine = sizeof(uint16_t) * M * kNSub * kBX, smem_keys = sizeof(uint32_t) * kCap;
    constexpr size_t smem = smem_refine > smem_keys ? smem_refine : smem_keys;
    static std::atomic<int> blocks_per_sm[64];          // per device; 0: not asked yet, -1: no cooperative launch
    int dev = 0;
    IQW_CUDA_OK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) return IQW_ERR_UNSUPPORTED;
    int bps = blocks_per_sm[dev].load();
    if (bps == 0) {
        int coop = 0;
        IQW_CUDA_OK(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
        IQW_CUDA_OK(cudaFuncSetAttribute(tail_kernel<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        IQW_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, tail_kernel<M>, kBX, smem));
        if (!coop || bps < 1) bps = -1;
        else if (bps > 8) bps = 8;
        blocks_per_sm[dev].store(bps);
    }
    if (bps < 0) return IQW_ERR_UNSUPPORTED;
    TailArgs args = a;
    void* params[] = {&args};
    if (cudaLaunchCooperativeKernel((const void*)tail_kernel<M>, dim3((unsigned)(sms * bps)), dim3(kBX), params, smem, s) !=
        cudaSuccess) {
        (void)cudaGetLastError();           // e.g. the grid cannot be co-resident right now: the caller runs the train
        return IQW_ERR_UNSUPPORTED;
    }
    return IQW_OK;
}

template <int M>
static int launch_select(cudaStream_t s, long long cols, const RankPlan& rp, const LongPlan& lp, const Work& w) {
    const size_t smem = sizeof(uint32_t) * ((size_t)M * (kSelBins + kSelBuf) + (size_t)lp.splits);
    IQW_CUDA_OK(cudaFuncSetAttribute(select_kernel<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    IQW_PROFILE("stats_select", s);
    select_kernel<M><<<(unsigned)cols, kSelThreads, smem, s>>>(cols, (int)lp.splits, rp, lp.bp, w);
    return IQW_OK;
}

// Calls f(std::integral_constant<int, M>) with M, the register-array size of the interval and bracket kernels, the
// smallest power of two >= n that is at least 2^LO (n <= 8 intervals or brackets)
template <int LO, class F>
static int dispatch_m(int n, F&& f) {
    int l = LO;
    while (l < 3 && (1 << l) < n) ++l;
    return dispatch<LO, 3>(l, [&](auto L) { return f(std::integral_constant<int, 1 << decltype(L)::value>{}); },
                           [] { return IQW_ERR_INVALID; });
}

// exact pipeline on every row: leaves the key of every target rank in w.r_key
static int run_exact(const float* p, long long rows, long long cols, const RankPlan& rp, bool want_sum, bool to_dB,
                     float eps, const Work& w, int sms, cudaStream_t s) {
    const long long col_tiles = (cols + kBX - 1) / kBX;
    Grid g;
    if (int rc = plan_grid(rows, col_tiles, col_tiles, 16, sms, &g)) return rc;
    const unsigned cthreads = 128, cblocks = (unsigned)((cols + cthreads - 1) / cthreads);

    long long stride = rows / 2048;
    if (stride < 1) stride = 1;
    long long rsplits = (rows + stride - 1) / stride / 64;
    if (rsplits < 1) rsplits = 1;
    if (rsplits > 64) rsplits = 64;
    // (range, l0, scan0, 7 x (refine, scan), collect, resolve)
    IQW_PROFILE_TRAIN("stats_exact", s, rp.n_ranks > 0 ? 3 + 2 * kRefineLevels + 2 : 2);
    { IQW_PROFILE_FINE("stats_range", s);
      range_kernel<<<dim3((unsigned)col_tiles, (unsigned)rsplits), kBX, 0, s>>>(p, cols, rows, stride, w); }

    {
        IQW_PROFILE_FINE("stats_l0", s);
        const size_t smem = sizeof(uint16_t) * kNB0 * kBX;
        auto l0 = [&](auto kernel) {
            cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            kernel<<<g.grid, kBX, smem, s>>>(p, cols, rows, g.rows_per_split, eps, w);
        };
        if (want_sum && to_dB) l0(l0_kernel<true, true>);
        else if (want_sum) l0(l0_kernel<true, false>);
        else l0(l0_kernel<false, false>);
    }
    if (rp.n_ranks > 0) {
        { IQW_PROFILE_FINE("stats_scan", s);
          scan0_kernel<<<cblocks, cthreads, 0, s>>>(cols, rp, w); }
        if (int rc = dispatch_m<1>(rp.n_ranks, [&](auto M) {
                return launch_interval_train<M>(g, s, p, rows, cols, rp, w, cblocks, cthreads);
            }))
            return rc;
    }
    IQW_CUDA_OK(cudaGetLastError());
    return IQW_OK;
}

static int reset_work(const Work& w, cudaStream_t s) {
    // range_hi is the first field of the zero region; the 0xFF region follows it directly
    IQW_CUDA_OK(cudaMemsetAsync(w.range_hi, 0, w.zero_bytes, s));
    IQW_CUDA_OK(cudaMemsetAsync(reinterpret_cast<char*>(w.range_hi) + w.zero_bytes, 0xFF, w.ff_bytes, s));
    return IQW_OK;
}

}  // namespace iqw

using namespace iqw;

extern "C" int iqw_debug_set_sample_margin(double sigmas, int extra) {
    g_margin_sigmas = sigmas;
    g_margin_extra = extra;
    return IQW_OK;
}

// rows > 0: columns of at least `rows` rows take the sampled path; rows < 0: the sample is rows / (-rows) of a
// column (between kSampleRowsMin and kSampleRows rows); 0: both defaults
extern "C" int iqw_debug_set_sample_min_rows(int64_t rows) {
    if (rows < 0) { g_sample_share.store(-rows); return IQW_OK; }
    if (rows == 0) g_sample_share.store(8);
    g_sample_min_rows.store(rows < 1 ? kSampleMinRows : rows);
    return IQW_OK;
}

extern "C" int iqw_debug_time_stats_counters(const void* d_workspace, int64_t n_cols, uint32_t* host_out16) {
    if (!d_workspace || !host_out16 || n_cols < 1) return fail(IQW_ERR_INVALID, "bad argument");
    Work w{};
    carve_work(const_cast<void*>(d_workspace), n_cols, 0, 0, &w);
    IQW_CUDA_OK(cudaMemcpy(host_out16, w.pending, 16 * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return IQW_OK;
}

extern "C" size_t iqw_time_stats_workspace_bytes(int64_t n_channels, int64_t n_rows, int64_t n_cols,
                                                 int32_t n_stats) {
    (void)n_channels;
    if (n_cols <= 0) return 256;
    if (n_rows < g_sample_min_rows.load() || n_stats < 1) return carve_work(nullptr, n_cols, 0, 0, nullptr);
    LongPlan lp{};
    plan_long_shape(n_rows, n_cols, &lp);
    const int groups = n_stats < kMaxGroups ? n_stats : kMaxGroups;
    return carve_work(nullptr, n_cols, lp.splits, cap_budget(lp, groups), nullptr);
}

extern "C" int iqw_time_stats_f32(const float* d_p, int64_t n_channels, int64_t n_rows,
                                  int64_t n_cols, int64_t p_channel_stride, const iqw_stat* stats,
                                  int32_t n_stats, int32_t to_dB, float eps, float* d_out,
                                  void* d_workspace, size_t workspace_bytes, void* stream) {
    iqw::DeviceGuard _dev_guard(d_p);
    if (!d_p || !stats || !d_out || !d_workspace) return fail(IQW_ERR_INVALID, "null pointer argument");
    if (n_stats < 1 || n_stats > kMaxStats)
        return fail(IQW_ERR_INVALID, "n_stats=%d outside 1..%d", n_stats, kMaxStats);
    if (n_channels < 0 || n_rows < 1 || n_cols < 1)
        return fail(IQW_ERR_INVALID, "empty matrix (rows=%lld cols=%lld)", (long long)n_rows, (long long)n_cols);
    if (n_rows >= 0xFFFFFFFFll) return fail(IQW_ERR_UNSUPPORTED, "n_rows >= 2^32");
    if (((uintptr_t)d_workspace & 255) != 0) return fail(IQW_ERR_INVALID, "workspace not 256-byte aligned");

    RankPlan rp{};
    StatPlan st{};
    bool want_sum = false, want_minmax = false;
    if (int rc = build_plans(stats, n_stats, n_rows, &rp, &st, &want_sum)) return rc;
    for (int i = 0; i < n_stats; ++i)
        want_minmax |= stats[i].kind == IQW_STAT_MAX || stats[i].kind == IQW_STAT_MIN;
    if (n_cols >= (1ll << 27)) return fail(IQW_ERR_UNSUPPORTED, "n_cols >= 2^27");

    // long-column (sampled, one-read) path?
    LongPlan lp{};
    const bool sampled = n_rows >= g_sample_min_rows.load() && rp.n_ranks > 0 &&
                         build_long_plan(rp, n_rows, n_cols, n_stats, &lp);
    Work w{};
    const size_t need = sampled ? carve_work(d_workspace, n_cols, lp.splits, lp.bp.cap_sum, &w)
                                : carve_work(d_workspace, n_cols, 0, 0, &w);
    if (workspace_bytes < need)
        return fail(IQW_ERR_WORKSPACE, "workspace %zu bytes < required %zu", workspace_bytes, need);

    cudaStream_t s = static_cast<cudaStream_t>(stream);
    int sms = 0;
    if (int rc = device_sm_count(&sms)) return rc;
    const long long col_tiles = (n_cols + kBX - 1) / kBX;
    const unsigned cthreads = 128, cblocks = (unsigned)((n_cols + cthreads - 1) / cthreads);
    if (sampled)
        IQW_CUDA_OK(cudaFuncSetAttribute(sample_brackets_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)kSampleSmem));

    for (int64_t c = 0; c < n_channels; ++c) {
        const float* p = d_p + c * p_channel_stride;
        float* out = d_out + c * (int64_t)n_stats * n_cols;
        { IQW_PROFILE_FINE("stats_init", s); if (int rc = reset_work(w, s)) return rc; }

        if (!sampled) {
            if (int rc = run_exact(p, n_rows, n_cols, rp, want_sum, to_dB != 0, eps, w, sms, s)) return rc;
        } else {
            { IQW_PROFILE("stats_sample", s);
              sample_brackets_kernel<<<(unsigned)((n_cols + kSampleCols - 1) / kSampleCols), kSampleThreads,
                                       kSampleSmem, s>>>(p, n_cols, lp.sample, lp.bp, w); }
            if (int rc = dispatch_m<0>(lp.bp.n_groups, [&](auto M) {
                    return launch_bracket_pass<M>(s, p, n_cols, n_rows, lp, want_minmax, want_sum, to_dB != 0, eps, w);
                }))
                return rc;
            { IQW_PROFILE("stats_scan", s);
              scan_brackets_kernel<<<cblocks, cthreads, 0, s>>>(n_cols, n_rows, rp, lp.bp.n_groups, w); }
            if (int rc = dispatch_m<0>(lp.bp.n_groups, [&](auto M) { return launch_select<M>(s, n_cols, rp, lp, w); }))
                return rc;
            // whatever select could not settle from the lists (missed brackets, overflowed lists,
            // heavy ties) is refined from the matrix; these exit at once when nothing is open
            // few tile slots x many row splits: when one column misses, the whole GPU reads its tile
            Grid g;
            if (int rc = plan_grid(n_rows, col_tiles, 4, 32, sms, &g)) return rc;
            // what select left open (nothing, as a rule) and the result rows: one cooperative launch
            TailArgs ta{p, n_rows, n_cols, g.grid.x, g.grid.y, g.rows_per_split, rp, st, to_dB, eps, w, out};
            int rc_tail = IQW_OK;
            { IQW_PROFILE("stats_tail", s);
              rc_tail = dispatch_m<1>(rp.n_ranks, [&](auto M) { return launch_tail<M>(s, ta, sms); }); }
            if (rc_tail == IQW_ERR_UNSUPPORTED) {
                // no cooperative launch on this device: the same steps as a train of kernels, then finalize
                IQW_PROFILE_TRAIN("stats_tail_train", s, 2 * kRefineLevels + 3);
                if (int rc = dispatch_m<1>(rp.n_ranks, [&](auto M) {
                        return launch_interval_train<M>(g, s, p, n_rows, n_cols, rp, w, cblocks, cthreads);
                    }))
                    return rc;
                { IQW_PROFILE_FINE("stats_finalize", s);
                  finalize_kernel<<<cblocks, cthreads, 0, s>>>(n_rows, n_cols, st, to_dB, eps, w, out); }
            } else if (rc_tail != IQW_OK) {
                return rc_tail;
            }
        }
        if (!sampled) {
            IQW_PROFILE("stats_finalize", s);
            finalize_kernel<<<cblocks, cthreads, 0, s>>>(n_rows, n_cols, st, to_dB, eps, w, out);
        }
        IQW_CUDA_OK(cudaGetLastError());
    }
    return IQW_OK;
}
