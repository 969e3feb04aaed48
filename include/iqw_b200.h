/* iqw_b200.h -- C-ABI of the B200-native iqwaveform spectral-analysis hot path.
 *
 * The reference (dgkuester/iqwaveform 0.52.0, pure Python) has no FFI: its "backend boundary" is
 * the per-call switch on the array type (numpy -> scipy.fft / numpy, cupy -> cuFFT / cupy) inside
 * four public functions.  Each entry point below replaces the device-side work that one of those
 * functions delegates to its array backend; the Python package `iqwaveform_b200` keeps the
 * reference's signatures on top of them (see INTEGRATION.md for the ctypes binding a reference
 * maintainer would add).  Paths are relative to /root/reference/src/iqwaveform/.
 *
 * Conventions
 *  - every pointer named d_* is DEVICE memory on the current CUDA device; the caller owns all
 *    buffers, including workspaces; nothing here allocates or frees caller-visible memory (the
 *    library keeps one small immutable twiddle table per (device, nfft), built on first use)
 *  - `stream` is a cudaStream_t passed as void*; all work is enqueued asynchronously on it
 *  - complex64 is interleaved (re, im) float32; sizes are in ELEMENTS unless named *_bytes
 *  - return value: 0 on success, a negative iqw_status otherwise; iqw_last_error() returns a
 *    thread-local description of the last failure; no C++ exception crosses this boundary
 */
#ifndef IQW_B200_H
#define IQW_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IQW_ABI_VERSION 10

typedef enum iqw_status {
    IQW_OK = 0,
    IQW_ERR_INVALID = -1,      /* bad argument (null pointer, size, range) */
    IQW_ERR_UNSUPPORTED = -2,  /* valid in the reference but not built here (e.g. nfft not 2^k) */
    IQW_ERR_CUDA = -3,         /* a CUDA runtime call failed; text in iqw_last_error() */
    IQW_ERR_WORKSPACE = -4     /* workspace too small */
} iqw_status;

typedef enum iqw_stft_mode {
    IQW_STFT_COMPLEX = 0,  /* complex64 STFT                    (fourier.py:927 stft)            */
    IQW_STFT_POWER = 1,    /* float32 |X|^2                     (fourier.py:1203 spectrogram)    */
    IQW_STFT_DB = 2        /* float32 10*log10(|X|^2 + eps)     (power_analysis.py:168 powtodB)  */
} iqw_stft_mode;

/* statistic kinds for iqw_time_stats_f32 / iqw_bin_power_c64 (power_analysis.py:73-101) */
typedef enum iqw_stat_kind {
    IQW_STAT_QUANTILE = 0, /* numpy 'linear' quantile: lerp(a[rank_lo], a[rank_hi], gamma)        */
    IQW_STAT_MEAN = 1,     /* 'mean' and 'rms'                                                    */
    IQW_STAT_MAX = 2,      /* 'max' and 'peak'                                                    */
    IQW_STAT_MIN = 3,
    IQW_STAT_MEDIAN = 4,   /* numpy median: 0.5*(a[(n-1)/2] + a[n/2])                             */
    IQW_STAT_ORDER = 5     /* the order statistic a[rank_lo] itself (no interpolation)            */
} iqw_stat_kind;

/* one requested statistic (one output row).  For QUANTILE the host supplies the float32 index
 * arithmetic of numpy's 'linear' method -- rank_lo = floor((n-1)*q), rank_hi, gamma = frac --
 * computed exactly as numpy does (python: iqwaveform_b200._plan.quantile_plan). */
typedef struct iqw_stat {
    int32_t kind;     /* iqw_stat_kind */
    int64_t rank_lo;  /* QUANTILE only, 0-based order statistic */
    int64_t rank_hi;
    float gamma;
} iqw_stat;

int iqw_abi_version(void);
const char* iqw_last_error(void);

/* ---------------------------------------------------------------------------------------------
 * Kernel 1: overlapped-frame gather * window -> FFT -> {complex | |X|^2 | dB} -> band trim.
 * Replaces fourier.py:545-581 (_stack_stft_windows) + 1016-1028 (no-overlap branch) +
 * fourier.py:200-218 (fft) + power_analysis.py:251-255 (envtopow) + 196-204 (powtodB) +
 * the band slice of fourier.py:1289-1295, in ONE pass over the samples.
 *
 *   d_x           (n_channels, n_samples) complex64, row stride x_channel_stride elements
 *   d_window      nfft float32 coefficients that multiply a frame.  The caller folds in the
 *                 (-1)^n fft-shift, the 1/nfft and (norm=None) the COLA scale, exactly as the
 *                 reference does on the host (fourier.py:1002-1010, 1033, 571-580)
 *   nfft          power of two, 16 <= nfft <= 65536 (others: IQW_ERR_UNSUPPORTED).  Up to 8192 a
 *                 frame is transformed inside one CTA's shared memory; 16384..65536 run as a
 *                 two-kernel four-step FFT through d_workspace
 *   hop           nfft - noverlap >= 1;  frame m covers samples [m*hop, m*hop + nfft)
 *   n_frames      T <= (n_samples - nfft)/hop + 1
 *   bin_lo,bin_hi output bins [bin_lo, bin_hi) of the fft-shifted spectrum (0, nfft = all)
 *   d_out         (n_channels, n_frames, bin_hi-bin_lo), complex64 (COMPLEX) or float32,
 *                 C-contiguous, channel stride out_channel_stride elements
 *   d_workspace   >= iqw_stft_workspace_bytes(nfft, n_channels, n_frames) bytes, 16-byte aligned;
 *                 may be NULL when that is 0 (nfft <= 8192).  Any size >= one frame (8*nfft bytes)
 *                 works: frames are processed in chunks that fit
 */
size_t iqw_stft_workspace_bytes(int32_t nfft, int64_t n_channels, int64_t n_frames);
int iqw_stft_c64(const void* d_x, int64_t n_channels, int64_t n_samples, int64_t x_channel_stride,
                 const float* d_window, int32_t nfft, int64_t hop, int64_t n_frames, int32_t mode,
                 float eps, int32_t bin_lo, int32_t bin_hi, void* d_out,
                 int64_t out_channel_stride, void* d_workspace, size_t workspace_bytes, void* stream);

/* Kernel 1 for frame lengths that are not a power of two (the reference takes nfft = round(fs/resolution),
 * fourier.py:1250-1255, and any length goes to scipy.fft / cuFFT, fourier.py:200-218): Bluestein's chirp-z
 * transform -- gather x window x chirp -> M-point FFT -> x filter spectrum -> M-point inverse FFT -> chirp ->
 * epilogue -- inside one CTA, M = the power of two >= 2*nfft - 1.  The host supplies the three tables
 * (python: iqwaveform_b200._plan.bluestein_tables, float64 design):
 *   d_pre   nfft complex64: frame coefficient (window, (-1)^n, 1/nfft ...) times exp(-i pi n^2 / nfft)
 *   d_bh    m complex64:    FFT_m of the wrapped chirp exp(+i pi j^2 / nfft), divided by m
 *   d_post  nfft complex64: exp(-i pi k^2 / nfft)
 * nfft <= 4096 (m <= 8192); the other arguments are those of iqw_stft_c64. */
int iqw_stft_bluestein_c64(const void* d_x, int64_t n_channels, int64_t n_samples, int64_t x_channel_stride,
                           const void* d_pre, const void* d_bh, const void* d_post, int32_t nfft, int32_t m,
                           int64_t hop, int64_t n_frames, int32_t mode, float eps, int32_t bin_lo,
                           int32_t bin_hi, void* d_out, int64_t out_channel_stride, void* stream);
/* Longer frames (m = 16384 .. 65536): the same transform composed from three elementwise kernels around two
 * calls of iqw_stft_c64 (nfft = m, hop = m, all-ones window, complex output) on a (n_frames, m) scratch:
 *   pre:  a[f][j] = x[f*hop + j] * pre[j] (j < nfft), 0 otherwise      then  A = FFT rows(a)
 *   mul:  A[f][k] = conj(A[f][k] * bh[k]) in place                      then  r = FFT rows(A)
 *   post: X[f][k] = post[k] * conj(r[f][k]), k in [bin_lo, bin_hi)  ->  d_out (n_frames, bin_hi - bin_lo) */
int iqw_bluestein_pre_c64(const void* d_x, int64_t hop, const void* d_pre, int32_t nfft, int32_t m,
                          int64_t n_frames, void* d_a, void* stream);
int iqw_bluestein_mul_c64(void* d_a, const void* d_bh, int32_t m, int64_t n_frames, void* stream);
int iqw_bluestein_post_c64(const void* d_a, const void* d_post, int32_t m, int64_t n_frames, int32_t mode,
                           float eps, int32_t bin_lo, int32_t bin_hi, void* d_out, void* stream);

/* Kernel 1 with the reducible time statistics fused into its epilogue: persistence spectrum with
 * statistics drawn from {mean, rms, max, peak, min} WITHOUT materialising the spectrogram (8 B per
 * sample of HBM traffic instead of 24).  Replaces fourier.py:1287-1301 (spectrogram, band slice, powtodB)
 * + fourier.py:1322-1325 (np.max / np.min / np.mean over the time axis) for that case.  Every frame slot
 * of the grid keeps max, min and a compensated sum of the bins it owns over its frames; a small second
 * kernel combines the partial rows.  mean averages the dB values when to_dB (like the reference, which
 * converts the spectrogram first); max / min are taken on the power and converted once (monotone map).
 *   stats        kinds IQW_STAT_MEAN / MAX / MIN only (others: IQW_ERR_UNSUPPORTED)
 *   nfft         power of two, 16 <= nfft <= 8192
 *   d_out        (n_channels, n_stats, bin_hi - bin_lo) float32
 *   d_workspace  >= iqw_stft_reduce_workspace_bytes(nfft) bytes
 * The other arguments are those of iqw_stft_c64. */
size_t iqw_stft_reduce_workspace_bytes(int32_t nfft);
int iqw_stft_reduce_c64(const void* d_x, int64_t n_channels, int64_t n_samples, int64_t x_channel_stride,
                        const float* d_window, int32_t nfft, int64_t hop, int64_t n_frames, int32_t to_dB,
                        float eps, int32_t bin_lo, int32_t bin_hi, const iqw_stat* stats, int32_t n_stats,
                        float* d_out, void* d_workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Kernel 2: statistics over the time axis of a (n_channels, n_rows, n_cols) float32 matrix
 * (rows = frames, cols = bins): exact order statistics + numpy 'linear' lerp, mean, max, min.
 * Replaces fourier.py:1311-1325 (np.quantile / stat ufuncs over axis) and, with to_dB != 0,
 * the in-place powtodB of fourier.py:1298-1299 (applied to the selected order statistics, which
 * is identical because 10*log10(p + eps) is monotone; 'mean' averages the dB values of every
 * element, as the reference does).
 *
 *   d_p            input matrix; row stride = n_cols, channel stride p_channel_stride elements
 *   stats          HOST array of n_stats requests (copied during the call)
 *   d_out          (n_channels, n_stats, n_cols) float32, C-contiguous
 *   d_workspace    >= iqw_time_stats_workspace_bytes(...) bytes, 256-byte aligned
 */
size_t iqw_time_stats_workspace_bytes(int64_t n_channels, int64_t n_rows, int64_t n_cols,
                                      int32_t n_stats);
int iqw_time_stats_f32(const float* d_p, int64_t n_channels, int64_t n_rows, int64_t n_cols,
                       int64_t p_channel_stride, const iqw_stat* stats, int32_t n_stats,
                       int32_t to_dB, float eps, float* d_out, void* d_workspace,
                       size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Kernel 3: per-bin envelope power of contiguous bins of bin_len samples.
 * Replaces power_analysis.py:380-385 (to_blocks + envtopow + mean/max/min detector).
 *
 *   d_x        (n_channels, >= n_bins*bin_len) complex64, row stride x_channel_stride elements
 *   d_mean / d_max / d_min   each NULL or (n_channels, n_bins) float32
 *   d_workspace  >= iqw_bin_power_workspace_bytes(...) bytes, 256-byte aligned (only touched when
 *                there are too few bins to fill the GPU and bins are split across CTAs)
 */
size_t iqw_bin_power_workspace_bytes(int64_t n_channels, int64_t bin_len, int64_t n_bins);
int iqw_bin_power_c64(const void* d_x, int64_t n_channels, int64_t x_channel_stride,
                      int64_t bin_len, int64_t n_bins, float* d_mean, float* d_max, float* d_min,
                      void* d_workspace, size_t workspace_bytes, void* stream);

/* |x|^2 of (n_channels, n_bins, bin_len) complex64 written TRANSPOSED as float32
 * (n_channels, bin_len, n_bins), so that the median / quantile detectors of iq_to_bin_power
 * (power_analysis.py:382-385 with kind='median' or a float) run through iqw_time_stats_f32,
 * whose statistics axis is the row axis.  Replaces power_analysis.py:251-255 for that case. */
int iqw_envtopow_transposed_c64(const void* d_x, int64_t n_channels, int64_t x_channel_stride,
                                int64_t bin_len, int64_t n_bins, float* d_out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Elementwise power transforms (power_analysis.py:168-298): float32 out, one streaming pass.
 *   op 0 powtodB  : 10*log10(abs(x) + eps)   (use_abs == 0: 10*log10(x + eps))
 *   op 1 dBtopow  : 10**(x/10)
 *   op 2 envtopow : abs(x)**2
 *   op 3 envtodB  : 20*log10(abs(x) + eps)   (use_abs == 0: 20*log10(x + eps))
 * iqw_elementwise_c64 takes complex64 input and supports ops 2 and 3 (abs is the modulus).
 */
typedef enum iqw_ew_op { IQW_EW_POWTODB = 0, IQW_EW_DBTOPOW = 1, IQW_EW_ENVTOPOW = 2, IQW_EW_ENVTODB = 3 } iqw_ew_op;
int iqw_elementwise_f32(int32_t op, const float* d_in, float* d_out, int64_t n, int32_t use_abs, float eps,
                        void* stream);
int iqw_elementwise_c64(int32_t op, const void* d_in, float* d_out, int64_t n, float eps, void* stream);

/* (batch, rows, cols) complex64 -> (batch, cols, rows): brings a capture whose time axis is not the last one
 * ((N, C) with axis = 0, util.py:400-442) to the (channels, time) layout of the kernels without a framework
 * copy on the data path.  cols <= 2 097 120, batch <= 65535. */
int iqw_transpose_c64(const void* d_in, int64_t batch, int64_t rows, int64_t cols, void* d_out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Kernel 4: inverse STFT with overlap-add, optionally band-masked / zero-padded / filtered
 * (SURVEY.md 8f rank 3: istft, ola_filter, oaresample).
 * Replaces fourier.py:1060-1105 (istft: ifft + the (-1)^n 'rect' window) + fourier.py:584-649
 * (_unstack_stft_windows) and, with a bin range, fourier.py:710-723 (zero_stft_by_freq, the
 * filter step of ola_filter, fourier.py:1108-1181), in ONE pass over the frames.
 *
 *   d_y          (n_channels, n_frames, y_bins) complex64 STFT in the fft-shifted bin order that
 *                iqw_stft_c64 produces; channel stride y_channel_stride elements
 *   nfft         power of two, 16 <= nfft <= 8192
 *   hop          nfft/hop must be 1, 2, 4, 8 or 16 (the reference's own summation is only an
 *                overlap-add when hop divides nfft)
 *   bin_lo,bin_hi  bins outside [bin_lo, bin_hi) are taken as zero (0, nfft = no mask)
 *   y_bins       bins STORED per frame: nfft (whole frames; the band is a read mask -- ola_filter),
 *                or bin_hi - bin_lo (only the band is stored and sits at bins [bin_lo, bin_hi) of a
 *                longer frame: the zero padding of the upsampling oaresample, fourier.py:1694-1699)
 *   d_bin_gain   NULL, or nfft complex64 gains that multiply the bins (the frequency-domain FIR of
 *                stft_fir_lowpass, fourier.py:803-826)
 *   scale        factor applied to every output sample after the overlap-add (oaresample's
 *                x.size/size_in*scale, fourier.py:1723; 1 otherwise)
 *   d_out        (n_channels, n_frames*hop + nfft - hop) complex64, channel stride
 *                out_channel_stride elements: every sample is the plain sum of the frames that
 *                cover it (no division by the window overlap, like the reference); the caller
 *                trims it (`size` argument of the reference) by slicing
 */
int iqw_istft_c64(const void* d_y, int64_t n_channels, int64_t n_frames, int64_t y_channel_stride,
                  int32_t nfft, int64_t hop, int32_t bin_lo, int32_t bin_hi, int32_t y_bins,
                  const void* d_bin_gain, float scale, void* d_out, int64_t out_channel_stride,
                  void* stream);

/* Plain batched inverse DFT of row A4's public pair fft / ifft (fourier.py:221-246, the scipy.fft.ifft
 * / cuFFT-inverse call): out[r][n] = 1/nfft * sum_k y[r][k] * exp(+2*pi*i*k*n/nfft), bins and samples
 * in NATURAL order.  Kernel 4 with hop = nfft and without the (-1)^n of the baked-in shift.  d_y and
 * d_out are (n_rows, nfft) complex64, C-contiguous; nfft a power of two, 16..8192.  (The forward
 * transform of fourier.py:200-218 needs no entry of its own: iqw_stft_c64 with an all-ones window,
 * hop = nfft, n_frames = n_rows and mode COMPLEX is the unnormalised natural-order DFT of every row,
 * for nfft up to 65536.) */
int iqw_ifft_c64(const void* d_y, int64_t n_rows, int32_t nfft, void* d_out, void* stream);

/* The whole of ola_filter (fourier.py:1108-1181 with nfft_out == nfft) in ONE kernel: overlapped
 * frame gather * window -> FFT -> zero the bins outside [bin_lo, bin_hi) -> inverse FFT -> (-1)^n ->
 * overlap-add.  The STFT is never written: 8 B read + 8 B written per sample.  d_x / d_window /
 * nfft / hop / n_frames as for iqw_stft_c64 (the window carries (-1)^n, 1/nfft and the COLA
 * scale); d_out as for iqw_istft_c64.  Same result as iqw_stft_c64 (complex) + iqw_istft_c64. */
int iqw_ola_filter_c64(const void* d_x, int64_t n_channels, int64_t n_samples, int64_t x_channel_stride,
                       const float* d_window, int32_t nfft, int64_t hop, int64_t n_frames,
                       int32_t bin_lo, int32_t bin_hi, void* d_out, int64_t out_channel_stride,
                       void* stream);


/* ---------------------------------------------------------------------------------------------
 * Kernel 5: counts[row][i] = number of samples x of the row with searchsorted(edges, x, side) == i,
 * i = 0 .. n_edges (SURVEY.md 8f rank 4).  The device part of power_analysis.py:552-583
 * (sample_ccdf: side 'left', then N - cumsum) and util.py:497-543 (histogram_last_axis: side
 * 'right', columns 1 .. n_edges-1 are the histogram).
 *
 *   d_a       (n_rows, n_cols) float32, C-contiguous      d_edges  n_edges float64, ascending
 *   d_counts  (n_rows, n_edges + 1) int64, zeroed by the call.  n_edges <= 4096
 */
int iqw_edge_counts_f32(const float* d_a, int64_t n_rows, int64_t n_cols, const double* d_edges,
                        int32_t n_edges, int32_t side_right, int64_t* d_counts, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Kernel 6: polyphase FIR filter / rational resampler with the semantics of scipy.signal.upfirdn
 * (zero padding only): zero-stuff by `up`, convolve in full with the L taps h, keep every `down`-th
 * sample.  Replaces the reference's fourier.upfirdn (fourier.py:1476-1495: scipy.signal.upfirdn on
 * the host, the NVRTC polyphase kernel of cuda.py on cupy arrays).
 *
 *   y[n] = sum_{j < Lp} hp[p][j] * x[i0 - j],  t = n*down, p = t mod up, i0 = t div up
 *
 *   d_x           (n_channels, n_in) complex64, row stride x_channel_stride elements; d_x[0] is the
 *                 sample of GLOBAL index x_first (0 for a whole capture; a time shard passes the first
 *                 sample it holds).  Samples outside [x_first, x_first + n_in) read as zero
 *   d_taps        the polyphase table hp[p][j] = h[p + j*up] for p < min(up, n_taps) and
 *                 j < Lp = ceil(n_taps/up), zero-padded: float32 (taps_complex = 0) or complex64
 *                 (python: iqwaveform_b200._plan.upfirdn_polyphase).  At most 32768 floats
 *                 (16384 real or 8192 complex taps for any up; larger: IQW_ERR_UNSUPPORTED)
 *   out_first     global index of the first output; the call writes outputs
 *                 [out_first, out_first + n_out) to d_out (n_channels, n_out) complex64, channel stride
 *                 out_channel_stride elements
 * The summation order of an output depends only on its global index and (up, down, n_taps), so shards
 * of one capture concatenate to the bits of a single call. */
int iqw_upfirdn_c64(const void* d_x, int64_t n_channels, int64_t n_in, int64_t x_channel_stride, int64_t x_first,
                    const void* d_taps, int32_t taps_complex, int32_t n_taps, int32_t up, int32_t down,
                    int64_t out_first, int64_t n_out, void* d_out, int64_t out_channel_stride, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Kernel 7: FFT convolution of complex64 rows with an M-tap filter by overlap-save, the output windows
 * of scipy.signal.oaconvolve.  Replaces the reference's fourier.oaconvolve (fourier.py:1496-1509:
 * scipy.signal.oaconvolve on the host, cupyx on cupy arrays).
 *
 *   y[n] = sum_{k < n_taps} h[k] * x[n - k],  n a global index of the full convolution
 *
 *   d_x           (n_channels, n_in) complex64, row stride x_channel_stride elements; d_x[0] is the
 *                 sample of GLOBAL index x_first (0 for a whole capture; a time shard passes the first
 *                 sample it holds).  Samples outside [x_first, x_first + n_in) read as zero
 *   d_hspec       H = fft(h, nfft) / nfft, complex64, one row (hspec_channel_stride = 0: the same
 *                 filter for every channel) or one row per channel (hspec_channel_stride = nfft)
 *                 (python: iqwaveform_b200._plan.oaconvolve_spectrum)
 *   nfft, discard blocks of nfft samples keep their last nfft - discard; nfft/discard in {2, 4, 8, 16},
 *                 discard >= n_taps - 1 (else IQW_ERR_INVALID).  Built: the (nfft, discard) pairs
 *                 that python's _plan.oaconvolve_plan picks for 1..4097 taps; other pairs return
 *                 IQW_ERR_UNSUPPORTED
 *   out_first     global index of the first output; the call writes outputs
 *                 [out_first, out_first + n_out) to d_out (n_channels, n_out) complex64, channel stride
 *                 out_channel_stride elements
 * Blocks are anchored at global index 0, never at out_first: a window of the full convolution is a
 * bitwise crop of it, and time shards that hold each of their blocks' in-range samples (the discard
 * before their first output) concatenate to the bits of a single call. */
int iqw_oaconvolve_c64(const void* d_x, int64_t n_channels, int64_t n_in, int64_t x_channel_stride, int64_t x_first,
                       const void* d_hspec, int64_t hspec_channel_stride, int32_t n_taps, int32_t nfft,
                       int32_t discard, int64_t out_first, int64_t n_out, void* d_out, int64_t out_channel_stride,
                       void* stream);

/* ---------------------------------------------------------------------------------------------
 * Exact order statistics of a float32 matrix whose ROWS are spread over several GPUs (the
 * time-sharded persistence spectrum; no reference counterpart -- the reference calls np.quantile
 * on the whole spectrogram in one process, fourier.py:1317-1320).  Most-significant-digit radix
 * select on order-preserving uint32 keys (key = bits ^ 0x80000000 for non-negative floats,
 * ~bits for negative ones), 8 bits per level, levels 0..3, inside a key interval [lo, hi] per
 * column and statistic that the caller seeds with a bracket known to hold the statistic
 * (0 .. 0xFFFFFFFF always works; a tight bracket makes the passes HBM-bound because only rows
 * inside the interval touch the histograms):
 *
 *   iqw_bracket_collect_f32  ONE pass over this device's rows: rows with key < lo per statistic
 *                         -> d_below rows 0..n_sel-1; rows inside ANY [lo, hi] are copied to the
 *                         candidate store in d_workspace; d_below row n_sel counts, per column,
 *                         the store segments that overflowed (heavy ties): if its sum over the
 *                         devices is non-zero anywhere, use iqw_radix_count_f32 instead of
 *                         iqw_candidate_count_f32 below.  n_sel <= 8 per call.
 *   iqw_candidate_count_f32  like iqw_radix_count_f32, over the candidate store
 *   iqw_radix_count_f32   counts of THIS device's rows with lo <= key <= hi by key digit
 *                         (key >> (24 - 8*level)) & 255, per statistic and column; with d_below,
 *                         also the rows with key < lo.  Both outputs are zeroed by the call.
 *   (caller)              all_reduce(SUM) of d_counts (and d_below) over the devices holding rows;
 *                         at level 0 the caller subtracts the summed d_below from d_rank
 *   iqw_radix_descend     walks the summed counts: the digit that holds the residual rank is
 *                         appended to the prefix, the rank is made relative to that bucket and
 *                         [lo, hi] is intersected with the bucket.  After level 3 d_prefix holds
 *                         the keys of the order statistics.  A rank outside the counted rows ends
 *                         as the key of NaN.
 *   iqw_order_stats_finish_f32  dB (optional) of the selected values + numpy 'linear' lerp /
 *                         median, as the last step of iqw_time_stats_f32 does.
 *
 *   d_p        (n_rows, n_cols) float32, C-contiguous; n_rows may be 0
 *   d_lo,d_hi  (n_sel, n_cols) uint32 keys, in/out of iqw_radix_descend
 *   d_prefix   (n_sel, n_cols) uint32        d_rank  (n_sel, n_cols) int64, in/out
 *   d_counts   (n_sel, n_cols, 256) int32    d_below NULL or (n_sel, n_cols) int32
 *              (iqw_bracket_collect_f32: (n_sel + 1, n_cols), required)
 *   d_workspace >= iqw_bracket_collect_workspace_bytes(n_rows, n_cols) bytes (about 1/8 of the
 *              matrix), 256-byte aligned; the same n_rows / n_cols go to iqw_candidate_count_f32
 *   sel_rank   HOST array: the 0-based global rank each of the n_sel rows of d_keys answers
 *   stats      HOST array of QUANTILE / MEDIAN requests whose ranks are all in sel_rank
 *   d_out      (n_stats, n_cols) float32
 */
size_t iqw_bracket_collect_workspace_bytes(int64_t n_rows, int64_t n_cols);
int iqw_bracket_collect_f32(const float* d_p, int64_t n_rows, int64_t n_cols, int32_t n_sel,
                            const uint32_t* d_lo, const uint32_t* d_hi, int32_t* d_below,
                            void* d_workspace, size_t workspace_bytes, void* stream);
int iqw_candidate_count_f32(const void* d_workspace, int64_t n_rows, int64_t n_cols, int32_t n_sel,
                            const uint32_t* d_lo, const uint32_t* d_hi, int32_t level,
                            int32_t* d_counts, void* stream);
int iqw_radix_count_f32(const float* d_p, int64_t n_rows, int64_t n_cols, int32_t n_sel,
                        const uint32_t* d_lo, const uint32_t* d_hi, int32_t level,
                        int32_t* d_counts, int32_t* d_below, void* stream);
int iqw_radix_descend(const int32_t* d_counts, int32_t n_sel, int64_t n_cols, int32_t level,
                      int64_t* d_rank, uint32_t* d_prefix, uint32_t* d_lo, uint32_t* d_hi,
                      void* stream);
int iqw_order_stats_finish_f32(const uint32_t* d_keys, int32_t n_sel, const int64_t* sel_rank,
                               int64_t n_rows_total, int64_t n_cols, const iqw_stat* stats,
                               int32_t n_stats, int32_t to_dB, float eps, float* d_out, void* stream);

/* Tuning aid: bytes of scratch iqw_stft_workspace_bytes asks for (nfft > 8192); frames are
 * processed in chunks of that size. */
int iqw_debug_set_stft_scratch_cap(size_t bytes);

/* Tuning aid: columns of at least this many rows take the sampled one-read path of iqw_time_stats_f32
 * (default 16384; 0 restores it); shorter ones the exact multi-pass pipeline.  Results are exact either way.
 * Set it before iqw_time_stats_workspace_bytes: the workspace layout depends on the path.
 * A NEGATIVE value sets the sample size instead: rows / (-value) of a column, between 2048 and 8192 rows (default 8). */
int iqw_debug_set_sample_min_rows(int64_t rows);

/* Tuning aid: which kernel-1 geometry serves nfft 1024 / 2048 / 4096.  0 = automatic (the two-pass
 * kernel, csrc/iqw_stft2p.cu: 32 / 64 values per thread, one shared-memory exchange per frame, frames
 * staged by bulk copies (TMA) when every frame start is 16-byte aligned), 1 = always the three-pass kernel
 * (csrc/iqw_stft.cu: 16 values per thread, two exchanges), 2 = two-pass with plain global loads, 3 = two-pass
 * staged (same as 0).  The same switch serves nfft 8192 .. 65536: 0 = the one-pass kernel that keeps the frame
 * in (distributed) shared memory, a thread-block cluster of 2 / 4 CTAs at nfft 32768 / 65536
 * (csrc/iqw_stft3p.cu), 1 = the three-pass kernel (8192) / the two-kernel four-step path through the
 * workspace (16384 .. 65536).  All compute the same transform; results differ by float32 rounding only. */
int iqw_debug_set_stft_variant(int variant);

/* Test aid: width of the brackets the row sample puts around each target rank on the long-column
 * path of iqw_time_stats_f32 (default 5 sigma + 2 ranks).  Results are exact for ANY setting -- a
 * bracket that misses its rank is refined like any other interval -- which is what the tests use
 * this for (margin 0 makes about half of the brackets miss). */
int iqw_debug_set_sample_margin(double sigmas, int extra_ranks);

/* Test aid: counters of the LAST channel iqw_time_stats_f32 processed with this workspace
 * (synchronises the device): out[0] intervals still to refine, [1] intervals collected from the
 * matrix, [2] ranks whose bracket missed, [3] brackets of columns whose candidate lists
 * overflowed, [4]/[5] brackets handed from the candidate lists back to the matrix passes (heavy
 * ties), [6] inconsistent candidate lists (a bug if ever non-zero), [7] brackets settled from the
 * candidate lists alone (the fast path), [8] 1 if the bracket pass compared order-preserving keys
 * instead of raw float bits (some bracket bound was negative), [9..15] reserved. */
int iqw_debug_time_stats_counters(const void* d_workspace, int64_t n_cols, uint32_t* host_out16);

/* ---------------------------------------------------------------------------------------------
 * Measurement aid (no reference counterpart): kernel launches of the library are bracketed by CUDA
 * events on the launching stream.  level 0: off.  level 1: the heavy kernels one by one, and each
 * train of small follow-up kernels (the fallback chain of iqw_time_stats_f32) as ONE scope, so that
 * a timed region carries ~12 events per persistence-spectrum step instead of ~46 (which cost 2 % of
 * it).  level 2: every launch.  iqw_profile_report writes one text line per scope name,
 * "<name> <launches covered> <total_ms>\n"; call it after synchronising the stream(s).
 */
int iqw_profile_enable(int level);
int iqw_profile_reset(void);
int iqw_profile_report(char* buf, size_t capacity);

#ifdef __cplusplus
}
#endif
#endif /* IQW_B200_H */
