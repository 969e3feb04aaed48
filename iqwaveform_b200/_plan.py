"""host-side planning: window design, numpy-compatible quantile index arithmetic, axis arrays.

Everything here is O(nfft) or O(n_statistics) work done once per configuration and cached; it is
the part of the reference that already lives on the host for every backend
(/root/reference/src/iqwaveform/fourier.py:70-157, 248-269, 348-357, 1184-1200; util.py:121-141).
"""
from __future__ import annotations

import functools
import math
from numbers import Number

import numpy as np

from . import _lib

INF = float('inf')


def isroundmod(value: float, div: float, atol: float = 1e-6) -> bool:
    """util.py:136-141"""
    return abs(math.remainder(value / div, 1)) <= atol


def find_float_inds(seq) -> list[bool]:
    """util.py:121-133: True where the statistic reads as a float (a quantile)"""
    flags = []
    for s in seq:
        try:
            float(s)
        except ValueError:
            flags.append(False)
        else:
            flags.append(True)
    return flags


def fftfreq(n: int, d: float) -> np.ndarray:
    """fourier.py:248-269: monotonic frequency axis (the fft-shift is baked into the window)"""
    fnyq = 1 / (2 * np.float64(d))
    if n % 2 == 0:
        return np.linspace(-fnyq, fnyq - 2 * fnyq / n, n, dtype='float64')
    return np.linspace(-fnyq + fnyq / n, fnyq - fnyq / n, n, dtype='float64')


@functools.lru_cache(16)
def stft_axes(fs: float, nfft: int, time_size: int, overlap_frac: float):
    """fourier.py:348-357"""
    freqs = fftfreq(nfft, 1 / fs)
    times = np.arange(time_size) * ((1 - overlap_frac) * nfft / fs)
    return freqs, times


@functools.lru_cache()
def freq_band_edges(n: int, d: float, cutoff_low, cutoff_hi):
    """fourier.py:1184-1200.  The upper edge is the index of the LAST bin <= cutoff_hi used as an
    exclusive stop (the edge bin itself is dropped), as the reference does."""
    freqs = fftfreq(n, d)
    ilo = 0 if cutoff_low is None else int(np.where(freqs >= cutoff_low)[0][0])
    if cutoff_hi is None or cutoff_hi >= freqs[-1]:
        ihi = freqs.size
    else:
        ihi = int(np.where(freqs <= cutoff_hi)[0][-1])
    return ilo, ihi


# ---------------------------------------------------------------------------------------------
# windows
# ---------------------------------------------------------------------------------------------
def _enbw(window, n: int) -> float:
    from scipy import signal

    w = signal.windows.get_window(window, n, fftbins=True)
    w = w / np.sqrt(np.mean(np.abs(w) ** 2))
    return len(w) * np.sum(w ** 2) / np.sum(w) ** 2


@functools.lru_cache()
def find_window_param_from_enbw(window_name: str, enbw: float, *, nfft: int = 4096,
                                atol: float = 1e-6) -> float:
    """fourier.py:289-332: bisect the single window parameter that realises an ENBW (in bins)"""
    from scipy.optimize import bisect

    if enbw < 1 + 1 / nfft:
        raise ValueError('enbw must be greater than 1')
    if window_name == 'kaiser':
        a, b = np.pi * 1e-2, min(enbw ** 2, nfft // 2 - 1) * np.pi
    elif window_name == 'dpss':
        a, b = 1e-2, min(enbw ** 2, nfft // 2 - 1)
    elif window_name == 'chebwin':
        a, b = 45, 1000
    else:
        raise ValueError('window_name must be one of ("kaiser", "dpss", "chebwin")')
    return bisect(lambda p: _enbw((window_name, p), nfft) - enbw, a, b, xtol=atol)


@functools.lru_cache(1024)
def design_window(name_or_tuple, nwindow: int, nzero: int = 0, *, norm: bool = True) -> np.ndarray:
    """fourier.py:110-152 with fftshift=True, float32 result: scipy window (periodic, float64) ->
    trailing zeros -> unit mean square over the padded length -> (-1)^n -> float32"""
    from scipy import signal

    if isinstance(name_or_tuple, tuple):
        base, *suffix = name_or_tuple[0].rsplit('_by_enbw', 1)
        if suffix:
            param = find_window_param_from_enbw(base, name_or_tuple[1], nfft=nwindow)
            name_or_tuple = (base, param)
    w = signal.windows.get_window(name_or_tuple, nwindow, fftbins=True)
    ntotal = nwindow + nzero
    if ntotal % 2:
        raise NotImplementedError('odd frame length is not built (complex phase-ramp window)')
    if nzero:
        padded = np.zeros(ntotal, dtype=w.dtype)
        padded[:nwindow] = w
        w = padded
    if norm:
        w = w / np.sqrt(np.mean(np.abs(w) ** 2))
    sign = np.ones(ntotal)
    sign[1::2] = -1.0
    return (sign * w).astype(np.float32)


# ---------------------------------------------------------------------------------------------
# overlap-add filter planning (host side of fourier.py:652-723, 1108-1181)
# ---------------------------------------------------------------------------------------------
_COLA = {'hamming': (2, 1 / 2), 'blackman': (3, 2 / 3), 'blackmanharris': (5, 4 / 5)}   # divisor, overlap


def ola_overlap(array_size: int, window, nfft: int, nfft_out, extend: bool) -> tuple[int, int, float]:
    """(nfft_out, noverlap, overlap fraction) of ola_filter with the reference's checks, in the
    reference's order (fourier.py:656-691): window name, divisibility, whole hops in the input"""
    nfft_out = nfft if nfft_out is None else nfft_out
    if window in (None, 'rect'):
        raise ValueError('unexpected matching error')       # what the reference raises for them
    try:
        divisor, frac = _COLA[window]
    except (KeyError, TypeError):
        raise TypeError('ola_filter argument "window" must be one of ("hamming", "blackman", or "blackmanharris")')
    if nfft_out % divisor:
        raise ValueError(f'{window!r} window COLA requires output nfft_out % {divisor} == 0')
    noverlap = round(nfft_out * frac)
    if array_size % noverlap and not extend:
        raise ValueError(f'x.size ({array_size}) is not an integer multiple of noverlap ({noverlap})')
    return nfft_out, noverlap, frac


@functools.lru_cache()
def enbw_symmetric_f32(window, n: int) -> np.float32:
    """ENBW in bins of the SYMMETRIC window (fftbins=False), accumulated in float32 on the
    float32 unit-power window, which is what ola_filter adds to its passband edges
    (fourier.py:1146, 270-279)"""
    from scipy import signal

    w = signal.windows.get_window(window, n, fftbins=False)
    w = (w / np.sqrt(np.mean(np.abs(w) ** 2))).astype(np.float32)
    return len(w) * np.sum(w ** 2) / np.sum(w) ** 2


def ola_mask_bins(nfft: int, fs: float, n_frames: int, lo, hi) -> tuple[int, int]:
    """bins [ilo, ihi) that zero_stft_by_freq keeps (fourier.py:710-723).  The reference derives
    the sample spacing it hands to the band-edge search from the FRAME count times the bin
    spacing, so passbands in Hz select every bin; reproduced as is for drop-in behaviour."""
    freqs = fftfreq(nfft, 1.0 / fs)
    step = float(freqs[1] - freqs[0])
    return freq_band_edges(nfft, n_frames * step, lo, hi)


def downsample_copy_range(nfft_in: int, nfft_out: int, edge_lo, edge_hi) -> tuple[int, int]:
    """input bins kept when frames of nfft_in bins shrink to nfft_out (fourier.py:813-847): the
    nfft_out bins around the centre of [edge_lo, edge_hi) (the whole spectrum when both are None)"""
    edge_lo = 0 if edge_lo is None else edge_lo
    edge_hi = nfft_in if edge_hi is None else edge_hi
    width = min(edge_hi - edge_lo, nfft_out)
    first = (edge_hi + edge_lo) // 2 - width // 2
    return max(first, 0), min(first + width, nfft_in)


@functools.lru_cache(32)
def fir_lowpass_gain(size: int, sample_rate: float, cutoff: float, transition: float) -> np.ndarray:
    """complex64 per-bin gain of stft_fir_lowpass (fourier.py:766-826, window='rect'): the FFT of the
    firwin2 taps in the fft-shifted bin order of the STFT; designed on the host like the windows"""
    from scipy import signal

    if cutoff == float('inf'):
        taps = np.ones(size, dtype=np.complex64)
    else:
        taps = np.array(signal.firwin2(size, [0, cutoff, cutoff + transition, sample_rate / 2], [1.0, 1, 0.0, 0.0],
                                       window='rect', fs=sample_rate)).astype(np.complex64)
    sign = np.ones(size, dtype=np.float32)
    sign[1::2] = -1.0
    sign = sign.astype(np.complex64)
    return (np.fft.fft(taps * sign) * sign).astype(np.complex64)


@functools.lru_cache(64)
def bluestein_tables(window, nfft: int, nzero: int, norm, hop: int):
    """(pre, bh, post, m) of the chirp-z evaluation of an nfft-point DFT, nfft even and not a power of two
    (csrc/iqw_stft_bluestein.cu).  Designed in float64; n^2 is reduced mod 2*nfft as an integer so the
    chirp phase is exact for any length."""
    c = stft_coefficients(window, nfft, nzero, norm, hop).astype(np.float64)
    n = np.arange(nfft, dtype=np.int64)
    ph = (n * n) % (2 * nfft)
    chirp = np.exp(-1j * np.pi * ph / nfft)                 # exp(-i pi n^2 / N)
    m = 1 << int(2 * nfft - 2).bit_length()                 # power of two >= 2N - 1
    b = np.zeros(m, dtype=np.complex128)
    b[:nfft] = np.conj(chirp)
    b[m - nfft + 1:] = np.conj(chirp[1:][::-1])             # b[m - j] = b[j]
    bh = np.fft.fft(b) / m
    return ((c * chirp).astype(np.complex64), bh.astype(np.complex64), chirp.astype(np.complex64), m)


def window_key(window):
    """hashable form of a window argument"""
    if window is None:
        return 'rect'
    if isinstance(window, list):
        return tuple(window)
    return window


@functools.lru_cache(256)
def stft_coefficients(window, nfft: int, nzero: int, norm, hop: int) -> np.ndarray:
    """float32 coefficient multiplying each sample of a frame: fp32(fp32(w)/nfft)
    (fourier.py:1002-1010, 1019, 1033) and, for norm=None with overlap, / sum|.[::hop]|
    (fourier.py:571-580)."""
    w = design_window(window, nfft - nzero, nzero, norm=(norm == 'power'))
    c = w / nfft
    if hop != nfft and norm is None:
        c = c / np.abs(c[::hop]).sum()
    return np.ascontiguousarray(c, dtype=np.float32)


# ---------------------------------------------------------------------------------------------
# statistics
# ---------------------------------------------------------------------------------------------
_NAMED = {
    'min': _lib.STAT_MIN, 'max': _lib.STAT_MAX, 'peak': _lib.STAT_MAX,
    'mean': _lib.STAT_MEAN, 'rms': _lib.STAT_MEAN, 'median': _lib.STAT_MEDIAN,
}


def quantile_plan(n: int, q) -> tuple[int, int, float]:
    """(rank_lo, rank_hi, gamma) exactly as numpy 2.x 'linear' computes them for float32 data and
    a float32 q (numpy/lib/_function_base_impl.py:126-129, 4633-4654, 4765-4785): the virtual
    index (n-1)*q is evaluated in float32."""
    q32 = np.float32(q)
    if not (0.0 <= q32 <= 1.0):
        raise ValueError('Quantiles must be in the range [0, 1]')
    v = np.float32(n - 1) * q32
    if v >= np.float32(n - 1):
        return n - 1, n - 1, 0.0
    lo = int(np.floor(v))
    return lo, lo + 1, float(np.float32(v - np.float32(lo)))


def stat_requests(statistics, n_rows: int):
    """translate the reference's `statistics` list (power_analysis.py:73-101; floats, float-like
    strings, 'min'/'max'/'peak'/'mean'/'rms'/'median') into C requests, in caller order"""
    reqs = []
    for s, is_q in zip(statistics, find_float_inds(tuple(statistics))):
        r = _lib.iqw_stat()
        if is_q:
            lo, hi, g = quantile_plan(n_rows, float(s))
            r.kind, r.rank_lo, r.rank_hi, r.gamma = _lib.STAT_QUANTILE, lo, hi, g
        elif isinstance(s, str):
            if s not in _NAMED:
                raise ValueError(f'kind argument must be one of {_NAMED.keys()}')
            r.kind = _NAMED[s]
        elif callable(s):
            raise NotImplementedError('callable statistics are not built (arbitrary python)')
        else:
            raise ValueError(f'invalid statistic ufunc "{s}"')
        reqs.append(r)
    return reqs


def distinct_ranks(reqs, n_rows: int) -> set:
    ranks = set()
    for r in reqs:
        if r.kind == _lib.STAT_QUANTILE:
            ranks.update((r.rank_lo, r.rank_hi))
        elif r.kind == _lib.STAT_ORDER:
            ranks.add(r.rank_lo)
        elif r.kind == _lib.STAT_MEDIAN:
            ranks.update(((n_rows - 1) // 2, n_rows // 2))
    return ranks


def split_requests(reqs, n_rows: int):
    """group request indices so that each group needs <= MAX_RANKS_PER_CALL distinct ranks"""
    groups, cur, cur_ranks = [], [], set()
    for i, r in enumerate(reqs):
        ranks = distinct_ranks([r], n_rows)
        if cur and len(cur_ranks | ranks) > _lib.MAX_RANKS_PER_CALL:
            groups.append(cur)
            cur, cur_ranks = [], set()
        cur.append(i)
        cur_ranks |= ranks
    if cur:
        groups.append(cur)
    return groups


# polyphase table limit of iqw_upfirdn_c64: 16384 real or 8192 complex taps for any up
UPFIRDN_MAX_TABLE_FLOATS = 32768


def upfirdn_output_len(n_taps: int, n_in: int, up: int, down: int) -> int:
    """output length of scipy.signal.upfirdn (scipy's _output_len): the full convolution of the
    zero-stuffed input, (n_in - 1)*up + n_taps samples, kept every `down`-th, rounded up"""
    if n_in < 1:
        return 0
    return ((n_in - 1) * up + n_taps - 1) // down + 1


def upfirdn_polyphase(h: np.ndarray, up: int) -> np.ndarray:
    """polyphase table hp[p][j] = h[p + j*up], p < min(up, len(h)), j < ceil(len(h)/up), zero-padded.
    Rows p >= len(h) would be all zero and are left out (the kernel treats them as zero)."""
    L = h.shape[0]
    lp = -(-L // up)
    padded = np.zeros(lp * up, dtype=h.dtype)
    padded[:L] = h
    return np.ascontiguousarray(padded.reshape(lp, up).T[:min(up, L)])


def upfirdn_phase_index(n: np.ndarray, up: int, down: int) -> tuple[np.ndarray, np.ndarray]:
    """(p, i0) of global output indices n: y[n] = sum_j hp[p][j] * x[i0 - j]"""
    t = np.asarray(n, dtype=np.int64) * down
    return t % up, t // up


# filters longer than this would need nfft > 8192 (discard nfft/2 >= M - 1): not built
OACONVOLVE_MAX_TAPS = 4097


@functools.lru_cache(maxsize=None)
def oaconvolve_plan(n_taps: int) -> tuple[int, int]:
    """(nfft, discard) of the overlap-save blocks of iqw_oaconvolve_c64 for an M-tap filter: nfft a
    power of two in 16..8192, discard D = nfft/R with R in {2, 4, 8, 16} and D >= M - 1, hop = nfft - D.
    Minimises the transform work per output, log2(nfft) * nfft / hop (exactly: log2(nfft) * R / (R - 1));
    a tie goes to the smaller nfft."""
    from fractions import Fraction
    if not 1 <= n_taps <= OACONVOLVE_MAX_TAPS:
        raise ValueError(f'oaconvolve plan: need 1 <= n_taps <= {OACONVOLVE_MAX_TAPS} (got {n_taps})')
    best = None
    for log2n in range(4, 14):
        for r in (2, 4, 8, 16):
            nfft = 1 << log2n
            if nfft // r < n_taps - 1:
                continue
            cost = Fraction(log2n * r, r - 1)
            if best is None or cost < best[0]:
                best = (cost, nfft, nfft // r)
    return best[1], best[2]


def oaconvolve_window(mode: str, n1: int, n2: int) -> tuple[int, int]:
    """(first, length) of the output of scipy.signal.oaconvolve along the convolved axis, as a window
    of the full convolution (length n1 + n2 - 1); n1 is the length of in1 along that axis"""
    L = n1 + n2 - 1
    if mode == 'full':
        return 0, L
    if mode == 'same':
        return (L - n1) // 2, n1
    if mode == 'valid':
        return min(n1, n2) - 1, max(n1, n2) - min(n1, n2) + 1
    raise ValueError("acceptable mode flags are 'valid', 'same', or 'full'")


def oaconvolve_spectrum(h: np.ndarray, nfft: int) -> np.ndarray:
    """H = fft(h, nfft) / nfft along the last axis, computed in float64 and rounded once to complex64
    (the 1/nfft of the inverse transform is folded in)"""
    h = np.asarray(h)
    H = np.fft.fft(h.astype(np.complex128), nfft, axis=-1) / nfft
    return np.ascontiguousarray(H.astype(np.complex64))
