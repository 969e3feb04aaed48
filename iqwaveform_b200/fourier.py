"""B200-native ``stft`` / ``spectrogram`` / ``persistence_spectrum`` with the reference signatures.

Mirrors /root/reference/src/iqwaveform/fourier.py:927-1057 (stft), 1203-1233 (spectrogram) and
1236-1327 (power_spectral_density == the north-star's persistence_spectrum).  The host side does
what the reference does on the host for every backend (parameter validation, window design, axis
arrays, band edges); all sample-rate work runs in the CUDA library behind include/iqw_b200.h.

Deliberate differences from what the reference *returns* (SURVEY.md section 0):
* quantile rows of ``power_spectral_density`` hold the values the reference computes and then
  loses (``fourier.py:1319-1320`` writes them into a temporary copy);
* overlapped ``stft`` works for any ``axis`` (the reference only for the last axis), and 1-D input
  to ``power_spectral_density`` works; the output layout is the one the reference produces
  wherever the reference works.
* ``spectrogram`` takes two additive keyword arguments, ``dB=`` and ``eps=``, fusing the
  ``powtodB(spectrogram(...))`` composition the reference's callers use (``figures.py:486``).
"""
from __future__ import annotations

import ctypes
import threading

import numpy as np
import torch

from . import _arrays, _lib, _plan
from .util import Domain, get_input_domain
from ._plan import INF

__all__ = ['GraphedCall', 'fft', 'ifft', 'zero_stft_by_freq', 'stft', 'istft', 'ola_filter', 'oaresample', 'upfirdn', 'oaconvolve', 'iq_to_stft_spectrogram', 'channelize_power', 'spectrogram', 'power_spectral_density', 'persistence_spectrum',
           'fftfreq', 'get_window', 'equivalent_noise_bandwidth']

fftfreq = _plan.fftfreq

_window_cache: dict = {}
_window_lock = threading.Lock()


def get_window(name_or_tuple, nwindow: int, nzero: int = 0, *, norm: bool = True,
               fftshift: bool = False) -> np.ndarray:
    """host window design (fourier.py:70-157), float32"""
    w = _plan.design_window(_plan.window_key(name_or_tuple), nwindow, nzero, norm=norm)
    if not fftshift:
        w = w.copy()
        w[1::2] *= -1.0
    return w


def equivalent_noise_bandwidth(window, N: int) -> float:
    """fourier.py:272-286: ENBW in bins"""
    return float(_plan._enbw(_plan.window_key(window), N))


def _device_window(window, nfft: int, nzero: int, norm, hop: int, device) -> torch.Tensor:
    key = (_plan.window_key(window), nfft, nzero, norm, hop, device.index)
    with _window_lock:
        w = _window_cache.get(key)
        if w is None:
            c = _plan.stft_coefficients(key[0], nfft, nzero, norm, hop)
            w = torch.from_numpy(c).to(device)
            _window_cache[key] = w
    return w


_bluestein_cache: dict = {}


def _device_bluestein(window, nfft: int, nzero: int, norm, hop: int, device):
    key = (_plan.window_key(window), nfft, nzero, norm, hop, device.index)
    with _window_lock:
        t = _bluestein_cache.get(key)
        if t is None:
            pre, bh, post, m = _plan.bluestein_tables(key[0], nfft, nzero, norm, hop)
            t = _bluestein_cache[key] = (torch.from_numpy(pre).to(device), torch.from_numpy(bh).to(device),
                                         torch.from_numpy(post).to(device), m)
    return t


BLUESTEIN_SCRATCH_BYTES = 1 << 30        # composed path: frames per pass so that the two scratch rows fit


def _stft_bluestein(x2, tables, nfft, hop, f0, nf, mode, eps, bin_lo, bin_hi, out, T, ranged):
    """frame lengths that are not a power of two (fourier.py:1250-1255 + 200-218): the chirp-z kernel
    inside one CTA up to nfft 4096, beyond that the same transform composed from three elementwise
    kernels around two calls of the large power-of-two FFT on a scratch of (frames, m) rows"""
    pre, bh, post, m = tables
    C, N = x2.shape
    nb = bin_hi - bin_lo
    esz = 8 if mode == _lib.STFT_COMPLEX else 4
    sp = _stream_ptr(x2.device)
    if m <= 8192:
        _lib.check(_lib.lib.iqw_stft_bluestein_c64(
            ctypes.c_void_p(x2.data_ptr() + f0 * hop * 8), C, (nf - 1) * hop + nfft if ranged else N,
            x2.stride(0) if C > 1 else N, ctypes.c_void_p(pre.data_ptr()), ctypes.c_void_p(bh.data_ptr()),
            ctypes.c_void_p(post.data_ptr()), nfft, m, hop, nf, mode, eps, bin_lo, bin_hi,
            ctypes.c_void_p(out.data_ptr() + f0 * nb * esz), T * nb, sp))
        return
    key = (m, x2.device.index)
    with _window_lock:
        ones = _ones_cache.get(key)
        if ones is None:
            ones = _ones_cache[key] = torch.ones(m, dtype=torch.float32, device=x2.device)
    chunk = max(1, BLUESTEIN_SCRATCH_BYTES // (2 * m * 8))
    a = torch.empty((min(chunk, nf), m), dtype=torch.complex64, device=x2.device)
    b = torch.empty_like(a)
    ws_bytes = _lib.lib.iqw_stft_workspace_bytes(m, 1, a.shape[0])
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x2.device) if ws_bytes else None

    def rows_fft(src, dst, k):
        _lib.check(_lib.lib.iqw_stft_c64(
            ctypes.c_void_p(src.data_ptr()), 1, k * m, k * m, ctypes.c_void_p(ones.data_ptr()), m, m, k,
            _lib.STFT_COMPLEX, 0.0, 0, m, ctypes.c_void_p(dst.data_ptr()), k * m,
            ctypes.c_void_p(ws.data_ptr()) if ws_bytes else None, ws_bytes, sp))

    for c in range(C):
        for g0 in range(f0, f0 + nf, chunk):
            k = min(chunk, f0 + nf - g0)
            _lib.check(_lib.lib.iqw_bluestein_pre_c64(
                ctypes.c_void_p(x2.data_ptr() + (c * x2.stride(0) + g0 * hop) * 8), hop, ctypes.c_void_p(pre.data_ptr()),
                nfft, m, k, ctypes.c_void_p(a.data_ptr()), sp))
            rows_fft(a, b, k)
            _lib.check(_lib.lib.iqw_bluestein_mul_c64(ctypes.c_void_p(b.data_ptr()), ctypes.c_void_p(bh.data_ptr()), m, k, sp))
            rows_fft(b, a, k)
            _lib.check(_lib.lib.iqw_bluestein_post_c64(
                ctypes.c_void_p(a.data_ptr()), ctypes.c_void_p(post.data_ptr()), m, k, mode, eps, bin_lo, bin_hi,
                ctypes.c_void_p(out.data_ptr() + ((c * T + g0) * nb) * esz), sp))


def _stream_ptr(device) -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _frame_count(n: int, nfft: int, noverlap: int, truncate: bool) -> int:
    if noverlap == 0:
        if n % nfft and not truncate:
            raise ValueError(f'axis 0 size {n} is not a factor of block size {nfft}')
        return n // nfft
    # overlap path: the partial tail frame is dropped whatever `truncate` says (fourier.py:568-569)
    if n < nfft:
        raise ValueError('window shape cannot be larger than input array shape')
    return (n - nfft) // (nfft - noverlap) + 1


def _host_checks(x, axis: int, nfft: int, noverlap: int, truncate: bool) -> None:
    """the reference's shape errors, raised before any byte moves to the device"""
    shape = getattr(x, 'shape', None)
    if shape is None:
        raise TypeError('unrecognized object type')
    ndim = len(shape)
    ax = axis + ndim if axis < 0 else axis
    if not 0 <= ax < ndim:
        raise ValueError(f'axis {axis} exceeds the number of dimensions')
    size = 1
    for d in shape:
        size *= d
    if size == 0:
        raise IndexError('cannot form blocks on arrays of size 0')
    if nfft < 1 or not 0 <= noverlap < nfft:
        raise ValueError('need 0 <= noverlap < nperseg')
    _frame_count(shape[ax], nfft, noverlap, truncate)


def _check_window_arg(window):
    if window is None or isinstance(window, str):
        return
    if isinstance(window, (tuple, list)) and len(window) and isinstance(window[0], str):
        return
    raise NotImplementedError(
        'array-valued windows are not built (they raise UnboundLocalError in the reference, '
        'fourier.py:1012)')


def _stft_device(x2: torch.Tensor, *, window, nfft: int, noverlap: int, nzero: int, norm,
                 truncate: bool, mode: int, eps: float = 0.0, bin_lo: int = 0, bin_hi=None,
                 out: torch.Tensor | None = None, frames: tuple | None = None) -> torch.Tensor:
    """(C, N) complex64 on the device -> (C, T, nbins).  `frames=(f0, f1)` computes only that frame
    range (C must be 1) into rows f0..f1 of `out`: used to transform a capture while it is still
    arriving from the host."""
    if x2.dtype != torch.complex64:
        raise NotImplementedError(f'only complex64 waveforms are built (got {x2.dtype})')
    if nfft < 1 or not 0 <= noverlap < nfft:
        raise ValueError('need 0 <= noverlap < nperseg')
    C, N = x2.shape
    if x2.numel() == 0:
        raise IndexError('cannot form blocks on arrays of size 0')
    hop = nfft - noverlap
    T = _frame_count(N, nfft, noverlap, truncate)
    bin_hi = nfft if bin_hi is None else bin_hi
    nb = bin_hi - bin_lo
    pow2 = nfft & (nfft - 1) == 0
    if pow2:
        _check_fft_size(nfft, 65536, 'stft')        # before anything is allocated
        w = _device_window(window, nfft, nzero, norm, hop, x2.device)
    else:
        if nfft % 2:
            raise NotImplementedError('odd frame lengths are not built (the reference multiplies them by a '
                                      'complex phase-ramp window, fourier.py:139-146)')
        if 2 * nfft - 1 > 65536:
            raise NotImplementedError(f'frame length {nfft}: lengths that are not a power of two are built up to 32768')
        tables = _device_bluestein(window, nfft, nzero, norm, hop, x2.device)
    dtype = torch.complex64 if mode == _lib.STFT_COMPLEX else torch.float32
    if out is None:
        out = torch.empty((C, T, nb), dtype=dtype, device=x2.device)
    elif out.shape != (C, T, nb) or out.dtype != dtype or not out.is_contiguous():
        raise ValueError(f'out must be a contiguous {dtype} tensor of shape {(C, T, nb)}')
    if T == 0 or C == 0:
        return out
    f0, f1 = (0, T) if frames is None else frames
    if frames is not None and (C != 1 or not 0 <= f0 <= f1 <= T):
        raise ValueError('frames=(f0, f1) needs a single channel and 0 <= f0 <= f1 <= T')
    if f1 == f0:
        return out
    nf = f1 - f0
    esz = 8 if mode == _lib.STFT_COMPLEX else 4
    if not pow2:
        _stft_bluestein(x2, tables, nfft, hop, f0, nf, mode, eps, bin_lo, bin_hi, out, T, frames is not None)
        return out
    ws_bytes = _lib.lib.iqw_stft_workspace_bytes(nfft, C, nf)     # > 0 only for nfft > 8192
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x2.device) if ws_bytes else None
    _lib.check(_lib.lib.iqw_stft_c64(
        ctypes.c_void_p(x2.data_ptr() + f0 * hop * 8), C, (nf - 1) * hop + nfft if frames is not None else N,
        x2.stride(0) if C > 1 else N,
        ctypes.c_void_p(w.data_ptr()), nfft, hop, nf, mode, eps, bin_lo, bin_hi,
        ctypes.c_void_p(out.data_ptr() + f0 * nb * esz), T * nb,
        ctypes.c_void_p(ws.data_ptr()) if ws_bytes else None, ws_bytes, _stream_ptr(x2.device)))
    return out


def stft(x, *, fs: float, window, nperseg: int = 256, noverlap: int = 0, nzero: int = 0,
         axis: int = 0, truncate: bool = True, norm: str | None = None, overwrite_x=False,
         return_axis_arrays=True, out=None):
    """short-time Fourier transform; same arguments and return value as the reference
    (fourier.py:927-1057).  Output index k is frequency index k - nfft/2 (no fftshift needed)."""
    if norm not in ('power', None):
        raise TypeError('norm must be "power" or None')
    _check_window_arg(window)
    _host_checks(x, axis, int(nperseg), int(noverlap), truncate)
    xd, res = _arrays.to_device(x)
    x2, lead, trail = _arrays.as_channels(xd, axis)
    y = _stft_device(x2, window=window, nfft=int(nperseg), noverlap=int(noverlap), nzero=int(nzero),
                     norm=norm, truncate=truncate, mode=_lib.STFT_COMPLEX,
                     out=out if (out is not None and not trail) else None)
    y = res.give_back(_arrays.restore_layout(y, lead, trail, 2))
    if not return_axis_arrays:
        return y
    ax = axis if axis >= 0 else axis + xd.ndim
    freqs, times = _plan.stft_axes(fs, int(nperseg), y.shape[ax], noverlap / nperseg)
    return freqs, times, y


def _istft_device(y3: torch.Tensor, nfft: int, noverlap: int, bin_lo: int = 0, bin_hi=None,
                  out: torch.Tensor | None = None, gain: torch.Tensor | None = None, scale: float = 1.0) -> torch.Tensor:
    """(C, T, bins) complex64 STFT on the device -> (C, T*hop + noverlap) complex64 waveform: band
    mask / zero padding, optional per-bin gain, inverse FFT, (-1)^n, overlap-add and a final scale in
    one kernel (csrc/iqw_istft.cu).  `bins` is nfft (whole frames; [bin_lo, bin_hi) is a read mask)
    or bin_hi - bin_lo (the frames hold only that band of an nfft-bin spectrum)."""
    if y3.dtype != torch.complex64:
        raise NotImplementedError(f'only complex64 STFTs are built (got {y3.dtype})')
    C, T, nb = y3.shape
    bin_hi = nfft if bin_hi is None else bin_hi
    if nb != nfft and nb != bin_hi - bin_lo:
        raise ValueError(f'the axis after the frame axis must hold nfft = {nfft} bins, got {nb}')
    hop = nfft - noverlap
    if hop < 1 or noverlap < 0:
        raise ValueError('need 0 <= noverlap < nfft')
    if nfft % hop:
        raise NotImplementedError(
            'istft: nfft must be a multiple of the hop (the reference adds groups of nfft // hop '
            'frames, fourier.py:628-647, which is not an overlap-add otherwise)')
    if T < 1 or C < 1:
        raise IndexError('cannot invert an STFT without frames')
    if not y3.is_contiguous():
        y3 = y3.contiguous()
    n_out = T * hop + noverlap
    if out is None:
        out = torch.empty((C, n_out), dtype=torch.complex64, device=y3.device)
    elif out.shape != (C, n_out) or out.dtype != torch.complex64 or not out.is_contiguous() or out.device != y3.device:
        raise ValueError(f'out must be a contiguous complex64 device tensor of shape {(C, n_out)}')
    if gain is not None and (gain.shape != (nfft,) or gain.dtype != torch.complex64 or not gain.is_contiguous()):
        raise ValueError('gain must be a contiguous complex64 vector of nfft bins')
    _lib.check(_lib.lib.iqw_istft_c64(
        ctypes.c_void_p(y3.data_ptr()), C, T, T * nb, nfft, hop, bin_lo, bin_hi, nb,
        ctypes.c_void_p(gain.data_ptr()) if gain is not None else None, float(scale),
        ctypes.c_void_p(out.data_ptr()), n_out, _stream_ptr(y3.device)))
    return out


_ones_cache: dict = {}


def _check_fft_size(n: int, largest: int, what: str) -> None:
    if n < 16 or n > largest or n & (n - 1):
        raise NotImplementedError(f'{what}: transform size {n}: powers of two from 16 to {largest} are built')


def fft(x, axis=-1, out=None, overwrite_x=False, plan=None, workers=None):
    """forward complex DFT along `axis`, unnormalised, natural bin order; same arguments as the
    reference (fourier.py:200-218, where it is scipy.fft.fft or cuFFT).  Runs kernel 1 with an
    all-ones window and hop = nfft, so every row of the batch is one "frame".  `plan` and `workers`
    are accepted and ignored (no FFT library is involved); `overwrite_x` is ignored (the kernel needs
    no scratch).  complex64, power-of-two sizes 16..65536."""
    xd, res = _arrays.to_device(x)
    x2, lead, trail = _arrays.as_channels(xd, axis)
    if x2.dtype != torch.complex64:
        raise NotImplementedError(f'only complex64 input is built (got {x2.dtype})')
    R, n = x2.shape
    _check_fft_size(n, 65536, 'fft')
    if x2.numel() == 0:
        raise IndexError('cannot transform arrays of size 0')
    if not x2.is_contiguous():
        x2 = x2.contiguous()
    key = (n, x2.device.index)
    with _window_lock:
        w = _ones_cache.get(key)
        if w is None:
            w = _ones_cache[key] = torch.ones(n, dtype=torch.float32, device=x2.device)
    direct = out is not None and not trail and isinstance(out, torch.Tensor) and out.is_cuda \
        and out.dtype == torch.complex64 and out.is_contiguous() and out.numel() == x2.numel()
    y = out.view(R, n) if direct else torch.empty((R, n), dtype=torch.complex64, device=x2.device)
    ws_bytes = _lib.lib.iqw_stft_workspace_bytes(n, 1, R)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x2.device) if ws_bytes else None
    _lib.check(_lib.lib.iqw_stft_c64(
        ctypes.c_void_p(x2.data_ptr()), 1, R * n, R * n, ctypes.c_void_p(w.data_ptr()), n, n, R,
        _lib.STFT_COMPLEX, 0.0, 0, n, ctypes.c_void_p(y.data_ptr()), R * n,
        ctypes.c_void_p(ws.data_ptr()) if ws_bytes else None, ws_bytes, _stream_ptr(x2.device)))
    if direct:
        return out
    y = res.give_back(_arrays.restore_layout(y, lead, trail, 1))
    if out is not None:         # any other `out` the reference would accept: filled by a copy
        out[...] = y if isinstance(out, torch.Tensor) else np.asarray(y)
        return out
    return y


def ifft(x, axis=-1, out=None, overwrite_x=False, plan=None, workers=None):
    """inverse complex DFT along `axis`, scaled by 1/n, natural order; same arguments as the reference
    (fourier.py:221-246).  Runs kernel 4 with hop = nfft and without the fft-shift sign
    (``iqw_ifft_c64``).  complex64, power-of-two sizes 16..8192."""
    xd, res = _arrays.to_device(x)
    x2, lead, trail = _arrays.as_channels(xd, axis)
    if x2.dtype != torch.complex64:
        raise NotImplementedError(f'only complex64 input is built (got {x2.dtype})')
    R, n = x2.shape
    _check_fft_size(n, 8192, 'ifft')
    if x2.numel() == 0:
        raise IndexError('cannot transform arrays of size 0')
    if not x2.is_contiguous():
        x2 = x2.contiguous()
    direct = out is not None and not trail and isinstance(out, torch.Tensor) and out.is_cuda \
        and out.dtype == torch.complex64 and out.is_contiguous() and out.numel() == x2.numel()
    y = out.view(R, n) if direct else torch.empty((R, n), dtype=torch.complex64, device=x2.device)
    _lib.check(_lib.lib.iqw_ifft_c64(ctypes.c_void_p(x2.data_ptr()), R, n, ctypes.c_void_p(y.data_ptr()),
                                     _stream_ptr(x2.device)))
    if direct:
        return out
    y = res.give_back(_arrays.restore_layout(y, lead, trail, 1))
    if out is not None:
        out[...] = y if isinstance(out, torch.Tensor) else np.asarray(y)
        return out
    return y


def zero_stft_by_freq(freqs, xstft, *, passband, axis=0):
    """band-pass in the STFT domain by zeroing bins IN PLACE; same arguments as the reference
    (fourier.py:707-720).  Device STFTs only (it is a memset of two bin ranges; inside `ola_filter`
    the same mask is a read predicate of kernel 4 and costs nothing).  `axis` is the frame axis, the
    bin axis follows it; like the reference, the bin spacing comes from `freqs` and the sample rate
    is taken as ``xstft.shape[axis] * freq_step``."""
    if not (isinstance(xstft, torch.Tensor) and xstft.is_cuda):
        raise TypeError('zero_stft_by_freq works in place on a device STFT (torch CUDA tensor)')
    freqs = np.asarray(freqs)
    freq_step = float(freqs[1] - freqs[0])
    fs = xstft.shape[axis] * freq_step
    if passband[0] is None or passband[1] is None:
        # the reference turns a None edge into slice(0, None) / slice(None, None) and clears the whole
        # STFT (fourier.py:717-718); reproduced, not repaired (ola_filter never gets here: its
        # passband arithmetic raises TypeError on None first)
        return xstft.zero_()
    ilo, ihi = _plan.freq_band_edges(freqs.size, fs, *passband)
    nb = xstft.shape[axis + 1]
    ilo, ihi = min(ilo, nb), min(ihi, nb)
    xstft.narrow(axis + 1, 0, ilo).zero_()
    xstft.narrow(axis + 1, ihi, nb - ihi).zero_()
    return xstft


def _trim_center(x: torch.Tensor, size, axis: int) -> torch.Tensor:
    """fourier.py:1098-1103: drop trim//2 samples at the start and the rest of the excess at the end"""
    if size is None:
        return x
    trim = x.shape[axis] - size
    if trim <= 0:
        return x
    return x.narrow(axis, trim // 2, size)


def istft(y, size=None, *, nfft: int, noverlap: int, out=None, overwrite_x=False, axis: int = 0):
    """reconstruct a waveform from its STFT; same arguments as the reference (fourier.py:1060-1105).
    ``axis`` is the frame axis of ``y`` and ``axis + 1`` its (fft-shifted) bin axis; the result has the
    waveform axis in their place.  Like the reference this is the plain overlap-add of the inverse
    transformed frames -- it inverts ``stft(..., norm=None)``, whose window carries the COLA scale."""
    yd, res = _arrays.to_device(y)
    if axis < 0:
        axis += yd.ndim
    if not 0 <= axis < yd.ndim - 1:
        raise ValueError('axis must address the frame axis, with the bin axis right after it')
    lead, trail = tuple(yd.shape[:axis]), tuple(yd.shape[axis + 2:])
    T, nb = yd.shape[axis], yd.shape[axis + 1]
    if trail:       # frames and bins last
        yd = yd.movedim((axis, axis + 1), (-2, -1))
    y3 = yd.reshape(-1, T, nb)
    x = _istft_device(y3, int(nfft), int(noverlap),
                      out=out if (out is not None and not trail and not lead) else None)
    x = _arrays.restore_layout(x, lead, trail, 1)
    return res.give_back(_trim_center(x, size, axis))


def ola_filter(x, *, fs: float, nfft: int, window='hamming', passband, nfft_out: int | None = None,
               frequency_shift=False, axis: int = 0, extend=False, out=None, overwrite_x=False,
               fused: bool = True):
    """band-pass filter by STFT overlap-and-add; same arguments as the reference
    (fourier.py:1108-1181): ``stft(norm=None, truncate=False)`` with a COLA window, the bins outside
    the passband zeroed, ``istft`` trimmed to the input size -- run as ONE kernel that never writes
    the STFT (``fused=False``, an additive argument, runs the stft and istft kernels one after the
    other instead; same result).  The resampling variants (``nfft_out != nfft``,
    ``frequency_shift``) are not built.
    NOTE the reference's passband arithmetic (fourier.py:714-715) works on a frequency axis scaled by
    the frame count, so passbands given in Hz keep every bin; this is reproduced, not repaired."""
    xd, res = _arrays.to_device(x)
    nfft = int(nfft)
    nfft_out, noverlap, frac = _plan.ola_overlap(xd.numel(), window, nfft, nfft_out, bool(extend))
    if nfft_out != nfft or frequency_shift:
        raise NotImplementedError('ola_filter: resampling (nfft_out != nfft, frequency_shift) is not built')
    enbw = _plan.enbw_symmetric_f32(window, nfft_out)
    lo, hi = passband[0] + enbw, passband[1] - enbw         # TypeError for None, as in the reference
    _host_checks(xd, axis, nfft, noverlap, False)
    x2, lead, trail = _arrays.as_channels(xd, axis)
    if x2.dtype != torch.complex64:
        raise NotImplementedError(f'only complex64 waveforms are built (got {x2.dtype})')
    C, N = x2.shape
    hop = nfft - noverlap
    T = _frame_count(N, nfft, noverlap, False)
    if T < 1:
        raise ValueError('the waveform is shorter than one frame')
    ilo, ihi = _plan.ola_mask_bins(nfft, fs, T, lo, hi)
    if fused:
        w = _device_window(window, nfft, 0, None, hop, x2.device)
        xf = torch.empty((C, T * hop + noverlap), dtype=torch.complex64, device=x2.device)
        _lib.check(_lib.lib.iqw_ola_filter_c64(
            ctypes.c_void_p(x2.data_ptr()), C, N, x2.stride(0) if C > 1 else N, ctypes.c_void_p(w.data_ptr()),
            nfft, hop, T, ilo, ihi, ctypes.c_void_p(xf.data_ptr()), xf.shape[1], _stream_ptr(x2.device)))
    else:
        y = _stft_device(x2, window=window, nfft=nfft, noverlap=noverlap, nzero=0, norm=None,
                         truncate=False, mode=_lib.STFT_COMPLEX)
        xf = _istft_device(y, nfft_out, noverlap, bin_lo=ilo, bin_hi=ihi)
    ax = axis if axis >= 0 else axis + xd.ndim
    xf = _arrays.restore_layout(xf, lead, trail, 1)
    return res.give_back(_trim_center(xf, round(xd.shape[ax] * nfft_out / nfft), ax))


def spectrogram(x, *, fs: float, window, nperseg: int = 256, noverlap: int = 0, nzero: int = 0,
                axis: int = 0, truncate: bool = True, return_axis_arrays: bool = True,
                dB: bool = False, eps: float = 0.0):
    """power spectrogram (fourier.py:1203-1233); with ``dB=True`` the fused
    ``10*log10(power + eps)`` of power_analysis.py:168-206"""
    _check_window_arg(window)
    xd, res = _arrays.to_device(x)
    x2, lead, trail = _arrays.as_channels(xd, axis)
    p = _stft_device(x2, window=window, nfft=int(nperseg), noverlap=int(noverlap), nzero=int(nzero),
                     norm='power', truncate=truncate,
                     mode=_lib.STFT_DB if dB else _lib.STFT_POWER, eps=float(eps))
    p = res.give_back(_arrays.restore_layout(p, lead, trail, 2))
    if not return_axis_arrays:
        return p
    ax = axis if axis >= 0 else axis + xd.ndim
    freqs, times = _plan.stft_axes(fs, int(nperseg), p.shape[ax], noverlap / nperseg)
    return freqs, times, p


def oaresample(x, up, down, fs, *, window='hamming', overwrite_x=False, axis=1, frequency_shift=0,
               filter_bandwidth=None, transition_bandwidth=250e3, scale: float = 1.0):
    """resample by up/down through STFT overlap-and-add; same arguments as the reference
    (fourier.py:1627-1725).  `down` and `up` are the frame lengths of the forward and the inverse
    transform.  Two kernels: the STFT writes only the bins that survive (downsampling: the `up` bins
    around the centre, or around `frequency_shift`), the inverse kernel zero-pads (upsampling),
    applies the optional frequency-domain FIR low-pass and the final x.size/size_in*scale factor."""
    xd, res = _arrays.to_device(x)
    nfft, nfft_in_out = int(down), int(up)
    nfft_out, noverlap, frac = _plan.ola_overlap(xd.numel(), window, nfft, nfft_in_out, True)
    if frequency_shift == 0:
        edge_lo = edge_hi = None
    elif down < up:
        raise ValueError('frequency_shift is only supported when downsampling')
    elif _plan.isroundmod(frequency_shift, fs / nfft):
        shift = round(frequency_shift / (fs / nfft))
        edge_lo = nfft // 2 - nfft_out // 2 + shift
        edge_hi = edge_lo + nfft_out
        if edge_lo < 0:
            raise ValueError('frequency_shift is too small')
        if edge_hi > nfft:
            raise ValueError('frequency_shift is too large')
    else:
        raise ValueError('frequency_shift must be a multiple of fs/up')
    nov_in = round(nfft * frac)
    _host_checks(xd, axis, nfft, nov_in, False)
    x2, lead, trail = _arrays.as_channels(xd, axis)
    if nfft_out < nfft:         # downsample: only the kept bins are computed into memory
        lo, hi = _plan.downsample_copy_range(nfft, nfft_out, edge_lo, edge_hi)
        y = _stft_device(x2, window=window, nfft=nfft, noverlap=nov_in, nzero=0, norm=None, truncate=False,
                         mode=_lib.STFT_COMPLEX, bin_lo=lo, bin_hi=hi)
        place_lo, place_hi = 0, hi - lo
        if place_hi != nfft_out:
            raise NotImplementedError('oaresample: a passband narrower than the output frame is not built')
    else:                       # upsample (or equal): the input spectrum sits in the middle of the output frame
        y = _stft_device(x2, window=window, nfft=nfft, noverlap=nov_in, nzero=0, norm=None, truncate=False,
                         mode=_lib.STFT_COMPLEX)
        place_lo = (nfft_out - nfft) // 2
        place_hi = place_lo + nfft
    gain = None
    if filter_bandwidth is not None and np.isfinite(filter_bandwidth):
        g = _plan.fir_lowpass_gain(nfft_out, float(fs * up / down), float(filter_bandwidth / 2), float(transition_bandwidth))
        gain = torch.from_numpy(g).to(x2.device)
    n_out = y.shape[1] * (nfft_out - noverlap) + noverlap
    factor = (x2.shape[0] * n_out) / xd.numel() * scale
    xr = _istft_device(y, nfft_out, noverlap, bin_lo=place_lo, bin_hi=place_hi, gain=gain,
                       scale=float(np.float32(factor)))
    return res.give_back(_arrays.restore_layout(xr, lead, trail, 1))


_UPFIRDN_MODES = ('constant', 'wrap', 'edge', 'smooth', 'symmetric', 'reflect', 'antisymmetric', 'antireflect',
                  'line')


def _upfirdn_taps(h, up: int, down: int, mode='constant', cval=0) -> tuple[np.ndarray, int]:
    """scipy.signal.upfirdn's argument checks (ValueError) and what is not built here
    (NotImplementedError), all on the host; returns (polyphase table float32 | complex64, len(h))"""
    if isinstance(h, torch.Tensor):
        h = h.detach().cpu().numpy()
    h = np.asarray(h)
    if h.ndim != 1 or h.size == 0:
        raise ValueError('h must be 1-D with non-zero length')
    if up < 1 or down < 1:
        raise ValueError('Both up and down must be >= 1')
    if mode not in _UPFIRDN_MODES:
        raise ValueError(f'Unknown mode: {mode!r}')
    if mode != 'constant' or cval != 0:
        raise NotImplementedError("upfirdn: only mode='constant' with cval=0 (zero padding) is built")
    h = h.astype(np.complex64 if np.iscomplexobj(h) else np.float32)
    table = _plan.upfirdn_polyphase(h, up)
    if table.size * (2 if table.dtype == np.complex64 else 1) > _plan.UPFIRDN_MAX_TABLE_FLOATS:
        raise NotImplementedError(f'upfirdn: a polyphase table of {table.shape[0]} x {table.shape[1]} taps exceeds '
                                  f'{_plan.UPFIRDN_MAX_TABLE_FLOATS} floats (16384 real or 8192 complex taps)')
    return table, h.size


def _upfirdn_device(x2: torch.Tensor, table: np.ndarray, n_taps: int, up: int, down: int, *, x_first: int = 0,
                    out_first: int = 0, n_out: int) -> torch.Tensor:
    """(C, N) complex64 device rows holding global samples [x_first, x_first + N) -> (C, n_out) outputs
    [out_first, out_first + n_out) of the whole capture.  The kernel reads unit-stride rows: any other
    layout (a column of an (N, C) capture, a strided view) is copied first."""
    C, N = x2.shape
    if x2.stride(1) != 1 or (C > 1 and x2.stride(0) < N):
        x2 = x2.contiguous()
    y = torch.empty((C, n_out), dtype=torch.complex64, device=x2.device)
    if n_out == 0 or C == 0:
        return y
    taps = torch.from_numpy(table).to(x2.device)
    _lib.check(_lib.lib.iqw_upfirdn_c64(
        ctypes.c_void_p(x2.data_ptr()), C, N, x2.stride(0) if C > 1 else N, x_first, ctypes.c_void_p(taps.data_ptr()),
        int(table.dtype == np.complex64), n_taps, up, down, out_first, n_out, ctypes.c_void_p(y.data_ptr()), n_out,
        _stream_ptr(x2.device)))
    return y


def upfirdn(h, x, up=1, down=1, axis=-1, mode='constant', cval=0):
    """upsample by `up` (zero stuffing), FIR-filter with `h` in full, downsample by `down`, along `axis`;
    the arguments and output length of scipy.signal.upfirdn, which the reference forwards host arrays to
    (fourier.py:1476-1495).  Polyphase: only the taps that meet a non-zero sample are applied.

    Differences from scipy: the arithmetic is float32.  `h` (1-D, real or complex, any float dtype) is
    rounded once to float32 / complex64, and the result is always complex64 -- scipy returns
    complex128 for float64 taps.  `x` must be complex64.  Only zero padding is built (mode='constant',
    cval=0; other modes raise NotImplementedError, unknown ones ValueError), as in the reference's GPU
    path, and the polyphase table is limited to 32768 floats: 16384 real or 8192 complex taps, for any
    `up`."""
    up, down = int(up), int(down)
    table, n_taps = _upfirdn_taps(h, up, down, mode, cval)
    dtype = getattr(x, 'dtype', None)
    if dtype not in (np.complex64, torch.complex64):
        raise NotImplementedError(f'upfirdn: only complex64 x is built (got {dtype})')
    xd, res = _arrays.to_device(x)
    x2, lead, trail = _arrays.as_channels(xd, axis)
    n_out = _plan.upfirdn_output_len(n_taps, x2.shape[1], up, down)
    y = _upfirdn_device(x2, table, n_taps, up, down, n_out=n_out)
    return res.give_back(_arrays.restore_layout(y, lead, trail, 1))


def _as_operand(a):
    """a torch tensor as it is (host or device); anything else as a numpy array (no copy of arrays)"""
    if isinstance(a, torch.Tensor):
        return a
    if hasattr(a, '__dlpack__') and not isinstance(a, np.ndarray):
        return torch.from_dlpack(a)
    return np.asarray(a)


def _conv_axes(axes, nd: int) -> list[int]:
    """scipy.fft's normalisation of `axes` (ValueError for out-of-range, repeated or empty axes)"""
    if axes is None:
        return list(range(nd))
    import operator
    ax = [operator.index(axes)] if np.ndim(axes) == 0 else [operator.index(a) for a in axes]
    if not ax:
        raise ValueError('when provided, axes cannot be empty')
    ax = [a + nd if a < 0 else a for a in ax]
    if any(a < 0 or a >= nd for a in ax):
        raise ValueError('axes exceeds dimensionality of input')
    if len(set(ax)) != len(ax):
        raise ValueError('all axes must be unique')
    return ax


def _oaconvolve_roles(s1: tuple, s2: tuple, mode: str, axes):
    """scipy.signal.oaconvolve's argument checks (ValueError) for non-empty operands of shapes s1, s2, and
    what is not built (NotImplementedError).  Returns (a, signal_is_in1, per_row): the one convolved axis,
    which operand is the signal (the longer along a; in1 on a tie) and whether the filter has one row per
    signal row (else one row for all)."""
    if mode not in ('full', 'same', 'valid'):
        raise ValueError("acceptable mode flags are 'valid', 'same', or 'full'")
    nd = len(s1)
    ax = _conv_axes(axes, nd)
    conv = [a for a in ax if s1[a] != 1 and s2[a] != 1]
    if not all(s1[a] == s2[a] or s1[a] == 1 or s2[a] == 1 for a in range(nd) if a not in conv):
        raise ValueError(f'incompatible shapes for in1 and in2: {s1} and {s2}')
    if mode == 'valid' and not (all(s1[a] >= s2[a] for a in conv) or all(s2[a] >= s1[a] for a in conv)):
        raise ValueError("For 'valid' mode, one must be at least as large as the other in every dimension")
    if len(conv) > 1:
        raise NotImplementedError(f'oaconvolve: convolution along more than one axis ({conv}) is not built')
    # no axis with both sizes > 1: an elementwise product, i.e. a 1-tap convolution along the longest axis
    a = conv[0] if conv else max(ax, key=lambda i: (max(s1[i], s2[i]), i))
    signal_is_in1 = s1[a] >= s2[a]
    xs, hs = (s1, s2) if signal_is_in1 else (s2, s1)
    others = [i for i in range(nd) if i != a]
    per_row = any(hs[i] != 1 for i in others)
    if per_row and any(hs[i] != xs[i] for i in others):
        raise NotImplementedError(f'oaconvolve: a filter of shape {hs} against a signal of shape {xs} (several filters '
                                  f'per signal row, or a broadcast signal) is not built; the filter must have size 1 '
                                  f'or the signal\'s size on every axis but {a}')
    if hs[a] > _plan.OACONVOLVE_MAX_TAPS:
        raise NotImplementedError(f'oaconvolve: both operands are longer than {_plan.OACONVOLVE_MAX_TAPS} samples '
                                  f'along axis {a} ({s1[a]} and {s2[a]}); filters of more taps are not built')
    return a, signal_is_in1, per_row


def _oaconvolve_device(x2: torch.Tensor, hspec: np.ndarray, n_taps: int, nfft: int, discard: int, *,
                       x_first: int = 0, out_first: int, n_out: int) -> torch.Tensor:
    """(C, N) complex64 device rows holding global samples [x_first, x_first + N) -> (C, n_out) outputs
    [out_first, out_first + n_out) of the full convolution.  `hspec`: (1 | C, nfft) complex64 spectrum rows
    (_plan.oaconvolve_spectrum).  The kernel reads unit-stride rows: any other layout is copied first."""
    C, N = x2.shape
    if x2.stride(1) != 1 or (C > 1 and x2.stride(0) < N):
        x2 = x2.contiguous()
    y = torch.empty((C, n_out), dtype=torch.complex64, device=x2.device)
    if n_out == 0 or C == 0:
        return y
    hd = torch.from_numpy(hspec).to(x2.device)
    _lib.check(_lib.lib.iqw_oaconvolve_c64(
        ctypes.c_void_p(x2.data_ptr()), C, N, x2.stride(0) if C > 1 else N, x_first, ctypes.c_void_p(hd.data_ptr()),
        nfft if hspec.shape[0] > 1 else 0, n_taps, nfft, discard, out_first, n_out, ctypes.c_void_p(y.data_ptr()),
        n_out, _stream_ptr(x2.device)))
    return y


def oaconvolve(in1, in2, mode='full', axes=None):
    """convolve `in1` with `in2` along one axis by FFT overlap-save; the arguments, output shapes and
    ValueErrors of scipy.signal.oaconvolve, which the reference forwards host arrays to
    (fourier.py:1496-1509).  Along the convolved axis the longer operand is the signal (in1 on a tie) and
    the other the filter, of M taps; the result comes back as the signal's kind (numpy, CPU or CUDA torch).

    Built: a complex64 signal; a filter of any numeric dtype, real or complex, on the host or the device,
    of at most 4097 taps; one convolved axis, with a filter of size 1 on every other axis (one filter for
    every row) or of the signal's size there (one filter per row).  Anything else raises
    NotImplementedError.  An empty operand gives an empty array of shape (0,).

    Differences from scipy: the filter's spectrum fft(h, nfft) / nfft is computed in float64 and rounded
    once to complex64, the device arithmetic is float32 and the result is always complex64 (scipy returns
    complex128 for float64 operands).  The error follows the energy of each FFT block rather than each
    output: |y - y_exact| stays within a small multiple of 2^-24 * log2(nfft) * max_k |fft(h, nfft)_k| *
    rms(x over the block's nfft input samples) (DESIGN.md section 7).

    Cost outside the kernel: every call computes the spectrum on the host (a filter on the device is copied
    to the host first) and copies it to the device synchronously, rows x nfft x 8 bytes (64 KB per row at
    nfft 8192).  Next to a long capture this is small; for many short calls with the same filter it is a
    host round trip per call."""
    in1, in2 = _as_operand(in1), _as_operand(in2)
    s1, s2 = tuple(in1.shape), tuple(in2.shape)
    if len(s1) != len(s2):
        raise ValueError('in1 and in2 should have the same dimensionality')
    if not s1:
        raise NotImplementedError('oaconvolve: 0-d operands are not built')
    if 0 in s1 or 0 in s2:
        if isinstance(in1, torch.Tensor):
            return torch.empty((0,), dtype=torch.complex64, device=in1.device)
        return np.empty((0,), np.complex64)
    a, signal_is_in1, per_row = _oaconvolve_roles(s1, s2, mode, axes)
    x, h = (in1, in2) if signal_is_in1 else (in2, in1)
    if x.dtype not in (np.complex64, torch.complex64):
        raise NotImplementedError(f'oaconvolve: only a complex64 signal is built (got {x.dtype})')
    if isinstance(h, torch.Tensor):
        h = h.detach().cpu().numpy()
    if not (np.issubdtype(h.dtype, np.number) or h.dtype == np.bool_):
        raise NotImplementedError(f'oaconvolve: a filter of dtype {h.dtype} is not built')
    n_taps = h.shape[a]
    first, n_out = _plan.oaconvolve_window(mode, s1[a], s2[a])
    nfft, discard = _plan.oaconvolve_plan(n_taps)
    hspec = _plan.oaconvolve_spectrum(np.moveaxis(h, a, -1).reshape(-1, n_taps), nfft)
    xd, res = _arrays.to_device(x)
    if mode == 'same' and not signal_is_in1:
        # scipy centres 'same' on in1's shape on every axis: where the (broadcast) filter in1 has size 1, the
        # one row kept is the middle one of the signal
        for i in range(xd.ndim):
            if i != a and s1[i] != xd.shape[i]:
                xd = xd.narrow(i, (xd.shape[i] - 1) // 2, 1)
    x2, lead, trail = _arrays.as_channels(xd, a)
    y = _oaconvolve_device(x2, hspec, n_taps, nfft, discard, out_first=first, n_out=n_out)
    return res.give_back(_arrays.restore_layout(y, lead, trail, 1))


def _python_slice(n: int, start: int, stop_from_end: int) -> tuple[int, int]:
    """bounds of range(n)[start:-stop_from_end] -- including python's [a:-0] == [a:0] (empty)"""
    lo, hi, _ = slice(start, -stop_from_end).indices(n)
    return lo, max(hi, lo)


def iq_to_stft_spectrogram(iq, window, nfft: int, Ts, overlap=True, analysis_bandwidth=None):
    """power spectrogram of a 1-D capture as a pandas DataFrame (index: frame times, columns:
    frequencies); same arguments as the reference (fourier.py:1421-1456).  The analysis-bandwidth
    trim is done by the STFT kernel (only the kept bins are computed into memory)."""
    import pandas as pd

    shape = getattr(iq, 'shape', None)
    if shape is None:
        raise TypeError('unrecognized object type')
    if len(shape) != 1:
        raise ValueError('iq_to_stft_spectrogram takes a 1-D waveform (a DataFrame is 2-D)')
    nfft = int(nfft)
    noverlap = nfft // 2 if overlap else 0
    _check_window_arg(window)
    _host_checks(iq, 0, nfft, noverlap, True)
    T = _frame_count(shape[0], nfft, noverlap, True)
    freqs, times = _plan.stft_axes(1.0 / Ts, nfft, T, noverlap / nfft)
    lo, hi = 0, nfft
    if analysis_bandwidth is not None:
        throwaway = nfft * (1 - analysis_bandwidth * Ts)
        if T > 1 and np.abs(throwaway - np.rint(throwaway)) > 1e-6:
            raise ValueError(f'analysis bandwidth yield integral number of samples, but got {throwaway}')
        lo, hi = _python_slice(nfft, int(np.floor(throwaway / 2)), int(np.ceil(throwaway // 2)))
    xd, _ = _arrays.to_device(iq)
    if hi > lo:
        p = _stft_device(xd.reshape(1, -1), window=window, nfft=nfft, noverlap=noverlap, nzero=0, norm='power',
                         truncate=True, mode=_lib.STFT_POWER, bin_lo=lo, bin_hi=hi)[0]
        values = _arrays.Residence('numpy').give_back(p)
    else:
        values = np.empty((T, 0), dtype=np.float32)
    return pd.DataFrame(values, columns=freqs[lo:hi], index=times)


def channelize_power(iq, Ts: float, fft_size_per_channel: int, *, analysis_bins_per_channel: int, window,
                     fft_overlap_per_channel=0, channel_count: int = 1, axis=0):
    """time series of the power in each of `channel_count` adjacent channels; the reference's
    arguments and return values (fourier.py:1330-1418).  The reference itself raises TypeError at its
    first statement (it forwards the window as ``w=``, which ``stft`` does not accept, fourier.py:1387-1390);
    this is the function with the window passed as ``window=``, everything else as written there --
    including ``X[:, s:-s]`` being EMPTY when no bins are skipped."""
    if axis != 0:
        raise NotImplementedError('sorry, only axis=0 implemented for now')
    if analysis_bins_per_channel > fft_size_per_channel:
        raise ValueError('the number of analysis bins cannot be greater than FFT size')
    shape = getattr(iq, 'shape', None)
    if shape is None:
        raise TypeError('unrecognized object type')
    if len(shape) != 1:
        raise NotImplementedError('channelize_power is built for 1-D captures')
    nfft = int(fft_size_per_channel * channel_count)
    noverlap = int(fft_overlap_per_channel * channel_count)
    _check_window_arg(window)
    _host_checks(iq, 0, nfft, noverlap, True)
    skip = channel_count * (fft_size_per_channel - analysis_bins_per_channel)
    if skip % 2 == 1:
        raise ValueError('must pass an even number of bins to skip')
    T = _frame_count(shape[0], nfft, noverlap, True)
    freqs, times = _plan.stft_axes(1.0 / Ts, nfft, T, noverlap / nfft)
    lo, hi = _python_slice(nfft, skip // 2, skip // 2)
    freqs = freqs[lo:hi]
    xd, res = _arrays.to_device(iq)
    nb = hi - lo
    if channel_count != 1 and nb == 0:
        raise IndexError('index 0 is out of bounds for axis 0 with size 0')     # freqs[0] of an empty band
    if channel_count != 1 and nb % analysis_bins_per_channel:
        raise ValueError(f'axis 0 size {nb} is not a factor of block size {analysis_bins_per_channel}')
    group = nb if channel_count == 1 else analysis_bins_per_channel
    n_groups = 1 if channel_count == 1 else (nb // group if group else 0)
    power = torch.zeros((T, n_groups), dtype=torch.float32, device=xd.device)
    if nb > 0 and T > 0:
        X = _stft_device(xd.reshape(1, -1), window=window, nfft=nfft, noverlap=noverlap, nzero=0, norm='power',
                         truncate=True, mode=_lib.STFT_COMPLEX, bin_lo=lo, bin_hi=hi)      # (1, T, nb)
        # sum of |X|^2 over each group of bins: kernel 3 on the flattened (T*nb) band, mean * size
        ws_bytes = _lib.lib.iqw_bin_power_workspace_bytes(1, group, T * n_groups)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=xd.device)
        _lib.check(_lib.lib.iqw_bin_power_c64(
            ctypes.c_void_p(X.data_ptr()), 1, T * nb, group, T * n_groups, ctypes.c_void_p(power.data_ptr()), None,
            None, ctypes.c_void_p(ws.data_ptr()), ws_bytes, _stream_ptr(xd.device)))
        power *= float(group)
    if channel_count == 1:
        return times, res.give_back(power[:, 0])
    return freqs[:analysis_bins_per_channel], times, res.give_back(power)


def time_statistics(p: torch.Tensor, statistics, *, dB: bool, eps: float = 1e-25,
                    out: torch.Tensor | None = None, counters: list | None = None,
                    requests: list | None = None) -> torch.Tensor:
    """statistics over axis 1 of a (C, T, nbins) float32 device tensor -> (C, nstat, nbins).
    The device-side part of fourier.py:1311-1325.  `requests` (prebuilt iqw_stat records) replaces
    `statistics` when the caller has done the rank arithmetic itself."""
    if p.dtype != torch.float32 or p.ndim != 3:
        raise ValueError('expected a (channels, frames, bins) float32 tensor')
    if not p.is_contiguous():
        p = p.contiguous()
    C, T, nb = p.shape
    if T < 1:
        raise ValueError('cannot take statistics over zero frames')
    reqs = list(requests) if requests is not None else _plan.stat_requests(list(statistics), T)
    if out is None:
        out = torch.empty((C, len(reqs), nb), dtype=torch.float32, device=p.device)
    ws_bytes = _lib.lib.iqw_time_stats_workspace_bytes(C, T, nb, len(reqs))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=p.device)
    groups = _plan.split_requests(reqs, T)
    for g in groups:
        arr = (_lib.iqw_stat * len(g))(*[reqs[i] for i in g])
        sub = out if len(groups) == 1 else torch.empty((C, len(g), nb), dtype=torch.float32,
                                                       device=p.device)
        _lib.check(_lib.lib.iqw_time_stats_f32(
            ctypes.c_void_p(p.data_ptr()), C, T, nb, T * nb, arr, len(g), int(bool(dB)), eps,
            ctypes.c_void_p(sub.data_ptr()), ctypes.c_void_p(ws.data_ptr()), ws_bytes,
            _stream_ptr(p.device)))
        if sub is not out:
            out[:, g, :] = sub
        if counters is not None:      # test aid: path counters of the last channel (synchronises)
            c16 = (ctypes.c_uint32 * 16)()
            _lib.check(_lib.lib.iqw_debug_time_stats_counters(ctypes.c_void_p(ws.data_ptr()), nb, c16))
            counters.append(dict(zip(('refine', 'collect', 'missed_ranks', 'overflowed', 'select_to_collect',
                                      'select_to_refine', 'inconsistent', 'selected', 'key_mode'), list(c16))))
    return out


def _psd_frame_plan(fs, resolution, fractional_overlap, fractional_window):
    """nfft, noverlap, nzero of a persistence spectrum and the reference's checks (fourier.py:1250-1262)"""
    if _plan.isroundmod(fs, resolution):
        nfft = round(fs / resolution)
        noverlap = round(fractional_overlap * nfft)
    else:
        raise ValueError('sample_rate_Hz/resolution must be a counting number')
    if _plan.isroundmod((1 - fractional_window) * nfft, 1):
        nzero = round((1 - fractional_window) * nfft)
    else:
        raise ValueError(
            '(1-fractional_window) * (sample_rate/frequency_resolution) must be a counting number')
    return nfft, noverlap, nzero


def power_spectral_density(x, *, fs: float, bandwidth=INF, window, resolution: float,
                           fractional_overlap=0, fractional_window: float = 1, statistics,
                           truncate=True, dB=True, axis=0):
    """persistence spectrum: per-bin statistics over time of the (dB) power spectrogram.
    Same arguments as the reference (fourier.py:1236-1327); returns (channels, nstat, nbins)
    float32 for (channels, time) input with axis=1, (nstat, nbins) for 1-D input."""
    nfft, noverlap, nzero = _psd_frame_plan(fs, resolution, fractional_overlap, fractional_window)
    statistics = list(statistics)
    _plan.stat_requests(statistics, 2)          # validates names before any device work
    domain = get_input_domain()
    if domain == Domain.FREQUENCY:
        return _psd_from_stft(x, fs=fs, nfft=nfft, bandwidth=bandwidth, statistics=statistics,
                              truncate=truncate, dB=dB, axis=axis)
    if domain != Domain.TIME:
        raise ValueError(f'unsupported persistence spectrum domain "{domain}"')
    _check_window_arg(window)
    _host_checks(x, axis, nfft, noverlap, True)

    bin_lo, bin_hi = 0, nfft
    if truncate and bandwidth != INF:
        bin_lo, bin_hi = _plan.freq_band_edges(nfft, 1.0 / fs, -bandwidth / 2, +bandwidth / 2)

    host = _host_rows(x, axis)
    if host is not None and host[0].numel() * 8 >= STREAM_MIN_BYTES:
        return _psd_from_host(*host, window=window, nfft=nfft, noverlap=noverlap, nzero=nzero,
                              bin_lo=bin_lo, bin_hi=bin_hi, statistics=statistics, dB=dB)

    xd, res = _arrays.to_device(x)
    x2, lead, trail = _arrays.as_channels(xd, axis)

    if _reducible(statistics, nfft) and x2.dtype == torch.complex64:
        # mean / max / min only: fused into kernel 1, no spectrogram in memory (8 B/sample of HBM traffic)
        out = _psd_reduce_device(x2, window=window, nfft=nfft, noverlap=noverlap, nzero=nzero, bin_lo=bin_lo,
                                 bin_hi=bin_hi, statistics=statistics, dB=dB)
        return res.give_back(_arrays.restore_layout(out, lead, trail, 2))

    C = x2.shape[0]
    dev = x2.device
    out = torch.empty((C, len(statistics), bin_hi - bin_lo), dtype=torch.float32, device=dev)
    T = _frame_count(x2.shape[1], nfft, noverlap, True)
    spg_bytes = T * (bin_hi - bin_lo) * 4

    def one_channel(c, scratch):
        p = _stft_device(x2[c:c + 1], window=window, nfft=nfft, noverlap=noverlap, nzero=nzero,
                         norm='power', truncate=True, mode=_lib.STFT_POWER, bin_lo=bin_lo,
                         bin_hi=bin_hi, out=scratch)
        time_statistics(p, statistics, dB=bool(dB), eps=1e-25, out=out[c:c + 1])
        return p

    # Several channels: the STFT -> statistics chains of consecutive channels run on two alternating
    # streams with a spectrogram buffer each, so that the tail of one channel's statistics (ALU /
    # issue bound, partly idle SMs) overlaps the next channel's STFT (FMA / shared-memory bound):
    # 3-4 % more throughput at config-3 size, bit-identical results.  Needs room for two spectrograms.
    if C >= 2 and spg_bytes >= PIPELINE_MIN_BYTES and torch.cuda.mem_get_info(dev)[0] > 2.5 * spg_bytes:
        main = torch.cuda.current_stream(dev)
        pair = _channel_streams.get(dev.index)
        if pair is None:
            pair = _channel_streams[dev.index] = (torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev))
        bufs = [torch.empty((1, T, bin_hi - bin_lo), dtype=torch.float32, device=dev) for _ in range(2)]
        for s in pair:
            s.wait_stream(main)
        for c in range(C):
            with torch.cuda.stream(pair[c % 2]):
                one_channel(c, bufs[c % 2])
        for s in pair:
            main.wait_stream(s)
    else:
        scratch = None
        for c in range(C):      # one channel's spectrogram in flight at a time (8 GB at config 3)
            scratch = one_channel(c, scratch)
    return res.give_back(_arrays.restore_layout(out, lead, trail, 2))


def _reducible(statistics, nfft: int) -> bool:
    """statistics that combine over time without the spectrogram (fourier.py:1322-1325 for 'max', 'min',
    'mean' and their aliases), at a frame size the fused kernel is built for"""
    if nfft < 16 or nfft > 8192 or nfft & (nfft - 1):
        return False
    kinds = {r.kind for r in _plan.stat_requests(list(statistics), 2)}
    return bool(kinds) and kinds <= {_lib.STAT_MEAN, _lib.STAT_MAX, _lib.STAT_MIN}


def _psd_reduce_device(x2: torch.Tensor, *, window, nfft, noverlap, nzero, bin_lo, bin_hi, statistics, dB,
                       frames: tuple | None = None, out: torch.Tensor | None = None) -> torch.Tensor:
    """(C, N) complex64 on the device -> (C, nstat, nbins) through iqw_stft_reduce_c64.  `frames=(f0, f1)`
    reduces only that frame range (C must be 1): the host path combines such partial results."""
    C, N = x2.shape
    hop = nfft - noverlap
    T = _frame_count(N, nfft, noverlap, True)
    if T < 1:
        raise ValueError('cannot take statistics over zero frames')
    f0, f1 = (0, T) if frames is None else frames
    reqs = _plan.stat_requests(list(statistics), f1 - f0)
    nb = bin_hi - bin_lo
    w = _device_window(window, nfft, nzero, 'power', hop, x2.device)
    if out is None:
        out = torch.empty((C, len(reqs), nb), dtype=torch.float32, device=x2.device)
    ws_bytes = _lib.lib.iqw_stft_reduce_workspace_bytes(nfft)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x2.device)
    arr = (_lib.iqw_stat * len(reqs))(*reqs)
    _lib.check(_lib.lib.iqw_stft_reduce_c64(
        ctypes.c_void_p(x2.data_ptr() + f0 * hop * 8), C, (f1 - f0 - 1) * hop + nfft if frames is not None else N,
        x2.stride(0) if C > 1 else N, ctypes.c_void_p(w.data_ptr()), nfft, hop, f1 - f0, int(bool(dB)), 1e-25,
        bin_lo, bin_hi, arr, len(reqs), ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(ws.data_ptr()), ws_bytes,
        _stream_ptr(x2.device)))
    return out


def _combine_reduced(parts: list, counts: list, statistics) -> torch.Tensor:
    """combine (nstat, nbins) results of consecutive frame ranges: max of max, min of min, frame-count
    weighted mean of means (in float64)"""
    kinds = [r.kind for r in _plan.stat_requests(list(statistics), 2)]
    stack = torch.stack(parts)                      # (n_parts, nstat, nbins)
    wts = torch.tensor(counts, dtype=torch.float64, device=stack.device)
    rows = []
    for i, k in enumerate(kinds):
        col = stack[:, i]
        if k == _lib.STAT_MAX:
            rows.append(col.amax(0))
        elif k == _lib.STAT_MIN:
            rows.append(col.amin(0))
        else:
            rows.append(((col.double() * wts[:, None]).sum(0) / wts.sum()).float())
    return torch.stack(rows)


PIPELINE_MIN_BYTES = 64 << 20    # spectrograms at least this large: two-stream pipeline over channels
_channel_streams: dict = {}
STREAM_MIN_BYTES = 64 << 20      # host captures at least this large are transformed while they arrive
STREAM_CHUNKS = 16
_copy_streams: dict = {}


def _host_rows(x, axis):
    """(rows tensor (C, N) on the host with contiguous rows, kind, squeeze) for a host capture whose
    time axis is the last one, else None"""
    if isinstance(x, np.ndarray):
        kind, t = 'numpy', (_arrays.from_numpy_readonly_ok(x) if x.dtype == np.complex64 else None)
    elif isinstance(x, torch.Tensor) and not x.is_cuda:
        kind, t = 'torch_cpu', (x if x.dtype == torch.complex64 else None)
    else:
        return None
    if t is None or t.ndim not in (1, 2):
        return None
    ax = axis + t.ndim if axis < 0 else axis
    if ax != t.ndim - 1 or t.stride(-1) != 1:
        return None
    return (t.reshape(1, -1) if t.ndim == 1 else t), kind, t.ndim == 1


def _psd_from_host(xh, kind, squeeze, *, window, nfft, noverlap, nzero, bin_lo, bin_hi, statistics, dB):
    """persistence spectrum of a HOST capture: the host->device copy runs in chunks on a copy stream
    and the STFT of the frames that are complete follows each chunk on the compute stream, so only the
    time statistics remain after the last byte has arrived (the copy is the bottleneck: 8 B/sample
    over PCIe).  Same kernels and frame arithmetic as the device path, hence identical results."""
    dev = _arrays._device()
    main = torch.cuda.current_stream(dev)
    cs = _copy_streams.get(dev.index)
    if cs is None:
        cs = _copy_streams[dev.index] = torch.cuda.Stream(device=dev)
    C, N = xh.shape
    hop = nfft - noverlap
    T = _frame_count(N, nfft, noverlap, True)
    nb = bin_hi - bin_lo
    out = torch.empty((C, len(statistics), nb), dtype=torch.float32, device=dev)
    spg = None if _reducible(statistics, nfft) else torch.empty((1, T, nb), dtype=torch.float32, device=dev)
    bufs = [torch.empty((1, N), dtype=torch.complex64, device=dev) for _ in range(min(C, 2))]
    for b in bufs:
        b.record_stream(cs)
    step = -(-N // STREAM_CHUNKS)
    step = max(nfft, -(-step // hop) * hop)
    freed = [None, None]                      # event after the last kernel that read bufs[i]
    fused = _reducible(statistics, nfft)      # mean / max / min only: each chunk is reduced as it lands
    for c in range(C):
        xd = bufs[c % 2]
        cs.wait_stream(main) if c == 0 else None
        if freed[c % 2] is not None:
            cs.wait_event(freed[c % 2])
        done = 0
        parts, counts = [], []
        for s0 in range(0, N, step):
            s1 = min(N, s0 + step)
            with torch.cuda.stream(cs):
                xd[0, s0:s1].copy_(xh[c, s0:s1], non_blocking=True)
                ev = cs.record_event()
            main.wait_event(ev)
            f1 = min(T, (s1 - nfft) // hop + 1) if s1 >= nfft else 0
            if f1 > done:
                if fused:
                    parts.append(_psd_reduce_device(xd, window=window, nfft=nfft, noverlap=noverlap, nzero=nzero,
                                                    bin_lo=bin_lo, bin_hi=bin_hi, statistics=statistics, dB=dB,
                                                    frames=(done, f1))[0])
                    counts.append(f1 - done)
                else:
                    _stft_device(xd, window=window, nfft=nfft, noverlap=noverlap, nzero=nzero, norm='power',
                                 truncate=True, mode=_lib.STFT_POWER, bin_lo=bin_lo, bin_hi=bin_hi, out=spg,
                                 frames=(done, f1))
                done = f1
        freed[c % 2] = main.record_event()
        if fused:
            out[c] = _combine_reduced(parts, counts, statistics)
        else:
            time_statistics(spg, statistics, dB=bool(dB), eps=1e-25, out=out[c:c + 1])
    res = _arrays.Residence(kind)
    return res.give_back(out[0] if squeeze else out)


def _psd_from_stft(X, *, fs, nfft, bandwidth, statistics, truncate, dB, axis):
    """``Domain.FREQUENCY`` branch (fourier.py:1277-1285, 1303-1307): X is an STFT (C, T, nfft),
    complex64, time on `axis` = 1.  dB is envtodB(X, eps=1e-25) = 20*log10(|X| + 1e-25), otherwise
    envtopow; then the statistics over time.  The band trim is applied to the result rows (the
    statistics of a bin do not depend on the other bins), so nothing is copied."""
    from .power_analysis import _elementwise
    shape = getattr(X, 'shape', None)
    if shape is None:
        raise TypeError('unrecognized object type')
    ax = axis + len(shape) if axis < 0 else axis
    if len(shape) != 3 or ax != 1 or shape[2] != nfft:
        raise ValueError(f'frequency-domain input must be (channels, frames, {nfft}) with the time axis 1')
    Xd, res = _arrays.to_device(X)
    if Xd.dtype != torch.complex64:
        raise NotImplementedError(f'only complex64 STFTs are built (got {Xd.dtype})')
    spg = _elementwise(Xd, _lib.EW_ENVTODB if dB else _lib.EW_ENVTOPOW, eps=1e-25 if dB else 0.0)
    out = time_statistics(spg, statistics, dB=False)
    if truncate and bandwidth != INF:
        ilo, ihi = _plan.freq_band_edges(nfft, 1.0 / fs, -bandwidth / 2, +bandwidth / 2)
        out = out[:, :, ilo:ihi].contiguous()
    return res.give_back(out)


persistence_spectrum = power_spectral_density


class GraphedCall:
    """a fixed-shape call of one of this module's device functions captured ONCE as a CUDA graph and
    replayed: for small problems (BASELINE configs[0]: 15 M samples, ~25 kernel launches of a few
    microseconds each) the launch latency of the individual kernels is most of the time.

        g = GraphedCall(persistence_spectrum, x, fs=..., window=..., resolution=..., statistics=...)
        y = g(x_next)         # x_next is copied into the captured input buffer, the graph is replayed

    The result tensor is reused by every replay (clone it to keep it).  Shapes, dtypes and keyword
    arguments are frozen at capture; results are bit-identical to the plain call (same kernels)."""

    def __init__(self, fn, x: torch.Tensor, **kw):
        if not (isinstance(x, torch.Tensor) and x.is_cuda):
            raise TypeError('GraphedCall captures device work: pass a CUDA tensor')
        self._x = x.clone()
        side = torch.cuda.Stream(device=x.device)
        side.wait_stream(torch.cuda.current_stream(x.device))
        with torch.cuda.stream(side):          # warm-up outside the capture: twiddle / window tables, allocator
            for _ in range(2):
                fn(self._x, **kw)
        torch.cuda.current_stream(x.device).wait_stream(side)
        torch.cuda.synchronize(x.device)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.out = fn(self._x, **kw)

    def __call__(self, x: torch.Tensor | None = None):
        if x is not None and x.data_ptr() != self._x.data_ptr():
            self._x.copy_(x)
        self.graph.replay()
        return self.out
