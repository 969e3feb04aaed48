"""numpy references of pfb_synthesize shared by the host and device tests: the definition and the factorisation
in float64, a complex64 emulation of the two kernels' arithmetic, the per-output error normaliser of the
documented bound, and the prototype pair of the reconstruction recipe."""
import numpy as np
import scipy.fft as sf
import scipy.signal as ss

from iqwaveform_b200 import _plan


def _phase(k, n, K):
    """exp(+2j pi k n / K) with k * n reduced mod K in integers"""
    return np.exp(2j * np.pi * (np.multiply.outer(k, n) % K) / K)


def direct64(y, g, hop):
    """the definition, frame by frame, in float64: xr[t] = sum_m sum_k g[t - m hop] y[m, k] W^-((k - K/2) t)"""
    y = np.asarray(y, np.complex128)
    g = np.asarray(g, np.float64)
    T, K = y.shape
    out = np.zeros(_plan.pfb_synth_len(T, g.size, hop), np.complex128)
    k = np.arange(K) - K // 2
    for m in range(T):
        n = m * hop + np.arange(g.size)
        out[n] += g * (y[m] @ _phase(k, n, K))
    return out


def _unrotate_idx(m, hop, K):
    return ((np.arange(K) - K // 2)[None, :] * ((np.asarray(m) * hop) % K)[:, None]) % K


def fact64(y, g, hop):
    """the kernels' factorisation in float64: unrotate, K * IFFT, unfold with the folded, sign-applied taps"""
    y = np.asarray(y, np.complex128)
    T, K = y.shape
    Lg = np.size(g)
    P = -(-Lg // K)
    gp = np.zeros(P * K)
    gp[:Lg] = np.asarray(g, np.float64)
    gs = gp.reshape(P, K) * np.where(np.arange(K) % 2, -1.0, 1.0)
    u = np.fft.ifft(y * np.exp(2j * np.pi * _unrotate_idx(np.arange(T), hop, K) / K), axis=1) * K
    out = np.zeros((T - 1) * hop + P * K, np.complex128)
    for m in range(T):
        out[m * hop:m * hop + P * K] += (gs * u[m][None, :]).ravel()
    return out[:_plan.pfb_synth_len(T, Lg, hop)]


def emulate(y_buf, taps, n_taps, hop, *, frame_first=0, n_frames_total, out_first, n_out):
    """the kernels' arithmetic in numpy for outputs [out_first, out_first + n_out) from a buffer holding global
    frames [frame_first, frame_first + len(y_buf)): complex64 unrotation by the complex64 W_K table, scipy's
    complex64 FFT between conjugates, and the unfold as one fused multiply-add per term and component (the
    product exact in float64, one rounding), frames in ascending order.  Usable as `compute` of
    distributed.pfb_synthesize_time_sharded."""
    y_buf = np.asarray(y_buf, np.complex64)
    K = taps.shape[1]
    gs = taps.ravel()
    acc = np.zeros(n_out, np.complex64)
    if n_out == 0:
        return acc
    m = frame_first + np.arange(y_buf.shape[0])
    W = np.exp(-2j * np.pi * np.arange(K) / K).astype(np.complex64)
    yc = (np.conj(y_buf) * W[_unrotate_idx(m, hop, K)]).astype(np.complex64)
    u = np.conj(sf.fft(yc, axis=1, workers=1)).astype(np.complex64)
    t = out_first + np.arange(n_out)
    m_hi = np.minimum(n_frames_total - 1, t // hop)
    m_lo = np.maximum(0, -((n_taps - 1 - t) // hop))              # ceil((t - Lg + 1) / hop)
    for d in range(-(-n_taps // hop) + 1):
        mm = m_lo + d
        ok = mm <= m_hi
        if not ok.any():
            break
        n = t[ok] - mm[ok] * hop
        term = gs[n].astype(np.float64) * u[mm[ok] - frame_first, n % K].astype(np.complex128)
        acc[ok] = (acc[ok].astype(np.complex128) + term).astype(np.complex64)
    return acc


def norm(y, taps, n_taps, hop):
    """2^-24 (log2 K + Q) S(t) per output, S(t) = sqrt(sum_m gs[t - m hop]^2 ||y_m||^2) in float64 of the float32
    taps and the complex64 frames, Q = ceil(Lg / hop)"""
    T, K = np.shape(y)
    e = np.sum(np.abs(np.asarray(y, np.complex128)) ** 2, axis=1)
    g2 = taps.ravel()[:n_taps].astype(np.float64) ** 2
    S2 = np.zeros(_plan.pfb_synth_len(T, n_taps, hop))
    for m in range(T):
        S2[m * hop:m * hop + n_taps] += g2 * e[m]
    return 2.0 ** -24 * (np.log2(K) + -(-n_taps // hop)) * np.sqrt(S2)


def recipe(K, L=None):
    """the 2x oversampled pair of the docstring: h = firwin(L, 1/K), g = firwin(L, 2/K) scaled by
    hop / (K sum g h), hop = K/2, L = 8K by default"""
    L = 8 * K if L is None else L
    h = ss.firwin(L, 1.0 / K, window=('kaiser', 9.0))
    g = ss.firwin(L, 2.0 / K, window=('kaiser', 9.0))
    return h, g * (K // 2) / (K * np.sum(g * h)), K // 2


def snr_db(x, xr, edge):
    """reconstruction SNR over the interior x[edge : len(x) - edge] (the edges get fewer terms)"""
    x = np.asarray(x, np.complex128)[edge:x.size - edge]
    e = np.asarray(xr, np.complex128)[edge:edge + x.size] - x
    return 10 * np.log10(np.sum(np.abs(x) ** 2) / np.sum(np.abs(e) ** 2))
