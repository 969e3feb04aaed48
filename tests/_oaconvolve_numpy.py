"""numpy reference of oaconvolve shared by the host tests: a complex64 emulation of the kernel's blocks."""
import numpy as np
import scipy.fft as sf


def emulate(x_buf, hspec, n_taps, nfft, discard, *, x_first, out_first, n_out):
    """the kernel's blocks in numpy complex64: block b reads global samples [b*hop - D, b*hop - D + nfft)
    of the buffer that holds [x_first, x_first + len(x_buf)) (zero elsewhere), forward FFT, times H,
    inverse as conj(FFT(conj(.))), keeps samples D.. as outputs [b*hop, b*hop + hop).  One block at a time,
    so that a block's bits cannot depend on what else is transformed with it.  Usable as `compute` of
    distributed.oaconvolve_time_sharded."""
    x_buf = np.asarray(x_buf)
    H = hspec[0]
    hop = nfft - discard
    y = np.zeros(n_out, np.complex64)
    if n_out == 0:
        return y
    for b in range(out_first // hop, (out_first + n_out - 1) // hop + 1):
        g0 = b * hop - discard - x_first
        blk = np.zeros(nfft, np.complex64)
        lo, hi = max(g0, 0), min(g0 + nfft, x_buf.size)
        if hi > lo:
            blk[lo - g0:hi - g0] = x_buf[lo:hi]
        kept = np.conj(sf.fft(np.conj(sf.fft(blk, workers=1) * H), workers=1))[discard:]
        n0 = b * hop - out_first
        a0, a1 = max(n0, 0), min(n0 + hop, n_out)
        y[a0:a1] = kept[a0 - n0:a1 - n0]
    return y
