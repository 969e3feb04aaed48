"""oaconvolve host logic without a GPU: the overlap-save plan, scipy's output windows, the argument checks
that run before any device work, and a numpy complex64 emulation of the kernel's blocks -- against
scipy.signal.convolve in float64 within the documented bound, and run shard by shard with the time-shard
planner's spans, bitwise equal to one call."""
import numpy as np
import pytest
import scipy.fft as sf
import scipy.signal as ss
import torch

import iqwaveform_b200 as iqw
from iqwaveform_b200 import _plan
from iqwaveform_b200 import distributed as D

# the (nfft, nfft/discard) pairs csrc/iqw_oaconvolve.cu instantiates (oaconvolve_built)
BUILT = {(16, 4), (16, 8), (16, 16), (32, 4), (64, 4), (256, 8), (512, 8), (1024, 8), (2048, 8), (4096, 8),
         (8192, 2), (8192, 4), (8192, 8)}


def _emulate(x_buf, hspec, n_taps, nfft, discard, *, x_first, out_first, n_out):
    """the kernel's blocks in numpy complex64: block b reads global samples [b*hop - D, b*hop - D + nfft)
    of the buffer that holds [x_first, x_first + len(x_buf)) (zero elsewhere), forward FFT, times H,
    inverse as conj(FFT(conj(.))), keeps samples D.. as outputs [b*hop, b*hop + hop).  One block at a time,
    so that a block's bits cannot depend on what else is transformed with it."""
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


def _bound(x, h, mode, n1, n2, factor):
    """factor * 2^-24 * log2(nfft) * max_k |fft(h, nfft)_k| * rms(x over the nfft input samples of the
    output's block), per output of the window"""
    M = h.size
    nfft, discard = _plan.oaconvolve_plan(M)
    hop = nfft - discard
    first, n_out = _plan.oaconvolve_window(mode, n1, n2)
    p = np.concatenate([np.zeros(discard), np.abs(x.astype(np.complex128)) ** 2, np.zeros(nfft)])
    cs = np.concatenate([[0.0], np.cumsum(p)])
    b = (first + np.arange(n_out)) // hop
    rms = np.sqrt((cs[b * hop + nfft] - cs[b * hop]) / nfft)
    return factor * 2.0 ** -24 * np.log2(nfft) * np.abs(np.fft.fft(h.astype(np.complex128), nfft)).max() * rms


def _signal(rng, n):
    return (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)


def test_plan_rule():
    from fractions import Fraction
    for M in range(1, _plan.OACONVOLVE_MAX_TAPS + 1):
        nfft, d = _plan.oaconvolve_plan(M)
        assert d >= M - 1 and nfft % d == 0 and (nfft // d) in (2, 4, 8, 16) and 16 <= nfft <= 8192
        assert (nfft, nfft // d) in BUILT, (M, nfft, d)
        cost = Fraction(int(np.log2(nfft)) * nfft, nfft - d)
        for log2n in range(4, 14):
            for r in (2, 4, 8, 16):
                n2 = 1 << log2n
                if n2 // r >= M - 1:
                    c2 = Fraction(log2n * n2, n2 - n2 // r)
                    assert cost < c2 or (cost == c2 and nfft <= n2), (M, nfft, d, n2, r)
    assert _plan.oaconvolve_plan(161) == (2048, 256)
    assert _plan.oaconvolve_plan(4097) == (8192, 4096)
    for bad in (0, 4098):
        with pytest.raises(ValueError):
            _plan.oaconvolve_plan(bad)


SIZES = (1, 2, 5, 64, 100, 333)


@pytest.mark.parametrize('mode', ['full', 'same', 'valid'])
def test_window_is_scipy(mode):
    """scipy's output of every mode is the window [first, first + n) of its full convolution (integer
    operands: the direct sums are exact)"""
    rng = np.random.default_rng(2)
    for n1 in SIZES:
        for n2 in SIZES:
            a = rng.integers(-9, 9, n1).astype(np.float64)
            b = rng.integers(-9, 9, n2).astype(np.float64)
            full = ss.convolve(a, b, method='direct')
            want = ss.convolve(a, b, mode=mode, method='direct')
            first, n = _plan.oaconvolve_window(mode, n1, n2)
            assert ss.oaconvolve(a, b, mode=mode).shape == (n,)
            np.testing.assert_array_equal(full[first:first + n], want)
    with pytest.raises(ValueError):
        _plan.oaconvolve_window('bogus', 3, 4)


def test_spectrum_is_float64_rounded_once():
    h = np.random.default_rng(3).standard_normal((2, 33))
    H = _plan.oaconvolve_spectrum(h, 256)
    assert H.dtype == np.complex64 and H.shape == (2, 256) and H.flags.c_contiguous
    np.testing.assert_array_equal(H, (np.fft.fft(h, 256) / 256).astype(np.complex64))


def test_argument_errors_before_device_work():
    x = np.zeros(64, np.complex64)
    with pytest.raises(ValueError, match='dimensionality'):
        iqw.oaconvolve(x, np.ones((2, 3)))
    with pytest.raises(ValueError, match='acceptable mode'):
        iqw.oaconvolve(x, np.ones(3), mode='bogus')
    with pytest.raises(ValueError, match='incompatible shapes'):
        iqw.oaconvolve(np.zeros((3, 64), np.complex64), np.ones((2, 5)), axes=1)
    with pytest.raises(ValueError, match="'valid' mode"):
        iqw.oaconvolve(np.zeros((5, 3), np.complex64), np.ones((3, 5)), mode='valid')
    with pytest.raises(ValueError, match='exceeds'):
        iqw.oaconvolve(x, np.ones(3), axes=1)
    with pytest.raises(ValueError, match='unique'):
        iqw.oaconvolve(np.zeros((3, 64), np.complex64), np.ones((1, 3)), axes=[1, -1])
    with pytest.raises(ValueError, match='empty'):
        iqw.oaconvolve(x, np.ones(3), axes=[])
    # what is not built
    for bad in (np.zeros(64, np.complex128), np.zeros(64, np.float32), torch.zeros(64, dtype=torch.float32)):
        with pytest.raises(NotImplementedError, match='complex64'):
            iqw.oaconvolve(bad, np.ones(4))
    with pytest.raises(NotImplementedError, match='complex64'):
        iqw.oaconvolve(np.zeros(4, np.complex64), np.ones(100))   # the longer operand is the signal
    with pytest.raises(NotImplementedError, match='more than one axis'):
        iqw.oaconvolve(np.zeros((5, 64), np.complex64), np.ones((3, 4)))
    with pytest.raises(NotImplementedError, match='not built'):
        iqw.oaconvolve(np.zeros((1, 64), np.complex64), np.ones((3, 4)), axes=1)     # broadcast signal
    with pytest.raises(NotImplementedError, match='not built'):
        iqw.oaconvolve(np.zeros((2, 3, 64), np.complex64), np.ones((2, 1, 4)), axes=2)
    with pytest.raises(NotImplementedError, match='4097'):
        iqw.oaconvolve(np.zeros(5000, np.complex64), np.ones(4098))
    with pytest.raises(NotImplementedError, match='0-d'):
        iqw.oaconvolve(np.complex64(1), np.float32(2))
    # empty operands: an empty (0,) array, as scipy's
    for a, b in ((np.zeros(0, np.complex64), np.ones(3)), (x, np.ones(0)), (np.zeros((0, 4), np.complex64), np.ones((1, 2)))):
        got = iqw.oaconvolve(a, b)
        assert isinstance(got, np.ndarray) and got.shape == ss.oaconvolve(a, b).shape == (0,)


@pytest.mark.parametrize('M', [1, 2, 33, 129, 161, 1025, 4097])
@pytest.mark.parametrize('cplx', [False, True])
def test_emulation_within_bound_of_float64(M, cplx):
    rng = np.random.default_rng(M + cplx)
    h = rng.standard_normal(M) + (1j * rng.standard_normal(M) if cplx else 0)
    N = 30000
    x = _signal(rng, N)
    x[12000:12050] *= 1000                               # +60 dB burst
    nfft, discard = _plan.oaconvolve_plan(M)
    hspec = _plan.oaconvolve_spectrum(h[None], nfft)
    for mode in ('full', 'same', 'valid'):
        first, n = _plan.oaconvolve_window(mode, N, M)
        got = _emulate(x, hspec, M, nfft, discard, x_first=0, out_first=first, n_out=n)
        want = ss.convolve(x.astype(np.complex128), h, mode=mode)
        err = np.abs(got - want)
        # 3x: scipy's float32 FFT reaches 2.2 units on the 16-point blocks of a 2-tap filter, < 2 elsewhere
        assert np.all(err <= _bound(x, h, mode, N, M, 3)), float(np.max(err / _bound(x, h, mode, N, M, 1)))


@pytest.mark.parametrize('world', [1, 2, 3, 4, 5])
@pytest.mark.parametrize('mode', ['full', 'same', 'valid'])
def test_shards_are_bitwise_one_call(world, mode):
    """the shard planner's spans hold every in-range sample of each block: the emulation run shard by
    shard is bitwise the unsharded emulation (cases include shards shorter than one block)"""
    rng = np.random.default_rng(world)
    for N, M in [(20000, 161), (9000, 1025), (5000, 4097), (300, 33), (40, 5), (7, 2), (4097, 4097)]:
        h = rng.standard_normal(M)
        x = _signal(rng, N)
        nfft, discard = _plan.oaconvolve_plan(M)
        first, n = _plan.oaconvolve_window(mode, N, M)
        single = _emulate(x, _plan.oaconvolve_spectrum(h[None], nfft), M, nfft, discard, x_first=0,
                          out_first=first, n_out=n)
        group = D.ThreadGroup(world)
        outs, parts = [], []
        for r in range(world):
            sh = D.oaconvolve_shard(N, M, mode, world, r)
            assert sh.n_out == n and 0 <= sh.sample0 <= sh.sample1 <= N
            outs += list(range(sh.out0, sh.out1))
            parts.append(np.asarray(D.oaconvolve_time_sharded(x[sh.sample0:sh.sample1], h, mode, n_samples=N,
                                                              group=group.member(r), compute=_emulate)))
        assert outs == list(range(n))
        assert np.array_equal(np.concatenate(parts), single), (N, M)


def test_shard_halo_is_the_discard():
    nfft, discard = _plan.oaconvolve_plan(161)
    hop = nfft - discard
    sh = D.oaconvolve_shard(100000, 161, 'full', 2, 1)
    assert sh.sample0 == sh.out0 // hop * hop - discard
    assert sh.sample1 == 100000


def test_shard_rejects_a_wrong_halo_and_a_short_capture():
    sh = D.oaconvolve_shard(1000, 33, 'full', 2, 1)
    x = np.zeros(sh.sample1 - sh.sample0 + 1, np.complex64)
    with pytest.raises(ValueError, match='expects a 1-D shard'):
        D.oaconvolve_time_sharded(x, np.ones(33), n_samples=1000, group=D.ThreadGroup(2).member(1), compute=_emulate)
    with pytest.raises(NotImplementedError):
        D.oaconvolve_shard(10, 33, 'full', 2, 0)
