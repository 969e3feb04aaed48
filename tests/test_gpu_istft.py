"""kernel 4 (fused band mask -> inverse FFT -> overlap-add) through the C-ABI and the reference's
`istft` / `ola_filter` signatures, against the numpy oracle and the committed reference outputs."""
import numpy as np
import pytest
import torch

import _tol
from conftest import load_golden
import iqwaveform_b200 as iqw
from oracle import iqw_oracle as orc
from oracle.make_golden import synth

pytestmark = pytest.mark.gpu


def _check(got, want):
    got = np.asarray(got)
    assert got.shape == want.shape and got.dtype == np.complex64
    tol = _tol.waveform_tol(np.moveaxis(want, -1, -1))
    assert np.all(np.abs(got - want) <= tol), float(np.max(np.abs(got - want) / tol))


@pytest.mark.parametrize('name', ['istft_hamming_256_128', 'istft_bh_1024_768', 'istft_rect_64_0'])
def test_istft_golden(name):
    p, a = load_golden(name)
    x = iqw.istft(a['y'], p['size'], nfft=p['nperseg'], noverlap=p['noverlap'], axis=p['axis'])
    _check(x, a['x'])


@pytest.mark.parametrize('name', ['ola_hamming_512_all', 'ola_hamming_512_band'])
def test_ola_filter_golden(name):
    p, a = load_golden(name)
    p['passband'] = tuple(p['passband'])
    _check(iqw.ola_filter(a['x'], **p), a['out'])


@pytest.mark.parametrize('nfft', [16, 32, 64, 128, 256, 512, 1024, 2048, 4096, 8192])
@pytest.mark.parametrize('R', [1, 2, 4, 8, 16])
def test_istft_matches_oracle(nfft, R):
    hop = nfft // R
    T = 37
    x = synth(nfft + R, (2, (T - 1) * hop + nfft))
    y = orc.stft(x, fs=1e6, window='hamming', nperseg=nfft, noverlap=nfft - hop, axis=1, truncate=False,
                 return_axis_arrays=False)
    if R > (8 if nfft in (32, 64) else 16):
        # nfft/hop larger than the values a thread holds: the library refuses the geometry
        with pytest.raises(NotImplementedError):
            iqw.istft(torch.from_numpy(y).cuda(), nfft=nfft, noverlap=nfft - hop, axis=1)
        return
    want = orc.istft(y.copy(), None, nfft=nfft, noverlap=nfft - hop, axis=1)
    got = iqw.istft(torch.from_numpy(y).cuda(), nfft=nfft, noverlap=nfft - hop, axis=1)
    _check(got.cpu().numpy(), want)


@pytest.mark.parametrize('shape,axis', [((5000,), 0), ((3, 4096), 1), ((2, 3, 2048), 2), ((2, 2048, 3), 1), ((1536, 2), 0)])
def test_istft_layouts_and_trim(shape, axis):
    """any frame axis, leading and trailing axes, numpy in -> numpy out, centre trim"""
    nfft, nov = 128, 64
    x = synth(7, shape[:axis] + shape[axis + 1:] + (shape[axis],))
    x = np.moveaxis(x, -1, axis)
    # the oracle's stft needs the time axis last
    y = np.moveaxis(orc.stft(np.moveaxis(x, axis, -1), fs=1e6, window='hamming', nperseg=nfft, noverlap=nov,
                             axis=x.ndim - 1, truncate=False, return_axis_arrays=False), (-2, -1), (axis, axis + 1))
    for size in (None, x.shape[axis], x.shape[axis] - 37, 10 ** 9):
        want = orc.istft(y.copy(), size, nfft=nfft, noverlap=nov, axis=axis)
        got = iqw.istft(y.copy(), size, nfft=nfft, noverlap=nov, axis=axis)
        assert isinstance(got, np.ndarray) and got.shape == want.shape
        tol = _tol.waveform_tol(np.moveaxis(want, axis, -1))
        assert np.all(np.abs(np.moveaxis(got, axis, -1) - np.moveaxis(want, axis, -1)) <= tol)


def test_istft_many_frames_and_ranges():
    """more frames than one range per slot: every range boundary must be seamless"""
    nfft, nov = 64, 48
    x = synth(3, (3, 400000))
    y = orc.stft(x, fs=1e6, window='hamming', nperseg=nfft, noverlap=nov, axis=1, truncate=False,
                 return_axis_arrays=False)
    want = orc.istft(y.copy(), x.shape[1], nfft=nfft, noverlap=nov, axis=1)
    got = iqw.istft(torch.from_numpy(y).cuda(), x.shape[1], nfft=nfft, noverlap=nov, axis=1)
    _check(got.cpu().numpy(), want)


def test_stft_istft_round_trip_is_the_identity():
    """COLA window + norm=None: the overlap-add of the inverse frames returns the capture (away from
    the first and last noverlap samples, where fewer frames overlap); full path on the device"""
    n = 1 << 24
    g = torch.Generator('cuda').manual_seed(5)
    x = torch.randn(n, dtype=torch.complex64, device='cuda', generator=g)
    for nfft, nov in [(4096, 2048), (1024, 512), (256, 128)]:
        y = iqw.stft(x, fs=1e6, window='hamming', nperseg=nfft, noverlap=nov, truncate=False, return_axis_arrays=False)
        xr = iqw.istft(y, n, nfft=nfft, noverlap=nov)
        assert xr.shape == x.shape
        err = (xr[nov:-nov] - x[nov:-nov]).abs().max().item()
        assert err < 2e-6 * x.abs().max().item(), err


@pytest.mark.parametrize('passband', [(-2e5, 2e5), (-1.3647444248199463 - 2e-6, 1.3647444248199463 + 1e-6)])
@pytest.mark.parametrize('shape,axis', [((8192,), 0), ((3, 4096), 1)])
def test_ola_filter_matches_oracle(passband, shape, axis):
    x = synth(10, shape)
    kw = dict(fs=1e6, nfft=512, window='hamming', passband=passband, axis=axis)
    _check(iqw.ola_filter(x.copy(), **kw), orc.ola_filter(x.copy(), **kw))


@pytest.mark.parametrize('nfft', [16, 64, 256, 1024, 2048, 4096, 8192])
def test_fused_ola_filter_equals_the_two_kernel_chain(nfft):
    """one kernel (no STFT in memory) against stft -> masked istft.  With the forward transform of the
    chain on the three-pass geometry the fused kernel shares (variant 1) it is the same arithmetic, bit
    for bit; with the default forward kernel (two-pass at nfft 1024..4096) the two differ by float32
    rounding only (waveform tolerance of tests/_tol.py)."""
    from iqwaveform_b200 import _lib
    x = torch.from_numpy(synth(nfft, (3, nfft * 40))).cuda()
    e = float(orc.enbw_symmetric('hamming', nfft))
    try:
        _lib.check(_lib.lib.iqw_debug_set_stft_variant(1))
        for pb in [(-2e5, 2e5), (-e - 2e-6 * 512 / nfft, e + 1e-6 * 512 / nfft)]:
            kw = dict(fs=1e6, nfft=nfft, window='hamming', passband=pb, axis=1)
            a = iqw.ola_filter(x, **kw)
            b = iqw.ola_filter(x, fused=False, **kw)
            assert torch.equal(a, b)
        # a long capture: many frame ranges per channel
        xl = torch.from_numpy(synth(1, (2, nfft * 3000 if nfft <= 256 else nfft * 300))).cuda()
        kw = dict(fs=1e6, nfft=nfft, window='hamming', passband=(-1e5, 1e5), axis=1)
        fused = iqw.ola_filter(xl, **kw)
        assert torch.equal(fused, iqw.ola_filter(xl, fused=False, **kw))
    finally:
        _lib.check(_lib.lib.iqw_debug_set_stft_variant(0))
    chain = iqw.ola_filter(xl, fused=False, **kw).cpu().numpy()
    assert np.all(np.abs(chain - fused.cpu().numpy()) <= _tol.waveform_tol(fused.cpu().numpy()))


def test_errors_follow_the_reference():
    x = synth(10, (8192,))
    kw = dict(fs=1e6, nfft=512, window='hamming', passband=(-1e5, 1e5))
    for bad, exc in [(dict(window='hann'), TypeError), (dict(window='blackman'), ValueError),
                     (dict(nfft=100), ValueError), (dict(passband=(None, 1e5)), TypeError),
                     (dict(nfft_out=256), NotImplementedError)]:
        with pytest.raises(exc):
            iqw.ola_filter(x, **dict(kw, **bad))
    y = np.zeros((4, 256), np.complex64)
    with pytest.raises(NotImplementedError):
        iqw.istft(y, nfft=256, noverlap=100)          # hop does not divide nfft
    with pytest.raises(ValueError):
        iqw.istft(y, nfft=128, noverlap=64)           # bin axis is not nfft long
    with pytest.raises(NotImplementedError):
        iqw.istft(np.zeros((4, 256), np.complex128), nfft=256, noverlap=128)


@pytest.mark.parametrize('name', ['oares_down_1024_512', 'oares_up_512_1024_fir', 'oares_shift_1024_256'])
def test_oaresample_golden(name):
    p, a = load_golden(name)
    _check(iqw.oaresample(a['x'], **p), a['out'])


@pytest.mark.parametrize('shape,axis', [((2, 16384), 1), ((16384,), 0), ((32768, 2), 0)])
@pytest.mark.parametrize('kw', [dict(up=512, down=1024), dict(up=1024, down=512), dict(up=1024, down=1024),
                                dict(up=256, down=1024, frequency_shift=1e6 / 1024 * 100),
                                dict(up=512, down=1024, filter_bandwidth=0.3e6, transition_bandwidth=50e3),
                                dict(up=2048, down=1024, filter_bandwidth=0.6e6, scale=0.5),
                                dict(up=8192, down=64), dict(up=32, down=4096)])
def test_oaresample_matches_oracle(shape, axis, kw):
    x = synth(14, shape[:axis] + shape[axis + 1:] + (shape[axis],))
    want = orc.oaresample(x.copy(), fs=1e6, axis=x.ndim - 1, window='hamming', **kw)
    got = iqw.oaresample(np.moveaxis(x, -1, axis).copy(), fs=1e6, axis=axis, window='hamming', **kw)
    _check(np.moveaxis(got, axis, -1), want)


def test_oaresample_errors_and_device_path():
    x = synth(14, (2, 16384))
    for bad, exc in [(dict(up=768, down=1024), NotImplementedError), (dict(up=1024, down=512, frequency_shift=1e3), ValueError),
                     (dict(up=512, down=1024, frequency_shift=123.0), ValueError),
                     (dict(up=256, down=1024, frequency_shift=0.45e6), ValueError), (dict(up=511, down=1024), ValueError)]:
        with pytest.raises(exc):
            iqw.oaresample(x, fs=1e6, axis=1, window='hamming', **bad)
    with pytest.raises(TypeError):
        iqw.oaresample(x, 512, 1024, 1e6, window='hann')
    xd = torch.from_numpy(x).cuda()
    a = iqw.oaresample(xd, 512, 1024, 1e6)
    assert a.is_cuda and a.shape == (2, 8192)
    # sanity, not parity: a 2:1 decimation keeps a slow tone (the cropped-spectrum overlap-add is only
    # approximately shift-invariant, hence the per-cent level bound)
    n = np.arange(1 << 16)
    tone = np.exp(2j * np.pi * 0.01 * n).astype(np.complex64)
    d = iqw.oaresample(tone, 512, 1024, 1e6, axis=0)
    assert d.shape == (1 << 15,)
    want = np.exp(2j * np.pi * 0.02 * np.arange(1 << 15))
    assert np.max(np.abs(d[2048:-2048] - want[2048:-2048])) < 5e-2
