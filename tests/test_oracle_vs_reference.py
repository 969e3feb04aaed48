"""the numpy oracle against the unmodified reference, bit-for-bit: against the live reference where it is installed,
else against the digests recorded from these comparisons (tests/_reference_digests.py)."""
import numpy as np
import pytest

from _reference_digests import RECORD, recorded, recorded_cpu_count
from oracle import iqw_oracle as orc
from oracle import ref_shim
from oracle.make_golden import synth

ref = ref_shim.load()


@pytest.fixture(autouse=True)
def _recorded_fft_threads(monkeypatch):
    """against the recorded digests, the oracle's FFTs run on as many threads as when the digests were recorded"""
    if ref is None and not RECORD:
        monkeypatch.setattr(orc, 'CPU_COUNT', recorded_cpu_count())


@pytest.mark.parametrize('window', ['hann', 'blackmanharris', ('kaiser', 8.0), 'rect', 'hamming'])
@pytest.mark.parametrize('nfft,noverlap', [(1024, 512), (256, 192), (2048, 0), (64, 48), (100, 50)])
@pytest.mark.parametrize('norm', ['power', None])
def test_stft(window, nfft, noverlap, norm):
    x = synth(1, (2, 20011))
    f2, t2, y2 = orc.stft(x.copy(), fs=1e6, window=window, nperseg=nfft, noverlap=noverlap,
                          axis=1, norm=norm)
    if recorded(ref, f2, t2, y2):
        return
    f, t, y = ref.fourier.stft(x.copy(), fs=1e6, window=window, nperseg=nfft, noverlap=noverlap,
                               axis=1, norm=norm)
    assert np.array_equal(f, f2) and np.array_equal(t, t2)
    assert np.array_equal(y.view(np.float32), y2.view(np.float32))


def test_spectrogram_nzero_1d():
    x = synth(2, (30000,))
    _, _, p2 = orc.spectrogram(x.copy(), fs=1e6, window='hann', nperseg=512, noverlap=256,
                               nzero=128, axis=0)
    if recorded(ref, p2):
        return
    _, _, p = ref.fourier.spectrogram(x.copy(), fs=1e6, window='hann', nperseg=512, noverlap=256,
                                      nzero=128, axis=0)
    assert np.array_equal(p, p2)


@pytest.mark.parametrize('dB', [True, False])
def test_persistence(dB):
    x = synth(3, (2, 1 << 16))
    stats = [0.1, 'mean', 0.5, 'max', 'min', 0.999, 'median', 'rms', 'peak']
    kw = dict(fs=1e6, window='hann', resolution=1e6 / 1024, fractional_overlap=0.5,
              statistics=stats, axis=1, bandwidth=0.5e6, dB=dB)
    o = orc.persistence_spectrum(x.copy(), **kw)
    if recorded(ref, o):
        return
    r = ref.fourier.power_spectral_density(x.copy(), **kw)
    isq = np.array(orc.find_float_inds(stats))
    assert r.shape == o.shape
    assert np.array_equal(r[:, ~isq], o[:, ~isq])          # rows the reference does return
    # rows the reference loses: rebuild them from the reference's own pieces
    _, _, sp = ref.fourier.spectrogram(x.copy(), fs=1e6, window='hann', nperseg=1024,
                                       noverlap=512, axis=1)
    ilo, ihi = ref.fourier._freq_band_edges(1024, 1e-6, -0.25e6, 0.25e6)
    sp = sp[..., ilo:ihi]
    if dB:
        sp = ref.power_analysis.powtodB(sp, eps=1e-25, out=sp)
    q = np.quantile(sp, np.array([0.1, 0.5, 0.999], dtype=np.float32), axis=1)
    assert np.array_equal(np.moveaxis(q, 0, 1), o[:, isq])


@pytest.mark.parametrize('kind', ['mean', 'max', 'min', 'median', 'peak', 'rms', 0.3])
def test_bin_power(kind):
    x = synth(4, (2, 30000))
    b1 = orc.iq_to_bin_power(x[0], 1e-6, 250e-6, kind=kind)
    b2 = orc.iq_to_bin_power(x, 1e-6, 300e-6, kind=kind, axis=1, truncate=True)
    b3 = orc.iq_to_bin_power(x.T.copy(), 1e-6, 300e-6, kind=kind, axis=0, truncate=True)
    if recorded(ref, b1, b2, b3):
        return
    a = ref.power_analysis.iq_to_bin_power(x[0], 1e-6, 250e-6, kind=kind)
    assert np.array_equal(a, b1)
    a = ref.power_analysis.iq_to_bin_power(x, 1e-6, 300e-6, kind=kind, axis=1, truncate=True)
    assert np.array_equal(a, b2)
    a = ref.power_analysis.iq_to_bin_power(x.T.copy(), 1e-6, 300e-6, kind=kind, axis=0, truncate=True)
    assert np.array_equal(a, b3)


def test_error_paths_match():
    """the error types are the reference's: checked on the reference too where it is installed"""
    x = synth(5, (1000,))
    for mod in (orc,) if ref is None else (ref.fourier, orc):
        with pytest.raises(TypeError):
            mod.stft(x, fs=1.0, window='hann', nperseg=64, norm='bogus')
        with pytest.raises(ValueError):
            mod.stft(x, fs=1.0, window='hann', nperseg=64, noverlap=0, truncate=False)
        with pytest.raises(ValueError):
            mod.power_spectral_density(x[None], fs=1e6, window='hann', resolution=3e3,
                                       statistics=['mean'], axis=1)
    for fn in (orc.iq_to_bin_power,) if ref is None else (ref.power_analysis.iq_to_bin_power, orc.iq_to_bin_power):
        with pytest.raises(ValueError):
            fn(x, 1.0, 2.5)
        with pytest.raises(ValueError):
            fn(x, 1.0, 300.0)
        with pytest.raises(ValueError):
            fn(x, 1.0, 100.0, kind='bogus')


def test_elementwise_transforms_match_reference():
    """powtodB / dBtopow / envtopow / envtodB restatements vs the unmodified reference (generic
    array branch, power_analysis.py:196-204, 226-229, 251-255, 286-296)"""
    rng = np.random.default_rng(9)
    p = rng.exponential(1e-3, 5000).astype(np.float32)
    z = (rng.standard_normal(5000) + 1j * rng.standard_normal(5000)).astype(np.complex64)
    d = rng.uniform(-100, 20, 5000).astype(np.float32)
    got = [orc.powtodB(p.copy()), orc.powtodB(p.copy(), eps=1e-9), orc.powtodB_noabs(p), orc.dBtopow(d),
           orc.envtopow(z), orc.envtodB(z), orc.envtodB(p, abs=False, eps=1e-6)]
    if recorded(ref, got):
        return
    pa = ref.power_analysis
    assert np.array_equal(got[0], pa.powtodB(p.copy()))
    assert np.array_equal(got[1], pa.powtodB(p.copy(), eps=1e-9))
    assert np.array_equal(got[2], pa.powtodB(p.copy(), abs=False))
    assert np.array_equal(got[3], pa.dBtopow(d.copy()))
    assert np.array_equal(got[4], pa.envtopow(z.copy()))
    assert np.array_equal(got[5], pa.envtodB(z.copy()))
    assert np.array_equal(got[6], pa.envtodB(p.copy(), abs=False, eps=1e-6))


def test_iq_to_cyclic_power_matches_reference():
    x = synth(12, (3, 60000))
    kw = dict(Ts=1e-6, detector_period=1e-5, cyclic_period=1e-3)
    got = orc.iq_to_cyclic_power(x.copy(), axis=1, **kw)
    assert set(got) == {'rms', 'peak'}
    if recorded(ref, got):
        return
    want = ref.power_analysis.iq_to_cyclic_power(x.copy(), axis=1, **kw)
    assert set(got) == set(want) == {'rms', 'peak'}
    for d in want:
        for k in want[d]:
            assert np.array_equal(got[d][k], want[d][k]), (d, k)


def test_frequency_domain_persistence_matches_reference():
    """Domain.FREQUENCY branch (fourier.py:1277-1285, 1303-1307): named rows against the reference
    (its quantile rows are uninitialised memory, SURVEY fact 0.2)"""
    x = synth(8, (2, 40000))
    _, _, X = orc.stft(x, fs=1e6, window='hann', nperseg=256, noverlap=128, axis=1, norm='power')
    stats = ['mean', 'max', 'min']
    cases = [(dB, bw) for dB in (True, False) for bw in (float('inf'), 0.5e6)]
    got = [orc.persistence_spectrum_from_stft(X.copy(), fs=1e6, bandwidth=bw, resolution=1e6 / 256,
                                              fractional_overlap=0.5, statistics=stats, dB=dB, axis=1)
           for dB, bw in cases]
    if recorded(ref, got):
        return
    for (dB, bw), g in zip(cases, got):
        with ref.util.set_input_domain('frequency'):
            want = ref.fourier.power_spectral_density(X.copy(), fs=1e6, bandwidth=bw, window='hann',
                                                      resolution=1e6 / 256, fractional_overlap=0.5,
                                                      statistics=stats, dB=dB, axis=1)
        assert g.shape == want.shape and np.array_equal(g, want), (dB, bw)


@pytest.mark.parametrize('shape,axis', [((4096 * 3,), 0), ((3, 2048 * 5), 1), ((2, 3, 4096), 2)])
@pytest.mark.parametrize('nfft,noverlap', [(256, 128), (256, 192), (64, 0), (128, 112), (1024, 512)])
def test_istft(shape, axis, nfft, noverlap):
    """the frames come from the oracle's stft (equal to the reference's, test_stft)"""
    x = synth(9, shape)
    _, _, y = orc.stft(x.copy(), fs=1e6, window='hamming', nperseg=nfft, noverlap=noverlap, truncate=False,
                       axis=axis)
    sizes = (None, x.shape[axis], x.shape[axis] - 37)
    got = [orc.istft(y.copy(), size, nfft=nfft, noverlap=noverlap, axis=axis) for size in sizes]
    if recorded(ref, got):
        return
    for size, b in zip(sizes, got):
        a = ref.fourier.istft(y.copy(), size, nfft=nfft, noverlap=noverlap, axis=axis)
        assert a.shape == b.shape and np.array_equal(a.view(np.float32), b.view(np.float32))


@pytest.mark.parametrize('shape,axis', [((8192,), 0), ((3, 4096), 1)])
@pytest.mark.parametrize('passband', [(-2e5, 2e5), (-1.3647444248199463 - 2e-6, 1.3647444248199463 + 1e-6)])
def test_ola_filter(shape, axis, passband):
    x = synth(10, shape)
    kw = dict(fs=1e6, nfft=512, window='hamming', passband=passband, axis=axis)
    b = orc.ola_filter(x.copy(), **kw)
    if recorded(ref, b):
        return
    a = ref.fourier.ola_filter(x.copy(), **kw)
    assert a.shape == b.shape and np.array_equal(a.view(np.float32), b.view(np.float32))


def test_ola_filter_errors_match():
    x = synth(10, (8192,))
    for kw, exc in [(dict(window='hann'), TypeError), (dict(window='blackman'), ValueError),
                    (dict(window='hamming', nfft=100), ValueError)]:
        full = dict(dict(fs=1e6, nfft=512, window='hamming', passband=(-1e5, 1e5)), **kw)
        for f in (orc.ola_filter,) if ref is None else (ref.fourier.ola_filter, orc.ola_filter):
            with pytest.raises(exc):
                f(x.copy(), **full)


def test_sample_ccdf_and_histogram_last_axis():
    rng = np.random.default_rng(3)
    p = (rng.standard_normal(100000) ** 2).astype(np.float32)
    p[::97] = 1.0
    ccdf = [(edges, density) for edges in (np.linspace(0, 4, 41), np.array([1.0]),
                                           np.array([0.5, 1.0, 1.0, 2.0], dtype=np.float32))
            for density in (True, False)]
    x = rng.standard_normal((3, 5, 4000)).astype(np.float32)
    x[0, 0, :10] = 2.0
    hist = ((40, (-2.0, 2.0)), (7, None), (np.array([-1.0, 0.0, 0.25, 3.0]), None))
    got_ccdf = [orc.sample_ccdf(p, edges, density=density) for edges, density in ccdf]
    got_hist = [orc.histogram_last_axis(x, bins, rg) for bins, rg in hist]
    if recorded(ref, got_ccdf, got_hist):
        return
    for (edges, density), b in zip(ccdf, got_ccdf):
        a = ref.power_analysis.sample_ccdf(p, edges, density=density)
        assert a.dtype == b.dtype and np.array_equal(a, b)
    for (bins, rg), (h2, e2) in zip(hist, got_hist):
        h, e = ref.util.histogram_last_axis(x, bins, rg)
        assert h.shape == h2.shape and np.array_equal(h, h2) and np.array_equal(e, e2)


@pytest.mark.parametrize('overlap,bw', [(True, None), (True, 0.5e6), (False, 0.75e6), (True, 1e6)])
def test_iq_to_stft_spectrogram(overlap, bw):
    x = synth(12, (20000,))
    b = orc.iq_to_stft_spectrogram(x.copy(), 'hann', 256, 1e-6, overlap=overlap, analysis_bandwidth=bw)
    if recorded(ref, b):
        return
    a = ref.fourier.iq_to_stft_spectrogram(x.copy(), 'hann', 256, 1e-6, overlap=overlap, analysis_bandwidth=bw)
    assert a.shape == b.shape and np.array_equal(a.values, b.values)
    assert np.array_equal(a.columns.values, b.columns.values) and np.array_equal(a.index.values, b.index.values)


def test_channelize_power_is_the_reference_with_the_window_forwarded():
    """the reference raises before doing anything (w= is not an argument of stft); the oracle is the
    same statements with window=, checked against the reference's own building blocks"""
    x = synth(13, (30000,))
    cases = [(4, 0), (4, 32), (1, 0)]
    got = [orc.channelize_power(x.copy(), 1e-6, 64, analysis_bins_per_channel=48, window='hann', channel_count=cc,
                                fft_overlap_per_channel=ov) for cc, ov in cases]
    if recorded(ref, got):
        return
    with pytest.raises(TypeError):
        ref.fourier.channelize_power(x, 1e-6, 64, analysis_bins_per_channel=48, window='hann', channel_count=4)
    for (cc, ov), g in zip(cases, got):
        f, t, X = ref.fourier.stft(x.copy(), fs=1e6, window='hann', nperseg=64 * cc, noverlap=ov * cc, norm='power', axis=0)
        s = cc * 16 // 2
        X, f = X[:, s:-s], f[s:-s]
        if cc == 1:
            assert np.array_equal(g[0], t) and np.array_equal(g[1], ref.power_analysis.envtopow(X).sum(axis=1))
        else:
            want = ref.power_analysis.envtopow(X.reshape(X.shape[0], cc, 48)).sum(axis=2)
            assert np.array_equal(g[0], f[:48]) and np.array_equal(g[1], t) and np.array_equal(g[2], want)


@pytest.mark.parametrize('shape,axis', [((2, 16384), 1), ((16384,), 0)])
@pytest.mark.parametrize('kw', [dict(up=512, down=1024), dict(up=1024, down=512), dict(up=1024, down=1024),
                                dict(up=256, down=1024, frequency_shift=1e6 / 1024 * 100),
                                dict(up=512, down=1024, filter_bandwidth=0.3e6, transition_bandwidth=50e3),
                                dict(up=2048, down=1024, filter_bandwidth=0.6e6, scale=0.5),
                                dict(up=768, down=1024)])
def test_oaresample(shape, axis, kw):
    x = synth(14, shape)
    b = orc.oaresample(x.copy(), fs=1e6, axis=axis, window='hamming', **kw)
    if recorded(ref, b):
        return
    a = ref.fourier.oaresample(x.copy(), fs=1e6, axis=axis, window='hamming', **kw)
    assert a.shape == b.shape and a.dtype == b.dtype
    assert np.array_equal(a.view(np.float32), b.view(np.float32))


def test_util_helpers_equal_the_reference():
    """row U of SURVEY 8a: the product's host helpers against the reference's own (host logic only)"""
    from iqwaveform_b200 import util as U
    a = np.arange(120).reshape(2, 3, 20)
    calls = [('isroundmod', (v, d), {}) for v, d in [(1e6, 1e3), (1e6, 3e3), (0.3, 0.1), (15.36e6, 15e3), (1.0, 0.3)]]
    calls += [('find_float_inds', (('0.5', 'mean', 0.1, 'max', '1e-3'),), {})]
    calls += [('float_dtype_like', (x, m), {})
              for x in (np.zeros(2, np.complex64), np.zeros(2, np.complex128), np.zeros(2, np.float16),
                        np.zeros(2, np.int32), 1.5)
              for m in (None, 'float32', 'float64')]
    calls += [('dtype_change_float', (p, q), {})
              for p, q in [(np.complex128, np.float32), (np.float64, np.float32), (np.complex64, np.float64),
                           (np.float16, np.complex64)]]
    calls += [('axis_slice', (a, 1, None, 2), dict(axis=ax)) for ax in (0, 1, 2, -1)]
    calls += [('axis_index', (a, np.array([0, 2])), dict(axis=1))]
    calls += [('to_blocks', (a, size), dict(truncate=trunc, axis=ax))
              for size, ax, trunc in [(5, 2, False), (5, -1, False), (3, 2, True), (1, 0, False), (2, 0, False)]]
    got = [getattr(U, name)(*args, **kw) for name, args, kw in calls]
    if recorded(ref, got):
        return
    R = ref.util
    for (name, args, kw), g in zip(calls, got):
        want = getattr(R, name)(*args, **kw)
        if name == 'isroundmod':
            assert bool(g) == bool(want), (name, args)
        elif isinstance(want, np.ndarray):
            assert np.array_equal(g, want), (name, args, kw)
        else:
            assert g == want, (name, args)


@pytest.mark.parametrize('n', [16, 100, 1024, 8192])
def test_fft_ifft(n):
    """row A4's public pair (fourier.py:200-246)"""
    x = synth(n, (3, n))
    got = [orc.fft(x, axis=1), orc.ifft(x, axis=1), orc.fft(x.T.copy(), axis=0)]
    if recorded(ref, got):
        return
    assert np.array_equal(ref.fourier.fft(x.copy(), axis=1).view(np.float32), got[0].view(np.float32))
    assert np.array_equal(ref.fourier.ifft(x.copy(), axis=1).view(np.float32), got[1].view(np.float32))
    assert np.array_equal(ref.fourier.fft(x.T.copy(), axis=0), got[2])


@pytest.mark.parametrize('passband', [(-0.2e6, 0.1e6), (-3.0, 2.0), (-1e9, 1e9), (None, 2.0), (-3.0, None)])
def test_zero_stft_by_freq(passband):
    """the frames come from the oracle's stft (equal to the reference's, test_stft)"""
    x = synth(5, (2, 9000))
    f, _, y = orc.stft(x, fs=1e6, window='hamming', nperseg=256, noverlap=128, axis=1)
    b = orc.zero_stft_by_freq(f, y.copy(), passband=passband, axis=1)
    if recorded(ref, b):
        return
    a = ref.fourier.zero_stft_by_freq(f, y.copy(), passband=passband, axis=1)
    assert np.array_equal(a.view(np.float32), b.view(np.float32))
