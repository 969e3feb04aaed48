"""the numpy oracle against the committed fixtures (outputs of the unmodified reference):
bit-for-bit, on CPU.  This is what pins the oracle on the GPU box, where the reference is absent."""
import numpy as np
import pytest

from conftest import load_golden
from oracle import iqw_oracle as orc

STFT = ['stft_hann_256_128_power', 'stft_hann_256_128_cola', 'stft_bh_512_0_power',
        'stft_kaiser_64_48_power', 'stft_hann_1024_512_nzero']
SPG = ['spg_bh_2048_1024', 'spg_hann_1024_768', 'spg_rect_4096_0']
PSD = ['psd_hann_1024_half', 'psd_hann_4096_trim', 'psd_bh_256_linear']


@pytest.fixture(autouse=True)
def _fixture_fft_threads(monkeypatch):
    """the reference runs its FFTs on os.cpu_count() // 2 threads, and the thread count changes the last bits of some
    transforms: the oracle uses the CPU count of the machine that wrote the fixtures (8; only then does
    spg_bh_2048_1024 match), whatever machine runs the test"""
    monkeypatch.setattr(orc, 'CPU_COUNT', 8)


@pytest.mark.parametrize('name', STFT)
def test_stft_bitwise(name):
    p, a = load_golden(name)
    f, t, y = orc.stft(a['x'], **p)
    assert np.array_equal(f, a['freqs']) and np.array_equal(t, a['times'])
    assert y.dtype == np.complex64
    assert np.array_equal(y.view(np.float32), a['y'].view(np.float32))


@pytest.mark.parametrize('name', SPG)
def test_spectrogram_bitwise(name):
    p, a = load_golden(name)
    f, t, pw = orc.spectrogram(a['x'], **p)
    assert np.array_equal(f, a['freqs']) and np.array_equal(t, a['times'])
    assert pw.dtype == np.float32 and np.array_equal(pw, a['power'])
    assert np.array_equal(orc.powtodB(pw.copy()), a['dB'])


@pytest.mark.parametrize('name', PSD)
def test_persistence_bitwise(name):
    p, a = load_golden(name)
    out = orc.persistence_spectrum(a['x'], **p)
    isq = a['is_quantile']
    assert out.dtype == np.float32
    assert np.array_equal(out[:, ~isq, :], a['named_rows'])
    assert np.array_equal(out[:, isq, :], a['quantile_rows'])


def test_bin_power_bitwise():
    p, a = load_golden('binpower_1536')
    for kind in ('mean', 'max', 'min', 'median', 'rms', 'peak'):
        assert np.array_equal(orc.iq_to_bin_power(a['x'], kind=kind, **p), a[kind])
    assert np.array_equal(orc.iq_to_bin_power(a['x'], kind=0.25, **p), a['q25'])


def test_quantile_restatement_matches_numpy_bitwise():
    rng = np.random.default_rng(5)
    qs = np.array([0.0, 0.1, 0.25, 0.5, 0.9, 0.99, 0.999, 1.0], dtype=np.float32)
    for n in (1, 2, 3, 10, 77, 1000, 29999, 488280):
        cols = 3 if n > 100000 else 17
        a = rng.standard_normal((n, cols)).astype(np.float32)
        want = np.quantile(a, qs, axis=0)
        got = orc.quantile_from_sorted(np.sort(a, axis=0), qs)
        assert np.array_equal(got, want), n


def test_known_answers():
    """indexing known-answers that involve no FFT accuracy (SURVEY.md section 4.3)"""
    nfft, hop = 64, 16
    n = 1000
    # ramp with a rectangular window: centre (DC) bin of frame m = mean of the frame
    x = np.arange(n).astype(np.complex64)
    _, t, y = orc.stft(x, fs=1.0, window='rect', nperseg=nfft, noverlap=nfft - hop, norm='power')
    T = (n - nfft) // hop + 1
    assert y.shape == (T, nfft)
    m = np.arange(T)
    np.testing.assert_allclose(y[:, nfft // 2].real, m * hop + (nfft - 1) / 2, rtol=1e-6)
    assert np.array_equal(t, m * float(hop))
    # unit impulse: non-zero only in frames that contain it
    s = 333
    x = np.zeros(n, np.complex64); x[s] = 1
    _, _, p = orc.spectrogram(x, fs=1.0, window='rect', nperseg=nfft, noverlap=nfft - hop)
    hit = (m * hop <= s) & (s < m * hop + nfft)
    assert np.all(p[hit].min(axis=1) > 0) and np.all(p[~hit] == 0)
    # bin-centred tone at index k lands in output bin k + nfft/2 with power A^2 (rect: ENBW 1)
    k, A = 5, 2.0
    x = (A * np.exp(2j * np.pi * k * np.arange(n) / nfft)).astype(np.complex64)
    _, _, p = orc.spectrogram(x, fs=1.0, window='rect', nperseg=nfft, noverlap=0)
    assert np.all(p.argmax(axis=1) == k + nfft // 2)
    np.testing.assert_allclose(p.max(axis=1), A * A, rtol=1e-5)
    # band edges: upper edge bin is dropped (fourier.py:1198)
    assert orc.freq_band_edges(256, 1 / 256, -64, 64) == (64, 192)


ISTFT = ['istft_hamming_256_128', 'istft_bh_1024_768', 'istft_rect_64_0']
OLA = ['ola_hamming_512_all', 'ola_hamming_512_band']


@pytest.mark.parametrize('name', ISTFT)
def test_istft_bitwise(name):
    p, a = load_golden(name)
    x = orc.istft(a['y'], p['size'], nfft=p['nperseg'], noverlap=p['noverlap'], axis=p['axis'])
    assert x.dtype == np.complex64 and x.shape == a['x'].shape
    assert np.array_equal(x.view(np.float32), a['x'].view(np.float32))


@pytest.mark.parametrize('name', OLA)
def test_ola_filter_bitwise(name):
    p, a = load_golden(name)
    p['passband'] = tuple(p['passband'])
    out = orc.ola_filter(a['x'], **p)
    assert out.dtype == np.complex64 and out.shape == a['out'].shape
    assert np.array_equal(out.view(np.float32), a['out'].view(np.float32))
    if name.endswith('band'):       # the mask really removed something
        assert np.abs(out).mean() < 0.8 * np.abs(a['x']).mean()


def test_ccdf_and_histogram_bitwise():
    _, a = load_golden('ccdf_power_61')
    assert np.array_equal(orc.sample_ccdf(a['p'], a['edges'], density=True), a['density'])
    assert np.array_equal(orc.sample_ccdf(a['p'], a['edges'], density=False), a['counts'])
    p, a = load_golden('hist_db_50')
    h, e = orc.histogram_last_axis(a['x'], p['bins'], tuple(p['range']))
    assert np.array_equal(h, a['hist']) and np.array_equal(e, a['edges'])


@pytest.mark.parametrize('name', ['oares_down_1024_512', 'oares_up_512_1024_fir', 'oares_shift_1024_256'])
def test_oaresample_bitwise(name):
    p, a = load_golden(name)
    out = orc.oaresample(a['x'], **p)
    assert out.dtype == np.complex64 and out.shape == a['out'].shape
    assert np.array_equal(out.view(np.float32), a['out'].view(np.float32))
