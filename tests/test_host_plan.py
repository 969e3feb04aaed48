"""host-side logic of the product package: window design, numpy-compatible quantile arithmetic,
band edges, statistic parsing, and the reference's error behaviour (all before any device work)."""
import numpy as np
import pytest

import iqwaveform_b200 as iqw
from iqwaveform_b200 import _lib, _plan
from oracle import iqw_oracle as orc


@pytest.mark.parametrize('window', ['hann', 'blackmanharris', ('kaiser', 8.0), 'rect', None])
@pytest.mark.parametrize('nfft,nzero,hop', [(1024, 0, 512), (256, 64, 64), (4096, 0, 4096), (64, 0, 16)])
@pytest.mark.parametrize('norm', ['power', None])
def test_window_coefficients_bitwise(window, nfft, nzero, hop, norm):
    want = orc.stft_window_coefficients(window, nfft, nzero, norm, hop)
    got = _plan.stft_coefficients(_plan.window_key(window), nfft, nzero, norm, hop)
    assert got.dtype == np.float32 and np.array_equal(got, want)


def test_enbw_window():
    w = _plan.design_window(('kaiser_by_enbw', 2.0), 1024)
    assert abs(_plan._enbw(('kaiser', _plan.find_window_param_from_enbw('kaiser', 2.0, nfft=1024)), 1024) - 2.0) < 1e-4
    assert w.shape == (1024,)
    assert abs(iqw.equivalent_noise_bandwidth('hann', 4096) - 1.5) < 1e-9


def test_quantile_plan_matches_numpy_bitwise():
    rng = np.random.default_rng(0)
    for n in (1, 2, 7, 1000, 29999, 488280, 976561):
        a = np.sort(rng.standard_normal(n).astype(np.float32))
        for q in (0.0, 0.1, 0.25, 0.5, 0.9, 0.99, 0.999, 1.0, 1 / 3):
            lo, hi, g = _plan.quantile_plan(n, q)
            d = a[hi] - a[lo]
            g32 = np.float32(g)
            r = a[hi] - d * (np.float32(1) - g32) if g32 >= 0.5 else a[lo] + d * g32
            assert np.float32(r) == np.quantile(a, np.float32(q)), (n, q)
    assert _plan.quantile_plan(488280, 0.999)[2] == 0.71875       # SURVEY.md row Q
    with pytest.raises(ValueError):
        _plan.quantile_plan(10, 1.5)


def test_axes_and_band_edges():
    assert np.array_equal(_plan.fftfreq(1024, 1e-6), orc.fftfreq(1024, 1e-6))
    f, t = _plan.stft_axes(1e6, 256, 45, 0.5)
    f2, t2 = orc.stft_axes(1e6, 256, 45, 0.5)
    assert np.array_equal(f, f2) and np.array_equal(t, t2)
    assert _plan.freq_band_edges(256, 1 / 256, -64, 64) == (64, 192)
    assert _plan.freq_band_edges(4096, 1e-8, -25e6, 25e6) == orc.freq_band_edges(4096, 1e-8, -25e6, 25e6)


def test_stat_requests():
    reqs = _plan.stat_requests([0.5, '0.99', 'mean', 'rms', 'max', 'peak', 'min', 'median'], 101)
    kinds = [r.kind for r in reqs]
    assert kinds == [_lib.STAT_QUANTILE, _lib.STAT_QUANTILE, _lib.STAT_MEAN, _lib.STAT_MEAN,
                     _lib.STAT_MAX, _lib.STAT_MAX, _lib.STAT_MIN, _lib.STAT_MEDIAN]
    assert (reqs[0].rank_lo, reqs[0].rank_hi, reqs[0].gamma) == (50, 51, 0.0)
    with pytest.raises(ValueError):
        _plan.stat_requests(['bogus'], 10)
    # more than 8 distinct ranks are split into several calls
    many = _plan.stat_requests([i / 10 for i in range(1, 10)], 100000)
    groups = _plan.split_requests(many, 100000)
    assert len(groups) > 1 and sorted(sum(groups, [])) == list(range(9))
    for g in groups:
        assert len(_plan.distinct_ranks([many[i] for i in g], 100000)) <= _lib.MAX_RANKS_PER_CALL


def test_error_behaviour_matches_reference():
    """same exception types for the same conditions as the reference (SURVEY.md 8b), raised on the
    host before anything touches the device"""
    x = np.zeros(1000, np.complex64)
    with pytest.raises(TypeError):
        iqw.stft(x, fs=1.0, window='hann', nperseg=64, norm='bogus')
    with pytest.raises(ValueError):
        iqw.stft(x, fs=1.0, window='hann', nperseg=64, noverlap=0, truncate=False)
    with pytest.raises(IndexError):
        iqw.stft(x[:0], fs=1.0, window='hann', nperseg=64)
    with pytest.raises(ValueError):
        iqw.power_spectral_density(x[None], fs=1e6, window='hann', resolution=3e3,
                                   statistics=['mean'], axis=1)
    with pytest.raises(ValueError):
        iqw.power_spectral_density(x[None], fs=1e6, window='hann', resolution=1e6 / 64,
                                   fractional_window=0.999, statistics=['mean'], axis=1)
    with pytest.raises(ValueError):
        iqw.power_spectral_density(x[None], fs=1e6, window='hann', resolution=1e6 / 64,
                                   statistics=['bogus'], axis=1)
    with pytest.raises(ValueError):
        iqw.iq_to_bin_power(x, 1.0, 2.5)
    with pytest.raises(ValueError):
        iqw.iq_to_bin_power(x, 1.0, 300.0)
    with pytest.raises(ValueError):
        iqw.iq_to_bin_power(x, 1.0, 100.0, kind='bogus')
    with pytest.raises(IndexError):
        iqw.iq_to_bin_power(x[:0], 1.0, 100.0)
    with pytest.raises(TypeError):
        iqw.iq_to_bin_power([1, 2, 3], 1.0, 1.0)
    assert iqw.persistence_spectrum is iqw.power_spectral_density


def test_no_cpu_fallback():
    """without a CUDA device the package raises instead of computing on the CPU; checked in a child process that
    sees no device, so that the test also runs on a machine with a GPU"""
    import os
    import subprocess
    import sys

    code = ('import numpy as np, pytest, iqwaveform_b200 as iqw\n'
            "with pytest.raises(RuntimeError, match='no CPU fallback'):\n"
            "    iqw.spectrogram(np.zeros(1000, np.complex64), fs=1.0, window='hann', nperseg=64)\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, '-c', code], cwd=root, env=dict(os.environ, CUDA_VISIBLE_DEVICES=''),
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_util_helpers_known_answers():
    import torch
    from iqwaveform_b200 import util as U
    assert U.isroundmod(1e6, 1e3) and not U.isroundmod(1e6, 3e3) and U.isroundmod(0.3, 0.1)
    assert list(U.isroundmod(np.array([1.0, 1.5]), 0.5)) == [True, True] and not U.isroundmod(np.array([1.1]), 0.5)[0]
    assert U.find_float_inds(('0.5', 'mean', 0.1, '1e-3')) == [True, False, True, True]
    for x, want in [(np.zeros(2, np.complex64), 'float32'), (np.zeros(2, np.complex128), 'float64'),
                    (np.zeros(2, np.float16), 'float16'), (np.zeros(2, np.int32), 'float32'), (1.5, 'float64'),
                    (torch.zeros(2, dtype=torch.complex64), 'float32'), (torch.zeros(2, dtype=torch.float64), 'float64')]:
        assert U.float_dtype_like(x) == np.dtype(want)
    assert U.float_dtype_like(np.zeros(2, np.float16), 'float32') == np.dtype('float32')
    assert U.dtype_change_float(np.complex128, np.float32) is np.complex64
    assert U.dtype_change_float('float64', 'complex64') is np.float32
    with pytest.raises(ValueError):
        U.dtype_change_float(np.int32, np.float32)
    a = np.arange(24).reshape(2, 3, 4)
    assert np.array_equal(U.axis_slice(a, 1, None, axis=1), a[:, 1:]) and np.array_equal(U.axis_slice(a, 0, 4, 2), a[..., 0:4:2])
    assert np.array_equal(U.axis_index(a, np.array([True, False, True]), axis=1), a[:, [0, 2]])
    assert U.to_blocks(a, 2, axis=2).shape == (2, 3, 2, 2) and U.to_blocks(a, 2, axis=-1).shape == (2, 3, 2, 2)
    assert U.to_blocks(np.arange(10), 4, truncate=True).shape == (2, 4)
    assert U.to_blocks(torch.arange(10), 5).shape == (2, 5)
    with pytest.raises(ValueError):
        U.to_blocks(np.arange(10), 4)
    with pytest.raises(TypeError):
        U.to_blocks(np.arange(10), 2.0)
    with pytest.raises(IndexError):
        U.to_blocks(np.zeros(0), 2)
