"""pfb_synthesize host logic without a GPU: the argument checks that run before any device work, the output
length, the time-shard planner, the factorisation against the definition and the adjoint identity in float64,
the reconstruction recipe, and a numpy complex64 emulation of the kernels' arithmetic -- against the float64
factorisation within the documented bound, and run shard by shard, bitwise equal to one call."""
import numpy as np
import pytest
import scipy.signal as ss
import torch

import iqwaveform_b200 as iqw
from iqwaveform_b200 import _plan
from iqwaveform_b200 import distributed as D

from _pfb_numpy import direct64 as analysis64
from _pfb_numpy import fold64, prototype
from _pfb_synth_numpy import direct64, emulate, fact64, norm, recipe, snr_db


def test_argument_errors_before_device_work():
    y = np.zeros((10, 64), np.complex64)
    g = np.ones(256)
    for bad_g in (np.ones((2, 8)), np.ones(0), np.float32(1.0)):
        with pytest.raises(ValueError, match='g must be 1-D'):
            iqw.pfb_synthesize(y, bad_g)
    for hop in (0, -1, 65, 32.0, True):
        with pytest.raises(ValueError, match='hop'):
            iqw.pfb_synthesize(y, g, hop)
    with pytest.raises(ValueError, match='at least one frame'):
        iqw.pfb_synthesize(np.zeros((0, 64), np.complex64), g)
    for axis in (1, -1, 2, -3):
        with pytest.raises(ValueError, match='axis'):
            iqw.pfb_synthesize(y, g, axis=axis)
    with pytest.raises(ValueError, match='axis'):
        iqw.pfb_synthesize(np.zeros(64, np.complex64), g)
    with pytest.raises(ValueError, match='even integer'):
        iqw.pfb_synthesize(np.zeros((10, 63), np.complex64), g)
    # what is not built
    for bad in (np.zeros((10, 64), np.complex128), np.zeros((10, 64), np.float32),
                torch.zeros((10, 64), dtype=torch.float32)):
        with pytest.raises(NotImplementedError, match='complex64'):
            iqw.pfb_synthesize(bad, g)
    with pytest.raises(NotImplementedError, match='complex prototypes'):
        iqw.pfb_synthesize(y, g.astype(np.complex64))
    for K in (2, 8, 48, 96, 16384):
        with pytest.raises(NotImplementedError, match='powers of two'):
            iqw.pfb_synthesize(np.zeros((2, K), np.complex64), np.ones(8))
    with pytest.raises(NotImplementedError, match='16 \\* nchannels'):
        iqw.pfb_synthesize(y, np.ones(16 * 64 + 1))
    with pytest.raises(NotImplementedError, match='32768'):
        iqw.pfb_synthesize(np.zeros((2, 8192), np.complex64), np.ones(32769))


def test_output_length():
    assert _plan.pfb_synth_len(1, 100, 7) == 100
    assert _plan.pfb_synth_len(5, 8192, 512) == 4 * 512 + 8192
    # the analysis bank's capture length when the prototypes have the same length and the capture ends on a frame
    for N, L, hop in [(100000, 8192, 1024), (5000, 1000, 48), (300, 256, 1)]:
        T = _plan.pfb_frame_count(N, L, hop)
        assert _plan.pfb_synth_len(T, L, hop) == N - (N - L) % hop


SHARD_GEOMETRIES = [(100, 8192, 1024, 1024), (200, 8192, 1024, 512), (80, 1000, 64, 48), (300, 256, 16, 1),
                    (3, 33, 16, 16), (1, 32768, 8192, 8192), (20, 100, 1024, 1024), (7, 20, 32, 29), (1, 5, 16, 16)]


@pytest.mark.parametrize('world', [1, 2, 3, 5, 8, 64])
def test_shard_planner(world):
    """the shards tile [0, n_out), and each reads exactly the frames its outputs need"""
    for T, Lg, K, hop in SHARD_GEOMETRIES:
        n_out = _plan.pfb_synth_len(T, Lg, hop)
        outs = []
        for r in range(world):
            sh = D.pfb_synth_shard(T, Lg, K, hop, world, r)
            assert sh.n_out == n_out and 0 <= sh.frame0 <= sh.frame1 <= T
            outs += list(range(sh.out0, sh.out1))
            need = {m for t in range(sh.out0, sh.out1) for m in range(T) if 0 <= t - m * hop < Lg}
            assert set(range(sh.frame0, sh.frame1)) == need, (T, Lg, K, hop, world, r)
        assert outs == list(range(n_out))
    assert D.pfb_synth_shard(10, 100, 64, None, 2, 0) == D.pfb_synth_shard(10, 100, 64, 64, 2, 0)
    with pytest.raises(ValueError):
        D.pfb_synth_shard(0, 100, 64, 64, 2, 0)


@pytest.mark.parametrize('K,Lg,hop', [(16, 64, 16), (16, 100, 8), (32, 256, 24), (64, 64, 64), (64, 500, 48),
                                      (16, 10, 16), (16, 40, 1)])
def test_factorisation_is_the_definition(K, Lg, hop):
    rng = np.random.default_rng(K + Lg + hop)
    y = rng.standard_normal((9, K)) + 1j * rng.standard_normal((9, K))
    g = prototype(Lg, K)
    a, b = direct64(y, g, hop), fact64(y, g, hop)
    assert np.abs(a - b).max() <= 1e-12 * np.abs(a).max()


@pytest.mark.parametrize('K,L,hop', [(16, 64, 16), (16, 128, 8), (32, 256, 24), (64, 500, 48)])
def test_adjoint_of_the_analysis_bank(K, L, hop):
    """<A x, y> = <x, A^H y>, A = pfb_channelize with h, A^H = pfb_synthesize with g = h"""
    rng = np.random.default_rng(K * L)
    h = prototype(L, K)
    x = rng.standard_normal(L + 17 * hop) + 1j * rng.standard_normal(L + 17 * hop)
    Ax = analysis64(x, h, K, hop)
    y = rng.standard_normal(Ax.shape) + 1j * rng.standard_normal(Ax.shape)
    AHy = fact64(y, h, hop)
    lhs, rhs = np.vdot(y, Ax), np.vdot(AHy, x[:AHy.size])
    assert abs(lhs - rhs) <= 1e-13 * abs(lhs)


@pytest.mark.parametrize('K', [16, 256])
def test_recipe_reconstructs(K):
    """the hop = K/2 pair of the docstring, in float64, over the interior"""
    h, g, hop = recipe(K)
    x = capture(np.random.default_rng(K), 24 * 8 * K)
    xr = fact64(fold64(x, h, K, hop), g, hop)
    assert snr_db(x, xr, 8 * K) >= 79.5


def test_root_hann_p1_reconstructs_exactly():
    K = 64
    w = np.sqrt(ss.windows.hann(K, sym=False))
    x = capture(np.random.default_rng(1), 4000)
    xr = fact64(fold64(x, w, K, K // 2), w / K, K // 2)
    assert np.abs(xr[K:-K] - x[K:xr.size - K]).max() <= 1e-12


def capture(rng, n):
    return (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)


def _frames(rng, T, K):
    """complex64 frames with a +60 dB burst frame"""
    y = (rng.standard_normal((T, K)) + 1j * rng.standard_normal((T, K))).astype(np.complex64)
    y[T // 2] *= 1000
    return y


EMU_CASES = [(16, 128, 8), (16, 100, 1), (64, 512, 32), (64, 512, 64), (32, 512, 20), (256, 2048, 128),
             (256, 4000, 96), (1024, 1024, 1024), (1024, 8192, 512), (4096, 16384, 2048), (16, 256, 16)]


@pytest.mark.parametrize('K,Lg,hop', EMU_CASES)
def test_emulation_within_bound_of_float64(K, Lg, hop):
    rng = np.random.default_rng(K * 7 + Lg + hop)
    h, g, _ = recipe(K, Lg)
    taps = _plan.pfb_taps(g, K)
    T = max(4, 12 * -(-Lg // hop))
    y = _frames(rng, T, K)
    n_out = _plan.pfb_synth_len(T, Lg, hop)
    got = emulate(y, taps, Lg, hop, n_frames_total=T, out_first=0, n_out=n_out)
    want = fact64(y, taps.ravel()[:Lg] * np.where(np.arange(Lg) % 2, -1, 1), hop)
    nrm = norm(y, taps, Lg, hop)
    r = np.abs(got - want)[nrm > 0] / nrm[nrm > 0]
    assert r.max() <= 2, float(r.max())
    assert np.all(got[nrm == 0] == 0)


@pytest.mark.parametrize('world', [1, 2, 3, 4, 7])
def test_shards_are_bitwise_one_call(world):
    for T, Lg, K, hop in [(40, 1024, 64, 64), (30, 4000, 256, 128), (50, 1000, 64, 37), (60, 256, 16, 1),
                          (9, 33, 16, 16), (12, 20, 32, 29)]:
        rng = np.random.default_rng(T + world)
        g = prototype(Lg, K)
        y = _frames(rng, T, K)
        taps = _plan.pfb_taps(g, K)
        single = emulate(y, taps, Lg, hop, n_frames_total=T, out_first=0, n_out=_plan.pfb_synth_len(T, Lg, hop))
        group = D.ThreadGroup(world)
        parts = []
        for r in range(world):
            sh = D.pfb_synth_shard(T, Lg, K, hop, world, r)
            parts.append(np.asarray(D.pfb_synthesize_time_sharded(y[sh.frame0:sh.frame1], g, hop, n_frames=T,
                                                                  group=group.member(r), compute=emulate)))
        assert np.array_equal(np.concatenate(parts), single), (T, Lg, K, hop)


def test_shard_rejects_a_wrong_halo():
    sh = D.pfb_synth_shard(20, 100, 16, 8, 2, 1)
    y = np.zeros((sh.frame1 - sh.frame0 + 1, 16), np.complex64)
    with pytest.raises(ValueError, match='expects a shard'):
        D.pfb_synthesize_time_sharded(y, np.ones(100), 8, n_frames=20, group=D.ThreadGroup(2).member(1),
                                      compute=emulate)
    with pytest.raises(ValueError, match='frames, nchannels'):
        D.pfb_synthesize_time_sharded(np.zeros(16, np.complex64), np.ones(100), 8, n_frames=20,
                                      group=D.ThreadGroup(2).member(1), compute=emulate)
