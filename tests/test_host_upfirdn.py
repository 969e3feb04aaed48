"""upfirdn host logic without a GPU: scipy's output length, the polyphase table, the time-shard planner
(with a numpy direct-formula stand-in for the kernel) and the argument checks that run before any
device work."""
import numpy as np
import pytest
import scipy.signal as ss
import torch
from scipy.signal._upfirdn import _output_len

import iqwaveform_b200 as iqw
from iqwaveform_b200 import _plan
from iqwaveform_b200 import distributed as D


def _direct(x_buf, table, n_taps, up, down, *, x_first, out_first, n_out):
    """float64 y[n] = sum_j hp[p][j] * x[i0 - j] over global outputs [out_first, out_first + n_out), reading
    only the buffer that holds global samples [x_first, x_first + len(x_buf)) (zero elsewhere)"""
    x_buf = np.asarray(x_buf).astype(np.complex128)
    rows, lp = table.shape
    p, i0 = _plan.upfirdn_phase_index(np.arange(out_first, out_first + n_out), up, down)
    y = np.zeros(n_out, np.complex128)
    for j in range(lp):
        idx = i0 - j - x_first
        ok = (idx >= 0) & (idx < x_buf.size) & (p < rows)
        y[ok] += table[p[ok], j].astype(np.complex128) * x_buf[idx[ok]]
    return y


GRID = [(L, n, up, down) for L in (1, 2, 7, 16, 161) for n in (1, 2, 5, 64, 999)
        for up, down in ((1, 1), (2, 1), (1, 2), (3, 2), (4, 6), (147, 160), (160, 147), (8, 8), (5, 1), (1, 16))]


def test_output_len_matches_scipy():
    for L, n, up, down in GRID:
        assert _plan.upfirdn_output_len(L, n, up, down) == _output_len(L, n, up, down), (L, n, up, down)


@pytest.mark.parametrize('up', [1, 2, 3, 4, 147, 300])
@pytest.mark.parametrize('L', [1, 5, 161, 3201])
def test_polyphase_table_reassembles_h(up, L):
    h = np.random.default_rng(L + up).standard_normal(L).astype(np.float32)
    t = _plan.upfirdn_polyphase(h, up)
    lp = -(-L // up)
    assert t.shape == (min(up, L), lp)
    back = np.zeros(lp * up, np.float32)
    for p in range(t.shape[0]):
        back[p::up] = t[p]
    assert np.array_equal(back[:L], h) and not back[L:].any()


def test_direct_formula_is_scipy():
    rng = np.random.default_rng(1)
    for L, n, up, down in GRID[::3]:
        h = rng.standard_normal(L).astype(np.float32)
        x = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
        want = ss.upfirdn(h.astype(np.float64), x.astype(np.complex128), up, down)
        t = _plan.upfirdn_polyphase(h, up)
        got = _direct(x, t, L, up, down, x_first=0, out_first=0, n_out=want.size)
        np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize('world', [1, 2, 3, 4, 5])
def test_shard_planner_tiles_outputs_and_holds_every_input(world):
    rng = np.random.default_rng(world)
    for L, n, up, down in [(161, 5000, 1, 8), (3201, 4000, 147, 160), (81, 700, 4, 1), (129, 3, 1, 1),
                           (7, 1, 3, 2), (40, 300, 160, 147), (16, 257, 5, 3)]:
        h = rng.standard_normal(L).astype(np.float32)
        x = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
        want = ss.upfirdn(h.astype(np.float64), x.astype(np.complex128), up, down)
        outs, parts = [], []
        group = D.ThreadGroup(world)
        for r in range(world):
            sh = D.upfirdn_shard(n, L, up, down, world, r)
            assert sh.n_out == want.size
            assert 0 <= sh.sample0 <= sh.sample1 <= n
            outs += list(range(sh.out0, sh.out1))
            parts.append(np.asarray(D.upfirdn_time_sharded(x[sh.sample0:sh.sample1], h, up, down, n_samples=n,
                                                           group=group.member(r), compute=_direct)))
        assert outs == list(range(want.size))
        np.testing.assert_allclose(np.concatenate(parts), want, rtol=1e-10, atol=1e-10)


def test_shard_rejects_a_wrong_halo():
    sh = D.upfirdn_shard(1000, 33, 2, 3, 2, 1)
    x = np.zeros(sh.sample1 - sh.sample0 + 1, np.complex64)
    with pytest.raises(ValueError, match='expects a 1-D shard'):
        D.upfirdn_time_sharded(x, np.ones(33), 2, 3, n_samples=1000, group=D.ThreadGroup(2).member(1), compute=_direct)


def test_argument_errors_before_device_work():
    x = np.zeros(64, np.complex64)
    for h in (np.ones((2, 3)), np.ones(0), 1.0):
        with pytest.raises(ValueError, match='1-D'):
            iqw.upfirdn(h, x)
    for up, down in ((0, 1), (1, 0), (-1, 2)):
        with pytest.raises(ValueError, match='>= 1'):
            iqw.upfirdn(np.ones(4), x, up, down)
    with pytest.raises(ValueError, match='Unknown mode'):
        iqw.upfirdn(np.ones(4), x, mode='nonsense')
    for mode in ('wrap', 'edge', 'symmetric', 'reflect', 'line'):
        with pytest.raises(NotImplementedError, match='constant'):
            iqw.upfirdn(np.ones(4), x, mode=mode)
    with pytest.raises(NotImplementedError, match='constant'):
        iqw.upfirdn(np.ones(4), x, cval=1.0)
    for bad in (np.zeros(64, np.complex128), np.zeros(64, np.float32), torch.zeros(64, dtype=torch.float32)):
        with pytest.raises(NotImplementedError, match='complex64'):
            iqw.upfirdn(np.ones(4), bad)
    # the limit is on the table (32768 floats), which up = 1 fills with the taps themselves
    with pytest.raises(NotImplementedError, match='exceeds'):
        iqw.upfirdn(np.ones(32769), x)
    with pytest.raises(NotImplementedError, match='exceeds'):
        iqw.upfirdn(np.ones(16385, np.complex64), x)
    with pytest.raises(NotImplementedError, match='exceeds'):
        iqw.upfirdn(np.ones(20000), x, 19999)         # 19999 rows x 2 taps


def test_table_limit_admits_the_documented_sizes_for_any_up():
    from iqwaveform_b200 import fourier
    for up in (1, 2, 3, 7, 100, 147, 4097, 8191, 16383, 16384, 100000):
        fourier._upfirdn_taps(np.ones(16384), up, 1)
        fourier._upfirdn_taps(np.ones(8192, np.complex128), up, 1)
