"""sosfilt host logic without a GPU: scipy's argument checks and what is not built, the state-space form and the
chunk fold in float64 against scipy, the time-shard planner, the numpy emulation of kernel 10 within the error
bound, emulated shards (threads and gloo) bitwise equal to one emulated call, and the workspace queries."""
import os
import socket
import threading

import numpy as np
import pytest
import scipy.signal as ss
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import iqwaveform_b200 as iqw
from iqwaveform_b200 import _lib, _plan, fourier
from iqwaveform_b200 import distributed as D

from _sosfilt_numpy import FILTERS, NumpyOps, emulate, ratio, reference, signal, zf_unit

HOST_FACTOR = 6


def test_argument_errors():
    x = np.zeros(64, np.complex64)
    with pytest.raises(ValueError, match=r'sos array must be shape \(n_sections, 6\)'):
        iqw.sosfilt(np.ones((2, 5)), x)
    with pytest.raises(ValueError, match=r'sos\[:, 3\] should be all ones'):
        iqw.sosfilt([[1, 0, 0, 2, 0, 0]], x)
    with pytest.raises(NotImplementedError, match='real coefficients'):
        iqw.sosfilt([[1, 0, 0, 1, 0.5j, 0]], x)
    with pytest.raises(NotImplementedError, match='17 sections'):
        iqw.sosfilt(np.tile([1, 0, 0, 1, 0, 0], (17, 1)), x)
    with pytest.raises(NotImplementedError, match='unstable'):
        iqw.sosfilt([[1, 0, 0, 1, -2.1, 1.2]], x)
    with pytest.raises(NotImplementedError, match='unstable'):
        iqw.sosfilt([[1, 0, 0, 1, 0, 1.0001]], x)
    for bad in (np.zeros(64, np.complex128), np.zeros(64, np.float32), torch.zeros(64)):
        with pytest.raises(NotImplementedError, match='complex64'):
            iqw.sosfilt([[1, 0, 0, 1, 0, 0]], bad)
    sos = ss.butter(4, 0.1, output='sos')
    with pytest.raises(ValueError, match='Invalid zi shape') as e:
        iqw.sosfilt(sos, np.zeros((3, 64), np.complex64), axis=0, zi=np.zeros((2, 3, 64)))
    # scipy's own message, word for word
    with pytest.raises(ValueError) as s:
        ss.sosfilt(sos, np.zeros((3, 64), np.complex64), axis=0, zi=np.zeros((2, 3, 64)))
    assert str(e.value) == str(s.value)


def test_sos_reaches_the_library_row_by_row():
    """a Fortran-ordered array or a transposed tensor view gives the same C-ordered float32 coefficients"""
    sos = ss.ellip(8, 0.1, 80, 0.05, output='sos')
    want = fourier._sosfilt_sos(sos)
    assert want.flags.c_contiguous
    for other in (np.asfortranarray(sos), torch.from_numpy(np.ascontiguousarray(sos.T)).T):
        got = fourier._sosfilt_sos(other)
        assert got.flags.c_contiguous and np.array_equal(got, want)
        assert np.array_equal(np.frombuffer(got.tobytes(), np.float32), want.reshape(-1))


def test_poles_on_the_unit_circle_are_accepted():
    for sos in ([[1, 0, 0, 1, -1, 0]], [[1, 0, 0, 1, -2, 1]], [[1, 0, 0, 1, 0, 1]], [[1, 0, 0, 1, 1, 0]]):
        assert fourier._sosfilt_sos(sos).dtype == np.float32


def test_state_space_matches_scipy_float64():
    rng = np.random.default_rng(1)
    for sos in FILTERS.values():
        sos = np.asarray(sos, np.float32).astype(np.float64)
        A, B, C, D_ = _plan.sosfilt_state_space(sos)
        x = rng.standard_normal(500) + 1j * rng.standard_normal(500)
        z = (rng.standard_normal(2 * len(sos)) + 1j * rng.standard_normal(2 * len(sos)))
        want, zf = ss.sosfilt(sos, x, zi=z.reshape(-1, 2))
        y = np.empty_like(x)
        for n in range(x.size):
            y[n] = C @ z + D_ * x[n]
            z = A @ z + B * x[n]
        scale = np.abs(want).max()
        assert np.abs(y - want).max() <= 1e-12 * scale
        assert np.abs(z - zf.reshape(-1)).max() <= 1e-12 * max(1.0, np.abs(zf).max())


def test_chunk_fold_gives_scipy_final_state():
    rng = np.random.default_rng(2)
    L = 64
    for sos in FILTERS.values():
        sos = np.asarray(sos, np.float32).astype(np.float64)
        S = len(sos)
        P = _plan.sosfilt_powers(sos, L, 1, 1)[0]
        x = rng.standard_normal(16 * L) + 1j * rng.standard_normal(16 * L)
        _, want = ss.sosfilt(sos, x, zi=np.zeros((S, 2)))
        t = np.zeros(2 * S, complex)
        for c in range(16):
            _, b = ss.sosfilt(sos, x[c * L:(c + 1) * L], zi=np.zeros((S, 2)))
            t = P @ t + b.reshape(-1)
        assert np.abs(t - want.reshape(-1)).max() <= 1e-10 * max(1.0, np.abs(want).max())


@pytest.mark.parametrize('S', [1, 4, 8, 9, 16])
def test_planner_aligns_and_covers(S):
    L, G, _ = fourier._sosfilt_geometry(S)
    for n in (0, 1, L * G - 1, L * G, 5 * L * G + 17):
        for world in (1, 2, 3, 7):
            spans = [D.sosfilt_shard(n, S, world, r) for r in range(world)]
            assert spans[0].sample0 == 0 and spans[-1].sample1 == n
            for a, b in zip(spans, spans[1:]):
                assert a.sample1 == b.sample0
            for sh in spans:
                assert (sh.out0, sh.out1, sh.n_out) == (sh.sample0, sh.sample1, n)
                assert sh.sample0 % (L * G) == 0 or sh.sample0 == n


def _emulation_ratios(name, n, rng):
    """(y without zi, y with zi, zf with zi) of the emulation of one row of n samples, in units of the bound"""
    sos32 = fourier._sosfilt_sos(FILTERS[name])
    S = len(sos32)
    x = signal(rng, n)
    y, _ = emulate(x, sos32)
    y64, e32 = reference(x, sos32)
    r0 = ratio(y, y64, e32)
    zi = (rng.standard_normal((S, 2)) + 1j * rng.standard_normal((S, 2))).astype(np.complex64)
    y, zf = emulate(x, sos32, zi)
    y64, e32, zf64, zf32 = reference(x, sos32, zi)
    return r0, ratio(y, y64, e32), ratio(zf.reshape(-1), zf64.reshape(-1), zf_unit(zf32, zf64, e32))


@pytest.mark.parametrize('name', sorted(FILTERS))
def test_emulation_within_bound(name):
    rng = np.random.default_rng(3)
    L, G, _ = fourier._sosfilt_geometry(len(FILTERS[name]))
    worst = np.zeros(3)
    for n in (1 << 20, 3 * L * G + L // 2 + 3, L * G, L - 1, 1):
        r = _emulation_ratios(name, n, rng)
        assert max(r) <= HOST_FACTOR, (name, n, r)
        worst = np.maximum(worst, r)
    print(f'{name}: worst y {worst[0]:.2f} / y with zi {worst[1]:.2f} / zf {worst[2]:.2f} units')


@pytest.mark.parametrize('name', ['ellip8', 'butter32'])
def test_emulation_within_bound_over_carry_blocks(name):
    """rows longer than one carry block of H groups: the block folds, the fold over blocks with A^(LGH) from zi, and
    the expansion of each block's groups all reach the result"""
    L, G, H = fourier._sosfilt_geometry(len(FILTERS[name]))
    r = _emulation_ratios(name, (H + 1) * L * G + 17, np.random.default_rng(11))
    assert max(r) <= HOST_FACTOR, (name, r)
    print(f'{name} over {H + 1} groups: y {r[0]:.2f} / y with zi {r[1]:.2f} / zf {r[2]:.2f} units')


def _case(world_seed=4, groups=5):
    sos32 = fourier._sosfilt_sos(FILTERS['ellip8'])
    L, G, _ = fourier._sosfilt_geometry(len(sos32))
    n = groups * L * G + 1234
    x = signal(np.random.default_rng(world_seed), n)
    zi = (np.arange(2 * len(sos32)) * (1 - 0.5j)).reshape(-1, 2).astype(np.complex64)
    return sos32, n, x, zi


def _run_rank(group, world, rank, sos32, n, x, zi, gather):
    sh = D.sosfilt_shard(n, len(sos32), world, rank)
    return D.sosfilt_time_sharded(x[sh.sample0:sh.sample1], sos32, n_samples=n, zi=zi, group=group,
                                  compute=NumpyOps(), gather=gather)


def _on_threads(world, run):
    tg = D.ThreadGroup(world)
    out, errors = [None] * world, []

    def body(r):
        try:
            out[r] = run(tg.member(r), r)
        except Exception as e:       # noqa: BLE001
            errors.append(e)
            tg._barrier.abort()
    threads = [threading.Thread(target=body, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        raise errors[0]
    return out


@pytest.mark.parametrize('world', [2, 3])
@pytest.mark.parametrize('with_zi', [False, True])
def test_emulated_shards_are_one_call(world, with_zi):
    sos32, n, x, zi = _case()
    zi = zi if with_zi else None
    want_y, want_zf = emulate(x, sos32, zi)
    for got in _on_threads(world, lambda g, r: _run_rank(g, world, r, sos32, n, x, zi, gather=True)):
        y, zf = got if with_zi else (got, None)
        assert np.array_equal(y.numpy(), want_y)
        if with_zi:
            assert np.array_equal(zf.numpy(), want_zf)


def test_emulated_shards_over_carry_blocks_are_one_call():
    """130 groups = three carry blocks, split over 3 ranks: every rank's start states come from the fold over
    blocks of the gathered list"""
    _, _, H = fourier._sosfilt_geometry(4)
    sos32, n, x, zi = _case(6, groups=2 * H + 2)
    want_y, want_zf = emulate(x, sos32, zi)
    for y, zf in _on_threads(3, lambda g, r: _run_rank(g, 3, r, sos32, n, x, zi, gather=True)):
        assert np.array_equal(y.numpy(), want_y) and np.array_equal(zf.numpy(), want_zf)


def test_emulated_shards_without_gather_concatenate():
    sos32, n, x, zi = _case(5)
    want_y, _ = emulate(x, sos32)
    out = _on_threads(3, lambda g, r: _run_rank(g, 3, r, sos32, n, x, None, gather=False))
    assert np.array_equal(np.concatenate([o.numpy() for o in out]), want_y)


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        sos32, n, x, zi = _case()
        want_y, want_zf = emulate(x, sos32, zi)
        y, zf = _run_rank(None, world, rank, sos32, n, x, zi, gather=True)
        assert np.array_equal(y.numpy(), want_y) and np.array_equal(zf.numpy(), want_zf)
        open(os.path.join(out_dir, f'ok{rank}'), 'w').close()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize('world', [2, 3])
def test_emulated_shards_over_gloo(tmp_path, world):
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    assert all((tmp_path / f'ok{r}').exists() for r in range(world))


def test_workspace_queries_need_no_gpu():
    L, G, H = fourier._sosfilt_geometry(4)
    assert (L, G, H) == (512, 128, 64)
    n = 3 * L * G + 1
    ws = _lib.lib.iqw_sosfilt_workspace_bytes(2, n, 4)
    assert ws == 2 * 4 * G * 8 * 8 + 2 * 4 * 8 * 16 + 2 * 1 * 8 * 16
    assert _lib.lib.iqw_sosfilt_carry_workspace_bytes(2, 65, 4) == 2 * 2 * 8 * 16
    assert _lib.lib.iqw_sosfilt_workspace_bytes(1, 100, 17) == 0
    assert _lib.lib.iqw_sosfilt_geometry(17, (__import__('ctypes').c_int32 * 3)()) == _lib.IQW_ERR_UNSUPPORTED
