"""sosfilt on the GPU against scipy's float64 sosfilt of the same float32 sos: per row, max |y - y64| <= 8 E32 (E32
the error of scipy's complex64 sosfilt) with a floor of a few ulp of max |y64|.  Every built S, lengths around L
and L*G, zi / zf and streaming in pieces, bitwise run-to-run, row-alone-vs-batch and unaligned-view equality,
layouts and residence, the entry point's status codes, and time shards (threads on one GPU; NCCL with >= 2
GPUs), bitwise equal to one call."""
import ctypes
import os
import socket
import threading

import numpy as np
import pytest
import scipy.signal as ss
import torch

import iqwaveform_b200 as iqw
from iqwaveform_b200 import _lib, fourier
from iqwaveform_b200 import distributed as D

from _sosfilt_numpy import FILTERS, ratio, reference, signal, zf_unit

pytestmark = pytest.mark.gpu

FACTOR = 8


def _sos(S, seed):
    """a stable S-section filter: the probe's filters where S matches, else a Butterworth / Chebyshev design"""
    for sos in FILTERS.values():
        if len(sos) == S and seed == 0:
            return sos
    return (ss.butter if seed % 2 else ss.cheby1)(2 * S, *((0.5,) if seed % 2 == 0 else ()),
                                                  0.05 + 0.1 * (S % 5), output='sos')


@pytest.mark.parametrize('S', range(1, 17))
def test_parity_every_built_size(cuda_device, S):
    rng = np.random.default_rng(S)
    L, G, _ = fourier._sosfilt_geometry(S)
    worst = 0.0
    for seed in (0, 1):
        sos32 = fourier._sosfilt_sos(_sos(S, seed))
        for n in (1, L - 1, L + 1, L * G - 1, L * G + 1, 2 * L * G + 3 * L + 5):
            x = np.stack([signal(rng, n), signal(rng, n, burst=False)])
            y = iqw.sosfilt(sos32, torch.from_numpy(x).to(cuda_device)).cpu().numpy()
            y64, e32 = reference(x, sos32)
            assert y.dtype == np.complex64 and y.shape == x.shape
            for r in range(2):
                worst = max(worst, ratio(y[r], y64[r], e32[r]))
                assert worst <= FACTOR, (S, seed, n, r)
    print(f'S = {S}: worst {worst:.2f} units')


@pytest.mark.parametrize('name', ['ellip8', 'butter32'])
def test_parity_over_carry_blocks(cuda_device, name):
    """rows of H + 1 groups, beyond one carry block: the block folds, the fold over blocks with A^(LGH) from each
    row's zi, and each block's expansion of its groups' start states all reach y and zf"""
    rng = np.random.default_rng(12)
    sos32 = fourier._sosfilt_sos(FILTERS[name])
    S = len(sos32)
    L, G, H = fourier._sosfilt_geometry(S)
    n = (H + 1) * L * G + 17
    x = np.stack([signal(rng, n), signal(rng, n, burst=False)])
    zi = (rng.standard_normal((S, 2, 2)) + 1j * rng.standard_normal((S, 2, 2))).astype(np.complex64)
    y, zf = iqw.sosfilt(sos32, torch.from_numpy(x).to(cuda_device), zi=torch.from_numpy(zi).to(cuda_device))
    y, zf = y.cpu().numpy(), zf.cpu().numpy()
    worst = [0.0, 0.0]
    for r in range(2):
        y64, e32, zf64, zf32 = reference(x[r], sos32, zi[:, r])
        worst[0] = max(worst[0], ratio(y[r], y64, e32))
        worst[1] = max(worst[1], ratio(zf[:, r].reshape(-1), zf64.reshape(-1), zf_unit(zf32, zf64, e32)))
        assert max(worst) <= FACTOR, (name, r, worst)
    print(f'{name} over {H + 1} groups: worst y {worst[0]:.2f} / zf {worst[1]:.2f} units')


@pytest.mark.parametrize('name', sorted(FILTERS))
def test_zi_zf_and_pieces(cuda_device, name):
    rng = np.random.default_rng(7)
    sos32 = fourier._sosfilt_sos(FILTERS[name])
    S = len(sos32)
    L, G, _ = fourier._sosfilt_geometry(S)
    n = 3 * L * G + 999
    x = signal(rng, n)
    zi = (rng.standard_normal((S, 2)) + 1j * rng.standard_normal((S, 2))).astype(np.complex64)
    y, zf = iqw.sosfilt(sos32, x, zi=zi)
    y64, e32, zf64, zf32 = reference(x, sos32, zi)
    assert ratio(y, y64, e32) <= FACTOR
    assert zf.shape == (S, 2) and zf.dtype == np.complex64
    assert ratio(zf.reshape(-1), zf64.reshape(-1), zf_unit(zf32, zf64, e32)) <= FACTOR
    # two calls with zf -> zi against one call
    cut = L * G + 12345
    ya, za = iqw.sosfilt(sos32, x[:cut], zi=zi)
    yb, zb = iqw.sosfilt(sos32, x[cut:], zi=za)
    assert ratio(np.concatenate([ya, yb]), y64, e32) <= FACTOR
    assert ratio(zb.reshape(-1), zf64.reshape(-1), zf_unit(zf32, zf64, e32)) <= FACTOR
    print(f'{name}: y {ratio(y, y64, e32):.2f} / zf {ratio(zf.reshape(-1), zf64.reshape(-1), zf_unit(zf32, zf64, e32)):.2f}'
          f' / two pieces {ratio(np.concatenate([ya, yb]), y64, e32):.2f} units')


def test_bitwise_repeat_batch_and_unaligned(cuda_device):
    rng = np.random.default_rng(8)
    sos32 = fourier._sosfilt_sos(FILTERS['ellip8'])
    n = 300001
    x = torch.from_numpy(np.stack([signal(rng, n + 1) for _ in range(5)])).to(cuda_device)
    a = iqw.sosfilt(sos32, x)
    assert torch.equal(a, iqw.sosfilt(sos32, x))
    for r in range(5):
        assert torch.equal(iqw.sosfilt(sos32, x[r]), a[r])
    view = x[:, 1:]                                  # starts one sample in: unaligned rows, row pitch n + 1
    assert torch.equal(iqw.sosfilt(sos32, view), iqw.sosfilt(sos32, view.contiguous()))
    # the coefficients in any memory order
    sos = FILTERS['ellip8']
    for other in (np.asfortranarray(sos), torch.from_numpy(np.ascontiguousarray(sos.T)).T.to(cuda_device)):
        assert torch.equal(iqw.sosfilt(other, x), a)


def test_layouts_and_residence(cuda_device):
    """every layout and residence gives the bits of the same rows filtered as a (rows, N) CUDA tensor"""
    rng = np.random.default_rng(9)
    sos32 = fourier._sosfilt_sos(FILTERS['butter4'])
    x = (rng.standard_normal((3, 5000, 2)) + 1j * rng.standard_normal((3, 5000, 2))).astype(np.complex64)
    zi = (rng.standard_normal((2, 3, 2, 2)) + 1j * rng.standard_normal((2, 3, 2, 2))).astype(np.complex64)
    rows = np.moveaxis(x, 1, -1).reshape(6, 5000)
    zrows = np.moveaxis(zi, (0, 2), (-2, -1)).reshape(6, 2, 2).transpose(1, 0, 2)
    yc, zc = iqw.sosfilt(sos32, torch.from_numpy(rows).to(cuda_device), zi=torch.from_numpy(zrows).to(cuda_device))
    yc, zc = yc.cpu().numpy(), zc.cpu().numpy()
    for kind in ('numpy', 'cpu', 'cuda'):
        xin = x if kind == 'numpy' else torch.from_numpy(x).to('cpu' if kind == 'cpu' else cuda_device)
        zin = zi if kind == 'numpy' else torch.from_numpy(zi).to(xin.device)
        y, zf = iqw.sosfilt(sos32, xin, axis=1, zi=zin)
        assert type(y) is type(xin) and type(zf) is type(xin)
        if kind != 'numpy':
            assert y.is_cuda == zf.is_cuda == (kind == 'cuda')
            y, zf = y.cpu().numpy(), zf.cpu().numpy()
        assert y.shape == x.shape and zf.shape == zi.shape
        assert np.array_equal(np.moveaxis(y, 1, -1).reshape(6, 5000), yc)
        assert np.array_equal(np.moveaxis(zf, (0, 2), (-2, -1)).reshape(6, 2, 2).transpose(1, 0, 2), zc)
    y0 = iqw.sosfilt(sos32, x, axis=0)
    assert np.array_equal(np.moveaxis(y0, 0, -1), iqw.sosfilt(sos32, np.ascontiguousarray(np.moveaxis(x, 0, -1))))
    # empty time axis: empty y, zf = zi
    y, zf = iqw.sosfilt(sos32, np.zeros((3, 0), np.complex64), zi=np.ones((2, 3, 2), np.complex64))
    assert y.shape == (3, 0) and np.array_equal(zf, np.ones((2, 3, 2), np.complex64))


def test_entry_point_status_codes(cuda_device):
    sos = np.asarray(ss.butter(2, 0.1, output='sos'), np.float32)
    x = torch.zeros(1000, dtype=torch.complex64, device=cuda_device)
    y = torch.empty_like(x)
    powers = fourier._sosfilt_powers(sos, cuda_device)
    ws_bytes = _lib.lib.iqw_sosfilt_workspace_bytes(1, 1000, 1)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=cuda_device)
    s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: ctypes.c_void_p(t.data_ptr())     # noqa: E731

    def call(sos_arr=sos, S=1, nbytes=ws_bytes, wsp=None, rows=1):
        return _lib.lib.iqw_sosfilt_c64(p(x), rows, 1000, 1000, sos_arr.ctypes.data_as(ctypes.c_void_p), S,
                                        p(powers), None, p(y), 1000, None, wsp or p(ws), nbytes, s)
    assert call() == _lib.IQW_OK
    assert call(S=17) == _lib.IQW_ERR_UNSUPPORTED
    assert call(S=0) == _lib.IQW_ERR_UNSUPPORTED
    bad = sos.copy()
    bad[0, 3] = 2
    assert call(sos_arr=bad) == _lib.IQW_ERR_INVALID
    assert call(nbytes=ws_bytes - 1) == _lib.IQW_ERR_WORKSPACE
    assert call(wsp=ctypes.c_void_p(ws.data_ptr() + 8)) == _lib.IQW_ERR_INVALID
    assert call(rows=-1) == _lib.IQW_ERR_INVALID
    assert call(rows=70000) == _lib.IQW_ERR_UNSUPPORTED
    assert 'sosfilt' in _lib.lib.iqw_last_error().decode()
    torch.cuda.synchronize()


def _sharded_case(cuda_device):
    sos32 = fourier._sosfilt_sos(FILTERS['ellip16'])
    L, G, H = fourier._sosfilt_geometry(len(sos32))
    n = (2 * H + 3) * L * G + 4321                  # three carry blocks
    x = torch.from_numpy(signal(np.random.default_rng(10), n)).to(cuda_device)
    zi = torch.full((len(sos32), 2), 0.5 + 0.25j, dtype=torch.complex64, device=cuda_device)
    return sos32, n, x, zi


@pytest.mark.parametrize('world', [2, 3, 5])
def test_time_shards_on_threads_are_one_call(cuda_device, world):
    sos32, n, x, zi = _sharded_case(cuda_device)
    want_y, want_zf = iqw.sosfilt(sos32, x, zi=zi)
    tg = D.ThreadGroup(world)
    out, errors = [None] * world, []

    def body(r):
        try:
            sh = D.sosfilt_shard(n, len(sos32), world, r)
            out[r] = D.sosfilt_time_sharded(x[sh.sample0:sh.sample1], sos32, n_samples=n, zi=zi, group=tg.member(r),
                                            gather=True)
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
    for y, zf in out:
        assert torch.equal(y, want_y) and torch.equal(zf, want_zf)


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _nccl_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=torch.device('cuda', rank))
    try:
        dev = torch.device('cuda', rank)
        sos32, n, x, zi = _sharded_case(dev)
        want_y, want_zf = iqw.sosfilt(sos32, x, zi=zi)
        sh = D.sosfilt_shard(n, len(sos32), world, rank)
        y, zf = D.sosfilt_time_sharded(x[sh.sample0:sh.sample1], sos32, n_samples=n, zi=zi, gather=True)
        assert torch.equal(y, want_y) and torch.equal(zf, want_zf)
        open(os.path.join(out_dir, f'ok{rank}'), 'w').close()
    finally:
        dist.destroy_process_group()


def test_time_shards_over_nccl_are_one_call(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    import torch.multiprocessing as mp
    world = min(torch.cuda.device_count(), 4)
    mp.spawn(_nccl_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    assert all((tmp_path / f'ok{r}').exists() for r in range(world))
