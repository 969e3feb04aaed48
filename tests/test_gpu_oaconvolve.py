"""oaconvolve on the GPU against scipy.signal.convolve in float64 (same complex64 samples, same filter):
|y - y64| <= 8 * 2^-24 * log2(nfft) * max_k |fft(h, nfft)_k| * rms(x over the output's block of nfft input
samples).  Roles, modes, per-row filters, layouts, the unaligned view, the error paths, bitwise crops and
run-to-run bit equality, agreement with the direct upfirdn kernel, and time shards (threads on one GPU;
NCCL with >= 2 GPUs)."""
import ctypes
import os
import socket

import numpy as np
import pytest
import scipy.signal as ss
import torch

import iqwaveform_b200 as iqw
from iqwaveform_b200 import _lib, _plan
from iqwaveform_b200 import distributed as D

pytestmark = pytest.mark.gpu

FACTOR = 8


def _signal(rng, shape):
    return (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(np.complex64)


def _taps(rng, M, cplx):
    h = rng.standard_normal(M) + (1j * rng.standard_normal(M) if cplx else 0)
    return h.astype(np.complex64 if cplx else np.float32)


def _bound_1d(x, h, mode, n1, n2):
    M = h.size
    nfft, discard = _plan.oaconvolve_plan(M)
    hop = nfft - discard
    first, n_out = _plan.oaconvolve_window(mode, n1, n2)
    p = np.concatenate([np.zeros(discard), np.abs(x.astype(np.complex128)) ** 2, np.zeros(nfft)])
    cs = np.concatenate([[0.0], np.cumsum(p)])
    b = (first + np.arange(n_out)) // hop
    rms = np.sqrt((cs[b * hop + nfft] - cs[b * hop]) / nfft)
    hmax = np.abs(np.fft.fft(h.astype(np.complex128), nfft)).max()
    return FACTOR * 2.0 ** -24 * np.log2(nfft) * hmax * rms


def _check_1d(got, x, h, mode, x_is_in1=True):
    """got = oaconvolve(x, h, mode) (x_is_in1) or oaconvolve(h, x, mode), 1-D"""
    x64 = x.astype(np.complex128)
    h64 = h.astype(np.complex128 if np.iscomplexobj(h) else np.float64)
    want = ss.convolve(x64, h64, mode=mode) if x_is_in1 else ss.convolve(h64, x64, mode=mode)
    got = np.asarray(got)
    assert got.shape == want.shape and got.dtype == np.complex64
    n1, n2 = (x.size, h.size) if x_is_in1 else (h.size, x.size)
    bound = _bound_1d(x, h, mode, n1, n2)
    err = np.abs(got.astype(np.complex128) - want)
    assert np.all(err <= bound), f'{float(np.max(err / bound)) * FACTOR} bound units'


# one or more filter lengths for each (nfft, nfft/discard) pair the plan picks: 1-2 (16, 16), 3 (16, 8),
# 5 (16, 4), 9 (32, 4), 17 (64, 4), 33 (256, 8), 65 (512, 8), 129 (1024, 8), 161 (2048, 8), 300 (4096, 8),
# 1025 (8192, 8), 2000 (8192, 4), 4097 (8192, 2)
MS = [1, 2, 3, 5, 9, 17, 33, 65, 129, 161, 300, 1025, 2000, 4097]


@pytest.mark.parametrize('cplx', [False, True])
@pytest.mark.parametrize('M', MS)
def test_parity_modes_and_roles(cuda_device, M, cplx):
    rng = np.random.default_rng(M * 2 + cplx)
    h = _taps(rng, M, cplx)
    nfft, _ = _plan.oaconvolve_plan(M)
    for N in sorted({max(M, nfft // 2 + 3), M + 7, 3 * nfft + 11, 200003}):
        x = _signal(rng, N)
        x[N // 3] *= 1000                                  # +60 dB burst
        xd = torch.from_numpy(x).to(cuda_device)
        for mode in ('full', 'same', 'valid'):
            _check_1d(iqw.oaconvolve(xd, h, mode).cpu(), x, h, mode)
            _check_1d(iqw.oaconvolve(h, xd, mode).cpu(), x, h, mode, x_is_in1=False)     # in1 shorter than in2


@pytest.mark.parametrize('M', [161, 4097])
def test_parity_long_capture(cuda_device, M):
    rng = np.random.default_rng(M)
    h = _taps(rng, M, False)
    x = _signal(rng, (1 << 22) + 12345)
    _check_1d(iqw.oaconvolve(torch.from_numpy(x).to(cuda_device), h).cpu(), x, h, 'full')


def test_filters_of_any_dtype_and_residence(cuda_device):
    rng = np.random.default_rng(1)
    x = _signal(rng, 5000)
    xd = torch.from_numpy(x).to(cuda_device)
    h = rng.standard_normal(65)
    ref = iqw.oaconvolve(xd, h)
    _check_1d(ref.cpu(), x, h, 'full')
    for hh in (list(h), torch.from_numpy(h).to(cuda_device), torch.from_numpy(h)):
        assert torch.equal(iqw.oaconvolve(xd, hh), ref)           # the spectrum is float64 either way
    hi = rng.integers(-3, 4, 17)
    _check_1d(iqw.oaconvolve(xd, hi).cpu(), x, hi, 'full')


@pytest.mark.parametrize('M,cplx', [(161, False), (1025, False), (4097, False), (129, True)])
def test_agrees_with_direct_upfirdn(cuda_device, M, cplx):
    rng = np.random.default_rng(M + 5)
    h = _taps(rng, M, cplx)
    x = _signal(rng, 300000)
    xd = torch.from_numpy(x).to(cuda_device)
    got = iqw.oaconvolve(xd, h).cpu().numpy().astype(np.complex128)
    direct = iqw.upfirdn(h, xd).cpu().numpy().astype(np.complex128)
    # both sides within their own bound of the exact result; the FFT side's bound dominates
    bound = _bound_1d(x, h, 'full', x.size, M) + 2.0 ** -24 * (8 + 2 * np.sqrt(M)) * ss.convolve(
        np.abs(x.astype(np.complex128)), np.abs(h.astype(np.complex128)))
    assert np.all(np.abs(got - direct) <= bound)


@pytest.mark.parametrize('M', [1, 33, 161, 1025, 4097])
def test_same_and_valid_are_bitwise_crops_of_full(cuda_device, M):
    rng = np.random.default_rng(M + 9)
    h = _taps(rng, M, True)
    x = torch.from_numpy(_signal(rng, (2, 70001))).to(cuda_device)
    full = iqw.oaconvolve(x, h[None], axes=1)
    for mode in ('same', 'valid'):
        first, n = _plan.oaconvolve_window(mode, 70001, M)
        assert torch.equal(iqw.oaconvolve(x, h[None], mode, axes=1), full[:, first:first + n])
    first, n = _plan.oaconvolve_window('same', M, 70001)
    assert torch.equal(iqw.oaconvolve(h[None], x, 'same', axes=1), full[:1, first:first + n])  # in1 = filter row


@pytest.mark.parametrize('M,cplx', [(2, False), (161, False), (1025, True), (4097, False)])
def test_two_calls_are_bitwise_equal(cuda_device, M, cplx):
    rng = np.random.default_rng(M + 13)
    h = _taps(rng, M, cplx)
    x = torch.from_numpy(_signal(rng, (3, 1 << 17))).to(cuda_device)
    assert torch.equal(iqw.oaconvolve(x, h[None], axes=1), iqw.oaconvolve(x, h[None], axes=1))


def test_per_row_filters(cuda_device):
    rng = np.random.default_rng(17)
    C, N, M = 3, 20000, 200
    x = _signal(rng, (C, N))
    h = np.stack([_taps(rng, M, c == 1) for c in range(C)])
    got = iqw.oaconvolve(torch.from_numpy(x).to(cuda_device), h, 'same', axes=-1).cpu().numpy()
    assert got.shape == ss.oaconvolve(x, h, 'same', axes=-1).shape == (C, N)
    for c in range(C):
        _check_1d(got[c], x[c], h[c], 'same')
    # one filter for all rows, as (1, M) and as the default axes=None with a size-1 row axis
    got = iqw.oaconvolve(torch.from_numpy(x).to(cuda_device), h[1:2]).cpu().numpy()
    for c in range(C):
        _check_1d(got[c], x[c], h[1], 'full')


def test_layouts_and_residence(cuda_device):
    rng = np.random.default_rng(19)
    M = 81
    h = _taps(rng, M, False)
    x2 = _signal(rng, (3, 4000))
    for kind in ('numpy', 'torch_cpu', 'torch_cuda'):
        arg = {'numpy': x2, 'torch_cpu': torch.from_numpy(x2), 'torch_cuda': torch.from_numpy(x2).to(cuda_device)}[kind]
        y = iqw.oaconvolve(arg, h[None], 'valid')
        assert type(y) is (np.ndarray if kind == 'numpy' else torch.Tensor)
        if kind != 'numpy':
            assert y.is_cuda == (kind == 'torch_cuda')
            y = y.cpu()
        for c in range(3):
            _check_1d(np.asarray(y)[c], x2[c], h, 'valid')
    xt = np.ascontiguousarray(x2.T)                                                   # (N, C), axis 0
    y = iqw.oaconvolve(torch.from_numpy(xt).to(cuda_device), h[:, None], axes=0).cpu().numpy()
    assert y.shape == (4000 + M - 1, 3)
    for c in range(3):
        _check_1d(y[:, c], xt[:, c], h, 'full')
    wide = torch.from_numpy(_signal(rng, 9000)).to(cuda_device)                      # strided view
    assert torch.equal(iqw.oaconvolve(wide[::2], h), iqw.oaconvolve(wide[::2].contiguous(), h))
    # in1 the (1, M) filter against a (4, N) signal: 'same' centres on in1's shape, keeping the middle row
    x4 = _signal(rng, (4, 1000))
    got = iqw.oaconvolve(h[None], torch.from_numpy(x4).to(cuda_device), 'same').cpu().numpy()
    want = ss.oaconvolve(h[None].astype(np.float64), x4.astype(np.complex128), 'same')
    assert got.shape == want.shape == (1, M)
    _check_1d(got[0], x4[1], h, 'same', x_is_in1=False)


@pytest.mark.parametrize('M', [33, 161, 4097])
def test_unaligned_channel_view(cuda_device, M):
    """x[..., 1:] of a contiguous (C, N + 1) capture: rows start 8 bytes off 16-byte alignment"""
    rng = np.random.default_rng(23)
    h = _taps(rng, M, False)
    x = _signal(rng, (2, 30001))
    xd = torch.from_numpy(x).to(cuda_device)[:, 1:]
    assert xd.data_ptr() % 16 == 8
    got = iqw.oaconvolve(xd, h[None])
    for c in range(2):
        _check_1d(got[c].cpu(), x[c, 1:], h, 'full')
    assert torch.equal(got, iqw.oaconvolve(xd.contiguous(), h[None]))


def test_errors_on_device_input(cuda_device):
    x = torch.zeros(64, dtype=torch.complex64, device=cuda_device)
    with pytest.raises(ValueError):
        iqw.oaconvolve(x, np.ones((2, 2)))
    with pytest.raises(ValueError):
        iqw.oaconvolve(x, np.ones(3), mode='bogus')
    with pytest.raises(NotImplementedError):
        iqw.oaconvolve(x.to(torch.complex128), np.ones(3))
    with pytest.raises(NotImplementedError):
        iqw.oaconvolve(x.real.contiguous(), np.ones(3))
    with pytest.raises(NotImplementedError):
        iqw.oaconvolve(torch.zeros(5000, dtype=torch.complex64, device=cuda_device), np.ones(4098))
    got = iqw.oaconvolve(x[:0], np.ones(3))
    assert got.is_cuda and got.shape == (0,)


def test_entry_point_status_codes(cuda_device):
    """the C entry point validates nfft, nfft/discard and discard >= n_taps - 1 before any launch"""
    x = torch.zeros(4096, dtype=torch.complex64, device=cuda_device)
    hs = torch.zeros(8192, dtype=torch.complex64, device=cuda_device)
    y = torch.zeros(4096, dtype=torch.complex64, device=cuda_device)
    sp = ctypes.c_void_p(torch.cuda.current_stream(cuda_device).cuda_stream)

    def call(nfft, discard, n_taps, hstride=0):
        return _lib.lib.iqw_oaconvolve_c64(ctypes.c_void_p(x.data_ptr()), 1, 4096, 4096, 0, ctypes.c_void_p(hs.data_ptr()),
                                           hstride, n_taps, nfft, discard, 0, 4096, ctypes.c_void_p(y.data_ptr()), 4096, sp)

    assert call(2048, 256, 161) == _lib.IQW_OK
    assert call(1000, 125, 3) == _lib.IQW_ERR_UNSUPPORTED          # not a power of two
    assert call(16384, 8192, 3) == _lib.IQW_ERR_UNSUPPORTED        # above 8192
    assert call(2048, 96, 3) == _lib.IQW_ERR_UNSUPPORTED           # nfft/discard not a power of two
    assert call(2048, 64, 3) == _lib.IQW_ERR_UNSUPPORTED           # nfft/discard = 32
    assert call(1024, 512, 3) == _lib.IQW_ERR_UNSUPPORTED          # a pair the plan never picks
    assert call(2048, 256, 258) == _lib.IQW_ERR_INVALID            # discard < n_taps - 1
    assert call(2048, 256, 0) == _lib.IQW_ERR_INVALID
    assert call(2048, 256, 161, hstride=5) == _lib.IQW_ERR_INVALID
    torch.cuda.synchronize()


def test_every_planned_pair_is_built(cuda_device):
    """every (nfft, discard) that _plan.oaconvolve_plan returns for 1..4097 taps is instantiated in the
    library: the entry point accepts it with the longest filter the discard admits"""
    pairs = sorted({_plan.oaconvolve_plan(M) for M in range(1, _plan.OACONVOLVE_MAX_TAPS + 1)})
    assert len(pairs) == 13
    x = torch.zeros(20000, dtype=torch.complex64, device=cuda_device)
    y = torch.zeros(20000, dtype=torch.complex64, device=cuda_device)
    sp = ctypes.c_void_p(torch.cuda.current_stream(cuda_device).cuda_stream)
    for nfft, discard in pairs:
        hs = torch.zeros(nfft, dtype=torch.complex64, device=cuda_device)
        rc = _lib.lib.iqw_oaconvolve_c64(ctypes.c_void_p(x.data_ptr()), 1, 20000, 20000, 0, ctypes.c_void_p(hs.data_ptr()),
                                         0, discard + 1, nfft, discard, 0, 20000, ctypes.c_void_p(y.data_ptr()), 20000, sp)
        assert rc == _lib.IQW_OK, (nfft, discard, _lib.lib.iqw_last_error())
    torch.cuda.synchronize()


SHARD_CASES = [(100003, 161), (77777, 1025), (50001, 4097), (5000, 33), (9000, 2)]


@pytest.mark.parametrize('world', [2, 3])
@pytest.mark.parametrize('mode', ['full', 'same', 'valid'])
@pytest.mark.parametrize('n,M', SHARD_CASES)
def test_time_shards_equal_single_call(cuda_device, world, mode, n, M):
    import threading
    rng = np.random.default_rng(n + world)
    h = _taps(rng, M, M == 1025)
    x = torch.from_numpy(_signal(rng, n)).to(cuda_device)
    single = iqw.oaconvolve(x, h, mode)
    group = D.ThreadGroup(world)
    parts = [None] * world

    def run(r):
        sh = D.oaconvolve_shard(n, M, mode, world, r)
        parts[r] = D.oaconvolve_time_sharded(x[sh.sample0:sh.sample1].clone(), h, mode, n_samples=n,
                                             group=group.member(r))
        torch.cuda.synchronize()

    threads = [threading.Thread(target=run, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert torch.equal(torch.cat(parts), single)


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _nccl_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device('cuda', rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=dev)
    try:
        for n, M in SHARD_CASES[:3]:
            rng = np.random.default_rng(n)
            h = _taps(rng, M, False)
            x = torch.from_numpy(_signal(rng, n)).to(dev)
            sh = D.oaconvolve_shard(n, M, 'same', world, rank)
            got = D.oaconvolve_time_sharded(x[sh.sample0:sh.sample1].contiguous(), h, 'same', n_samples=n, gather=True)
            assert torch.equal(got, iqw.oaconvolve(x, h, 'same'))
        open(os.path.join(out_dir, f'ok{rank}'), 'w').close()
    finally:
        dist.destroy_process_group()


def test_time_shards_over_nccl(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip('needs at least 2 GPUs')
    import torch.multiprocessing as mp
    world = 2
    mp.spawn(_nccl_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    assert all((tmp_path / f'ok{r}').exists() for r in range(world))
