"""upfirdn on the GPU against scipy.signal.upfirdn in float64 (same float32-rounded taps, same complex64
samples): |y - y64| <= 2^-24 * (8 + 2*sqrt(Lp)) * upfirdn(|h|, |x|).  Layouts, the unaligned path, the
error paths, run-to-run bit equality and time shards (threads on one GPU; NCCL with >= 2 GPUs)."""
import os
import socket

import numpy as np
import pytest
import scipy.signal as ss
import torch

import iqwaveform_b200 as iqw
from iqwaveform_b200 import distributed as D

pytestmark = pytest.mark.gpu


def _signal(rng, shape):
    x = rng.standard_normal(shape) + 1j * rng.standard_normal(shape)
    return x.astype(np.complex64)


def _taps(rng, L, cplx):
    h = rng.standard_normal(L) + (1j * rng.standard_normal(L) if cplx else 0)
    return h.astype(np.complex64 if cplx else np.float32)


def _check(got, h, x, up, down, axis=-1):
    """the documented bound, per element"""
    h64 = h.astype(np.complex128 if np.iscomplexobj(h) else np.float64)
    x64 = x.astype(np.complex128)
    want = ss.upfirdn(h64, x64, up, down, axis=axis)
    scale = ss.upfirdn(np.abs(h64), np.abs(x64), up, down, axis=axis)
    lp = -(-h.size // up)
    got = np.asarray(got)
    assert got.shape == want.shape and got.dtype == np.complex64
    err = np.abs(got.astype(np.complex128) - want)
    bound = 2.0 ** -24 * (8 + 2 * np.sqrt(lp)) * scale
    worst = float(np.max(err - bound)) if err.size else 0.0
    assert worst <= 0.0, f'{float(np.max(err / np.maximum(bound, 1e-300)))} bound units'


UPS = [1, 2, 3, 4, 147]
DOWNS = [1, 2, 8, 16, 160]


@pytest.mark.parametrize('cplx', [False, True])
@pytest.mark.parametrize('down', DOWNS)
@pytest.mark.parametrize('up', UPS)
def test_parity_grid(cuda_device, up, down, cplx):
    rng = np.random.default_rng(up * 1000 + down + cplx)
    for L in (1, 5, 33, 161, 1024):
        h = _taps(rng, L, cplx)
        for n in (3, 700, 5000):              # shorter and longer than the filter
            x = _signal(rng, n)
            _check(iqw.upfirdn(h, torch.from_numpy(x).to(cuda_device), up, down).cpu(), h, x, up, down)


@pytest.mark.parametrize('L,up,down,cplx', [(16384, 1, 16, False), (16384, 147, 160, False), (16384, 3, 1, False),
                                            (8192, 1, 1, True), (8192, 4, 1, True), (4097, 1, 16, False),
                                            (3201, 147, 160, False), (8192, 147, 160, True)])
def test_parity_long_filters(cuda_device, L, up, down, cplx):
    rng = np.random.default_rng(L + up + down)
    h = _taps(rng, L, cplx)
    x = _signal(rng, 40000)
    x[12345] *= 1e4                            # +80 dB burst
    _check(iqw.upfirdn(h, torch.from_numpy(x).to(cuda_device), up, down).cpu(), h, x, up, down)


def test_large_decimation_and_interpolation(cuda_device):
    rng = np.random.default_rng(5)
    x = _signal(rng, 20000)
    for up, down, L in ((1, 1000, 2001), (1000, 1, 3000), (7, 999, 64), (999, 7, 5000)):
        h = _taps(rng, L, False)
        _check(iqw.upfirdn(h, torch.from_numpy(x).to(cuda_device), up, down).cpu(), h, x, up, down)


def test_layouts_and_residence(cuda_device):
    rng = np.random.default_rng(7)
    h = _taps(rng, 61, False)
    up, down = 3, 2
    x2 = _signal(rng, (3, 1000))
    for kind in ('numpy', 'torch_cpu', 'torch_cuda'):
        arg = {'numpy': x2, 'torch_cpu': torch.from_numpy(x2), 'torch_cuda': torch.from_numpy(x2).to(cuda_device)}[kind]
        y = iqw.upfirdn(h, arg, up, down, axis=1)
        assert type(y) is (np.ndarray if kind == 'numpy' else torch.Tensor)
        if kind != 'numpy':
            assert y.is_cuda == (kind == 'torch_cuda')
            y = y.cpu()
        _check(y, h, x2, up, down, axis=1)
    _check(iqw.upfirdn(h, x2[0], up, down), h, x2[0], up, down)                    # 1-D
    xt = np.ascontiguousarray(x2.T)                                                 # (N, C), axis 0
    _check(iqw.upfirdn(h, torch.from_numpy(xt).to(cuda_device), up, down, axis=0).cpu(), h, xt, up, down, axis=0)
    x3 = _signal(rng, (2, 500, 3))                                                  # 3-D, middle axis
    _check(iqw.upfirdn(h, torch.from_numpy(x3).to(cuda_device), up, down, axis=1).cpu(), h, x3, up, down, axis=1)
    h64 = h.astype(np.float64)                    # any float dtype of taps: rounded to float32 once
    assert torch.equal(iqw.upfirdn(h64, torch.from_numpy(x2).to(cuda_device), up, down),
                       iqw.upfirdn(h, torch.from_numpy(x2).to(cuda_device), up, down))


@pytest.mark.parametrize('up,down,L', [(1, 8, 161), (147, 160, 3201), (1, 1, 129)])
def test_unaligned_channel_view(cuda_device, up, down, L):
    """x[..., 1:] of a contiguous (C, N + 1) capture: rows start 8 bytes off 16-byte alignment"""
    rng = np.random.default_rng(11)
    h = _taps(rng, L, False)
    x = _signal(rng, (2, 3001))
    xd = torch.from_numpy(x).to(cuda_device)[:, 1:]
    assert xd.data_ptr() % 16 == 8
    got = iqw.upfirdn(h, xd, up, down)
    _check(got.cpu(), h, x[:, 1:], up, down)
    assert torch.equal(got, iqw.upfirdn(h, xd.contiguous(), up, down))


def test_errors_on_device_input(cuda_device):
    x = torch.zeros(64, dtype=torch.complex64, device=cuda_device)
    with pytest.raises(ValueError):
        iqw.upfirdn(np.ones((2, 2)), x)
    with pytest.raises(ValueError):
        iqw.upfirdn(np.ones(0), x)
    with pytest.raises(ValueError):
        iqw.upfirdn(np.ones(3), x, 0, 1)
    with pytest.raises(ValueError):
        iqw.upfirdn(np.ones(3), x, 1, 0)
    with pytest.raises(ValueError):
        iqw.upfirdn(np.ones(3), x, mode='bogus')
    with pytest.raises(NotImplementedError):
        iqw.upfirdn(np.ones(3), x, mode='reflect')
    with pytest.raises(NotImplementedError):
        iqw.upfirdn(np.ones(3), x, cval=2)
    with pytest.raises(NotImplementedError):
        iqw.upfirdn(np.ones(3), x.to(torch.complex128))
    with pytest.raises(NotImplementedError):
        iqw.upfirdn(np.ones(3), x.real.contiguous())
    with pytest.raises(NotImplementedError):
        iqw.upfirdn(np.ones(32769), x)
    with pytest.raises(ValueError):
        iqw.upfirdn(np.ones(3), x, axis=2)


@pytest.mark.parametrize('up,down,L,cplx', [(1, 8, 161, False), (147, 160, 3201, False), (4, 1, 81, False),
                                            (1, 1, 129, True), (3, 7, 2000, False)])
def test_two_calls_are_bitwise_equal(cuda_device, up, down, L, cplx):
    rng = np.random.default_rng(13)
    h = _taps(rng, L, cplx)
    x = torch.from_numpy(_signal(rng, (2, 1 << 16))).to(cuda_device)
    assert torch.equal(iqw.upfirdn(h, x, up, down), iqw.upfirdn(h, x, up, down))


# (n, L, up, down): uneven splits; 147/160 and 3/2 shards start mid-way through the phase cycle
SHARD_CASES = [(100003, 161, 1, 8), (77777, 3201, 147, 160), (50001, 81, 4, 1), (60000, 129, 1, 1),
               (40000, 4097, 1, 16), (33333, 31, 3, 2), (20011, 2000, 160, 147)]


@pytest.mark.parametrize('world', [2, 3])
@pytest.mark.parametrize('n,L,up,down', SHARD_CASES)
def test_time_shards_equal_single_call(cuda_device, world, n, L, up, down):
    import threading
    rng = np.random.default_rng(n + world)
    h = _taps(rng, L, up == 1 and down == 1)
    x = torch.from_numpy(_signal(rng, n)).to(cuda_device)
    single = iqw.upfirdn(h, x, up, down)
    group = D.ThreadGroup(world)
    parts = [None] * world
    starts = []

    def run(r):
        sh = D.upfirdn_shard(n, L, up, down, world, r)
        parts[r] = D.upfirdn_time_sharded(x[sh.sample0:sh.sample1].clone(), h, up, down, n_samples=n,
                                          group=group.member(r))
        torch.cuda.synchronize()

    for r in range(world):
        starts.append(D.upfirdn_shard(n, L, up, down, world, r).out0)
    threads = [threading.Thread(target=run, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if up > 1:
        assert any((s * down) % up for s in starts[1:]), 'some shard must start off phase 0'
    assert torch.equal(torch.cat(parts), single)


@pytest.mark.parametrize('n,L,up,down', [SHARD_CASES[0], SHARD_CASES[1], SHARD_CASES[5]])
def test_time_shards_of_strided_halos(cuda_device, n, L, up, down):
    """shards taken as a column of an (N, C) capture, and as a step-2 view, are not unit-stride rows: the result
    is still bitwise the single call on the same samples"""
    rng = np.random.default_rng(n + 17)
    h = _taps(rng, L, False)
    cap = torch.from_numpy(_signal(rng, (n, 3))).to(cuda_device)
    col = cap[:, 1]
    single = iqw.upfirdn(h, col.contiguous(), up, down)
    wide = torch.from_numpy(_signal(rng, 2 * n)).to(cuda_device)
    single_wide = iqw.upfirdn(h, wide[::2].contiguous(), up, down)
    world = 3
    parts, parts_wide = [], []
    for r in range(world):
        sh = D.upfirdn_shard(n, L, up, down, world, r)
        halo = col[sh.sample0:sh.sample1]
        assert halo.numel() < 2 or halo.stride(0) == 3
        parts.append(D.upfirdn_time_sharded(halo, h, up, down, n_samples=n, group=D.ThreadGroup(world).member(r)))
        halo = wide[::2][sh.sample0:sh.sample1]
        parts_wide.append(D.upfirdn_time_sharded(halo, h, up, down, n_samples=n,
                                                 group=D.ThreadGroup(world).member(r)))
    assert torch.equal(torch.cat(parts), single)
    assert torch.equal(torch.cat(parts_wide), single_wide)


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
        for n, L, up, down in SHARD_CASES[:3]:
            rng = np.random.default_rng(n)
            h = _taps(rng, L, False)
            x = torch.from_numpy(_signal(rng, n)).to(dev)
            sh = D.upfirdn_shard(n, L, up, down, world, rank)
            got = D.upfirdn_time_sharded(x[sh.sample0:sh.sample1].contiguous(), h, up, down, n_samples=n, gather=True)
            assert torch.equal(got, iqw.upfirdn(h, x, up, down))
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
