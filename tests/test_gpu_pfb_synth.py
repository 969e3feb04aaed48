"""pfb_synthesize on the GPU against the float64 factorisation of the same float32 taps and complex64 frames:
|xr - xr64| <= 8 * 2^-24 * (log2 K + Q) * S(t).  Every built K with several prototype lengths and hops, the
adjoint identity against the device pfb_channelize, round-trip reconstruction, excision of a channel, layouts,
the unaligned view, residence, run-to-run bit equality, the entry point's status codes, and time shards
(threads on one GPU; NCCL with >= 2 GPUs)."""
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

from _pfb_numpy import prototype
from _pfb_synth_numpy import fact64, norm, recipe, snr_db

pytestmark = pytest.mark.gpu

FACTOR = 8
KS = [1 << j for j in range(4, 14)]


def _frames(rng, T, K, burst=True):
    y = (rng.standard_normal((T, K)) + 1j * rng.standard_normal((T, K))).astype(np.complex64)
    if burst:
        y[T // 2] *= 1000
    return y


def _check(xr, y, g, hop):
    """xr against the float64 factorisation within FACTOR units of the bound; returns the worst ratio"""
    xr = xr.cpu().numpy() if isinstance(xr, torch.Tensor) else np.asarray(xr)
    K = y.shape[1]
    taps = _plan.pfb_taps(g, K)
    want = fact64(y, np.asarray(g, np.float32).astype(np.float64), hop)
    assert xr.shape == want.shape and xr.dtype == np.complex64
    nrm = norm(y, taps, np.size(g), hop)
    assert np.all(xr[nrm == 0] == 0)
    r = float((np.abs(xr - want)[nrm > 0] / nrm[nrm > 0]).max())
    assert r <= FACTOR, (K, np.size(g), hop, r)
    return r


@pytest.mark.parametrize('K', KS)
def test_parity_every_built_size(cuda_device, K):
    rng = np.random.default_rng(K)
    odd = K // 2 + 1 if K // 2 % 2 == 0 else K // 2
    worst = 0.0
    for Lg in (K, 2 * K - K // 3, 8 * K, 16 * K):
        if Lg > _plan.PFB_MAX_TAPS:
            continue
        g = prototype(Lg, K).astype(np.float32)
        for hop in (K, K // 2, 3 * K // 4, odd) + ((1,) if K <= 64 and Lg <= 8 * K else ()):
            Q = -(-Lg // hop)
            y = _frames(rng, 2 * Q + 3, K)
            xr = iqw.pfb_synthesize(torch.from_numpy(y).to(cuda_device), g, hop)
            worst = max(worst, _check(xr, y, g, hop))
    print(f'K={K}: worst {worst:.3f} units of 2^-24 (log2 K + Q) S(t)')


@pytest.mark.parametrize('K,L,hop', [(64, 512, 64), (256, 2048, 128), (1024, 8192, 768), (16, 100, 5)])
def test_adjoint_of_the_device_analysis_bank(cuda_device, K, L, hop):
    """<A x, y> = <x, A^H y> with A = pfb_channelize(., h) and A^H = pfb_synthesize(., h), float64 products"""
    rng = np.random.default_rng(K + hop)
    h = prototype(L, K)
    n = L + 60 * hop
    x = torch.from_numpy((rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)).to(cuda_device)
    Ax = iqw.pfb_channelize(x, h, K, hop)
    y = torch.from_numpy(_frames(rng, Ax.shape[0], K, burst=False)).to(cuda_device)
    AHy = iqw.pfb_synthesize(y, h, hop)
    lhs = torch.vdot(y.flatten().to(torch.complex128), Ax.flatten().to(torch.complex128)).item()
    rhs = torch.vdot(AHy.to(torch.complex128), x[:AHy.shape[0]].to(torch.complex128)).item()
    assert abs(lhs - rhs) <= 1e-5 * abs(lhs)


@pytest.mark.parametrize('K', [64, 1024, 4096])
def test_round_trip_recipe(cuda_device, K):
    h, g, hop = recipe(K)
    rng = np.random.default_rng(K)
    n = 40 * 8 * K
    x = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
    xr = iqw.pfb_synthesize(iqw.pfb_channelize(torch.from_numpy(x).to(cuda_device), h, K, hop), g, hop)
    s = snr_db(x, xr.cpu().numpy(), 8 * K)
    print(f'K={K}: round trip {s:.1f} dB')
    assert s >= 78


def test_round_trip_root_hann(cuda_device):
    K = 256
    w = np.sqrt(ss.windows.hann(K, sym=False))
    x = (np.random.default_rng(2).standard_normal((2, 50000)) * [[1], [1j]]).astype(np.complex64)
    xr = iqw.pfb_synthesize(iqw.pfb_channelize(x, w, K, K // 2), w / K, K // 2)
    assert xr.shape[0] == 2 and isinstance(xr, np.ndarray)
    for c in range(2):
        assert snr_db(x[c], xr[c], K) >= 110


@pytest.mark.parametrize('K', [64, 1024])
def test_excision_of_a_channel(cuda_device, K):
    """a tone at the centre of channel k0: zeroing column k0 leaves it below -80 dB of its amplitude"""
    h, g, hop = recipe(K)
    n = np.arange(30 * 8 * K)
    k0 = K // 2 + 5
    A = 30.0
    tone = A * np.exp(2j * np.pi * ((k0 - K // 2) * n % K) / K)
    rng = np.random.default_rng(K)
    x = (tone + rng.standard_normal(n.size) + 1j * rng.standard_normal(n.size)).astype(np.complex64)
    y = iqw.pfb_channelize(torch.from_numpy(x).to(cuda_device), h, K, hop)
    y[:, k0] = 0
    xr = iqw.pfb_synthesize(y, g, hop).cpu().numpy().astype(np.complex128)
    s, e = 8 * K, xr.size - 8 * K
    left = np.abs(np.vdot(tone[s:e], xr[s:e])) / np.vdot(tone[s:e], tone[s:e]).real
    assert 20 * np.log10(left) <= -80


def test_layouts_and_residence(cuda_device):
    rng = np.random.default_rng(7)
    K, Lg, hop, T = 256, 1024, 128, 40
    g = prototype(Lg, K)
    y = (rng.standard_normal((3, 4, T, K)) + 1j * rng.standard_normal((3, 4, T, K))).astype(np.complex64)
    ref = np.stack([np.stack([iqw.pfb_synthesize(y[i, j], g, hop) for j in range(4)]) for i in range(3)])
    n_out = _plan.pfb_synth_len(T, Lg, hop)
    assert ref.shape == (3, 4, n_out)
    _check(ref[1, 2], y[1, 2], g, hop)
    got = iqw.pfb_synthesize(y, g, hop)                                         # 4-D numpy in, numpy out
    assert isinstance(got, np.ndarray)
    np.testing.assert_array_equal(got, ref)
    got = iqw.pfb_synthesize(torch.from_numpy(y), torch.from_numpy(g), hop)      # CPU torch in and out
    assert isinstance(got, torch.Tensor) and not got.is_cuda
    np.testing.assert_array_equal(got.numpy(), ref)
    yt = torch.from_numpy(np.ascontiguousarray(np.moveaxis(y, (2, 3), (0, 1)))).to(cuda_device)   # (T, K, 3, 4)
    got = iqw.pfb_synthesize(yt, g, hop, axis=0)
    assert got.is_cuda and got.shape == (n_out, 3, 4)
    np.testing.assert_array_equal(np.moveaxis(got.cpu().numpy(), 0, 2), ref)
    y1 = torch.from_numpy(np.ascontiguousarray(np.moveaxis(y[0], 0, 2))).to(cuda_device)   # (T, K, 4), axis -3
    got = iqw.pfb_synthesize(y1, g, hop, axis=-3)
    np.testing.assert_array_equal(np.moveaxis(got.cpu().numpy(), 1, 0), ref[0])
    empty = iqw.pfb_synthesize(np.zeros((0, T, K), np.complex64), g, hop)
    assert empty.shape == (0, n_out)
    # the round trip with the defaults keeps the layout of the capture
    x = torch.from_numpy(np.ascontiguousarray(rng.standard_normal((5000, 3)).astype(np.complex64))).to(cuda_device)
    assert iqw.pfb_synthesize(iqw.pfb_channelize(x, g, K, hop, axis=0), g, hop, axis=0).shape == (4992, 3)


@pytest.mark.parametrize('K,Lg,hop', [(64, 512, 64), (1024, 8192, 512), (16, 100, 5)])
def test_unaligned_view(cuda_device, K, Lg, hop):
    """frames that start 8 bytes past a 16-byte boundary"""
    rng = np.random.default_rng(K)
    T = 30
    flat = torch.from_numpy((rng.standard_normal(3 * T * K + 1) + 1j * rng.standard_normal(3 * T * K + 1))
                            .astype(np.complex64)).to(cuda_device)
    v = flat[1:].view(3, T, K)
    assert v.data_ptr() % 16 == 8
    g = prototype(Lg, K)
    got = iqw.pfb_synthesize(v, g, hop)
    assert torch.equal(got, iqw.pfb_synthesize(v.clone(), g, hop))
    _check(got[2], v[2].cpu().numpy(), g, hop)


@pytest.mark.parametrize('K,hop', [(1024, 1024), (1024, 512), (64, 37), (8192, 8192), (16, 1)])
def test_two_calls_are_bitwise_equal(cuda_device, K, hop):
    Lg = min(8 * K, _plan.PFB_MAX_TAPS)
    y = torch.from_numpy(_frames(np.random.default_rng(K), 300, K)).to(cuda_device)
    g = prototype(Lg, K)
    assert torch.equal(iqw.pfb_synthesize(y, g, hop), iqw.pfb_synthesize(y, g, hop))


def test_errors_on_device_input(cuda_device):
    y = torch.zeros((8, 64), dtype=torch.complex64, device=cuda_device)
    with pytest.raises(NotImplementedError, match='complex64'):
        iqw.pfb_synthesize(y.to(torch.complex128), np.ones(64))
    with pytest.raises(NotImplementedError, match='complex prototypes'):
        iqw.pfb_synthesize(y, torch.ones(64, dtype=torch.complex64, device=cuda_device))
    got = iqw.pfb_synthesize(y, torch.ones(64, device=cuda_device))            # taps on the device
    assert got.is_cuda and got.shape == (7 * 64 + 64,)


def test_entry_point_status_codes(cuda_device):
    """the C entry point validates K, the prototype's limits, hop, the output and frame ranges, pointers, strides
    and the workspace before any launch"""
    y = torch.zeros(1 << 16, dtype=torch.complex64, device=cuda_device)
    t = torch.zeros(32768, dtype=torch.float32, device=cuda_device)
    out = torch.zeros(1 << 16, dtype=torch.complex64, device=cuda_device)
    ws = torch.zeros(1 << 19, dtype=torch.uint8, device=cuda_device)
    sp = ctypes.c_void_p(torch.cuda.current_stream(cuda_device).cuda_stream)
    P = ctypes.c_void_p

    def call(n_taps=256, nfft=64, hop=64, n_frames=10, frame_first=0, T=10, out_first=0, n_out=None, C=1,
             y_stride=None, out_stride=None, ws_bytes=None, yp=y, tp=t, op=out, wp=ws):
        n_out = (T - 1) * hop + n_taps - out_first if n_out is None else n_out
        ws_bytes = _lib.lib.iqw_pfb_synthesize_workspace_bytes(C, n_frames, nfft) if ws_bytes is None else ws_bytes
        return _lib.lib.iqw_pfb_synthesize_c64(
            P(yp.data_ptr() if yp is not None else None), C, n_frames,
            n_frames * nfft if y_stride is None else y_stride, frame_first, T,
            P(tp.data_ptr() if tp is not None else None), n_taps, nfft, hop, out_first, n_out,
            P(op.data_ptr() if op is not None else None), n_out if out_stride is None else out_stride,
            P(wp.data_ptr() if wp is not None else None), ws_bytes, sp)

    assert _lib.lib.iqw_pfb_synthesize_workspace_bytes(3, 10, 64) == 3 * 10 * 64 * 8
    assert call() == _lib.IQW_OK
    assert call(n_out=(10 - 1) * 64 + 257) == _lib.IQW_ERR_INVALID          # past (T - 1) hop + Lg
    assert call(n_frames=9) == _lib.IQW_ERR_INVALID                         # the last output needs frame 9
    assert call(n_frames=9, n_out=9 * 64) == _lib.IQW_OK                    # ... which [0, 576) does not
    assert call(n_frames=3, frame_first=7, out_first=576) == _lib.IQW_ERR_INVALID   # [576, 832) needs frames 6..9
    assert call(n_frames=4, frame_first=6, out_first=576) == _lib.IQW_OK
    assert call(n_frames=0, frame_first=1, T=2, n_taps=10, out_first=12, n_out=40, yp=None, wp=None) == _lib.IQW_OK
    assert call(n_frames=3, frame_first=8) == _lib.IQW_ERR_INVALID          # frames past T
    assert call(nfft=1000, hop=1000) == _lib.IQW_ERR_UNSUPPORTED            # not a power of two
    assert call(nfft=8, hop=8) == _lib.IQW_ERR_UNSUPPORTED                  # below 16
    assert call(nfft=16384, hop=16384) == _lib.IQW_ERR_UNSUPPORTED          # above 8192
    assert call(n_taps=16 * 64 + 1) == _lib.IQW_ERR_UNSUPPORTED             # 17 segments
    assert call(n_taps=32769, nfft=4096, hop=4096, n_frames=1, T=1) == _lib.IQW_ERR_UNSUPPORTED
    assert call(n_taps=0) == _lib.IQW_ERR_INVALID
    assert call(hop=0) == _lib.IQW_ERR_INVALID
    assert call(hop=65) == _lib.IQW_ERR_INVALID
    assert call(n_frames=-1) == _lib.IQW_ERR_INVALID
    assert call(T=0, n_frames=0, n_out=1) == _lib.IQW_ERR_INVALID
    assert call(yp=None) == _lib.IQW_ERR_INVALID
    assert call(tp=None) == _lib.IQW_ERR_INVALID
    assert call(op=None) == _lib.IQW_ERR_INVALID
    assert call(wp=None) == _lib.IQW_ERR_INVALID
    assert call(C=2, y_stride=10 * 64 - 1) == _lib.IQW_ERR_INVALID
    assert call(C=2, out_stride=10) == _lib.IQW_ERR_INVALID
    assert call(C=2) == _lib.IQW_OK
    assert call(ws_bytes=10 * 64 * 8 - 1) == _lib.IQW_ERR_INVALID
    assert call(n_out=0) == _lib.IQW_OK
    torch.cuda.synchronize()


SHARD_CASES = [(300, 8192, 1024, 1024), (201, 8192, 1024, 512), (700, 1000, 64, 37), (2000, 256, 16, 1),
               (12, 32768, 8192, 8192), (50, 100, 256, 256)]


@pytest.mark.parametrize('world', [2, 3])
@pytest.mark.parametrize('T,Lg,K,hop', SHARD_CASES)
def test_time_shards_equal_single_call(cuda_device, world, T, Lg, K, hop):
    import threading
    rng = np.random.default_rng(T + world)
    g = prototype(Lg, K)
    y = torch.from_numpy(_frames(rng, T, K)).to(cuda_device)
    single = iqw.pfb_synthesize(y, g, hop)
    group = D.ThreadGroup(world)
    parts = [None] * world

    def run(r):
        sh = D.pfb_synth_shard(T, Lg, K, hop, world, r)
        parts[r] = D.pfb_synthesize_time_sharded(y[sh.frame0:sh.frame1].clone(), g, hop, n_frames=T,
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
        for T, Lg, K, hop in SHARD_CASES[:3]:
            g = prototype(Lg, K)
            y = torch.from_numpy(_frames(np.random.default_rng(T), T, K)).to(dev)
            sh = D.pfb_synth_shard(T, Lg, K, hop, world, rank)
            got = D.pfb_synthesize_time_sharded(y[sh.frame0:sh.frame1].contiguous(), g, hop, n_frames=T, gather=True)
            assert torch.equal(got, iqw.pfb_synthesize(y, g, hop))
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
