"""gather=True of the sharded entry points without a GPU: every rank gets the whole result, bitwise the single
call of the same numpy compute -- with the ranks as threads of one `ThreadGroup` (world sizes 2 and 3), and for
the four filter ops also as processes over gloo."""
import os
import socket
import threading

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from iqwaveform_b200 import _plan, fourier
from iqwaveform_b200 import distributed as D
from oracle import iqw_oracle as orc
from oracle.make_golden import synth

from _oaconvolve_numpy import emulate as oaconvolve_emulate
from _pfb_numpy import emulate as pfb_emulate
from _pfb_numpy import prototype
from _pfb_synth_numpy import emulate as pfb_synth_emulate
from _upfirdn_numpy import direct as upfirdn_direct


def _spectrogram():
    N, nfft, nov = 5001, 64, 48
    x = synth(1, (N,))
    kw = dict(fs=1e6, window='hann', nperseg=nfft, noverlap=nov)
    want = orc.spectrogram(x, axis=0, return_axis_arrays=False, **kw)

    def run(group, world, rank):
        sh = D.frame_shard(N, nfft, nov, world, rank)
        return D.spectrogram_time_sharded(x[sh.sample0:sh.sample1], n_samples=N, group=group, gather=True,
                                          compute=lambda a, **k: orc.spectrogram(np.asarray(a), **k), **kw)
    return want, run


def _bin_power():
    N, Ts, Tbin = 1007, 1e-6, 1e-5
    x = synth(2, (N,))
    want = orc.iq_to_bin_power(x, Ts, Tbin, kind='max', truncate=True)

    def run(group, world, rank):
        sh = D.bin_shard(N, 10, world, rank)
        return D.iq_to_bin_power_sharded(x[sh.sample0:sh.sample1], Ts, Tbin, n_samples=N, kind='max', group=group,
                                         compute=lambda a, *p, **k: orc.iq_to_bin_power(np.asarray(a), *p, **k))
    return want, run


def _persistence():
    C, N = 5, 4096
    x = synth(3, (C, N))
    kw = dict(fs=1e6, window='hann', resolution=1e6 / 64, fractional_overlap=0.5, statistics=[0.5, 'mean', 'max'],
              dB=True)
    want = orc.persistence_spectrum(x, axis=1, **kw)

    def run(group, world, rank):
        mine = D.channel_shard(C, world, rank)
        return D.persistence_spectrum_sharded(x[mine.start:mine.stop], n_channels=C, group=group,
                                              compute=lambda a, **k: orc.persistence_spectrum(np.asarray(a), **k),
                                              **kw)
    return want, run


def _upfirdn():
    n, L, up, down = 1000, 33, 2, 3
    h = np.random.default_rng(4).standard_normal(L)
    x = synth(4, (n,))
    table, _ = fourier._upfirdn_taps(h, up, down)
    want = upfirdn_direct(x, table, L, up, down, x_first=0, out_first=0, n_out=_plan.upfirdn_output_len(L, n, up, down))

    def run(group, world, rank):
        sh = D.upfirdn_shard(n, L, up, down, world, rank)
        return D.upfirdn_time_sharded(x[sh.sample0:sh.sample1], h, up, down, n_samples=n, group=group,
                                      compute=upfirdn_direct, gather=True)
    return want, run


def _oaconvolve():
    N, M, mode = 3000, 161, 'same'
    h = np.random.default_rng(5).standard_normal(M)
    x = synth(5, (N,))
    nfft, discard = _plan.oaconvolve_plan(M)
    first, n = _plan.oaconvolve_window(mode, N, M)
    want = oaconvolve_emulate(x, _plan.oaconvolve_spectrum(h[None], nfft), M, nfft, discard, x_first=0,
                              out_first=first, n_out=n)

    def run(group, world, rank):
        sh = D.oaconvolve_shard(N, M, mode, world, rank)
        return D.oaconvolve_time_sharded(x[sh.sample0:sh.sample1], h, mode, n_samples=N, group=group,
                                         compute=oaconvolve_emulate, gather=True)
    return want, run


def _pfb():
    N, L, K, hop = 3000, 256, 16, 12
    h = prototype(L, K)
    x = synth(6, (N,))
    want = pfb_emulate(x, _plan.pfb_taps(h, K), L, K, hop, n_frames=_plan.pfb_frame_count(N, L, hop))

    def run(group, world, rank):
        sh = D.pfb_shard(N, L, K, hop, world, rank)
        return D.pfb_channelize_time_sharded(x[sh.sample0:sh.sample1], h, K, hop, n_samples=N, group=group,
                                             compute=pfb_emulate, gather=True)
    return want, run


def _pfb_synth():
    T, Lg, K, hop = 40, 100, 16, 8
    g = prototype(Lg, K)
    y = synth(7, (T, K))
    want = pfb_synth_emulate(y, _plan.pfb_taps(g, K), Lg, hop, n_frames_total=T, out_first=0,
                             n_out=_plan.pfb_synth_len(T, Lg, hop))

    def run(group, world, rank):
        sh = D.pfb_synth_shard(T, Lg, K, hop, world, rank)
        return D.pfb_synthesize_time_sharded(y[sh.frame0:sh.frame1], g, hop, n_frames=T, group=group,
                                             compute=pfb_synth_emulate, gather=True)
    return want, run


FILTER_OPS = {'upfirdn': _upfirdn, 'oaconvolve': _oaconvolve, 'pfb_channelize': _pfb, 'pfb_synthesize': _pfb_synth}
OPS = dict(FILTER_OPS, spectrogram=_spectrogram, iq_to_bin_power=_bin_power, persistence_spectrum=_persistence)


def _on_threads(world, run):
    """run(group, world, rank) for every rank of one ThreadGroup, each on a thread of its own -> the results in
    rank order.  A rank that raises breaks the group's barrier, so that the others stop waiting for it."""
    group = D.ThreadGroup(world)
    out, errors = [None] * world, []

    def one(r):
        try:
            out[r] = run(group.member(r), world, r)
        except BaseException as e:
            errors.append(e)
            group._barrier.abort()

    threads = [threading.Thread(target=one, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        raise errors[0]
    return out


@pytest.mark.parametrize('world', [2, 3])
@pytest.mark.parametrize('op', sorted(OPS))
def test_thread_group_gathers_the_whole_result(op, world):
    want, run = OPS[op]()
    for got in _on_threads(world, run):
        assert got.shape == want.shape
        assert np.array_equal(got.numpy(), want)


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        for op in FILTER_OPS.values():
            want, run = op()
            got = run(None, world, rank)
            assert got.shape == want.shape and np.array_equal(got.numpy(), want), op.__name__
        open(os.path.join(out_dir, f'ok{rank}'), 'w').close()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize('world', [2, 3])
def test_filter_ops_gather_over_gloo(tmp_path, world):
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    assert all((tmp_path / f'ok{r}').exists() for r in range(world))
