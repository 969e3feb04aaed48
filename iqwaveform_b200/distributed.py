"""one-process-per-GPU sharding of the hot path (no counterpart in the reference, which is
single-process: SURVEY.md section 2.1 / 8e).

The path shards without any collective on the data path, with one exception (the last bullet):

* channels are independent                     -> `channel_shard`  (persistence spectrum, config 3)
* STFT frames are independent                  -> `frame_shard`    (stft / spectrogram, config 2):
  rank r owns frames [f0, f1) and reads samples [f0*hop, (f1-1)*hop + nfft): the last
  `noverlap` samples are the halo shared with the next rank
* power bins are independent                   -> `bin_shard`      (iq_to_bin_power, config 4):
  shards are aligned to whole bins, so the halo is zero
* upfirdn outputs are independent              -> `upfirdn_shard`  (upfirdn): rank r owns outputs
  [out0, out1) and reads the Lp - 1 samples before its first input as the halo
* oaconvolve outputs are independent           -> `oaconvolve_shard` (oaconvolve): rank r owns outputs
  [out0, out1) and reads every in-range sample of the overlap-save blocks they fall in -- a halo of
  the discard D (not M - 1) before them and the rest of its last block after them
* exact quantiles of ONE capture split in time -> `persistence_spectrum_time_sharded`: the only
  real exchange step of the path -- per-bin digit counts of a radix select are all_reduced
  (`select_order_statistics`; kernels in csrc/iqw_rowsplit.cu)

Only the small results are exchanged: `gather_rows` is one `all_gather` over NCCL (CUDA tensors)
or gloo (CPU tensors, used by the CPU tests) of the per-rank result rows.
"""
from __future__ import annotations

from typing import Callable, NamedTuple

import numpy as np
import torch
import torch.distributed as dist

__all__ = ['channel_shard', 'frame_shard', 'bin_shard', 'gather_rows', 'persistence_spectrum_sharded',
           'persistence_spectrum_time_sharded', 'select_order_statistics', 'CudaShardOps', 'ThreadGroup',
           'bind_to_gpu_numa_node', 'spectrogram_time_sharded', 'iq_to_bin_power_sharded', 'upfirdn_shard',
           'upfirdn_time_sharded', 'oaconvolve_shard', 'oaconvolve_time_sharded']


def _split(n: int, world: int, rank: int) -> tuple[int, int]:
    """contiguous, balanced split of range(n): the first n % world ranks get one extra item"""
    if world < 1 or not 0 <= rank < world:
        raise ValueError(f'rank {rank} outside world of {world}')
    base, extra = divmod(n, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def channel_shard(n_channels: int, world: int, rank: int) -> range:
    return range(*_split(n_channels, world, rank))


class FrameShard(NamedTuple):
    frame0: int     # first frame of this rank
    frame1: int     # one past its last frame
    sample0: int    # first sample it reads
    sample1: int    # one past the last sample it reads (includes the halo)
    n_frames: int   # frames of the whole capture


def frame_shard(n_samples: int, nfft: int, noverlap: int, world: int, rank: int) -> FrameShard:
    """time-axis shard of an STFT with the reference's framing (fourier.py:568-569, 1016-1028:
    T = (N - nfft)//hop + 1 with overlap, N//nfft without; no padding, partial tail dropped)"""
    hop = nfft - noverlap
    if hop < 1 or nfft < 1:
        raise ValueError('need 0 <= noverlap < nfft')
    if noverlap == 0:
        T = n_samples // nfft
    else:
        T = (n_samples - nfft) // hop + 1 if n_samples >= nfft else 0
    f0, f1 = _split(T, world, rank)
    if f1 == f0:
        return FrameShard(f0, f1, f0 * hop, f0 * hop, T)
    return FrameShard(f0, f1, f0 * hop, (f1 - 1) * hop + nfft, T)


class BinShard(NamedTuple):
    bin0: int
    bin1: int
    sample0: int
    sample1: int
    n_bins: int


def bin_shard(n_samples: int, bin_len: int, world: int, rank: int) -> BinShard:
    """bin-aligned time shard for iq_to_bin_power (power_analysis.py:380: whole bins only)"""
    if bin_len < 1:
        raise ValueError('bin length must be >= 1 sample')
    n_bins = n_samples // bin_len
    b0, b1 = _split(n_bins, world, rank)
    return BinShard(b0, b1, b0 * bin_len, b1 * bin_len, n_bins)


def gather_rows(local: torch.Tensor, sizes: list[int] | None = None, axis: int = 0, group=None) -> torch.Tensor:
    """all_gather of per-rank result rows along `axis`.  `sizes[r]` = rows of rank r when shards are
    ragged (default: every rank has local.shape[axis] rows).  Works on the backend of the group:
    NCCL for CUDA tensors, gloo for CPU tensors."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return local
    world = dist.get_world_size(group)
    local = local.movedim(axis, 0).contiguous()
    if sizes is None:
        sizes = [local.shape[0]] * world
    if len(sizes) != world or sizes[dist.get_rank(group)] != local.shape[0]:
        raise ValueError('sizes must list the row count of every rank')
    rest = tuple(local.shape[1:])
    # equal-sized exchange (padded to the largest shard): one collective, KB-MB payloads
    m = max(sizes)
    send = local
    if local.shape[0] < m:
        send = torch.zeros((m,) + rest, dtype=local.dtype, device=local.device)
        send[:local.shape[0]] = local
    recv = [torch.empty((m,) + rest, dtype=local.dtype, device=local.device) for _ in range(world)]
    dist.all_gather(recv, send, group=group)
    out = torch.cat([r[:n] for r, n in zip(recv, sizes)], dim=0)
    return out.movedim(0, axis)


def bind_to_gpu_numa_node(device_index: int) -> str | None:
    """pin the calling process to the CPUs of the NUMA node its GPU hangs off, so that the pinned
    host buffers it allocates afterwards (first touch) and its copy threads sit next to that GPU's
    PCIe root: with one process per GPU, host->device copies of all ranks otherwise share one
    socket's memory and the inter-socket link.  Returns the cpu list it bound to, or None when the
    topology is not visible (no sysfs entry, single node, restricted cpuset) -- never raises."""
    import os
    try:
        pr = torch.cuda.get_device_properties(device_index)
        bdf = f'{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0'
        with open(f'/sys/bus/pci/devices/{bdf}/numa_node') as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f'/sys/devices/system/node/node{node}/cpulist') as f:
            cpulist = f.read().strip()
        cpus = set()
        for part in cpulist.split(','):
            a, _, b = part.partition('-')
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return cpulist
    except Exception:       # no GPU, no sysfs, restricted cpuset ...: binding is an optimisation only
        return None


def _world(group=None) -> tuple[int, int]:
    if hasattr(group, 'iqw_all_reduce'):      # in-process stand-in for a process group (tests, probes)
        return group.size(), group.rank()
    if dist.is_initialized():
        return dist.get_world_size(group), dist.get_rank(group)
    return 1, 0


def _all_reduce(t: torch.Tensor, op: str, group=None) -> None:
    """in-place all_reduce over `group`: a torch.distributed group (NCCL / gloo), or any object with
    rank(), size() and iqw_all_reduce(tensor, op) -- e.g. `ThreadGroup`, which lets several shards of
    one capture be driven from threads of one process on one GPU"""
    if hasattr(group, 'iqw_all_reduce'):
        group.iqw_all_reduce(t, op)
    else:
        dist.all_reduce(t, op={'sum': dist.ReduceOp.SUM, 'min': dist.ReduceOp.MIN, 'max': dist.ReduceOp.MAX}[op],
                        group=group)


class ThreadGroup:
    """`ThreadGroup(n).member(r)` objects act as the `group` of rank r of n for the time-sharded
    functions when the n ranks are threads of ONE process (all shards on one GPU, or a CPU test):
    all_reduce is a barrier plus an elementwise reduction over the members' tensors."""

    def __init__(self, n: int):
        import threading
        self.n = n
        self._barrier = threading.Barrier(n)
        self._slots: list = [None] * n

    def member(self, r: int):
        return _ThreadMember(self, r)


class _ThreadMember:
    def __init__(self, owner: ThreadGroup, r: int):
        self._o, self._r = owner, r

    def rank(self) -> int:
        return self._r

    def size(self) -> int:
        return self._o.n

    def iqw_all_reduce(self, t: torch.Tensor, op: str) -> None:
        o = self._o
        o._slots[self._r] = t
        o._barrier.wait()
        stacked = torch.stack(list(o._slots))
        res = {'sum': stacked.sum(0), 'min': stacked.amin(0), 'max': stacked.amax(0)}[op].to(t.dtype)
        if t.is_cuda:
            torch.cuda.synchronize()
        o._barrier.wait()
        t.copy_(res)
        if t.is_cuda:
            torch.cuda.synchronize()
        o._barrier.wait()


def persistence_spectrum_sharded(x_local, *, n_channels: int, group=None, compute: Callable | None = None, **kw):
    """channel-sharded persistence spectrum: `x_local` holds this rank's channels
    (`channel_shard(n_channels, world, rank)`, shape (C_local, N)); every rank returns the full
    (n_channels, nstat, nbins) result.  `compute` defaults to the CUDA `persistence_spectrum`."""
    if compute is None:
        from .fourier import persistence_spectrum as compute
    world, rank = _world(group)
    # every rank derives this from the arguments alone, so all of them raise together: a raise on a
    # subset of the ranks ahead of the all_gather would leave the others blocked in the collective
    if n_channels < 1:
        raise ValueError('n_channels must be >= 1')
    if world > n_channels:
        raise ValueError(f'{world} ranks for {n_channels} channels: every rank needs at least one channel '
                         f'(run the call on a sub-group of {n_channels} ranks)')
    mine = channel_shard(n_channels, world, rank)
    if x_local.shape[0] != len(mine):
        raise ValueError(f'rank {rank} expects {len(mine)} channels, got {x_local.shape[0]}')
    kw = dict(kw, axis=1)
    out = compute(x_local, **kw)
    if world == 1:
        return out
    out = torch.as_tensor(out)
    return gather_rows(out, [len(channel_shard(n_channels, world, r)) for r in range(world)], 0, group)


_REDUCIBLE = {'mean': 'sum', 'rms': 'sum', 'max': 'max', 'peak': 'max', 'min': 'min'}


class CudaShardOps:
    """the per-rank device work of the time-sharded persistence spectrum, through the C-ABI.
    (The CPU tests substitute a numpy stand-in with the same five methods to run the host logic
    and the collectives over gloo.)"""

    def power_spectrogram(self, x, *, window, nfft, noverlap, nzero, bin_lo, bin_hi):
        """this rank's frames: (T_local, nbins) float32 power on the device"""
        from . import _arrays, _lib, fourier
        xd, _ = _arrays.to_device(x)
        if xd.numel() == 0:
            return torch.empty((0, bin_hi - bin_lo), dtype=torch.float32, device=xd.device)
        return fourier._stft_device(xd.reshape(1, -1), window=window, nfft=nfft, noverlap=noverlap, nzero=nzero,
                                    norm='power', truncate=True, mode=_lib.STFT_POWER, bin_lo=bin_lo,
                                    bin_hi=bin_hi)[0]

    def named_statistics(self, p, names, dB):
        from . import fourier
        return fourier.time_statistics(p[None], list(names), dB=bool(dB), eps=1e-25)[0]

    def local_order_statistics(self, p, local_ranks):
        """(len(local_ranks), nbins) float32: the order statistics of THIS rank's rows at the given
        0-based local ranks (kernel 2, no interpolation, no dB)"""
        from . import _lib, fourier
        reqs = []
        for r in local_ranks:
            q = _lib.iqw_stat()
            q.kind, q.rank_lo, q.rank_hi, q.gamma = _lib.STAT_ORDER, r, r, 0.0
            reqs.append(q)
        return fourier.time_statistics(p[None], None, dB=False, requests=reqs)[0]

    def bracket_collect(self, p, lo, hi):
        """one pass over this rank's rows: (store, below) -- the rows inside any bracket go to the
        candidate store; below is (n_sel + 1, nbins) int32: rows under each bracket, and in the last
        row the number of overflowed store segments"""
        import ctypes
        from . import _lib, fourier
        n_sel, nb = lo.shape
        nbytes = _lib.lib.iqw_bracket_collect_workspace_bytes(p.shape[0], nb)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=lo.device)
        below = torch.empty((n_sel + 1, nb), dtype=torch.int32, device=lo.device)
        _lib.check(_lib.lib.iqw_bracket_collect_f32(
            ctypes.c_void_p(p.data_ptr() if p.shape[0] else None), p.shape[0], nb, n_sel,
            ctypes.c_void_p(lo.data_ptr()), ctypes.c_void_p(hi.data_ptr()), ctypes.c_void_p(below.data_ptr()),
            ctypes.c_void_p(ws.data_ptr()), nbytes, fourier._stream_ptr(lo.device)))
        return (ws, p.shape[0]), below

    def candidate_count(self, store, lo, hi, level):
        """(n_sel, nbins, 256) int32 digit counts of the stored candidates inside [lo, hi]"""
        import ctypes
        from . import _lib, fourier
        ws, n_rows = store
        n_sel, nb = lo.shape
        counts = torch.empty((n_sel, nb, 256), dtype=torch.int32, device=lo.device)
        _lib.check(_lib.lib.iqw_candidate_count_f32(
            ctypes.c_void_p(ws.data_ptr()), n_rows, nb, n_sel, ctypes.c_void_p(lo.data_ptr()),
            ctypes.c_void_p(hi.data_ptr()), level, ctypes.c_void_p(counts.data_ptr()), fourier._stream_ptr(lo.device)))
        return counts

    def radix_count(self, p, lo, hi, level, want_below):
        """(n_sel, nbins, 256) int32 counts of this rank's rows with lo <= key <= hi by key digit
        `level`, and (n_sel, nbins) int32 rows with key < lo (or None)"""
        import ctypes
        from . import _lib, fourier
        n_sel, nb = lo.shape
        counts = torch.empty((n_sel, nb, 256), dtype=torch.int32, device=lo.device)
        below = torch.empty((n_sel, nb), dtype=torch.int32, device=lo.device) if want_below else None
        _lib.check(_lib.lib.iqw_radix_count_f32(
            ctypes.c_void_p(p.data_ptr() if p.shape[0] else None), p.shape[0], nb, n_sel,
            ctypes.c_void_p(lo.data_ptr()), ctypes.c_void_p(hi.data_ptr()), level,
            ctypes.c_void_p(counts.data_ptr()), ctypes.c_void_p(below.data_ptr()) if want_below else None,
            fourier._stream_ptr(lo.device)))
        return counts, below

    def radix_descend(self, counts, rank, prefix, lo, hi, level):
        import ctypes
        from . import _lib, fourier
        _lib.check(_lib.lib.iqw_radix_descend(
            ctypes.c_void_p(counts.data_ptr()), prefix.shape[0], prefix.shape[1], level,
            ctypes.c_void_p(rank.data_ptr()), ctypes.c_void_p(prefix.data_ptr()), ctypes.c_void_p(lo.data_ptr()),
            ctypes.c_void_p(hi.data_ptr()), fourier._stream_ptr(prefix.device)))

    def finish(self, keys, sel_rank, n_rows_total, reqs, dB):
        """(len(reqs), nbins) float32 quantile / median rows from the selected keys"""
        import ctypes
        from . import _lib, fourier
        out = torch.empty((len(reqs), keys.shape[1]), dtype=torch.float32, device=keys.device)
        _lib.check(_lib.lib.iqw_order_stats_finish_f32(
            ctypes.c_void_p(keys.data_ptr()), len(sel_rank), (ctypes.c_int64 * len(sel_rank))(*sel_rank),
            n_rows_total, keys.shape[1], (_lib.iqw_stat * len(reqs))(*reqs), len(reqs), int(bool(dB)), 1e-25,
            ctypes.c_void_p(out.data_ptr()), fourier._stream_ptr(keys.device)))
        return out


def _keys_of(v: torch.Tensor) -> torch.Tensor:
    """order-preserving uint32 keys of float32 values, as int64 (so that MIN / MAX reduce them)"""
    b = v.contiguous().view(torch.int32).to(torch.int64) & 0xFFFFFFFF
    return torch.where(b >= 0x80000000, b ^ 0xFFFFFFFF, b ^ 0x80000000)


def _as_u32_storage(k: torch.Tensor) -> torch.Tensor:
    """int64 keys -> int32 tensor holding the same 32 bits (what the C-ABI reads as uint32)"""
    return torch.where(k >= 0x80000000, k - (1 << 32), k).to(torch.int32).contiguous()


MAX_SEL_PER_PASS = 8


def _rank_groups(sel_rank: list[int]) -> list[list[int]]:
    """indices of `sel_rank` (ascending ranks) grouped into runs of consecutive ranks"""
    groups: list[list[int]] = []
    for i, r in enumerate(sel_rank):
        if groups and 0 <= r - sel_rank[groups[-1][-1]] <= 1:
            groups[-1].append(i)
        else:
            groups.append([i])
    return groups


def select_order_statistics(p: torch.Tensor, sel_rank: list[int], n_rows_total: int | None = None, *, group=None,
                            ops=None, bracket: bool = True, info: dict | None = None) -> torch.Tensor:
    """keys (order-preserving uint32 images of float32, stored in an int32 tensor) of the global
    order statistics `sel_rank` of every column of a matrix whose rows are spread over the ranks
    of `group`: `p` holds this rank's rows (possibly none), `n_rows_total` is the row count over
    all ranks.  Every rank ends with the same (len(sel_rank), n_cols) keys.

    1. bracket: the local order statistic at rank floor(j*n_local/n_total) on every rank; the MIN
       and MAX of those over the ranks enclose the global statistic j (fewer than j+1 rows lie
       below the MIN, at least j+1 at or below the MAX) -- two all_reduce of (n_sel, n_cols) keys
    2. collect: one pass over the local rows counts the rows below each bracket and keeps the rows
       inside any bracket -- one all_reduce(SUM) of (n_sel + 1, n_cols) counts
    3. four count -> all_reduce(SUM) -> descend rounds over the kept rows, 8 key bits each (over
       the whole matrix if some rank's candidate store overflowed: heavy ties)
    `bracket=False` skips 1-2 and counts every row at every level (same result)."""
    ops = ops or CudaShardOps()
    if len(sel_rank) > MAX_SEL_PER_PASS:
        return torch.cat([select_order_statistics(p, sel_rank[i:i + MAX_SEL_PER_PASS], n_rows_total, group=group,
                                                  ops=ops, bracket=bracket, info=info)
                          for i in range(0, len(sel_rank), MAX_SEL_PER_PASS)])
    world, _ = _world(group)
    n_local, nb = p.shape
    n_sel = len(sel_rank)
    if n_rows_total is None:
        if world > 1:
            raise ValueError('n_rows_total is required when rows are spread over several ranks')
        n_rows_total = n_local
    dev = p.device
    rank = torch.tensor(sel_rank, dtype=torch.int64).reshape(n_sel, 1).expand(n_sel, nb).contiguous().to(dev)
    prefix = torch.zeros((n_sel, nb), dtype=torch.int32, device=dev)
    store = None
    if bracket and n_rows_total > 0:
        if n_local:
            vals = ops.local_order_statistics(p, [min(j * n_local // n_rows_total, n_local - 1) for j in sel_rank])
            # kernel 2 orders -0.0 and +0.0 as equal: a zero stands for either key
            klo = torch.where(vals == 0, _keys_of(torch.full_like(vals, -0.0)), _keys_of(vals))
            khi = torch.where(vals == 0, _keys_of(torch.zeros_like(vals)), _keys_of(vals))
        else:       # no rows: neutral elements of MIN / MAX
            klo = torch.full((n_sel, nb), 0xFFFFFFFF, dtype=torch.int64, device=dev)
            khi = torch.zeros((n_sel, nb), dtype=torch.int64, device=dev)
        if world > 1:
            _all_reduce(klo, 'min', group)
            _all_reduce(khi, 'max', group)
        # statistics at neighbouring ranks (the two ends of one quantile) share one bracket: the
        # collect pass is bound by its compares per row, and any enclosing interval is valid
        grp = _rank_groups(sel_rank)
        glo = torch.stack([klo[g].amin(0) for g in grp])
        ghi = torch.stack([khi[g].amax(0) for g in grp])
        of = torch.tensor([k for k, g in enumerate(grp) for _ in g], device=dev)
        lo, hi = _as_u32_storage(glo[of]), _as_u32_storage(ghi[of])
        store, below = ops.bracket_collect(p, _as_u32_storage(glo), _as_u32_storage(ghi))
        if world > 1:
            _all_reduce(below, 'sum', group)
        rank -= below[of]
        if bool(below[len(grp)].any()):      # identical on every rank (summed), so all take the same branch
            store = None
        if info is not None:
            info['candidate_store'] = store is not None
    else:
        lo = torch.zeros((n_sel, nb), dtype=torch.int32, device=dev)
        hi = torch.full((n_sel, nb), -1, dtype=torch.int32, device=dev)
    for level in range(4):
        if store is not None:
            counts = ops.candidate_count(store, lo, hi, level)
        else:
            counts, below = ops.radix_count(p, lo, hi, level, level == 0 and not bracket)
            if below is not None:
                if world > 1:
                    _all_reduce(below, 'sum', group)
                rank -= below
        if world > 1:
            _all_reduce(counts, 'sum', group)
        ops.radix_descend(counts, rank, prefix, lo, hi, level)
    return prefix


def persistence_spectrum_time_sharded(x_halo, *, n_samples: int, fs: float, window, resolution: float,
                                      statistics, fractional_overlap=0, fractional_window: float = 1,
                                      bandwidth=float('inf'), truncate=True, dB=True, group=None, ops=None):
    """time-sharded persistence spectrum of ONE long 1-D capture of `n_samples` samples: `x_halo`
    holds this rank's samples [shard.sample0, shard.sample1) of `frame_shard` (halo included);
    every rank returns the (nstat, nbins) result of the whole capture.

    * 'mean'/'rms' (over dB values when dB=True, like the reference), 'max'/'peak', 'min': one
      all_reduce of a row each (frame-count-weighted SUM, MAX, MIN)
    * quantiles and 'median': EXACT, by a bracketed radix select on the distributed spectrogram
      (`select_order_statistics`: 2 all_reduce of bracket keys + 5 of per-bin counts; one pass over
      the local spectrogram + kernel 2 on it for the bracket), then the
      reference's float32 'linear' interpolation on the dB of the selected values.  The quantile index
      arithmetic uses the frame count of the whole capture (fourier.py:1317-1320)."""
    from . import _lib, _plan, fourier
    ops = ops or CudaShardOps()
    world, rank = _world(group)
    nfft, noverlap, nzero = fourier._psd_frame_plan(fs, resolution, fractional_overlap, fractional_window)
    sh = frame_shard(n_samples, nfft, noverlap, world, rank)
    if x_halo.shape[-1] != sh.sample1 - sh.sample0 or x_halo.ndim != 1:
        raise ValueError(f'rank {rank} expects a 1-D shard of {sh.sample1 - sh.sample0} samples, got {tuple(x_halo.shape)}')
    T = sh.n_frames
    if T < 1:
        raise ValueError('cannot take statistics over zero frames')
    if T >= 1 << 31:
        raise NotImplementedError('more than 2^31-1 frames')
    statistics = list(statistics)
    reqs = _plan.stat_requests(statistics, T)
    bin_lo, bin_hi = 0, nfft
    if truncate and bandwidth != float('inf'):
        bin_lo, bin_hi = _plan.freq_band_edges(nfft, 1.0 / fs, -bandwidth / 2, +bandwidth / 2)

    p = ops.power_spectrogram(x_halo, window=window, nfft=nfft, noverlap=noverlap, nzero=nzero,
                              bin_lo=bin_lo, bin_hi=bin_hi)
    n_local = sh.frame1 - sh.frame0
    assert p.shape == (n_local, bin_hi - bin_lo)
    out = torch.empty((len(reqs), p.shape[1]), dtype=torch.float32, device=p.device)

    named = [i for i, r in enumerate(reqs) if r.kind in (_lib.STAT_MEAN, _lib.STAT_MAX, _lib.STAT_MIN)]
    if named:
        if n_local:
            rows = ops.named_statistics(p, [statistics[i] for i in named], dB)
        else:       # a rank without frames contributes the neutral element of each reduction
            neutral = {'sum': 0.0, 'max': float('-inf'), 'min': float('inf')}
            rows = torch.stack([torch.full((p.shape[1],), neutral[_REDUCIBLE[statistics[i]]], dtype=torch.float32,
                                           device=p.device) for i in named])
        for k, i in enumerate(named):
            row = rows[k].clone()
            how = _REDUCIBLE[statistics[i]]
            if world > 1:
                if how == 'sum':
                    row.mul_(n_local / T)
                _all_reduce(row, how, group)
            out[i] = row

    order = [i for i in range(len(reqs)) if i not in named]
    if order:
        sel_rank = sorted(_plan.distinct_ranks([reqs[i] for i in order], T))
        keys = select_order_statistics(p, sel_rank, T, group=group, ops=ops)
        out[order] = ops.finish(keys, sel_rank, T, [reqs[i] for i in order], dB)
    return out


def spectrogram_time_sharded(x_halo, *, n_samples: int, nperseg: int, noverlap: int = 0, group=None,
                             compute: Callable | None = None, gather: bool = False, **kw):
    """time-sharded spectrogram of a 1-D capture of `n_samples` samples: `x_halo` holds this rank's
    samples [shard.sample0, shard.sample1) (halo included).  Returns this rank's frames
    (T_local, nfft) or, with gather=True, all frames on every rank."""
    if compute is None:
        from .fourier import spectrogram as compute
    world, rank = _world(group)
    sh = frame_shard(n_samples, nperseg, noverlap, world, rank)
    if x_halo.shape[-1] != sh.sample1 - sh.sample0:
        raise ValueError(f'rank {rank} expects {sh.sample1 - sh.sample0} samples, got {x_halo.shape[-1]}')
    p = compute(x_halo, nperseg=nperseg, noverlap=noverlap, axis=0, return_axis_arrays=False, **kw)
    p = torch.as_tensor(p)
    assert p.shape[0] == sh.frame1 - sh.frame0
    if not gather or world == 1:
        return p
    sizes = [(lambda s: s.frame1 - s.frame0)(frame_shard(n_samples, nperseg, noverlap, world, r)) for r in range(world)]
    return gather_rows(p, sizes, 0, group)


def iq_to_bin_power_sharded(x_local, Ts: float, Tbin: float, *, n_samples: int, kind='mean', group=None,
                            compute: Callable | None = None):
    """bin-sharded iq_to_bin_power of a 1-D capture: `x_local` holds samples
    [shard.sample0, shard.sample1); every rank returns all n_bins values."""
    if compute is None:
        from .power_analysis import iq_to_bin_power as compute
    world, rank = _world(group)
    bin_len = round(Tbin / Ts)
    sh = bin_shard(n_samples, bin_len, world, rank)
    if x_local.shape[-1] != sh.sample1 - sh.sample0:
        raise ValueError(f'rank {rank} expects {sh.sample1 - sh.sample0} samples, got {x_local.shape[-1]}')
    out = torch.as_tensor(compute(x_local, Ts, Tbin, kind=kind, axis=0, truncate=True))
    if world == 1:
        return out
    sizes = [(lambda s: s.bin1 - s.bin0)(bin_shard(n_samples, bin_len, world, r)) for r in range(world)]
    return gather_rows(out, sizes, 0, group)


class UpfirdnShard(NamedTuple):
    out0: int       # first output of this rank
    out1: int       # one past its last output
    sample0: int    # first sample it reads
    sample1: int    # one past the last sample it reads (includes the halo)
    n_out: int      # outputs of the whole capture


def upfirdn_shard(n_in: int, n_taps: int, up: int, down: int, world: int, rank: int) -> UpfirdnShard:
    """time-axis shard of upfirdn: outputs split evenly; the samples are those the rank's outputs read,
    y[n] = sum_{j < Lp} hp[p][j] * x[n*down div up - j], clamped to [0, n_in)"""
    from . import _plan
    if n_taps < 1 or up < 1 or down < 1:
        raise ValueError('need n_taps, up, down >= 1')
    n_out = _plan.upfirdn_output_len(n_taps, n_in, up, down)
    o0, o1 = _split(n_out, world, rank)
    lp = -(-n_taps // up)
    if o1 == o0:
        s = min(o0 * down // up, n_in)
        return UpfirdnShard(o0, o1, s, s, n_out)
    s0 = max(0, o0 * down // up - (lp - 1))
    s1 = min(n_in, (o1 - 1) * down // up + 1)
    return UpfirdnShard(o0, o1, s0, max(s0, s1), n_out)


def upfirdn_time_sharded(x_halo, h, up: int = 1, down: int = 1, *, n_samples: int, group=None,
                         compute: Callable | None = None, gather: bool = False):
    """time-sharded upfirdn of a 1-D complex64 capture of `n_samples` samples: `x_halo` holds this rank's
    samples [shard.sample0, shard.sample1) of `upfirdn_shard` (halo included).  Returns this rank's
    outputs [out0, out1) or, with gather=True, all outputs on every rank; the concatenation is bitwise
    the single-GPU `upfirdn`.  `compute(x_halo, table, n_taps, up, down, x_first=, out_first=, n_out=)`
    defaults to the CUDA kernel."""
    from . import fourier
    up, down = int(up), int(down)
    table, n_taps = fourier._upfirdn_taps(h, up, down)
    world, rank = _world(group)
    sh = upfirdn_shard(n_samples, n_taps, up, down, world, rank)
    if x_halo.ndim != 1 or x_halo.shape[0] != sh.sample1 - sh.sample0:
        raise ValueError(f'rank {rank} expects a 1-D shard of {sh.sample1 - sh.sample0} samples, got {tuple(x_halo.shape)}')
    if compute is None:
        from . import _arrays
        xd, _ = _arrays.to_device(x_halo)
        if xd.dtype != torch.complex64:
            raise NotImplementedError(f'upfirdn: only complex64 x is built (got {xd.dtype})')
        y = fourier._upfirdn_device(xd.reshape(1, -1), table, n_taps, up, down, x_first=sh.sample0,
                                    out_first=sh.out0, n_out=sh.out1 - sh.out0)[0]
    else:
        y = torch.as_tensor(compute(x_halo, table, n_taps, up, down, x_first=sh.sample0, out_first=sh.out0,
                                    n_out=sh.out1 - sh.out0))
    if not gather or world == 1:
        return y
    sizes = [(lambda s: s.out1 - s.out0)(upfirdn_shard(n_samples, n_taps, up, down, world, r)) for r in range(world)]
    return gather_rows(y, sizes, 0, group)


class OaconvolveShard(NamedTuple):
    out0: int       # first output of this rank (index into the output of the chosen mode)
    out1: int       # one past its last output
    sample0: int    # first sample it reads
    sample1: int    # one past the last sample it reads (includes the halo)
    n_out: int      # outputs of the whole capture in the chosen mode


def oaconvolve_shard(n_in: int, n_taps: int, mode: str, world: int, rank: int) -> OaconvolveShard:
    """time-axis shard of oaconvolve(x, h, mode) for a capture of n_in samples and an n_taps filter:
    the outputs of the mode are split evenly; the samples are every in-range sample of the overlap-save
    blocks those outputs fall in (block b reads [b*hop - D, b*hop - D + nfft)), clamped to [0, n_in).
    Every block is then computed from the same samples as in one call, so the shards' concatenation is
    bitwise the single-GPU result."""
    from . import _plan
    if n_taps < 1 or n_in < n_taps:
        raise NotImplementedError(f'oaconvolve time shards need 1 <= n_taps <= n_in (got {n_taps}, {n_in})')
    nfft, discard = _plan.oaconvolve_plan(n_taps)
    hop = nfft - discard
    first, n_out = _plan.oaconvolve_window(mode, n_in, n_taps)
    o0, o1 = _split(n_out, world, rank)
    if o1 == o0:
        s = min(max(0, (first + o0) // hop * hop - discard), n_in)
        return OaconvolveShard(o0, o1, s, s, n_out)
    b0, b1 = (first + o0) // hop, (first + o1 - 1) // hop
    s0 = min(n_in, max(0, b0 * hop - discard))
    s1 = min(n_in, b1 * hop - discard + nfft)
    return OaconvolveShard(o0, o1, s0, max(s0, s1), n_out)


def oaconvolve_time_sharded(x_halo, h, mode: str = 'full', *, n_samples: int, group=None,
                            compute: Callable | None = None, gather: bool = False):
    """time-sharded oaconvolve(x, h, mode) of a 1-D complex64 capture x of `n_samples` samples and a 1-D
    filter h no longer than it: `x_halo` holds this rank's samples [shard.sample0, shard.sample1) of
    `oaconvolve_shard` (halo included).  Returns this rank's outputs [out0, out1) or, with gather=True, all
    outputs on every rank; the concatenation is bitwise the single-GPU `oaconvolve`.
    `compute(x_halo, hspec, n_taps, nfft, discard, x_first=, out_first=, n_out=)` defaults to the CUDA
    kernel."""
    from . import _plan, fourier
    if isinstance(h, torch.Tensor):
        h = h.detach().cpu().numpy()
    h = np.asarray(h)
    if h.ndim != 1 or h.size == 0:
        raise ValueError('oaconvolve_time_sharded: h must be 1-D with non-zero length')
    world, rank = _world(group)
    sh = oaconvolve_shard(n_samples, h.size, mode, world, rank)
    if x_halo.ndim != 1 or x_halo.shape[0] != sh.sample1 - sh.sample0:
        raise ValueError(f'rank {rank} expects a 1-D shard of {sh.sample1 - sh.sample0} samples, got {tuple(x_halo.shape)}')
    nfft, discard = _plan.oaconvolve_plan(h.size)
    hspec = _plan.oaconvolve_spectrum(h[None], nfft)
    first, _ = _plan.oaconvolve_window(mode, n_samples, h.size)
    kw = dict(x_first=sh.sample0, out_first=first + sh.out0, n_out=sh.out1 - sh.out0)
    if compute is None:
        from . import _arrays
        xd, _ = _arrays.to_device(x_halo)
        if xd.dtype != torch.complex64:
            raise NotImplementedError(f'oaconvolve: only a complex64 signal is built (got {xd.dtype})')
        y = fourier._oaconvolve_device(xd.reshape(1, -1), hspec, h.size, nfft, discard, **kw)[0]
    else:
        y = torch.as_tensor(compute(x_halo, hspec, h.size, nfft, discard, **kw))
    if not gather or world == 1:
        return y
    sizes = [(lambda s: s.out1 - s.out0)(oaconvolve_shard(n_samples, h.size, mode, world, r)) for r in range(world)]
    return gather_rows(y, sizes, 0, group)
