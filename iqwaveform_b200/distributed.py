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
* pfb_channelize frames are independent         -> `pfb_shard` (pfb_channelize): rank r owns frames
  [f0, f1) and reads [f0*hop, (f1 - 1)*hop + L), a halo of L - hop samples
* pfb_synthesize outputs are independent         -> `pfb_synth_shard` (pfb_synthesize): rank r owns outputs
  [o0, o1) and reads the frames that cover them, a halo of about Lg / hop - 1 frames
* sosfilt is recursive                        -> `sosfilt_shard` (sosfilt): rank r owns the samples of whole
  groups of kernel 10 and reads no halo; instead the ranks all_gather the zero-state final state of every
  group, and each folds the whole list into the start states of its own groups (`sosfilt_time_sharded`)
* exact quantiles of ONE capture split in time -> `persistence_spectrum_time_sharded`: the only
  real exchange step of the path -- per-bin digit counts of a radix select are all_reduced
  (`select_order_statistics`; kernels in csrc/iqw_rowsplit.cu)

Every time-axis planner returns a record of one layout: (first item the rank owns, one past its last, first
item of the input it reads, one past the last it reads -- halo included --, items of the whole capture).  The
owned items are frames, bins or outputs; the input is samples, or frames for `pfb_synth_shard`.  The field
names say which; `_time_sharded` reads the records by position.

Only the small results are exchanged: `gather_rows` is one `all_gather` over NCCL (CUDA tensors)
or gloo (CPU tensors, used by the CPU tests) of the per-rank result rows, or an exchange between the
threads of a `ThreadGroup`.
"""
from __future__ import annotations

from typing import Callable, NamedTuple

import torch
import torch.distributed as dist

__all__ = ['channel_shard', 'frame_shard', 'bin_shard', 'gather_rows', 'persistence_spectrum_sharded',
           'persistence_spectrum_time_sharded', 'select_order_statistics', 'CudaShardOps', 'ThreadGroup',
           'bind_to_gpu_numa_node', 'spectrogram_time_sharded', 'iq_to_bin_power_sharded', 'upfirdn_shard',
           'upfirdn_time_sharded', 'oaconvolve_shard', 'oaconvolve_time_sharded', 'pfb_shard',
           'pfb_channelize_time_sharded', 'pfb_synth_shard', 'pfb_synthesize_time_sharded', 'sosfilt_shard',
           'SosfiltShardOps', 'sosfilt_time_sharded']


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
    NCCL for CUDA tensors, gloo for CPU tensors; or between the threads of a `ThreadGroup`."""
    world, rank = _world(group)
    if world == 1:
        return local
    local = local.movedim(axis, 0).contiguous()
    if sizes is None:
        sizes = [local.shape[0]] * world
    if len(sizes) != world or sizes[rank] != local.shape[0]:
        raise ValueError('sizes must list the row count of every rank')
    rest = tuple(local.shape[1:])
    # equal-sized exchange (padded to the largest shard): one collective, KB-MB payloads
    m = max(sizes)
    send = local
    if local.shape[0] < m:
        send = torch.zeros((m,) + rest, dtype=local.dtype, device=local.device)
        send[:local.shape[0]] = local
    if hasattr(group, 'iqw_all_reduce'):
        recv = group.iqw_all_gather(send)
    else:
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
    all_reduce is a barrier plus an elementwise reduction over the members' tensors, all_gather a
    barrier plus a copy of each."""

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

    def _exchange(self, t: torch.Tensor, combine: Callable):
        """combine(the members' tensors in rank order), once every member has posted its `t`; no member
        returns before all have combined"""
        o = self._o
        o._slots[self._r] = t
        o._barrier.wait()
        res = combine(list(o._slots))
        if t.is_cuda:
            torch.cuda.synchronize()
        o._barrier.wait()
        return res

    def iqw_all_reduce(self, t: torch.Tensor, op: str) -> None:
        def reduce(ts):
            stacked = torch.stack(ts)
            return {'sum': stacked.sum(0), 'min': stacked.amin(0), 'max': stacked.amax(0)}[op].to(t.dtype)
        t.copy_(self._exchange(t, reduce))
        if t.is_cuda:
            torch.cuda.synchronize()
        self._o._barrier.wait()

    def iqw_all_gather(self, t: torch.Tensor) -> list[torch.Tensor]:
        # copies: a member may change its tensor as soon as the exchange is over
        return self._exchange(t, lambda ts: [s.clone() for s in ts])


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


def _time_sharded(x_halo, plan: Callable, run: Callable, compute: Callable | None, default: Callable, *, group,
                  gather: bool, ndim: int | None = 1, unit: str = 'samples'):
    """the steps every time-sharded entry point shares.  `plan(world, rank)` returns a shard record (the layout
    of the module docstring) whose read span `x_halo` holds: along its first axis and with `ndim` axes, or along
    its last axis when ndim is None.  Returns `run(compute, shard)` (`compute` defaulting to `default`) as a
    tensor or, with `gather`, the owned items of all ranks on every rank."""
    world, rank = _world(group)
    sh = plan(world, rank)
    own0, own1, read0, read1, _ = sh
    n = read1 - read0
    if ndim is None:
        bad, want = x_halo.shape[-1] != n, f'{n} {unit}'
    else:
        bad = x_halo.ndim != ndim or x_halo.shape[0] != n
        want = f'a {"1-D " if ndim == 1 else ""}shard of {n} {unit}'
    if bad:
        raise ValueError(f'rank {rank} expects {want}, got {tuple(x_halo.shape)}')
    y = torch.as_tensor(run(default if compute is None else compute, sh))
    assert y.shape[0] == own1 - own0
    if not gather:
        return y
    return gather_rows(y, [s[1] - s[0] for s in (plan(world, r) for r in range(world))], 0, group)


def _on_device(device_op: Callable, not_built: str) -> Callable:
    """`device_op` of (C, ...) complex64 rows on the device as the `compute` of a rank's shard: the shard goes to
    the device as one row.  `not_built` is the NotImplementedError message for a shard of another dtype."""
    def compute(x, *args, **kw):
        from . import _arrays
        xd, _ = _arrays.to_device(x)
        if xd.dtype != torch.complex64:
            raise NotImplementedError(f'{not_built} (got {xd.dtype})')
        return device_op(xd[None], *args, **kw)[0]
    return compute


def spectrogram_time_sharded(x_halo, *, n_samples: int, nperseg: int, noverlap: int = 0, group=None,
                             compute: Callable | None = None, gather: bool = False, **kw):
    """time-sharded spectrogram of a 1-D capture of `n_samples` samples: `x_halo` holds this rank's
    samples [shard.sample0, shard.sample1) (halo included).  Returns this rank's frames
    (T_local, nfft) or, with gather=True, all frames on every rank."""
    from . import fourier
    return _time_sharded(x_halo, lambda w, r: frame_shard(n_samples, nperseg, noverlap, w, r),
                         lambda f, sh: f(x_halo, nperseg=nperseg, noverlap=noverlap, axis=0, return_axis_arrays=False,
                                         **kw),
                         compute, fourier.spectrogram, group=group, gather=gather, ndim=None)


def iq_to_bin_power_sharded(x_local, Ts: float, Tbin: float, *, n_samples: int, kind='mean', group=None,
                            compute: Callable | None = None):
    """bin-sharded iq_to_bin_power of a 1-D capture: `x_local` holds samples
    [shard.sample0, shard.sample1); every rank returns all n_bins values."""
    from . import power_analysis
    bin_len = round(Tbin / Ts)
    return _time_sharded(x_local, lambda w, r: bin_shard(n_samples, bin_len, w, r),
                         lambda f, sh: f(x_local, Ts, Tbin, kind=kind, axis=0, truncate=True),
                         compute, power_analysis.iq_to_bin_power, group=group, gather=True, ndim=None)


class OutputShard(NamedTuple):
    out0: int       # first output of this rank (for oaconvolve: an index into the output of the chosen mode)
    out1: int       # one past its last output
    sample0: int    # first sample it reads
    sample1: int    # one past the last sample it reads (includes the halo)
    n_out: int      # outputs of the whole capture


def upfirdn_shard(n_in: int, n_taps: int, up: int, down: int, world: int, rank: int) -> OutputShard:
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
        return OutputShard(o0, o1, s, s, n_out)
    s0 = max(0, o0 * down // up - (lp - 1))
    s1 = min(n_in, (o1 - 1) * down // up + 1)
    return OutputShard(o0, o1, s0, max(s0, s1), n_out)


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
    return _time_sharded(x_halo, lambda w, r: upfirdn_shard(n_samples, n_taps, up, down, w, r),
                         lambda f, sh: f(x_halo, table, n_taps, up, down, x_first=sh.sample0, out_first=sh.out0,
                                         n_out=sh.out1 - sh.out0),
                         compute, _on_device(fourier._upfirdn_device, 'upfirdn: only complex64 x is built'),
                         group=group, gather=gather)


def oaconvolve_shard(n_in: int, n_taps: int, mode: str, world: int, rank: int) -> OutputShard:
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
        return OutputShard(o0, o1, s, s, n_out)
    b0, b1 = (first + o0) // hop, (first + o1 - 1) // hop
    s0 = min(n_in, max(0, b0 * hop - discard))
    s1 = min(n_in, b1 * hop - discard + nfft)
    return OutputShard(o0, o1, s0, max(s0, s1), n_out)


def oaconvolve_time_sharded(x_halo, h, mode: str = 'full', *, n_samples: int, group=None,
                            compute: Callable | None = None, gather: bool = False):
    """time-sharded oaconvolve(x, h, mode) of a 1-D complex64 capture x of `n_samples` samples and a 1-D
    filter h no longer than it: `x_halo` holds this rank's samples [shard.sample0, shard.sample1) of
    `oaconvolve_shard` (halo included).  Returns this rank's outputs [out0, out1) or, with gather=True, all
    outputs on every rank; the concatenation is bitwise the single-GPU `oaconvolve`.
    `compute(x_halo, hspec, n_taps, nfft, discard, x_first=, out_first=, n_out=)` defaults to the CUDA
    kernel."""
    from . import _plan, fourier
    h = fourier._as_operand(h)
    if h.ndim != 1 or h.shape[0] == 0:
        raise ValueError('oaconvolve_time_sharded: h must be 1-D with non-zero length')
    hspec, n_taps, nfft, discard = fourier._oaconvolve_filter(h, 0)
    first, _ = _plan.oaconvolve_window(mode, n_samples, n_taps)
    return _time_sharded(x_halo, lambda w, r: oaconvolve_shard(n_samples, n_taps, mode, w, r),
                         lambda f, sh: f(x_halo, hspec, n_taps, nfft, discard, x_first=sh.sample0,
                                         out_first=first + sh.out0, n_out=sh.out1 - sh.out0),
                         compute, _on_device(fourier._oaconvolve_device,
                                             'oaconvolve: only a complex64 signal is built'),
                         group=group, gather=gather)


def pfb_shard(n_samples: int, n_taps: int, nchannels: int, hop: int | None, world: int, rank: int) -> FrameShard:
    """time-axis shard of pfb_channelize(x, h, nchannels, hop) for a capture of n_samples samples and an n_taps
    prototype: the frames are split evenly, and rank r reads the samples [frame0*hop, (frame1 - 1)*hop + L) of
    its frames -- a halo of L - hop samples past the frame0*hop of the next rank.  A frame's bits depend only
    on its samples and its global index, so the shards' concatenation is bitwise the single-GPU result."""
    from . import _plan
    hop = nchannels if hop is None else hop
    if n_taps < 1 or not 1 <= hop <= nchannels:
        raise ValueError(f'pfb time shards need n_taps >= 1 and 1 <= hop <= nchannels (got {n_taps}, {hop})')
    T = _plan.pfb_frame_count(n_samples, n_taps, hop)
    f0, f1 = _split(T, world, rank)
    if f1 == f0:
        s = min(f0 * hop, n_samples)
        return FrameShard(f0, f1, s, s, T)
    return FrameShard(f0, f1, f0 * hop, (f1 - 1) * hop + n_taps, T)


def pfb_channelize_time_sharded(x_halo, h, nchannels, hop=None, *, n_samples: int, group=None,
                                compute: Callable | None = None, gather: bool = False):
    """time-sharded pfb_channelize(x, h, nchannels, hop) of a 1-D complex64 capture x of `n_samples` samples:
    `x_halo` holds this rank's samples [shard.sample0, shard.sample1) of `pfb_shard` (halo included).  Returns
    this rank's frames [frame0, frame1) as a (frames, nchannels) tensor or, with gather=True, all frames on
    every rank; the concatenation is bitwise the single-GPU `pfb_channelize`.
    `compute(x_halo, taps, n_taps, nchannels, hop, x_first=, frame_first=, n_frames=)` defaults to the CUDA
    kernel."""
    from . import fourier
    taps, L, K, hop = fourier._pfb_args(h, nchannels, hop)
    return _time_sharded(x_halo, lambda w, r: pfb_shard(n_samples, L, K, hop, w, r),
                         lambda f, sh: f(x_halo, taps, L, K, hop, x_first=sh.sample0, frame_first=sh.frame0,
                                         n_frames=sh.frame1 - sh.frame0),
                         compute, _on_device(fourier._pfb_device, 'pfb_channelize: only a complex64 signal is built'),
                         group=group, gather=gather)


class PfbSynthShard(NamedTuple):
    out0: int       # first output of this rank
    out1: int       # one past its last output
    frame0: int     # first frame it reads
    frame1: int     # one past the last frame it reads (includes the halo)
    n_out: int      # outputs of the whole capture


def pfb_synth_shard(n_frames: int, n_taps: int, nchannels: int, hop: int | None, world: int,
                    rank: int) -> PfbSynthShard:
    """time-axis shard of pfb_synthesize(y, g, hop) for n_frames frames and an n_taps synthesis prototype: the
    (T - 1) * hop + Lg outputs are split evenly, and rank r reads the frames [max(0, ceil((o0 - Lg + 1) / hop)),
    min(T, floor((o1 - 1) / hop) + 1)) that cover its outputs [o0, o1) (an empty range where they all fall in a
    gap between frames, Lg < hop).  An output sums the same terms in the same order wherever it is computed, so
    the shards' concatenation is bitwise the single-GPU result."""
    from . import _plan
    hop = nchannels if hop is None else hop
    if n_taps < 1 or not 1 <= hop <= nchannels or n_frames < 1:
        raise ValueError(f'pfb synthesis shards need n_taps >= 1, 1 <= hop <= nchannels and n_frames >= 1 '
                         f'(got {n_taps}, {hop}, {n_frames})')
    n_out = _plan.pfb_synth_len(n_frames, n_taps, hop)
    o0, o1 = _split(n_out, world, rank)
    f0 = max(0, -(-(o0 - n_taps + 1) // hop))
    f1 = min(n_frames, (o1 - 1) // hop + 1) if o1 > o0 else f0
    f0 = min(f0, n_frames)
    return PfbSynthShard(o0, o1, f0, max(f0, f1), n_out)


def pfb_synthesize_time_sharded(y_halo, g, hop=None, *, n_frames: int, group=None, compute: Callable | None = None,
                                gather: bool = False):
    """time-sharded pfb_synthesize(y, g, hop) of n_frames frame-major frames y (T, K) complex64: `y_halo` holds
    this rank's frames [shard.frame0, shard.frame1) of `pfb_synth_shard` (halo included) as a (frames, K)
    array.  Returns this rank's outputs [out0, out1) or, with gather=True, all outputs on every rank; the
    concatenation is bitwise the single-GPU `pfb_synthesize`.
    `compute(y_halo, taps, n_taps, hop, frame_first=, n_frames_total=, out_first=, n_out=)` defaults to the CUDA
    kernels."""
    from . import fourier
    if y_halo.ndim != 2:
        raise ValueError(f'pfb_synthesize_time_sharded: y_halo must be (frames, nchannels), got {tuple(y_halo.shape)}')
    taps, Lg, K, hop = fourier._pfb_args(g, y_halo.shape[1], hop, what='pfb_synthesize', name='g')
    return _time_sharded(y_halo, lambda w, r: pfb_synth_shard(n_frames, Lg, K, hop, w, r),
                         lambda f, sh: f(y_halo, taps, Lg, hop, frame_first=sh.frame0, n_frames_total=n_frames,
                                         out_first=sh.out0, n_out=sh.out1 - sh.out0),
                         compute, _on_device(fourier._pfb_synth_device,
                                             'pfb_synthesize: only complex64 frames are built'),
                         group=group, gather=gather, ndim=2, unit='frames')


def sosfilt_shard(n_samples: int, n_sections: int, world: int, rank: int) -> OutputShard:
    """time-axis shard of sosfilt for a capture of n_samples samples and n_sections sections: kernel 10's groups
    of L*G samples (anchored at sample 0) are split evenly, so every boundary but the capture's end falls on a
    multiple of L*G.  There is no halo: the samples read are the samples owned."""
    from . import fourier
    L, G, _ = fourier._sosfilt_geometry(n_sections)
    span = L * G
    g0, g1 = _split(-(-n_samples // span), world, rank)
    s0, s1 = min(g0 * span, n_samples), min(g1 * span, n_samples)
    return OutputShard(s0, s1, s0, s1, n_samples)


class SosfiltShardOps:
    """the per-rank device steps of `sosfilt_time_sharded`, through the C-ABI entry points that iqw_sosfilt_c64
    itself runs, so that the shards reproduce one call bit for bit.  One instance serves one shard: `states`
    keeps the chunk states in a workspace that `apply` reads.  (The CPU tests substitute a numpy stand-in with
    the same three methods.)"""

    def __init__(self):
        self._ws = None

    @staticmethod
    def _rows(x):
        from . import _arrays
        xd, _ = _arrays.to_device(x)
        if xd.dtype != torch.complex64:
            raise NotImplementedError(f'sosfilt: only complex64 x is built (got {xd.dtype})')
        return xd.reshape(1, -1).contiguous()

    def states(self, x, sos32) -> torch.Tensor:
        """(n_groups, 2S) complex128: the zero-state final state of each group of the shard"""
        import ctypes
        from . import _lib, fourier
        x2 = self._rows(x)
        S, N = len(sos32), x2.shape[1]
        L, G, _ = fourier._sosfilt_geometry(S)
        g = torch.empty((-(-N // (L * G)), 2 * S), dtype=torch.complex128, device=x2.device)
        ws_bytes = _lib.lib.iqw_sosfilt_workspace_bytes(1, N, S)
        self._ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x2.device)
        _lib.check(_lib.lib.iqw_sosfilt_states_c64(
            ctypes.c_void_p(x2.data_ptr()), 1, N, N, sos32.ctypes.data_as(ctypes.c_void_p), S,
            ctypes.c_void_p(fourier._sosfilt_powers(sos32, x2.device).data_ptr()), ctypes.c_void_p(g.data_ptr()),
            ctypes.c_void_p(self._ws.data_ptr()), ws_bytes, fourier._stream_ptr(x2.device)))
        return g

    def carry(self, g: torch.Tensor, sos32, zi: torch.Tensor | None) -> torch.Tensor:
        """the group states of the whole capture (n_groups, 2S) -> the start state of each group, from zi (2S,)"""
        import ctypes
        from . import _lib, fourier
        S = len(sos32)
        g = g.to(torch.complex128).contiguous().clone()
        if zi is not None:
            zi = zi.to(g.device).to(torch.complex64).contiguous()
        ws_bytes = _lib.lib.iqw_sosfilt_carry_workspace_bytes(1, g.shape[0], S)
        ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=g.device)
        _lib.check(_lib.lib.iqw_sosfilt_carry_c64(
            ctypes.c_void_p(g.data_ptr()), 1, g.shape[0], ctypes.c_void_p(zi.data_ptr() if zi is not None else None),
            S, ctypes.c_void_p(fourier._sosfilt_powers(sos32, g.device).data_ptr()), ctypes.c_void_p(ws.data_ptr()),
            ws_bytes, fourier._stream_ptr(g.device)))
        return g

    def apply(self, x, sos32, s: torch.Tensor, want_zf: bool):
        """the shard's output from the start states s (n_groups, 2S) of its groups -> (y, zf (2S,) or None)"""
        import ctypes
        from . import _lib, fourier
        x2 = self._rows(x)
        S, N = len(sos32), x2.shape[1]
        s = s.to(x2.device).to(torch.complex128).contiguous()
        y = torch.empty_like(x2)
        zf = torch.zeros(2 * S, dtype=torch.complex64, device=x2.device) if want_zf else None
        if N:
            _lib.check(_lib.lib.iqw_sosfilt_apply_c64(
                ctypes.c_void_p(x2.data_ptr()), 1, N, N, sos32.ctypes.data_as(ctypes.c_void_p), S,
                ctypes.c_void_p(fourier._sosfilt_powers(sos32, x2.device).data_ptr()), ctypes.c_void_p(s.data_ptr()),
                ctypes.c_void_p(self._ws.data_ptr()), self._ws.numel(), ctypes.c_void_p(y.data_ptr()), N,
                ctypes.c_void_p(zf.data_ptr() if zf is not None else None), fourier._stream_ptr(x2.device)))
        return y[0], zf


def sosfilt_time_sharded(x_local, sos, *, n_samples: int, zi=None, group=None, compute=None, gather: bool = False):
    """time-sharded sosfilt(sos, x) of a 1-D complex64 capture x of `n_samples` samples: `x_local` holds this
    rank's samples [shard.sample0, shard.sample1) of `sosfilt_shard`.  Each rank runs the states pass on its
    samples; one all_gather shares every group's zero-state final state; every rank folds the whole list in the
    order of one call (a small float64 computation) and filters its own samples from the start states of its
    groups.  Returns this rank's outputs or, with gather=True, all outputs on every rank -- and with `zi` (shape
    (n_sections, 2)) the pair (y, zf), zf the final state of the whole capture on every rank.  The concatenation
    is bitwise the single-GPU `sosfilt`.  `compute` is an object with the methods of `SosfiltShardOps`
    (default: a new `SosfiltShardOps`)."""
    from . import fourier
    sos32 = fourier._sosfilt_sos(sos)
    S = len(sos32)
    zi_t = None
    if zi is not None:
        zi_t = torch.as_tensor(fourier._as_operand(zi))
        if tuple(zi_t.shape) != (S, 2):
            raise ValueError(f'Invalid zi shape. With axis=-1, an input with shape {(n_samples,)!r}, and an sos '
                             f'array with {S} sections, zi must have shape {(S, 2)!r}, got {tuple(zi_t.shape)!r}.')
        zi_t = zi_t.to(torch.complex64).reshape(2 * S)
    world, rank = _world(group)
    L, G, _ = fourier._sosfilt_geometry(S)
    span = L * G
    groups = [-(-(sh.sample1 - sh.sample0) // span) for sh in (sosfilt_shard(n_samples, S, world, r)
                                                                 for r in range(world))]
    last = max([r for r in range(world) if groups[r] > 0], default=world - 1)
    zf = []

    def run(ops, sh):
        g_local = ops.states(x_local, sos32)
        g_all = torch.view_as_complex(gather_rows(torch.view_as_real(g_local.contiguous()), groups, 0, group)
                                      .contiguous())
        first = sum(groups[:rank])
        s = ops.carry(g_all, sos32, zi_t)[first:first + groups[rank]]
        y, f = ops.apply(x_local, sos32, s, want_zf=zi_t is not None and rank == last)
        if zi_t is not None:
            if n_samples == 0:
                f = zi_t
            elif rank != last:
                f = torch.zeros(2 * S, dtype=torch.complex64, device=y.device)
            f = torch.view_as_real(f.to(y.device).reshape(1, 2 * S))
            zf.append(torch.view_as_complex(gather_rows(f, None, 0, group)[last].contiguous()).reshape(S, 2))
        return y

    y = _time_sharded(x_local, lambda w, r: sosfilt_shard(n_samples, S, w, r), run, compute, SosfiltShardOps(),
                      group=group, gather=gather)
    return y if zi is None else (y, zf[0])
