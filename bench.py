#!/usr/bin/env python
"""bench.py -- headline benchmark: complex IQ GS/s of persistence_spectrum on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[2], the configuration the metric is quoted on): persistence
spectrum of 100 MS/s complex64 captures, 10 s per channel (1e9 samples), nfft 4096 Hann, 50 %
overlap, quantiles [0.1, 0.5, 0.9, 0.999], dB.  Channels are independent, so the job shards by
channel with no data-path collective: ONE channel per GPU ("weak" scaling; 8 GPUs = the full
8-channel config), plus the NCCL all_gather of the (4, 4096) result rows the north-star names.

A step = one full pass of the hot path over one channel per GPU:
    kernel 1 (STFT -> |X|^2, 8 GB in / 8 GB out)  ->  kernel 2 (exact per-bin order statistics).
`value`  : device-resident input, CUDA events on the launching stream, max over ranks.
`e2e`    : the same call with the capture in pinned HOST memory (host->device copy of 8 GB and
           device->host read of the result inside the timed region).
`roofline`: dominant kernel's algorithmic bytes / its measured duration (library profile events
           recorded inside the timed region) against MEASURED_PEAKS.json.
`cpu_baseline`: the reference's own power_spectral_density (unmodified package installed to
           baseline/_ref by __graft_entry__.build(), imported through oracle/ref_shim.py;
           kind "reference") on a bounded sample of the workload; the numpy/scipy oracle port
           (kind "port") only when baseline/_ref is absent.
--impl reference times that CPU arm alone (rank 0), as the reference arm.
`extra.configs`: one-shot timings (best of 3) of BASELINE configs[1], configs[3] (30 s half-capture)
           and the configs[4] sweep, N = 1 only.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FS = 100e6
NFFT = 4096
OVERLAP = 0.5
STATS = [0.1, 0.5, 0.9, 0.999]
WINDOW = 'hann'
SAMPLES_PER_CHANNEL = 1_000_000_000
CPU_SAMPLE = 1 << 25          # bounded sample for the CPU arms (0.34 s of one channel)
METRIC = 'complex IQ GS/s for persistence_spectrum'
UNIT = 'GS/s'


def workload_config(n_gpus, samples):
    """the workload both arms name (identical in the GPU and the reference line).  The GPU arm processes
    it in full every step; the CPU arms process the bounded sample stated under `cpu_arms_step`."""
    return {
        'workload': 'BASELINE configs[2] persistence_spectrum, sharded by channel: 1 channel per GPU',
        'channels': n_gpus, 'channels_per_gpu': 1, 'samples_per_channel': samples,
        'sample_rate_hz': FS, 'nfft': NFFT, 'window': WINDOW, 'overlap': OVERLAP,
        'statistics': STATS, 'dB': True,
        'frames_per_channel': (samples - NFFT) // (NFFT // 2) + 1,
        'cpu_arms_step': {'what': 'cpu_baseline and --impl reference: ONE CPU process (rank 0 at every N) on a '
                                  'bounded sample of one channel per step, same nfft/window/overlap/statistics',
                          'channels': 1, 'samples_per_channel': CPU_SAMPLE,
                          'frames_per_channel': (CPU_SAMPLE - NFFT) // (NFFT // 2) + 1},
        'l2': 'no flush: per-step input (8 B/sample) and spectrogram (8 B/sample) exceed the 126 MB L2',
        'collective': 'nccl all_gather of the (4, 4096) fp32 result per channel' if n_gpus > 1 else 'none',
    }


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference
# ------------------------------------------------------------------------------------------------
def cpu_capture(n, seed=1234):
    import numpy as np

    rng = np.random.default_rng(seed)
    x = np.empty(n, dtype=np.complex64)
    chunk = 1 << 22
    for s in range(0, n, chunk):
        m = min(chunk, n - s)
        k = np.arange(s, s + m, dtype=np.float64)
        z = (rng.standard_normal(m) + 1j * rng.standard_normal(m)) * math.sqrt(0.5)
        for f, a in ((0.0651, 0.5), (-0.2148, 0.05), (0.3256, 3.0)):
            z += a * np.exp(2j * np.pi * ((f * k) % 1.0))
        x[s:s + m] = z
    return x


def reference_api():
    """-> (persistence-spectrum callable, kind).  kind "reference": the UNMODIFIED reference package
    (fourier.py:1236-1327, stock code path) from /root/reference or its installed copy baseline/_ref;
    kind "port": the numpy/scipy oracle restatement, only when neither is present"""
    from oracle import ref_shim

    ref = ref_shim.load()
    if ref is not None:
        return ref.fourier.power_spectral_density, 'reference'
    from oracle import iqw_oracle as orc

    return orc.persistence_spectrum, 'port'


def cpu_step(x, fn=None):
    fn = fn or reference_api()[0]
    return fn(x[None, :], fs=FS, window=WINDOW, resolution=FS / NFFT, fractional_overlap=OVERLAP,
              statistics=STATS, dB=True, axis=1)


def cpu_cores():
    return max((os.cpu_count() or 1) // 2, 1)


def cpu_sample_note(kind):
    what = ('the reference\'s own iqwaveform.fourier.power_spectral_density, unmodified (baseline/_ref)'
            if kind == 'reference' else 'numpy/scipy oracle port of the reference (baseline/_ref absent)')
    return (f'1 channel x {CPU_SAMPLE} samples per step ({CPU_SAMPLE / FS:.3f} s of the 10 s capture), same '
            f'nfft/overlap/statistics; {what}; scipy.fft workers = cpu_count//2 = {cpu_cores()} of '
            f'{os.cpu_count()} cores (the reference policy, fourier.py:214), numpy stages single-threaded '
            f'as in the reference')


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return None
    fn, kind = reference_api()
    x = cpu_capture(CPU_SAMPLE)
    for _ in range(max(args.warmup, 1)):
        cpu_step(x, fn)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_step(x, fn)
    dt = time.perf_counter() - t0
    value = CPU_SAMPLE * args.steps / dt / 1e9
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': max(args.warmup, 1), 'ms_per_step': dt / args.steps * 1e3,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic',
        # same `config` as the GPU arm (the workload the metric is quoted on); what one step of THIS arm
        # really processes is config.cpu_arms_step and the `step_processed` key below
        'config': workload_config(args.gpus, SAMPLES_PER_CHANNEL),
        'step_processed': {'channels': 1, 'samples_per_channel': CPU_SAMPLE, 'processes': 1,
                           'note': 'one CPU process at every N; value = samples processed / wall time'},
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cpu_cores(), 'kind': kind,
                         'sample': cpu_sample_note(kind)},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    return line


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region"""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '50',
                 '-i', str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.25)
        self.proc.terminate()
        self.thread.join(timeout=2)
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'samples': len(sm), 'reasons': sorted(reasons)}


def device_capture(torch, n, seed, device):
    g = torch.Generator(device=device).manual_seed(seed)
    x = torch.empty(n, dtype=torch.complex64, device=device)
    xr = torch.view_as_real(x)
    chunk = 1 << 26
    for s in range(0, n, chunk):
        m = min(chunk, n - s)
        xr[s:s + m].normal_(0.0, math.sqrt(0.5), generator=g)
        k = torch.arange(s, s + m, device=device, dtype=torch.float64)
        for f, a in ((0.0651, 0.5), (-0.2148, 0.05), (0.3256, 3.0)):
            ph = (2 * math.pi) * torch.remainder(f * k, 1.0)
            xr[s:s + m, 0] += (a * torch.cos(ph)).float()
            xr[s:s + m, 1] += (a * torch.sin(ph)).float()
    return x


def measured_peak():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            return float(json.load(f)['hbm_gbs']), 'MEASURED_PEAKS.json hbm_gbs (of measured)'
    except (OSError, KeyError, ValueError):
        return 6650.0, 'B200_PROFILING.md fallback 6.65 TB/s (of fallback)'


def ncu_traffic(kernel):
    """dram bytes per launch from the committed ncu --set full capture of this workload, if any"""
    try:
        with open(os.path.join(ROOT, 'profiles', 'ncu_traffic.json')) as f:
            return json.load(f).get(kernel)
    except (OSError, ValueError):
        return None


def _timed(torch, fn, reps=3):
    out = fn(); del out
    torch.cuda.synchronize()
    best = float('inf')
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(reps):
        e0.record(); out = fn(); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1)); del out
    return best


def extra_configs(torch, iqw, dev, peak):
    """one-shot timings of the other BASELINE.json configs on one GPU: device-resident synthetic input
    larger than L2, CUDA events on the launching stream, best of 3 after one warm-up call"""
    rows = []

    def row(name, n, ms, bps):
        gbs = n * bps / ms / 1e6
        rows.append({'config': name, 'samples': n, 'ms': round(ms, 4), 'GS_per_s': round(n / ms / 1e6, 2),
                     'algorithmic_bytes_per_sample': bps, 'algorithmic_GBps': round(gbs, 1),
                     'frac_of_measured_hbm_peak': round(gbs / peak, 4)})

    # configs[0]: the reference's own CPU-runnable case, plain call and as one captured CUDA graph
    n = 15_360_000
    x = device_capture(torch, n, 1, dev).view(1, n)
    kw0 = dict(fs=15.36e6, window='hann', resolution=15e3, fractional_overlap=0.5, statistics=[0.5, 0.99], dB=True, axis=1)
    row('configs[0] persistence_spectrum 15.36 MS/s x 1 s, nfft 1024 hann 50 %, q = [0.5, 0.99]', n,
        _timed(torch, lambda: iqw.persistence_spectrum(x, **kw0), reps=5), 24)
    g = iqw.GraphedCall(iqw.persistence_spectrum, x, **kw0)
    row('configs[0] same call replayed as one CUDA graph (iqw.GraphedCall)', n, _timed(torch, lambda: g(), reps=5), 24)
    del x, g
    # configs[1]: stft/spectrogram, 100 MS/s x 10 s, nfft 2048 Blackman-Harris, 50 % overlap, dB
    n = 1_000_000_000
    x = device_capture(torch, n, 2, dev)
    kw = dict(fs=100e6, window='blackmanharris', nperseg=2048, noverlap=1024, return_axis_arrays=False)
    row('configs[1] spectrogram dB, 1e9 samples, nfft 2048 blackmanharris 50 %', n,
        _timed(torch, lambda: iqw.spectrogram(x, dB=True, **kw)), 16)
    row('configs[1] spectrogram power, same capture', n, _timed(torch, lambda: iqw.spectrogram(x, **kw)), 16)
    # configs[2] with reducible statistics only: no spectrogram is materialised (8 B/sample compulsory)
    kw3 = dict(fs=FS, window=WINDOW, resolution=FS / NFFT, fractional_overlap=OVERLAP, dB=True, axis=1)
    row('configs[2] persistence_spectrum statistics=[mean, max] (fused, nothing materialised)', n,
        _timed(torch, lambda: iqw.persistence_spectrum(x.view(1, n), statistics=['mean', 'max'], **kw3)), 8)
    del x
    torch.cuda.empty_cache()
    # configs[3]: iq_to_bin_power, 1 ms bins at 245.76 MS/s; the 30 s half-capture one GPU of a pair holds
    n = 245_760 * 30_000
    x = torch.empty(n, dtype=torch.complex64, device=dev)
    xr = torch.view_as_real(x)
    for s0 in range(0, n, 1 << 28):
        xr[s0:s0 + (1 << 28)].normal_(0.0, 0.7)
    for kind in ('mean', 'peak'):
        row(f'configs[3] iq_to_bin_power {kind}, 1 ms bins, 245.76 MS/s x 30 s (59 GB)', n,
            _timed(torch, lambda: iqw.iq_to_bin_power(x, 1 / 245.76e6, 1e-3, kind=kind)), 8)
    del x, xr
    torch.cuda.empty_cache()
    # configs[4]: nfft sweep at 50 % and 75 % overlap
    n = 1 << 28
    x = torch.randn(n, dtype=torch.complex64, device=dev)
    for nfft in (64, 256, 1024, 8192, 65536):
        for ov in (0.5, 0.75):
            nov = int(nfft * ov)
            row(f'configs[4] spectrogram nfft {nfft} overlap {ov:.2f}', n,
                _timed(torch, lambda: iqw.spectrogram(x, fs=1e8, window='hann', nperseg=nfft, noverlap=nov,
                                                      return_axis_arrays=False)), 8 + 4 * nfft / (nfft - nov))
    del x
    torch.cuda.empty_cache()
    return rows


def dump_outputs(out_dir, arrays):
    """what the last timed step returned, one float32 `<name>.npy` per array: the inputs are regenerated from fixed
    seeds, so two builds run with the same arguments can be compared output for output"""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), t.float().cpu().numpy())


def run_b200(args):
    import torch
    import torch.distributed as dist

    import iqwaveform_b200 as iqw
    from iqwaveform_b200 import _lib

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a GPU (the product path has no CPU fallback)')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    numa_cpus = None
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        # one process per GPU: keep each rank's pinned host buffer on the socket its GPU hangs off
        numa_cpus = iqw.distributed.bind_to_gpu_numa_node(local)
        dist.init_process_group('nccl', device_id=dev)
    n = args.samples
    warmup = max(args.warmup, 3)

    x = device_capture(torch, n, 1234 + 1000 * rank, dev).view(1, n)
    kw = dict(fs=FS, window=WINDOW, resolution=FS / NFFT, fractional_overlap=OVERLAP,
              statistics=STATS, dB=True, axis=1)

    gathered = {}

    def step(inp):
        out = iqw.persistence_spectrum(inp, **kw)
        if world > 1:       # the (4, 4096) rows of every channel on every rank: one NCCL all_gather
            gathered['rows'] = iqw.distributed.gather_rows(out if out.is_cuda else out.to(dev))
        return out

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local) if rank == 0 else None     # clocks under load: warm-up + timed region
    for _ in range(warmup):
        step(x)
    barrier()

    # ---- device-resident timed region --------------------------------------------------------
    _lib.profile(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        out = step(x)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump = {'persistence_spectrum': out}
        if world > 1:
            dump['gathered_rows'] = gathered['rows']
        dump_outputs(args.dump_outputs, dump)
    del out
    prof = _lib.profile_report()
    _lib.profile(False)
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = world * n * args.steps / (ms * 1e-3) / 1e9

    # ---- N > 1: the gathered rows of a FOREIGN channel equal rank 0's own computation of that channel --
    shard_parity = None
    if world > 1:
        rows = gathered['rows'].clone()                 # (world, 4, 4096) of the last timed step
        if rank == 0:
            other = world - 1                           # the capture of the last rank, regenerated from its seed
            xf = device_capture(torch, n, 1234 + 1000 * other, dev).view(1, n)
            mine = iqw.persistence_spectrum(xf, **kw)
            shard_parity = bool(torch.equal(mine[0], rows[other])) and bool(torch.isfinite(rows).all())
            del xf, mine
        barrier()

    # ---- end to end: pinned host input, result read back ---------------------------------------
    e2e = None
    if not args.no_e2e:
        host = torch.empty((1, n), dtype=torch.complex64, pin_memory=True)
        host.copy_(x)
        torch.cuda.synchronize()
        res = step(host)          # warm-up (allocator, pinned result buffer)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            res = step(host)
        barrier()
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
        # the ceiling of this metric: the same pinned buffer copied to the device and nothing else, every
        # rank at the same time (shared PCIe uplinks / host memory included), same barrier bracket
        dst = torch.empty((1, n), dtype=torch.complex64, device=dev)
        dst.copy_(host, non_blocking=True)
        barrier()
        c0 = time.perf_counter()
        for _ in range(3):
            dst.copy_(host, non_blocking=True)
        barrier()
        dc = (time.perf_counter() - c0) / 3
        t = torch.tensor([dc], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dc = float(t.item())
        del dst
        e2e = {'value': world * n * args.steps / dt / 1e9, 'unit': UNIT,
               'h2d_bytes_per_step': world * n * 8,
               'd2h_bytes_per_step': world * res.numel() * 4,
               'ms_per_step': dt / args.steps * 1e3,
               'api': 'iqwaveform_b200.persistence_spectrum(pinned CPU torch tensor) -> CPU tensor',
               'h2d_ceiling': {'value': world * n / dc / 1e9, 'unit': UNIT, 'ms_per_step': dc * 1e3,
                               'GBps_per_gpu': n * 8 / dc / 1e9,
                               'what': 'measured here: pure pinned host->device copy of the same buffers, all '
                                       'ranks at once, max over ranks, mean of 3'},
               'frac_of_h2d_ceiling': round((dc * args.steps) / dt, 4),
               'host_cpus_rank0': numa_cpus}
        del host

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return None

    # ---- roofline of the dominant kernel -------------------------------------------------------
    T = (n - NFFT) // (NFFT // 2) + 1
    alg_bytes = {                       # algorithmic bytes per launch (DESIGN.md section 5)
        'stft_kernel': 8 * n + 4 * T * NFFT,            # read each sample once, write |X|^2 once
        'stats_bracket_pass': 4 * T * NFFT,             # read |X|^2 once (candidate lists are overhead)
    }
    peak, peak_src = measured_peak()
    stages, launches = [], 0
    for name, (cnt, tot) in sorted(prof.items(), key=lambda kv: -kv[1][1]):
        launches += cnt
        avg = tot / cnt
        b = alg_bytes.get(name)
        gbs = b / (avg * 1e-3) / 1e9 if (b and avg > 0.01) else None
        stages.append({'kernel': name, 'launches': cnt, 'avg_ms': round(avg, 4),
                       'share': round(tot / ms, 4),
                       'algorithmic_GBps': round(gbs, 1) if gbs else None,
                       'frac': round(gbs / peak, 4) if gbs else None})
    top = next(s for s in stages if s['algorithmic_GBps'])
    roofline = {'bound': 'hbm', 'kernel': top['kernel'], 'achieved': top['algorithmic_GBps'],
                'peak': peak, 'unit': 'GB/s', 'frac': top['frac'], 'peak_source': peak_src,
                'traffic': ncu_traffic(top['kernel']),
                'algorithmic_bytes_per_launch': alg_bytes[top['kernel']],
                'avg_launch_ms': top['avg_ms'], 'share_of_step': top['share'],
                # whole pipeline against the two lower bounds of SURVEY.md 8d
                # (per GPU: the aggregate value divided by the number of GPUs, each against one GPU's peak)
                'pipeline_materialise_once_frac': round(24 * value / world / peak, 4),
                'pipeline_compulsory_frac': round(8 * value / world / peak, 4),
                'stages': stages}

    # ---- CPU baseline on a bounded sample ------------------------------------------------------
    cpu = None
    if world == 1 and not args.no_cpu:
        fn, kind = reference_api()
        xc = cpu_capture(CPU_SAMPLE)
        cpu_step(xc, fn)
        best = float('inf')
        for _ in range(2):
            t0 = time.perf_counter(); cpu_step(xc, fn); best = min(best, time.perf_counter() - t0)
        cpu = {'value': CPU_SAMPLE / best / 1e9, 'unit': UNIT, 'cores': cpu_cores(), 'kind': kind,
               'sample': cpu_sample_note(kind) + '; best of 2 after 1 warm-up'}

    # ---- the other BASELINE configs, one-shot (N = 1 only) -----------------------------------------
    extra = None
    if world == 1 and not args.no_extra:
        del x
        torch.cuda.empty_cache()
        extra = {'configs': extra_configs(torch, iqw, dev, peak)}

    line = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
        'warmup': warmup, 'ms_per_step': ms / args.steps, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(world, n), 'clocks': clocks, 'e2e': e2e,
        'gpu_launches': launches, 'roofline': roofline, 'cpu_baseline': cpu, 'impl': 'b200',
    }
    if shard_parity is not None:
        line['shard_parity'] = shard_parity
        line['shard_parity_what'] = ('rank 0 regenerated the last rank\'s capture from its seed, ran the '
                                     'persistence spectrum locally and compared it bit for bit (torch.equal) '
                                     'with that channel\'s rows of the NCCL all_gather')
    if extra is not None:
        line['extra'] = extra
    if world > 1:
        dist.destroy_process_group()
    return line


class QuietStdout:
    """everything libraries print to fd 1 while the benchmark runs (NCCL's version banner, ...)
    goes to stderr, so that stdout carries exactly one JSON line"""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--samples', type=int, default=SAMPLES_PER_CHANNEL,
                    help='samples per channel (default: the full 10 s capture)')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-extra', action='store_true', help='skip the one-shot timings of the other configs')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the result of the last timed step as DIR/persistence_spectrum.npy (float32, '
                         '4 quantile rows x 4096 bins per channel) and, on more than one GPU, the all-gathered rows '
                         'of every channel as DIR/gathered_rows.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs writes the outputs of the GPU path (--impl b200)')
    if args.impl == 'reference':
        with QuietStdout():
            line = run_reference(args)
        if line is not None:
            print(json.dumps(line), flush=True)
        return 0
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if args.gpus > 1 and world == 1:
        # convenience: re-launch under torchrun, one rank per GPU
        cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1',
               f'--nproc-per-node={args.gpus}', '--master-addr', '127.0.0.1', '--master-port', '29517',
               os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    with QuietStdout():
        line = run_b200(args)
    if line is not None:
        print(json.dumps(line), flush=True)
    return 0


if __name__ == '__main__':
    sys.exit(main())
