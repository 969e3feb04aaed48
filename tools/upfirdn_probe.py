"""upfirdn throughput on one GPU: workloads W1-W5 of DESIGN.md "Kernel 6" on one channel of 2^28 complex64
samples (2.15 GB, larger than L2), generated on the device from a seed.

Per workload: CUDA events over --iters calls after a warm-up (best and median), GS/s of input, the time
over the HBM floor ((8 n_in + 8 n_out) bytes over the device-to-device copy bandwidth measured in the same
run) and over the FP32 floor (FMA lane-slots over 128 x SMs x max SM clock; real taps take 2 lane-slots
per tap and output, complex taps 4), which floor binds, the SM clock read while the workload runs (the
idle clock is recorded once at the start), and the kernel that served it (torch.profiler, one extra call).
Bars: torch.nn.functional.conv1d over the zero-stuffed input (re / im as channels, stride = down; a
benchmark-only stand-in for the reference's cupy kernel, checked against scipy at a
small size), and scipy.signal.upfirdn on the host at 1/16 of the samples (the reference's host path).

    python tools/upfirdn_probe.py --out profiles/upfirdn_r03.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = {   # name: (up, down, n_taps, complex taps, what)
    'W1': (1, 8, 161, False, 'decimate by 8, 161 real taps'),
    'W2': (147, 160, 3201, False, 'resample 147/160, 3201 real taps'),
    'W3': (4, 1, 81, False, 'upsample by 4, 81 real taps'),
    'W4': (1, 1, 129, True, 'filter, 129 complex taps'),
    'W5': (1, 16, 4097, False, 'narrow channel: decimate by 16, 4097 real taps'),
}


def smi(q: str) -> list[str]:
    """read-only nvidia-smi query of GPU 0"""
    out = subprocess.run(['nvidia-smi', '-i', '0', f'--query-gpu={q}', '--format=csv,noheader'], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    return [s.strip() for s in out.split(',')]


def gpu_info() -> dict:
    name, power, sm, smax = smi('name,power.limit,clocks.sm,clocks.max.sm')
    return {'name': name, 'power_limit': power, 'clocks_sm_idle': sm, 'clocks_max_sm': smax,
            'sm_count': torch.cuda.get_device_properties(0).multi_processor_count, 'torch': torch.__version__}


def clock_under_load(fn, seconds: float = 1.0) -> str:
    """the SM clock read while `fn` runs back to back for `seconds` (the query is taken mid-way)"""
    import threading
    got = {}

    def query():
        time.sleep(seconds / 3)
        got['sm'] = smi('clocks.sm')[0]

    t = threading.Thread(target=query)
    t0 = time.perf_counter()
    t.start()
    while time.perf_counter() - t0 < seconds or t.is_alive():
        fn()
        torch.cuda.synchronize()
    t.join()
    return got['sm']


def timed(fn, iters: int, warmup: int) -> list[float]:
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return ms


def copy_bandwidth(x: torch.Tensor, iters: int) -> float:
    """bytes read + written per second of a device-to-device copy of x"""
    y = torch.empty_like(x)
    ms = timed(lambda: y.copy_(x), iters, 3)
    return 2 * x.numel() * x.element_size() / (min(ms) * 1e-3)


def conv1d_upfirdn(h: torch.Tensor, x: torch.Tensor, up: int, down: int, n_out: int) -> torch.Tensor:
    """benchmark-only stand-in: zero-stuff, then conv1d with (re, im) as channels and stride = down"""
    import torch.nn.functional as F
    L = h.numel()
    xs = torch.zeros((2, x.numel() * up + 2 * (L - 1) + down), dtype=torch.float32, device=x.device)
    xs[:, L - 1:L - 1 + x.numel() * up:up] = torch.view_as_real(x).T
    hf = h.flip(0)
    if h.is_complex():
        w = torch.stack([torch.stack([hf.real, -hf.imag]), torch.stack([hf.imag, hf.real])])
    else:
        z = torch.zeros_like(hf)
        w = torch.stack([torch.stack([hf, z]), torch.stack([z, hf])])
    y = F.conv1d(xs[None], w.float(), stride=down)[0, :, :n_out]
    return torch.complex(y[0], y[1])


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument('--log2n', type=int, default=28)
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--workloads', default=','.join(WORKLOADS))
    ap.add_argument('--skip-bars', action='store_true')
    ap.add_argument('--out', default=None)
    args = ap.parse_args()

    import scipy.signal as ss
    import iqwaveform_b200 as iqw
    from iqwaveform_b200 import _plan

    assert torch.cuda.is_available(), 'the probe measures the GPU; there is no CPU fallback'
    dev = torch.device('cuda', 0)
    info = gpu_info()
    n_in = 1 << args.log2n
    g = torch.Generator(device=dev).manual_seed(20261020)
    x = torch.randn(n_in, dtype=torch.complex64, device=dev, generator=g)
    bw = copy_bandwidth(x, args.iters)
    clock_hz = float(info['clocks_max_sm'].split()[0]) * 1e6
    fma_rate = 128 * info['sm_count'] * clock_hz
    res = {'gpu': info, 'n_in': n_in, 'copy_bandwidth_TBps': bw / 1e12, 'fp32_lane_slots_per_s': fma_rate,
           'iters': args.iters, 'workloads': {}}
    print(json.dumps(res['gpu']), f'copy {bw / 1e12:.2f} TB/s', flush=True)

    rng = np.random.default_rng(3)
    for name in args.workloads.split(','):
        up, down, L, cplx, what = WORKLOADS[name]
        h = rng.standard_normal(L) + (1j * rng.standard_normal(L) if cplx else 0)
        h = (h / np.abs(h).sum()).astype(np.complex64 if cplx else np.float32)
        n_out = _plan.upfirdn_output_len(L, n_in, up, down)
        fn = lambda: iqw.upfirdn(h, x, up, down)       # noqa: E731
        ms = timed(fn, args.iters, args.warmup)
        best, med = min(ms), float(np.median(ms))
        sm_load = clock_under_load(fn)
        hbm_ms = (8 * n_in + 8 * n_out) / bw * 1e3
        lane_slots = n_out * (L / up) * (4 if cplx else 2)
        fp32_ms = lane_slots / fma_rate * 1e3
        row = {'what': what, 'up': up, 'down': down, 'n_taps': L, 'complex_taps': cplx, 'n_out': n_out,
               'best_ms': best, 'median_ms': med, 'GSps_in': n_in / (best * 1e-3) / 1e9,
               'hbm_floor_ms': hbm_ms, 'fp32_floor_ms': fp32_ms, 'binds': 'HBM' if hbm_ms >= fp32_ms else 'FP32',
               'floor_over_time': max(hbm_ms, fp32_ms) / best, 'clocks_sm_under_load': sm_load}
        # which kernel served it, and its own time (torch.profiler, one call)
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        row['profiler_kernels'] = {e.key: e.device_time_total / 1e3 for e in prof.key_averages()
                                   if 'upfirdn' in e.key}
        if not args.skip_bars:
            small = 4096
            xs = x[:small]
            want = ss.upfirdn(h.astype(np.complex128 if cplx else np.float64), xs.cpu().numpy().astype(np.complex128),
                              up, down)
            got = conv1d_upfirdn(torch.from_numpy(h).to(dev), xs, up, down, want.size).cpu().numpy()
            row['conv1d_check_max_rel_err'] = float(np.max(np.abs(got - want)) / np.max(np.abs(want)))
            try:
                cms = timed(lambda: conv1d_upfirdn(torch.from_numpy(h).to(dev), x, up, down, n_out), 5, 1)
                row['conv1d_best_ms'] = min(cms)
                row['conv1d_GSps_in'] = n_in / (min(cms) * 1e-3) / 1e9
            except RuntimeError as e:       # e.g. out of memory for the zero-stuffed input
                row['conv1d_error'] = str(e).splitlines()[0]
                torch.cuda.empty_cache()
            xh = x[:n_in // 16].cpu().numpy()
            t0 = time.perf_counter()
            ss.upfirdn(h, xh, up, down)
            row['scipy_cpu_MSps_in'] = xh.size / (time.perf_counter() - t0) / 1e6
        res['workloads'][name] = row
        print(name, json.dumps({k: v for k, v in row.items() if k != 'what'}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
