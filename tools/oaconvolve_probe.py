"""oaconvolve throughput on one GPU: one channel of 2^28 complex64 samples (2.15 GB, larger than L2), full mode,
generated on the device from a seed, for the filters of DESIGN.md "Kernel 7".

Per workload: CUDA events over --iters calls after a warm-up (best and median), GS/s of output, the time over
the HBM floor (16 B per output sample over the device-to-device copy bandwidth measured in the same run) and
over the FP32 floor ((2*5*nfft*log2(nfft)/hop + 6) flop per output over 2 x 128 x SMs x max SM clock), the
kernel's share of the call time (torch.profiler, one extra call), and in the same run:
  * upfirdn(h, x) with the same taps (the direct kernel; the crossover),
  * the fused ola_filter kernel (iqw_ola_filter_c64, rect window, every bin kept) at the same nfft with
    hop = nfft: the same two transforms per block, so its blocks/s times oaconvolve's hop is the rate
    oaconvolve would reach at ola_filter's speed (ola_filter cannot take hop = nfft - nfft/R),
  * scipy.signal.oaconvolve on the host at 1/16 of the samples.

    python tools/oaconvolve_probe.py --out profiles/oaconvolve_r04.json
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

from upfirdn_probe import clock_under_load, copy_bandwidth, gpu_info, timed  # noqa: E402

WORKLOADS = {   # name: (n_taps, complex taps, what)
    'F161': (161, False, '161 real taps (firwin)'),
    'F1025': (1025, False, '1025 real taps (firwin)'),
    'F4097': (4097, False, '4097 real taps (firwin)'),
    'C129': (129, True, '129 complex taps (firwin, shifted by fs/8)'),
}


def taps(M: int, cplx: bool) -> np.ndarray:
    import scipy.signal as ss
    h = ss.firwin(M, 0.1)
    if cplx:
        return (h * np.exp(2j * np.pi * np.arange(M) / 8)).astype(np.complex64)
    return h.astype(np.float32)


def ola_blocks_per_s(x: torch.Tensor, nfft: int, iters: int) -> float:
    """blocks per second of the fused ola_filter kernel at hop = nfft (rect window, every bin kept)"""
    from iqwaveform_b200 import _lib
    n_frames = x.numel() // nfft
    w = torch.ones(nfft, dtype=torch.float32, device=x.device)
    out = torch.empty(n_frames * nfft, dtype=torch.complex64, device=x.device)
    sp = ctypes.c_void_p(torch.cuda.current_stream(x.device).cuda_stream)

    def fn():
        _lib.check(_lib.lib.iqw_ola_filter_c64(ctypes.c_void_p(x.data_ptr()), 1, x.numel(), x.numel(),
                                               ctypes.c_void_p(w.data_ptr()), nfft, nfft, n_frames, 0, nfft,
                                               ctypes.c_void_p(out.data_ptr()), out.numel(), sp))
    ms = timed(fn, iters, 3)
    return n_frames / (min(ms) * 1e-3)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument('--log2n', type=int, default=28)
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--workloads', default=','.join(WORKLOADS))
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
    flop_rate = 2 * 128 * info['sm_count'] * clock_hz
    res = {'gpu': info, 'n_in': n_in, 'mode': 'full', 'copy_bandwidth_TBps': bw / 1e12, 'fp32_flop_per_s': flop_rate,
           'iters': args.iters, 'workloads': {}}
    print(json.dumps(res['gpu']), f'copy {bw / 1e12:.2f} TB/s', flush=True)

    ola_cache = {}
    for name in args.workloads.split(','):
        M, cplx, what = WORKLOADS[name]
        h = taps(M, cplx)
        nfft, discard = _plan.oaconvolve_plan(M)
        hop = nfft - discard
        n_out = n_in + M - 1
        fn = lambda: iqw.oaconvolve(x, h)       # noqa: E731
        ms = timed(fn, args.iters, args.warmup)
        best, med = min(ms), float(np.median(ms))
        hbm_ms = 16 * n_out / bw * 1e3
        flop = (2 * 5 * nfft * np.log2(nfft) / hop + 6) * n_out
        fp32_ms = flop / flop_rate * 1e3
        row = {'what': what, 'n_taps': M, 'complex_taps': cplx, 'nfft': nfft, 'discard': discard, 'hop': hop,
               'n_out': n_out, 'best_ms': best, 'median_ms': med, 'GSps_out': n_out / (best * 1e-3) / 1e9,
               'hbm_floor_ms': hbm_ms, 'fp32_floor_ms': fp32_ms, 'binds': 'HBM' if hbm_ms >= fp32_ms else 'FP32',
               'floor_over_time': max(hbm_ms, fp32_ms) / best, 'clocks_sm_under_load': clock_under_load(fn)}
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        wall_ms = (time.perf_counter() - t0) * 1e3
        kern = {e.key: e.device_time_total / 1e3 for e in prof.key_averages() if 'oaconvolve' in e.key}
        row['profiler_kernels_ms'] = kern
        row['kernel_share_of_best_call'] = sum(kern.values()) / best
        row['profiled_call_wall_ms'] = wall_ms
        # the direct kernel with the same taps
        ums = timed(lambda: iqw.upfirdn(h, x), max(3, args.iters // 4), 1)
        row['upfirdn_best_ms'] = min(ums)
        row['upfirdn_GSps_out'] = n_out / (min(ums) * 1e-3) / 1e9
        row['speedup_over_upfirdn'] = min(ums) / best
        # ola_filter's transform rate at the same nfft, as outputs/s at this hop
        if nfft not in ola_cache:
            ola_cache[nfft] = ola_blocks_per_s(x, nfft, args.iters)
        row['ola_filter_blocks_per_s'] = ola_cache[nfft]
        row['ola_equivalent_GSps_out'] = ola_cache[nfft] * hop / 1e9
        row['over_ola_equivalent'] = row['GSps_out'] / row['ola_equivalent_GSps_out']
        xh = x[:n_in // 16].cpu().numpy()
        t0 = time.perf_counter()
        ss.oaconvolve(xh, h)
        row['scipy_cpu_MSps_out'] = (xh.size + M - 1) / (time.perf_counter() - t0) / 1e6
        res['workloads'][name] = row
        print(name, json.dumps({k: v for k, v in row.items() if k != 'what'}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
