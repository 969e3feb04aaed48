"""pfb_synthesize throughput on one GPU: one channel, frames made by pfb_channelize of a seeded 2^28-sample
complex64 capture on the device, the workloads of DESIGN.md "Kernel 9".

Per workload: CUDA events over --iters calls after a warm-up (best and median), GS/s of output, the HBM floors --
the two-kernel design moves 8 K/hop (read y) + 8 K/hop (write u) + 8 K/hop (read u once) + 8 (write) bytes per
output sample, a fused kernel 8 K/hop + 8 -- over the device-to-device copy bandwidth measured in the same run,
and floor / time; each kernel's share of a call (torch.profiler, a separate call); the rate relative to
pfb_channelize at the same (K, L, hop), output samples of one against input samples of the other; the
round-trip SNR of S2 over the interior; and the card's name and power limit.

    python tools/pfb_synth_probe.py --out profiles/pfb_synth_r06.json
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(ROOT))
sys.path.insert(0, ROOT)

from upfirdn_probe import clock_under_load, copy_bandwidth, gpu_info, timed  # noqa: E402

WORKLOADS = {   # name: (K, L = Lg, hop as a fraction of K, reconstruction pair)
    'S1': (1024, 8192, 1, False),
    'S2': (1024, 8192, 2, True),
    'S3': (64, 1024, 1, False),
    'S4': (8192, 32768, 1, False),
}


def prototypes(K: int, L: int, hop: int, pair: bool) -> tuple[np.ndarray, np.ndarray]:
    """(h, g): the docstring's reconstruction pair, or the same Kaiser firwin prototype for both"""
    import scipy.signal as ss
    h = ss.firwin(L, 1.0 / K, window=('kaiser', 9.0))
    if not pair:
        return h.astype(np.float32), h.astype(np.float32)
    g = ss.firwin(L, 2.0 / K, window=('kaiser', 9.0))
    return h.astype(np.float32), (g * hop / (K * np.sum(g * h))).astype(np.float32)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument('--log2n', type=int, default=28)
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--workloads', default=','.join(WORKLOADS))
    ap.add_argument('--out', default=None)
    args = ap.parse_args()

    import iqwaveform_b200 as iqw
    from iqwaveform_b200 import _plan

    assert torch.cuda.is_available(), 'the probe measures the GPU; there is no CPU fallback'
    dev = torch.device('cuda', 0)
    info = gpu_info()
    N = 1 << args.log2n
    gen = torch.Generator(device=dev).manual_seed(20261021)
    x = torch.randn(N, dtype=torch.complex64, device=dev, generator=gen)
    bw = copy_bandwidth(x, args.iters)
    res = {'gpu': info, 'n_in': N, 'copy_bandwidth_TBps': bw / 1e12, 'iters': args.iters, 'workloads': {}}
    print(json.dumps(res['gpu']), f'copy {bw / 1e12:.2f} TB/s', flush=True)

    for name in args.workloads.split(','):
        K, L, div, pair = WORKLOADS[name]
        hop = K // div
        h, g = prototypes(K, L, hop, pair)
        y = iqw.pfb_channelize(x, h, K, hop)
        T = y.shape[0]
        n_out = _plan.pfb_synth_len(T, L, hop)
        fn = lambda: iqw.pfb_synthesize(y, g, hop)       # noqa: E731
        ms = timed(fn, args.iters, args.warmup)
        best, med = min(ms), float(np.median(ms))
        two_ms = n_out * (24 * K / hop + 8) / bw * 1e3
        fused_ms = n_out * (8 * K / hop + 8) / bw * 1e3
        row = {'K': K, 'L': L, 'hop': hop, 'n_frames': T, 'n_out': n_out, 'best_ms': best, 'median_ms': med,
               'GSps_out': n_out / (best * 1e-3) / 1e9, 'hbm_floor_two_kernel_ms': two_ms,
               'hbm_floor_fused_ms': fused_ms, 'two_kernel_floor_over_time': two_ms / best,
               'fused_floor_over_time': fused_ms / best, 'clocks_sm_under_load': clock_under_load(fn)}
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        kern = {e.key: e.device_time_total / 1e3 for e in prof.key_averages() if 'pfb' in e.key}
        row['profiler_kernels_ms'] = kern
        row['kernel_share_of_best_call'] = {k: v / best for k, v in kern.items()}
        cms = timed(lambda: iqw.pfb_channelize(x, h, K, hop), args.iters, args.warmup)
        row['channelize_best_ms'] = min(cms)
        row['channelize_GSps_in'] = N / (min(cms) * 1e-3) / 1e9
        row['rate_over_channelize'] = row['GSps_out'] / row['channelize_GSps_in']
        if pair:
            xr = fn()
            e = 8 * K
            ref = x[e:n_out - e].to(torch.complex128)
            err = xr[e:n_out - e].to(torch.complex128) - ref
            row['round_trip_snr_dB'] = float(10 * torch.log10(ref.abs().square().sum() / err.abs().square().sum()))
            del xr, ref, err
        del y
        torch.cuda.empty_cache()
        res['workloads'][name] = row
        print(name, json.dumps(row), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
