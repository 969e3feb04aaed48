"""sosfilt throughput on one GPU: the workloads of DESIGN.md "Kernel 10" on one row of 2^28 samples and on 8 rows
of 2^25 (seeded complex64 noise on the device).

Per workload and shape: CUDA events over --iters calls after a warm-up (best and median) and the rate; each
pass's time from the library's per-launch event scopes (a separate run); the floors, computed from counts -- HBM:
24 B/sample (x read twice, y written once) at the device-to-device copy bandwidth measured in the same run;
FP32: 20 S fused multiply-adds per sample over the two passes at 37 T FMA/s -- and floor / time for the binding
one; scipy's complex64 sosfilt on this host's CPU at 2^22 samples; and the card's name and power limit.

    python tools/sosfilt_probe.py --out profiles/sosfilt_r07.json
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np
import scipy.signal as ss
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(ROOT))
sys.path.insert(0, ROOT)

from upfirdn_probe import copy_bandwidth, gpu_info, timed  # noqa: E402

WORKLOADS = {
    'I1': ('DC blocker [1, -1, 0, 1, -0.999, 0]', lambda: np.array([[1, -1, 0, 1, -0.999, 0]])),
    'I2': ('butter(4, 0.002)', lambda: ss.butter(4, 0.002, output='sos')),
    'I3': ('ellip(8, 0.1, 80, 0.05)', lambda: ss.ellip(8, 0.1, 80, 0.05, output='sos')),
    'I4': ('ellip(16, 0.1, 100, 0.2)', lambda: ss.ellip(16, 0.1, 100, 0.2, output='sos')),
    'I5': ('butter(32, 0.3)', lambda: ss.butter(32, 0.3, output='sos')),
}
FMA_PER_S = 37e12


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--iters', type=int, default=10)
    ap.add_argument('--log2n', type=int, default=28)
    ap.add_argument('--cpu-log2n', type=int, default=22)
    args = ap.parse_args()
    import iqwaveform_b200 as iqw
    from iqwaveform_b200 import _lib, fourier

    dev = torch.device('cuda', 0)
    g = torch.Generator(device=dev).manual_seed(7)
    n = 1 << args.log2n
    x1 = torch.randn((1, n), dtype=torch.complex64, device=dev, generator=g)
    x8 = x1.reshape(8, n // 8)
    bw = copy_bandwidth(x1, 10)
    rng = np.random.default_rng(7)
    xc = (rng.standard_normal(1 << args.cpu_log2n) + 1j * rng.standard_normal(1 << args.cpu_log2n)).astype(np.complex64)
    out = {'gpu': gpu_info(), 'copy_bandwidth_TBps': bw / 1e12, 'samples': n, 'workloads': {}}
    for name, (desc, make) in WORKLOADS.items():
        sos32 = fourier._sosfilt_sos(make())
        S = len(sos32)
        rad = max(abs(np.roots([1, a1, a2])).max() for a1, a2 in sos32[:, 4:6].astype(np.float64))
        hbm_ms = 24 * n / bw * 1e3
        fp32_ms = 20 * S * n / FMA_PER_S * 1e3
        floor = max(hbm_ms, fp32_ms)
        w = {'sos': desc, 'S': S, 'max_pole_radius': float(rad), 'hbm_floor_ms': hbm_ms, 'fp32_floor_ms': fp32_ms,
             'binding': 'HBM' if hbm_ms >= fp32_ms else 'FP32', 'shapes': {}}
        for shape, x in (('1 x 2^%d' % args.log2n, x1), ('8 x 2^%d' % (args.log2n - 3), x8)):
            ms = timed(lambda: iqw.sosfilt(sos32, x), args.iters, 2)
            _lib.profile(True, fine=True)
            for _ in range(3):
                iqw.sosfilt(sos32, x)
            torch.cuda.synchronize()
            rep = _lib.profile_report()
            _lib.profile(False)
            passes = {k: v[1] / v[0] for k, v in rep.items() if k.startswith('sosfilt')}
            w['shapes'][shape] = {'best_ms': min(ms), 'median_ms': float(np.median(ms)),
                                  'GS_per_s': n / min(ms) / 1e6, 'floor_over_time': floor / min(ms),
                                  'pass_ms': passes}
        t0 = time.perf_counter()
        ss.sosfilt(sos32, xc)
        cpu_s = time.perf_counter() - t0
        w['scipy_cpu'] = {'samples': xc.size, 'seconds': cpu_s, 'MS_per_s': xc.size / cpu_s / 1e6}
        out['workloads'][name] = w
        print(name, json.dumps(w), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(out, f, indent=1)


if __name__ == '__main__':
    main()
