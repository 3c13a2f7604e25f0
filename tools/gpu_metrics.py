"""Timings of the image quality kernels and of the Wald-protocol evaluation -> one JSON (default profiles/metrics_b200.json).

    python tools/gpu_metrics.py [--out profiles/metrics_b200.json]

(a) dsen2_image_quality alone (CUDA events, mean of 20 runs after a warm-up; inputs larger than L2) at the Wald full tile
    5490^2 x 6 (float32 and float64 estimates against a uint16 reference) and at 10980^2 x 6, with and without nodata; the
    bytes of both images read once per unit time, against a device-to-device copy measured in the same run.
(b) The stages of evaluate.wald_device on a full bench.synth_tile (10980^2, a seeded random DSen2).
(c) The numpy oracle on a 1000^2 x 6 crop on the host cores.
The card's name, power limit and maximum SM clock are read in the same run."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from dsen2_b200 import _capi, evaluate, metrics  # noqa: E402
from dsen2_b200.DSen2Net import s2model  # noqa: E402
from oracle import metrics_oracle as mo  # noqa: E402


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, power, clock = [s.strip() for s in q.split(',')]
    return {'name': name, 'power_limit': power, 'max_sm_clock': clock}


def timed(fn, reps=20):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def copy_peak():
    x = torch.empty(4 << 30, dtype=torch.uint8, device='cuda')
    y = torch.empty_like(x)
    ms = timed(lambda: y.copy_(x), 10)
    return 2 * x.numel() / ms / 1e6                     # GB/s, read + write


def kernel_case(n, est_dtype, nodata, peak):
    g = torch.Generator(device='cuda').manual_seed(n)
    ref = (torch.rand((n, n, 6), generator=g, device='cuda') * 8000 + 500).round_().to(torch.int16)
    if nodata is not None:
        ref[:, : n // 10] = 0                            # a swath edge of nodata
    est = ref.to(est_dtype) + torch.randn((n, n, 6), generator=g, device='cuda', dtype=est_dtype) * 100
    ref = ref.view(torch.uint16)
    H, W, C, ce, cr, v = metrics.check_args(est.shape, est.dtype, ref.shape, ref.dtype, nodata)
    lib = _capi.lib()
    nbytes = lib.dsen2_image_quality_workspace_bytes(H, W, C)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device='cuda')
    sums = torch.empty((5 * C + 2,), dtype=torch.float64, device='cuda')

    def run():
        _capi.check(lib.dsen2_image_quality(_capi.ptr(est), ce, _capi.ptr(ref), cr, H, W, C, int(v is not None),
                                            0.0 if v is None else v, _capi.ptr(ws), nbytes, _capi.ptr(sums),
                                            _capi.stream_ptr()), "dsen2_image_quality")
    ms = timed(run)
    read = est.numel() * est.element_size() + ref.numel() * 2
    del est, ref, ws
    torch.cuda.empty_cache()
    return {'size': n, 'bands': 6, 'est': str(est_dtype)[6:], 'ref': 'uint16', 'nodata': nodata, 'ms': round(ms, 3),
            'bytes_read_once': read, 'GB_per_s': round(read / ms / 1e6, 1), 'share_of_copy_rate': round(read / ms / 1e6 / peak, 3)}


def wald_stages():
    d10, d20 = bench.synth_tile(torch, 10980, 10980, 'cuda')
    d10, d20 = d10.contiguous(), d20.contiguous()
    m = s2model(((4, None, None), (6, None, None)), num_layers=6, feature_size=128, seed=0)
    runs = []
    for _ in range(3):                                   # the first run warms up
        res = evaluate.wald_device(m, d10, d20)
        runs.append({k: round(v, 2) for k, v in res['times_ms'].items()})
    t = runs[-1]
    return {'tile': '10980^2 x 4 + 5490^2 x 6 float32 (bench.synth_tile), degraded to 5490^2 / 2745^2',
            'model': 'DSen2 6 x 128, seeded random weights', 'runs_ms': runs[1:],
            'metrics_share_of_sr': round(t['metrics'] / t['sr'], 4),
            'dsen2_uiq': res['dsen2']['uiq'], 'bicubic_uiq': res['bicubic']['uiq']}


def oracle_crop():
    rng = np.random.RandomState(0)
    ref = rng.randint(500, 8000, (1000, 1000, 6)).astype(np.uint16)
    est = (ref + rng.randn(1000, 1000, 6) * 100).astype(np.float32)
    t0 = time.perf_counter()
    mo.sums(est, ref)
    return {'size': '1000^2 x 6', 'host_cores': os.cpu_count(), 's': round(time.perf_counter() - t0, 2)}


def main():
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'metrics_b200.json'))
    path = ap.parse_args().out
    out = {'card': card()}
    peak = copy_peak()
    out['copy_rate_GB_per_s'] = round(peak, 1)
    out['kernel'] = [kernel_case(n, dt, nd, peak) for n, dt in ((5490, torch.float32), (5490, torch.float64),
                                                                (10980, torch.float32))
                     for nd in (None, 0)]
    out['wald_full_tile'] = wald_stages()
    out['oracle_host'] = oracle_crop()
    out['card_after'] = card()
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, 'w') as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == '__main__':
    main()
