"""What ``nodata`` costs and saves on a full 10980 x 10980 uint16 tile (one GPU).

The synthetic tile of ``bench.synth_tile`` is set to 0 in every band outside a straight, slightly slanted swath edge
(cut on the 60 m grid, so all resolutions agree) at coverages 100 / 75 / 50 / 25 / 0 %, and at 100 % with square holes
cut through patch interiors.  Per coverage: the active-patch fraction, device-resident and facade (numpy uint16 in ->
numpy out) ms per tile with ``nodata=None`` and ``nodata=0`` (alternating, after warm-up), the nodata kernels' own time
(CUDA events), and a full-size check that valid pixels are bit-identical between the two modes and nodata pixels are 0.
DSen2 at every coverage, VDSen2 device-resident at 50 %.  Writes one JSON (default profiles/nodata_b200.json).

    python tools/gpu_nodata.py [--out profiles/nodata_b200.json] [--reps 3]
"""
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
from bench import synth_tile  # noqa: E402
from dsen2_b200 import supres  # noqa: E402
from dsen2_b200.DSen2Net import s2model  # noqa: E402

N = 10980


def card():
    p = torch.cuda.get_device_properties(0)
    uuid = str(p.uuid)
    uuid = uuid if uuid.startswith('GPU-') else 'GPU-' + uuid
    q = subprocess.run(['nvidia-smi', '-i', uuid, '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip()
    return {'torch_name': p.name, 'nvidia_smi': q}


def valid_mask60(kind):
    """bool (N/6, N/6) on the 60 m grid: True where the ground was imaged."""
    n = N // 6
    y, x = torch.meshgrid(torch.arange(n, device='cuda', dtype=torch.float32) + 0.5,
                          torch.arange(n, device='cuda', dtype=torch.float32) + 0.5, indexing='ij')
    if kind == 'holes':                        # 48 x 48 px holes every 102 px: they cut through patch interiors
        return ~(((y.long() % 17) < 8) & ((x.long() % 17) < 8) & (y.long() // 17 % 2 == 0))
    c = float(kind)
    if c >= 1.0:
        return torch.ones((n, n), dtype=torch.bool, device='cuda')
    if c <= 0.0:
        return torch.zeros((n, n), dtype=torch.bool, device='cuda')
    return x < c * n + 0.1 * (y - n / 2)       # slanted swath edge; covered area = c of the tile


def up(m, k):
    return m.repeat_interleave(k, 0).repeat_interleave(k, 1)


def timed(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3


def measure(model, f10, f20, kind, reps, facade):
    m60 = valid_mask60(kind)
    g10, g20 = f10 * up(m60, 6)[..., None], f20 * up(m60, 3)[..., None]     # float32: torch has no uint16 masked fill
    nod = (g10 == 0).all(-1) & up((g20 == 0).all(-1), 2)
    d10, d20 = g10.to(torch.uint16), g20.to(torch.uint16)
    del g10, g20
    out_a = torch.empty((N, N, model.out_channels), dtype=torch.float32, device='cuda')
    out_b = torch.empty_like(out_a)
    filled = supres.patch_counts(N // 2, N // 2, 64, 4)[1]
    active = int(supres.active_patches(d10, d20, nodata=0).numel())
    run = {None: lambda: supres.super_resolve_device(model, d10, d20, out=out_a),
           0: lambda: supres.super_resolve_device(model, d10, d20, out=out_b, nodata=0)}
    for mode in (None, 0):                     # warm-up of both modes at this coverage
        run[mode]()
    dev = {'none': [], 'nodata0': []}
    for _ in range(reps):
        for mode, key in ((None, 'none'), (0, 'nodata0')):
            dev[key].append(round(timed(run[mode]), 2))
    # the nodata kernels' own time: CUDA events of one more call
    timers = {}
    supres.super_resolve_device(model, d10, d20, out=out_b, nodata=0, timers=timers)
    torch.cuda.synchronize()
    kern = {k: round(sum(e0.elapsed_time(e1) for e0, e1, _ in timers.get(k, [])), 4) for k in ('nodata_patches', 'nodata_fill')}
    valid_same = bool(torch.equal(out_a[~nod].view(torch.int32), out_b[~nod].view(torch.int32)))
    nodata_is_v = bool((out_b[nod] == 0).all())
    rec = {'coverage': kind, 'filled_patches': filled, 'active_patches': active, 'active_fraction': round(active / filled, 4),
           'nodata_pixel_fraction': round(float(nod.float().mean()), 4), 'device_ms': dev,
           'nodata_kernels_ms': kern, 'valid_pixels_bit_identical': valid_same, 'nodata_pixels_equal_v': nodata_is_v}
    del out_a, out_b
    if facade:
        h10, h20 = d10.cpu().numpy(), d20.cpu().numpy()
        hout = np.empty((N, N, model.out_channels), np.float32)
        fr = {None: lambda: supres.DSen2_20(h10, h20, model=model, out=hout),
              0: lambda: supres.DSen2_20(h10, h20, model=model, out=hout, nodata=0)}
        for mode in (None, 0):
            fr[mode]()
        fac = {'none': [], 'nodata0': []}
        for _ in range(reps):
            for mode, key in ((None, 'none'), (0, 'nodata0')):
                fac[key].append(round(timed(fr[mode]), 2))
        rec['facade_ms'] = fac
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'nodata_b200.json'))
    ap.add_argument('--reps', type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.cuda.set_device(0)
    res = {'card': card(), 'tile': '%d x %d uint16, bench.synth_tile, 20 m path' % (N, N),
           'timing': 'host clock around each call, ending in a device synchronise; modes alternate; after one warm-up '
                     'call of each mode per coverage',
           'dsen2': [], 'vdsen2': []}
    f10, f20 = synth_tile(torch, N, N, 'cuda')
    m = s2model(((4, None, None), (6, None, None)), num_layers=6, feature_size=128, seed=0)
    for kind in ('1.0', '0.75', '0.5', '0.25', '0.0', 'holes'):
        res['dsen2'].append(measure(m, f10, f20, kind, args.reps, facade=True))
    mv = s2model(((4, None, None), (6, None, None)), num_layers=32, feature_size=256, seed=0)
    res['vdsen2'].append(measure(mv, f10, f20, '0.5', 2, facade=False))
    res['card_after'] = card()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, 'w') as fh:
        json.dump(res, fh, indent=1)
    print('wrote', args.out)


if __name__ == '__main__':
    main()
