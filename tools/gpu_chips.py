"""Chip stacks against one call per chip, and against the full tile (one GPU).

DSen2 20 m (6 x 128, he_uniform seed 0), uint16 images (random integer DN, seeded), float32 and uint16 output, for
120 x 120 x 4096 chips (BigEarthNet), 256 x 256 x 1024 (SEN12MS) and 600 x 600 x 64 (the reference's demo size):
  (a) a loop of single-image ``DSen2_20`` calls over the first ``--loop-chips`` chips, reported per chip;
  (b) ``DSen2_20(stack)`` numpy -> numpy (a fresh output array, as a caller gets it);
  (c) ``super_resolve_device`` on the device-resident stack (preallocated output);
  (d) input preparation and last layer per patch (CUDA events of the 'prep' / 'conv_tail' launches of separate calls of
      (c)), against the full 10980 x 10980 tile of ``bench.synth_tile`` through the 3-D path in the same run.
Host clock around calls that end in a synchronise; one warm-up call of every mode first, then the modes alternate; mean
and spread of ``--reps`` (at least 3).  (b) is checked bit for bit against (a) on the chips (a) covered.  The card's name,
power limit and max SM clock are read in the same run.  Writes one JSON (default profiles/chips_b200.json).

    python tools/gpu_chips.py [--out profiles/chips_b200.json] [--reps 3] [--loop-chips 256]
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(ROOT))
sys.path.insert(0, ROOT)
from bench import synth_tile  # noqa: E402
from dsen2_b200 import supres  # noqa: E402
from dsen2_b200.DSen2Net import s2model  # noqa: E402
from dsen2_b200.patches import patch_counts  # noqa: E402
from gpu_u16_output import alternate, card, mean  # noqa: E402

GEOMETRIES = [(120, 4096), (256, 1024), (600, 64)]
TILE = 10980
OUT = {'float32': (np.float32, None), 'uint16': (np.uint16, torch.uint16)}


def spread(xs):
    return [min(xs), max(xs)]


def per_patch_us(model, call, reps, patches):
    """'prep' / 'conv_tail': microseconds per patch from the CUDA events of the launches, mean of ``reps`` calls."""
    res = {'prep': [], 'conv_tail': []}
    for _ in range(reps):
        timers = {}
        call(timers)
        torch.cuda.synchronize()
        for k in res:
            res[k].append(sum(e0.elapsed_time(e1) for e0, e1, _ in timers[k]) * 1e3 / patches)
    return {k: round(sum(v) / len(v), 3) for k, v in res.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(os.path.dirname(ROOT), 'profiles', 'chips_b200.json'))
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--loop-chips', type=int, default=256)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.cuda.set_device(0)
    reps = max(3, args.reps)
    res = {'card': card(),
           'model': 'DSen2 20 m (6 x 128, he_uniform seed 0)',
           'images': 'uint16, random integer DN in [1, 12000), seeded',
           'timing': 'host clock around each call, ending in a device synchronise; one warm-up call of every mode, then '
                     'the modes alternate; mean and [min, max] of %d; prep / conv_tail: CUDA events of separate calls' % reps}
    m = s2model(((4, None, None), (6, None, None)), num_layers=6, feature_size=128, seed=0)

    # ---- the full tile through the 3-D path, device-resident
    f10, f20 = synth_tile(torch, TILE, TILE, 'cuda')
    t10, t20 = f10.to(torch.uint16), f20.to(torch.uint16)
    del f10, f20
    tile_patches = patch_counts(TILE // 2, TILE // 2, 64, 4)[1]
    tile = {}
    for name, (_np_dt, t_dt) in OUT.items():
        out = torch.empty((TILE, TILE, 6), dtype=t_dt or torch.float32, device='cuda')
        ms = alternate({'tile': lambda: supres.super_resolve_device(m, t10, t20, out=out, out_dtype=t_dt)}, reps)['tile']
        tile[name] = {'ms': ms, 'ms_mean': mean(ms), 'patches': tile_patches,
                      'patches_per_s': round(tile_patches / (mean(ms) / 1e3)),
                      'out_mpix_per_s': round(TILE * TILE / (mean(ms) / 1e3) / 1e6, 1),
                      'per_patch_us': per_patch_us(m, lambda tm: supres.super_resolve_device(
                          m, t10, t20, out=out, out_dtype=t_dt, timers=tm), reps, tile_patches)}
        del out
    res['full_tile'] = tile
    del t10, t20
    torch.cuda.empty_cache()

    rows = []
    for H, N in GEOMETRIES:
        g = torch.Generator(device='cuda').manual_seed(1000 + H)
        d10 = torch.randint(1, 12000, (N, H, H, 4), generator=g, device='cuda', dtype=torch.int32).to(torch.uint16)
        d20 = torch.randint(1, 12000, (N, H // 2, H // 2, 6), generator=g, device='cuda', dtype=torch.int32).to(torch.uint16)
        h10, h20 = d10.cpu().numpy(), d20.cpu().numpy()
        ppc = patch_counts(H // 2, H // 2, 64, 4)[1]
        k = min(N, args.loop_chips)
        for name, (np_dt, t_dt) in OUT.items():
            dout = torch.empty((N, H, H, 6), dtype=t_dt or torch.float32, device='cuda')
            loop_out = np.empty((k, H, H, 6), np_dt)

            def loop():
                for i in range(k):
                    supres.DSen2_20(h10[i], h20[i], model=m, out=loop_out[i], out_dtype=np_dt)
            stack_out = {}

            def stack():
                stack_out['v'] = supres.DSen2_20(h10, h20, model=m, out_dtype=np_dt)

            def device():
                supres.super_resolve_device(m, d10, d20, out=dout, out_dtype=t_dt)
            ms = alternate({'a_loop': loop, 'b_stack_numpy': stack, 'c_stack_device': device}, reps)
            a = mean(ms['a_loop']) / k
            b, c = mean(ms['b_stack_numpy']), mean(ms['c_stack_device'])
            row = {'chip': '%d x %d' % (H, H), 'chips': N, 'patches_per_chip': ppc, 'patches': N * ppc, 'out_dtype': name,
                   'ms': ms, 'ms_spread': {kk: spread(v) for kk, v in ms.items()},
                   'a_loop_ms_per_chip': round(a, 3), 'a_loop_chips': k,
                   'b_stack_numpy_ms': b, 'c_stack_device_ms': c,
                   'b_ms_per_chip': round(b / N, 4), 'c_ms_per_chip': round(c / N, 4),
                   'speedup_b_over_a': round(a * N / b, 2),
                   'b_over_c': round(b / c, 3),
                   'c_patches_per_s': round(N * ppc / (c / 1e3)),
                   'c_patches_per_s_vs_full_tile': round(N * ppc / (c / 1e3) / tile[name]['patches_per_s'], 3),
                   'b_patches_per_s': round(N * ppc / (b / 1e3)),
                   'c_out_mpix_per_s': round(N * H * H / (c / 1e3) / 1e6, 1),
                   'b_out_mpix_per_s': round(N * H * H / (b / 1e3) / 1e6, 1),
                   'per_patch_us': per_patch_us(m, lambda tm: supres.super_resolve_device(
                       m, d10, d20, out=dout, out_dtype=t_dt, timers=tm), reps, N * ppc),
                   'b_equals_a_bitwise': bool(np.array_equal(stack_out['v'][:k].view(np.uint8),
                                                             loop_out.view(np.uint8))),
                   'c_equals_b_bitwise': bool(np.array_equal(dout.cpu().numpy().view(np.uint8),
                                                             stack_out['v'].view(np.uint8)))}
            print(json.dumps({kk: v for kk, v in row.items() if kk not in ('ms', 'per_patch_us')}), flush=True)
            rows.append(row)
            del dout, stack_out
        del d10, d20, h10, h20
        torch.cuda.empty_cache()
    res['rows'] = rows
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res['card']), json.dumps({k: (v['ms_mean'], v['patches_per_s']) for k, v in tile.items()}))


if __name__ == '__main__':
    main()
