"""Scene lists against one call per scene, and against the full tile (one GPU).

DSen2 (6 x 128, he_uniform seed 0), uint16 images (random integer DN, seeded), float32 output, three workloads:
  grid   : the 10980 x 10980 tile cut into 256 x 256 chips with its 228-px remainder row and column (43 x 43 = 1849
           scenes of four sizes), the chips being numpy views of the one product;
  random : 2000 scenes of seeded random even sizes in [112, 600] (each axis);
  60m    : 500 scenes (60 m path) of seeded random sizes, multiples of 6 in [168, 600].
Per workload:
  (a) a loop of 3-D ``DSen2_20`` / ``DSen2_60`` calls, one per scene;
  (b) ``DSen2_20_scenes`` / ``DSen2_60_scenes`` numpy -> numpy;
  (c) ``super_resolve_scenes_device`` on the device-resident list (preallocated outputs);
  patches/s of (c) against the full tile's (3-D path, same run), and prep / last-layer microseconds per patch (CUDA
  events of the 'prep' / 'conv_tail' launches of separate calls of (c)).
Host clock around calls that end in a synchronise; one warm-up call of every mode first, then the modes alternate; mean
and [min, max] of ``--reps`` (at least 3).  (b) is checked bit for bit against (a) and (c).  The card's name, power limit
and max SM clock are read in the same run.  Writes one JSON (default profiles/scenes_b200.json).

    python tools/gpu_scenes.py [--out profiles/scenes_b200.json] [--reps 3]
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
from gpu_chips import per_patch_us, spread  # noqa: E402
from gpu_u16_output import alternate, card, mean  # noqa: E402

TILE = 10980


def grid_windows(size, chip):
    starts = list(range(0, size, chip))
    return [(y, x, min(chip, size - y), min(chip, size - x)) for y in starts for x in starts]


def random_sizes(rng, n, lo, hi, step):
    return [(int(rng.randint(lo // step, hi // step + 1)) * step, int(rng.randint(lo // step, hi // step + 1)) * step)
            for _ in range(n)]


def lists_of(rng, sizes, run_60):
    divs = (1, 2, 6) if run_60 else (1, 2)
    return [[rng.randint(1, 12000, size=(H // d, W // d, c)).astype(np.uint16) for H, W in sizes]
            for d, c in zip(divs, (4, 6, 2))]


def workload(name, model, lists, sizes, run_60, reps, tile_pps):
    r, P, B = (6, 192, 12) if run_60 else (2, 128, 8)
    patches = sum(patch_counts(H // r, W // r, P // r, B // r)[1] for H, W in sizes)
    single = supres.DSen2_60 if run_60 else supres.DSen2_20
    many = supres.DSen2_60_scenes if run_60 else supres.DSen2_20_scenes
    dev = [[torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in l] for l in lists]
    douts = [torch.empty((H, W, model.out_channels), device='cuda') for H, W in sizes]
    loop_out = [np.empty((H, W, model.out_channels), np.float32) for H, W in sizes]
    got = {}

    def loop():
        for i in range(len(sizes)):
            single(*[l[i] for l in lists], model=model, out=loop_out[i])

    def scenes():
        got['b'] = many(*lists, model=model)

    def device():
        supres.super_resolve_scenes_device(model, *dev, outs=douts)
    ms = alternate({'a_loop': loop, 'b_scenes_numpy': scenes, 'c_scenes_device': device}, reps)
    a, b, c = mean(ms['a_loop']), mean(ms['b_scenes_numpy']), mean(ms['c_scenes_device'])
    same = lambda x, y: np.array_equal(x.view(np.uint8), y.view(np.uint8))
    row = {'workload': name, 'scenes': len(sizes), 'distinct_sizes': len(set(sizes)), 'patches': patches,
           'out_mpix': round(sum(H * W for H, W in sizes) / 1e6, 1),
           'ms': ms, 'ms_spread': {k: spread(v) for k, v in ms.items()},
           'a_loop_ms': a, 'b_scenes_numpy_ms': b, 'c_scenes_device_ms': c,
           'speedup_b_over_a': round(a / b, 2), 'b_over_c': round(b / c, 3),
           'c_patches_per_s': round(patches / (c / 1e3)),
           'c_patches_per_s_vs_full_tile': round(patches / (c / 1e3) / tile_pps, 3),
           'per_patch_us': per_patch_us(model, lambda tm: supres.super_resolve_scenes_device(model, *dev, outs=douts,
                                                                                             timers=tm), reps, patches),
           'b_equals_a_bitwise': all(same(x, y) for x, y in zip(got['b'], loop_out)),
           'c_equals_b_bitwise': all(same(d.cpu().numpy(), y) for d, y in zip(douts, got['b']))}
    print(json.dumps({k: v for k, v in row.items() if k not in ('ms', 'per_patch_us')}), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(os.path.dirname(ROOT), 'profiles', 'scenes_b200.json'))
    ap.add_argument('--reps', type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.cuda.set_device(0)
    reps = max(3, args.reps)
    res = {'card': card(),
           'model': 'DSen2 (6 x 128, he_uniform seed 0), 20 m and 60 m',
           'images': 'uint16, random integer DN in [1, 12000), seeded (grid: bench.synth_tile); float32 output',
           'timing': 'host clock around each call, ending in a device synchronise; one warm-up call of every mode, then '
                     'the modes alternate; mean and [min, max] of %d; prep / conv_tail: CUDA events of separate calls' % reps}
    m20 = s2model(((4, None, None), (6, None, None)), num_layers=6, feature_size=128, seed=0)
    m60 = s2model(((4, None, None), (6, None, None), (2, None, None)), num_layers=6, feature_size=128, seed=0)

    f10, f20 = synth_tile(torch, TILE, TILE, 'cuda')
    t10, t20 = f10.to(torch.uint16), f20.to(torch.uint16)
    del f10, f20
    tile_patches = patch_counts(TILE // 2, TILE // 2, 64, 4)[1]
    out = torch.empty((TILE, TILE, 6), device='cuda')
    ms = alternate({'tile': lambda: supres.super_resolve_device(m20, t10, t20, out=out)}, reps)['tile']
    tile = {'ms': ms, 'ms_mean': mean(ms), 'patches': tile_patches, 'patches_per_s': round(tile_patches / (mean(ms) / 1e3)),
            'per_patch_us': per_patch_us(m20, lambda tm: supres.super_resolve_device(m20, t10, t20, out=out, timers=tm),
                                         reps, tile_patches)}
    res['full_tile'] = tile
    h10, h20 = t10.cpu().numpy(), t20.cpu().numpy()
    del t10, t20, out
    torch.cuda.empty_cache()

    rows = []
    wins = grid_windows(TILE, 256)
    lists = [[h10[y:y + h, x:x + w] for y, x, h, w in wins], [h20[y // 2:(y + h) // 2, x // 2:(x + w) // 2]
                                                              for y, x, h, w in wins]]
    rows.append(workload('grid 10980 / 256', m20, lists, [(h, w) for _, _, h, w in wins], False, reps,
                         tile['patches_per_s']))
    del lists, h10, h20
    rng = np.random.RandomState(7)
    sizes = random_sizes(rng, 2000, 112, 600, 2)
    rows.append(workload('random 2000 in [112, 600]', m20, lists_of(rng, sizes, False), sizes, False, reps,
                         tile['patches_per_s']))
    sizes = random_sizes(rng, 500, 168, 600, 6)
    rows.append(workload('60m 500 in [168, 600]', m60, lists_of(rng, sizes, True), sizes, True, reps,
                         tile['patches_per_s']))
    res['rows'] = rows
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res['card']), json.dumps({'tile_ms': tile['ms_mean'], 'tile_pps': tile['patches_per_s']}))


if __name__ == '__main__':
    main()
