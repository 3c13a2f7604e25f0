"""What the radiometric offset (``add_offset=-1000``) costs against no offset, and what it saves against the host workaround
(one GPU).

Full 10980 x 10980 uint16 tile P = ``bench.synth_tile`` + 1000 (a product in the convention of processing baseline 04.00;
values below 13 001), DSen2 20 m, he_uniform weights (seed 0):
  * device-resident ``super_resolve_device`` on P without and with ``add_offset=-1000``, float32 and uint16 output (host
    clock around calls ending in a synchronise), and the input preparation / last layer alone (CUDA events of the 'prep' /
    'conv_tail' launches of separate calls);
  * the facade numpy -> numpy, uint16 in and out: ``add_offset=-1000`` against what a caller does without it
    (``astype(float32) - 1000`` on the host, the float32 facade, then ``+ 1000`` and the numpy quantisation), and the uint16
    facade without an offset;
  * full size: out(P, -1000) == out(S) + 1000 bit for bit (S = P - 1000, the same scene in the old convention), and the
    quantisation of that for uint16 output.
Modes alternate, after one warm-up call of each.  Writes one JSON (default profiles/add_offset_b200.json).

    python tools/gpu_add_offset.py [--out profiles/add_offset_b200.json] [--reps 3]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(ROOT))
sys.path.insert(0, ROOT)
from bench import synth_tile  # noqa: E402
from dsen2_b200 import supres  # noqa: E402
from dsen2_b200.DSen2Net import s2model  # noqa: E402
from gpu_u16_output import alternate, as_int, card, expected_dev, mean, user_quantise  # noqa: E402

N = 10980
A = -1000.0
U16, F32 = torch.uint16, torch.float32


def kernel_ms(model, d10, d20, out, reps, **kw):
    """Per kind ('prep', 'conv_tail'): ms per tile from the CUDA events of the launches, one list entry per call."""
    res = {'prep': [], 'conv_tail': []}
    for _ in range(reps):
        timers = {}
        supres.super_resolve_device(model, d10, d20, out=out, timers=timers, **kw)
        torch.cuda.synchronize()
        for k in res:
            res[k].append(round(sum(e0.elapsed_time(e1) for e0, e1, _ in timers[k]), 3))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(os.path.dirname(ROOT), 'profiles', 'add_offset_b200.json'))
    ap.add_argument('--reps', type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.cuda.set_device(0)
    reps = max(3, args.reps)
    res = {'card': card(),
           'tile': '%d x %d uint16, bench.synth_tile + 1000, DSen2 20 m (6 x 128, he_uniform seed 0)' % (N, N),
           'timing': 'host clock around each call, ending in a device synchronise; modes alternate, after one warm-up '
                     'call of each; prep / conv_tail: CUDA events around those launches of separate calls'}
    f10, f20 = synth_tile(torch, N, N, 'cuda')
    s10, s20 = f10.to(U16), f20.to(U16)
    p10, p20 = (f10 + 1000).to(U16), (f20 + 1000).to(U16)      # float, then uint16: no elementwise uint16 kernel needed
    res['input_max'] = int(max(float(f10.max()), float(f20.max()))) + 1000
    del f10, f20
    m = s2model(((4, None, None), (6, None, None)), num_layers=6, feature_size=128, seed=0)

    # ---- device-resident, the same product P without and with the offset
    shape = (N, N, 6)
    outs = {k: torch.empty(shape, dtype=F32 if k.startswith('float32') else U16, device='cuda')
            for k in ('float32', 'float32_offset', 'uint16', 'uint16_offset')}
    kw = {'float32': {}, 'float32_offset': {'add_offset': A}, 'uint16': {'out_dtype': U16},
          'uint16_offset': {'out_dtype': U16, 'add_offset': A}}
    ms = alternate({k: (lambda k=k: supres.super_resolve_device(m, p10, p20, out=outs[k], **kw[k])) for k in outs}, reps)
    kern = {k: kernel_ms(m, p10, p20, outs[k], reps, **kw[k]) for k in outs}
    mm = {k: mean(v) for k, v in ms.items()}
    rec = {'device_ms': ms, 'device_ms_mean': mm,
           'offset_over_none': {'float32': round(mm['float32_offset'] / mm['float32'], 4),
                                'uint16': round(mm['uint16_offset'] / mm['uint16'], 4)},
           'kernel_ms': kern,
           'kernel_ms_mean': {k: {kk: mean(vv) for kk, vv in v.items()} for k, v in kern.items()}}
    # full size: out(P, -1000) == out(S) + 1000, and its quantisation
    ref = supres.super_resolve_device(m, s10, s20) + 1000.0
    rec['float32_equals_old_product_plus_1000'] = bool(torch.equal(outs['float32_offset'].view(torch.int32),
                                                                   ref.view(torch.int32)))
    rec['uint16_equals_quantised_old_product_plus_1000'] = bool(torch.equal(as_int(outs['uint16_offset']),
                                                                            expected_dev(ref)))
    rec['values'] = int(ref.numel())
    rec['negative_after_offset'] = int((ref.round() < 0).sum())
    rec['uint16_zeros_with_offset'] = int((as_int(outs['uint16_offset']) == 0).sum())
    res['device_20m'] = rec
    print(json.dumps(rec), flush=True)
    del outs, ref
    torch.cuda.empty_cache()

    # ---- the facade, numpy -> numpy, uint16 in and out
    a10, a20 = p10.cpu().numpy(), p20.cpu().numpy()
    del s10, s20, p10, p20
    torch.cuda.empty_cache()
    o_off, o_none, o_f = np.empty(shape, np.uint16), np.empty(shape, np.uint16), np.empty(shape, np.float32)
    got = {}

    def host_workaround():
        off = np.float32(-A)
        f = supres.DSen2_20(a10.astype(np.float32) - off, a20.astype(np.float32) - off, model=m, out=o_f)
        got['w'] = user_quantise(f + off)
    fac = {'uint16_add_offset': lambda: supres.DSen2_20(a10, a20, model=m, out=o_off, out_dtype=np.uint16, add_offset=A),
           'host_workaround': host_workaround,
           'uint16_no_offset': lambda: supres.DSen2_20(a10, a20, model=m, out=o_none, out_dtype=np.uint16)}
    ms = alternate(fac, reps)
    t0 = time.perf_counter()
    g10, g20 = a10.astype(np.float32) - np.float32(-A), a20.astype(np.float32) - np.float32(-A)
    t1 = time.perf_counter()
    user_quantise(o_f + np.float32(-A))
    t2 = time.perf_counter()
    del g10, g20
    res['facade'] = {'ms': ms, 'ms_mean': {k: mean(v) for k, v in ms.items()},
                     'host_input_pass_ms': round((t1 - t0) * 1e3, 1), 'host_output_pass_ms': round((t2 - t1) * 1e3, 1),
                     'workaround': 'a.astype(np.float32) - 1000 per input, the float32 facade, then '
                                   'np.clip(np.rint(f + 1000), 0, 65535).astype(np.uint16)',
                     'add_offset_equals_workaround': bool(np.array_equal(o_off, got['w']))}
    print(json.dumps(res['facade']), flush=True)
    res['card_after'] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as fh:
        json.dump(res, fh, indent=1)
    print('wrote', args.out)


if __name__ == '__main__':
    main()
