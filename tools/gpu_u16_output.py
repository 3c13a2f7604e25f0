"""What uint16 digital-number output (``out_dtype=uint16``) costs and saves against float32 output (one GPU).

Full 10980 x 10980 uint16 tile of ``bench.synth_tile``, DSen2 20 m, he_uniform weights (seed 0):
  * device-resident ``super_resolve_device`` float32 vs uint16 output (host clock around calls ending in a synchronise),
    and the last layer alone (CUDA events of the 'conv_tail' launches);
  * ``HostPipeline.run`` pinned -> pinned: ms and device -> host bytes;
  * the facade numpy -> numpy: float32 out, float32 out + the host quantisation a user runs today, uint16 out;
  * nodata=0 at 50 % coverage (``gpu_nodata.valid_mask60``), float32 vs uint16 output;
  * a full-size check that the uint16 output is the numpy quantisation of the float output, and how many values clamped.
Then DSen2 60 m and VDSen2 20 m device-resident on a 3360 x 3360 tile.  Modes alternate, after one warm-up call of each.
Writes one JSON (default profiles/u16_output_b200.json).

    python tools/gpu_u16_output.py [--out profiles/u16_output_b200.json] [--reps 3]
"""
import argparse
import json
import os
import subprocess
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
from gpu_nodata import up, valid_mask60  # noqa: E402

N = 10980
U16, F32 = torch.uint16, torch.float32


def card():
    p = torch.cuda.get_device_properties(0)
    uuid = str(p.uuid)
    uuid = uuid if uuid.startswith('GPU-') else 'GPU-' + uuid
    q = subprocess.run(['nvidia-smi', '-i', uuid, '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip()
    return {'torch_name': p.name, 'nvidia_smi': q}


def timed(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3


def alternate(fns, reps):
    """{mode: fn} -> {mode: [ms]}: one warm-up call of each mode, then ``reps`` rounds with the modes alternating."""
    for fn in fns.values():
        fn()
    res = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            res[k].append(round(timed(fn), 2))
    return res


def mean(xs):
    return round(sum(xs) / len(xs), 2)


def quantise_np(f):
    """The numpy reference of the uint16 output."""
    return np.clip(np.rint(np.nan_to_num(f, nan=0)), 0, 65535).astype(np.uint16)


def user_quantise(f):
    """What a caller of the float32 facade runs to get digital numbers."""
    return np.clip(np.rint(f), 0, 65535).astype(np.uint16)


def as_int(u):
    """uint16 CUDA tensor -> int32 values (through an int16 view: elementwise uint16 kernels are not needed)."""
    return u.view(torch.int16).to(torch.int32) & 0xFFFF


def expected_dev(f, nodata_mask=None, v=None):
    """q(f) on the device (torch.round rounds half to even), with the nodata rule when ``nodata_mask`` is given."""
    q = torch.nan_to_num(f, nan=0.0).round_().clamp_(0, 65535).to(torch.int32)
    if nodata_mask is not None:
        m = nodata_mask[..., None].expand_as(q)
        q[(q == v) & ~m] = 65534 if v == 65535 else v + 1
        q[m] = v
    return q


def device_section(model, d10, d20, d60, reps, label):
    H, W = int(d10.shape[0]), int(d10.shape[1])
    outs = {F32: torch.empty((H, W, model.out_channels), dtype=F32, device='cuda'),
            U16: torch.empty((H, W, model.out_channels), dtype=U16, device='cuda')}
    run = {'float32': lambda: supres.super_resolve_device(model, d10, d20, d60, out=outs[F32]),
           'uint16': lambda: supres.super_resolve_device(model, d10, d20, d60, out=outs[U16], out_dtype=U16)}
    ms = alternate(run, reps)
    tail = {'float32': [], 'uint16': []}
    for _ in range(reps):                       # the last layer alone: CUDA events around its launches, separate calls
        for k, dt in (('float32', F32), ('uint16', U16)):
            timers = {}
            supres.super_resolve_device(model, d10, d20, d60, out=outs[dt], out_dtype=dt if dt == U16 else None,
                                        timers=timers)
            torch.cuda.synchronize()
            tail[k].append(round(sum(e0.elapsed_time(e1) for e0, e1, _ in timers['conv_tail']), 3))
    same = bool(torch.equal(as_int(outs[U16]), expected_dev(outs[F32])))
    rec = {'what': label, 'device_ms': ms, 'device_ms_mean': {k: mean(v) for k, v in ms.items()},
           'uint16_over_float32': round(mean(ms['uint16']) / mean(ms['float32']), 4),
           'conv_tail_ms': tail, 'conv_tail_ms_mean': {k: mean(v) for k, v in tail.items()},
           'uint16_equals_quantised_float': same}
    print(json.dumps(rec), flush=True)
    return rec, outs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(os.path.dirname(ROOT), 'profiles', 'u16_output_b200.json'))
    ap.add_argument('--reps', type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.cuda.set_device(0)
    reps = max(3, args.reps)
    res = {'card': card(), 'tile': '%d x %d uint16, bench.synth_tile, DSen2 20 m (6 x 128, he_uniform seed 0)' % (N, N),
           'timing': 'host clock around each call, ending in a device synchronise; modes alternate, after one warm-up '
                     'call of each; conv_tail: CUDA events around the last-layer launches of separate calls'}
    f10, f20 = synth_tile(torch, N, N, 'cuda')
    d10, d20 = f10.to(U16), f20.to(U16)
    m = s2model(((4, None, None), (6, None, None)), num_layers=6, feature_size=128, seed=0)

    # ---- device-resident + the full-size check
    rec, outs = device_section(m, d10, d20, None, reps, 'DSen2 20 m, %d^2, device-resident' % N)
    f = outs[F32]
    rf = torch.nan_to_num(f, nan=0.0).round()
    rec['values'] = int(f.numel())
    rec['clamped_at_0'] = int((rf < 0).sum())
    rec['clamped_at_65535'] = int((rf > 65535).sum())
    rec['nan'] = int(torch.isnan(f).sum())
    del rf
    host_f = f.cpu().numpy()
    host_u = outs[U16].cpu().numpy()
    rec['numpy_check_full_size'] = bool(np.array_equal(quantise_np(host_f), host_u))
    res['device_20m'] = rec
    del outs, f, host_u
    print('full-size numpy check:', rec['numpy_check_full_size'], flush=True)

    # ---- HostPipeline.run, pinned -> pinned
    h10, h20 = d10.cpu().pin_memory(), d20.cpu().pin_memory()
    pipes = {k: supres.HostPipeline(m, N, N, dtype=U16, out_dtype=dt) for k, dt in (('float32', F32), ('uint16', U16))}
    houts = {k: torch.empty((N, N, 6), dtype=dt).pin_memory() for k, dt in (('float32', F32), ('uint16', U16))}
    ms = alternate({k: (lambda k=k: pipes[k].run(h10, h20, hout=houts[k])) for k in pipes}, reps)
    res['host_pipeline_pinned'] = {'ms': ms, 'ms_mean': {k: mean(v) for k, v in ms.items()},
                                   'd2h_bytes': {k: int(p.d2h_bytes) for k, p in pipes.items()},
                                   'h2d_bytes': {k: int(p.h2d_bytes) for k, p in pipes.items()},
                                   'uint16_equals_quantised_float': bool(np.array_equal(quantise_np(houts['float32'].numpy()),
                                                                                        houts['uint16'].numpy()))}
    print(json.dumps(res['host_pipeline_pinned']), flush=True)
    del pipes, houts, h10, h20
    supres._pipe_cache.clear()
    torch.cuda.empty_cache()

    # ---- the facade, numpy -> numpy
    a10, a20 = d10.cpu().numpy(), d20.cpu().numpy()
    o_f = np.empty((N, N, 6), np.float32)
    o_u = np.empty((N, N, 6), np.uint16)
    got = {}

    def f32_then_quantise():
        got['q'] = user_quantise(supres.DSen2_20(a10, a20, model=m, out=o_f))
    fac = {'float32': lambda: supres.DSen2_20(a10, a20, model=m, out=o_f),
           'float32_then_numpy_quantise': f32_then_quantise,
           'uint16': lambda: supres.DSen2_20(a10, a20, model=m, out=o_u, out_dtype=np.uint16)}
    ms = alternate(fac, reps)
    t0 = time.perf_counter()
    user_quantise(o_f)
    q_ms = (time.perf_counter() - t0) * 1e3
    res['facade'] = {'ms': ms, 'ms_mean': {k: mean(v) for k, v in ms.items()},
                     'numpy_quantise_alone_ms': round(q_ms, 1),
                     'quantise': 'np.clip(np.rint(x), 0, 65535).astype(np.uint16) on the float32 facade output',
                     'uint16_equals_numpy_quantised_float': bool(np.array_equal(quantise_np(o_f), o_u)),
                     'uint16_equals_user_quantised_float': bool(np.array_equal(got['q'], o_u))}
    print(json.dumps(res['facade']), flush=True)
    del o_f, o_u, got, host_f
    supres._pipe_cache.clear()
    torch.cuda.empty_cache()

    # ---- nodata = 0 at 50 % coverage, device-resident
    m60 = valid_mask60('0.5')
    g10, g20 = f10 * up(m60, 6)[..., None], f20 * up(m60, 3)[..., None]
    nod = (g10 == 0).all(-1) & up((g20 == 0).all(-1), 2)
    n10, n20 = g10.to(U16), g20.to(U16)
    del g10, g20
    outs = {F32: torch.empty((N, N, 6), dtype=F32, device='cuda'), U16: torch.empty((N, N, 6), dtype=U16, device='cuda')}
    ms = alternate({'float32': lambda: supres.super_resolve_device(m, n10, n20, out=outs[F32], nodata=0),
                    'uint16': lambda: supres.super_resolve_device(m, n10, n20, out=outs[U16], nodata=0, out_dtype=U16)},
                   reps)
    exp = expected_dev(outs[F32], nod, 0)
    res['nodata_50pct'] = {'nodata_pixel_fraction': round(float(nod.float().mean()), 4), 'device_ms': ms,
                           'device_ms_mean': {k: mean(v) for k, v in ms.items()},
                           'uint16_equals_contract': bool(torch.equal(as_int(outs[U16]), exp)),
                           'valid_values_moved_off_0': int(((torch.nan_to_num(outs[F32], nan=0.0).round() <= 0)
                                                            & ~nod[..., None]).sum())}
    print(json.dumps(res['nodata_50pct']), flush=True)
    del outs, exp, nod, n10, n20, f10, f20, d10, d20
    torch.cuda.empty_cache()

    # ---- 3360^2: DSen2 60 m and VDSen2 20 m
    T = 3360
    s10, s20, s60 = [t.to(U16) for t in synth_tile(torch, T, T, 'cuda', with_60=True)]
    m6 = s2model(((4, None, None), (6, None, None), (2, None, None)), num_layers=6, feature_size=128, seed=0)
    res['device_60m_3360'] = device_section(m6, s10, s20, s60, reps, 'DSen2 60 m, %d^2, device-resident' % T)[0]
    mv = s2model(((4, None, None), (6, None, None)), num_layers=32, feature_size=256, seed=0)
    res['device_vdsen2_3360'] = device_section(mv, s10, s20, None, reps, 'VDSen2 20 m, %d^2, device-resident' % T)[0]
    res['card_after'] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as fh:
        json.dump(res, fh, indent=1)
    print('wrote', args.out)


if __name__ == '__main__':
    main()
