"""Quality of DSen2 and of the bicubic baseline under Wald's protocol, on the device.

    python -m dsen2_b200.evaluate PRODUCT [--run_60] [--deep] [--weights F | --random-weights] [--roi_x_y x1,y1,x2,y2]
                                  [--nodata V] [--add_offset A] [--json OUT]
    python -m dsen2_b200.evaluate --predictions DATA_PATH [--run_60] [--nodata V] [--json OUT]

Wald's protocol scores a super-resolution method where the truth is known: every band is degraded by the resolution ratio r
(2 for the 20 m bands, 6 for the 60 m bands), the method brings the degraded target bands back to their native resolution,
and the result is compared with the native bands.  ``wald_device`` runs what ``create_patches --test_data`` writes and
``demoDSen2`` scores, without leaving the GPU: ``down_pixel_aggr_device`` (``patches.downPixelAggr``'s arithmetic, then
float32), ``supres.super_resolve_device``, the bicubic baseline ``imresize_device(degraded target, r)`` and
``metrics.quality_device`` (RMSE, SRE, SAM, UIQ) of both against the native target bands.

Product mode reads a SAFE product or an ``.npz`` container through the ROI, UTM and band selection of ``create_patches``.
``--predictions`` scores every ``test/<scene>/`` (``test60/`` with ``--run_60``) holding the ``<nr>-predict.npy`` of
``supres_train --predict``, against ``no_tiling/data20_gt.npy`` (``data60_gt.npy``), with the bicubic baseline computed from
``no_tiling/data20.npy`` (``data60.npy``).  Both print per scene a table of the per-band and overall values of DSen2 and
bicubic; ``--json`` writes them with the stage times (SRE of a perfect estimate is +inf, written as ``Infinity``).
"""
import argparse
import glob
import json
import os
import sys

import numpy as np

from . import _capi, metrics, supres
from .create_patches import read_bands
from .imresize import imresize_device
from .patches import down_pixel_aggr_device  # noqa: F401  (part of this module's interface)

_STAGES = ('degrade', 'sr', 'bicubic', 'metrics')


def _name(dt):
    return str(dt)[len('torch.'):] if str(dt).startswith('torch.') else np.dtype(dt).name


def check_wald(model, shapes, dtypes, nodata=None, add_offset=None):
    """Rejects with ``ValueError`` what ``wald_device`` cannot run: inputs other than (H, W, 4), (H/2, W/2, 6)[, (H/6, W/6, 2)]
    float32 or uint16, a model with another number of inputs, 10 m sizes that are not multiples of 4 (20 m path) or 36
    (60 m path), degraded scenes smaller than one patch stride (10 m size < 224 or < 1008), and the ``nodata`` /
    ``add_offset`` the measures or the network refuse.  Returns (H, W, r)."""
    run_60 = len(shapes) == 3
    if len(shapes) != len(model.in_channels):
        raise ValueError("the model takes %d inputs, got %d images" % (len(model.in_channels), len(shapes)))
    r, mult, least = (6, 36, 1008) if run_60 else (2, 4, 224)
    if len(shapes[0]) != 3:
        raise ValueError("images must be HWC, got shape %s" % (tuple(shapes[0]),))
    H, W = int(shapes[0][0]), int(shapes[0][1])
    if H % mult or W % mult:
        raise ValueError("10 m size %dx%d must be a multiple of %d for the %d m path" % (H, W, mult, 60 if run_60 else 20))
    if min(H, W) < least:
        raise ValueError("10 m size %dx%d: the scene degraded by %d is smaller than one patch stride (%d px at 10 m)"
                         % (H, W, r, least))
    for sh, dt, div, c in zip(shapes, dtypes, (1, 2, 6), model.in_channels):
        if tuple(int(s) for s in sh) != (H // div, W // div, c):
            raise ValueError("expected an image of shape %s, got %s" % ((H // div, W // div, c), tuple(sh)))
        if _name(dt) not in ('float32', 'uint16'):
            raise ValueError("images must be float32 or uint16, got %s" % _name(dt))
    target = shapes[-1]
    metrics.check_args(target, 'float32', target, dtypes[-1], nodata)
    supres.check_add_offset(add_offset, model)
    return H, W, r


def wald_device(model, d10, d20, d60=None, nodata=None, add_offset=None):
    """Wald's protocol on native-resolution CUDA HWC bands (uint16 or float32; ``d60`` selects the 60 m path).
    Returns a dict: ``dsen2`` and ``bicubic``, the measures (``metrics``) of each against the native target bands (``d20``,
    or ``d60``), masked by ``nodata`` on those bands (the network runs without nodata); ``sr`` (float32) and ``baseline``
    (float64), the two estimates on the device; ``times_ms``, the device time of each stage.  ``add_offset`` goes to the
    network (``supres.super_resolve_device``)."""
    imgs = [d10, d20] + ([d60] if d60 is not None else [])
    _H, _W, r = check_wald(model, [tuple(t.shape) for t in imgs], [t.dtype for t in imgs], nodata, add_offset)
    torch = _capi.require_cuda()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(_STAGES) + 1)]
    ev[0].record()
    low = [down_pixel_aggr_device(t, r).to(torch.float32) for t in imgs]
    ev[1].record()
    sr = supres.super_resolve_device(model, *low, add_offset=add_offset)
    ev[2].record()
    h, w = int(low[-1].shape[0]), int(low[-1].shape[1])
    baseline = imresize_device(low[-1], [float(r), float(r)], [h * r, w * r])
    ev[3].record()
    sums = torch.stack([metrics.sums_device(sr, imgs[-1], nodata), metrics.sums_device(baseline, imgs[-1], nodata)])
    ev[4].record()
    sums = sums.cpu().numpy()
    C = int(imgs[-1].shape[2])
    return {'dsen2': metrics.measures(sums[0], C), 'bicubic': metrics.measures(sums[1], C), 'sr': sr, 'baseline': baseline,
            'times_ms': {s: ev[i].elapsed_time(ev[i + 1]) for i, s in enumerate(_STAGES)}}


def _fmt(v, spec):
    return '-' if v is None else format(v, spec)


def print_table(title, dsen2, bicubic):
    print(title)
    print('%-8s %11s %11s %10s %10s %9s %9s' % ('band', 'RMSE DSen2', 'RMSE bicub', 'SRE DSen2', 'SRE bicub', 'UIQ DSen2',
                                                'UIQ bicub'))
    for b in range(len(dsen2['rmse_bands'])):
        print('%-8s %11s %11s %10s %10s %9s %9s' % (
            b, _fmt(dsen2['rmse_bands'][b], '.3f'), _fmt(bicubic['rmse_bands'][b], '.3f'), _fmt(dsen2['sre_bands'][b], '.3f'),
            _fmt(bicubic['sre_bands'][b], '.3f'), _fmt(dsen2['uiq_bands'][b], '.5f'), _fmt(bicubic['uiq_bands'][b], '.5f')))
    print('%-8s %11s %11s %10s %10s %9s %9s' % (
        'overall', _fmt(dsen2['rmse'], '.3f'), _fmt(bicubic['rmse'], '.3f'), _fmt(dsen2['sre'], '.3f'),
        _fmt(bicubic['sre'], '.3f'), _fmt(dsen2['uiq'], '.5f'), _fmt(bicubic['uiq'], '.5f')))
    print('SAM (degrees): DSen2 %s, bicubic %s;  %d pixels scored' % (_fmt(dsen2['sam'], '.4f'), _fmt(bicubic['sam'], '.4f'),
                                                                      dsen2['pixels']))


def _model(run_60, deep, weights, random_weights):
    from .DSen2Net import s2model
    shape = ((4, None, None), (6, None, None)) + (((2, None, None),) if run_60 else ())
    layers, features = (32, 256) if deep else (6, 128)
    if random_weights:
        return s2model(shape, num_layers=layers, feature_size=features, seed=0)
    model = s2model(shape, num_layers=layers, feature_size=features)
    model.load_weights(weights or supres.weight_file(deep, run_60))
    return model


def _upload(torch, a):
    a = np.ascontiguousarray(a if a.dtype in (np.uint16, np.float32) else a.astype(np.float32))
    return torch.from_numpy(a).cuda()


def evaluate_product(args):
    nodata = None if args.nodata is None else float(args.nodata)
    model = _model(args.run_60, args.deep, args.weights, args.random_weights)
    bands = read_bands(args.product, args.roi_x_y, args.run_60)
    if bands is None:
        return None
    imgs = [bands[0], bands[1]] + ([bands[2]] if args.run_60 else [])
    check_wald(model, [a.shape for a in imgs], [a.dtype for a in imgs], nodata, args.add_offset)
    torch = _capi.require_cuda()
    res = wald_device(model, *[_upload(torch, a) for a in imgs], nodata=nodata, add_offset=args.add_offset)
    name = os.path.split(args.product.rstrip('/'))[1]
    print_table('%s (%d m -> 10 m, Wald protocol, ROI %s)' % (name, 60 if args.run_60 else 20, list(bands[3])),
                res['dsen2'], res['bicubic'])
    return [{'scene': name, 'roi': list(bands[3]), 'dsen2': res['dsen2'], 'bicubic': res['bicubic'],
             'times_ms': res['times_ms']}]


def evaluate_predictions(args):
    sub, gt, low, r = ('test60', 'data60_gt', 'data60', 6) if args.run_60 else ('test', 'data20_gt', 'data20', 2)
    found = []
    for scene in sorted(glob.glob(os.path.join(args.predictions, sub, '*', ''))):
        preds = sorted(glob.glob(os.path.join(scene, '*-predict.npy')))
        if preds:
            found.append((scene, preds))
    if not found:
        raise ValueError("no %s/<scene>/*-predict.npy under %s" % (sub, args.predictions))
    loaded = []
    for scene, preds in found:                           # every array is read and checked before the device is touched
        ref = np.load(os.path.join(scene, 'no_tiling', gt + '.npy'))
        lo = np.load(os.path.join(scene, 'no_tiling', low + '.npy'))
        if tuple(lo.shape[:2]) != (ref.shape[0] // r, ref.shape[1] // r) or lo.ndim != 3 or lo.shape[2] != ref.shape[2]:
            raise ValueError("%s: %s %s does not match %s %s" % (scene, low, lo.shape, gt, ref.shape))
        ests = []
        for p in preds:
            est = np.load(p)
            metrics.check_args(est.shape, est.dtype, ref.shape, ref.dtype, args.nodata)
            ests.append((p, est))
        metrics.check_args(ref.shape, 'float64', ref.shape, ref.dtype, args.nodata)
        loaded.append((scene, ref, lo, ests))
    torch = _capi.require_cuda()
    out = []
    for scene, ref, lo, ests in loaded:
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        d_ref = torch.from_numpy(np.ascontiguousarray(ref)).cuda()
        d_low = torch.from_numpy(np.ascontiguousarray(lo, dtype=np.float64 if lo.dtype == np.float64 else np.float32)).cuda()
        ev[0].record()
        baseline = imresize_device(d_low, [float(r), float(r)], [lo.shape[0] * r, lo.shape[1] * r])
        ev[1].record()
        q_bc = metrics.quality_device(baseline, d_ref, args.nodata)
        ev[2].record()
        name = os.path.basename(os.path.dirname(scene))
        for path, est in ests:
            t0 = torch.cuda.Event(enable_timing=True)
            t1 = torch.cuda.Event(enable_timing=True)
            d_est = torch.from_numpy(np.ascontiguousarray(est)).cuda()
            t0.record()
            q = metrics.quality_device(d_est, d_ref, args.nodata)
            t1.record()
            t1.synchronize()
            print_table('%s: %s (%d m -> 10 m)' % (name, os.path.basename(path), 60 if args.run_60 else 20), q, q_bc)
            out.append({'scene': name, 'prediction': os.path.basename(path), 'dsen2': q, 'bicubic': q_bc,
                        'times_ms': {'bicubic': ev[0].elapsed_time(ev[1]), 'metrics_bicubic': ev[1].elapsed_time(ev[2]),
                                     'metrics': t0.elapsed_time(t1)}})
    return out


def build_parser():
    p = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    p.add_argument('product', nargs='?', help='A Sentinel-2 SAFE directory (read through GDAL) or a .npz product container.')
    p.add_argument('--predictions', metavar='DATA_PATH', help='Score the *-predict.npy of test/<scene>/ (test60/) instead.')
    p.add_argument('--run_60', action='store_true', help='The 60 m path (60 m -> 10 m); default 20 m -> 10 m.')
    p.add_argument('--deep', action='store_true', help='VDSen2 (32 resBlocks x 256 features).')
    w = p.add_mutually_exclusive_group()
    w.add_argument('--weights', help='Weight file (default: the shipped file of supres.MDL_PATH).')
    w.add_argument('--random-weights', action='store_true', help='Seeded he_uniform weights instead of a weight file.')
    p.add_argument('--roi_x_y', default='', help='Region of interest on the 10 m bands: x_1,y_1,x_2,y_2 (36-pixel rounded).')
    p.add_argument('--nodata', type=float, help='Reference pixels whose every target band equals this value are not scored.')
    p.add_argument('--add_offset', type=float, help='Radiometric offset of the product (e.g. -1000), passed to the network.')
    p.add_argument('--json', help='Write the values and the stage times to this file.')
    return p


def main(argv=None):
    p = build_parser()
    args = p.parse_args(argv)
    if (args.product is None) == (args.predictions is None):
        p.error('give either a PRODUCT or --predictions DATA_PATH')
    if args.predictions is not None:
        res = evaluate_predictions(args)
    else:
        res = evaluate_product(args)
        if res is None:
            return 1
    if args.json:
        with open(args.json, 'w') as fh:
            json.dump({'mode': 'predictions' if args.predictions else 'product', 'run_60': args.run_60, 'scenes': res},
                      fh, indent=1)
    return 0


if __name__ == '__main__':
    sys.exit(main())
