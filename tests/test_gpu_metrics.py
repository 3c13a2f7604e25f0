"""Image quality kernels (csrc/metrics.cu) against the numpy oracle, at full tile size against a float64 torch restatement,
and the Wald-protocol evaluation (dsen2_b200/evaluate.py) end to end."""
import json
import math
import os
import shutil

import numpy as np
import pytest
import torch

from dsen2_b200 import create_patches, evaluate, metrics, supres, supres_train
from dsen2_b200.DSen2Net import s2model
from dsen2_b200.imresize import imresize
from dsen2_b200.patches import downPixelAggr
from oracle import metrics_oracle as mo
from test_s2_tiles import _product

pytestmark = pytest.mark.gpu

NP = {'float32': np.float32, 'float64': np.float64, 'uint16': np.uint16}


def _pair(H, W, C, est_dt, ref_dt, nodata, seed):
    """ref: smooth field + noise in ref_dt; est: ref + noise in est_dt; a block flat in both images, a few zero estimate
    vectors; with nodata v, random holes and a swath edge of v in every band of ref."""
    rng = np.random.RandomState(seed)
    yy, xx = np.mgrid[0:H, 0:W]
    base = 3000 + 1500 * np.sin(yy[:, :, None] / 17.0 + np.arange(C)) * np.cos(xx[:, :, None] / 23.0)
    ref = base + rng.randn(H, W, C) * 200
    est = ref + rng.randn(H, W, C) * 150
    est[rng.rand(H, W) < 0.002] = 0
    ref[H // 4:H // 4 + 20, W // 3:W // 3 + 30] = 1234
    est[H // 4:H // 4 + 20, W // 3:W // 3 + 30] = 1200
    ref = ref.astype(NP[ref_dt]) if ref_dt != 'uint16' else np.clip(np.rint(ref), 1, 65535).astype(np.uint16)
    est = est.astype(NP[est_dt]) if est_dt != 'uint16' else np.clip(np.rint(est), 0, 65535).astype(np.uint16)
    if nodata is not None:
        ref[rng.rand(H, W) < 0.01] = nodata
        ref[xx > 2 * yy + W // 2] = nodata
    return est, ref


def _check_sums(got, want, C):
    got, want = np.asarray(got).reshape(-1), np.asarray(want).reshape(-1)
    for b in range(C):
        E, S, n, Q, U = got[5 * b:5 * b + 5]
        e, s, m, q, u = want[5 * b:5 * b + 5]
        assert (n, U) == (m, u), (b, n, m, U, u)
        assert abs(E - e) <= 1e-12 * abs(e) and abs(S - s) <= 1e-12 * abs(s), (b, E, e, S, s)
        if u:
            assert abs(Q / U - q / u) <= 1e-9, (b, Q / U, q / u)
    assert got[5 * C + 1] == want[5 * C + 1]
    if want[5 * C + 1]:
        assert abs(math.degrees(got[5 * C] / got[5 * C + 1]) - math.degrees(want[5 * C] / want[5 * C + 1])) <= 1e-6


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


DT = ('float32', 'float64', 'uint16')


@pytest.mark.parametrize('est_dt', DT)
@pytest.mark.parametrize('ref_dt', DT)
def test_every_dtype_pair_against_the_oracle(est_dt, ref_dt):
    for nodata, seed in ((None, 1), (0, 2)):
        est, ref = _pair(203, 517, 6, est_dt, ref_dt, nodata, seed)
        _check_sums(metrics.sums_device(_dev(est), _dev(ref), nodata).cpu().numpy(), mo.sums(est, ref, nodata), 6)


@pytest.mark.parametrize('C', [1, 2, 4, 6, 16])
@pytest.mark.parametrize('nodata', [None, 7])
def test_band_counts_against_the_oracle(C, nodata):
    est, ref = _pair(203, 517, C, 'float32', 'uint16', nodata, 10 + C)
    got = metrics.quality_device(_dev(est), _dev(ref), nodata)
    _check_sums(metrics.sums_device(_dev(est), _dev(ref), nodata).cpu().numpy(), mo.sums(est, ref, nodata), C)
    want = mo.quality(est, ref, nodata)
    assert got['pixels'] == want['pixels'] and got['uiq_windows'] == want['uiq_windows']
    assert got['sam_pixels'] == want['sam_pixels']
    assert abs(got['rmse'] - want['rmse']) <= 1e-12 * want['rmse'] and abs(got['uiq'] - want['uiq']) <= 1e-9


def test_flat_uint16_windows_are_skipped_exactly():
    est, ref = _pair(120, 140, 3, 'uint16', 'uint16', None, 4)
    sums = metrics.sums_device(_dev(est), _dev(ref)).cpu().numpy()
    want = mo.sums(est, ref)
    _check_sums(sums, want, 3)
    assert all(sums[5 * b + 4] == 113 * 133 - 13 * 23 for b in range(3))     # the 20 x 30 block flat in both images


@pytest.mark.parametrize('H, W', [(5, 40), (40, 7), (1, 1), (8, 8), (9, 300)])
def test_small_images(H, W):
    est, ref = _pair(H, W, 4, 'float64', 'float32', None, 5)
    sums = metrics.sums_device(_dev(est), _dev(ref)).cpu().numpy()
    _check_sums(sums, mo.sums(est, ref), 4)
    assert sums[4] == max(0, H - 7) * max(0, W - 7)


def test_all_nodata_reference_is_none():
    ref = np.full((30, 40, 6), 3, np.uint16)
    q = metrics.quality(np.ones((30, 40, 6), np.float32), ref, nodata=3)
    assert q['rmse'] is q['sre'] is q['sam'] is q['uiq'] is None and q['pixels'] == q['sam_pixels'] == 0
    assert q['uiq_windows'] == [0] * 6 and q['rmse_bands'] == [None] * 6


def test_deterministic():
    est, ref = _pair(700, 900, 6, 'float32', 'uint16', 0, 6)
    a = metrics.sums_device(_dev(est), _dev(ref), 0)
    b = metrics.sums_device(_dev(est), _dev(ref), 0)
    assert torch.equal(a, b)


def _torch_restatement(est, ref):
    """float64 per band (E, S, sum Q, windows) with plain torch sums and avg_pool2d windows, and the SAM mean (degrees)."""
    F = torch.nn.functional
    out = []
    for b in range(ref.shape[2]):
        x = est[:, :, b].double()[None, None]
        y = ref[:, :, b].double()[None, None]
        pool = lambda t: F.avg_pool2d(t, 8, stride=1)
        mx, my = pool(x), pool(y)
        vx, vy, cxy = pool(x * x) - mx * mx, pool(y * y) - my * my, pool(x * y) - mx * my
        den = (vx + vy) * (mx * mx + my * my)
        q = 4 * cxy * mx * my / den
        use = den != 0
        out.append((float(((x - y) ** 2).sum()), float(y.sum()), float(q[use].sum()), int(use.sum())))
        del x, y, mx, my, vx, vy, cxy, den, q
    ang, cnt = 0.0, 0
    for r0 in range(0, ref.shape[0], 1024):
        xe, xr = est[r0:r0 + 1024].double(), ref[r0:r0 + 1024].double()
        ne, nr = (xe * xe).sum(2).sqrt(), (xr * xr).sum(2).sqrt()
        nz = (ne > 0) & (nr > 0)
        c = ((xe * xr).sum(2)[nz] / (ne[nz] * nr[nz])).clamp(-1, 1)
        ang += float(torch.acos(c).sum())
        cnt += int(nz.sum())
    return out, math.degrees(ang / cnt), cnt


@pytest.mark.parametrize('n, est_dtype', [(5490, torch.float32), (10980, torch.float64)])
def test_full_size_against_torch(n, est_dtype):
    g = torch.Generator(device='cuda').manual_seed(n)
    ref = (torch.rand((n, n, 6), generator=g, device='cuda') * 8000 + 500).round_().to(torch.int32).to(torch.int16)
    ref = ref.view(torch.uint16)
    est = (ref.view(torch.int16).to(est_dtype) + torch.randn((n, n, 6), generator=g, device='cuda', dtype=est_dtype) * 100)
    sums = metrics.sums_device(est, ref).cpu().numpy()
    refi = ref.view(torch.int16)
    want, sam, cnt = _torch_restatement(est, refi)
    for b, (E, S, Q, U) in enumerate(want):
        assert sums[5 * b + 2] == n * n and sums[5 * b + 4] == U == (n - 7) ** 2
        assert abs(sums[5 * b] - E) <= 1e-6 * E and abs(sums[5 * b + 1] - S) <= 1e-6 * S
        assert abs(sums[5 * b + 3] / sums[5 * b + 4] - Q / U) <= 1e-6
    assert sums[31] == cnt and abs(math.degrees(sums[30] / sums[31]) - sam) <= 1e-6


def _crop(scene, n=576):
    d10, d20, d60 = scene
    return d10[:n, :n], d20[:n // 2, :n // 2], d60[:n // 6, :n // 6]


def _check_measures(got, want):
    assert got['pixels'] == want['pixels'] and got['sam_pixels'] == want['sam_pixels']
    assert got['uiq_windows'] == want['uiq_windows']
    for k in ('rmse', 'sre'):
        assert abs(got[k] - want[k]) <= 1e-12 * abs(want[k]), k
    for a, b in zip(got['rmse_bands'] + got['sre_bands'], want['rmse_bands'] + want['sre_bands']):
        assert abs(a - b) <= 1e-12 * abs(b)
    assert abs(got['uiq'] - want['uiq']) <= 1e-9 and abs(got['sam'] - want['sam']) <= 1e-6
    assert all(abs(a - b) <= 1e-9 for a, b in zip(got['uiq_bands'], want['uiq_bands']))


@pytest.mark.parametrize('name, u16, nodata', [('malmo', False, None), ('shark', True, 0)])
def test_wald_20m_end_to_end(name, u16, nodata, malmo, shark):
    d10, d20, _ = _crop(malmo if name == 'malmo' else shark)
    if u16:
        d10, d20 = d10.astype(np.uint16), d20.astype(np.uint16)
    m = s2model(((4, None, None), (6, None, None)), num_layers=6, feature_size=128, seed=0)
    res = evaluate.wald_device(m, _dev(d10), _dev(d20), nodata=nodata)
    lr10, lr20 = downPixelAggr(d10, 2).astype(np.float32), downPixelAggr(d20, 2).astype(np.float32)
    sr = supres.DSen2_20(lr10, lr20, model=m)
    bc = imresize(lr20, 2)
    assert np.array_equal(res['sr'].cpu().numpy(), sr) and np.array_equal(res['baseline'].cpu().numpy(), bc)
    _check_measures(res['dsen2'], mo.quality(sr, d20, nodata))
    _check_measures(res['bicubic'], mo.quality(bc, d20, nodata))
    assert set(res['times_ms']) == {'degrade', 'sr', 'bicubic', 'metrics'}


def test_wald_60m_end_to_end():
    rng = np.random.RandomState(60)
    n = 1080

    def field(h, w, c):
        return np.clip(np.repeat(np.repeat(rng.randint(500, 6000, (h // 12 + 1, w // 12 + 1, c)), 12, 0), 12, 1)[:h, :w] +
                       rng.randint(0, 300, (h, w, c)), 0, 65535).astype(np.uint16)
    d10, d20, d60 = field(n, n, 4), field(n // 2, n // 2, 6), field(n // 6, n // 6, 2)
    m = s2model(((4, None, None), (6, None, None), (2, None, None)), num_layers=6, feature_size=128, seed=0)
    res = evaluate.wald_device(m, _dev(d10), _dev(d20), _dev(d60))
    lr = [downPixelAggr(a, 6).astype(np.float32) for a in (d10, d20, d60)]
    sr = supres.DSen2_60(*lr, model=m)
    bc = imresize(lr[2], 6)
    assert np.array_equal(res['sr'].cpu().numpy(), sr) and np.array_equal(res['baseline'].cpu().numpy(), bc)
    _check_measures(res['dsen2'], mo.quality(sr, d60))
    _check_measures(res['bicubic'], mo.quality(bc, d60))


KEYS = {'rmse', 'sre', 'sam', 'uiq', 'rmse_bands', 'sre_bands', 'uiq_bands', 'pixels', 'sam_pixels', 'uiq_windows'}


def test_cli_product_and_predictions(tmp_path):
    path = _product(tmp_path, H=504, W=504)
    out = str(tmp_path / 'product.json')
    assert evaluate.main([path, '--random-weights', '--nodata', '0', '--json', out]) == 0
    res = json.load(open(out))
    assert res['mode'] == 'product' and len(res['scenes']) == 1
    s = res['scenes'][0]
    assert set(s['dsen2']) == KEYS == set(s['bicubic']) and set(s['times_ms']) == {'degrade', 'sr', 'bicubic', 'metrics'}
    assert s['dsen2']['pixels'] <= 252 * 252 and len(s['dsen2']['rmse_bands']) == 6
    # test data, a saved random model's predictions, and their scores
    prefix = str(tmp_path / 'data') + '/'
    os.makedirs(prefix)
    assert create_patches.main([path, '--test_data', '--save_prefix', prefix]) == 0
    shutil.move(prefix + 'test/product.npz', prefix + 'test/S2X_TEST.SAFE')       # supres_train --predict reads *SAFE
    weights = str(tmp_path / 's2_038_lr_1e-04.hdf5')
    s2model(((4, None, None), (6, None, None)), num_layers=6, feature_size=128, seed=3).save_weights(weights)
    assert supres_train.main(['--predict', weights, '--path', prefix]) == 0
    out = str(tmp_path / 'pred.json')
    assert evaluate.main(['--predictions', prefix, '--json', out]) == 0
    res = json.load(open(out))
    assert res['mode'] == 'predictions' and [s['scene'] for s in res['scenes']] == ['S2X_TEST.SAFE']
    s = res['scenes'][0]
    assert s['prediction'] == 's2_038_-predict.npy' and set(s['dsen2']) == KEYS
    gt = np.load(prefix + 'test/S2X_TEST.SAFE/no_tiling/data20_gt.npy')
    pred = np.load(prefix + 'test/S2X_TEST.SAFE/s2_038_-predict.npy')
    _check_measures(s['dsen2'], mo.quality(pred, gt))
    bc = imresize(np.load(prefix + 'test/S2X_TEST.SAFE/no_tiling/data20.npy'), 2)
    _check_measures(s['bicubic'], mo.quality(bc, gt))
