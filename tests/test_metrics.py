"""Image quality measures without a GPU: properties of the numpy oracle (oracle/metrics_oracle.py), and every ValueError of
metrics.quality, evaluate.wald_device and the evaluate CLI, raised before a CUDA device is needed."""
import math

import numpy as np
import pytest
import torch

from dsen2_b200 import demoDSen2, evaluate, metrics
from dsen2_b200.DSen2Net import s2model
from oracle import metrics_oracle as mo
from test_s2_tiles import _product


def _img(rng, H, W, C, lo=200, hi=6000):
    return rng.randint(lo, hi, (H, W, C)).astype(np.float32)


def test_identical_images():
    ref = _img(np.random.RandomState(0), 30, 41, 4)
    q = mo.quality(ref, ref)
    assert q['rmse'] == 0 and q['sre'] == math.inf and all(s == math.inf for s in q['sre_bands'])
    assert q['sam'] < 1e-6                                   # acos of a rounded 1
    assert all(abs(u - 1) < 1e-12 for u in q['uiq_bands']) and q['uiq_windows'] == [23 * 34] * 4
    assert q['pixels'] == q['sam_pixels'] == 30 * 41


def test_scaled_estimate_has_no_spectral_angle():
    rng = np.random.RandomState(1)
    ref = _img(rng, 17, 19, 6)
    q = mo.quality(ref.astype(np.float64) * 1.7, ref)
    assert q['sam'] < 1e-6 and q['rmse'] > 0


def test_overall_rmse_is_demo_rmse():
    rng = np.random.RandomState(2)
    ref = _img(rng, 33, 29, 6)
    est = ref + rng.randn(33, 29, 6).astype(np.float32) * 40
    q = mo.quality(est, ref)
    want = demoDSen2.RMSE(est, ref)
    assert abs(q['rmse'] - want) <= 1e-12 * want
    assert all(abs(r - np.sqrt(np.mean((est[:, :, b].astype(np.float64) - ref[:, :, b]) ** 2))) <= 1e-12 * r
               for b, r in enumerate(q['rmse_bands']))


def test_flat_uint16_blocks_and_nodata_skip_windows():
    """Windows inside a block where both images are flat have a zero denominator and are skipped; windows touching a nodata
    pixel of the reference are not scored, and neither is the pixel."""
    rng = np.random.RandomState(3)
    ref = rng.randint(100, 9000, (40, 50, 2)).astype(np.uint16)
    est = rng.randint(100, 9000, (40, 50, 2)).astype(np.uint16)
    ref[5:21, 10:30] = 777                                   # 16 x 20 flat block in both images, both bands
    est[5:21, 10:30] = 1234
    q = mo.quality(est, ref)
    windows = 33 * 43
    assert q['uiq_windows'] == [windows - 9 * 13] * 2
    ref[30, 40] = 0                                          # one nodata pixel: all bands 0
    ref[31, 41, 0] = 0                                       # only one band 0: still valid
    q = mo.quality(est, ref, nodata=0)
    assert q['pixels'] == 40 * 50 - 1
    assert q['uiq_windows'] == [windows - 9 * 13 - 64] * 2   # the 8 x 8 origins whose window covers (30, 40)


def test_measures_of_the_product_module_match_the_oracle_on_raw_sums():
    rng = np.random.RandomState(4)
    ref = _img(rng, 20, 24, 3)
    est = ref + rng.randn(20, 24, 3).astype(np.float32) * 30
    ref[2, 3] = 0
    got = metrics.measures(mo.sums(est, ref, 0), 3)
    want = mo.quality(est, ref, 0)
    for k, v in want.items():
        assert np.allclose(np.array(got[k], np.float64), np.array(v, np.float64), rtol=1e-13, atol=0), k


def test_all_nodata_reference_gives_none():
    ref = np.full((9, 9, 2), 5, np.uint16)
    est = np.ones((9, 9, 2), np.float32)
    q = mo.quality(est, ref, nodata=5)
    got = metrics.measures(mo.sums(est, ref, 5), 2)
    for d in (q, got):
        assert d['rmse'] is d['sre'] is d['sam'] is d['uiq'] is None
        assert d['rmse_bands'] == d['sre_bands'] == d['uiq_bands'] == [None, None] and d['pixels'] == 0


@pytest.mark.parametrize('est, ref, nodata, what', [
    (np.zeros((8, 9, 3), np.float32), np.zeros((9, 8, 3), np.float32), None, 'same shape'),
    (np.zeros((8, 9), np.float32), np.zeros((8, 9), np.float32), None, 'HWC'),
    (np.zeros((8, 9, 17), np.float32), np.zeros((8, 9, 17), np.float32), None, 'at most 16'),
    (np.zeros((8, 9, 3), np.int32), np.zeros((8, 9, 3), np.float32), None, 'float32, float64 or uint16'),
    (np.zeros((8, 9, 3), np.float32), np.zeros((8, 9, 3), np.float16), None, 'float32, float64 or uint16'),
    (np.zeros((8, 9, 3), np.float32), np.zeros((8, 9, 3), np.float32), float('nan'), 'NaN'),
    (np.zeros((8, 9, 3), np.float32), np.zeros((8, 9, 3), np.uint16), 1.5, 'uint16 value'),
    (np.zeros((8, 9, 3), np.float32), np.zeros((8, 9, 3), np.uint16), -1, 'uint16 value'),
    (np.zeros((8, 9, 3), np.float32), np.zeros((8, 9, 3), np.float64), 0.1, 'float32 value'),
])
def test_quality_rejects_before_the_device(est, ref, nodata, what):
    with pytest.raises(ValueError, match=what):
        metrics.quality(est, ref, nodata)


def _cpu(shape, dtype=torch.float32):
    return torch.zeros(shape, dtype=dtype)


M20 = s2model(((4, None, None), (6, None, None)), num_layers=1, feature_size=128, seed=0)
M60 = s2model(((4, None, None), (6, None, None), (2, None, None)), num_layers=1, feature_size=128, seed=0)


@pytest.mark.parametrize('model, shapes, kw, what', [
    (M20, [(226, 228, 4), (113, 114, 6)], {}, 'multiple of 4'),
    (M20, [(220, 240, 4), (110, 120, 6)], {}, 'smaller than one patch stride'),
    (M60, [(1044, 1026, 4), (522, 513, 6), (174, 171, 2)], {}, 'multiple of 36'),
    (M60, [(972, 1080, 4), (486, 540, 6), (162, 180, 2)], {}, 'smaller than one patch stride'),
    (M20, [(224, 224, 4), (112, 112, 5)], {}, 'expected an image of shape'),
    (M20, [(224, 224, 4), (112, 112, 6), (37, 37, 2)], {}, 'takes 2 inputs'),
    (M20, [(224, 224, 4), (112, 112, 6)], dict(nodata=float('nan')), 'NaN'),
    (M20, [(224, 224, 4), (112, 112, 6)], dict(add_offset=float('inf')), 'finite'),
])
def test_wald_rejects_before_the_device(model, shapes, kw, what):
    with pytest.raises(ValueError, match=what):
        evaluate.wald_device(model, *[_cpu(s) for s in shapes], **kw)


def test_wald_rejects_other_dtypes_and_uint16_nodata():
    with pytest.raises(ValueError, match='float32 or uint16'):
        evaluate.wald_device(M20, _cpu((224, 224, 4), torch.float64), _cpu((112, 112, 6)))
    with pytest.raises(ValueError, match='uint16 value'):
        evaluate.wald_device(M20, _cpu((224, 224, 4)), _cpu((112, 112, 6), torch.uint16), nodata=0.5)


def test_cli_rejects_before_the_device(tmp_path):
    path = _product(tmp_path, H=144, W=216)
    with pytest.raises(ValueError, match='smaller than one patch stride'):
        evaluate.main([path, '--random-weights'])
    with pytest.raises(ValueError, match='smaller than one patch stride'):
        evaluate.main([path, '--random-weights', '--run_60', '--roi_x_y', '0,0,99,99'])   # rounded to 72 x 72
    (tmp_path / 'big').mkdir()
    big = _product(tmp_path / 'big', H=252, W=252)
    with pytest.raises(ValueError, match='NaN'):
        evaluate.main([big, '--random-weights', '--nodata', 'nan'])
    with pytest.raises(ValueError, match='finite'):
        evaluate.main([big, '--random-weights', '--add_offset', 'inf'])
    with pytest.raises(ValueError, match='no test/<scene>'):
        evaluate.main(['--predictions', str(tmp_path)])
    with pytest.raises(SystemExit):
        evaluate.main([path, '--predictions', str(tmp_path)])
    with pytest.raises(SystemExit):
        evaluate.main([path, '--weights', 'w.hdf5', '--random-weights'])
