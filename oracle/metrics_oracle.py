"""numpy float64 restatement of the image quality measures of dsen2_b200/metrics.py (RMSE, SRE, SAM, UIQ).

Only the tests and the measurement tool import it.  ``sums`` gives the raw sums in the layout of ``dsen2_image_quality``;
``quality`` the measures from them, restated here rather than taken from the product package.
"""
import math

import numpy as np
from numpy.lib.stride_tricks import sliding_window_view


def valid_mask(ref, nodata=None):
    """(H, W) bool: False where every band of ``ref`` equals ``nodata`` in ref's element type."""
    ref = np.asarray(ref)
    if nodata is None:
        return np.ones(ref.shape[:2], bool)
    v = ref.dtype.type(nodata)
    return ~np.all(ref == v, axis=2)


def uiq_band(x, y, valid):
    """(sum of Q, used windows) of one band: 8 x 8 windows moved one pixel at a time whose 64 pixels are valid, two-pass
    population moments, a window used iff its denominator is not zero."""
    H, W = x.shape
    if H < 8 or W < 8:
        return 0.0, 0
    full = sliding_window_view(valid, (8, 8)).all(axis=(2, 3))
    xw = sliding_window_view(x, (8, 8))
    yw = sliding_window_view(y, (8, 8))
    mx = xw.mean(axis=(2, 3))
    my = yw.mean(axis=(2, 3))
    dx = xw - mx[:, :, None, None]
    dy = yw - my[:, :, None, None]
    vx = (dx * dx).mean(axis=(2, 3))
    vy = (dy * dy).mean(axis=(2, 3))
    cxy = (dx * dy).mean(axis=(2, 3))
    den = (vx + vy) * (mx * mx + my * my)
    use = full & (den != 0)
    q = 4 * cxy[use] * mx[use] * my[use] / den[use]
    return float(q.sum()), int(use.sum())


def sums(est, ref, nodata=None):
    """float64 (5 C + 2,): per band E_b, S_b, n, sum Q_b, used windows; then the sum of spectral angles (radians) and the
    number of pixels they are taken over."""
    ok = valid_mask(ref, nodata)
    x = np.asarray(est).astype(np.float64)
    y = np.asarray(ref).astype(np.float64)
    C = y.shape[2]
    xv, yv = x[ok], y[ok]
    n = xv.shape[0]
    out = []
    for b in range(C):
        d = xv[:, b] - yv[:, b]
        qs, used = uiq_band(x[:, :, b], y[:, :, b], ok)
        out += [float(np.sum(d * d)), float(np.sum(yv[:, b])), float(n), qs, float(used)]
    dot = np.sum(xv * yv, axis=1)
    nx = np.sqrt(np.sum(xv * xv, axis=1))
    ny = np.sqrt(np.sum(yv * yv, axis=1))
    nz = (nx > 0) & (ny > 0)
    ang = np.arccos(np.clip(dot[nz] / (nx[nz] * ny[nz]), -1.0, 1.0))
    out += [float(ang.sum()), float(nz.sum())]
    return np.array(out)


def quality(est, ref, nodata=None):
    """The measures of dsen2_b200.metrics (same dict keys) from ``sums``."""
    s = sums(est, ref, nodata)
    C = np.asarray(ref).shape[2]
    E, S, n, Q, U = (s[0:5 * C].reshape(C, 5)[:, k] for k in range(5))
    n = n[0]
    with np.errstate(divide='ignore'):
        sre = [None if n == 0 else (math.inf if e == 0 else float(10 * np.log10((t / n) ** 2 / (e / n))))
               for e, t in zip(E, S)]
    uiq = [float(q / u) if u else None for q, u in zip(Q, U)]
    have = [u for u in uiq if u is not None]
    return {
        'rmse': float(np.sqrt(E.sum() / (n * C))) if n else None,
        'sre': float(np.mean(sre)) if n else None,
        'sam': float(np.degrees(s[5 * C] / s[5 * C + 1])) if s[5 * C + 1] else None,
        'uiq': float(np.mean(have)) if have else None,
        'rmse_bands': [float(np.sqrt(e / n)) if n else None for e in E],
        'sre_bands': sre, 'uiq_bands': uiq,
        'pixels': int(n), 'sam_pixels': int(s[5 * C + 1]), 'uiq_windows': [int(u) for u in U],
    }
