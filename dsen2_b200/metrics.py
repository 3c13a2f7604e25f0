"""Image quality on the device: RMSE, SRE, SAM and UIQ of an estimate against a reference (csrc/metrics.cu).

These are the measures the DSen2 paper reports.  ``est`` and ``ref`` are HWC (H, W, C) images with 1 <= C <= 16, each one
float32, float64 or uint16 on its own; every value is read exactly as float64 and all arithmetic is float64.

- Valid pixels: all of them without ``nodata``; with ``nodata=v`` a pixel is invalid iff every band of the REFERENCE
  equals v in the reference's element type (a float64 reference takes only float32 values of v).
- Per band b over the n valid pixels, E_b = sum (est - ref)^2 and S_b = sum ref: RMSE_b = sqrt(E_b / n) and
  SRE_b = 10 log10((S_b / n)^2 / (E_b / n)) dB (+inf when E_b = 0).
- UIQ_b: the mean Wang-Bovik Q = 4 cov mean_est mean_ref / ((var_est + var_ref)(mean_est^2 + mean_ref^2)) over the 8 x 8
  windows (origins one pixel apart) whose 64 pixels are valid and whose denominator is not zero (population moments, means
  first, then centred sums).
- SAM: the mean spectral angle acos(clamp(<est, ref> / (|est| |ref|), -1, 1)) in degrees over the valid pixels where both
  vectors are non-zero.
- Overall: RMSE = sqrt(sum_b E_b / (n C)) (``demoDSen2.RMSE`` when no pixel is excluded), SRE and UIQ the means of the
  per-band values (UIQ over the bands that have a used window).  A measure without pixels or windows is None.

The result is a dict: overall ``rmse``, ``sre``, ``sam``, ``uiq``; per-band lists ``rmse_bands``, ``sre_bands``,
``uiq_bands``; counts ``pixels``, ``sam_pixels`` and per-band ``uiq_windows``.
"""
import math

import numpy as np

from . import _capi

MAX_BANDS = 16
_CODES = {'float32': _capi.IMG_F32, 'uint16': _capi.IMG_U16, 'float64': _capi.IMG_F64}


def _dtype_name(dt):
    name = str(dt)
    return name[len('torch.'):] if name.startswith('torch.') else np.dtype(dt).name


def check_args(est_shape, est_dtype, ref_shape, ref_dtype, nodata):
    """(H, W, C, est code, ref code, nodata as float or None) of a call; ``ValueError`` for anything the kernel does not
    take: shapes that differ or are not HWC, C outside 1..16, another dtype, a NaN nodata, and a nodata that is not an
    integer in [0, 65535] with a uint16 reference."""
    est_shape, ref_shape = tuple(int(s) for s in est_shape), tuple(int(s) for s in ref_shape)
    if est_shape != ref_shape or len(ref_shape) != 3 or min(ref_shape) < 1:
        raise ValueError("est and ref must be HWC images of the same shape, got %s and %s" % (est_shape, ref_shape))
    H, W, C = ref_shape
    if C > MAX_BANDS:
        raise ValueError("at most %d bands, got %d" % (MAX_BANDS, C))
    names = (_dtype_name(est_dtype), _dtype_name(ref_dtype))
    if any(n not in _CODES for n in names):
        raise ValueError("est and ref must each be float32, float64 or uint16, got %s and %s" % names)
    v = None
    if nodata is not None:
        v = float(nodata)
        if math.isnan(v):
            raise ValueError("nodata must not be NaN")
        if names[1] == 'uint16' and not (v.is_integer() and 0 <= v <= 65535):
            raise ValueError("nodata %r is not a uint16 value (an integer in [0, 65535])" % (nodata,))
        if names[1] == 'float64' and float(np.float32(v)) != v:       # the C call takes nodata as a float
            raise ValueError("nodata %r of a float64 reference must be a float32 value" % (nodata,))
    return H, W, C, _CODES[names[0]], _CODES[names[1]], v


def sums_device(est, ref, nodata=None):
    """The 5 C + 2 raw float64 sums of ``dsen2_image_quality`` (per band E_b, S_b, n, sum Q_b, used windows; then the sum
    of spectral angles in radians and the SAM pixel count) as a CUDA tensor.  ``est`` / ``ref``: CUDA tensors."""
    H, W, C, ce, cr, v = check_args(est.shape, est.dtype, ref.shape, ref.dtype, nodata)
    torch = _capi.require_cuda()
    if not (est.is_cuda and ref.is_cuda and est.device == ref.device):
        raise ValueError("est and ref must be CUDA tensors on one device")
    est, ref = est.contiguous(), ref.contiguous()
    lib = _capi.lib()
    nbytes = lib.dsen2_image_quality_workspace_bytes(H, W, C)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=ref.device)
    sums = torch.empty((5 * C + 2,), dtype=torch.float64, device=ref.device)
    with torch.cuda.device(ref.device):
        rc = lib.dsen2_image_quality(_capi.ptr(est), ce, _capi.ptr(ref), cr, H, W, C, int(v is not None),
                                     0.0 if v is None else v, _capi.ptr(ws), nbytes, _capi.ptr(sums), _capi.stream_ptr())
    _capi.check(rc, "dsen2_image_quality")
    return sums


def measures(sums, C):
    """The measures (module docstring) from the raw sums (a length 5 C + 2 sequence)."""
    s = [float(x) for x in sums]
    band = [s[5 * b:5 * b + 5] for b in range(C)]
    n = band[0][2]
    ang, nsam = s[5 * C], s[5 * C + 1]
    rmse_b = [math.sqrt(E / n) if n else None for E, _S, _n, _q, _u in band]
    sre_b = []
    for E, S, _n, _q, _u in band:
        if not n:
            sre_b.append(None)
        elif E == 0:
            sre_b.append(math.inf)
        else:
            r = (S / n) ** 2 / (E / n)
            sre_b.append(10 * math.log10(r) if r > 0 else -math.inf)
    uiq_b = [q / u if u else None for _E, _S, _n, q, u in band]
    have = [u for u in uiq_b if u is not None]
    return {
        'rmse': math.sqrt(sum(b[0] for b in band) / (n * C)) if n else None,
        'sre': sum(sre_b) / C if n else None,
        'sam': math.degrees(ang / nsam) if nsam else None,
        'uiq': sum(have) / len(have) if have else None,
        'rmse_bands': rmse_b, 'sre_bands': sre_b, 'uiq_bands': uiq_b,
        'pixels': int(n), 'sam_pixels': int(nsam), 'uiq_windows': [int(b[4]) for b in band],
    }


def quality_device(est, ref, nodata=None):
    """Measures of the CUDA HWC tensor ``est`` against ``ref`` (module docstring); one device -> host read of the sums."""
    sums = sums_device(est, ref, nodata)
    return measures(sums.cpu().numpy(), int(ref.shape[2]))


def quality(est, ref, nodata=None):
    """``quality_device`` for numpy arrays, uploaded in their own dtype."""
    est, ref = np.asarray(est), np.asarray(ref)
    check_args(est.shape, est.dtype, ref.shape, ref.dtype, nodata)
    torch = _capi.require_cuda()
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return quality_device(up(est), up(ref), nodata)
