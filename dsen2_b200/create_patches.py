"""Training / test patch generation -- mirror of ``training/create_patches.py`` (same options, same directory layout).

    python -m dsen2_b200.create_patches <product> [--roi_x_y x1,y1,x2,y2] [--test_data] [--write_images]
                                        [--save_prefix ../data/] [--run_60] [--true_data]

The reference script is one function around GDAL (``create_patches.py:19-316``).  Here the GDAL-free core is in functions
(ROI rounding to 36-pixel boundaries ``:60-71``, band selection ``:27-30,147-187``, the degradation to the training scale
``:219-232``, the ``train/ | train60/ | test/ | test60/ | true/`` layout with ``roi.json`` and the untiled arrays ``:241-316``)
and the product comes from the same sources as the tile driver: a GDAL data set where ``osgeo`` is importable, else a ``.npz``
product container (``dsen2_b200.s2_tiles_supres.NpzSource``).  The arithmetic runs on the GPU: ``patches.downPixelAggr``
(Gaussian sigma = 1/s + s x s mean, bit-identical to scipy), ``patches.save_*`` (crops, tiling, bilinear upsampling).
"""
import argparse
import json
import os
import re
import struct
import zlib

import numpy as np

from . import patches
from .s2_tiles_supres import choose_utm, get_band_short_name, open_source, read_windows

BANDS_20 = "B2,B3,B4,B5,B6,B7,B8,B8A,B11,B12"                   # create_patches.py:27-30
BANDS_60 = "B1,B2,B3,B4,B5,B6,B7,B8,B8A,B9,B11,B12"


def clamp_roi_36(x1, y1, x2, y2, xsize, ysize):
    """``:60-71``: clamp the ROI into the 10 m raster and SHRINK it to 36-pixel boundaries (a whole number of 60 m pixels of
    the 6x degraded image)."""
    xmin = max(min(x1, x2, xsize - 1), 0)
    xmax = min(max(x1, x2, 0), xsize - 1)
    ymin = max(min(y1, y2, ysize - 1), 0)
    ymax = min(max(y1, y2, 0), ysize - 1)
    return (int(xmin / 36) * 36, int(ymin / 36) * 36, int((xmax + 1) / 36) * 36 - 1, int((ymax + 1) / 36) * 36 - 1)


def validate_description(description):
    """``:128-135`` (no ENVI special case here, unlike the tile driver)."""
    m = re.match(r"(.*?), central wavelength (\d+) nm", description)
    if m:
        return m.group(1) + " (" + m.group(2) + " nm)"
    pos = description.find(',')
    return description[:pos] + description[(pos + 1):]


def select_bands(desc10, desc20, desc60, run_60):
    """``:27-30,147-187``: every wanted band is taken from the FIRST resolution that offers it.
    -> ((names, indices) for 10 / 20 / 60 m)."""
    wanted = re.split(',', BANDS_60 if run_60 else BANDS_20)
    out = []
    for descs in (desc10, desc20, desc60):
        names, idx = [], []
        for b, d in enumerate(descs):
            short = get_band_short_name(validate_description(d))
            if short in wanted:
                wanted.remove(short)
                names.append(short)
                idx.append(b)
        out.append((names, idx))
    return tuple(out)


def write_png(path, img01):
    """``save_band``'s ``imageio.imsave`` of a float image in [0, 1] (``:199-205``): 8-bit PNG, grey or RGB."""
    a = np.asarray(img01, np.float64)
    a = (np.clip(a, 0.0, 1.0) * 255 + 0.5).astype(np.uint8)
    if a.ndim == 2:
        a = a[:, :, None]
    h, w, c = a.shape
    raw = b''.join(b'\x00' + a[y].tobytes() for y in range(h))

    def chunk(tag, data):
        body = tag + data
        return struct.pack('>I', len(data)) + body + struct.pack('>I', zlib.crc32(body) & 0xffffffff)
    with open(path, 'wb') as f:
        f.write(b'\x89PNG\r\n\x1a\n' + chunk(b'IHDR', struct.pack('>IIBBBBB', w, h, 8, {1: 0, 3: 2}[c], 0, 0, 0)) +
                chunk(b'IDAT', zlib.compress(raw, 6)) + chunk(b'IEND', b''))


def save_band(save_prefix, data, name, percentile_data=None):
    """``:199-205``: clip to the 1st..99th percentile, scale to [0, 1], write ``<save_prefix><name>.png``."""
    if percentile_data is None:
        percentile_data = data
    mi, ma = np.percentile(percentile_data, (1, 99))
    band = (np.clip(data, mi, ma) - mi) / (ma - mi)
    os.makedirs(os.path.dirname(save_prefix + name), exist_ok=True)
    write_png(save_prefix + name + ".png", band)


def _mkdirs(*dirs):
    for d in dirs:
        if not os.path.isdir(d):
            os.mkdir(d)


def write_patches(data10, data20, data60, name, roi, test_data=False, save_prefix="../data/", write_images=False, run_60=False,
                  true_data=False):
    """``create_patches.py:207-316`` from the loaded bands on: degrade to the training scale, then write the patch files.
    ``roi`` = (xmin, ymin, xmax, ymax) on the 10 m raster, ``name`` = the product's directory name."""
    xmin, ymin, xmax, ymax = roi
    if np.sum(data10[:, :, 0] < 1) > 0:
        print('The selected image has some blank pixels')
    scale20, scale60 = 2, 6
    data10_gt, data20_gt, data60_gt = data10, data20, data60
    data10_lr = data20_lr = data60_lr = None
    if not true_data:                                        # Wald's protocol: the input resolution becomes the label (:219-232)
        s = scale60 if run_60 else scale20
        data10_lr = patches.downPixelAggr(data10_gt, SCALE=s)
        data20_lr = patches.downPixelAggr(data20_gt, SCALE=s)
        if run_60:
            data60_lr = patches.downPixelAggr(data60_gt, SCALE=s)
    print(name)
    if test_data:
        sub, s = ('test60/', scale60) if run_60 else ('test/', scale20)
        out = save_prefix + sub + name + '/'
        _mkdirs(save_prefix + sub, out)
        print('Writing files for testing to:{}'.format(out))
        if run_60:
            patches.save_test_patches60(data10_lr, data20_lr, data60_lr, out)
        else:
            patches.save_test_patches(data10_lr, data20_lr, out)
        with open(out + 'roi.json', 'w') as f:
            json.dump([xmin // s, ymin // s, (xmax + 1) // s, (ymax + 1) // s], f)
        _mkdirs(out + 'no_tiling/')
        print("Now saving the whole image without tiling...")
        if run_60:
            np.save(out + 'no_tiling/' + 'data60_gt', data60_gt.astype(np.float32))
            np.save(out + 'no_tiling/' + 'data60', data60_lr.astype(np.float32))
        else:
            np.save(out + 'no_tiling/' + 'data20_gt', data20_gt.astype(np.float32))
            save_band(save_prefix, data10_lr[:, :, 0:3], '/test/' + name + '/RGB')
        np.save(out + 'no_tiling/' + 'data10', data10_lr.astype(np.float32))
        np.save(out + 'no_tiling/' + 'data20', data20_lr.astype(np.float32))
    elif write_images:
        print('Creating RGB images...')
        save_band(save_prefix, data10_lr[:, :, 0:3], '/raw/rgbs/' + name + 'RGB')
        save_band(save_prefix, data20_lr[:, :, 0:3], '/raw/rgbs/' + name + 'RGB20')
    elif true_data:
        out = save_prefix + 'true/' + name + '/'
        _mkdirs(save_prefix + 'true/', out)
        print('Writing files for testing to:{}'.format(out))
        patches.save_test_patches60(data10_gt, data20_gt, data60_gt, out, patchSize=384, border=12)
        with open(out + 'roi.json', 'w') as f:
            json.dump([xmin, ymin, xmax + 1, ymax + 1], f)
        _mkdirs(out + 'no_tiling/')
        print("Now saving the whole image without tiling...")
        np.save(out + 'no_tiling/' + 'data10', data10_gt.astype(np.float32))
        np.save(out + 'no_tiling/' + 'data20', data20_gt.astype(np.float32))
        np.save(out + 'no_tiling/' + 'data60', data60_gt.astype(np.float32))
    else:
        sub = 'train60/' if run_60 else 'train/'
        out = save_prefix + sub + name + '/'
        _mkdirs(save_prefix + sub, out)
        print('Writing files for training to:{}'.format(out))
        if run_60:
            patches.save_random_patches60(data60_gt, data10_lr, data20_lr, data60_lr, out)
        else:
            patches.save_random_patches(data20_gt, data10_lr, data20_lr, out)
    print("Success.")


def read_bands(data_file, roi_x_y=None, run_60=False, true_data=False):
    """``create_patches.py:19-205``: the bands of the ROI (rounded to 36-pixel boundaries) of the UTM zone with the largest
    coverage, 10 / 20 / 60 m, in the product's own dtype -> (data10, data20, data60, (xmin, ymin, xmax, ymax)), or None
    for an empty region.  ``data_file``: a SAFE directory (its ``MTD_MSIL1C.xml`` is opened through GDAL) or a ``.npz``
    product container."""
    path = data_file if data_file.endswith('.npz') else data_file + '/MTD_MSIL1C.xml'
    src = open_source(path)
    cands = []
    for desc, (xs, ys) in src.candidates():
        if roi_x_y:
            x1, y1, x2, y2 = [float(x) for x in re.split(',', roi_x_y)]
            roi = clamp_roi_36(x1, y1, x2, y2, xs, ys)
        else:
            roi = (0, 0, xs - 1, ys - 1)
        cands.append((desc, roi))
    utm_idx, utm, (xmin, ymin, xmax, ymax), _ = choose_utm(cands)
    print("Selected UTM Zone:", utm)
    print("Selected pixel region: xmin=%d, ymin=%d, xmax=%d, ymax=%d:" % (xmin, ymin, xmax, ymax))
    print("Image size: width=%d x height=%d" % (xmax - xmin + 1, ymax - ymin + 1))
    if xmax < xmin or ymax < ymin:
        print("Invalid region of interest / UTM Zone combination")
        return None
    ds = src.open(utm_idx)
    (n10, i10), (n20, i20), (n60, i60) = select_bands(ds.descriptions(0), ds.descriptions(1), ds.descriptions(2), run_60)
    for label, names in (("10m", n10), ("20m", n20), ("60m", n60)):
        print("Selected %s bands: %s" % (label, " ".join(names)))
    w10, w20, w60 = read_windows(xmin, ymin, xmax, ymax)
    data10 = ds.read(0, w10, i10) if i10 else None
    data20 = ds.read(1, w20, i20) if i20 else None
    data60 = ds.read(2, w60, i60) if i60 else None
    if (run_60 or true_data) and data60 is None:
        raise SystemExit("the product has none of the 60 m bands B1 / B9 that --run_60 / --true_data need")
    return data10, data20, data60, (xmin, ymin, xmax, ymax)


def readS2fromFile(data_file, test_data=False, roi_x_y=None, save_prefix="../data/", write_images=False, run_60=False,
                   true_data=False):
    """``create_patches.py:19-316``.  ``data_file``: a SAFE directory (its ``MTD_MSIL1C.xml`` is opened through GDAL) or a
    ``.npz`` product container."""
    bands = read_bands(data_file, roi_x_y, run_60, true_data)
    if bands is None:
        return 0
    data10, data20, data60, roi = bands
    name = os.path.split(data_file.rstrip('/'))[1]           # :234-238
    write_patches(data10, data20, data60, name, roi, test_data, save_prefix, write_images, run_60, true_data)
    return 0


def build_parser():
    p = argparse.ArgumentParser(description="Read Sentinel-2 data and write training / test patches (B200 build).",
                                formatter_class=argparse.ArgumentDefaultsHelpFormatter)
    p.add_argument("data_file", help="A Sentinel-2 SAFE directory (read through GDAL) or a .npz product container.")
    p.add_argument("--roi_x_y", default="", help="Region of interest as pixel locations on the 10m bands: x_1,y_1,x_2,y_2.")
    p.add_argument("--test_data", default=False, action="store_true", help="Store test patches in a separate dir.")
    p.add_argument("--write_images", default=False, action="store_true", help="Write quick-look PNG images of the degraded bands.")
    p.add_argument("--save_prefix", default="../data/", help="Prefix for all output files (use a trailing /).")
    p.add_argument("--run_60", default=False, action="store_true", help="Create patches also from the 60m channels.")
    p.add_argument("--true_data", default=False, action="store_true", help="Create patches for S2 without ground truth.")
    return p


def main(argv=None):
    args = build_parser().parse_args(argv)
    print('I will proceed with file {}'.format(args.data_file))
    return readS2fromFile(args.data_file, args.test_data, args.roi_x_y, args.save_prefix, args.write_images, args.run_60,
                          args.true_data)


if __name__ == '__main__':
    raise SystemExit(main())
