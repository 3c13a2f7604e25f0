"""Mirror of the reference's user-facing tile driver ``testing/s2_tiles_supres.py``: read the 10 / 20 / 60 m bands of a
Sentinel-2 product, super-resolve the 60 m bands (``DSen2_60``) and the 20 m bands (``DSen2_20``) to 10 m, write them out.

The reference is a flat script bound to GDAL for reading (JP2 sub-datasets) and writing (GeoTIFF / ENVI / npz).  GDAL is not
part of this image, so the script is split here into

* the GDAL-free core -- region-of-interest arithmetic (``:127-140,165-173``), pixel <-> projected coordinate inversion
  (``:150-158``), UTM-zone choice (``:174-193``), band selection (``:236-303``), the read windows per resolution
  (``:311-329``), the 60 m -> 20 m chaining (``:332-342,385-390``), band ordering / naming of the output (``:367-416``),
  the geotransform shift (``:397-400``) and the npz writer (``:419-420``) -- as functions, tested on synthetic arrays;
* two sources / sinks behind one small interface: ``GdalSource`` (used when ``osgeo`` is importable; same calls as the
  reference) and ``NpzSource`` (a ``.npz`` container of the three band stacks + descriptions + geotransform, which is also
  what ``--output_file_format npz`` style post-processing chains and the tests use).

    python -m dsen2_b200.s2_tiles_supres <data_file> [output_file] [--roi_x_y x1,y1,x2,y2] [--run_60]
                                         [--copy_original_bands] [--output_file_format npz|GTiff|ENVI ...]
                                         [--nodata VALUE] [--output_dtype float64|uint16] [--add_offset VALUE]

``--nodata`` is an extension of the reference's options: pixels whose every input band holds VALUE (0 outside the footprint
of a partly covered granule) stay VALUE in the output, which records VALUE as its nodata value.  ``--output_dtype uint16``
(another extension) writes the super-resolved bands as uint16 digital numbers, the input's own format, rounded and saturated
on the GPU (``supres.DSen2_20(out_dtype=)``); VALUE must then be a uint16 value.  The default ``float64`` is the reference's
output.  ``--add_offset VALUE`` (an extension) is the radiometric offset of the product, as its metadata states it
(RADIO_ADD_OFFSET / BOA_ADD_OFFSET: -1000 for processing baseline 04.00 and later): it is added to the inputs before the
network and subtracted from its output on the GPU (``supres.DSen2_20(add_offset=)``), so the super-resolved bands are in the
product's own convention, like the bands ``--copy_original_bands`` copies.  ``--nodata`` stays the value the product stores.
"""
import argparse
import math
import os
import re
import sys
from collections import defaultdict

import numpy as np

BANDS_20 = 'B2,B3,B4,B5,B6,B7,B8,B8A,B11,B12'                       # s2_tiles_supres.py:86-89
BANDS_60 = 'B1,B2,B3,B4,B5,B6,B7,B8,B8A,B9,B11,B12'


# ---------------------------------------------------------------------------------------------- #
# region of interest (s2_tiles_supres.py:127-140, 165-173)
# ---------------------------------------------------------------------------------------------- #
def clamp_roi(x1, y1, x2, y2, xsize, ysize):
    """Two corner points (any order, 10 m pixel units) -> (xmin, ymin, xmax, ymax) inside the raster, enlarged / shrunk to
    60 m pixel boundaries (multiples of 6) exactly as the reference does: min down, max+1 down."""
    xmin = max(min(x1, x2, xsize - 1), 0)
    xmax = min(max(x1, x2, 0), xsize - 1)
    ymin = max(min(y1, y2, ysize - 1), 0)
    ymax = min(max(y1, y2, 0), ysize - 1)
    xmin = int(xmin / 6) * 6
    xmax = int((xmax + 1) / 6) * 6 - 1
    ymin = int(ymin / 6) * 6
    ymax = int((ymax + 1) / 6) * 6 - 1
    return xmin, ymin, xmax, ymax


def full_roi(xsize, ysize):
    """No ROI given: the whole raster, NOT rounded (s2_tiles_supres.py:136-140)."""
    return 0, 0, xsize - 1, ysize - 1


def projected_to_pixel(geotransform, xp, yp):
    """Projected coordinates -> integer pixel position by inverting the affine geotransform (``to_xy``, :150-158)."""
    xoff, a, b, yoff, d, e = geotransform
    xp -= xoff
    yp -= yoff
    det_inv = 1. / (a * e - d * b)
    x = (e * xp - b * yp) * det_inv
    y = (-d * xp + a * yp) * det_inv
    return int(x), int(y)


def choose_utm(candidates, select_utm=''):
    """``candidates``: [(description, (xmin, ymin, xmax, ymax))] for the 10 m (or unknown-resolution) sub-datasets in
    listing order.  Returns (index, utm string, roi, {utm: area}) -- the selected zone if named, else the one with the
    largest ROI coverage (:174-193)."""
    all_utms = defaultdict(int)
    best = (0, select_utm, (0, 0, 0, 0))
    largest_area = -1
    for idx, (desc, roi) in enumerate(candidates):
        xmin, ymin, xmax, ymax = roi
        area = (xmax - xmin + 1) * (ymax - ymin + 1)
        current = desc[desc.find("UTM"):]
        if area > all_utms[current]:
            all_utms[current] = area
        if current == select_utm:
            best = (idx, current, roi)
            break
        if area > largest_area:
            largest_area = area
            best = (idx, current, roi)
    return best[0], best[1], best[2], dict(all_utms)


# ---------------------------------------------------------------------------------------------- #
# band selection (s2_tiles_supres.py:221-303)
# ---------------------------------------------------------------------------------------------- #
def validate_description(description, output_file_format='GTiff'):
    m = re.match(r"(.*?), central wavelength (\d+) nm", description)
    if m:
        return m.group(1) + " (" + m.group(2) + " nm)"
    if output_file_format == 'ENVI' and ',' in description:      # ENVI band names must not contain commas
        pos = description.find(',')
        return description[:pos] + description[(pos + 1):]
    return description


def get_band_short_name(description):
    if ',' in description:
        return description[:description.find(',')]
    if ' ' in description:
        return description[:description.find(' ')]
    return description[:3]


def select_bands(desc10, desc20, desc60, run_60, output_file_format='GTiff'):
    """Band descriptions of the three sub-datasets -> per resolution (short names, indices) of the bands to load, and the
    validated description of every selected band.  A band is taken from the FIRST resolution that lists it (:270-303)."""
    wanted = (BANDS_60 if run_60 else BANDS_20).split(',')
    out, descriptions = [], {}
    for descs in (desc10, desc20, desc60):
        names, indices = [], []
        for b, raw in enumerate(descs):
            desc = validate_description(raw, output_file_format)
            short = get_band_short_name(desc)
            if short in wanted:
                wanted.remove(short)
                names.append(short)
                indices.append(b)
                descriptions[short] = desc
        out.append((names, indices))
    return out[0], out[1], out[2], descriptions


def read_windows(xmin, ymin, xmax, ymax):
    """(xoff, yoff, xsize, ysize) of the ROI at 10 / 20 / 60 m (:311-329; integer division like the reference)."""
    w, h = xmax - xmin + 1, ymax - ymin + 1
    return ((xmin, ymin, w, h), (xmin // 2, ymin // 2, w // 2, h // 2), (xmin // 6, ymin // 6, w // 6, h // 6))


# ---------------------------------------------------------------------------------------------- #
# super-resolution chaining and output assembly (s2_tiles_supres.py:332-342, 385-416)
# ---------------------------------------------------------------------------------------------- #
def super_resolve(data10, data20, data60, names10, names20, names60, deep=False, models=None, nodata=None,
                  out_dtype=None, add_offset=None):
    """The 60 m bands first, then the 20 m bands; returns (sr (H, W, n20 [+ n60]) or None, short names of its bands).
    ``models`` (extension): {'20': S2Model, '60': S2Model} instead of the shipped weight files; ``nodata`` (extension):
    the nodata value of both calls (``supres.DSen2_20``); ``out_dtype`` (extension): their output type (float32 if None,
    or np.uint16); ``add_offset`` (extension): the product's radiometric offset, for both calls."""
    from . import supres
    models = models or {}
    extra = {} if nodata is None else {'nodata': nodata}
    if out_dtype is not None:
        extra['out_dtype'] = out_dtype
    if add_offset is not None:
        extra['add_offset'] = add_offset
    sr60 = None
    if names60 and names20 and names10:
        print("Super-resolving the 60m data into 10m bands")
        sr60 = supres.DSen2_60(data10, data20, data60, deep=deep, model=models.get('60'), **extra)
    sr20 = None
    if names10 and names20:
        print("Super-resolving the 20m data into 10m bands")
        sr20 = supres.DSen2_20(data10, data20, deep=deep, model=models.get('20'), **extra)
    if sr20 is None:
        return None, []
    if sr60 is not None:
        return np.concatenate((sr20, sr60), axis=2), list(names20) + list(names60)
    return sr20, list(names20)


def assemble_output(data10, names10, sr, sr_names, descriptions, copy_original_bands):
    """Ordered [(description, (H, W) array)]: optionally the original 10 m bands, then "SR" + description of every
    super-resolved band (:405-413)."""
    out = []
    if copy_original_bands:
        for bi, bn in enumerate(names10):
            out.append((descriptions[bn], data10[:, :, bi]))
    for bi, bn in enumerate(sr_names):
        out.append(("SR" + descriptions[bn], sr[:, :, bi]))
    return out


def shift_geotransform(geotransform, xmin, ymin):
    """Upper-left corner of the ROI in projected metres: 10 m pixels (:397-400)."""
    geot = list(geotransform)
    geot[0] += xmin * 10
    geot[3] -= ymin * 10
    return tuple(geot)


def save_npz(output_file, bands, nodata=None, add_offset=None):
    """``np.savez(output_file, bands=bands)`` with bands = {description: array} (:419-420); with ``nodata`` / ``add_offset``
    also a ``nodata`` / ``add_offset`` entry holding the value."""
    extra = {name: np.float64(v) for name, v in (('nodata', nodata), ('add_offset', add_offset)) if v is not None}
    np.savez(output_file, bands=dict(bands), **extra)


# ---------------------------------------------------------------------------------------------- #
# sources
# ---------------------------------------------------------------------------------------------- #
class NpzSource:
    """A product held in one ``.npz``: ``data10 (H,W,C10)``, ``data20 (H/2,W/2,C20)``, ``data60 (H/6,W/6,C60)``,
    ``desc10 / desc20 / desc60`` (band descriptions as GDAL reports them), optional ``geotransform`` (6 numbers),
    ``projection`` (WKT string) and ``utm`` (description suffix)."""

    def __init__(self, path):
        z = np.load(path, allow_pickle=False)
        self.data = [z['data10'], z['data20'], z['data60']]
        self.desc = [[str(s) for s in z['desc%d' % r]] for r in (10, 20, 60)]
        self.geotransform = tuple(float(v) for v in z['geotransform']) if 'geotransform' in z.files else (0., 10., 0., 0., 0., -10.)
        self.projection = str(z['projection']) if 'projection' in z.files else ''
        self.utm = str(z['utm']) if 'utm' in z.files else 'UTM 32N'

    def candidates(self):
        h, w = self.data[0].shape[:2]
        return [("10m resolution, " + self.utm, (w, h))]

    def open(self, idx):
        return self

    def descriptions(self, res):
        return self.desc[res]

    def read(self, res, window, indices):
        xoff, yoff, xs, ys = window
        return np.ascontiguousarray(self.data[res][yoff:yoff + ys, xoff:xoff + xs][:, :, indices])


class GdalSource:  # pragma: no cover - needs osgeo, which is not in this image
    """The reference's reading calls (:97-118, 200-219, 311-329) behind the same interface."""

    def __init__(self, path):
        from osgeo import gdal
        self.gdal = gdal
        raster = gdal.Open(path)
        self.sets = {10: [], 20: [], 60: [], 0: []}
        for dsname, dsdesc in raster.GetSubDatasets():
            key = 10 if '10m resolution' in dsdesc else 20 if '20m resolution' in dsdesc else 60 if '60m resolution' in dsdesc else 0
            self.sets[key].append((dsname, dsdesc))
        self.ds = None

    def candidates(self):
        out = []
        for dsname, dsdesc in self.sets[10] + self.sets[0]:
            ds = self.gdal.Open(dsname)
            out.append((dsdesc, (ds.RasterXSize, ds.RasterYSize)))
        return out

    def open(self, idx, utm=''):
        pick10 = self.sets[0][0] if not self.sets[10] else self.sets[10][idx]
        pick = lambda sets: next((s for s in sets if utm and utm in s[1]), sets[idx])
        self.ds = [self.gdal.Open(pick10[0]), self.gdal.Open(pick(self.sets[20])[0]), self.gdal.Open(pick(self.sets[60])[0])]
        self.geotransform = self.ds[0].GetGeoTransform()
        self.projection = self.ds[0].GetProjection()
        return self

    def descriptions(self, res):
        ds = self.ds[res]
        return [ds.GetRasterBand(b + 1).GetDescription() for b in range(ds.RasterCount)]

    def read(self, res, window, indices):
        xoff, yoff, xs, ys = window
        arr = self.ds[res].ReadAsArray(xoff=xoff, yoff=yoff, xsize=xs, ysize=ys, buf_xsize=xs, buf_ysize=ys)
        return np.rollaxis(arr, 0, 3)[:, :, indices]


def open_source(path):
    if path.endswith('.npz'):
        return NpzSource(path)
    try:
        import osgeo  # noqa: F401
    except ImportError:
        raise SystemExit("reading %s needs GDAL (osgeo), which is not installed; a .npz product container "
                         "(see dsen2_b200.s2_tiles_supres.NpzSource) works without it" % path)
    return GdalSource(path)


def output_file_formats():
    """``--list_output_file_formats`` (:64-78): the raster drivers GDAL can create files with, as "name: long name (ext)";
    ``npz`` is always there (the reference falls back to it when the driver is missing, :409-411)."""
    lines = ["npz: compressed python/numpy file, one array per band (npz)"]
    try:
        from osgeo import gdal
    except ImportError:
        return lines
    for didx in range(gdal.GetDriverCount()):  # pragma: no cover - needs osgeo, which is not in this image
        driver = gdal.GetDriver(didx)
        metadata = driver.GetMetadata() if driver else {}
        if metadata.get(gdal.DCAP_CREATE) == 'YES' and metadata.get(gdal.DCAP_RASTER) == 'YES':
            name = driver.GetDescription()
            if "DMD_LONGNAME" in metadata:
                name += ": " + metadata["DMD_LONGNAME"]
            if "DMD_EXTENSIONS" in metadata:
                name += " (" + metadata["DMD_EXTENSIONS"] + ")"
            lines.append(name)
    return lines


# ---------------------------------------------------------------------------------------------- #
# command line (same options as the reference, :14-64)
# ---------------------------------------------------------------------------------------------- #
def build_parser():
    p = argparse.ArgumentParser(description="Perform super-resolution on Sentinel-2 with DSen2 (B200 build).",
                                formatter_class=argparse.ArgumentDefaultsHelpFormatter)
    p.add_argument("data_file", help="An input Sentinel-2 data file (ZIP / SAFE .xml through GDAL, or a .npz product container).")
    p.add_argument("output_file", nargs="?", help="A target data file.")
    p.add_argument("--roi_lon_lat", default="", help="Region of interest, WGS84: lon_1,lat_1,lon_2,lat_2 (needs GDAL/osr).")
    p.add_argument("--roi_x_y", default="", help="Region of interest as pixel locations on the 10m bands: x_1,y_1,x_2,y_2.")
    p.add_argument("--list_bands", action="store_true", help="List bands in the input file and exit.")
    p.add_argument("--run_60", action="store_true", help="Also super-resolve the 60m bands (B1, B9).")
    p.add_argument("--list_UTM", action="store_true", help="List all UTM zones present in the input file.")
    p.add_argument("--select_UTM", default="", help="Select a UTM zone (default: largest ROI coverage).")
    p.add_argument("--list_output_file_formats", action="store_true",
                   help="List the raster output file formats GDAL can create (and npz) and exit.")
    p.add_argument("--output_file_format", default="GTiff", help="GDAL driver name, or npz.")
    p.add_argument("--copy_original_bands", action="store_true", help="Also copy the original 10m bands into the output.")
    p.add_argument("--save_prefix", default="", help="Prefix for all output files.")
    p.add_argument("--nodata", type=float, default=None,
                   help="Extension: input value of pixels without data (e.g. 0).  Pixels whose every band holds it stay "
                        "nodata in the output, which records the value; empty patches are not computed.")
    p.add_argument("--output_dtype", choices=("float64", "uint16"), default="float64",
                   help="Extension: data type of the written bands.  uint16: digital numbers like the input, rounded and "
                        "clipped to [0, 65535] on the GPU; a computed value equal to --nodata is moved one step off it.")
    p.add_argument("--add_offset", type=float, default=None, metavar="VALUE",
                   help="Extension: radiometric offset of the product, as RADIO_ADD_OFFSET (L1C) / BOA_ADD_OFFSET (L2A) in "
                        "its metadata.  Products of processing baseline 04.00 and later (from 25 January 2022, and the "
                        "reprocessed archive) want --add_offset -1000.  It is added to the inputs before the network and "
                        "subtracted from the output on the GPU; the output stays in the product's convention.")
    return p


def parse_args(argv=None):
    parser = build_parser()
    args = parser.parse_args(argv)
    if args.output_dtype == "uint16" and args.nodata is not None and \
            not (args.nodata.is_integer() and 0 <= args.nodata <= 65535):
        parser.error("--nodata %r is not a uint16 value (an integer in [0, 65535]), as --output_dtype uint16 needs"
                     % args.nodata)
    if args.add_offset is not None and not math.isfinite(args.add_offset):
        parser.error("--add_offset %r is not a finite number" % args.add_offset)
    return args


def main(argv=None, models=None):
    args = parse_args(argv)
    if args.list_output_file_formats:                # before the input is opened, as in the reference (:64-79)
        for line in output_file_formats():
            print(line)
        return 0
    src = open_source(args.data_file)
    if args.roi_lon_lat and not isinstance(src, GdalSource):
        raise SystemExit("--roi_lon_lat needs GDAL/osr for the coordinate transformation; use --roi_x_y")
    cands = []
    for desc, (xs, ys) in src.candidates():
        if args.roi_x_y:
            x1, y1, x2, y2 = [float(x) for x in re.split(',', args.roi_x_y)]
            roi = clamp_roi(x1, y1, x2, y2, xs, ys)
        else:
            roi = full_roi(xs, ys)
        cands.append((desc, roi))
    utm_idx, utm, (xmin, ymin, xmax, ymax), all_utms = choose_utm(cands, args.select_UTM)
    if args.list_UTM:
        print("List of UTM zones (with ROI coverage in pixels):")
        for u in all_utms:
            print("%s (%d)" % (u, all_utms[u]))
        return 0
    print("Selected UTM Zone:", utm)
    print("Selected pixel region: xmin=%d, ymin=%d, xmax=%d, ymax=%d:" % (xmin, ymin, xmax, ymax))
    print("Image size: width=%d x height=%d" % (xmax - xmin + 1, ymax - ymin + 1))
    if xmax < xmin or ymax < ymin:
        print("Invalid region of interest / UTM Zone combination")
        return 0
    ds = src.open(utm_idx)
    fmt = args.output_file_format
    (n10, i10), (n20, i20), (n60, i60), descriptions = select_bands(ds.descriptions(0), ds.descriptions(1), ds.descriptions(2),
                                                                    args.run_60, fmt)
    for label, names in (("10m", n10), ("20m", n20), ("60m", n60)):
        print("Selected %s bands: %s" % (label, " ".join(names)))
    if args.list_bands:
        return 0
    output_file = args.output_file
    if not output_file:
        print("Error: you must provide the name of an output file. I will set it identical to the input...")
        output_file = os.path.split(args.data_file)[1] + '.tif'
    output_file = args.save_prefix + output_file
    if fmt == 'ENVI' and output_file[-4:].lower() == '.hdr':
        output_file = output_file[:-4] + '.bin'
    w10, w20, w60 = read_windows(xmin, ymin, xmax, ymax)
    data10 = ds.read(0, w10, i10) if i10 else None
    data20 = ds.read(1, w20, i20) if i20 else None
    data60 = ds.read(2, w60, i60) if i60 else None
    u16 = args.output_dtype == "uint16"
    sr, sr_names = super_resolve(data10, data20, data60, n10, n20, n60, models=models, nodata=args.nodata,
                                 out_dtype=np.uint16 if u16 else None, add_offset=args.add_offset)
    if sr is None:
        print("No super-resolution performed, exiting")
        return 0
    bands = assemble_output(data10, n10, sr, sr_names, descriptions, args.copy_original_bands)
    driver = None
    if fmt != "npz":
        try:
            from osgeo import gdal
            driver = gdal.GetDriverByName(fmt)
            md = driver.GetMetadata() if driver else {}
            if not (driver and md.get(gdal.DCAP_CREATE) == 'YES'):
                driver = None
        except ImportError:
            driver = None
        if driver is None:
            print("Gdal doesn't support creating %s files" % fmt)
            print("Writing to npz as a fallback")
            fmt = "npz"
    print("Writing%s the super-resolved bands in %s" % (" the original 10m bands and" if args.copy_original_bands else "",
                                                          output_file))
    geot = shift_geotransform(ds.geotransform, xmin, ymin)
    if fmt == "npz":
        save_npz(output_file, bands, args.nodata, args.add_offset)
    else:  # pragma: no cover - needs osgeo
        from osgeo import gdal
        result = driver.Create(output_file, data10.shape[1], data10.shape[0], len(bands),
                               gdal.GDT_UInt16 if u16 else gdal.GDT_Float64)
        result.SetGeoTransform(geot)
        result.SetProjection(ds.projection)
        for bidx, (desc, data) in enumerate(bands):
            result.GetRasterBand(bidx + 1).SetDescription(desc)
            result.GetRasterBand(bidx + 1).WriteArray(data)
            if args.nodata is not None:
                result.GetRasterBand(bidx + 1).SetNoDataValue(args.nodata)
    for desc, _ in bands:
        print(desc)
    return 0


if __name__ == '__main__':
    sys.exit(main())
