"""Host-side mirror of the reference ``testing/supres.py``: ``DSen2_20`` / ``DSen2_60``.

Same signatures, ``SCALE`` / ``MDL_PATH`` module constants and weight-file naming (supres.py:11-12,57,60).
The whole tile stays on the GPU between the upload of the inputs and the download of the stitched
image.  Per patch batch: one input-preparation kernel (extract + bilinear + /2000 fused, straight from the images),
then the 14 (DSen2, 6 x 128) or 66 (VDSen2, 32 x 256) tcgen05 convolutions, the last one writing the stitched
x2000 canvas.

Nodata (an extension): with ``nodata=v``, an output pixel whose every input band (10 m, 20 m[, 60 m]) equals v is nodata
and comes out as v; only the patches that own a pixel with data run the network.  Every other pixel is bit-identical to
the output without ``nodata``.

Digital-number output (an extension): with ``out_dtype=uint16`` the last layer rounds and saturates its values on the
device and writes a uint16 canvas: NaN becomes 0, every other value is rint(clip(f, 0, 65535)) (half to even) of the float f
the float32 output holds.  With ``nodata=v`` as well, nodata pixels are v, and a valid value that would round to v is
written as v + 1 (65534 for v = 65535), so no computed value reads as nodata.

Radiometric offset (an extension): in Sentinel-2 products of processing baseline 04.00 and later, reflectance is
(DN + add_offset) / 10000, with the add_offset of their metadata (RADIO_ADD_OFFSET / BOA_ADD_OFFSET, -1000); the network
expects DN = 10000 x reflectance.  With ``add_offset=a`` every band value x of the input images, as held on the device
(uint16, or float32 as staged), becomes fl32(x + a) before the preparation, and every output value f becomes fl32(f - a):
the output is in the product's own convention (quantised after that for uint16 output).  Nodata is still decided on the
stored values, and nodata pixels are written as the stored v.

Chip stacks (an extension): 4-D inputs (N, H, W, 4), (N, H/2, W/2, 6)[, (N, H/6, W/6, 2)] are N same-size scenes, the
datasets of machine learning (BigEarthNet 120 x 120, SEN12MS 256 x 256).  The output is (N, H, W, Cout), and chip i of it
is bit for bit what the 3-D call on chip i returns, for every ``out_dtype`` / ``add_offset``; but every device launch
runs the patches of many chips.  Patches are numbered over the stack, chip * ppc + patch with ppc the filled patches of
one chip, and a launch may straddle chips.  All float32 or all uint16; ``nodata`` is not supported with stacks.
"""

import math
import os

import numpy as np

from . import _capi, sharding
from .DSen2Net import S2Model, s2model
from .patches import bilinear_up_device, extract_patches_device, patch_counts, recompose_device

SCALE = 2000
MDL_PATH = '../models/'

_GEOM = {False: dict(patch=128, border=8, ratio=2), True: dict(patch=192, border=12, ratio=6)}
_model_cache = {}


def weight_file(deep=False, run_60=False):
    """File-name convention of supres.py:57,60."""
    if deep:
        return MDL_PATH + ('s2_034_lr_1e-04.hdf5' if run_60 else 's2_033_lr_1e-04.hdf5')
    return MDL_PATH + ('s2_030_lr_1e-05.hdf5' if run_60 else 's2_032_lr_1e-04.hdf5')


def _load_model(input_shape, deep, run_60):
    path = weight_file(deep, run_60)
    st = os.stat(path)                      # FileNotFoundError (OSError) when the weights are missing, as h5py
    key = (os.path.abspath(path), st.st_mtime_ns, st.st_size)
    if key not in _model_cache:
        model = s2model(input_shape, num_layers=32, feature_size=256) if deep else \
            s2model(input_shape, num_layers=6, feature_size=128)
        print('Symbolic Model Created.')
        model.load_weights(path)
        _model_cache[key] = model
    print("Predicting using file: {}".format(path))
    return _model_cache[key]


def default_device_batch(W, P, B):
    """Patches per launch: whole patch rows of the tile when a row is a reasonable batch (a full Sentinel-2 tile has 99
    patches of 128 per row), so that the chunks of ``HostPipeline`` (whole rows) split into equal batches; about 4.9 M
    patch pixels otherwise.  Larger batches only amortise launch overhead and the last wave of each launch: measured on
    one box 559-561 ms per tile with 99 patches per launch, 553-555 ms with 198 or 297."""
    nx = -(-W // (P - 2 * B))
    target = max(1, (300 * 128 * 128) // (P * P))
    if nx > 2 * target:
        return target
    return nx * max(1, target // nx)


def check_nodata(nodata, model, uint16_images):
    """The ``nodata`` argument as the float the kernels compare with (None stays None).  Rejected, not clamped: NaN, a
    value that is not an integer in [0, 65535] for uint16 images, a network without resBlocks (``model`` None: no
    network involved)."""
    if nodata is None:
        return None
    v = float(nodata)
    if math.isnan(v):
        raise ValueError("nodata must not be NaN")
    if uint16_images and not (v.is_integer() and 0 <= v <= 65535):
        raise ValueError("nodata %r is not a uint16 value (an integer in [0, 65535])" % (nodata,))
    if model is not None and not model.xin16:
        raise ValueError("nodata needs a network with resBlocks (num_layers > 0)")
    return v


def check_add_offset(add_offset, model):
    """The ``add_offset`` argument as the float32 value the kernels use, as a Python float (None stays None).  Rejected with
    ``ValueError``: anything but a real number, a value that is not finite in float32, and a network without resBlocks (its
    separate extract / network / recompose kernels take no offset; ``model`` None: not checked)."""
    if add_offset is None:
        return None
    a = np.asarray(add_offset)
    if a.ndim != 0 or a.dtype.kind not in 'iuf':
        raise ValueError("add_offset must be a number, got %r" % (add_offset,))
    with np.errstate(over='ignore'):
        v = np.float32(a)
    if not np.isfinite(v):
        raise ValueError("add_offset %r is not a finite float32 value" % (add_offset,))
    if model is not None and not model.xin16:
        raise ValueError("add_offset needs a network with resBlocks (num_layers > 0)")
    return float(v)


_OUT_DTYPES = {'float32': False, 'uint16': True}


def check_out_dtype(out_dtype, model):
    """True when ``out_dtype`` (a numpy or torch dtype; None = float32) asks for uint16 digital numbers, False for float32.
    Rejected with ``ValueError``: any other type, and uint16 with a network without resBlocks (it runs the separate
    extract / network / recompose kernels, which write float32; ``model`` None: not checked)."""
    if out_dtype is None:
        return False
    name = str(out_dtype)
    if name.startswith('torch.'):
        name = name[len('torch.'):]
    else:
        try:
            name = np.dtype(out_dtype).name
        except TypeError:
            name = None
    if name not in _OUT_DTYPES:
        raise ValueError("out_dtype must be float32 or uint16, got %r" % (out_dtype,))
    u16 = _OUT_DTYPES[name]
    if u16 and model is not None and not model.xin16:
        raise ValueError("uint16 output needs a network with resBlocks (num_layers > 0)")
    return u16


def _check_out(out, shape, dtype, what):
    if out is not None and (out.dtype != dtype or tuple(out.shape) != tuple(shape)):
        raise ValueError("%s must be %s of shape %s, got %s of shape %s"
                         % (what, dtype, tuple(shape), out.dtype, tuple(out.shape)))


def _zeros_canvas(torch, shape, u16, device):
    """Zero-filled device canvas: float32, or uint16 (zeroed through an int16 view: no CUDA fill of uint16 is needed)."""
    if not u16:
        return torch.zeros(shape, dtype=torch.float32, device=device)
    out = torch.empty(shape, dtype=torch.uint16, device=device)
    out.view(torch.int16).zero_()
    return out


def _nodata_args(d10, d20, d60, nodata):
    torch = _capi.require_cuda()
    g = _GEOM[d60 is not None]
    H, W = int(d10.shape[0]), int(d10.shape[1])
    img_dtype = _capi.IMG_U16 if d10.dtype == torch.uint16 else _capi.IMG_F32
    ptr = _capi.ptr
    return (ptr(d10), ptr(d20), ptr(d60), img_dtype, H, W, g['patch'], g['border']), float(nodata)


def _scan_active(d10, d20, d60, first_patch, num_patches, nodata, ids, count, count_host, timers=None):
    """Enqueue ``dsen2_nodata_patches`` for the range on the current stream (active ids -> ``ids``, their number ->
    ``count``) and the copy of the count into the pinned ``count_host``; returns the event that follows the copy."""
    torch = _capi.require_cuda()
    imgs, v = _nodata_args(d10, d20, d60, nodata)
    S2Model._timed(timers, 'nodata_patches', num_patches, lambda: _capi.check(_capi.lib().dsen2_nodata_patches(
        *imgs, first_patch, num_patches, v, _capi.ptr(ids), _capi.ptr(count), _capi.stream_ptr()), "dsen2_nodata_patches"))
    count_host.copy_(count, non_blocking=True)
    ev = torch.cuda.Event()
    ev.record()
    return ev


def _run_active(model, d10, d20, d60, first_patch, num_patches, nodata, ids, out, device_batch, timers=None,
                add_offset=None):
    """The network over the active patches ``ids`` (batches of at most ``device_batch``), then nodata into the nodata
    pixels the range owns -- after the last layer, which also stitches active patches' values over their nodata pixels.
    A uint16 ``out`` gets network values moved off v (``avoid``) and the uint16 fill.  The fill writes v as it is: the
    offset applies to network values only."""
    torch = _capi.require_cuda()
    g = _GEOM[d60 is not None]
    u16 = out.dtype == torch.uint16
    avoid = int(nodata) if u16 else None
    for i in range(0, int(ids.shape[0]), device_batch):
        batch = ids[i:i + device_batch]
        model.forward_images(d10, d20, d60, g['patch'], g['border'], 0, int(batch.shape[0]), out, float(SCALE),
                             timers=timers, patch_ids=batch, avoid=avoid, add_offset=add_offset)
    imgs, v = _nodata_args(d10, d20, d60, nodata)
    name = 'dsen2_nodata_fill_u16' if u16 else 'dsen2_nodata_fill'
    fill = getattr(_capi.lib(), name)
    S2Model._timed(timers, 'nodata_fill', num_patches, lambda: _capi.check(fill(
        *imgs, first_patch, num_patches, v, model.out_channels, _capi.ptr(out), _capi.stream_ptr()), name))


def _active(d10, d20, d60, first_patch, num_patches, nodata, timers=None):
    """Active patch ids of the range: a CUDA int32 tensor, after one device -> host read of their number."""
    torch = _capi.require_cuda()
    ids = torch.empty((max(1, num_patches),), dtype=torch.int32, device=d10.device)
    count = torch.empty((1,), dtype=torch.int32, device=d10.device)
    count_host = torch.empty((1,), dtype=torch.int32).pin_memory()
    _scan_active(d10, d20, d60, first_patch, num_patches, nodata, ids, count, count_host, timers).synchronize()
    return ids[:int(count_host[0])]


def _filled_range(d10, run_60, first_patch, num_patches):
    g = _GEOM[run_60]
    r, P, B = g['ratio'], g['patch'], g['border']
    H, W = int(d10.shape[0]), int(d10.shape[1])
    if H % r or W % r:
        raise ValueError("10 m image size %dx%d must be a multiple of %d" % (H, W, r))
    _, filled = patch_counts(H // r, W // r, P // r, B // r)
    if num_patches is None:
        num_patches = filled - first_patch
    if first_patch < 0 or first_patch + num_patches > filled:
        raise ValueError("patch range [%d, %d) outside the %d patches of this tile"
                         % (first_patch, first_patch + num_patches, filled))
    return num_patches


def active_patches(d10, d20, d60=None, nodata=0, first_patch=0, num_patches=None):
    """Ascending indices (CUDA int32 tensor) of the patches of [first_patch, first_patch+num_patches) that own a pixel
    with data: the patches ``super_resolve_device(..., nodata=nodata)`` runs through the network."""
    torch = _capi.require_cuda()
    nodata = check_nodata(nodata, None, d10.dtype == torch.uint16)
    num_patches = _filled_range(d10, d60 is not None, first_patch, num_patches)
    return _active(d10, d20, d60, first_patch, num_patches, nodata)


def _stack_geometry(model, shapes, dtypes, nodata):
    """(N, H, W, ppc) of a chip stack with images of ``shapes`` and element types ``dtypes`` (numpy names), ppc the filled
    patches of one chip.  Rejected with ``ValueError``: ``nodata``, a network without resBlocks, leading sizes that
    differ, shapes other than (N, H/d, W/d, C), mixed or other element types, and chips the 3-D path rejects: sizes that
    are not multiples of the ratio, chips smaller than one patch stride (112 px at 20 m, 168 px at 60 m)."""
    if nodata is not None:
        raise ValueError("nodata is not supported with chip stacks")
    if not model.xin16:
        raise ValueError("chip stacks need a network with resBlocks (num_layers > 0)")
    if len(set(dtypes)) != 1 or dtypes[0] not in ('float32', 'uint16'):
        raise ValueError("chip stack images must all be float32 or all be uint16, got %s" % (list(dtypes),))
    if any(len(sh) != 4 for sh in shapes) or len({int(sh[0]) for sh in shapes}) != 1:
        raise ValueError("chip stacks must be 4-D with the same number of chips, got shapes %s" % (list(shapes),))
    g = _GEOM[len(shapes) == 3]
    r, P, B = g['ratio'], g['patch'], g['border']
    N, H, W = (int(v) for v in shapes[0][:3])
    if H % r or W % r:
        raise ValueError("10 m chip size %dx%d must be a multiple of %d" % (H, W, r))
    for sh, div, c in zip(shapes, (1, 2, 6), model.in_channels):
        if tuple(int(v) for v in sh) != (N, H // div, W // div, c):
            raise ValueError("expected a chip stack of shape %s, got %s" % ((N, H // div, W // div, c), tuple(sh)))
    if min(H, W) < P - 2 * B:
        raise ValueError("chips of %dx%d are smaller than one patch stride (%d)" % (H, W, P - 2 * B))
    return N, H, W, patch_counts(H // r, W // r, P // r, B // r)[1]


def _super_resolve_chips(model, d10, d20, d60, first_patch, num_patches, out, device_batch, timers, nodata, out_dtype,
                         add_offset):
    import torch
    # rejected before the device is touched (add_offset: by the caller)
    u16 = check_out_dtype(out_dtype, model)
    imgs = [t for t in (d10, d20, d60) if t is not None]
    N, H, W, ppc = _stack_geometry(model, [tuple(t.shape) for t in imgs], [str(t.dtype)[len('torch.'):] for t in imgs],
                                   nodata)
    g = _GEOM[d60 is not None]
    shape = (N, H, W, model.out_channels)
    _check_out(out, shape, torch.uint16 if u16 else torch.float32, "out")
    if num_patches is None:
        num_patches = N * ppc - first_patch
    if first_patch < 0 or num_patches < 0 or first_patch + num_patches > N * ppc:
        raise ValueError("patch range [%d, %d) outside the %d patches of %d chips"
                         % (first_patch, first_patch + num_patches, N * ppc, N))
    _capi.require_cuda()
    if out is None:
        out = _zeros_canvas(torch, shape, u16, d10.device)
    if device_batch is None:
        device_batch = default_device_batch(W, g['patch'], g['border'])
    for p0 in range(first_patch, first_patch + num_patches, device_batch):
        nb = min(device_batch, first_patch + num_patches - p0)
        model.forward_images(d10, d20, d60, g['patch'], g['border'], p0, nb, out, float(SCALE), timers=timers,
                             add_offset=add_offset)
    return out


def super_resolve_device(model, d10, d20, d60=None, first_patch=0, num_patches=None, out=None, device_batch=None,
                         timers=None, nodata=None, out_dtype=None, add_offset=None):
    """Device-level pipeline.  d10/d20(/d60): CUDA HWC tensors, all float32 or all uint16.  Processes patches
    [first_patch, first_patch+num_patches) of the FILLED patch list (surplus zero patches of
    patches.py:32-39 are never read by recompose_images, so they are skipped) and writes the pixels those
    patches own into ``out`` (H, W, Cout) of ``out_dtype`` (torch.float32 when None, or torch.uint16: see the module
    docstring; allocated zero-filled if None).  ``nodata``: see the module docstring; the active patches are found on
    the device, and their number is the one value read back.  ``add_offset``: see the module docstring.

    Chip stacks (4-D images, module docstring): ``first_patch`` / ``num_patches`` index the flat patch list of the stack
    (chip * ppc + patch), ``out`` is (N, H, W, Cout), and a device batch may straddle chips."""
    add_offset = check_add_offset(add_offset, model)
    if d10.dim() == 4:
        return _super_resolve_chips(model, d10, d20, d60, first_patch, num_patches, out, device_batch, timers, nodata,
                                    out_dtype, add_offset)
    torch = _capi.require_cuda()
    u16 = check_out_dtype(out_dtype, model)
    nodata = check_nodata(nodata, model, d10.dtype == torch.uint16 or u16)
    run_60 = d60 is not None
    g = _GEOM[run_60]
    r, P, B = g['ratio'], g['patch'], g['border']
    H, W = int(d10.shape[0]), int(d10.shape[1])
    plr, blr = P // r, B // r
    shape = (H, W, model.out_channels)
    _check_out(out, shape, torch.uint16 if u16 else torch.float32, "out")
    num_patches = _filled_range(d10, run_60, first_patch, num_patches)
    if out is None:
        out = _zeros_canvas(torch, shape, u16, d10.device)
    if device_batch is None:
        device_batch = default_device_batch(W, P, B)
    # recompose_images' "lone patch is returned uncropped" branch (patches.py:375-376) keys on the ALLOCATED patch count
    # (k_i+1)(k_j+1), which is 1 only for images smaller than one stride -- inputs get_test_patches itself cannot tile
    # (and dsen2_prep16_from_images rejects); every image that reaches this point is stitched and cropped.
    if nodata is not None:
        ids = _active(d10, d20, d60, first_patch, num_patches, nodata, timers)
        _run_active(model, d10, d20, d60, first_patch, num_patches, nodata, ids, out, device_batch, timers, add_offset)
        return out
    for p0 in range(first_patch, first_patch + num_patches, device_batch):
        nb = min(device_batch, first_patch + num_patches - p0)
        if model.xin16:                          # fused: images -> x_in16 -> network -> stitched canvas
            model.forward_images(d10, d20, d60, P, B, p0, nb, out, float(SCALE), timers=timers, add_offset=add_offset)
            continue
        # a network without resblocks: separate extract / bilinear / network / stitch kernels
        if run_60:
            xs = [extract_patches_device(d10, 6, plr, blr, p0, nb, divisor=SCALE),
                  bilinear_up_device(extract_patches_device(d20, 3, plr, blr, p0, nb), 2, post_divisor=SCALE),
                  bilinear_up_device(extract_patches_device(d60, 1, plr, blr, p0, nb), 6, post_divisor=SCALE)]
        else:
            xs = [extract_patches_device(d10, 2, plr, blr, p0, nb, divisor=SCALE),
                  bilinear_up_device(extract_patches_device(d20, 1, plr, blr, p0, nb), 2, post_divisor=SCALE)]
        pred = model.forward_device(xs, timers=timers)
        recompose_device(pred, B, H, W, first_patch=p0, mul=float(SCALE), out=out)
    return out


def _np_dtype_of(torch, dt):
    return {torch.float32: np.float32, torch.uint16: np.uint16}[dt]


class _Slot:
    """One slot of the pinned staging ring: input rows of a chunk per resolution + the output rectangles it owns."""

    def __init__(self, torch, shapes_in, dtype, out_elems, out_dtype):
        self.inp = [torch.empty(s, dtype=dtype).pin_memory() for s in shapes_in]
        self.out = torch.empty((out_elems,), dtype=out_dtype).pin_memory()
        self.ev_h2d, self.ev_d2h = torch.cuda.Event(), torch.cuda.Event()
        self.used_in = self.used_out = False


def _staging_pool(torch, dev):
    """The worker threads that fill and drain the pinned staging slots (numpy releases the GIL for the copies)."""
    from concurrent.futures import ThreadPoolExecutor
    return ThreadPoolExecutor(max_workers=4, thread_name_prefix='dsen2-stage', initializer=torch.cuda.set_device,
                              initargs=(dev,))


class HostPipeline:
    """Host-buffer front end: tile inputs / output live in HOST memory; the patch range is cut into chunks of whole
    patch rows and chunk k+1's input rows upload while chunk k computes and chunk k-1's owned output rows download
    (three CUDA streams, one device-resident tile).  Reusable across calls of one shape.

    Host buffers may be pinned torch tensors (copied directly, fully asynchronous) or ordinary pageable numpy arrays
    -- what a caller of ``DSen2_20`` holds.  Pageable arrays go through a ring of pinned staging slots filled / drained
    by worker threads (numpy releases the GIL for the copies), so neither the page-locked upload nor the first-touch
    page faults of a freshly allocated output serialise with the GPU.  ``dtype``: element type of the device-resident
    images, float32 or uint16 (Sentinel-2 digital numbers as GDAL delivers them, s2_tiles_supres.py:311-315: half the
    bytes over PCIe; ``dsen2_prep16_from_images`` converts exactly, results are bit-identical).  ``out_dtype``: element
    type of the output canvas and of the host output, float32 (None) or uint16 (module docstring: half the bytes back)."""

    RING = 3

    def __init__(self, model, H, W, run_60=False, device=None, chunk_patch_rows=None, device_batch=None, dtype=None,
                 out_dtype=None):
        u16 = check_out_dtype(out_dtype, model)
        torch = _capi.require_cuda()
        self.torch, self.model, self.run_60 = torch, model, run_60
        self.H, self.W = int(H), int(W)
        g = _GEOM[run_60]
        self.r, self.P, self.B = g['ratio'], g['patch'], g['border']
        if self.H % self.r or self.W % self.r:
            raise ValueError("10 m image size %dx%d must be a multiple of %d" % (H, W, self.r))
        self.dev = torch.device('cuda', torch.cuda.current_device()) if device is None else device
        self.dtype = torch.float32 if dtype is None else dtype
        if self.dtype not in (torch.float32, torch.uint16):
            raise ValueError("device images are float32 or uint16")
        self.ny, self.nx, self.S = sharding.tile_grid(self.H, self.W, self.P, self.B)
        self.chunk_rows, self.device_batch = chunk_patch_rows, device_batch
        mk = lambda h, w, c: torch.empty((h, w, c), dtype=self.dtype, device=self.dev)
        self.d10, self.d20 = mk(self.H, self.W, 4), mk(self.H // 2, self.W // 2, 6)
        self.d60 = mk(self.H // 6, self.W // 6, 2) if run_60 else None
        self.out_dtype = torch.uint16 if u16 else torch.float32
        self.canvas = _zeros_canvas(torch, (self.H, self.W, model.out_channels), u16, self.dev)
        self.up, self.down = torch.cuda.Stream(self.dev), torch.cuda.Stream(self.dev)
        self.h2d_bytes = self.d2h_bytes = 0
        self._slots, self._pool = None, None

    # ---- pinned host buffers: direct asynchronous copies ------------------------------------------------------------
    def _upload(self, h, d, div, r0, r1, done):
        """rows [r0, r1) of the 10 m grid -> rows of the (H/div) grid not uploaded yet."""
        a, b = r0 // div, -(-r1 // div)
        if done is not None:
            a = max(a, done)
        if b > a:
            d[a:b].copy_(h[a:b], non_blocking=True)
            self.h2d_bytes += (b - a) * d.shape[1] * d.shape[2] * d.element_size()
        return b if done is None else max(done, b)

    def _nodata_buffers(self, nodata, first_patch, num_patches, chunks):
        """Device id list of the range, device and pinned per-chunk counts: chunk k scans into its own slice / entry, so
        the upload stream never overwrites what an earlier chunk's network still reads."""
        torch = self.torch
        nodata = check_nodata(nodata, self.model, self.dtype == torch.uint16 or self.out_dtype == torch.uint16)
        if nodata is None:
            return None, None, None, None
        ids = torch.empty((max(1, num_patches),), dtype=torch.int32, device=self.dev)
        count = torch.empty((chunks,), dtype=torch.int32, device=self.dev)
        return nodata, ids, count, torch.empty((chunks,), dtype=torch.int32).pin_memory()

    def _compute(self, k, p0, cnt, first_patch, nodata, ids, count_host, ev_scan, timers, add_offset):
        """Chunk k's network on the current stream (its inputs are resident): the whole range, or -- with ``nodata`` --
        the active patches its scan found, then the nodata fill."""
        if nodata is None:
            super_resolve_device(self.model, self.d10, self.d20, self.d60, first_patch=p0, num_patches=cnt,
                                 out=self.canvas, device_batch=self.device_batch, timers=timers, out_dtype=self.out_dtype,
                                 add_offset=add_offset)
            return
        ev_scan.synchronize()                        # this chunk's upload and scan only, never an earlier network
        batch = self.device_batch or default_device_batch(self.W, self.P, self.B)
        a = p0 - first_patch
        _run_active(self.model, self.d10, self.d20, self.d60, p0, cnt, nodata, ids[a:a + int(count_host[k])], self.canvas,
                    batch, timers, add_offset)

    def run(self, h10, h20, h60=None, hout=None, first_patch=0, num_patches=None, timers=None, nodata=None,
            add_offset=None):
        """Pinned torch tensors in (dtype = the pipeline's), pinned (H, W, Cout) tensor of ``out_dtype`` out.  Rows of
        ``hout`` that the patch range owns only partly (the seam rows of a sharded range) are downloaded whole.  ``nodata``: see the
        module docstring; each chunk's patch scan runs on the upload stream right behind its upload.  ``add_offset``: see
        the module docstring."""
        add_offset = check_add_offset(add_offset, self.model)
        torch = self.torch
        filled = self.ny * self.nx
        if num_patches is None:
            num_patches = filled - first_patch
        if hout is None:
            hout = torch.empty((self.H, self.W, self.model.out_channels), dtype=self.out_dtype).pin_memory()
        _check_out(hout, self.canvas.shape, self.out_dtype, "hout")
        for h in (h10, h20) + ((h60,) if self.run_60 else ()):
            if h.dtype != self.dtype:
                raise ValueError("host image dtype %s does not match the pipeline's %s" % (h.dtype, self.dtype))
        plan = self._plan(first_patch, num_patches)
        nodata, ids, count, count_host = self._nodata_buffers(nodata, first_patch, num_patches, len(plan))
        self.h2d_bytes = self.d2h_bytes = 0
        main = torch.cuda.current_stream(self.dev)
        self.up.wait_stream(main)
        self.down.wait_stream(main)
        done10 = done20 = done60 = None           # rows already resident on the device (per resolution)
        for k, (p0, cnt, (r0, r1), rects) in enumerate(plan):
            ev_scan = None
            with torch.cuda.stream(self.up):
                done10 = self._upload(h10, self.d10, 1, r0, r1, done10)
                done20 = self._upload(h20, self.d20, 2, r0, r1, done20)
                if self.run_60:
                    done60 = self._upload(h60, self.d60, 6, r0, r1, done60)
                if nodata is not None:
                    a = p0 - first_patch
                    ev_scan = _scan_active(self.d10, self.d20, self.d60, p0, cnt, nodata, ids[a:a + cnt],
                                           count[k:k + 1], count_host[k:k + 1], timers)
                ev_up = torch.cuda.Event()
                ev_up.record(self.up)
            main.wait_event(ev_up)
            self._compute(k, p0, cnt, first_patch, nodata, ids, count_host, ev_scan, timers, add_offset)
            ev_c = torch.cuda.Event()
            ev_c.record(main)
            self.down.wait_event(ev_c)
            with torch.cuda.stream(self.down):
                for (y0, y1, x0, x1) in rects:
                    # Whole rows, also where the range starts / ends inside a patch row and owns only part of them: a
                    # strided (partial-width) device -> host copy goes through temporaries and synchronises.  The pixels
                    # of those rows that another rank owns come along as they are on this device (never computed here);
                    # `sharding.assemble` / `owned_rects` say which part of a row is this rank's.
                    hout[y0:y1].copy_(self.canvas[y0:y1], non_blocking=True)
                    self.d2h_bytes += (y1 - y0) * self.W * self.canvas.shape[2] * self.canvas.element_size()
        main.wait_stream(self.down)
        return hout

    def _plan(self, first_patch, num_patches):
        if self.chunk_rows is None:
            batch = self.device_batch or default_device_batch(self.W, self.P, self.B)
            middle, edge = sharding.auto_chunk_rows(num_patches, self.nx, batch)
        else:
            middle = edge = int(self.chunk_rows)
        return sharding.plan_chunks(first_patch, num_patches, self.H, self.W, self.P, self.B, middle, edge)

    # ---- pageable numpy arrays: pinned staging ring + worker threads -------------------------------------------------
    def _ring(self, plan):
        """Slots sized for the largest chunk of ``plan`` (allocated once per pipeline, grown on demand)."""
        torch = self.torch
        divs = (1, 2, 6) if self.run_60 else (1, 2)
        devs = (self.d10, self.d20, self.d60)
        rows = [max(-(-r1 // dv) - r0 // dv for _, _, (r0, r1), _ in plan) for dv in divs]
        shapes = [(rows[i], devs[i].shape[1], devs[i].shape[2]) for i in range(len(divs))]
        out_elems = max(sum((y1 - y0) * (x1 - x0) for (y0, y1, x0, x1) in rects) for _, _, _, rects in plan) \
            * self.canvas.shape[2]
        if self._slots is None or any(a.shape[0] < s[0] for a, s in zip(self._slots[0].inp, shapes)) \
                or self._slots[0].out.numel() < out_elems:
            self._slots = [_Slot(torch, shapes, self.dtype, out_elems, self.out_dtype) for _ in range(self.RING)]
        if self._pool is None:
            self._pool = _staging_pool(torch, self.dev)
        return self._slots

    def run_numpy(self, a10, a20, a60=None, out=None, first_patch=0, num_patches=None, timers=None, nodata=None,
                  add_offset=None):
        """Pageable numpy arrays in -> numpy (H, W, Cout) array of ``out_dtype`` out (allocated if None).  Arrays whose
        dtype is not the pipeline's are cast while they are staged (the offset applies to the staged values).  ``nodata``
        and ``add_offset`` as in ``run``."""
        add_offset = check_add_offset(add_offset, self.model)
        torch = self.torch
        filled = self.ny * self.nx
        if num_patches is None:
            num_patches = filled - first_patch
        C = self.model.out_channels
        np_out = _np_dtype_of(torch, self.out_dtype)
        if out is None:
            out = np.empty((self.H, self.W, C), np_out)
        _check_out(out, (self.H, self.W, C), np.dtype(np_out), "out")
        srcs = [a10, a20] + ([a60] if self.run_60 else [])
        divs = (1, 2, 6) if self.run_60 else (1, 2)
        devs = [self.d10, self.d20] + ([self.d60] if self.run_60 else [])
        plan = self._plan(first_patch, num_patches)
        nodata, ids, count, count_host = self._nodata_buffers(nodata, first_patch, num_patches, len(plan))
        slots = self._ring(plan)
        # rows of every resolution a chunk has to bring (those beyond what earlier chunks brought)
        need, done = [], [None] * len(divs)
        for _, _, (r0, r1), _ in plan:
            rows = []
            for i, dv in enumerate(divs):
                a, b = r0 // dv, -(-r1 // dv)
                if done[i] is not None:
                    a = max(a, done[i])
                rows.append((a, max(a, b)))
                done[i] = max(a, b) if done[i] is None else max(done[i], b)
            need.append(rows)
        self.h2d_bytes = self.d2h_bytes = 0

        def stage_in(k):
            slot = slots[k % self.RING]
            if slot.used_in:
                slot.ev_h2d.synchronize()            # the previous upload from this slot has left it
            for i, (a, b) in enumerate(need[k]):
                if b > a:
                    slot.inp[i][:b - a].numpy()[...] = srcs[i][a:b]

        def stage_out(rects, src, offs, part, parts):
            for (y0, y1, x0, x1), o in zip(rects, offs):
                h = y1 - y0
                ya, yb = y0 + h * part // parts, y0 + h * (part + 1) // parts
                if yb > ya:
                    view = src[o:o + h * (x1 - x0) * C].reshape(h, x1 - x0, C)
                    out[ya:yb, x0:x1] = view[ya - y0:yb - y0]

        main = torch.cuda.current_stream(self.dev)
        self.up.wait_stream(main)
        self.down.wait_stream(main)
        fin = {k: self._pool.submit(stage_in, k) for k in range(min(self.RING, len(plan)))}
        fout = {}
        for k, (p0, cnt, _rows, rects) in enumerate(plan):
            slot = slots[k % self.RING]
            fin.pop(k).result()
            with torch.cuda.stream(self.up):
                for i, (a, b) in enumerate(need[k]):
                    if b > a:
                        devs[i][a:b].copy_(slot.inp[i][:b - a], non_blocking=True)
                        self.h2d_bytes += (b - a) * devs[i].shape[1] * devs[i].shape[2] * devs[i].element_size()
                slot.ev_h2d.record(self.up)
                slot.used_in = True
                ev_scan = None
                if nodata is not None:
                    a = p0 - first_patch
                    ev_scan = _scan_active(self.d10, self.d20, self.d60, p0, cnt, nodata, ids[a:a + cnt],
                                           count[k:k + 1], count_host[k:k + 1], timers)
            main.wait_event(slot.ev_h2d)
            if k + self.RING < len(plan):
                fin[k + self.RING] = self._pool.submit(stage_in, k + self.RING)
            self._compute(k, p0, cnt, first_patch, nodata, ids, count_host, ev_scan, timers, add_offset)
            ev_c = torch.cuda.Event()
            ev_c.record(main)
            self.down.wait_event(ev_c)
            for f in fout.pop(k - self.RING, ()):    # the slot's previous contents have been copied out
                f.result()
            offs, o = [], 0
            with torch.cuda.stream(self.down):
                for (y0, y1, x0, x1) in rects:
                    nel = (y1 - y0) * (x1 - x0) * C
                    dst = slot.out[o:o + nel].view(y1 - y0, x1 - x0, C)
                    dst.copy_(self.canvas[y0:y1] if (x0 == 0 and x1 == self.W) else self.canvas[y0:y1, x0:x1],
                              non_blocking=True)
                    offs.append(o)
                    o += nel
                    self.d2h_bytes += nel * self.canvas.element_size()
                slot.ev_d2h.record(self.down)
            src = slot.out.numpy()

            def drain(part, parts, rects=rects, src=src, offs=offs, ev=slot.ev_d2h):
                ev.synchronize()
                stage_out(rects, src, offs, part, parts)
            fout[k] = [self._pool.submit(drain, part, 2) for part in range(2)]
        for fs in fout.values():
            for f in fs:
                f.result()
        main.wait_stream(self.down)
        return out


class ChipPipeline:
    """Host-buffer front end for stacks of same-size chips (module docstring).  The unit is whole chips: a chunk is the
    chips whose patches fill about one device batch (``default_device_batch``; at least one chip), so its inputs and
    outputs are contiguous slices of the stacks, one copy per resolution.  Chunk k+1 uploads while chunk k computes and
    chunk k-1 downloads, through a ring of device chunk buffers: a stack larger than device memory streams through.
    Pinned torch tensors are copied directly; pageable numpy arrays go through pinned staging slots (``_Slot``) filled and
    drained by worker threads, as in ``HostPipeline.run_numpy``.  ``dtype`` / ``out_dtype`` as for ``HostPipeline``.
    Reusable across calls of one chip shape and any number of chips."""

    RING = 3

    def __init__(self, model, H, W, run_60=False, device=None, chunk_chips=None, dtype=None, out_dtype=None):
        u16 = check_out_dtype(out_dtype, model)
        torch = _capi.require_cuda()
        self.torch, self.model, self.run_60 = torch, model, run_60
        self.H, self.W = int(H), int(W)
        self.dtype = torch.float32 if dtype is None else dtype
        self.out_dtype = torch.uint16 if u16 else torch.float32
        self.divs = (1, 2, 6) if run_60 else (1, 2)
        in_shapes = [(1, self.H // d, self.W // d, c) for d, c in zip(self.divs, model.in_channels)]
        _, _, _, self.ppc = _stack_geometry(model, in_shapes, [str(self.dtype)[len('torch.'):]] * len(in_shapes), None)
        g = _GEOM[run_60]
        self.device_batch = default_device_batch(self.W, g['patch'], g['border'])
        self.chunk = int(chunk_chips) if chunk_chips else max(1, self.device_batch // self.ppc)
        self.in_shapes = [(self.chunk,) + s[1:] for s in in_shapes]
        self.out_shape = (self.chunk, self.H, self.W, model.out_channels)
        self.dev = torch.device('cuda', torch.cuda.current_device()) if device is None else device
        # no zero fill: the chips of a chunk own every pixel of their canvases
        self.d_in = [[torch.empty(s, dtype=self.dtype, device=self.dev) for s in self.in_shapes] for _ in range(self.RING)]
        self.d_out = [torch.empty(self.out_shape, dtype=self.out_dtype, device=self.dev) for _ in range(self.RING)]
        self.ev_free = [torch.cuda.Event() for _ in range(self.RING)]      # the last download from a ring entry
        self.up, self.down = torch.cuda.Stream(self.dev), torch.cuda.Stream(self.dev)
        self._slots, self._pool = None, None

    def _check(self, srcs, dtype_names):
        N, _, _, _ = _stack_geometry(self.model, [tuple(a.shape) for a in srcs], dtype_names, None)
        if tuple(srcs[0].shape[1:3]) != (self.H, self.W):
            raise ValueError("chips of %dx%d do not match the pipeline's %dx%d" % (*srcs[0].shape[1:3], self.H, self.W))
        return N

    def _chunks(self, N):
        return [(c0, min(N, c0 + self.chunk)) for c0 in range(0, N, self.chunk)]

    def _compute(self, e, n, timers, add_offset):
        """The network over the n chips of ring entry e, on the current stream."""
        d = [t[:n] for t in self.d_in[e]] + [None] * (3 - len(self.divs))
        super_resolve_device(self.model, *d, out=self.d_out[e][:n], device_batch=self.device_batch, timers=timers,
                             out_dtype=self.out_dtype, add_offset=add_offset)

    def run(self, h10, h20, h60=None, hout=None, timers=None, add_offset=None):
        """Pinned torch stacks in (dtype = the pipeline's), pinned (N, H, W, Cout) tensor of ``out_dtype`` out."""
        add_offset = check_add_offset(add_offset, self.model)
        torch = self.torch
        srcs = [h10, h20] + ([h60] if self.run_60 else [])
        if any(h.dtype != self.dtype for h in srcs):
            raise ValueError("host image dtype does not match the pipeline's %s" % self.dtype)
        N = self._check(srcs, [str(h.dtype)[len('torch.'):] for h in srcs])
        if hout is None:
            hout = torch.empty((N,) + self.out_shape[1:], dtype=self.out_dtype).pin_memory()
        _check_out(hout, (N,) + self.out_shape[1:], self.out_dtype, "hout")
        main = torch.cuda.current_stream(self.dev)
        self.up.wait_stream(main)
        self.down.wait_stream(main)
        for k, (c0, c1) in enumerate(self._chunks(N)):
            e = k % self.RING
            with torch.cuda.stream(self.up):
                if k >= self.RING:
                    self.up.wait_event(self.ev_free[e])     # chunk k - RING has been computed and downloaded
                for d, h in zip(self.d_in[e], srcs):
                    d[:c1 - c0].copy_(h[c0:c1], non_blocking=True)
                ev_up = torch.cuda.Event()
                ev_up.record(self.up)
            main.wait_event(ev_up)
            self._compute(e, c1 - c0, timers, add_offset)
            ev_c = torch.cuda.Event()
            ev_c.record(main)
            self.down.wait_event(ev_c)
            with torch.cuda.stream(self.down):
                hout[c0:c1].copy_(self.d_out[e][:c1 - c0], non_blocking=True)
                self.ev_free[e].record(self.down)
        main.wait_stream(self.down)
        return hout

    def run_numpy(self, a10, a20, a60=None, out=None, timers=None, add_offset=None):
        """Pageable numpy stacks in -> numpy (N, H, W, Cout) array of ``out_dtype`` out (allocated if None).  The stacks'
        element type must be float32 or uint16; a type that is not the pipeline's is cast while it is staged."""
        add_offset = check_add_offset(add_offset, self.model)
        torch = self.torch
        srcs = [a10, a20] + ([a60] if self.run_60 else [])
        N = self._check(srcs, [a.dtype.name for a in srcs])
        np_out = np.dtype(_np_dtype_of(torch, self.out_dtype))
        if out is None:
            out = np.empty((N,) + self.out_shape[1:], np_out)
        _check_out(out, (N,) + self.out_shape[1:], np_out, "out")
        chunks = self._chunks(N)
        if not chunks:
            return out
        if self._slots is None:
            out_elems = int(np.prod(self.out_shape))
            self._slots = [_Slot(torch, self.in_shapes, self.dtype, out_elems, self.out_dtype) for _ in range(self.RING)]
            self._pool = _staging_pool(torch, self.dev)
        slots = self._slots

        def stage_in(k):
            slot = slots[k % self.RING]
            if slot.used_in:
                slot.ev_h2d.synchronize()            # the previous upload from this slot has left it
            c0, c1 = chunks[k]
            for buf, a in zip(slot.inp, srcs):
                buf[:c1 - c0].numpy()[...] = a[c0:c1]

        def drain(k, part, parts, ev, src):
            ev.synchronize()
            c0, c1 = chunks[k]
            a, b = c0 + (c1 - c0) * part // parts, c0 + (c1 - c0) * (part + 1) // parts
            if b > a:
                out[a:b] = src[a - c0:b - c0]

        main = torch.cuda.current_stream(self.dev)
        self.up.wait_stream(main)
        self.down.wait_stream(main)
        fin = {k: self._pool.submit(stage_in, k) for k in range(min(self.RING, len(chunks)))}
        fout = {}
        for k, (c0, c1) in enumerate(chunks):
            e, n = k % self.RING, c1 - c0
            slot = slots[e]
            fin.pop(k).result()
            with torch.cuda.stream(self.up):
                if k >= self.RING:
                    self.up.wait_event(self.ev_free[e])
                for d, buf in zip(self.d_in[e], slot.inp):
                    d[:n].copy_(buf[:n], non_blocking=True)
                slot.ev_h2d.record(self.up)
                slot.used_in = True
            main.wait_event(slot.ev_h2d)
            if k + self.RING < len(chunks):
                fin[k + self.RING] = self._pool.submit(stage_in, k + self.RING)
            self._compute(e, n, timers, add_offset)
            ev_c = torch.cuda.Event()
            ev_c.record(main)
            self.down.wait_event(ev_c)
            for f in fout.pop(k - self.RING, ()):    # the slot's previous contents have been copied out
                f.result()
            dst = slot.out[:n * int(np.prod(self.out_shape[1:]))].view((n,) + self.out_shape[1:])
            with torch.cuda.stream(self.down):
                dst.copy_(self.d_out[e][:n], non_blocking=True)
                slot.ev_d2h.record(self.down)
                self.ev_free[e].record(self.down)
            src = dst.numpy()
            fout[k] = [self._pool.submit(drain, k, part, 2, slot.ev_d2h, src) for part in range(2)]
        for fs in fout.values():
            for f in fs:
                f.result()
        main.wait_stream(self.down)
        return out


_pipe_cache = {}


def _pipeline_for(model, H, W, run_60, dtype, out_dtype):
    """HostPipeline objects (device-resident tile + pinned staging ring) are kept for the last shapes used, so a caller
    that super-resolves scene after scene pays the allocations once."""
    torch = _capi.require_cuda()
    key = (id(model), H, W, run_60, dtype, out_dtype, torch.cuda.current_device())
    pipe = _pipe_cache.get(key)
    if pipe is None or pipe.model is not model:
        if len(_pipe_cache) >= 2:
            _pipe_cache.clear()
        pipe = _pipe_cache[key] = HostPipeline(model, H, W, run_60=run_60, dtype=dtype, out_dtype=out_dtype)
    return pipe


_chip_pipe_cache = {}


def _chip_pipeline_for(model, H, W, run_60, dtype, out_dtype):
    """ChipPipeline objects (device chunk ring + pinned staging ring), kept for the last chip shapes used like
    ``_pipeline_for``, so a caller that works through a dataset stack after stack pays the allocations once."""
    torch = _capi.require_cuda()
    key = (id(model), H, W, run_60, dtype, out_dtype, torch.cuda.current_device())
    pipe = _chip_pipe_cache.get(key)
    if pipe is None or pipe.model is not model:
        if len(_chip_pipe_cache) >= 2:
            _chip_pipe_cache.clear()
        pipe = _chip_pipe_cache[key] = ChipPipeline(model, H, W, run_60=run_60, dtype=dtype, out_dtype=out_dtype)
    return pipe


def _run_chips(model, arrays, out=None, nodata=None, out_dtype=np.float32, add_offset=None):
    # rejected before the device is touched
    u16 = check_out_dtype(out_dtype, model)
    add_offset = check_add_offset(add_offset, model)
    arrays = [np.asarray(a) for a in arrays]
    N, H, W, _ = _stack_geometry(model, [a.shape for a in arrays], [a.dtype.name for a in arrays], nodata)
    np_out = np.dtype(np.uint16 if u16 else np.float32)
    _check_out(out, (N, H, W, model.out_channels), np_out, "out")
    if N == 0:
        return np.empty((0, H, W, model.out_channels), np_out) if out is None else out
    torch = _capi.require_cuda()
    dtype = torch.uint16 if arrays[0].dtype == np.uint16 else torch.float32
    pipe = _chip_pipeline_for(model, H, W, len(arrays) == 3, dtype, torch.uint16 if u16 else torch.float32)
    res = pipe.run_numpy(*arrays, out=out, add_offset=add_offset)
    torch.cuda.current_stream().synchronize()
    return res


def _run(model, arrays, out=None, nodata=None, out_dtype=np.float32, add_offset=None):
    # rejected before the device is touched
    u16 = check_out_dtype(out_dtype, model)
    add_offset = check_add_offset(add_offset, model)
    if nodata is not None:
        nodata = check_nodata(nodata, model,
                              u16 or (model.xin16 and all(np.asarray(a).dtype == np.uint16 for a in arrays)))
    a10 = np.asarray(arrays[0])
    if out is not None and a10.ndim >= 2:
        _check_out(out, (a10.shape[0], a10.shape[1], model.out_channels), np.dtype(np.uint16 if u16 else np.float32),
                   "out")
    torch = _capi.require_cuda()
    arrays = [np.asarray(a) for a in arrays]
    H, W = int(arrays[0].shape[0]), int(arrays[0].shape[1])
    for a, div, c in zip(arrays, (1, 2, 6), model.in_channels):
        if a.ndim != 3 or tuple(a.shape) != (H // div, W // div, c):
            raise ValueError("expected an image of shape %s (HWC, 10 m size %dx%d / %d), got %s"
                             % ((H // div, W // div, c), H, W, div, tuple(a.shape)))
    # uint16 digital numbers (GDAL, s2_tiles_supres.py:311-315) stay uint16 up to the input-preparation kernel; everything
    # else is staged as float32 (the reference divides by SCALE in floating point whatever the input type, supres.py:23-24)
    dtype = torch.uint16 if (model.xin16 and all(a.dtype == np.uint16 for a in arrays)) else torch.float32
    pipe = _pipeline_for(model, H, W, len(arrays) == 3, dtype, torch.uint16 if u16 else torch.float32)
    res = pipe.run_numpy(*arrays, out=out, nodata=nodata, add_offset=add_offset)
    torch.cuda.current_stream().synchronize()
    return res


def DSen2_20(d10, d20, deep=False, model=None, out=None, nodata=None, out_dtype=np.float32, add_offset=None):
    """supres.py:15-30.  d10 (H,W,4), d20 (H/2,W/2,6) -> (H,W,6) float32.  Extensions: ``model`` supplies a preloaded
    ``S2Model`` instead of the shipped hdf5 weights, ``out`` a preallocated (H,W,6) array of ``out_dtype`` to fill,
    ``nodata`` the input value of pixels without data (module docstring): they come out as ``nodata`` and empty patches are
    skipped; ``out_dtype`` np.uint16: digital numbers, rounded and saturated on the device (module docstring);
    ``add_offset`` the radiometric offset of the product (-1000 for processing baseline 04.00 and later; module docstring):
    removed from the inputs and restored on the output, on the device.  Chip stacks: d10 (N,H,W,4), d20 (N,H/2,W/2,6),
    all float32 or all uint16 -> (N,H,W,6) (module docstring)."""
    input_shape = ((4, None, None), (6, None, None))
    if model is None:
        model = _load_model(input_shape, deep, run_60=False)
    run = _run_chips if np.ndim(d10) == 4 else _run
    return run(model, [d10, d20], out, nodata, out_dtype, add_offset)


def DSen2_60(d10, d20, d60, deep=False, model=None, out=None, nodata=None, out_dtype=np.float32, add_offset=None):
    """supres.py:33-50.  + d60 (H/6,W/6,2) -> (H,W,2) float32 (or ``out_dtype``).  Chip stacks: + d60 (N,H/6,W/6,2) ->
    (N,H,W,2)."""
    input_shape = ((4, None, None), (6, None, None), (2, None, None))
    if model is None:
        model = _load_model(input_shape, deep, run_60=True)
    run = _run_chips if np.ndim(d10) == 4 else _run
    return run(model, [d10, d20, d60], out, nodata, out_dtype, add_offset)
