"""Host-side mirror of the reference ``utils/patches.py`` (test-time tiling / stitching).

Same names, argument meaning and return shapes as the reference functions
(``get_test_patches`` :19-80, ``get_test_patches60`` :83-156, ``interp_patches`` :11-16,
``recompose_images`` :374-405); the arithmetic runs in the CUDA kernels of
``csrc/patch_kernels.cu`` through the C ABI.  The ``*_device`` functions are the
torch-tensor level used by the engine (no host round trips).
"""
from math import ceil

import numpy as np

from . import _capi

VERBOSE = True   # recompose_images prints the canvas shape like the reference (patches.py:392)


def patch_counts(grid_h, grid_w, patch_lr, border_lr):
    """(allocated, filled) patch counts (patches.py:32-53)."""
    import ctypes
    a, f = ctypes.c_int(0), ctypes.c_int(0)
    rc = _capi.lib().dsen2_patch_counts(grid_h, grid_w, patch_lr, border_lr, ctypes.byref(a), ctypes.byref(f))
    if rc:
        raise ValueError(_capi.lib().dsen2_last_error().decode())
    return a.value, f.value


# ------------------------------------------------------------------------------------------ #
# device level
# ------------------------------------------------------------------------------------------ #
def extract_patches_device(img, ratio, patch_lr, border_lr, first_patch=0, num_patches=None, divisor=1.0, out=None):
    """img: CUDA float32 (H, W, C) contiguous -> (num_patches, C, p, p) float32."""
    torch = _capi.require_cuda()
    assert img.is_cuda and img.dtype == torch.float32 and img.is_contiguous() and img.dim() == 3
    H, W, C = img.shape
    if H % ratio or W % ratio:
        raise ValueError("image size %dx%d is not a multiple of the resolution ratio %d" % (H, W, ratio))
    gh, gw = H // ratio, W // ratio
    allocated, _ = patch_counts(gh, gw, patch_lr, border_lr)
    if num_patches is None:
        num_patches = allocated - first_patch
    p = patch_lr * ratio
    if out is None:
        out = torch.empty((num_patches, C, p, p), dtype=torch.float32, device=img.device)
    with torch.cuda.device(img.device):
        rc = _capi.lib().dsen2_extract_patches(_capi.ptr(img), gh, gw, C, ratio, patch_lr, border_lr, first_patch,
                                               num_patches, float(divisor), _capi.ptr(out), _capi.stream_ptr())
    if rc == -1:
        raise ValueError(_capi.lib().dsen2_last_error().decode())
    _capi.check(rc, "dsen2_extract_patches")
    return out


def bilinear_up_device(x, scale, post_divisor=1.0, out=None):
    """x: CUDA float32 (..., p, p) -> (..., p*scale, p*scale), mirror boundary (patches.py:11-16)."""
    torch = _capi.require_cuda()
    assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous()
    p = x.shape[-1]
    assert x.shape[-2] == p, "patches are square"
    planes = x.numel() // (p * p)
    if out is None:
        out = torch.empty(tuple(x.shape[:-2]) + (p * scale, p * scale), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        rc = _capi.lib().dsen2_bilinear_mirror_up(_capi.ptr(x), planes, p, scale, float(post_divisor),
                                                  _capi.ptr(out), _capi.stream_ptr())
    _capi.check(rc, "dsen2_bilinear_mirror_up")
    return out


def recompose_device(pred, border, H, W, first_patch=0, mul=1.0, out=None):
    """pred: CUDA float32 (n, C, P, P) holding patches [first_patch, first_patch+n) -> writes into (H, W, C)."""
    torch = _capi.require_cuda()
    assert pred.is_cuda and pred.dtype == torch.float32 and pred.is_contiguous() and pred.dim() == 4
    n, C, P, _ = pred.shape
    if out is None:
        out = torch.zeros((H, W, C), dtype=torch.float32, device=pred.device)
    with torch.cuda.device(pred.device):
        rc = _capi.lib().dsen2_recompose(_capi.ptr(pred), first_patch, n, C, P, border, H, W, float(mul),
                                         _capi.ptr(out), _capi.stream_ptr())
    if rc == -1:
        raise ValueError(_capi.lib().dsen2_last_error().decode())
    _capi.check(rc, "dsen2_recompose")
    return out


# ------------------------------------------------------------------------------------------ #
# numpy level: the reference's signatures
# ------------------------------------------------------------------------------------------ #
def _to_dev(a):
    torch = _capi.require_cuda()
    a = np.ascontiguousarray(np.asarray(a), dtype=np.float32)   # the reference casts on assignment into float32 stacks
    return torch.from_numpy(a).cuda()


def interp_patches(image_20, image_10_shape):
    image_20 = np.asarray(image_20)
    P = image_10_shape[2]
    s = P // image_20.shape[2]
    if image_20.shape[2] * s != P or tuple(image_10_shape[2:4]) != (P, P):
        raise ValueError("interp_patches supports square integer-factor upsampling only")
    if image_20.shape[0] == 0:
        return np.zeros(image_20.shape[0:2] + tuple(image_10_shape[2:4]), np.float32)
    return bilinear_up_device(_to_dev(image_20), s).cpu().numpy()


def get_test_patches(dset_10, dset_20, patchSize=128, border=4, interp=True):
    d10, d20 = _to_dev(dset_10), _to_dev(dset_20)
    if d10.shape[0] != 2 * d20.shape[0] or d10.shape[1] != 2 * d20.shape[1]:
        raise ValueError("dset_10 must be exactly twice the size of dset_20")
    plr, blr = patchSize // 2, border // 2
    image_10 = extract_patches_device(d10, 2, plr, blr)
    image_20 = extract_patches_device(d20, 1, plr, blr)
    if interp:
        image_20 = bilinear_up_device(image_20, 2)
    return image_10.cpu().numpy(), image_20.cpu().numpy()


def get_test_patches60(dset_10, dset_20, dset_60, patchSize=128, border=8, interp=True):
    d10, d20, d60 = _to_dev(dset_10), _to_dev(dset_20), _to_dev(dset_60)
    if (d10.shape[0] != 6 * d60.shape[0] or d10.shape[1] != 6 * d60.shape[1] or
            d20.shape[0] != 3 * d60.shape[0] or d20.shape[1] != 3 * d60.shape[1]):
        raise ValueError("dset_10 / dset_20 must be exactly 6x / 3x the size of dset_60")
    plr, blr = patchSize // 6, border // 6
    image_10 = extract_patches_device(d10, 6, plr, blr)
    image_20 = extract_patches_device(d20, 3, plr, blr)
    image_60 = extract_patches_device(d60, 1, plr, blr)
    if interp:
        image_20 = bilinear_up_device(image_20, 2)
        image_60 = bilinear_up_device(image_60, 6)
    return image_10.cpu().numpy(), image_20.cpu().numpy(), image_60.cpu().numpy()


def recompose_images(a, border, size=None):
    a = np.asarray(a)
    if a.shape[0] == 1:
        images = np.ascontiguousarray(a[0], dtype=np.float32)   # returned uncropped (patches.py:375-376)
        return images.transpose((1, 2, 0))
    H, W = int(size[0]), int(size[1])
    patch_size = a.shape[2] - border * 2
    x_tiles, y_tiles = int(ceil(W / float(patch_size))), int(ceil(H / float(patch_size)))
    if a.shape[0] < x_tiles * y_tiles:
        raise IndexError("index %d is out of bounds for axis 0 with size %d" % (a.shape[0], a.shape[0]))
    if VERBOSE:
        print((a.shape[1], H, W))
    used = a[:x_tiles * y_tiles]          # surplus (all-zero) patches are never read by the reference loop
    return recompose_device(_to_dev(used), border, H, W).cpu().numpy()


# ------------------------------------------------------------------------------------------ #
# training / prediction data sets on disk (utils/patches.py:274-350): plain numpy file I/O
# ------------------------------------------------------------------------------------------ #
def splitTrainVal(train_path, train, label):
    """utils/patches.py:274-285: boolean ``val_index.npy`` selects the validation patches."""
    try:
        val_ind = np.load(train_path + 'val_index.npy')
    except IOError:
        print("Please define the validation split indices, usually located in .../data/test/. To generate this file use"
              " createRandom.py")
        raise
    val_tr = [p[val_ind] for p in train]
    train = [p[~val_ind] for p in train]
    val_lb, label = label[val_ind], label[~val_ind]
    print("Loaded {} patches for training.".format(val_ind.shape[0]))
    return train, label, val_tr, val_lb


def OpenDataFiles(path, run_60, SCALE):
    """utils/patches.py:288-324: concatenate the per-scene ``data10/20[/60][_gt].npy`` stacks under ``train/`` or
    ``train60/``, divide by SCALE, split by ``val_index.npy`` -> (train list, label, val list, val label)."""
    import glob
    import os
    train_path = path + ('train60/' if run_60 else 'train/')
    names = ['data10', 'data20'] + (['data60', 'data60_gt'] if run_60 else ['data20_gt'])
    stacks = {k: [] for k in names}
    for dset in [os.path.basename(x) for x in sorted(glob.glob(train_path + '*SAFE'))]:
        for k in names:
            stacks[k].append(np.load(train_path + dset + '/' + k + '.npy'))
    data = {k: (np.concatenate(v) if v else None) for k, v in stacks.items()}
    if SCALE:
        for k in names:
            if data[k] is not None:
                data[k] = data[k] / SCALE          # float32 stacks stay float32 (the reference divides in place)
    if run_60:
        return splitTrainVal(train_path, [data['data10'], data['data20'], data['data60']], data['data60_gt'])
    return splitTrainVal(train_path, [data['data10'], data['data20']], data['data20_gt'])


def OpenDataFilesTest(path, run_60, SCALE, true_scale=False):
    """utils/patches.py:327-350: one scene's patch stacks + ``roi.json`` -> (input list, [height, width])."""
    import json
    if not SCALE:
        SCALE = 1
    train = [np.load(path + '/data10.npy') / SCALE, np.load(path + '/data20.npy') / SCALE]
    if run_60:
        train.append(np.load(path + '/data60.npy') / SCALE)
    with open(path + '/roi.json') as fh:
        roi = json.load(fh)
    image_size = [(roi[2] - roi[0]), (roi[3] - roi[1])]
    print("The image size is: {}".format(image_size))
    print("The SCALE is: {}".format(SCALE))
    print("The true_scale is: {}".format(true_scale))
    return train, image_size


# ------------------------------------------------------------------------------------------ #
# training-data generation (utils/patches.py:159-271, 353-371; used by training/create_patches.py)
# ------------------------------------------------------------------------------------------ #
def downPixelAggr(img, SCALE=2):
    """patches.py:353-371: Gaussian blur with sigma = 1/SCALE per band, then SCALE x SCALE pixel aggregation.
    Returns float64 like the reference (``np.zeros`` default dtype), squeezed.  An integer image (the uint16 digital numbers
    ``create_patches.py`` reads through GDAL) is blurred the way scipy blurs it: every pass stored in the image's dtype,
    i.e. truncated towards zero."""
    torch = _capi.require_cuda()
    img = np.asarray(img)
    if img.ndim == 2:
        img = img[:, :, None]
    integer = np.issubdtype(img.dtype, np.integer)
    if integer and (img.dtype.itemsize > 2 or (img.size and img.min() < 0)):
        raise ValueError("downPixelAggr: integer images must be uint8 / uint16 / non-negative int16 (exact in float32)")
    d = torch.from_numpy(np.ascontiguousarray(img, dtype=np.float32)).cuda()
    return np.squeeze(down_pixel_aggr_device(d, SCALE, integer=integer).cpu().numpy())



def down_pixel_aggr_device(img, scale, integer=None):
    """``downPixelAggr`` on the device: CUDA (H, W, C) float32 or uint16 -> CUDA float64 (H // scale, W // scale, C).
    ``integer``: blur as scipy blurs an integer image (every pass truncated); None = whether ``img`` is uint16.  A float32
    image holding the values of an integer image (``downPixelAggr``'s upload) passes ``integer=True``."""
    torch = _capi.require_cuda()
    if img.dim() != 3 or img.dtype not in (torch.float32, torch.uint16) or not img.is_cuda:
        raise ValueError("down_pixel_aggr_device: a CUDA (H, W, C) float32 or uint16 tensor, got %s %s"
                         % (img.dtype, tuple(img.shape)))
    if integer is None:
        integer = img.dtype == torch.uint16
    if img.dtype == torch.uint16:                        # uint16 -> float32 is exact; through int32 (the int16 bits)
        img = img.view(torch.int16).to(torch.int32).bitwise_and_(0xffff).to(torch.float32)
    img = img.contiguous()
    sigma = 1.0 / scale
    radius = int(4.0 * sigma + 0.5)                      # scipy.ndimage.gaussian_filter1d, truncate = 4.0
    x = np.arange(-radius, radius + 1)
    w = np.exp(-0.5 / (sigma * sigma) * x ** 2)
    w = w / w.sum()
    dw = torch.from_numpy(w).to(img.device)
    H, W, C = (int(s) for s in img.shape)
    tmp = torch.empty_like(img)
    out = torch.empty((H // scale, W // scale, C), dtype=torch.float64, device=img.device)
    with torch.cuda.device(img.device):
        rc = _capi.lib().dsen2_down_pixel_aggr(_capi.ptr(img), int(bool(integer)), H, W, C, scale, _capi.ptr(dw), radius,
                                               _capi.ptr(tmp), _capi.ptr(out), _capi.stream_ptr())
    _capi.check(rc, "dsen2_down_pixel_aggr")
    return out


def save_test_patches(dset_10, dset_20, file, patchSize=128, border=4, interp=True):
    """patches.py:159-167."""
    image_10, data20_interp = get_test_patches(dset_10, dset_20, patchSize=patchSize, border=border, interp=interp)
    print("Saving to file {}".format(file))
    np.save(file + 'data10', image_10)
    np.save(file + 'data20', data20_interp)
    print('Done!')


def save_test_patches60(dset_10, dset_20, dset_60, file, patchSize=192, border=12, interp=True):
    """patches.py:170-180."""
    image_10, data20_interp, data60_interp = get_test_patches60(dset_10, dset_20, dset_60, patchSize=patchSize,
                                                                border=border, interp=interp)
    print("Saving to file {}".format(file))
    np.save(file + 'data10', image_10)
    np.save(file + 'data20', data20_interp)
    np.save(file + 'data60', data60_interp)
    print('Done!')


def _random_crops(lowest, sizes_lr, nr_crop):
    from random import randrange
    for _ in range(nr_crop):
        x0 = randrange(0, lowest.shape[0] - sizes_lr[0])
        y0 = randrange(0, lowest.shape[1] - sizes_lr[1])
        yield x0, y0


def _crop_chw(d, x0, y0, h, w):
    return np.rollaxis(d[x0:x0 + h, y0:y0 + w], 2)


def save_random_patches(dset_20gt, dset_10, dset_20, file, NR_CROP=8000):
    """patches.py:183-224: random 16x16 (20 m) crops with their 32x32 counterparts; the 20 m stack is upsampled."""
    label_20 = np.zeros((NR_CROP, dset_20.shape[2], 32, 32), np.float32)
    image_20 = np.zeros((NR_CROP, dset_20.shape[2], 16, 16), np.float32)
    image_10 = np.zeros((NR_CROP, dset_10.shape[2], 32, 32), np.float32)
    for i, (x0, y0) in enumerate(_random_crops(dset_20, (16, 16), NR_CROP)):
        label_20[i] = _crop_chw(dset_20gt, 2 * x0, 2 * y0, 32, 32)
        image_20[i] = _crop_chw(dset_20, x0, y0, 16, 16)
        image_10[i] = _crop_chw(dset_10, 2 * x0, 2 * y0, 32, 32)
    np.save(file + 'data10', image_10)
    np.save(file + 'data20_gt', label_20)
    np.save(file + 'data20', interp_patches(image_20, image_10.shape))
    print('Done!')


def save_random_patches60(dset_60gt, dset_10, dset_20, dset_60, file, NR_CROP=500):
    """patches.py:227-271: random 16x16 (60 m) crops with their 48x48 (20 m) and 96x96 (10 m) counterparts."""
    label_60 = np.zeros((NR_CROP, dset_60.shape[2], 96, 96), np.float32)
    image_10 = np.zeros((NR_CROP, dset_10.shape[2], 96, 96), np.float32)
    image_20 = np.zeros((NR_CROP, dset_20.shape[2], 48, 48), np.float32)
    image_60 = np.zeros((NR_CROP, dset_60.shape[2], 16, 16), np.float32)
    for i, (x0, y0) in enumerate(_random_crops(dset_60, (16, 16), NR_CROP)):
        label_60[i] = _crop_chw(dset_60gt, 6 * x0, 6 * y0, 96, 96)
        image_10[i] = _crop_chw(dset_10, 6 * x0, 6 * y0, 96, 96)
        image_20[i] = _crop_chw(dset_20, 3 * x0, 3 * y0, 48, 48)
        image_60[i] = _crop_chw(dset_60, x0, y0, 16, 16)
    np.save(file + 'data10', image_10)
    np.save(file + 'data60_gt', label_60)
    np.save(file + 'data20', interp_patches(image_20, image_10.shape))
    np.save(file + 'data60', interp_patches(image_60, image_10.shape))
    print('Done!')
