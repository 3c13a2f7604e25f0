"""Every launch path of the resampling, stitching and nodata entry points against the CPU oracle.

The C entry points of ``csrc/patch_kernels.cu`` and ``csrc/nodata.cu`` pick a kernel from the channel count, the patch size,
the scale, pointer alignment or the tap count.  Each case names the kernel it is meant to reach and asserts, from a
``torch.profiler`` trace, that this kernel ran, so a change to the dispatch cannot move a case off its branch unnoticed.
The choice between the tiled passes and the direct form inside ``bicubic_tiled_kernel`` has no kernel name of its own: a
CPU restatement of that condition (``bicubic_forms``) asserts it from the tap tables."""
import numpy as np
import pytest

from oracle import imresize_oracle as io_
from oracle import patches_oracle as po
from test_gpu_nodata import oracle as nodata_oracle


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32 if a.dtype == np.float32 else np.uint64)


@pytest.fixture(scope='module')
def torch_mod():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from dsen2_b200 import patches
    patches.VERBOSE = False
    return torch


@pytest.fixture(scope='module')
def launched(torch_mod):
    """launched(fn) -> (fn(), set of the kernels fn launched), names as 'dsen2::kernel<template args>' without spaces."""
    torch = torch_mod
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile

    def run(fn):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            result = fn()
            torch.cuda.synchronize()
        names = set()
        for e in prof.events():
            if e.device_type == DeviceType.CUDA:
                n = e.name[5:] if e.name.startswith('void ') else e.name
                names.add(n.split('(')[0].replace(' ', ''))
        return result, names
    return run


def _ran(names, kernel):
    assert 'dsen2::' + kernel in names, (kernel, sorted(names))


def _on_device(torch, a, offset=0):
    """Copy of numpy ``a`` on the GPU starting ``offset`` elements past an allocation (which is 512-byte aligned)."""
    t = torch.from_numpy(np.ascontiguousarray(a))
    buf = torch.empty(t.numel() + offset, dtype=t.dtype, device='cuda')
    v = buf[offset:].view(t.shape)
    v.copy_(t)
    return v


def _nan_canvas(torch, shape, offset=0):
    buf = torch.full((int(np.prod(shape)) + offset,), float('nan'), dtype=torch.float32, device='cuda')
    return buf[offset:].view(shape)


# ---- bilinear (dsen2_bilinear_mirror_up) ------------------------------------------------------------------------------
SCALAR = 'bilinear_mirror_kernel'
BAND = 'bilinear_mirror_band_kernel<%d>'
# (p, s, input offset, output offset in floats, kernel).  One float of offset leaves the input 4-byte aligned (the x2_p64
# kernel wants 8) and the output 4-byte aligned (the band kernels' 16-byte row stores want 16).
BILINEAR = [
    (64, 2, 0, 0, 'bilinear_mirror_x2_p64_kernel'),
    (64, 2, 1, 0, BAND % 2),
    (64, 2, 0, 1, SCALAR),
    (16, 2, 0, 0, BAND % 2), (40, 2, 0, 0, BAND % 2), (2, 2, 0, 0, BAND % 2),        # 40: a short last band of rows
    (16, 6, 0, 0, BAND % 6), (40, 6, 0, 0, BAND % 6), (2, 6, 0, 0, BAND % 6),
    (8, 3, 0, 0, BAND % 0), (8, 4, 0, 0, BAND % 0), (8, 5, 0, 0, BAND % 0), (40, 3, 0, 0, BAND % 0),
    (3, 4, 1, 0, BAND % 0),
    (1, 2, 0, 0, SCALAR), (1, 6, 0, 0, SCALAR),                                         # one-pixel planes
    (7, 2, 0, 0, SCALAR), (3, 2, 0, 0, SCALAR), (3, 6, 0, 0, SCALAR),                   # P % 4 != 0
    (200, 6, 0, 0, SCALAR),                                                             # P > 1024
]


@pytest.mark.gpu
@pytest.mark.parametrize('p,s,in_off,out_off,kernel', BILINEAR,
                         ids=['p%d-s%d-in%d-out%d' % c[:4] for c in BILINEAR])
def test_bilinear_branch(torch_mod, launched, p, s, in_off, out_off, kernel):
    """Oracle within 2e-3 DN; ``post_divisor`` is one IEEE division of the undivided result; and the scalar kernel gives
    the same bits as the branch under test on the same planes."""
    torch = torch_mod
    from dsen2_b200 import patches
    P = p * s
    shape = (1, 2, p, p) if P > 1024 else (2, 3, p, p)
    x = (np.random.RandomState(100 * p + s).rand(*shape) * 10000).astype(np.float32)   # every plane different
    ref = po.interp_patches(x, shape[:2] + (P, P))
    xd = _on_device(torch, x, in_off)
    got = {}
    for div in (1.0, 2000.0):
        out = _nan_canvas(torch, shape[:2] + (P, P), out_off)
        _, names = launched(lambda: patches.bilinear_up_device(xd, s, div, out))
        _ran(names, kernel)
        got[div] = out.cpu().numpy()
    np.testing.assert_allclose(got[1.0], ref, rtol=0, atol=2e-3)
    assert np.array_equal(_bits(got[2000.0]), _bits(got[1.0] / np.float32(2000)))
    if kernel != SCALAR:
        out = _nan_canvas(torch, shape[:2] + (P, P), 1)
        _, names = launched(lambda: patches.bilinear_up_device(xd, s, 1.0, out))
        _ran(names, SCALAR)
        assert np.array_equal(_bits(out.cpu().numpy()), _bits(got[1.0]))


@pytest.mark.gpu
def test_bilinear_one_pixel_planes_read_only_their_pixel(torch_mod):
    """A 1x1 plane upsamples to its own value (up to the /30000 round trip), whatever the next plane or the memory
    after the last plane holds; through the public interp_patches and get_test_patches(patchSize=2, border=0)."""
    torch = torch_mod
    from dsen2_b200 import patches
    x = np.array([1000., 9000., 3.], np.float32).reshape(3, 1, 1, 1)
    for s in (2, 3, 6):
        got = patches.interp_patches(x, (3, 1, s, s))
        np.testing.assert_allclose(got, np.broadcast_to(x, (3, 1, s, s)), rtol=0, atol=2e-3)
    rng = np.random.RandomState(3)
    d10 = (rng.rand(6, 8, 4) * 5000).astype(np.float32)
    d20 = (rng.rand(3, 4, 6) * 5000).astype(np.float32)
    _, g20 = patches.get_test_patches(d10, d20, patchSize=2, border=0)
    _, r20 = po.get_test_patches(d10, d20, patchSize=2, border=0)
    np.testing.assert_allclose(g20, r20, rtol=0, atol=2e-3)


# ---- extract (dsen2_extract_patches) ----------------------------------------------------------------------------------
def _extract_kernel(C, aligned):
    return 'extract_patches_kernel<%d>' % C if C in (2, 4, 6) and aligned else 'extract_patches_generic_kernel'


def _extract_sources(C, seed, g20=(36, 41), g60=(18, 20)):
    """(image, ratio, patch_lr, border_lr, oracle stack) for the ratios 2, 1 (20 m tiling: patch 32 / border 4 at 10 m) and
    6, 3, 1 (60 m tiling: patch 48 / border 6).  36 and 18 are multiples of the stride (surplus zero patches); 41 and 20
    are not (a clamped last column)."""
    rng = np.random.RandomState(seed)
    im = lambda h, w: (rng.rand(h, w, C) * 10000).astype(np.float32)
    a10, a20 = im(2 * g20[0], 2 * g20[1]), im(*g20)
    r10, r20 = po.get_test_patches(a10, a20, 32, 4, interp=False)
    b10, b20, b60 = im(6 * g60[0], 6 * g60[1]), im(3 * g60[0], 3 * g60[1]), im(*g60)
    q10, q20, q60 = po.get_test_patches60(b10, b20, b60, 48, 6, interp=False)
    return [(a10, 2, 16, 2, r10), (a20, 1, 16, 2, r20), (b10, 6, 8, 1, q10), (b20, 3, 8, 1, q20), (b60, 1, 8, 1, q60)]


@pytest.mark.gpu
@pytest.mark.parametrize('C', [1, 2, 3, 4, 5, 6])
def test_extract_every_ratio_bit_exact(torch_mod, launched, C):
    torch = torch_mod
    from dsen2_b200 import patches
    for img, ratio, plr, blr, ref in _extract_sources(C, seed=C):
        d = _on_device(torch, img)
        for div in (1.0, 2000.0):
            got, names = launched(lambda: patches.extract_patches_device(d, ratio, plr, blr, divisor=div).cpu().numpy())
            _ran(names, _extract_kernel(C, True))
            assert np.array_equal(_bits(got), _bits(ref / np.float32(div))), (ratio, div)
        if C in (2, 4, 6):                                  # the same image 4 bytes off 16-byte alignment
            u = _on_device(torch, img, 1)
            got, names = launched(lambda: patches.extract_patches_device(u, ratio, plr, blr).cpu().numpy())
            _ran(names, 'extract_patches_generic_kernel')
            assert np.array_equal(_bits(got), _bits(ref)), ratio
        alloc, filled = patches.patch_counts(img.shape[0] // ratio, img.shape[1] // ratio, plr, blr)
        assert alloc == ref.shape[0]
        if filled < alloc:                                  # a range that runs into the surplus (zero) patches
            first = filled - 2
            got = patches.extract_patches_device(d, ratio, plr, blr, first, alloc - first, 2000.0).cpu().numpy()
            assert np.array_equal(_bits(got), _bits(ref[first:] / np.float32(2000)))
            assert not got[2:].any()


@pytest.mark.gpu
@pytest.mark.parametrize('C', [1, 4])
def test_extract_image_of_exactly_one_patch(torch_mod, launched, C):
    """Image + border == one patch: one filled patch, three surplus ones."""
    torch = torch_mod
    from dsen2_b200 import patches
    for img, ratio, plr, blr, ref in _extract_sources(C, seed=10 + C, g20=(12, 12), g60=(6, 6)):
        assert ref.shape[0] == 4 and ref[0].any() and not ref[1:].any()
        got, names = launched(lambda: patches.extract_patches_device(_on_device(torch, img), ratio, plr, blr).cpu().numpy())
        _ran(names, _extract_kernel(C, True))
        assert np.array_equal(_bits(got), _bits(ref)), ratio


# ---- recompose (dsen2_recompose) --------------------------------------------------------------------------------------
VEC4 = 'recompose_vec4_kernel<%d>'
# (C, P, border, H, W, pred offset, output offset, kernel).  S = P - 2 border = 24 unless noted; W mod S in {1, 2, 3}
# leaves the second-to-last patch column 1-3 owned columns, W mod S in {4, 8, 12} four or more on the vector path.
RECOMPOSE = [
    (6, 32, 4, 50, 52, 0, 0, VEC4 % 6), (6, 32, 4, 50, 56, 0, 0, VEC4 % 6), (6, 32, 4, 48, 60, 0, 0, VEC4 % 6),
    (2, 32, 4, 50, 52, 0, 0, VEC4 % 2), (2, 32, 4, 73, 76, 0, 0, VEC4 % 2),
    (1, 32, 4, 50, 52, 0, 0, 'recompose_kernel'), (3, 32, 4, 50, 52, 0, 0, 'recompose_kernel'),
    (4, 32, 4, 50, 52, 0, 0, 'recompose_kernel'),
    (6, 32, 2, 50, 60, 0, 0, 'recompose_kernel'),                                     # border % 4 != 0 (S = 28)
    (6, 32, 4, 50, 49, 0, 0, 'recompose_kernel'),                                     # W C % 4 != 0, W mod S = 1
    (2, 32, 4, 50, 51, 0, 0, 'recompose_kernel'),                                     # W C % 4 != 0, W mod S = 3
    (6, 32, 4, 50, 50, 0, 0, 'recompose_kernel'),                                     # (W - S) % 4 != 0, W mod S = 2
    (2, 32, 4, 49, 74, 0, 0, 'recompose_kernel'),                                     # (W - S) % 4 != 0, W mod S = 2
    (6, 30, 3, 50, 52, 0, 0, 'recompose_kernel'),                                     # P % 4 != 0
    (6, 32, 4, 50, 52, 0, 1, 'recompose_kernel'),                                     # output not 16-byte aligned
    (2, 32, 4, 50, 52, 1, 0, 'recompose_kernel'),                                     # input not 16-byte aligned
]


@pytest.mark.gpu
@pytest.mark.parametrize('C,P,B,H,W,pred_off,out_off,kernel', RECOMPOSE,
                         ids=['C%d-P%d-b%d-%dx%d-in%d-out%d' % c[:7] for c in RECOMPOSE])
def test_recompose_branch_bit_exact(torch_mod, launched, C, P, B, H, W, pred_off, out_off, kernel):
    """The whole canvas (NaN beforehand) from two patch ranges, against the oracle's last-writer-wins gather; mul is one
    IEEE product."""
    torch = torch_mod
    from dsen2_b200 import patches
    S = P - 2 * B
    n = -(-H // S) * -(-W // S)
    pred = (np.random.RandomState(H * W + C).rand(n, C, P, P) * 2 - 1).astype(np.float32)
    ref = po.recompose_images(pred, B, (H, W))
    k = n // 2 + 1
    for mul in (1.0, 2000.0):
        out = _nan_canvas(torch, (H, W, C), out_off)
        parts = [_on_device(torch, pred[k:], pred_off), _on_device(torch, pred[:k], pred_off)]

        def run():
            patches.recompose_device(parts[0], B, H, W, first_patch=k, mul=mul, out=out)
            patches.recompose_device(parts[1], B, H, W, first_patch=0, mul=mul, out=out)
        _, names = launched(run)
        _ran(names, kernel)
        assert np.array_equal(_bits(out.cpu().numpy()), _bits(ref * np.float32(mul))), mul


# ---- bicubic (dsen2_bicubic_imresize) ---------------------------------------------------------------------------------
def _sizes(shape, scale=None, output_shape=None):
    """(scale per axis, output size) as imresize.imresize derives them."""
    from math import ceil
    if scale is not None:
        return [float(scale)] * 2, [int(ceil(float(scale) * shape[k])) for k in range(2)]
    return [1.0 * output_shape[k] / shape[k] for k in range(2)], list(output_shape)


def bicubic_forms(shape, scale=None, output_shape=None):
    """Which form each block of dsen2_bicubic_imresize takes, restated from its dispatch in patch_kernels.cu:
    'grid-stride' (bicubic_kernel: fewer than 8 span columns fit the 40 KB intermediate) or the set of 'tiled' / 'direct'
    over the 16 x tcol output tiles of bicubic_tiled_kernel (direct: more than 8 taps on an axis, or a tile whose
    second-pass footprint spans more than span_cap input pixels)."""
    from dsen2_b200 import imresize
    h, w, C = shape
    sc, (oh, ow) = _sizes(shape, scale, output_shape)
    wy, iy = imresize.tap_tables(h, oh, sc[0])
    wx, ix = imresize.tap_tables(w, ow, sc[1])
    first = int(np.argsort(np.array(sc))[0])
    tcol = 64 if C >= 6 else (96 if C >= 3 else 128)
    span_cap = (40 * 1024 // 8) // ((16 if first == 0 else tcol) * C)
    if span_cap < 8:
        return first, {'grid-stride'}
    taps_fit = iy.shape[1] <= 8 and ix.shape[1] <= 8
    forms = set()
    for oy0 in range(0, oh, 16):
        for ox0 in range(0, ow, tcol):
            idx = ix[ox0:ox0 + tcol] if first == 0 else iy[oy0:oy0 + 16]
            forms.add('tiled' if taps_fit and idx.max() - idx.min() + 1 <= span_cap else 'direct')
    return first, forms


# (input shape, scale, output_shape, kernel name with T for the input type, forms)
BICUBIC = [
    ((60, 50, 1), 0.5, None, 'bicubic_tiled_kernel<T,true,0>', {'tiled'}),          # 8 taps: run-time tap counts
    ((60, 50, 2), 0.5, None, 'bicubic_tiled_kernel<T,true,0>', {'tiled'}),
    ((60, 50, 6), 0.5, None, 'bicubic_tiled_kernel<T,true,0>', {'tiled'}),
    ((50, 60, 1), None, (30, 30), 'bicubic_tiled_kernel<T,false,0>', {'tiled'}),    # 0.6 / 0.5: columns first
    ((60, 200, 6), 0.5, None, 'bicubic_tiled_kernel<T,true,0>', {'direct'}),        # taps fit, the span does not
    ((60, 48, 3), 1 / 3, None, 'bicubic_tiled_kernel<T,true,0>', {'direct'}),       # 9 .. 24 taps
    ((60, 48, 3), 1 / 4, None, 'bicubic_tiled_kernel<T,true,0>', {'direct'}),
    ((60, 48, 2), 1 / 6, None, 'bicubic_tiled_kernel<T,true,0>', {'direct'}),
    ((50, 40, 6), None, (20, 100), 'bicubic_tiled_kernel<T,true,0>', {'direct'}),   # 10 taps on one axis, 4 on the other
    ((30, 20, 3), 1.5, None, 'bicubic_tiled_kernel<T,true,4>', {'tiled'}),
    ((30, 20, 3), 2.5, None, 'bicubic_tiled_kernel<T,true,4>', {'tiled'}),
    ((30, 20, 3), None, (45, 50), 'bicubic_tiled_kernel<T,true,4>', {'tiled'}),     # 1.5 / 2.5: rows first
    ((30, 20, 3), None, (75, 30), 'bicubic_tiled_kernel<T,false,4>', {'tiled'}),    # 2.5 / 1.5: columns first
    ((20, 30, 48), 2, None, 'bicubic_kernel<T>', {'grid-stride'}),                  # C > 40, rows first
    ((25, 30, 11), None, (50, 45), 'bicubic_kernel<T>', {'grid-stride'}),           # C > 10, columns first
]
BICUBIC_IDS = ['%dx%dx%d-' % c[0] + ('x%.3g' % c[1] if c[1] else 'to%dx%d' % c[2]) for c in BICUBIC]


@pytest.mark.gpu
@pytest.mark.parametrize('shape,scale,output_shape,kernel,forms', BICUBIC, ids=BICUBIC_IDS)
def test_bicubic_branch_bit_exact(torch_mod, launched, shape, scale, output_shape, kernel, forms):
    """float64 products summed left to right in every branch: bit-identical to the oracle, float32 and float64 inputs."""
    from dsen2_b200 import imresize
    assert bicubic_forms(shape, scale, output_shape)[1] == forms
    x = np.random.RandomState(sum(shape)).rand(*shape) * 1e4
    for dt, T in ((np.float32, 'float'), (np.float64, 'double')):
        img = x.astype(dt)
        got, names = launched(lambda: imresize.imresize(img, scale, output_shape))
        _ran(names, kernel.replace('T', T))
        ref = io_.imresize(img, scale, output_shape)
        assert got.shape == ref.shape and got.dtype == np.float64
        assert np.array_equal(_bits(got), _bits(ref)), T


@pytest.mark.parametrize('shape,scale,output_shape', [c[:3] for c in BICUBIC], ids=BICUBIC_IDS)
def test_tap_tables_equal_oracle_contributions(shape, scale, output_shape):
    """No GPU: the device tap tables are the oracle's contributions, bit for bit."""
    from dsen2_b200 import imresize
    sc, out = _sizes(shape, scale, output_shape)
    for k in range(2):
        w, i = imresize.tap_tables(shape[k], out[k], sc[k])
        rw, ri = io_.contributions(shape[k], out[k], sc[k])
        assert w.dtype == np.float64 and i.dtype == np.int32
        assert np.array_equal(_bits(w), _bits(rw)) and np.array_equal(i, ri.astype(np.int32))


# ---- nodata scan and fill at thousands of patches (dsen2_nodata_patches, dsen2_nodata_fill[_u16]) -----------------------
# any patch / border that are multiples of r: S = 12 at 10 m gives 95 x 58 = 5510 and 50 x 43 = 2150 patches
NODATA = {20: dict(r=2, patch=16, border=2, H=1140, W=692, n=5510), 60: dict(r=6, patch=24, border=6, H=600, W=516, n=2150)}
COUNTS = [0, 1, 1023, 1024, 1025, 2048, 2049, None]                                  # None: to the last patch
FIRSTS = [0, 1, 437]


def _owner(g):
    S = g['patch'] - 2 * g['border']
    ty, _ = po.stitch_tile_of(np.arange(g['H']), g['H'], S)
    tx, nx = po.stitch_tile_of(np.arange(g['W']), g['W'], S)
    return ty[:, None] * nx + tx[None, :]


def _flag_patterns(n, rng):
    return {
        'all': np.arange(n), 'none': np.arange(0), 'alternating': np.arange(1, n, 2),
        'random': np.flatnonzero(rng.rand(n) < 0.3), 'only1023': np.array([1023]), 'only1024': np.array([1024]),
        'last': np.array([n - 1]),
        'runs': np.unique(np.concatenate([np.arange(1000, 1100), np.arange(2040, 2060), np.arange(n - 1030, n - 1010)])),
    }


def _images_with_active(g, owner, active, v, dtype, rng):
    """All inputs v except one band of one 10 m pixel, at a random place inside each active patch's owned area."""
    H, W, r = g['H'], g['W'], g['r']
    d10 = np.full((H, W, 4), v, dtype)
    d20 = np.full((H // 2, W // 2, 6), v, dtype)
    d60 = np.full((H // 6, W // 6, 2), v, dtype) if r == 6 else None
    flat = owner.ravel()
    order = np.argsort(flat, kind='stable')
    starts = np.searchsorted(flat[order], np.arange(g['n']))
    counts = np.bincount(flat, minlength=g['n'])
    if len(active):
        px = order[starts[active] + (rng.rand(len(active)) * counts[active]).astype(np.int64)]
        d10.reshape(-1, 4)[px, rng.randint(0, 4, len(px))] = v + 1
    return d10, d20, d60


def _scan(torch, lib, d, img_dtype, g, first, num, v):
    from dsen2_b200 import _capi
    ids = torch.full((max(num, 1),), -7, dtype=torch.int32, device='cuda')
    count = torch.full((1,), -7, dtype=torch.int32, device='cuda')
    rc = lib.dsen2_nodata_patches(*[_capi.ptr(t) for t in d], img_dtype, g['H'], g['W'], g['patch'], g['border'], first,
                                  num, float(v), _capi.ptr(ids), _capi.ptr(count), _capi.stream_ptr())
    _capi.check(rc, 'dsen2_nodata_patches')
    c = int(count.item())
    return ids[:c].cpu().numpy()


NODATA_CASES = [(20, np.uint16, 0.0), (20, np.float32, 777.0), (60, np.uint16, 0.0), (60, np.float32, 777.0)]
NODATA_IDS = ['%dm-%s' % (p, np.dtype(t).name) for p, t, _ in NODATA_CASES]


@pytest.mark.gpu
@pytest.mark.parametrize('path,dtype,v', NODATA_CASES, ids=NODATA_IDS)
def test_nodata_scan_thousands_of_patches(torch_mod, launched, path, dtype, v):
    """Flag patterns around the 1024-flag steps of the compaction, over ranges of 0 .. all patches from three starts:
    the ascending ids of the active patches in the range, against the oracle's mask and owner map."""
    torch = torch_mod
    from dsen2_b200 import _capi
    lib = _capi.lib()
    g = NODATA[path]
    code = _capi.IMG_U16 if dtype == np.uint16 else _capi.IMG_F32
    owner = _owner(g)
    rng = np.random.RandomState(path)
    for name, act in _flag_patterns(g['n'], rng).items():
        imgs = _images_with_active(g, owner, act, v, dtype, rng)
        _, expect, n = nodata_oracle(*imgs, v, g['patch'], g['border'])
        assert n == g['n'] and np.array_equal(expect, act), name
        d = [_on_device(torch, a) if a is not None else None for a in imgs]
        got, names = launched(lambda: _scan(torch, lib, d, code, g, 0, n, v))
        _ran(names, 'nodata_compact_kernel')
        assert np.array_equal(got, expect), name
        for first in FIRSTS:
            for num in COUNTS:
                num = n - first if num is None else num
                if first + num > n:
                    continue
                got = _scan(torch, lib, d, code, g, first, num, v)
                assert np.array_equal(got, expect[(expect >= first) & (expect < first + num)]), (name, first, num)


@pytest.mark.gpu
@pytest.mark.parametrize('path,dtype,v', NODATA_CASES, ids=NODATA_IDS)
def test_nodata_fill_thousands_of_patches(torch_mod, path, dtype, v):
    """v into exactly the nodata pixels the range owns, on float32 and uint16 canvases; every other pixel keeps the
    sentinel the canvas held."""
    torch = torch_mod
    from dsen2_b200 import _capi
    from test_gpu_nodata import make_scene
    lib = _capi.lib()
    g = NODATA[path]
    code = _capi.IMG_U16 if dtype == np.uint16 else _capi.IMG_F32
    imgs = make_scene(path, v, dtype, seed=path + 1)
    mask, _, n = nodata_oracle(*imgs, v, g['patch'], g['border'])
    assert n == g['n'] and mask.any() and not mask.all()
    owner = _owner(g)
    d = [_on_device(torch, a) if a is not None else None for a in imgs]
    cout = 6 if path == 20 else 2
    for first in FIRSTS:
        for num in COUNTS:
            num = n - first if num is None else num
            if first + num > n:
                continue
            hit = np.broadcast_to((mask & (owner >= first) & (owner < first + num))[:, :, None], (g['H'], g['W'], cout))
            f32 = torch.full((g['H'], g['W'], cout), -1.0, device='cuda')
            u16 = torch.full((g['H'], g['W'], cout), 12345, dtype=torch.int16, device='cuda')   # read as uint16
            args = [_capi.ptr(t) for t in d] + [code, g['H'], g['W'], g['patch'], g['border'], first, num, float(v), cout]
            _capi.check(lib.dsen2_nodata_fill(*args, _capi.ptr(f32), _capi.stream_ptr()), 'dsen2_nodata_fill')
            _capi.check(lib.dsen2_nodata_fill_u16(*args, _capi.ptr(u16), _capi.stream_ptr()), 'dsen2_nodata_fill_u16')
            exp32 = np.where(hit, np.float32(v), np.float32(-1)).astype(np.float32)
            exp16 = np.where(hit, np.uint16(v), np.uint16(12345)).astype(np.uint16)
            assert np.array_equal(_bits(f32.cpu().numpy()), _bits(exp32)), (first, num)
            assert np.array_equal(u16.cpu().numpy().view(np.uint16), exp16), (first, num)


@pytest.mark.gpu
def test_nodata_scan_full_tile(torch_mod, launched):
    """The production count: the 20 m scan of a 10980^2 uint16 tile (9801 patches) with a swath edge, a hole that empties
    four whole patches but one 10 m band pixel, and a lone valid pixel beyond the swath edge."""
    torch = torch_mod
    from dsen2_b200 import _capi
    T, P, B = 10980, 128, 8
    S = P - 2 * B
    g = dict(H=T, W=T, patch=P, border=B)
    gen = torch.Generator(device='cuda').manual_seed(9801)
    # int16 storage holds the uint16 values 1 .. 11999 bit for bit
    d10 = torch.randint(1, 12000, (T, T, 4), generator=gen, device='cuda', dtype=torch.int16)
    d20 = torch.randint(1, 12000, (T // 2, T // 2, 6), generator=gen, device='cuda', dtype=torch.int16)
    yc = torch.arange(T // 2, device='cuda')[:, None]
    xc = torch.arange(T // 2, device='cuda')[None, :]
    empty = xc > 0.35 * yc + 0.55 * (T // 2)                                  # on the 20 m grid
    empty[10 * S // 2:12 * S // 2, 5 * S // 2:7 * S // 2] = True              # patch rows 10-11 x columns 5-6
    d20[empty] = 0
    d10[empty.repeat_interleave(2, 0).repeat_interleave(2, 1)] = 0
    d10[11 * S + 5, 6 * S + 7, 2] = 3                                         # patch (11, 6) is active again
    d10[T - 3, T - 5, 0] = 1                                                  # beyond the swath edge
    # the oracle's rule: nodata iff every band of every input is v; owner = the last writer of the stitching
    mask = (d10 == 0).all(-1) & (d20 == 0).all(-1).repeat_interleave(2, 0).repeat_interleave(2, 1)
    ty, _ = po.stitch_tile_of(np.arange(T), T, S)
    tx, nx = po.stitch_tile_of(np.arange(T), T, S)
    owner = torch.from_numpy(ty[:, None] * nx + tx[None, :]).cuda()
    expect = torch.unique(owner[~mask]).cpu().numpy()
    del mask, owner
    assert 0 < len(expect) < 9801 and 11 * 99 + 6 in expect and 10 * 99 + 5 not in expect and 9800 in expect
    got, names = launched(lambda: _scan(torch, _capi.lib(), [d10, d20, None], _capi.IMG_U16, g, 0, 9801, 0))
    _ran(names, 'nodata_compact_kernel')
    assert np.array_equal(got, expect)
