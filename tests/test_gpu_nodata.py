"""Nodata-aware super-resolution (``nodata=v``): nodata pixels come out as v, every other pixel is bit-identical to the run
without ``nodata``, and only the patches that own a pixel with data are computed.  The oracle works from numpy masks and
the reference's stitching (``oracle.patches_oracle.recompose_images``), not from the product's tiling code."""
import ctypes

import numpy as np
import pytest

from oracle.patches_oracle import recompose_images

GEOM = {20: dict(r=2, P=128, B=8, H=1140, W=692), 60: dict(r=6, P=192, B=12, H=600, W=516)}
WIDTHS = {'dsen2': dict(num_layers=2, feature_size=128), 'vdsen2': dict(num_layers=1, feature_size=256)}


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def oracle(d10, d20, d60, v, P, B):
    """(nodata mask (H, W), ascending active patch ids): owners of valid pixels under last-writer-wins stitching."""
    m = (d10 == v).all(-1) & np.repeat(np.repeat((d20 == v).all(-1), 2, 0), 2, 1)
    if d60 is not None:
        m &= np.repeat(np.repeat((d60 == v).all(-1), 6, 0), 6, 1)
    H, W = m.shape
    S = P - 2 * B
    n = -(-H // S) * -(-W // S)
    stack = np.broadcast_to(np.arange(n, dtype=np.float32)[:, None, None, None], (n, 1, P, P))
    owner = recompose_images(stack, B, (H, W))[:, :, 0].astype(np.int64)
    return m, np.unique(owner[~m]), n


def make_scene(path, v, dtype, seed=0):
    """Random DN images with: a diagonal swath edge (empty to its right), holes inside patches, one empty patch row,
    pixels where only the 20 m input is nodata, and pixels inside empty ground where one of the four 10 m bands has data."""
    g = GEOM[path]
    r, H, W, S = g['r'], g['H'], g['W'], g['P'] - 2 * g['B']
    rng = np.random.RandomState(seed)
    d10 = rng.randint(1, 12000, size=(H, W, 4)).astype(np.float64)
    d20 = rng.randint(1, 12000, size=(H // 2, W // 2, 6)).astype(np.float64)
    d60 = rng.randint(1, 12000, size=(H // 6, W // 6, 2)).astype(np.float64) if path == 60 else None
    hc, wc = H // r, W // r                                   # the coarsest grid: empty regions are whole cells of it
    yc, xc = np.mgrid[0:hc, 0:wc]
    empty = xc > 0.35 * yc + 0.55 * wc                         # diagonal swath edge
    sc = S // r
    empty[sc:2 * sc] = True                                    # patch row 1 entirely empty
    empty[3 * sc // 4 - 6:3 * sc // 4 + 4, sc // 3:sc // 3 + 7] = True     # holes inside patch interiors
    empty[sc // 5:sc // 5 + 3, sc + sc // 2:sc + sc // 2 + 5] = True
    up = lambda a, k: np.repeat(np.repeat(a, k, 0), k, 1)
    d10[up(empty, r)] = v
    d20[up(empty, r // 2)] = v
    if d60 is not None:
        d60[empty] = v
    # only the 20 m input is nodata: these pixels have data and stay computed
    d20[20:24, 2:9] = v
    # one of four 10 m bands has data inside empty ground: inside the empty patch row and beyond the swath edge
    d10[S + S // 2:S + S // 2 + 3, S // 2:S // 2 + 2, 1] = v + 5
    d10[H - 7, W - 9, 3] = v + 1
    return [a.astype(dtype) if a is not None else None for a in (d10, d20, d60)]


@pytest.fixture(scope='module')
def torch_mod():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _model(path, width, seed=7):
    from dsen2_b200.DSen2Net import s2model
    shape = ((4, None, None), (6, None, None)) + (((2, None, None),) if path == 60 else ())
    return s2model(shape, seed=seed, **WIDTHS[width])


def _dev(torch, arrays):
    return [torch.from_numpy(a).cuda() if a is not None else None for a in arrays]


@pytest.mark.gpu
@pytest.mark.parametrize('dtype,v', [(np.uint16, 0), (np.float32, 777.0)], ids=['u16-v0', 'f32-v777'])
@pytest.mark.parametrize('width', ['dsen2', 'vdsen2'])
@pytest.mark.parametrize('path', [20, 60])
def test_contract_device_resident(torch_mod, path, width, dtype, v):
    torch = torch_mod
    from dsen2_b200 import supres
    g = GEOM[path]
    imgs = make_scene(path, v, dtype)
    mask, active, n = oracle(*imgs, v, g['P'], g['B'])
    assert 0 < len(active) < n and mask.any() and not mask.all()
    model = _model(path, width)
    d = _dev(torch, imgs)
    ref = supres.super_resolve_device(model, *d).cpu().numpy()
    got = supres.super_resolve_device(model, *d, nodata=v).cpu().numpy()
    assert np.array_equal(supres.active_patches(*d, nodata=v).cpu().numpy(), active)
    assert (got[mask] == np.float32(v)).all()
    assert np.array_equal(_bits(got[~mask]), _bits(ref[~mask]))


@pytest.mark.gpu
def test_uint16_nodata_other_than_zero_and_a_sharded_range(torch_mod):
    torch = torch_mod
    from dsen2_b200 import supres
    g = GEOM[20]
    imgs = make_scene(20, 4000, np.uint16, seed=2)
    mask, active, n = oracle(*imgs, 4000, g['P'], g['B'])
    model = _model(20, 'dsen2')
    d = _dev(torch, imgs)
    ref = supres.super_resolve_device(model, *d).cpu().numpy()
    got = supres.super_resolve_device(model, *d, nodata=4000).cpu().numpy()
    assert (got[mask] == 4000).all() and np.array_equal(_bits(got[~mask]), _bits(ref[~mask]))
    ids = supres.active_patches(*d, nodata=4000, first_patch=10, num_patches=40).cpu().numpy()
    assert np.array_equal(ids, active[(active >= 10) & (active < 50)])


@pytest.mark.gpu
def test_scene_without_nodata_pixels_is_unchanged(torch_mod):
    torch = torch_mod
    from dsen2_b200 import supres
    rng = np.random.RandomState(4)
    H, W = GEOM[20]['H'], GEOM[20]['W']
    d = _dev(torch, [rng.randint(1, 12000, size=s).astype(np.uint16) for s in ((H, W, 4), (H // 2, W // 2, 6))] + [None])
    model = _model(20, 'dsen2')
    ref = supres.super_resolve_device(model, *d).cpu().numpy()
    got = supres.super_resolve_device(model, *d, nodata=0).cpu().numpy()
    assert np.array_equal(_bits(got), _bits(ref))
    assert np.array_equal(supres.active_patches(*d, nodata=0).cpu().numpy(), np.arange(77))


@pytest.mark.gpu
@pytest.mark.parametrize('path', [20, 60])
def test_all_nodata_scene_launches_no_network(torch_mod, path):
    torch = torch_mod
    from dsen2_b200 import supres
    g = GEOM[path]
    H, W = g['H'], g['W']
    shapes = [(H, W, 4), (H // 2, W // 2, 6)] + ([(H // 6, W // 6, 2)] if path == 60 else [])
    d = _dev(torch, [np.full(s, 9, np.uint16) for s in shapes] + ([None] if path == 20 else []))
    model = _model(path, 'dsen2')
    timers = {}
    got = supres.super_resolve_device(model, *d, nodata=9, timers=timers).cpu().numpy()
    assert (got == 9).all()
    assert set(timers) == {'nodata_patches', 'nodata_fill'}, sorted(timers)
    assert supres.active_patches(*d, nodata=9).numel() == 0


@pytest.mark.gpu
def test_out_prefilled_is_entirely_written(torch_mod):
    torch = torch_mod
    from dsen2_b200 import supres
    imgs = make_scene(20, 0, np.uint16, seed=5)
    model = _model(20, 'dsen2')
    d = _dev(torch, imgs)
    ref = supres.super_resolve_device(model, *d, nodata=0).cpu().numpy()
    out = torch.full(ref.shape, -1.0, device='cuda')
    assert supres.super_resolve_device(model, *d, nodata=0, out=out) is out
    assert np.array_equal(_bits(out.cpu().numpy()), _bits(ref))


@pytest.mark.gpu
def test_host_routes_agree_on_sharded_ranges(torch_mod):
    """Pinned ``run`` and pageable ``run_numpy`` with two patch rows per chunk over ranges that start and end inside a patch
    row (what a rank of 3 owns), then the facade."""
    torch = torch_mod
    from dsen2_b200 import sharding, supres
    g = GEOM[20]
    H, W = g['H'], g['W']
    model = _model(20, 'dsen2')
    for dtype, tdtype in ((np.uint16, torch.uint16), (np.float32, torch.float32)):
        d10, d20, _ = make_scene(20, 0, dtype, seed=6)
        ref = supres.super_resolve_device(model, *_dev(torch, [d10, d20]), nodata=0).cpu().numpy()
        pipe = supres.HostPipeline(model, H, W, dtype=tdtype, chunk_patch_rows=2)
        h10, h20 = torch.from_numpy(d10).pin_memory(), torch.from_numpy(d20).pin_memory()
        hout = torch.full((H, W, 6), -1.0).pin_memory()
        got_np = np.full((H, W, 6), -1, np.float32)
        for r in (1, 2, 0):
            first, count = sharding.shard_range(77, r, 3)
            pipe.run(h10, h20, hout=hout, first_patch=first, num_patches=count, nodata=0)
            pipe.run_numpy(d10, d20, out=got_np, first_patch=first, num_patches=count, nodata=0)
        torch.cuda.synchronize()
        assert np.array_equal(_bits(hout.numpy()), _bits(ref))
        assert np.array_equal(_bits(got_np), _bits(ref))
        assert np.array_equal(_bits(supres.DSen2_20(d10, d20, model=model, nodata=0)), _bits(ref))


@pytest.mark.gpu
def test_facade_60m(torch_mod):
    torch = torch_mod
    from dsen2_b200 import supres
    imgs = make_scene(60, 0, np.uint16, seed=8)
    model = _model(60, 'dsen2')
    ref = supres.super_resolve_device(model, *_dev(torch, imgs), nodata=0).cpu().numpy()
    assert np.array_equal(_bits(supres.DSen2_60(*imgs, model=model, nodata=0)), _bits(ref))


@pytest.mark.gpu
def test_tile_driver_writes_nodata(torch_mod, tmp_path):
    from dsen2_b200 import s2_tiles_supres as st
    from dsen2_b200 import supres
    from test_s2_tiles import D10, D20, D60
    rng = np.random.RandomState(0)
    H, W = 240, 300
    data10 = rng.randint(1, 9000, (H, W, 4)).astype(np.uint16)
    data20 = rng.randint(1, 9000, (H // 2, W // 2, 6)).astype(np.uint16)
    data60 = rng.randint(1, 9000, (H // 6, W // 6, 3)).astype(np.uint16)
    data10[:120, :150] = 0                                     # empty corner
    data20[:60, :75] = 0
    data60[:20, :25] = 0
    path, out = str(tmp_path / 'product.npz'), str(tmp_path / 'sr.npz')
    np.savez(path, data10=data10, data20=data20, data60=data60, desc10=np.array(D10), desc20=np.array(D20),
             desc60=np.array(D60))
    model = _model(20, 'dsen2')
    assert st.main([path, out, '--output_file_format', 'npz', '--nodata', '0'], models={'20': model}) == 0
    z = np.load(out, allow_pickle=True)
    assert float(z['nodata']) == 0.0
    bands = z['bands'].item()
    expect = supres.DSen2_20(data10, data20, model=model, nodata=0)
    assert len(bands) == 6
    for i, (name, band) in enumerate(bands.items()):
        assert name.startswith('SR') and np.array_equal(_bits(band), _bits(expect[:, :, i]))
        assert (band[:120, :150] == 0).all() and (band[120:] != 0).any()


# ---- argument checks: no GPU needed ---------------------------------------------------------------------------------
def test_entry_points_reject_bad_arguments():
    from dsen2_b200 import _capi
    lib = _capi.lib()
    p = ctypes.c_void_p(256)                                   # never dereferenced: the checks come first
    U16 = _capi.IMG_U16
    # 1140 x 692 at 20 m: 77 filled patches
    assert lib.dsen2_nodata_patches(None, p, None, U16, 1140, 692, 128, 8, 0, 77, 0.0, p, p, None) == -1
    assert lib.dsen2_nodata_patches(p, p, None, U16, 1140, 692, 128, 8, 0, 77, 0.0, None, p, None) == -1
    assert lib.dsen2_nodata_patches(p, p, None, U16, 1140, 692, 128, 8, 0, 77, 0.0, p, None, None) == -1
    assert lib.dsen2_nodata_patches(p, p, None, U16, 1140, 692, 128, 8, 70, 8, 0.0, p, p, None) == -1   # past the end
    assert lib.dsen2_nodata_patches(p, p, None, U16, 1140, 692, 128, 8, -1, 8, 0.0, p, p, None) == -1
    assert lib.dsen2_nodata_patches(p, p, None, U16, 1141, 692, 128, 8, 0, 8, 0.0, p, p, None) == -1    # odd height
    assert lib.dsen2_nodata_patches(p, p, None, U16, 1140, 692, 128, 64, 0, 8, 0.0, p, p, None) == -1   # border
    assert lib.dsen2_nodata_patches(p, p, None, 7, 1140, 692, 128, 8, 0, 8, 0.0, p, p, None) == -1      # dtype
    assert lib.dsen2_nodata_patches(p, p, None, U16, 1140, 692, 128, 8, 0, 8, float('nan'), p, p, None) == -1
    assert lib.dsen2_nodata_fill(None, p, None, U16, 1140, 692, 128, 8, 0, 77, 0.0, 6, p, None) == -1
    assert lib.dsen2_nodata_fill(p, p, None, U16, 1140, 692, 128, 8, 0, 77, 0.0, 6, None, None) == -1
    assert lib.dsen2_nodata_fill(p, p, None, U16, 1140, 692, 128, 8, 0, 78, 0.0, 6, p, None) == -1
    assert lib.dsen2_nodata_fill(p, p, None, U16, 1140, 692, 128, 8, 0, 77, 0.0, 0, p, None) == -1
    assert lib.dsen2_nodata_fill(p, p, p, U16, 600, 520, 192, 12, 0, 8, 0.0, 2, p, None) == -1          # 520 % 6
    assert lib.dsen2_prep16_from_images_ids(p, p, None, U16, 1140, 692, 128, 8, None, 4, 2000.0, p, p, None) == -1
    assert lib.dsen2_prep16_from_images_ids(None, p, None, U16, 1140, 692, 128, 8, p, 4, 2000.0, p, p, None) == -1
    assert lib.dsen2_prep16_from_images_ids(p, p, None, U16, 1140, 692, 128, 8, p, -1, 2000.0, p, p, None) == -1
    assert lib.dsen2_prep16_from_images_ids(p, p, None, U16, 1140, 692, 129, 8, p, 4, 2000.0, p, p, None) == -1
    args = [p] * 6 + [4, 6, 128]
    assert lib.dsen2_conv_tail16_stitch_ids(*args, 4, 128, None, 8, 1140, 692, 2000.0, p, None) == -1
    assert lib.dsen2_conv_tail16_stitch_ids(*args, 4, 128, p, 64, 1140, 692, 2000.0, p, None) == -1     # no interior
    assert lib.dsen2_conv_tail16_stitch_ids(*args, 4, 128, p, 8, 100, 692, 2000.0, p, None) == -1       # image < stride
    assert lib.dsen2_conv_tail16_stitch_ids(*([p] * 5 + [None, 4, 6, 128]), 4, 128, p, 8, 1140, 692, 2000.0, p, None) == -1


def test_facade_rejects_bad_nodata_before_touching_the_device():
    from dsen2_b200 import supres
    from dsen2_b200.DSen2Net import s2model
    model = s2model(((4, None, None), (6, None, None)), num_layers=1, feature_size=128, seed=0)
    d10, d20 = np.zeros((240, 240, 4), np.uint16), np.zeros((120, 120, 6), np.uint16)
    for bad in (float('nan'), 65536, -1, 2.5):
        with pytest.raises(ValueError):
            supres.DSen2_20(d10, d20, model=model, nodata=bad)
    with pytest.raises(ValueError):
        supres.DSen2_20(d10.astype(np.float32), d20.astype(np.float32), model=model, nodata=float('nan'))
    flat = s2model(((4, None, None), (6, None, None)), num_layers=0, feature_size=128, seed=0)
    with pytest.raises(ValueError):
        supres.DSen2_20(d10, d20, model=flat, nodata=0)
    d60 = np.zeros((40, 40, 2), np.uint16)
    m60 = s2model(((4, None, None), (6, None, None), (2, None, None)), num_layers=1, feature_size=128, seed=0)
    with pytest.raises(ValueError):
        supres.DSen2_60(d10, d20, d60, model=m60, nodata=1e6)
