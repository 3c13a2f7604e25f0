"""Digital-number output (``out_dtype=uint16``): the last layer writes rint(clip(f, 0, 65535)) (NaN -> 0) of the float value
f the float32 output holds, bit for bit; with ``nodata=v`` nodata pixels are v and computed values equal to v move to v + 1
(65534 for v = 65535).  The oracle is numpy applied to the float output of the same model and inputs."""
import ctypes

import numpy as np
import pytest

from test_gpu_nodata import GEOM, _dev, _model, make_scene, oracle


def quantise(f):
    """What a user does with the float output today: the numpy reference of the uint16 output."""
    return np.clip(np.rint(np.nan_to_num(f, nan=0)), 0, 65535).astype(np.uint16)


def expected(f, mask, v):
    """uint16 output with nodata=v: v on the nodata mask, q(f) elsewhere with q(f) == v moved off v."""
    e = quantise(f)
    e[(e == v) & ~mask[..., None]] = 65534 if v == 65535 else v + 1
    e[mask] = v
    return e


@pytest.fixture(scope='module')
def torch_mod():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _clamping_model(torch, path, imgs):
    """Last-layer biases moved so that on ``imgs`` about half of band 0 saturates above 65535 and half of band 1 goes
    negative (the bias adds bias x 2000 DN: each band's median moves onto the clamp); 20 m: band 2 is NaN throughout (its
    uint16 value is 0)."""
    from dsen2_b200 import supres
    model = _model(path, 'dsen2')
    f = supres.super_resolve_device(model, *_dev(torch, imgs)).cpu().numpy()
    ws = model.get_weights()
    ws[-1] = ws[-1].copy()
    ws[-1][0] += (65535.0 - np.median(f[..., 0])) / supres.SCALE
    ws[-1][1] -= np.median(f[..., 1]) / supres.SCALE
    if path == 20:
        ws[-1][2] = np.nan
    model.set_weights(ws)
    return model


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', [np.uint16, np.float32], ids=['u16-images', 'f32-images'])
@pytest.mark.parametrize('width', ['dsen2', 'vdsen2'])
@pytest.mark.parametrize('path', [20, 60])
def test_uint16_output_is_the_quantised_float_output(torch_mod, path, width, dtype):
    torch = torch_mod
    from dsen2_b200 import supres
    imgs = make_scene(path, 0, dtype, seed=11)
    model = _model(path, width)
    d = _dev(torch, imgs)
    ref = supres.super_resolve_device(model, *d).cpu().numpy()
    out = supres.super_resolve_device(model, *d, out_dtype=torch.uint16)
    assert out.dtype == torch.uint16 and tuple(out.shape) == ref.shape
    got = out.cpu().numpy()
    assert np.array_equal(got, quantise(ref))
    assert len(np.unique(got)) > 1000                          # a real spread of values, not a constant


@pytest.mark.gpu
@pytest.mark.parametrize('path', [20, 60])
def test_clamps_nan_and_half_way_values_are_exercised(torch_mod, path):
    torch = torch_mod
    from dsen2_b200 import supres
    imgs = make_scene(path, 0, np.uint16, seed=12)
    model = _clamping_model(torch, path, imgs)
    d = _dev(torch, imgs)
    ref = supres.super_resolve_device(model, *d).cpu().numpy()
    got = supres.super_resolve_device(model, *d, out_dtype=torch.uint16).cpu().numpy()
    assert np.array_equal(got, quantise(ref))
    assert (ref[..., 0] > 65535.5).any() and (got[..., 0] == 65535).any()        # saturation above
    assert (ref[..., 1] < -0.5).any() and (got[..., 1] == 0).any()              # saturation below
    assert ((got[..., :2] > 0) & (got[..., :2] < 65535)).any()
    if path == 20:
        assert np.isnan(ref[..., 2]).all() and (got[..., 2] == 0).all()
    finite = np.isfinite(ref) & (ref > 0) & (ref < 65535)
    fl = np.floor(ref[finite])
    half = (ref[finite] - fl) == 0.5
    assert (half & (fl % 2 == 0)).any() and (half & (fl % 2 == 1)).any()        # ties to even, both ways


@pytest.mark.gpu
@pytest.mark.parametrize('path,v', [(20, 0), (60, 0), (20, 4000), (20, 65535)])
def test_nodata_with_uint16_output(torch_mod, path, v):
    torch = torch_mod
    from dsen2_b200 import supres
    g = GEOM[path]
    imgs = make_scene(path, v, np.uint16, seed=13)
    mask, _active, _n = oracle(*imgs, v, g['P'], g['B'])
    assert mask.any() and not mask.all()
    model = _clamping_model(torch, path, imgs)
    d = _dev(torch, imgs)
    ref = supres.super_resolve_device(model, *d).cpu().numpy()
    got = supres.super_resolve_device(model, *d, nodata=v, out_dtype=torch.uint16).cpu().numpy()
    assert (got[mask] == v).all()
    assert np.array_equal(got, expected(ref, mask, v))
    moved = (quantise(ref) == v) & ~mask[..., None]
    if v in (0, 65535):                                         # band 1 / band 0 clamp onto v: the rule is exercised
        assert moved.any() and (got[moved] == (1 if v == 0 else 65534)).all()
    assert not (got[~mask] == v).any()


@pytest.mark.gpu
@pytest.mark.parametrize('path', [20, 60])
def test_all_nodata_scene_launches_no_network_uint16(torch_mod, path):
    torch = torch_mod
    from dsen2_b200 import supres
    g = GEOM[path]
    H, W = g['H'], g['W']
    shapes = [(H, W, 4), (H // 2, W // 2, 6)] + ([(H // 6, W // 6, 2)] if path == 60 else [])
    d = _dev(torch, [np.full(s, 9, np.uint16) for s in shapes] + ([None] if path == 20 else []))
    model = _model(path, 'dsen2')
    timers = {}
    got = supres.super_resolve_device(model, *d, nodata=9, timers=timers, out_dtype=torch.uint16).cpu().numpy()
    assert got.dtype == np.uint16 and (got == 9).all()
    assert set(timers) == {'nodata_patches', 'nodata_fill'}, sorted(timers)


@pytest.mark.gpu
@pytest.mark.parametrize('nodata', [None, 0])
def test_host_routes_on_sharded_ranges_and_facades(torch_mod, nodata):
    """Pinned ``run`` and pageable ``run_numpy`` per rank of 3 (ranges start and end inside a patch row), assembled with
    ``sharding.assemble``; half the device -> host bytes of the float32 run; then the facades."""
    torch = torch_mod
    from dsen2_b200 import sharding, supres
    g = GEOM[20]
    H, W, P, B = g['H'], g['W'], g['P'], g['B']
    d10, d20, _ = make_scene(20, 0, np.uint16, seed=14)
    model = _clamping_model(torch, 20, [d10, d20, None])
    ref = supres.super_resolve_device(model, *_dev(torch, [d10, d20]), nodata=nodata,
                                      out_dtype=torch.uint16).cpu().numpy()
    pipe = supres.HostPipeline(model, H, W, dtype=torch.uint16, chunk_patch_rows=2, out_dtype=torch.uint16)
    pipe_f = supres.HostPipeline(model, H, W, dtype=torch.uint16, chunk_patch_rows=2)
    h10, h20 = torch.from_numpy(d10).pin_memory(), torch.from_numpy(d20).pin_memory()
    parts_run, parts_np = [], []
    for r in (1, 2, 0):
        first, count = sharding.shard_range(77, r, 3)
        y0, y1 = sharding.output_rows(first, count, H, W, P, B)
        hout = pipe.run(h10, h20, first_patch=first, num_patches=count, nodata=nodata)
        torch.cuda.synchronize()
        assert hout.dtype == torch.uint16 and hout.is_pinned()
        parts_run.append((first, count, y0, hout.numpy()[y0:y1].copy(), P, B))
        pipe_f.run(h10, h20, first_patch=first, num_patches=count, nodata=nodata)
        assert pipe.d2h_bytes * 2 == pipe_f.d2h_bytes > 0
        got = pipe.run_numpy(d10, d20, first_patch=first, num_patches=count, nodata=nodata)
        assert got.dtype == np.uint16
        parts_np.append((first, count, y0, got[y0:y1].copy(), P, B))
        pipe_f.run_numpy(d10, d20, first_patch=first, num_patches=count, nodata=nodata)
        assert pipe.d2h_bytes * 2 == pipe_f.d2h_bytes > 0
    torch.cuda.synchronize()
    for parts in (parts_run, parts_np):
        assert np.array_equal(sharding.assemble(np.zeros((H, W, 6), np.uint16), parts), ref)
    fac = supres.DSen2_20(d10, d20, model=model, nodata=nodata, out_dtype=np.uint16)
    assert fac.dtype == np.uint16 and np.array_equal(fac, ref)
    out = np.full((H, W, 6), 7, np.uint16)
    assert supres.DSen2_20(d10, d20, model=model, nodata=nodata, out_dtype=np.uint16, out=out) is out
    assert np.array_equal(out, ref)
    # the float32 facade of the same model, quantised on the host, is the same product
    assert np.array_equal(quantise(supres.DSen2_20(d10, d20, model=model)),
                          supres.DSen2_20(d10, d20, model=model, out_dtype=np.uint16))


@pytest.mark.gpu
def test_facade_60m_uint16(torch_mod):
    torch = torch_mod
    from dsen2_b200 import supres
    imgs = make_scene(60, 0, np.uint16, seed=15)
    model = _clamping_model(torch, 60, imgs)
    for nodata in (None, 0):
        ref = supres.super_resolve_device(model, *_dev(torch, imgs), nodata=nodata, out_dtype=torch.uint16).cpu().numpy()
        got = supres.DSen2_60(*imgs, model=model, nodata=nodata, out_dtype=np.uint16)
        assert got.dtype == np.uint16 and np.array_equal(got, ref)


@pytest.mark.gpu
def test_tile_driver_writes_uint16(torch_mod, tmp_path):
    torch = torch_mod
    from dsen2_b200 import s2_tiles_supres as st
    from dsen2_b200 import supres
    from test_s2_tiles import D10, D20, D60
    rng = np.random.RandomState(1)
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
    m20 = _clamping_model(torch, 20, [data10, data20, None])
    m60 = _clamping_model(torch, 60, [data10, data20, np.ascontiguousarray(data60[:, :, :2])])
    assert st.main([path, out, '--output_file_format', 'npz', '--nodata', '0', '--output_dtype', 'uint16', '--run_60'],
                   models={'20': m20, '60': m60}) == 0
    z = np.load(out, allow_pickle=True)
    assert float(z['nodata']) == 0.0
    bands = list(z['bands'].item().values())
    e20 = supres.DSen2_20(data10, data20, model=m20, nodata=0, out_dtype=np.uint16)
    e60 = supres.DSen2_60(data10, data20, data60[:, :, :2], model=m60, nodata=0, out_dtype=np.uint16)
    expect = np.concatenate((e20, e60), axis=2)
    assert len(bands) == 8
    for i, band in enumerate(bands):
        assert band.dtype == np.uint16 and np.array_equal(band, expect[:, :, i])
        assert (band[:120, :150] == 0).all() and (band[120:] != 0).all()


# ---- argument checks: no GPU needed ---------------------------------------------------------------------------------
def test_u16_entry_points_reject_bad_arguments():
    from dsen2_b200 import _capi
    lib = _capi.lib()
    p = ctypes.c_void_p(256)                                   # never dereferenced: the checks come first
    U16 = _capi.IMG_U16
    args = [p] * 6 + [4, 6, 128]                               # skip_ch0 4, cout 6, feature_size 128
    # 1140 x 692 at 20 m: 77 filled patches; n = 0 returns before the device is used
    st = lib.dsen2_conv_tail16_stitch_u16
    assert st(*args, 0, 128, 0, 8, 1140, 692, 2000.0, -1, p, None) == 0
    assert st(*args, 0, 128, 0, 8, 1140, 692, 2000.0, 65535, p, None) == 0
    assert st(*args, 4, 128, 0, 8, 1140, 692, 2000.0, -1, None, None) == -1                 # null canvas
    assert st(*([None] + [p] * 5 + [4, 6, 128]), 4, 128, 0, 8, 1140, 692, 2000.0, -1, p, None) == -1
    assert st(*args, 4, 128, 0, 8, 1140, 692, 2000.0, -2, p, None) == -1                    # avoid
    assert st(*args, 4, 128, 0, 8, 1140, 692, 2000.0, 65536, p, None) == -1
    assert st(*args, 4, 128, 0, 64, 1140, 692, 2000.0, -1, p, None) == -1                   # no interior
    assert st(*args, 4, 128, 0, 8, 100, 692, 2000.0, -1, p, None) == -1                     # image < stride
    assert st(*args, 4, 128, 75, 8, 1140, 692, 2000.0, -1, p, None) == -1                   # past the 77 patches
    assert st(*([p] * 6 + [4, 6, 96]), 4, 128, 0, 8, 1140, 692, 2000.0, -1, p, None) == -1  # feature size
    assert st(*([p] * 6 + [4, 8, 128]), 4, 128, 0, 8, 1140, 692, 2000.0, -1, p, None) == -1  # cout > 7
    ids = lib.dsen2_conv_tail16_stitch_ids_u16
    assert ids(*args, 0, 128, p, 8, 1140, 692, 2000.0, 0, p, None) == 0
    assert ids(*args, 4, 128, None, 8, 1140, 692, 2000.0, 0, p, None) == -1                 # null ids
    assert ids(*args, 4, 128, p, 8, 1140, 692, 2000.0, 0, None, None) == -1
    assert ids(*args, 4, 128, p, 8, 1140, 692, 2000.0, -7, p, None) == -1
    assert ids(*args, 4, 128, p, 64, 1140, 692, 2000.0, 0, p, None) == -1
    assert ids(*args, 4, 128, p, 8, 100, 692, 2000.0, 0, p, None) == -1
    fill = lib.dsen2_nodata_fill_u16
    assert fill(p, p, None, U16, 1140, 692, 128, 8, 0, 0, 65535.0, 6, p, None) == 0
    assert fill(None, p, None, U16, 1140, 692, 128, 8, 0, 77, 0.0, 6, p, None) == -1
    assert fill(p, p, None, U16, 1140, 692, 128, 8, 0, 77, 0.0, 6, None, None) == -1
    assert fill(p, p, None, U16, 1140, 692, 128, 8, 0, 78, 0.0, 6, p, None) == -1
    assert fill(p, p, None, U16, 1140, 692, 128, 8, 0, 77, 0.0, 0, p, None) == -1
    assert fill(p, p, p, U16, 600, 520, 192, 12, 0, 8, 0.0, 2, p, None) == -1                # 520 % 6
    for bad in (2.5, 70000.0, -1.0, 65536.0, float('nan'), float('inf')):
        assert fill(p, p, None, U16, 1140, 692, 128, 8, 0, 77, bad, 6, p, None) == -1, bad
    # the float entries keep their behaviour: a non-integer nodata is fine for a float canvas
    assert lib.dsen2_nodata_fill(p, p, None, _capi.IMG_F32, 1140, 692, 128, 8, 0, 0, 2.5, 6, p, None) == 0


def test_facade_rejects_bad_output_arguments_before_touching_the_device():
    from dsen2_b200 import supres
    from dsen2_b200.DSen2Net import s2model
    model = s2model(((4, None, None), (6, None, None)), num_layers=1, feature_size=128, seed=0)
    d10, d20 = np.zeros((240, 240, 4), np.uint16), np.zeros((120, 120, 6), np.uint16)
    f10, f20 = d10.astype(np.float32), d20.astype(np.float32)
    for bad in (np.float64, np.int16, 'uint8', object, 'no such type'):
        with pytest.raises(ValueError):
            supres.DSen2_20(d10, d20, model=model, out_dtype=bad)
    for out_dtype, out in ((np.uint16, np.zeros((240, 240, 6), np.float32)),
                           (np.uint16, np.zeros((240, 240, 5), np.uint16)),
                           (np.float32, np.zeros((240, 240, 6), np.uint16)),
                           (np.float32, np.zeros((120, 240, 6), np.float32))):
        with pytest.raises(ValueError):
            supres.DSen2_20(d10, d20, model=model, out=out, out_dtype=out_dtype)
    for bad in (2.5, 70000, -1, float('nan')):
        with pytest.raises(ValueError):                         # float32 images: only uint16 output makes these invalid
            supres.DSen2_20(f10, f20, model=model, nodata=bad, out_dtype=np.uint16)
    flat = s2model(((4, None, None), (6, None, None)), num_layers=0, feature_size=128, seed=0)
    with pytest.raises(ValueError):
        supres.DSen2_20(d10, d20, model=flat, out_dtype=np.uint16)
    d60 = np.zeros((40, 40, 2), np.uint16)
    m60 = s2model(((4, None, None), (6, None, None), (2, None, None)), num_layers=1, feature_size=128, seed=0)
    with pytest.raises(ValueError):
        supres.DSen2_60(d10, d20, d60, model=m60, nodata=70000, out_dtype=np.uint16)
    with pytest.raises(ValueError):
        supres.DSen2_60(d10, d20, d60, model=m60, out=np.zeros((240, 240, 2), np.float32), out_dtype='uint16')
    with pytest.raises(ValueError):
        supres.HostPipeline(model, 240, 240, out_dtype=np.float64)
    with pytest.raises(ValueError):
        supres.HostPipeline(flat, 240, 240, out_dtype=np.uint16)


def test_check_out_dtype_accepts_numpy_and_torch_types():
    import torch
    from dsen2_b200 import supres
    for t in (None, np.float32, 'float32', torch.float32):
        assert supres.check_out_dtype(t, None) is False
    for t in (np.uint16, 'uint16', np.dtype('<u2'), torch.uint16):
        assert supres.check_out_dtype(t, None) is True
    for t in (torch.int16, torch.float64, np.float16, 3):
        with pytest.raises(ValueError):
            supres.check_out_dtype(t, None)


def test_tile_driver_parser_errors(tmp_path, capsys):
    from dsen2_b200 import s2_tiles_supres as st
    missing = str(tmp_path / 'not_there.npz')                  # the product is never opened: the parser refuses first
    for argv in (['--output_dtype', 'uint16', '--nodata', '2.5'], ['--output_dtype', 'uint16', '--nodata', '70000'],
                 ['--output_dtype', 'uint16', '--nodata', '-1'], ['--output_dtype', 'uint16', '--nodata', 'nan'],
                 ['--output_dtype', 'float32']):
        with pytest.raises(SystemExit) as e:
            st.main([missing, str(tmp_path / 'o.npz')] + argv)
        assert e.value.code == 2, argv
    assert 'uint16' in capsys.readouterr().err
    args = st.parse_args([missing, '--output_dtype', 'uint16', '--nodata', '65535'])
    assert args.output_dtype == 'uint16' and args.nodata == 65535.0
    args = st.parse_args([missing, '--nodata', '2.5'])
    assert args.output_dtype == 'float64' and args.nodata == 2.5
