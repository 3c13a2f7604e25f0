"""Radiometric offset (``add_offset=a``): every input band value x, as the device holds it, becomes fl32(x + a) before the input
preparation, and every output value f becomes fl32(f - a) before it is stored (and quantised, for uint16 output).  So
``out(imgs, add_offset=a)`` is ``out(float32(imgs) + float32(a)) - float32(a)`` in float32 numpy, bit for bit, and a
current-convention product P = S + 1000 gives ``out(P, add_offset=-1000) == out(S) + float32(1000)``."""
import ctypes

import numpy as np
import pytest

from test_gpu_nodata import GEOM, _bits, _dev, _model, make_scene, oracle
from test_gpu_u16_output import expected, quantise

A = -1000.0                                                    # RADIO_ADD_OFFSET / BOA_ADD_OFFSET of baseline 04.00


@pytest.fixture(scope='module')
def torch_mod():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _same(a, b):
    """Bit-identical: float arrays by their bits, uint16 arrays by value."""
    if a.dtype == np.float32 or b.dtype == np.float32:
        return a.dtype == b.dtype and np.array_equal(_bits(a), _bits(b))
    return a.dtype == b.dtype and np.array_equal(a, b)


def _offset_reference(torch, model, imgs, a):
    """The float path on the offset inputs float32(x) + float32(a), minus float32(a): the contract in float32 numpy."""
    from dsen2_b200 import supres
    a32 = np.float32(a)
    shifted = [None if x is None else x.astype(np.float32) + a32 for x in imgs]
    return supres.super_resolve_device(model, *_dev(torch, shifted)).cpu().numpy() - a32


def _dark_model(torch, path, imgs, target):
    """A DSen2 model whose last-layer bias of band 1 is moved so that the median of that band's float output on ``imgs`` is
    ``target`` (the bias adds bias x 2000 to the output): with target = a, half of band 1 of fl32(f - a) is negative."""
    from dsen2_b200 import supres
    model = _model(path, 'dsen2')
    f = supres.super_resolve_device(model, *_dev(torch, imgs)).cpu().numpy()
    ws = model.get_weights()
    ws[-1] = ws[-1].copy()
    ws[-1][1] += (target - np.median(f[..., 1])) / supres.SCALE
    model.set_weights(ws)
    return model


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', [np.uint16, np.float32], ids=['u16-images', 'f32-images'])
@pytest.mark.parametrize('width', ['dsen2', 'vdsen2'])
@pytest.mark.parametrize('path', [20, 60])
def test_contract_device_resident(torch_mod, path, width, dtype):
    torch = torch_mod
    from dsen2_b200 import supres
    imgs = make_scene(path, 0, dtype, seed=21)
    model = _model(path, width)
    d = _dev(torch, imgs)
    got = supres.super_resolve_device(model, *d, add_offset=A).cpu().numpy()
    assert _same(got, _offset_reference(torch, model, imgs, A))
    assert not np.array_equal(got, supres.super_resolve_device(model, *d).cpu().numpy())


@pytest.mark.gpu
@pytest.mark.parametrize('path', [20, 60])
def test_non_integer_offset_rounds_as_float32_numpy(torch_mod, path):
    """float32 images with fractional values: for the small ones x + a is not a float32 value, so the add rounds."""
    torch = torch_mod
    from dsen2_b200 import supres
    a = -999.75
    rng = np.random.RandomState(22)
    imgs = [None if x is None else x + rng.uniform(0, 1, x.shape).astype(np.float32)
            for x in make_scene(path, 0, np.float32, seed=22)]
    assert any(((x.astype(np.float64) + a) != (x + np.float32(a)).astype(np.float64)).any() for x in imgs if x is not None)
    model = _model(path, 'dsen2')
    got = supres.super_resolve_device(model, *_dev(torch, imgs), add_offset=a).cpu().numpy()
    assert _same(got, _offset_reference(torch, model, imgs, a))


@pytest.mark.gpu
@pytest.mark.parametrize('path', [20, 60])
def test_current_product_equals_old_product_plus_1000(torch_mod, path):
    """P = S + 1000 (uint16): fl32(P - 1000) is S exactly, so the network sees what it sees for S, and the output is
    out(S) + 1000.  S holds values below 1000 DN (and 0 in its empty regions), so P - 1000 is small where S is."""
    torch = torch_mod
    from dsen2_b200 import supres
    S = [x for x in make_scene(path, 0, np.uint16, seed=23) if x is not None]
    P = [x + np.uint16(1000) for x in S]
    assert all((x < 1000).any() for x in S)
    facade = supres.DSen2_20 if path == 20 else supres.DSen2_60
    model = _model(path, 'dsen2')
    got = facade(*P, model=model, add_offset=-1000)
    assert _same(got, facade(*S, model=model) + np.float32(1000))
    # uint16 output: the quantisation of out(S) + 1000; a dark band 1 makes values below -1000 in out(S) clamp at 0
    dark = _dark_model(torch, path, S + [None] * (3 - len(S)), -1000.0)
    ref = facade(*S, model=dark) + np.float32(1000)
    got = facade(*P, model=dark, add_offset=-1000, out_dtype=np.uint16)
    assert _same(got, quantise(ref))
    assert (ref < -0.5).any() and (got == 0).any() and len(np.unique(got)) > 1000


@pytest.mark.gpu
@pytest.mark.parametrize('path', [20, 60])
def test_uint16_output_with_nodata(torch_mod, path):
    """nodata=0 is decided on the stored values: the same patches run as without the offset, nodata pixels are 0, and valid
    values are the quantised fl32(f - a) with a computed 0 written as 1."""
    torch = torch_mod
    from dsen2_b200 import supres
    g = GEOM[path]
    imgs = make_scene(path, 0, np.uint16, seed=24)
    mask, active, n = oracle(*imgs, 0, g['P'], g['B'])
    assert 0 < len(active) < n
    shifted = [None if x is None else x.astype(np.float32) + np.float32(A) for x in imgs]
    model = _dark_model(torch, path, shifted, A)
    ref = _offset_reference(torch, model, imgs, A)
    d = _dev(torch, imgs)
    t_plain, t_offset = {}, {}
    supres.super_resolve_device(model, *d, nodata=0, out_dtype=torch.uint16, timers=t_plain)
    got = supres.super_resolve_device(model, *d, nodata=0, out_dtype=torch.uint16, add_offset=A,
                                      timers=t_offset).cpu().numpy()
    assert (got[mask] == 0).all()
    assert _same(got, expected(ref, mask, 0))
    moved = (quantise(ref) == 0) & ~mask[..., None]
    assert moved.any() and (got[moved] == 1).all()
    assert np.array_equal(supres.active_patches(*d, nodata=0).cpu().numpy(), active)
    patches = lambda timers: sum(k for _e0, _e1, k in timers['prep'])
    assert patches(t_offset) == patches(t_plain) == len(active)


@pytest.mark.gpu
@pytest.mark.parametrize('out_dtype', ['float32', 'uint16'])
@pytest.mark.parametrize('nodata', [None, 0])
def test_host_routes_on_sharded_ranges(torch_mod, nodata, out_dtype):
    """Pinned ``run`` and pageable ``run_numpy`` per rank of 3 (ranges start and end inside a patch row), two patch rows per
    chunk, assembled with ``sharding.assemble``, then the facade: all equal the device-resident result."""
    torch = torch_mod
    from dsen2_b200 import sharding, supres
    g = GEOM[20]
    H, W, P, B = g['H'], g['W'], g['P'], g['B']
    d10, d20, _ = make_scene(20, 0, np.uint16, seed=25)
    model = _model(20, 'dsen2')
    tdt, ndt = (torch.uint16, np.uint16) if out_dtype == 'uint16' else (torch.float32, np.float32)
    ref = supres.super_resolve_device(model, *_dev(torch, [d10, d20]), nodata=nodata, out_dtype=tdt,
                                      add_offset=A).cpu().numpy()
    pipe = supres.HostPipeline(model, H, W, dtype=torch.uint16, chunk_patch_rows=2, out_dtype=tdt)
    h10, h20 = torch.from_numpy(d10).pin_memory(), torch.from_numpy(d20).pin_memory()
    parts_run, parts_np = [], []
    for r in (1, 2, 0):
        first, count = sharding.shard_range(77, r, 3)
        y0, y1 = sharding.output_rows(first, count, H, W, P, B)
        hout = pipe.run(h10, h20, first_patch=first, num_patches=count, nodata=nodata, add_offset=A)
        torch.cuda.synchronize()
        parts_run.append((first, count, y0, hout.numpy()[y0:y1].copy(), P, B))
        got = pipe.run_numpy(d10, d20, first_patch=first, num_patches=count, nodata=nodata, add_offset=A)
        parts_np.append((first, count, y0, got[y0:y1].copy(), P, B))
    for parts in (parts_run, parts_np):
        assert _same(sharding.assemble(np.zeros((H, W, 6), ndt), parts), ref)
    assert _same(supres.DSen2_20(d10, d20, model=model, nodata=nodata, out_dtype=ndt, add_offset=A), ref)


@pytest.mark.gpu
def test_tile_driver_add_offset(torch_mod, tmp_path):
    torch = torch_mod
    from dsen2_b200 import s2_tiles_supres as st
    from dsen2_b200 import supres
    from test_s2_tiles import D10, D20, D60
    rng = np.random.RandomState(3)
    H, W = 240, 300
    data10 = rng.randint(1000, 10000, (H, W, 4)).astype(np.uint16)      # a current product: DN = 10000 x rho + 1000
    data20 = rng.randint(1000, 10000, (H // 2, W // 2, 6)).astype(np.uint16)
    data60 = rng.randint(1000, 10000, (H // 6, W // 6, 3)).astype(np.uint16)
    data10[:120, :150] = 0                                     # empty corner: 0 stays the nodata value
    data20[:60, :75] = 0
    data60[:20, :25] = 0
    path = str(tmp_path / 'product.npz')
    np.savez(path, data10=data10, data20=data20, data60=data60, desc10=np.array(D10), desc20=np.array(D20),
             desc60=np.array(D60))
    m20 = _model(20, 'dsen2')
    out = str(tmp_path / 'sr.npz')
    assert st.main([path, out, '--add_offset', '-1000', '--output_file_format', 'npz'], models={'20': m20}) == 0
    z = np.load(out, allow_pickle=True)
    assert float(z['add_offset']) == -1000.0 and 'nodata' not in z.files
    bands = list(z['bands'].item().values())
    expect = supres.DSen2_20(data10, data20, model=m20, add_offset=-1000)
    assert len(bands) == 6
    for i, band in enumerate(bands):
        assert _same(band, expect[:, :, i])
    # uint16 output with nodata, both calls (60 m and 20 m)
    m60 = _model(60, 'dsen2')
    out = str(tmp_path / 'sr16.npz')
    assert st.main([path, out, '--add_offset', '-1000', '--output_file_format', 'npz', '--output_dtype', 'uint16',
                    '--nodata', '0', '--run_60'], models={'20': m20, '60': m60}) == 0
    z = np.load(out, allow_pickle=True)
    assert float(z['add_offset']) == -1000.0 and float(z['nodata']) == 0.0
    bands = list(z['bands'].item().values())
    e20 = supres.DSen2_20(data10, data20, model=m20, nodata=0, out_dtype=np.uint16, add_offset=-1000)
    e60 = supres.DSen2_60(data10, data20, data60[:, :, :2], model=m60, nodata=0, out_dtype=np.uint16, add_offset=-1000)
    expect = np.concatenate((e20, e60), axis=2)
    assert len(bands) == 8
    for i, band in enumerate(bands):
        assert _same(band, expect[:, :, i])
        assert (band[:120, :150] == 0).all()


# ---- argument checks: no GPU needed ---------------------------------------------------------------------------------
BAD = (float('nan'), float('inf'), -float('inf'), 1e39, '-1000', b'-1000', [-1000.0], np.array([-1000.0, 0.0]), object())


def test_bad_offsets_are_rejected_before_the_device_is_touched():
    from dsen2_b200 import supres
    from dsen2_b200.DSen2Net import s2model
    model = s2model(((4, None, None), (6, None, None)), num_layers=1, feature_size=128, seed=0)
    m60 = s2model(((4, None, None), (6, None, None), (2, None, None)), num_layers=1, feature_size=128, seed=0)
    flat = s2model(((4, None, None), (6, None, None)), num_layers=0, feature_size=128, seed=0)
    d10, d20, d60 = np.zeros((240, 240, 4), np.uint16), np.zeros((120, 120, 6), np.uint16), np.zeros((40, 40, 2), np.uint16)
    pipes = {}
    for m in (model, flat):                                    # pipelines without device buffers: the check comes first
        pipes[id(m)] = supres.HostPipeline.__new__(supres.HostPipeline)
        pipes[id(m)].model = m

    def calls(m, a):
        return (lambda: supres.DSen2_20(d10, d20, model=m, add_offset=a),
                lambda: supres.DSen2_20(d10, d20, model=m, add_offset=a, nodata=0, out_dtype=np.uint16),
                lambda: supres.super_resolve_device(m, None, None, add_offset=a),
                lambda: pipes[id(m)].run_numpy(d10, d20, add_offset=a),
                lambda: pipes[id(m)].run(None, None, add_offset=a))
    for bad in BAD:
        for call in calls(model, bad):
            with pytest.raises(ValueError):
                call()
        with pytest.raises(ValueError):
            supres.DSen2_60(d10, d20, d60, model=m60, add_offset=bad)
    for call in calls(flat, -1000):
        with pytest.raises(ValueError):
            call()
    # accepted: the float32 value the kernels use
    assert supres.check_add_offset(-1000, model) == -1000.0
    assert supres.check_add_offset(np.int16(-1000), None) == -1000.0
    assert supres.check_add_offset(np.float32(-999.75), None) == -999.75
    assert supres.check_add_offset(0.1, None) == float(np.float32(0.1))
    assert supres.check_add_offset(None, flat) is None


def test_offset_entry_points_reject_bad_arguments():
    from dsen2_b200 import _capi
    lib = _capi.lib()
    p = ctypes.c_void_p(256)                                   # never dereferenced: the checks come first
    U16, F32 = _capi.IMG_U16, _capi.IMG_F32
    nonfinite = (float('nan'), float('inf'), -float('inf'))
    # 1140 x 692 at 20 m: 77 filled patches; num_patches = 0 returns before the device is used
    prep = lib.dsen2_prep16_from_images_offset
    geo = (1140, 692, 128, 8)
    assert prep(p, p, None, U16, *geo, 0, None, 0, 2000.0, A, p, p, None) == 0
    assert prep(p, p, None, U16, *geo, 5000, p, 0, 2000.0, A, p, p, None) == 0           # ids: first_patch ignored
    for bad in nonfinite:
        assert prep(p, p, None, U16, *geo, 0, None, 0, 2000.0, bad, p, p, None) == -1
        assert prep(p, p, None, U16, *geo, 0, p, 4, 2000.0, bad, p, p, None) == -1
    assert prep(None, p, None, U16, *geo, 0, None, 4, 2000.0, A, p, p, None) == -1
    assert prep(p, None, None, U16, *geo, 0, p, 4, 2000.0, A, p, p, None) == -1
    assert prep(p, p, None, U16, *geo, 0, None, 4, 2000.0, A, None, p, None) == -1
    assert prep(p, p, None, U16, *geo, 0, p, 4, 2000.0, A, p, None, None) == -1
    assert prep(p, p, None, 7, *geo, 0, None, 4, 2000.0, A, p, p, None) == -1                # image type
    assert prep(p, p, None, U16, *geo, 5000, None, 4, 2000.0, A, p, p, None) == -1           # past the patches
    assert prep(p, p, None, U16, 1140, 692, 129, 8, 0, None, 4, 2000.0, A, p, p, None) == -1  # patch size
    st = lib.dsen2_conv_tail16_stitch_offset
    args = [p] * 6 + [4, 6, 128]                               # skip_ch0 4, cout 6, feature_size 128
    assert st(*args, 0, 128, 0, None, 8, 1140, 692, 2000.0, A, F32, -1, p, None) == 0
    assert st(*args, 0, 128, 0, p, 8, 1140, 692, 2000.0, A, U16, 0, p, None) == 0
    assert st(*args, 0, 128, 0, None, 8, 1140, 692, 2000.0, A, U16, 65535, p, None) == 0
    for bad in nonfinite:
        assert st(*args, 0, 128, 0, None, 8, 1140, 692, 2000.0, bad, F32, -1, p, None) == -1
        assert st(*args, 4, 128, 0, p, 8, 1140, 692, 2000.0, bad, U16, 0, p, None) == -1
    assert st(*args, 4, 128, 0, None, 8, 1140, 692, 2000.0, A, 7, -1, p, None) == -1              # canvas_dtype
    assert st(*args, 4, 128, 0, None, 8, 1140, 692, 2000.0, A, F32, 0, p, None) == -1             # avoid, float canvas
    assert st(*args, 4, 128, 0, None, 8, 1140, 692, 2000.0, A, U16, -2, p, None) == -1
    assert st(*args, 4, 128, 0, None, 8, 1140, 692, 2000.0, A, U16, 65536, p, None) == -1
    assert st(*args, 4, 128, 0, None, 8, 1140, 692, 2000.0, A, F32, -1, None, None) == -1         # null canvas
    assert st(*([None] + [p] * 5 + [4, 6, 128]), 4, 128, 0, p, 8, 1140, 692, 2000.0, A, U16, 0, p, None) == -1
    assert st(*([p] * 5 + [None, 4, 6, 128]), 4, 128, 0, None, 8, 1140, 692, 2000.0, A, F32, -1, p, None) == -1
    assert st(*args, 4, 128, 75, None, 8, 1140, 692, 2000.0, A, F32, -1, p, None) == -1           # past the 77 patches
    assert st(*args, 4, 128, 0, p, 64, 1140, 692, 2000.0, A, U16, 0, p, None) == -1               # no interior


def test_tile_driver_add_offset_option(tmp_path):
    from dsen2_b200 import s2_tiles_supres as st
    missing = str(tmp_path / 'not_there.npz')                  # the product is never opened: the parser refuses first
    assert st.parse_args([missing, '--add_offset', '-1000']).add_offset == -1000.0
    assert st.parse_args([missing, '--add_offset=-999.75', '--output_dtype', 'uint16']).add_offset == -999.75
    assert st.parse_args([missing]).add_offset is None
    for v in ('abc', '', 'nan', 'inf', '-inf', '-1e400'):
        with pytest.raises(SystemExit) as e:
            st.main([missing, str(tmp_path / 'o.npz'), '--add_offset=' + v])
        assert e.value.code == 2, v
    text = st.build_parser().format_help()
    assert '--add_offset' in text and '04.00' in text and '-1000' in text
    out = str(tmp_path / 'bands.npz')
    st.save_npz(out, [('SRB5', np.zeros((2, 2), np.float32))], None, -1000.0)
    z = np.load(out, allow_pickle=True)
    assert float(z['add_offset']) == -1000.0 and 'nodata' not in z.files
