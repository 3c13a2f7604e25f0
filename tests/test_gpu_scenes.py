"""Scene lists: N scenes of different sizes in one call.  Output scene i equals the 3-D call on scene i bit for bit, for every
option combination, also when device batches straddle scenes and when a flat patch range starts and ends inside a scene.
Without a GPU: the facade's ValueErrors and the C entry points' argument errors."""
import ctypes
import math

import numpy as np
import pytest

from test_gpu_chips import A, _same, model_for

SIZES = {20: [(112, 112), (120, 256), (256, 120), (228, 256), (112, 1000), (600, 600)],
         60: [(168, 168), (180, 240), (336, 174)]}


def make_scenes(path, sizes, dtype, seed=0):
    """Random integer-valued DN images per scene: lists of the 10 m, 20 m (and 60 m) bands."""
    rng = np.random.RandomState(seed)
    lists = [[], []] + ([[]] if path == 60 else [])
    for H, W in sizes:
        shapes = [(H, W, 4), (H // 2, W // 2, 6)] + ([(H // 6, W // 6, 2)] if path == 60 else [])
        for l, s in zip(lists, shapes):
            l.append(rng.randint(1, 12000, size=s).astype(dtype))
    return lists


def _facade(path):
    from dsen2_b200 import supres
    return supres.DSen2_20 if path == 20 else supres.DSen2_60


def _scenes_facade(path):
    from dsen2_b200 import supres
    return supres.DSen2_20_scenes if path == 20 else supres.DSen2_60_scenes


def _per_scene(path, model, lists, i, **kw):
    return _facade(path)(*[l[i] for l in lists], model=model, **kw)


@pytest.fixture(scope='module')
def torch_mod():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _dev(torch, lists):
    return [[torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in l] for l in lists]


def _counts(path, sizes):
    from dsen2_b200.patches import patch_counts
    r = 2 if path == 20 else 6
    P, B = (128, 8) if path == 20 else (192, 12)
    return [patch_counts(H // r, W // r, P // r, B // r)[1] for H, W in sizes]


# ---- 1. the list equals the per-scene calls, bit for bit -------------------------------------------------------------
OPTIONS = [(img, out, off) for img in (np.uint16, np.float32) for out in (np.float32, np.uint16) for off in (None, A)]
OPT_IDS = ['%s-in-%s-out-%s' % (np.dtype(i).name, np.dtype(o).name, 'offset' if a else 'plain') for i, o, a in OPTIONS]


@pytest.mark.gpu
@pytest.mark.parametrize('img,out_dtype,add_offset', OPTIONS, ids=OPT_IDS)
@pytest.mark.parametrize('path', [20, 60], ids=['20m', '60m'])
def test_ragged_list_equals_per_scene_calls(torch_mod, path, img, out_dtype, add_offset):
    torch = torch_mod
    from dsen2_b200 import supres
    model = model_for(path, 'dsen2')
    sizes = SIZES[path]
    lists = make_scenes(path, sizes, img, seed=len(sizes) + path)
    kw = dict(out_dtype=out_dtype, add_offset=add_offset)
    got = _scenes_facade(path)(*lists, model=model, **kw)
    d = _dev(torch, lists)
    dev = supres.super_resolve_scenes_device(model, *d, out_dtype=torch.uint16 if out_dtype == np.uint16 else None,
                                             add_offset=add_offset)
    assert isinstance(got, list) and len(got) == len(sizes) and len(dev) == len(sizes)
    for i, (H, W) in enumerate(sizes):
        ref = _per_scene(path, model, lists, i, **kw)
        assert got[i].shape == (H, W, model.out_channels) and got[i].dtype == out_dtype
        assert _same(got[i], ref), i
        assert _same(dev[i].cpu().numpy(), ref), i


@pytest.mark.gpu
@pytest.mark.parametrize('path', [20, 60], ids=['20m', '60m'])
def test_vdsen2_list_equals_per_scene_calls(torch_mod, path):
    model = model_for(path, 'vdsen2')
    sizes = [(112, 120), (240, 112)] if path == 20 else [(168, 180), (174, 168)]
    lists = make_scenes(path, sizes, np.uint16, seed=3)
    kw = dict(out_dtype=np.uint16, add_offset=A)
    got = _scenes_facade(path)(*lists, model=model, **kw)
    for i in range(len(sizes)):
        assert _same(got[i], _per_scene(path, model, lists, i, **kw)), i


# ---- 2. device batches and flat ranges that straddle scenes ----------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('batch', [5, 7, 11])
def test_straddling_device_batches(torch_mod, batch):
    torch = torch_mod
    from dsen2_b200 import supres
    model = model_for(20, 'dsen2')
    sizes = SIZES[20]
    counts = _counts(20, sizes)
    assert all(c % batch != 0 for c in counts if c > 1)
    d = _dev(torch, make_scenes(20, sizes, np.uint16, seed=batch))
    whole = supres.super_resolve_scenes_device(model, *d, add_offset=A)
    straddled = supres.super_resolve_scenes_device(model, *d, add_offset=A, device_batch=batch)
    for i in range(len(sizes)):
        assert _same(straddled[i].cpu().numpy(), whole[i].cpu().numpy()), i


@pytest.mark.gpu
def test_range_split_inside_a_scene(torch_mod):
    """Two ranks, each a contiguous half of the flat list, on NaN-filled canvases: the seam lies inside a scene; nothing
    outside each half's owned pixels is written, and the halves together equal the whole."""
    torch = torch_mod
    from dsen2_b200 import supres
    model = model_for(20, 'dsen2')
    sizes = SIZES[20]
    counts = _counts(20, sizes)
    firsts = np.concatenate([[0], np.cumsum(counts)])
    total = int(firsts[-1])
    half = int(firsts[4]) + 3                                  # inside scene 4 (112 x 1000: 9 patches)
    seam = 4
    assert firsts[seam] < half < firsts[seam + 1]
    d = _dev(torch, make_scenes(20, sizes, np.float32, seed=21))
    whole = [o.cpu().numpy() for o in supres.super_resolve_scenes_device(model, *d)]
    outs = [torch.full((H, W, 6), float('nan'), device='cuda') for H, W in sizes]
    res = supres.super_resolve_scenes_device(model, *d, outs=outs, first_patch=0, num_patches=half, device_batch=5)
    assert res is outs
    c = [o.cpu().numpy() for o in outs]
    for i in range(seam):
        assert _same(c[i], whole[i]), i
    for i in range(seam + 1, len(sizes)):
        assert np.isnan(c[i]).all(), i                         # nothing written past the seam scene
    assert np.isnan(c[seam]).any() and not np.isnan(c[seam]).all()
    written = ~np.isnan(c[seam])
    assert _same(c[seam][written], whole[seam][written])
    supres.super_resolve_scenes_device(model, *d, outs=outs, first_patch=half, num_patches=total - half, device_batch=7)
    for i in range(len(sizes)):
        assert _same(outs[i].cpu().numpy(), whole[i]), i


# ---- 3. host routes --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_pipeline_pinned_and_numpy_with_more_chunks_than_ring_entries(torch_mod):
    torch = torch_mod
    from dsen2_b200 import supres
    model = model_for(20, 'dsen2')
    rng = np.random.RandomState(30)
    sizes = [(int(rng.randint(56, 151)) * 2, int(rng.randint(56, 151)) * 2) for _ in range(17)]
    lists = make_scenes(20, sizes, np.uint16, seed=31)
    ref = [o.cpu().numpy() for o in supres.super_resolve_scenes_device(model, *_dev(torch, lists), out_dtype=torch.uint16)]
    pipe = supres.ScenePipeline(model, chunk_patches=10, dtype=torch.uint16, out_dtype=torch.uint16)
    assert len(pipe._plan(sizes)) > 2 * pipe.RING
    pinned = [[torch.from_numpy(a).pin_memory() for a in l] for l in lists]
    got = pipe.run(*pinned)
    torch.cuda.current_stream().synchronize()
    for i in range(len(sizes)):
        assert _same(got[i].numpy(), ref[i]), i
    outs = [np.full((H, W, 6), 7, np.uint16) for H, W in sizes]
    res = pipe.run_numpy(*lists, outs=outs)
    torch.cuda.current_stream().synchronize()
    assert res is outs
    for i in range(len(sizes)):
        assert _same(outs[i], ref[i]), i
    # a larger list through the same pipeline: the buffers grow
    big = [(600, 600), (112, 1000)] + sizes[:3]
    lists = make_scenes(20, big, np.uint16, seed=32)
    res = pipe.run_numpy(*lists)
    torch.cuda.current_stream().synchronize()
    for i in range(len(big)):
        assert _same(res[i], _per_scene(20, model, lists, i, out_dtype=np.uint16)), i


@pytest.mark.gpu
def test_windows_sliced_from_one_product(torch_mod):
    """Non-contiguous numpy views: windows of different sizes cut out of one product, as around field parcels."""
    from dsen2_b200 import supres
    model = model_for(20, 'dsen2')
    d10, d20 = make_scenes(20, [(720, 840)], np.uint16, seed=40)
    d10, d20 = d10[0], d20[0]
    wins = [(0, 0, 112, 112), (100, 240, 228, 256), (360, 20, 120, 600), (480, 600, 240, 240)]
    a10 = [d10[y:y + h, x:x + w] for y, x, h, w in wins]
    a20 = [d20[y // 2:(y + h) // 2, x // 2:(x + w) // 2] for y, x, h, w in wins]
    assert not a10[1].flags.c_contiguous and not a20[1].flags.c_contiguous
    out = [np.empty((h, w, 6), np.float32) for _, _, h, w in wins]
    got = supres.DSen2_20_scenes(a10, a20, model=model, out=out, add_offset=A)
    assert got is out
    for i in range(len(wins)):
        ref = supres.DSen2_20(np.ascontiguousarray(a10[i]), np.ascontiguousarray(a20[i]), model=model, add_offset=A)
        assert _same(got[i], ref), i


@pytest.mark.gpu
def test_empty_and_single_scene_lists(torch_mod):
    torch = torch_mod
    from dsen2_b200 import supres
    model = model_for(20, 'dsen2')
    assert supres.DSen2_20_scenes([], [], model=model) == []
    assert supres.super_resolve_scenes_device(model, [], []) == []
    lists = make_scenes(20, [(256, 120)], np.uint16, seed=12)
    got = supres.DSen2_20_scenes(*lists, model=model, out_dtype=np.uint16, add_offset=A)
    assert len(got) == 1
    assert _same(got[0], _per_scene(20, model, lists, 0, out_dtype=np.uint16, add_offset=A))
    m60 = model_for(60, 'dsen2')
    assert supres.DSen2_60_scenes([], [], [], model=m60, out_dtype=np.uint16) == []


@pytest.mark.gpu
def test_equal_size_list_equals_the_chip_stack(torch_mod):
    from dsen2_b200 import supres
    model = model_for(20, 'dsen2')
    lists = make_scenes(20, [(120, 120)] * 5, np.float32, seed=50)
    got = supres.DSen2_20_scenes(*lists, model=model, out_dtype=np.uint16)
    stack = supres.DSen2_20(np.stack(lists[0]), np.stack(lists[1]), model=model, out_dtype=np.uint16)
    for i in range(5):
        assert _same(got[i], stack[i]), i


@pytest.mark.gpu
def test_scene_of_a_list_against_the_oracle(torch_mod):
    from dsen2_b200 import supres
    from oracle import dsen2net_oracle as no
    model = model_for(20, 'dsen2')
    lists = make_scenes(20, [(112, 112), (120, 256), (228, 120)], np.float32, seed=60)
    got = supres.DSen2_20_scenes(*lists, model=model)
    ws = model.get_weights()
    ref = no.DSen2_20(lists[0][1], lists[1][1], [(ws[2 * i], ws[2 * i + 1]) for i in range(len(ws) // 2)])
    err = float(np.abs(got[1] - ref).max()) / supres.SCALE
    assert err <= 5e-3, err


# ---- without a GPU ---------------------------------------------------------------------------------------------------
def _cpu_model(path=20, num_layers=1):
    from dsen2_b200.DSen2Net import s2model
    shape = ((4, None, None), (6, None, None)) + (((2, None, None),) if path == 60 else ())
    return s2model(shape, num_layers=num_layers, feature_size=128, seed=0)


@pytest.mark.parametrize('case', ['lengths-differ', 'shape', 'not-hwc', 'mixed-in-scene', 'mixed-across-scenes', 'float64',
                                  'not-multiple', 'smaller-than-stride', '60m-120', 'out-length', 'out-shape',
                                  'out-dtype', 'nodata', 'no-resblocks'])
def test_facade_rejects_before_the_device(case):
    from dsen2_b200 import supres
    model = _cpu_model()
    d10s, d20s = make_scenes(20, [(120, 256), (112, 112)], np.uint16)
    kw = {}
    fn = supres.DSen2_20_scenes
    args = [d10s, d20s]
    if case == 'lengths-differ':
        args = [d10s, d20s[:1]]
    elif case == 'shape':
        args = [d10s, [d20s[0], d20s[1][:, :54]]]
    elif case == 'not-hwc':
        args = [[d10s[0], d10s[1][None]], d20s]
    elif case == 'mixed-in-scene':
        args = [d10s, [d20s[0], d20s[1].astype(np.float32)]]
    elif case == 'mixed-across-scenes':
        args = [[d10s[0], d10s[1].astype(np.float32)], [d20s[0], d20s[1].astype(np.float32)]]
    elif case == 'float64':
        args = [[a.astype(np.float64) for a in d10s], [a.astype(np.float64) for a in d20s]]
    elif case == 'not-multiple':
        args = [[d10s[0], np.zeros((121, 120, 4), np.uint16)], [d20s[0], np.zeros((60, 60, 6), np.uint16)]]
    elif case == 'smaller-than-stride':
        args = make_scenes(20, [(120, 120), (110, 200)], np.uint16)
    elif case == '60m-120':
        fn, model, args = supres.DSen2_60_scenes, _cpu_model(60), make_scenes(60, [(180, 180), (120, 180)], np.uint16)
    elif case == 'out-length':
        kw['out'] = [np.empty((120, 256, 6), np.float32)]
    elif case == 'out-shape':
        kw['out'] = [np.empty((120, 256, 6), np.float32), np.empty((112, 114, 6), np.float32)]
    elif case == 'out-dtype':
        kw.update(out=[np.empty((120, 256, 6), np.float32), np.empty((112, 112, 6), np.float32)], out_dtype=np.uint16)
    elif case == 'nodata':
        kw['nodata'] = 0
    elif case == 'no-resblocks':
        model = _cpu_model(num_layers=0)
    with pytest.raises(ValueError):
        fn(*args, model=model, **kw)


def test_device_facade_rejects_before_the_device():
    import torch
    from dsen2_b200 import supres
    model = _cpu_model()
    d10s, d20s = [[torch.from_numpy(a) for a in l] for l in make_scenes(20, [(120, 120), (112, 240)], np.uint16)]
    with pytest.raises(ValueError):
        supres.super_resolve_scenes_device(model, d10s, d20s[:1])
    with pytest.raises(ValueError):
        supres.super_resolve_scenes_device(model, d10s, [d20s[0], d20s[1][:, :100]])
    with pytest.raises(ValueError):
        supres.super_resolve_scenes_device(model, d10s, d20s, outs=[torch.empty((120, 120, 6))])
    with pytest.raises(ValueError):
        supres.super_resolve_scenes_device(model, d10s, d20s)              # CPU tensors


def _pp(vals, t=ctypes.c_void_p):
    return (t * len(vals))(*vals)


def test_scene_table_reports_argument_errors_without_a_gpu():
    from dsen2_b200 import _capi
    lib = _capi.lib()
    assert lib.dsen2_scene_table_bytes(0) == 0 and lib.dsen2_scene_table_bytes(3) == 3 * lib.dsen2_scene_table_bytes(1) > 0
    table = (ctypes.c_char * (lib.dsen2_scene_table_bytes(3) + 1))()
    total = ctypes.c_longlong(-1)

    def build(Hs=(120, 112, 256), Ws=(256, 112, 120), img10=1, img60=False, patch=128, border=8, pmap=None, cap=0, n=3,
              tot=True):
        p = lambda v: _pp([v] * 3)
        return lib.dsen2_scene_table(n, p(img10), p(2), p(3) if img60 else None, p(4), _pp(Hs, ctypes.c_int),
                                     _pp(Ws, ctypes.c_int), patch, border, table, pmap, cap,
                                     ctypes.byref(total) if tot else None)

    assert build() == 0 and total.value == 6 + 1 + 6                        # 2 x 3, 1 x 1, 3 x 2 patches
    pmap = (ctypes.c_int * 13)()
    assert build(pmap=pmap, cap=13) == 0 and list(pmap) == [0] * 6 + [1] + [2] * 6
    assert build(n=0) == 0 and total.value == 0
    for kw, msg in [(dict(n=-1), b'num_scenes'),
                    (dict(img10=0), b'scene 0: null pointer'),
                    (dict(tot=False), b'null pointer'),
                    (dict(Hs=(120, 113, 256)), b'scene 1: 10 m size'),
                    (dict(Hs=(120, 112, 110)), b'scene 2: image'),
                    (dict(Hs=(120, 112, 180), img60=True, patch=192, border=12), b'scene 0'),      # 256 % 6
                    (dict(patch=129), b'multiples'),
                    (dict(pmap=pmap, cap=12), b'map')]:
        assert build(**kw) == -1, kw
        assert msg in lib.dsen2_last_error(), (kw, lib.dsen2_last_error())


def test_scene_entry_points_report_argument_errors_without_a_gpu():
    from dsen2_b200 import _capi
    lib = _capi.lib()
    buf = (ctypes.c_char * 4096)()
    p = ctypes.cast(ctypes.byref(buf, 1024 - ctypes.addressof(buf) % 1024), ctypes.c_void_p)      # a non-null, aligned pointer
    U16, F32 = _capi.IMG_U16, _capi.IMG_F32

    def prep(table=p, num_scenes=3, total=12, first=0, count=12, add=0, offset=0.0, xin=p, img_dtype=U16):
        return lib.dsen2_prep16_from_scenes(table, p, num_scenes, total, img_dtype, 0, 128, 8, first, count, 2000.0, add,
                                            offset, xin, p, None)

    def tail(table=p, num_scenes=3, total=12, first=0, n=12, add=0, offset=0.0, canvas_dtype=F32, avoid=-1, x_hi=p):
        return lib.dsen2_conv_tail16_stitch_scenes(x_hi, p, p, p, p, p, 4, 6, 128, n, 128, first, 8, table, p, num_scenes,
                                                   total, 2000.0, add, offset, canvas_dtype, avoid, None)

    for fn in (prep, tail):
        cnt = 'count' if fn is prep else 'n'
        for kw, msg in [(dict(num_scenes=-1), b'num_scenes'),
                        (dict(table=None), b'null pointer'),
                        (dict(first=-1), b'outside'),
                        (dict(first=8, **{cnt: 5}), b'outside'),               # 13 > 12 patches
                        (dict(total=0, **{cnt: 1}), b'outside'),
                        (dict(total=1 << 31, **{cnt: 1}), b'outside'),
                        (dict(add=1, offset=math.inf), b'finite'),
                        (dict(add=1, offset=math.nan), b'finite'),
                        (dict(add=2), b'0 or 1')]:
            assert fn(**kw) == -1, (fn.__name__, kw)
            assert msg in lib.dsen2_last_error(), (fn.__name__, kw, lib.dsen2_last_error())
    assert prep(xin=None) == -1 and b'null pointer' in lib.dsen2_last_error()
    assert prep(img_dtype=5) == -1 and b'img_dtype' in lib.dsen2_last_error()
    assert tail(x_hi=None) == -1 and b'null pointer' in lib.dsen2_last_error()
    assert tail(canvas_dtype=7) == -1 and b'canvas_dtype' in lib.dsen2_last_error()
    assert tail(avoid=3) == -1 and b'avoid' in lib.dsen2_last_error()
