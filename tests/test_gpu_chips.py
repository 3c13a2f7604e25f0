"""Chip stacks: N same-size scenes (N, H, W, C) in one call.  Output chip i equals the 3-D call on chip i bit for bit, for
every option combination, also when device batches straddle chips and when a flat patch range starts and ends inside a
chip.  Without a GPU: the facade's ValueErrors and the C entry points' argument errors."""
import ctypes
import math

import numpy as np
import pytest

from test_gpu_nodata import _bits, _model

A = -1000.0
RATIO = {20: 2, 60: 6}


def make_stack(path, N, H, W, dtype, seed=0):
    """Random integer-valued DN stacks (N, H/d, W/d, C) of the 10 m, 20 m (and 60 m) bands."""
    rng = np.random.RandomState(seed)
    shapes = [(N, H, W, 4), (N, H // 2, W // 2, 6)] + ([(N, H // 6, W // 6, 2)] if path == 60 else [])
    return [rng.randint(1, 12000, size=s).astype(dtype) for s in shapes]


def _same(a, b):
    if a.dtype == np.float32 or b.dtype == np.float32:
        return a.dtype == b.dtype and a.shape == b.shape and np.array_equal(_bits(a), _bits(b))
    return a.dtype == b.dtype and np.array_equal(a, b)


def _facade(path):
    from dsen2_b200 import supres
    return supres.DSen2_20 if path == 20 else supres.DSen2_60


_models = {}


def model_for(path, width):
    if (path, width) not in _models:
        _models[(path, width)] = _model(path, width)
    return _models[(path, width)]


@pytest.fixture(scope='module')
def torch_mod():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _dev(torch, arrays):
    return [torch.from_numpy(a).cuda() for a in arrays]


def _per_chip(path, model, stack, i, **kw):
    return _facade(path)(*[x[i] for x in stack], model=model, **kw)


# ---- 1. the stack equals the per-chip calls, bit for bit ------------------------------------------------------------
GEOMETRIES = [(20, 120, 120), (20, 256, 256), (20, 120, 256), (20, 112, 112), (60, 180, 180), (60, 168, 240)]
OPTIONS = [(img, out, off) for img in (np.uint16, np.float32) for out in (np.float32, np.uint16) for off in (None, A)]


@pytest.mark.gpu
@pytest.mark.parametrize('img,out_dtype,add_offset', OPTIONS,
                         ids=['%s-in-%s-out-%s' % (np.dtype(i).name, np.dtype(o).name, 'offset' if a else 'plain')
                              for i, o, a in OPTIONS])
@pytest.mark.parametrize('path,H,W', GEOMETRIES, ids=['%dm-%dx%d' % g for g in GEOMETRIES])
def test_stack_equals_per_chip_calls(torch_mod, path, H, W, img, out_dtype, add_offset):
    torch = torch_mod
    from dsen2_b200 import supres
    model = model_for(path, 'dsen2')
    stack = make_stack(path, 3, H, W, img, seed=H + W)
    kw = dict(out_dtype=out_dtype, add_offset=add_offset)
    got = _facade(path)(*stack, model=model, **kw)
    dev = supres.super_resolve_device(model, *_dev(torch, stack), out_dtype=torch.uint16 if out_dtype == np.uint16 else None,
                                      add_offset=add_offset).cpu().numpy()
    assert got.shape == (3, H, W, model.out_channels) and got.dtype == out_dtype
    for i in range(3):
        ref = _per_chip(path, model, stack, i, **kw)
        assert _same(got[i], ref), i
        assert _same(dev[i], ref), i
    assert not _same(got[0], got[1])


@pytest.mark.gpu
@pytest.mark.parametrize('path,H,W', [(20, 120, 120), (60, 180, 180)], ids=['20m-120', '60m-180'])
@pytest.mark.parametrize('img,out_dtype,add_offset', [(np.float32, np.float32, None), (np.uint16, np.uint16, A)],
                         ids=['f32-plain', 'u16-offset'])
def test_vdsen2_stack_equals_per_chip_calls(torch_mod, path, H, W, img, out_dtype, add_offset):
    model = model_for(path, 'vdsen2')
    stack = make_stack(path, 2, H, W, img, seed=5)
    kw = dict(out_dtype=out_dtype, add_offset=add_offset)
    got = _facade(path)(*stack, model=model, **kw)
    for i in range(2):
        assert _same(got[i], _per_chip(path, model, stack, i, **kw)), i


# ---- 2. device batches and flat ranges that straddle chips -----------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('H,W,batch', [(120, 120, 7), (256, 256, 7), (120, 256, 5)])
def test_straddling_batches_and_ranks(torch_mod, H, W, batch):
    torch = torch_mod
    from dsen2_b200 import supres
    from dsen2_b200.patches import patch_counts
    model = model_for(20, 'dsen2')
    N = 5
    ppc = patch_counts(H // 2, W // 2, 64, 4)[1]
    assert batch % ppc != 0 and ppc % batch != 0
    d = _dev(torch, make_stack(20, N, H, W, np.uint16, seed=9))
    whole = supres.super_resolve_device(model, *d, add_offset=A)
    straddled = supres.super_resolve_device(model, *d, add_offset=A, device_batch=batch)
    assert _same(straddled.cpu().numpy(), whole.cpu().numpy())
    # two ranks, each half of the flat patch list: the seam lies inside a chip
    total = N * ppc
    half = total // 2
    assert half % ppc != 0
    canvas = torch.full((N, H, W, model.out_channels), float('nan'), device='cuda')
    supres.super_resolve_device(model, *d, first_patch=0, num_patches=half, out=canvas, add_offset=A, device_batch=batch)
    seam = half // ppc
    c = canvas.cpu().numpy()
    assert _same(c[:seam], whole[:seam].cpu().numpy())
    assert np.isnan(c[seam + 1:]).all()                                  # nothing written past the seam chip
    assert np.isnan(c[seam]).any() and not np.isnan(c[seam]).all()      # the seam chip: rank 0's patches only
    supres.super_resolve_device(model, *d, first_patch=half, num_patches=total - half, out=canvas, add_offset=A,
                                device_batch=batch)
    assert _same(canvas.cpu().numpy(), whole.cpu().numpy())


# ---- 3. host routes --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_pinned_pipeline_and_chunks_that_do_not_divide_the_stack(torch_mod):
    torch = torch_mod
    from dsen2_b200 import supres
    model = model_for(20, 'dsen2')
    N = 9
    stack = make_stack(20, N, 120, 120, np.uint16, seed=10)
    ref = supres.super_resolve_device(model, *_dev(torch, stack), out_dtype=torch.uint16).cpu().numpy()
    pipe = supres.ChipPipeline(model, 120, 120, chunk_chips=2, dtype=torch.uint16, out_dtype=torch.uint16)
    assert pipe.chunk == 2                                                  # 5 chunks through a ring of 3
    pinned = [torch.from_numpy(a).pin_memory() for a in stack]
    got = pipe.run(*pinned)
    torch.cuda.current_stream().synchronize()
    assert _same(got.numpy(), ref)
    out = np.full((N, 120, 120, 6), 7, np.uint16)
    res = pipe.run_numpy(*stack, out=out)
    torch.cuda.current_stream().synchronize()
    assert res is out and _same(out, ref)
    # the default chunk: 75 chips of 4 patches; 80 chips leave a chunk of 5
    N = 80
    stack = make_stack(20, N, 120, 120, np.float32, seed=11)
    ref = supres.super_resolve_device(model, *_dev(torch, stack)).cpu().numpy()
    assert supres.ChipPipeline(model, 120, 120).chunk == 75
    out = np.empty((N, 120, 120, 6), np.float32)
    res = supres.DSen2_20(*stack, model=model, out=out)
    assert res is out and _same(out, ref)


@pytest.mark.gpu
def test_single_chip_and_empty_stack(torch_mod):
    torch = torch_mod
    from dsen2_b200 import supres
    model = model_for(20, 'dsen2')
    stack = make_stack(20, 1, 256, 120, np.uint16, seed=12)
    got = supres.DSen2_20(*stack, model=model, out_dtype=np.uint16, add_offset=A)
    assert got.shape == (1, 256, 120, 6)
    assert _same(got[0], supres.DSen2_20(stack[0][0], stack[1][0], model=model, out_dtype=np.uint16, add_offset=A))
    empty = make_stack(20, 0, 120, 120, np.uint16)
    assert supres.DSen2_20(*empty, model=model).shape == (0, 120, 120, 6)
    assert tuple(supres.super_resolve_device(model, *_dev(torch, empty)).shape) == (0, 120, 120, 6)
    m60 = model_for(60, 'dsen2')
    empty60 = make_stack(60, 0, 180, 180, np.float32)
    assert supres.DSen2_60(*empty60, model=m60, out_dtype=np.uint16).dtype == np.uint16


# ---- 4. element offsets above 2^31 -----------------------------------------------------------------------------------
@pytest.mark.gpu
def test_chip_offsets_above_2_to_the_31(torch_mod):
    """40 000 uint16 chips of 120 x 120: the last chips start beyond element 2^31 of the 10 m stack (4.6 GB) and of the
    float32 output (13.8 GB).  Only the last three chips' patches run; they are random, the rest of the stack is zero."""
    torch = torch_mod
    from dsen2_b200 import supres
    model = model_for(20, 'dsen2')
    N, k = 40000, 3
    assert (N - k) * 120 * 120 * 4 > 2 ** 31 and (N - k) * 120 * 120 * 6 > 2 ** 31
    tail = make_stack(20, k, 120, 120, np.uint16, seed=13)
    d = [torch.zeros((N,) + a.shape[1:], dtype=torch.uint16, device='cuda') for a in tail]
    for t, a in zip(d, tail):
        t[N - k:] = torch.from_numpy(a).cuda()
    out = torch.empty((N, 120, 120, 6), dtype=torch.float32, device='cuda')
    supres.super_resolve_device(model, *d, first_patch=(N - k) * 4, num_patches=k * 4, out=out, add_offset=A)
    got = out[N - k:].cpu().numpy()
    del d, out
    torch.cuda.empty_cache()
    for i in range(k):
        assert _same(got[i], supres.DSen2_20(tail[0][i], tail[1][i], model=model, add_offset=A)), i


# ---- 5. the oracle on the BigEarthNet geometry -----------------------------------------------------------------------
@pytest.mark.gpu
def test_chip_of_a_stack_against_the_oracle(torch_mod):
    """120 x 120: two crops per axis whose starts are 8 px apart (0 and 8 on the 10 m grid)."""
    from dsen2_b200 import supres
    from oracle import dsen2net_oracle as no
    model = model_for(20, 'dsen2')
    stack = make_stack(20, 3, 120, 120, np.float32, seed=14)
    got = supres.DSen2_20(*stack, model=model)
    ws = model.get_weights()
    ref = no.DSen2_20(stack[0][1], stack[1][1], [(ws[2 * i], ws[2 * i + 1]) for i in range(len(ws) // 2)])
    err = float(np.abs(got[1] - ref).max()) / supres.SCALE
    assert err <= 5e-3, err


# ---- without a GPU ---------------------------------------------------------------------------------------------------
def _cpu_model(path=20, num_layers=1):
    from dsen2_b200.DSen2Net import s2model
    shape = ((4, None, None), (6, None, None)) + (((2, None, None),) if path == 60 else ())
    return s2model(shape, num_layers=num_layers, feature_size=128, seed=0)


@pytest.mark.parametrize('case', ['n-differ', 'shape', 'mixed-dtype', 'float64', 'out-shape', 'out-dtype', 'nodata',
                                  'no-resblocks', 'not-multiple', 'smaller-than-stride', '60m-120'])
def test_facade_rejects_before_the_device(case):
    from dsen2_b200 import supres
    model = _cpu_model()
    d10, d20 = make_stack(20, 3, 120, 120, np.uint16)
    kw = {}
    fn = supres.DSen2_20
    args = [d10, d20]
    if case == 'n-differ':
        args = [d10, d20[:2]]
    elif case == 'shape':
        args = [d10, d20[:, :, :58]]
    elif case == 'mixed-dtype':
        args = [d10, d20.astype(np.float32)]
    elif case == 'float64':
        args = [d10.astype(np.float64), d20.astype(np.float64)]
    elif case == 'out-shape':
        kw['out'] = np.empty((3, 120, 120, 6), np.float32)[:2]
    elif case == 'out-dtype':
        kw.update(out=np.empty((3, 120, 120, 6), np.float32), out_dtype=np.uint16)
    elif case == 'nodata':
        kw['nodata'] = 0
    elif case == 'no-resblocks':
        model = _cpu_model(num_layers=0)
    elif case == 'not-multiple':
        args = make_stack(20, 2, 121, 121, np.uint16)
        args[1] = np.zeros((2, 60, 60, 6), np.uint16)
    elif case == 'smaller-than-stride':
        args = make_stack(20, 2, 110, 110, np.uint16)
    elif case == '60m-120':
        fn, model, args = supres.DSen2_60, _cpu_model(60), make_stack(60, 2, 120, 120, np.uint16)
    with pytest.raises(ValueError):
        fn(*args, model=model, **kw)


def test_super_resolve_device_rejects_before_the_device():
    import torch
    from dsen2_b200 import supres
    model = _cpu_model()
    d10, d20 = [torch.from_numpy(a) for a in make_stack(20, 2, 120, 120, np.uint16)]
    with pytest.raises(ValueError):
        supres.super_resolve_device(model, d10, d20, nodata=0)
    with pytest.raises(ValueError):
        supres.super_resolve_device(model, d10, d20, first_patch=5, num_patches=4)        # 8 patches in the stack
    with pytest.raises(ValueError):
        supres.super_resolve_device(model, d10, d20[:1])


def test_chip_entry_points_report_argument_errors_without_a_gpu():
    from dsen2_b200 import _capi
    lib = _capi.lib()
    buf = (ctypes.c_char * 4096)()
    p = ctypes.cast(ctypes.byref(buf, 1024 - ctypes.addressof(buf) % 1024), ctypes.c_void_p)      # a non-null, aligned pointer
    U16, F32 = _capi.IMG_U16, _capi.IMG_F32

    def prep(img10=p, num_chips=3, H=120, W=120, first=0, count=12, add=0, offset=0.0, xin=p):
        return lib.dsen2_prep16_from_chips(img10, p, None, U16, num_chips, H, W, 128, 8, first, count, 2000.0, add, offset,
                                           xin, p, None)

    def tail(x_hi=p, num_chips=3, H=120, W=120, first=0, n=12, add=0, offset=0.0, canvas_dtype=F32, avoid=-1):
        return lib.dsen2_conv_tail16_stitch_chips(x_hi, p, p, p, p, p, 4, 6, 128, n, 128, first, 8, num_chips, H, W, 2000.0,
                                                  add, offset, canvas_dtype, avoid, p, None)

    for fn in (prep, tail):
        for kw, msg in [(dict(num_chips=-1), b'num_chips'),
                        (dict(first=-1), b''),
                        (dict(first=8, **({'count': 5} if fn is prep else {'n': 5})), b'outside'),   # 13 > 12 patches
                        (dict(num_chips=0, first=0, **({'count': 1} if fn is prep else {'n': 1})), b'outside'),
                        (dict(add=1, offset=math.inf), b'finite'),
                        (dict(add=1, offset=math.nan), b'finite'),
                        (dict(add=2), b'0 or 1'),
                        (dict(H=100, W=100), b''),                       # smaller than one patch stride
                        (dict(H=121, W=120), b'')]:                      # not a multiple of the ratio
            if fn is tail and 'H' in kw and kw['H'] == 121:
                continue                                                 # the canvas takes any size of at least one stride
            assert fn(**kw) == -1, (fn.__name__, kw)
            assert msg in lib.dsen2_last_error(), (fn.__name__, kw, lib.dsen2_last_error())
    assert prep(img10=None) == -1 and b'null pointer' in lib.dsen2_last_error()
    assert prep(xin=None) == -1 and b'null pointer' in lib.dsen2_last_error()
    assert tail(x_hi=None) == -1 and b'null pointer' in lib.dsen2_last_error()
    assert tail(canvas_dtype=7) == -1 and b'canvas_dtype' in lib.dsen2_last_error()
    assert tail(avoid=3) == -1 and b'avoid' in lib.dsen2_last_error()
    # 2^31 patches or more in the flat list
    assert prep(num_chips=1 << 29, first=0, count=1) == -1 and b'outside' in lib.dsen2_last_error()
    assert tail(num_chips=1 << 29, first=0, n=1) == -1 and b'outside' in lib.dsen2_last_error()
