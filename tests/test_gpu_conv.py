"""tcgen05 convolution path against the fp32 CPU oracle (oracle/dsen2net_oracle.py).

Tolerances: single layers are compared with a CPU convolution of the SAME fp16-rounded operands
(only the fp32 accumulation order and the final fp16 rounding differ): rtol 2e-3 / atol 2e-3.
Whole networks are held to the north-star gate: max |err| <= 5e-3 on the /2000-scaled output.
"""
import ctypes

import numpy as np
import pytest

import tile_schedule as ts

pytestmark = pytest.mark.gpu

GATE = 5e-3


@pytest.fixture(scope='module')
def env():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from dsen2_b200 import _capi
    return torch, _capi, _capi.lib()


def _conv_ref(torch, x_nhwc, w_hwio, bias):
    """fp32 conv of fp16-rounded operands; x (n,H,W,C) -> (n,H,W,Cout)."""
    import torch.nn.functional as F
    x = torch.from_numpy(x_nhwc.astype(np.float32)).permute(0, 3, 1, 2)
    w = torch.from_numpy(w_hwio.astype(np.float16).astype(np.float32)).permute(3, 2, 0, 1).contiguous()
    y = F.conv2d(x, w, torch.from_numpy(bias), padding=w_hwio.shape[0] // 2)
    return y.permute(0, 2, 3, 1).contiguous().numpy()


def _pack(torch, _capi, lib, w_hwio, cin_pad, cout_pad):
    cin, cout = w_hwio.shape[2], w_hwio.shape[3]
    src = torch.from_numpy(np.ascontiguousarray(w_hwio)).cuda()
    dst = torch.empty((9, cout_pad, cin_pad), dtype=torch.float16, device='cuda')
    _capi.check(lib.dsen2_pack_conv_weights(_capi.ptr(src), cin, cout, cin_pad, cout_pad, _capi.ptr(dst),
                                            _capi.stream_ptr()), 'pack')
    return dst


@pytest.mark.parametrize('shape', [(2, 32, 32), (1, 128, 128), (1, 192, 192), (3, 40, 24), (1, 8, 200), (5, 16, 8), ts.PATCH,
                                   ts.RAGGED])
@pytest.mark.parametrize('F', [128, 256])
def test_conv_relu_layer(env, shape, F):
    """First convolution of a resBlock (DSen2Net.py:10-11) for F = 128 (resident weights) and 256 (streamed weights); the
    ts.PATCH / ts.RAGGED cases run several tiles per CTA pair, as real runs do."""
    torch, _capi, lib = env
    n, H, W = shape
    rng = np.random.RandomState(H * 7 + W + F)
    x = (rng.randn(n, H, W, F).astype(np.float32)).astype(np.float16)
    lim = np.sqrt(6.0 / (9 * F))
    w = rng.uniform(-lim, lim, size=(3, 3, F, F)).astype(np.float32)
    bias = rng.randn(F).astype(np.float32) * 0.1
    tx = torch.from_numpy(x).cuda()
    tw = _pack(torch, _capi, lib, w, F, F)
    tb = torch.from_numpy(bias).cuda()
    out = torch.zeros((n, H, W, F), dtype=torch.float16, device='cuda')
    _capi.check(lib.dsen2_conv_relu(_capi.ptr(tx), _capi.ptr(tw), _capi.ptr(tb), n, H, W, F, _capi.ptr(out),
                                    _capi.stream_ptr()), 'conv relu')
    torch.cuda.synchronize()
    ref = np.maximum(_conv_ref(torch, x, w, bias), 0)
    got = out.cpu().numpy().astype(np.float32)
    ts.check(ts.pair_schedule(n, H, W), 'conv_relu F=%d' % F, np.abs(got - ref).max())
    np.testing.assert_allclose(got, ref, rtol=2e-3, atol=2e-3)
    assert lib.dsen2_conv_relu(_capi.ptr(tx), _capi.ptr(tw), _capi.ptr(tb), n, H, W, 192, _capi.ptr(out),
                               _capi.stream_ptr()) == -1                              # unsupported feature size is refused


@pytest.mark.parametrize('cfg', [dict(inp=(4, 6), L=2, F=128, P=32, n=3), dict(inp=(4, 6), L=6, F=128, P=128, n=2),
                                 dict(inp=(4, 6, 2), L=6, F=128, P=192, n=1), dict(inp=(4, 6), L=3, F=256, P=64, n=2)])
def test_s2model_predict_vs_oracle(env, cfg):
    from dsen2_b200.DSen2Net import s2model
    from oracle import dsen2net_oracle as no
    rng = np.random.RandomState(11)
    shape = tuple((c, None, None) for c in cfg['inp'])
    model = s2model(shape, num_layers=cfg['L'], feature_size=cfg['F'], seed=3)
    # non-zero biases so the bias path is exercised
    ws = model.get_weights()
    for i in range(1, len(ws), 2):
        ws[i] = (rng.randn(*ws[i].shape) * 0.05).astype(np.float32)
    model.set_weights(ws)
    xs = [(0.8 + 0.45 * rng.randn(cfg['n'], c, cfg['P'], cfg['P'])).clip(0, 6).astype(np.float32) for c in cfg['inp']]
    got = model.predict(xs)
    ref = no.predict(xs, [(ws[2 * i], ws[2 * i + 1]) for i in range(len(ws) // 2)])
    assert got.shape == ref.shape and got.dtype == np.float32
    err = np.abs(got - ref).max()
    print('max abs err', err, 'rms', np.sqrt(np.mean((got - ref) ** 2)))
    assert err <= GATE


@pytest.mark.parametrize('cfg', [dict(inp=(4, 6), L=2, F=128, P=64, n=3), dict(inp=(4, 6, 2), L=1, F=128, P=48, n=2),
                                 dict(inp=(4, 6), L=1, F=256, P=32, n=2), dict(inp=(4, 6), L=0, F=128, P=32, n=2)])
def test_c_entry_point_whole_forward(env, cfg):
    """dsen2_s2model_forward (the one-call C entry) == the per-layer sequence the Python host issues."""
    torch, _capi, lib = env
    from dsen2_b200.DSen2Net import s2model
    rng = np.random.RandomState(5)
    model = s2model(tuple((c, None, None) for c in cfg['inp']), num_layers=cfg['L'], feature_size=cfg['F'], seed=2)
    xs = [torch.from_numpy((0.8 + 0.4 * rng.randn(cfg['n'], c, cfg['P'], cfg['P'])).clip(0, 5).astype(np.float32)).cuda()
          for c in cfg['inp']]
    a = model.forward_device(xs).clone()
    b = model.forward_c(xs)
    torch.cuda.synchronize()
    assert torch.equal(a, b)


def test_DSen2_20_and_60_scene_vs_oracle(env, scene):
    """Both scenes of the reference's data/ directory that are present (Malmo, Shark Bay), 20 m and 60 m path."""
    from dsen2_b200 import supres
    from dsen2_b200.DSen2Net import s2model
    from oracle import dsen2net_oracle as no
    name, d10, d20, d60 = scene
    for run_60 in (False, True):
        shape = ((4, None, None), (6, None, None)) + (((2, None, None),) if run_60 else ())
        model = s2model(shape, num_layers=6, feature_size=128, seed=0)
        ws = model.get_weights()
        wl = [(ws[2 * i], ws[2 * i + 1]) for i in range(len(ws) // 2)]
        if run_60:
            got = supres.DSen2_60(d10, d20, d60, model=model)
            ref = no.DSen2_60(d10, d20, d60, wl)
            assert got.shape == (600, 600, 2)
        else:
            got = supres.DSen2_20(d10, d20, model=model)
            ref = no.DSen2_20(d10, d20, wl)
            assert got.shape == (600, 600, 6)
        assert got.dtype == np.float32
        err = np.abs(got - ref).max() / supres.SCALE
        print(name, 'run_60', run_60, 'max abs err (scaled)', err)
        assert err <= GATE


@pytest.mark.parametrize('seed', [11, 12, 13])
def test_DSen2_60_synthetic_scenes_vs_oracle(env, seed):
    """BASELINE config 2 names five 600 x 600 scenes for the 60 m path; two exist in the mount (above), the other three are
    seeded synthetic scenes with the dynamic range of the real ones (uint16 DN, smooth field + noise)."""
    from dsen2_b200 import supres
    from dsen2_b200.DSen2Net import s2model
    from oracle import dsen2net_oracle as no
    rng = np.random.RandomState(seed)

    def field(h, w, c):
        lo = rng.randn(h // 50 + 2, w // 50 + 2, c)
        up = np.kron(lo, np.ones((50, 50, 1)))[:h, :w]
        return np.clip(1600 + 900 * up + 150 * rng.randn(h, w, c), 0, 12000).round().astype(np.uint16)
    d10, d20, d60 = field(600, 600, 4), field(300, 300, 6), field(100, 100, 2)
    model = s2model(((4, None, None), (6, None, None), (2, None, None)), num_layers=6, feature_size=128, seed=seed)
    ws = model.get_weights()
    got = supres.DSen2_60(d10, d20, d60, model=model)                     # uint16 in, as GDAL delivers
    ref = no.DSen2_60(d10.astype(np.float32), d20.astype(np.float32), d60.astype(np.float32),
                      [(ws[2 * i], ws[2 * i + 1]) for i in range(len(ws) // 2)])
    err = np.abs(got - ref).max() / supres.SCALE
    print('synthetic scene', seed, 'max abs err (scaled)', err)
    assert got.shape == (600, 600, 2) and err <= GATE


def test_rmse_gate_on_the_shipped_scenes_when_the_blobs_exist(env):
    """The north-star acceptance gate: DSen2 RMSE against the simulated ground truth within 0.5 % of the notebook's recorded
    values (Running_Demo_in_the_colab.ipynb:170,209,236).  The three ground-truth scenes and both weight files are listed
    in the reference's .MISSING_LARGE_BLOBS and far larger than a test fixture, so this is skipped until they are supplied
    (directories named by DSEN2_DATA and DSEN2_MODELS)."""
    import os
    from dsen2_b200 import demoDSen2, supres
    data, models = os.environ.get('DSEN2_DATA', ''), os.environ.get('DSEN2_MODELS', '')
    if not data or not models:
        pytest.skip("DSEN2_DATA / DSEN2_MODELS do not name the ground-truth scenes and shipped weights")
    cases = [('S2B_MSIL1C_20170725_T43WFQ.mat', False, 31.2404), ('S2A_MSIL1C_20171028_T34HCH.mat', True, 20.4089),
             ('S2B_MSIL1C_20170928_T18TWL.mat', False, 64.2276)]
    weights = [os.path.join(models, f) for f in ('s2_032_lr_1e-04.hdf5', 's2_030_lr_1e-05.hdf5')]
    have = [c for c in cases if os.path.exists(os.path.join(data, c[0]))]
    if not have or not all(os.path.exists(w) for w in weights):
        pytest.skip("ground-truth scenes / shipped weights are missing blobs in this mount")
    old, old_data = supres.MDL_PATH, demoDSen2.DATA_PATH
    supres.MDL_PATH, demoDSen2.DATA_PATH = models.rstrip('/') + '/', data.rstrip('/') + '/'
    try:
        for fn, run_60, expected in have:
            if run_60:
                d10, d20, d60, gt = demoDSen2.readh5(fn, im60=True, imGT=True)
                sr = supres.DSen2_60(d10, d20, d60)
            else:
                d10, d20, gt = demoDSen2.readh5(fn, imGT=True)
                sr = supres.DSen2_20(d10, d20)
            rmse = demoDSen2.RMSE(sr, gt)
            print(fn, 'RMSE', rmse, 'notebook', expected)
            assert abs(rmse - expected) <= 0.005 * expected
    finally:
        supres.MDL_PATH, demoDSen2.DATA_PATH = old, old_data


def test_tile_driver_on_an_npz_product(env, tmp_path):
    """python -m dsen2_b200.s2_tiles_supres end to end (ROI, 60 m then 20 m network, npz output) == the facade calls on the
    same windows (testing/s2_tiles_supres.py:311-342,385-420)."""
    from dsen2_b200 import s2_tiles_supres as st, supres
    from dsen2_b200.DSen2Net import s2model
    rng = np.random.RandomState(2)
    H, W = 360, 420
    desc10 = ["B4, central wavelength 665 nm", "B3, central wavelength 560 nm", "B2, central wavelength 490 nm",
              "B8, central wavelength 842 nm"]
    desc20 = ["B%s, central wavelength %d nm" % b for b in (('5', 705), ('6', 740), ('7', 783), ('8A', 865), ('11', 1610), ('12', 2190))]
    desc60 = ["B1, central wavelength 443 nm", "B9, central wavelength 945 nm", "B10, central wavelength 1375 nm"]
    prod = str(tmp_path / 'p.npz')
    np.savez(prod, data10=rng.randint(0, 9000, (H, W, 4)).astype(np.uint16), data20=rng.randint(0, 9000, (H // 2, W // 2, 6)).astype(np.uint16),
             data60=rng.randint(0, 9000, (H // 6, W // 6, 3)).astype(np.uint16), desc10=np.array(desc10), desc20=np.array(desc20),
             desc60=np.array(desc60))
    models = {'20': s2model(((4, None, None), (6, None, None)), num_layers=1, feature_size=128, seed=1),
              '60': s2model(((4, None, None), (6, None, None), (2, None, None)), num_layers=1, feature_size=128, seed=2)}
    out = str(tmp_path / 'o.npz')
    assert st.main([prod, out, '--roi_x_y', '20,10,400,340', '--run_60', '--output_file_format', 'npz'], models=models) == 0
    bands = np.load(out, allow_pickle=True)['bands'].item()
    z = np.load(prod)
    xmin, ymin, xmax, ymax = st.clamp_roi(20., 10., 400., 340., W, H)
    w10, w20, w60 = st.read_windows(xmin, ymin, xmax, ymax)
    cut = lambda a, w, idx: np.ascontiguousarray(a[w[1]:w[1] + w[3], w[0]:w[0] + w[2]][:, :, idx])
    d10, d20, d60 = cut(z['data10'], w10, [0, 1, 2, 3]), cut(z['data20'], w20, list(range(6))), cut(z['data60'], w60, [0, 1])
    sr20 = supres.DSen2_20(d10, d20, model=models['20'])
    sr60 = supres.DSen2_60(d10, d20, d60, model=models['60'])
    assert list(bands) == ['SRB5 (705 nm)', 'SRB6 (740 nm)', 'SRB7 (783 nm)', 'SRB8A (865 nm)', 'SRB11 (1610 nm)', 'SRB12 (2190 nm)',
                           'SRB1 (443 nm)', 'SRB9 (945 nm)']
    assert np.array_equal(bands['SRB7 (783 nm)'], sr20[:, :, 2]) and np.array_equal(bands['SRB9 (945 nm)'], sr60[:, :, 1])


def test_VDSen2_depth32_scene_vs_oracle(env):
    """VDSen2 at its real depth (32 resblocks x 256 features, supres.py:55-57 deep=True shapes) through the facade:
    DSen2_20 on a 220 x 220 scene (4 patches of 128) and DSen2_60 on a 180 x 180 scene (4 patches of 192) -- sizes whose
    allocated patch stack has no surplus zero patches for the CPU oracle to grind through -- he_uniform weights with
    non-zero biases, against the fp32 CPU oracle.  Gate 5e-3 on the /2000-scaled output."""
    from dsen2_b200 import supres
    from dsen2_b200.DSen2Net import s2model
    from oracle import dsen2net_oracle as no
    rng = np.random.RandomState(32)
    for run_60, (H, W) in ((False, (220, 220)), (True, (180, 180))):
        shape = ((4, None, None), (6, None, None)) + (((2, None, None),) if run_60 else ())
        model = s2model(shape, num_layers=32, feature_size=256, seed=1)
        ws = model.get_weights()
        for i in range(1, len(ws), 2):
            ws[i] = (rng.randn(*ws[i].shape) * 0.02).astype(np.float32)
        model.set_weights(ws)
        wl = [(ws[2 * i], ws[2 * i + 1]) for i in range(len(ws) // 2)]
        d10 = rng.randint(200, 6000, size=(H, W, 4)).astype(np.float32)
        d20 = rng.randint(200, 6000, size=(H // 2, W // 2, 6)).astype(np.float32)
        if run_60:
            d60 = rng.randint(200, 6000, size=(H // 6, W // 6, 2)).astype(np.float32)
            got, ref = supres.DSen2_60(d10, d20, d60, model=model), no.DSen2_60(d10, d20, d60, wl)
            assert got.shape == (H, W, 2)
        else:
            got, ref = supres.DSen2_20(d10, d20, model=model), no.DSen2_20(d10, d20, wl)
            assert got.shape == (H, W, 6)
        err = np.abs(got - ref).max() / supres.SCALE
        print('VDSen2 32x256 run_60', run_60, 'max abs err (scaled)', err, 'output range', ref.min() / supres.SCALE,
              ref.max() / supres.SCALE)
        assert err <= GATE


def test_DSen2_20_single_filled_patch_is_stitched_and_cropped(env):
    """112 x 112 (golden case 'c'): one filled patch of four allocated -> recompose_images crops it (patches.py:375 keys
    on the allocated count); the facade must return (112, 112, 6), not the uncropped 128 x 128 patch."""
    from dsen2_b200 import supres
    from dsen2_b200.DSen2Net import s2model
    from oracle import dsen2net_oracle as no
    rng = np.random.RandomState(7)
    d10 = rng.randint(200, 6000, size=(112, 112, 4)).astype(np.float32)
    d20 = rng.randint(200, 6000, size=(56, 56, 6)).astype(np.float32)
    model = s2model(((4, None, None), (6, None, None)), num_layers=2, feature_size=128, seed=4)
    ws = model.get_weights()
    got = supres.DSen2_20(d10, d20, model=model)
    ref = no.DSen2_20(d10, d20, [(ws[2 * i], ws[2 * i + 1]) for i in range(len(ws) // 2)])
    assert got.shape == ref.shape == (112, 112, 6)
    assert np.abs(got - ref).max() / supres.SCALE <= GATE


def test_missing_weight_file_raises_oserror(env):
    from dsen2_b200 import supres
    old = supres.MDL_PATH
    supres.MDL_PATH = '/nonexistent/models/'
    try:
        with pytest.raises(OSError):
            supres.DSen2_20(np.zeros((128, 128, 4), np.float32), np.zeros((64, 64, 6), np.float32))
    finally:
        supres.MDL_PATH = old


def test_demo_driver_runs_on_a_scene_file(env, malmo, tmp_path, capsys):
    """python -m dsen2_b200.demoDSen2 (mirror of testing/demoDSen2.py) on a scene written as HDF5 the way the .mat
    files store it (arrays transposed), with random weights because the shipped hdf5 weights are missing blobs."""
    from dsen2_b200 import demoDSen2
    from dsen2_b200.hdf5 import write_hdf5
    d10, d20, d60 = malmo
    crop = lambda a, r: np.ascontiguousarray(a[:240 // r, :240 // r])
    tree = {'im10': crop(d10, 1).transpose().copy(), 'im20': crop(d20, 2).transpose().copy(),
            'im60': crop(d60, 6).transpose().copy()}
    write_hdf5(str(tmp_path / 'S2A_MSIL1C_20170527_T33UUB.mat'), tree, {})
    rc = demoDSen2.main(['--data', str(tmp_path) + '/', '--random-weights'])
    out = capsys.readouterr().out
    assert rc == 0 and out.count('super-resolved') == 2 and '(240, 240, 6)' in out and '(240, 240, 2)' in out
    assert out.count('skipping') == 5                      # the other scenes of the demo are not in the directory


def test_integration_md_ctypes_stub_runs_as_written(env):
    """The reference-side binding shown in INTEGRATION.md section 2 is executed verbatim (only the library path is
    resolved) and must give the facade's result bit for bit -- the document cannot drift from the ABI."""
    import os
    import re
    from dsen2_b200 import supres
    from dsen2_b200.DSen2Net import s2model
    torch, _capi, lib = env
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    text = open(os.path.join(root, 'INTEGRATION.md')).read()
    code = re.search(r"```python\n(# testing/supres_b200\.py.*?)```", text, re.S).group(1)
    code = code.replace('ctypes.CDLL("libdsen2_b200.so")', 'ctypes.CDLL(%r)' % _capi.LIB_PATH)
    ns = {}
    exec(compile(code, 'INTEGRATION.md', 'exec'), ns)
    rng = np.random.RandomState(21)
    d10 = rng.randint(0, 9000, size=(300, 412, 4)).astype(np.uint16)
    d20 = rng.randint(0, 9000, size=(150, 206, 6)).astype(np.uint16)
    model = s2model(((4, None, None), (6, None, None)), num_layers=6, feature_size=128, seed=8)
    wts, biases, _, _ = model._ensure_packed(torch.device('cuda', torch.cuda.current_device()))
    got = ns['DSen2_20'](d10, d20, (wts, biases))
    assert np.array_equal(got, supres.DSen2_20(d10, d20, model=model))
    assert np.array_equal(ns['DSen2_20'](d10.astype(np.float32), d20.astype(np.float32), (wts, biases)), got)
