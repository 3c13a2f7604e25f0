"""CTA-pair (cta_group::2) DSen2 fast path: input preparation, split-precision head / tail, stitch fusion.

Oracles: the prepared-input layout is checked bit-exactly against a numpy restatement of its definition
(include/dsen2_b200.h) built on the CPU patch oracle; the head / tail layers against float64 convolutions
of the SAME operands (hi + lo), so only accumulation order differs: rtol/atol 2e-5 (fp32-equivalent layers).
"""
import numpy as np
import pytest

from cases import CASES20, CASES60, synth
import tile_schedule as ts
from qtrunk import NORMAL, q_decode as _q_decode, q_encode as _q_encode, q_from_tiles as _q_from_tiles, q_to_tiles as _q_to_tiles

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def env():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from dsen2_b200 import _capi
    return torch, _capi, _capi.lib()


def _split(v):
    hi = v.astype(np.float16)
    lo = (v - hi.astype(np.float32)).astype(np.float16)
    return hi, lo


def _xin_expected(xcat):
    """xcat (n, C, P, P) float32 -> (hi, lo) (n, P, P, 64) float16 per the x_in definition."""
    n, C, P, _ = xcat.shape
    x = np.zeros((n, P, P + 2, 16), np.float32)
    x[:, :, 1:P + 1, :C] = xcat.transpose(0, 2, 3, 1)
    full = np.zeros((n, P, P, 64), np.float32)
    for t in range(3):
        full[..., t * 16:(t + 1) * 16] = x[:, :, t:t + P, :]
    return _split(full)


def _prep_patches(env, xs):
    torch, _capi, lib = env
    n, P = xs[0].shape[0], xs[0].shape[2]
    dx = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in xs]
    hi = torch.full((n, P, P, 64), 7.0, dtype=torch.float16, device='cuda')
    lo = torch.full((n, P, P, 64), 7.0, dtype=torch.float16, device='cuda')
    x2, c2 = (dx[2], xs[2].shape[1]) if len(xs) == 3 else (None, 0)
    _capi.check(lib.dsen2_prep_from_patches(_capi.ptr(dx[0]), xs[0].shape[1], _capi.ptr(dx[1]), xs[1].shape[1],
                                            _capi.ptr(x2), c2, n, P, _capi.ptr(hi), _capi.ptr(lo),
                                            _capi.stream_ptr()), 'prep_from_patches')
    torch.cuda.synchronize()
    return hi, lo


@pytest.mark.parametrize('chan', [(4, 6), (4, 6, 2)])
def test_prep_from_patches_layout_bit_exact(env, chan):
    rng = np.random.RandomState(sum(chan))
    n, P = 2, 40
    xs = [rng.uniform(0, 5, size=(n, c, P, P)).astype(np.float32) for c in chan]
    hi, lo = _prep_patches(env, xs)
    ehi, elo = _xin_expected(np.concatenate(xs, axis=1))
    assert np.array_equal(hi.cpu().numpy().view(np.uint16), ehi.view(np.uint16))
    assert np.array_equal(lo.cpu().numpy().view(np.uint16), elo.view(np.uint16))


@pytest.mark.parametrize('tag', sorted(CASES20)[:3] + sorted(CASES60)[:2])
def test_prep16_from_images_matches_patch_oracle(env, tag):
    """Fused extract + bilinear + /2000 == the CPU oracle's get_test_patches[60] then /2000, value for value
    (10 m bands bit-exact; upsampled bands within the 2e-3 DN the standalone bilinear kernel is held to); the same
    images as uint16 digital numbers (what GDAL delivers) prepare bit-identical inputs."""
    torch, _capi, lib = env
    from oracle import patches_oracle as po
    d10, d20, d60 = synth(tag)
    run60 = tag in CASES60
    if run60:
        ps = po.get_test_patches60(d10, d20, d60, 192, 12)
        P, B = 192, 12
    else:
        ps = po.get_test_patches(d10, d20, 128, 8)
        P, B = 128, 8
    H, W = d10.shape[:2]
    S = P - 2 * B
    filled = (-(-H // S)) * (-(-W // S))
    n = ps[0].shape[0]                                   # allocated (patches.py:32-39): surplus patches stay zero
    imgs = (d10, d20) + ((d60,) if run60 else ())
    outs = []
    for dt, code in ((np.float32, _capi.IMG_F32), (np.uint16, _capi.IMG_U16)):
        assert all(np.array_equal(a, a.astype(dt)) for a in imgs)
        t = [torch.from_numpy(a.astype(dt)).cuda() for a in imgs] + ([None] if not run60 else [])
        hi = torch.full((n, P, P, 16), 7.0, dtype=torch.float16, device='cuda')
        lo = torch.full_like(hi, 7.0)
        _capi.check(lib.dsen2_prep16_from_images(_capi.ptr(t[0]), _capi.ptr(t[1]), _capi.ptr(t[2]), code, H, W, P, B, 0, n,
                                                 2000.0, _capi.ptr(hi), _capi.ptr(lo), _capi.stream_ptr()), 'prep16_from_images')
        torch.cuda.synchronize()
        outs.append((hi.cpu().numpy(), lo.cpu().numpy()))
    hi, lo = outs[0]
    assert np.array_equal(hi.view(np.uint16), outs[1][0].view(np.uint16)) and np.array_equal(lo.view(np.uint16), outs[1][1].view(np.uint16))
    got = hi.astype(np.float32) + lo.astype(np.float32)
    xcat = np.concatenate([p / np.float32(2000) for p in ps], axis=1)
    exp_hi, exp_lo = _xin16_expected(xcat)
    exp = exp_hi.astype(np.float32) + exp_lo.astype(np.float32)
    assert n >= filled
    # 10 m bands: pure indexing, then IEEE division -> identical bits
    assert np.array_equal(hi[..., :4].view(np.uint16), exp_hi[..., :4].view(np.uint16))
    assert np.array_equal(lo[..., :4].view(np.uint16), exp_lo[..., :4].view(np.uint16))
    np.testing.assert_allclose(got, exp, rtol=0, atol=2e-3 / 2000 + 1e-7)
    if n > filled:   # surplus patches of the allocated stack are zero (patches.py:32-39)
        assert not hi[filled:].any()


def _xin16_expected(xcat):
    """xcat (n, C, P, P) float32 -> (hi, lo) (n, P, P, 16) float16: channel c = band c, zero above C."""
    n, C, P, _ = xcat.shape
    full = np.zeros((n, P, P, 16), np.float32)
    full[..., :C] = xcat.transpose(0, 2, 3, 1)
    return _split(full)


def _conv64(x_nhwc, w_hwio, bias):
    """float64 3x3 'same' cross-correlation; x (n,H,W,C) -> (n,H,W,Cout)."""
    import torch
    import torch.nn.functional as F
    x = torch.from_numpy(np.ascontiguousarray(x_nhwc, dtype=np.float64)).permute(0, 3, 1, 2)
    w = torch.from_numpy(np.ascontiguousarray(w_hwio, dtype=np.float64)).permute(3, 2, 0, 1).contiguous()
    y = F.conv2d(x, w, torch.from_numpy(bias.astype(np.float64)), padding=1)
    return y.permute(0, 2, 3, 1).contiguous().numpy()


@pytest.mark.parametrize('shape', [(2, 32, 32), (1, 128, 128), (3, 40, 24), (1, 8, 200), (5, 16, 8), ts.PATCH])
def test_conv_head_fp32_equivalent(env, shape):
    torch, _capi, lib = env
    n, H, W = shape
    F, C = 128, 10
    rng = np.random.RandomState(H + W)
    # head runs on square patches in production, but the kernel is shape-generic: use the NHWC layout directly
    xcat = rng.uniform(0, 5, size=(n, C, H, W)).astype(np.float32)
    xp = np.zeros((n, H, W + 2, 16), np.float32)
    xp[:, :, 1:W + 1, :C] = xcat.transpose(0, 2, 3, 1)
    full = np.concatenate([xp[:, :, t:t + W, :] for t in range(3)] + [np.zeros((n, H, W, 16), np.float32)], axis=-1)
    hi, lo = _split(full)
    lim = np.sqrt(6.0 / (9 * C))
    w = rng.uniform(-lim, lim, size=(3, 3, C, F)).astype(np.float32)
    bias = (rng.randn(F) * 0.1).astype(np.float32)
    tw = torch.empty((3, 2 * F, 64), dtype=torch.float16, device='cuda')
    _capi.check(lib.dsen2_pack_head_weights(_capi.ptr(torch.from_numpy(w).cuda()), C, F, _capi.ptr(tw),
                                            _capi.stream_ptr()), 'pack head')
    thi, tlo = torch.from_numpy(hi).cuda(), torch.from_numpy(lo).cuda()
    tb = torch.from_numpy(bias).cuda()
    ohi = torch.zeros((n, H, W, F), dtype=torch.float16, device='cuda')
    olo = torch.zeros_like(ohi)
    x32 = torch.full((n, H, W // 8, F // 4, 8, 4), -3.0, device='cuda')
    _capi.check(lib.dsen2_conv_head(_capi.ptr(thi), _capi.ptr(tlo), _capi.ptr(tw), _capi.ptr(tb), n, H, W, F,
                                    _capi.ptr(ohi), _capi.ptr(olo), _capi.ptr(x32), _capi.stream_ptr()), 'conv head')
    torch.cuda.synchronize()
    xin = (hi.astype(np.float64) + lo.astype(np.float64))[..., 16:16 + C]          # centre tap = the input itself
    w_hi = w.astype(np.float16)
    w_eff = w_hi.astype(np.float64) + (w - w_hi.astype(np.float32)).astype(np.float16).astype(np.float64)
    ref = np.maximum(_conv64(xin, w_eff, bias), 0)
    got = ohi.cpu().numpy().astype(np.float64) + olo.cpu().numpy().astype(np.float64)
    ts.check(ts.pair_schedule(n, H, W), 'conv_head', np.abs(got - ref).max())
    np.testing.assert_allclose(got, ref, rtol=2e-5, atol=2e-5)
    assert np.abs(got - np.maximum(_conv64(xcat.transpose(0, 2, 3, 1), w, bias), 0)).max() < 5e-5   # vs true fp32 layer
    # fp32 trunk seed, tile-row-major (n, H, W/8, F/4, 8, 4): the same values before the hi/lo split
    trunk = x32.cpu().numpy().transpose(0, 1, 2, 4, 3, 5).reshape(n, H, W, F)
    np.testing.assert_allclose(trunk, ref, rtol=2e-5, atol=2e-5)
    assert np.array_equal(trunk.astype(np.float16).view(np.uint16), ohi.cpu().numpy().view(np.uint16))


@pytest.mark.parametrize('shape,cout,ch0', [((2, 32, 32), 6, 4), ((1, 128, 128), 6, 4), ((1, 48, 48), 2, 10),
                                            ((3, 40, 24), 6, 4), (ts.PATCH, 6, 4)])
def test_conv_tail_nchw_fp32_equivalent(env, shape, cout, ch0):
    torch, _capi, lib = env
    n, H, W = shape
    F = 128
    rng = np.random.RandomState(H * 3 + cout)
    x = rng.randn(n, H, W, F).astype(np.float32)
    x_hi, x_lo = _split(x)
    xin = np.zeros((n, H, W, 64), np.float32)
    xin[..., 16:32] = rng.uniform(0, 4, size=(n, H, W, 16)).astype(np.float32)
    xin_hi, xin_lo = _split(xin)
    lim = np.sqrt(6.0 / (9 * F))
    w = rng.uniform(-lim, lim, size=(3, 3, F, cout)).astype(np.float32)
    bias = np.zeros(16, np.float32)
    bias[:cout] = rng.randn(cout) * 0.1
    tw = torch.empty((9, 32, F), dtype=torch.float16, device='cuda')
    _capi.check(lib.dsen2_pack_tail_weights(_capi.ptr(torch.from_numpy(w).cuda()), F, cout, _capi.ptr(tw),
                                            _capi.stream_ptr()), 'pack tail')
    dev = [torch.from_numpy(a).cuda() for a in (x_hi, x_lo, xin_hi, xin_lo, bias)]

    def tail(b0, m):
        out = torch.full((m, cout, H, W), -5.0, device='cuda')
        _capi.check(lib.dsen2_conv_tail(_capi.ptr(dev[0][b0:]), _capi.ptr(dev[1][b0:]), _capi.ptr(tw), _capi.ptr(dev[4]),
                                        _capi.ptr(dev[2][b0:]), _capi.ptr(dev[3][b0:]), ch0, cout, m, H, W, _capi.ptr(out),
                                        _capi.stream_ptr()), 'conv tail')
        torch.cuda.synchronize()
        return out.cpu().numpy()
    got = tail(0, n)
    # a tile's result does not depend on which CTA computes it, or after which tiles: the batch equals one launch per
    # patch (at most one tile per CTA) bit for bit
    alone = np.concatenate([tail(b, 1) for b in range(n)])
    assert np.array_equal(got.view(np.uint32), alone.view(np.uint32))
    xe = x_hi.astype(np.float64) + x_lo.astype(np.float64)
    w_hi = w.astype(np.float16)
    w_eff = w_hi.astype(np.float64) + (w - w_hi.astype(np.float32)).astype(np.float16).astype(np.float64)
    skip = (xin_hi.astype(np.float64) + xin_lo.astype(np.float64))[..., 16 + ch0:16 + ch0 + cout]
    conv = _conv64(xe, w_eff, bias[:cout])
    ref = (conv + skip).transpose(0, 3, 1, 2)
    ts.check(ts.pair_schedule(n, H, W), 'conv_tail cout=%d' % cout, np.abs(got - ref).max())
    # relative to the magnitudes the fp32 arithmetic carries: where the skip cancels the convolution (|conv| ~ 4, sum ~ 0.05)
    # the accumulation error of the convolution (~3e-5 at most) is all that is left
    scale = (np.abs(conv) + np.abs(skip)).transpose(0, 3, 1, 2)
    assert (np.abs(got - ref) <= 2e-5 + 2e-5 * scale).all(), np.abs(got - ref).max()


@pytest.mark.parametrize('shape,cout,ch0,F', [((2, 32, 32), 6, 4, 128), ((1, 128, 128), 6, 4, 256), ((1, 48, 48), 2, 10, 256),
                                              ((3, 40, 24), 6, 4, 256), ((1, 192, 192), 2, 10, 128), (ts.PATCH, 6, 4, 128),
                                              (ts.PATCH, 6, 4, 256), (ts.PATCH, 7, 9, 128), (ts.RAGGED, 1, 15, 256)])
def test_conv_tail16_nchw_fp32_equivalent(env, shape, cout, ch0, F):
    """Last layer (F -> cout, split hi + lo operands) + global skip from the 16-channel prepared input, F = 128 / 256.
    cout 7 (kTMaxCout: 126 of the 128 weight rows) with the skip reaching channel 15, and cout 1."""
    torch, _capi, lib = env
    n, H, W = shape
    rng = np.random.RandomState(H * 3 + cout + F)
    x_hi, x_lo = _split(rng.randn(n, H, W, F).astype(np.float32))
    xin_hi, xin_lo = _split(rng.uniform(0, 4, size=(n, H, W, 16)).astype(np.float32))
    lim = np.sqrt(6.0 / (9 * F))
    w = rng.uniform(-lim, lim, size=(3, 3, F, cout)).astype(np.float32)
    bias = np.zeros(16, np.float32)
    bias[:cout] = rng.randn(cout) * 0.1
    tw = torch.empty((128, F), dtype=torch.float16, device='cuda')
    _capi.check(lib.dsen2_pack_tail16_weights(_capi.ptr(torch.from_numpy(w).cuda()), F, cout, _capi.ptr(tw),
                                            _capi.stream_ptr()), 'pack tail')
    dev = [torch.from_numpy(a).cuda() for a in (x_hi, x_lo, xin_hi, xin_lo, bias)]
    out = torch.full((n, cout, H, W), -5.0, device='cuda')
    _capi.check(lib.dsen2_conv_tail16(_capi.ptr(dev[0]), _capi.ptr(dev[1]), _capi.ptr(tw), _capi.ptr(dev[4]),
                                      _capi.ptr(dev[2]), _capi.ptr(dev[3]), ch0, cout, F, n, H, W, _capi.ptr(out),
                                      _capi.stream_ptr()), 'conv tail16')
    torch.cuda.synchronize()
    xe = x_hi.astype(np.float64) + x_lo.astype(np.float64)
    w_hi = w.astype(np.float16)
    w_eff = w_hi.astype(np.float64) + (w - w_hi.astype(np.float32)).astype(np.float16).astype(np.float64)
    skip = (xin_hi.astype(np.float64) + xin_lo.astype(np.float64))[..., ch0:ch0 + cout]
    ref = (_conv64(xe, w_eff, bias[:cout]) + skip).transpose(0, 3, 1, 2)
    tol = 2e-5 if F == 128 else 6e-5          # fp32 accumulation order over K = 4 * 9 * F products
    got = out.cpu().numpy()
    ts.check(ts.tail_schedule(n, H, W), 'conv_tail16 F=%d cout=%d' % (F, cout), np.abs(got - ref).max())
    np.testing.assert_allclose(got, ref, rtol=tol, atol=tol)


@pytest.mark.parametrize('tag,F', [('a', 128), ('b', 128), ('c', 128), ('d', 128), ('b', 256)])
def test_conv_tail_stitch_matches_recompose(env, tag, F):
    """tail + stitch fusion == tail (NCHW) then recompose_images (CPU oracle) x 2000, exactly.  Case 'c' (112 x 112)
    fills ONE patch of the four allocated ones: it is stitched and cropped like any other (patches.py:375 keys on the
    allocated count)."""
    torch, _capi, lib = env
    from oracle import patches_oracle as po
    d10, _, _ = synth(tag)
    H, W = d10.shape[:2]
    P, B, cout = 128, 8, 6
    S = P - 2 * B
    ny, nx = -(-H // S), -(-W // S)
    n = ny * nx
    rng = np.random.RandomState(n)
    x_hi, x_lo = _split(rng.randn(n, P, P, F).astype(np.float32))
    xin_hi, xin_lo = _split(rng.uniform(0, 4, size=(n, P, P, 16)).astype(np.float32))
    lim = np.sqrt(6.0 / (9 * F))
    w = rng.uniform(-lim, lim, size=(3, 3, F, cout)).astype(np.float32)
    bias = np.zeros(16, np.float32)
    tw = torch.empty((128, F), dtype=torch.float16, device='cuda')
    _capi.check(lib.dsen2_pack_tail16_weights(_capi.ptr(torch.from_numpy(w).cuda()), F, cout, _capi.ptr(tw),
                                            _capi.stream_ptr()), 'pack tail')
    dev = [torch.from_numpy(a).cuda() for a in (x_hi, x_lo, xin_hi, xin_lo, bias)]
    pred = torch.empty((n, cout, P, P), device='cuda')
    _capi.check(lib.dsen2_conv_tail16(_capi.ptr(dev[0]), _capi.ptr(dev[1]), _capi.ptr(tw), _capi.ptr(dev[4]),
                                      _capi.ptr(dev[2]), _capi.ptr(dev[3]), 4, cout, F, n, P, P, _capi.ptr(pred),
                                      _capi.stream_ptr()), 'conv tail16')
    ts.report(ts.tail_schedule(n - n // 2, P, P, border=B), 'conv_tail16_stitch F=%d, larger shard' % F, float('nan'))
    canvas = torch.full((H, W, cout), -1.0, device='cuda')
    # two shards, second first: ownership (not launch order) decides every pixel
    half = n // 2
    for first, cnt in ((half, n - half), (0, half)):
        if cnt == 0:
            continue
        sl = slice(first, first + cnt)
        _capi.check(lib.dsen2_conv_tail16_stitch(_capi.ptr(dev[0][sl]), _capi.ptr(dev[1][sl]), _capi.ptr(tw),
                                                 _capi.ptr(dev[4]), _capi.ptr(dev[2][sl]), _capi.ptr(dev[3][sl]), 4, cout, F,
                                                 cnt, P, first, B, H, W, 2000.0, _capi.ptr(canvas), _capi.stream_ptr()),
                    'conv tail16 stitch')
    torch.cuda.synchronize()
    allocated = (H // 2 // 56 + 1) * (W // 2 // 56 + 1)
    full = np.zeros((allocated, cout, P, P), np.float32)      # the reference's stack carries the surplus zero patches
    full[:n] = pred.cpu().numpy()
    ref = po.recompose_images(full, B, (H, W)) * np.float32(2000)
    assert ref.shape == (H, W, cout)
    assert np.array_equal(canvas.cpu().numpy(), ref)


@pytest.mark.parametrize('shape', [(2, 32, 32), (1, 128, 128), (3, 40, 24), (1, 8, 200), (2, 192, 192), (2, 32, 32, 256),
                                   (1, 24, 72, 256), ts.PATCH, ts.RAGGED, ts.PATCH + (256,), ts.RAGGED + (256,)])
@pytest.mark.parametrize('want_lo', [False, True])
def test_conv_res32_fp32_trunk_update(env, shape, want_lo):
    """trunk32 <- trunk32 + 0.1 * (conv(t) + b) in place on the tile-row-major fp32 trunk; fp16 hi (and lo) copies.
    128 features (resident weights) and 256 (streamed; the training step of VDSen2)."""
    torch, _capi, lib = env
    n, H, W = shape[:3]
    F = shape[3] if len(shape) == 4 else 128
    rng = np.random.RandomState(H + 5 * W)
    t = np.maximum(rng.randn(n, H, W, F), 0).astype(np.float16)
    x = rng.randn(n, H, W, F).astype(np.float32)
    lim = np.sqrt(6.0 / (9 * F))
    w = rng.uniform(-lim, lim, size=(3, 3, F, F)).astype(np.float32)
    bias = (rng.randn(F) * 0.1).astype(np.float32)
    tw = torch.empty((9, F, F), dtype=torch.float16, device='cuda')
    _capi.check(lib.dsen2_pack_conv_weights(_capi.ptr(torch.from_numpy(w).cuda()), F, F, F, F, _capi.ptr(tw), _capi.stream_ptr()), 'pack')
    x_cm = np.ascontiguousarray(x.reshape(n, H, W // 8, 8, F // 4, 4).transpose(0, 1, 2, 4, 3, 5))
    tx, tt, tb = torch.from_numpy(x_cm).cuda(), torch.from_numpy(t).cuda(), torch.from_numpy(bias).cuda()
    hi = torch.zeros((n, H, W, F), dtype=torch.float16, device='cuda')
    lo = torch.zeros_like(hi) if want_lo else None
    _capi.check(lib.dsen2_conv_res32(_capi.ptr(tt), _capi.ptr(tw), _capi.ptr(tb), n, H, W, F, 0.1, _capi.ptr(tx),
                                     _capi.ptr(hi), _capi.ptr(lo), _capi.stream_ptr()), 'conv res32')
    torch.cuda.synchronize()
    ref = x.astype(np.float64) + 0.1 * _conv64(t.astype(np.float64), w.astype(np.float16).astype(np.float64), bias)
    got = tx.cpu().numpy().transpose(0, 1, 2, 4, 3, 5).reshape(n, H, W, F)
    tol = 2e-5 if F == 128 else 4e-5                  # fp32 accumulation over K = 9 F
    ts.check(ts.pair_schedule(n, H, W), 'conv_res32 F=%d lo=%s' % (F, want_lo), np.abs(got - ref).max())
    np.testing.assert_allclose(got, ref, rtol=tol, atol=tol)
    assert np.array_equal(hi.cpu().numpy().view(np.uint16), got.astype(np.float16).view(np.uint16))
    if want_lo:
        exp_lo = (got - got.astype(np.float16).astype(np.float32)).astype(np.float16)
        assert np.array_equal(lo.cpu().numpy().view(np.uint16), exp_lo.view(np.uint16))


# ---- fp16 + 8 bit trunk (include/dsen2_b200.h: dsen2_conv_head16_q / dsen2_conv_resq) -------------------------------
@pytest.mark.parametrize('shape', [(2, 32, 32), (1, 128, 128), (3, 40, 24), (1, 8, 200), (2, 192, 192), ts.PATCH, ts.RAGGED])
@pytest.mark.parametrize('last', [False, True])
def test_conv_resq_trunk_update(env, shape, last):
    """x <- x + 0.1 * (conv(t) + b) on the fp16 + 8 bit trunk, in place; the last block emits x_hi, x_lo for the tail."""
    torch, _capi, lib = env
    n, H, W = shape
    F = 128
    rng = np.random.RandomState(H + 5 * W)
    t = np.maximum(rng.randn(n, H, W, F), 0).astype(np.float16)
    x = rng.randn(n, H, W, F).astype(np.float32)
    x[0, 0, :, :4] = 0                                       # exact zeros stay exact zeros
    lim = np.sqrt(6.0 / (9 * F))
    w = rng.uniform(-lim, lim, size=(3, 3, F, F)).astype(np.float32)
    bias = (rng.randn(F) * 0.1).astype(np.float32)
    tw = torch.empty((9, F, F), dtype=torch.float16, device='cuda')
    _capi.check(lib.dsen2_pack_conv_weights(_capi.ptr(torch.from_numpy(w).cuda()), F, F, F, F, _capi.ptr(tw), _capi.stream_ptr()), 'pack')
    h0, q0 = _q_encode(x)
    x_seen = _q_decode(h0, q0)
    thi, tq = torch.from_numpy(h0).cuda(), torch.from_numpy(_q_to_tiles(q0)).cuda()
    tt, tb = torch.from_numpy(t).cuda(), torch.from_numpy(bias).cuda()
    lo = torch.zeros((n, H, W, F), dtype=torch.float16, device='cuda') if last else None
    _capi.check(lib.dsen2_conv_resq(_capi.ptr(tt), _capi.ptr(tw), _capi.ptr(tb), n, H, W, 0.1, _capi.ptr(thi),
                                    _capi.ptr(tq), _capi.ptr(lo), _capi.stream_ptr()), 'conv resq')
    torch.cuda.synchronize()
    ref = x_seen.astype(np.float64) + 0.1 * _conv64(t.astype(np.float64), w.astype(np.float16).astype(np.float64), bias)
    h = thi.cpu().numpy()
    sched = ts.pair_schedule(n, H, W)
    if last:
        got = h.astype(np.float64) + lo.cpu().numpy().astype(np.float64)
        ts.check(sched, 'conv_resq last', np.abs(got - ref).max())
        np.testing.assert_allclose(got, ref, rtol=2e-5, atol=2e-5)
        # x_hi = fp16(x): re-rounding hi + lo differs only where x sits within 2^-22 of a rounding tie (~2^-11 of the elements)
        assert np.mean(got.astype(np.float32).astype(np.float16).view(np.uint16) == h.view(np.uint16)) > 0.999
        assert np.array_equal(_q_from_tiles(tq.cpu().numpy()), q0)                       # bytes only read
    else:
        q = _q_from_tiles(tq.cpu().numpy())
        got = _q_decode(h, q)
        ts.check(sched, 'conv_resq', np.abs(got - ref).max())
        np.testing.assert_allclose(got, ref, rtol=2e-5, atol=2e-5)
        ok = np.abs(got) >= 2 * NORMAL
        h2, q2 = _q_encode(got[ok])
        assert np.array_equal(h2.view(np.uint16), h[ok].view(np.uint16)) and np.array_equal(q2, q[ok])
        assert not got[0, 0, :, :4].any() or np.abs(ref[0, 0, :, :4]).min() > 0        # no spurious zeros
    assert lib.dsen2_conv_resq(_capi.ptr(thi), _capi.ptr(tw), _capi.ptr(tb), n, H, W, 0.1, _capi.ptr(thi),
                               _capi.ptr(tq), None, _capi.stream_ptr()) == -1           # aliasing is refused


# ---- un-gathered 16-channel prepared input + nine-tap first layer (dsen2_prep16_* / dsen2_conv_head16_q) ------------
@pytest.mark.parametrize('chan', [(4, 6), (4, 6, 2)])
def test_prep16_from_patches_layout_bit_exact(env, chan):
    torch, _capi, lib = env
    rng = np.random.RandomState(sum(chan))
    n, P = 2, 40
    xs = [rng.uniform(0, 5, size=(n, c, P, P)).astype(np.float32) for c in chan]
    dx = [torch.from_numpy(a).cuda() for a in xs]
    hi = torch.full((n, P, P, 16), 7.0, dtype=torch.float16, device='cuda')
    lo = torch.full_like(hi, 7.0)
    x2, c2 = (dx[2], chan[2]) if len(chan) == 3 else (None, 0)
    _capi.check(lib.dsen2_prep16_from_patches(_capi.ptr(dx[0]), chan[0], _capi.ptr(dx[1]), chan[1], _capi.ptr(x2), c2, n, P,
                                              _capi.ptr(hi), _capi.ptr(lo), _capi.stream_ptr()), 'prep16_from_patches')
    torch.cuda.synchronize()
    ehi, elo = _xin16_expected(np.concatenate(xs, axis=1))
    assert np.array_equal(hi.cpu().numpy().view(np.uint16), ehi.view(np.uint16))
    assert np.array_equal(lo.cpu().numpy().view(np.uint16), elo.view(np.uint16))


@pytest.mark.parametrize('shape', [(2, 32, 32), (1, 128, 128), (3, 40, 24), (1, 8, 200), (5, 16, 8), (1, 192, 192), ts.PATCH,
                                   ts.RAGGED])
@pytest.mark.parametrize('F', [128, 256])
def test_conv_head16_q_nine_taps(env, shape, F):
    """First layer on the 16-channel input: nine shifted 32-byte-row descriptors, three products (hi*W_hi + hi*W_lo +
    lo*W_hi) per tap into one accumulator; fp32-equivalent.  F = 128 (DSen2) and 256 (VDSen2)."""
    torch, _capi, lib = env
    n, H, W = shape
    C = 12
    rng = np.random.RandomState(H + 3 * W + F)
    xcat = rng.uniform(0, 5, size=(n, C, H, W)).astype(np.float32)
    hi, lo = _xin16_expected(xcat) if H == W else _split(np.concatenate(
        [xcat.transpose(0, 2, 3, 1), np.zeros((n, H, W, 16 - C), np.float32)], axis=-1))
    lim = np.sqrt(6.0 / (9 * C))
    w = rng.uniform(-lim, lim, size=(3, 3, C, F)).astype(np.float32)
    bias = (rng.randn(F) * 0.1).astype(np.float32)
    tw = torch.empty((9, 2 * F, 16), dtype=torch.float16, device='cuda')
    _capi.check(lib.dsen2_pack_head16_weights(_capi.ptr(torch.from_numpy(w).cuda()), C, F, _capi.ptr(tw),
                                              _capi.stream_ptr()), 'pack head16')
    thi, tlo, tb = torch.from_numpy(hi).cuda(), torch.from_numpy(lo).cuda(), torch.from_numpy(bias).cuda()
    ohi = torch.zeros((n, H, W, F), dtype=torch.float16, device='cuda')
    oq = torch.full((n, H, W // 8, F // 16, 8, 16), 77, dtype=torch.int8, device='cuda')
    _capi.check(lib.dsen2_conv_head16_q(_capi.ptr(thi), _capi.ptr(tlo), _capi.ptr(tw), _capi.ptr(tb), n, H, W, F,
                                        _capi.ptr(ohi), _capi.ptr(oq), _capi.stream_ptr()), 'conv head16 q')
    torch.cuda.synchronize()
    xin = (hi.astype(np.float64) + lo.astype(np.float64))[..., :C]
    w_hi = w.astype(np.float16)
    w_eff = w_hi.astype(np.float64) + (w - w_hi.astype(np.float32)).astype(np.float16).astype(np.float64)
    ref = np.maximum(_conv64(xin, w_eff, bias), 0)         # (the kernel drops lo * W_lo: ~2^-22 of a product)
    got = _q_decode(ohi.cpu().numpy(), _q_from_tiles(oq.cpu().numpy()))
    ts.check(ts.pair_schedule(n, H, W), 'conv_head16_q F=%d' % F, np.abs(got - ref).max())
    np.testing.assert_allclose(got, ref, rtol=2e-5, atol=2e-5)
    assert np.abs(got - np.maximum(_conv64(xcat.transpose(0, 2, 3, 1), w, bias), 0)).max() < 5e-5   # vs the true fp32 layer


@pytest.mark.parametrize('shape', [ts.PATCH, ts.RAGGED])
def test_conv_head16_relu(env, shape):
    """The first layer of the 256-feature training step (dsen2_conv_head16_relu): the nine-tap three-product convolution of
    dsen2_conv_head16_q, relu -> NHWC fp16 and the seed of the fp32 trunk, tile-row-major (n, H, W/8, F/4, 8, 4)."""
    torch, _capi, lib = env
    n, H, W = shape
    C, F = 12, 256
    rng = np.random.RandomState(H + 3 * W + F)
    x = rng.uniform(0, 5, size=(n, H, W, C)).astype(np.float32)
    hi, lo = _split(np.concatenate([x, np.zeros((n, H, W, 16 - C), np.float32)], axis=-1))
    lim = np.sqrt(6.0 / (9 * C))
    w = rng.uniform(-lim, lim, size=(3, 3, C, F)).astype(np.float32)
    bias = (rng.randn(F) * 0.1).astype(np.float32)
    tw = torch.empty((9, 2 * F, 16), dtype=torch.float16, device='cuda')
    _capi.check(lib.dsen2_pack_head16_weights(_capi.ptr(torch.from_numpy(w).cuda()), C, F, _capi.ptr(tw),
                                              _capi.stream_ptr()), 'pack head16')
    thi, tlo, tb = torch.from_numpy(hi).cuda(), torch.from_numpy(lo).cuda(), torch.from_numpy(bias).cuda()
    ohi = torch.zeros((n, H, W, F), dtype=torch.float16, device='cuda')
    x32 = torch.full((n, H, W // 8, F // 4, 8, 4), -3.0, device='cuda')
    _capi.check(lib.dsen2_conv_head16_relu(_capi.ptr(thi), _capi.ptr(tlo), _capi.ptr(tw), _capi.ptr(tb), n, H, W, F,
                                           _capi.ptr(ohi), _capi.ptr(x32), _capi.stream_ptr()), 'conv head16 relu')
    torch.cuda.synchronize()
    xin = (hi.astype(np.float64) + lo.astype(np.float64))[..., :C]
    w_hi = w.astype(np.float16)
    w_eff = w_hi.astype(np.float64) + (w - w_hi.astype(np.float32)).astype(np.float16).astype(np.float64)
    ref = np.maximum(_conv64(xin, w_eff, bias), 0)         # (the kernel drops lo * W_lo: ~2^-22 of a product)
    trunk = x32.cpu().numpy().transpose(0, 1, 2, 4, 3, 5).reshape(n, H, W, F)
    ts.check(ts.pair_schedule(n, H, W), 'conv_head16_relu', np.abs(trunk - ref).max())
    np.testing.assert_allclose(trunk, ref, rtol=2e-5, atol=2e-5)
    assert np.abs(trunk - np.maximum(_conv64(x, w, bias), 0)).max() < 5e-5                       # vs the true fp32 layer
    assert np.array_equal(trunk.astype(np.float16).view(np.uint16), ohi.cpu().numpy().view(np.uint16))


@pytest.mark.parametrize('shape', [(2, 32, 32), (1, 128, 128), (3, 40, 24), ts.PATCH, ts.RAGGED])
@pytest.mark.parametrize('last', [False, True])
def test_conv_resq256_trunk_update(env, shape, last):
    """The 256-feature (VDSen2) resblock update on the fp16 + 8 bit trunk: two 64-channel passes per thread; the last
    block emits x_hi, x_lo for the last layer."""
    torch, _capi, lib = env
    n, H, W = shape
    F = 256
    rng = np.random.RandomState(H + 7 * W)
    t = np.maximum(rng.randn(n, H, W, F), 0).astype(np.float16)
    x = rng.randn(n, H, W, F).astype(np.float32)
    lim = np.sqrt(6.0 / (9 * F))
    w = rng.uniform(-lim, lim, size=(3, 3, F, F)).astype(np.float32)
    bias = (rng.randn(F) * 0.1).astype(np.float32)
    tw = torch.empty((9, F, F), dtype=torch.float16, device='cuda')
    _capi.check(lib.dsen2_pack_conv_weights(_capi.ptr(torch.from_numpy(w).cuda()), F, F, F, F, _capi.ptr(tw), _capi.stream_ptr()), 'pack')
    h0, q0 = _q_encode(x)
    x_seen = _q_decode(h0, q0)
    thi, tq = torch.from_numpy(h0).cuda(), torch.from_numpy(_q_to_tiles(q0)).cuda()
    tt, tb = torch.from_numpy(t).cuda(), torch.from_numpy(bias).cuda()
    lo = torch.zeros((n, H, W, F), dtype=torch.float16, device='cuda') if last else None
    _capi.check(lib.dsen2_conv_resq256(_capi.ptr(tt), _capi.ptr(tw), _capi.ptr(tb), n, H, W, 0.1, _capi.ptr(thi),
                                       _capi.ptr(tq), _capi.ptr(lo), _capi.stream_ptr()), 'conv resq256')
    torch.cuda.synchronize()
    ref = x_seen.astype(np.float64) + 0.1 * _conv64(t.astype(np.float64), w.astype(np.float16).astype(np.float64), bias)
    sched = ts.pair_schedule(n, H, W)
    if last:
        got = thi.cpu().numpy().astype(np.float64) + lo.cpu().numpy().astype(np.float64)
        ts.check(sched, 'conv_resq256 last', np.abs(got - ref).max())
        np.testing.assert_allclose(got, ref, rtol=3e-5, atol=3e-5)
        return
    h, q = thi.cpu().numpy(), _q_from_tiles(tq.cpu().numpy())
    got = _q_decode(h, q)
    ts.check(sched, 'conv_resq256', np.abs(got - ref).max())
    np.testing.assert_allclose(got, ref, rtol=3e-5, atol=3e-5)
    ok = np.abs(got) >= 2 * NORMAL
    h2, q2 = _q_encode(got[ok])
    assert np.array_equal(h2.view(np.uint16), h[ok].view(np.uint16)) and np.array_equal(q2, q[ok])
