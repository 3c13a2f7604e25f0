"""Training step (supres_train.py:137-144,218-230) on the GPU against the fp32 CPU oracle (oracle/train_oracle.py,
torch autograd + NAdam; parity unpinned by the reference -- Keras is not installable).

Tolerances: gradients flow through fp16 operands (fp32 accumulation), so each gradient tensor is compared to the fp32
autograd gradient relative to its own largest entry: max|g - g_ref| <= 2e-2 * max|g_ref|; building blocks are compared
with float64 restatements on the SAME fp16-rounded operands (rtol/atol 1e-3 or tighter).
"""
import numpy as np
import pytest

import tile_schedule as ts

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def env():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from dsen2_b200 import _capi
    return torch, _capi, _capi.lib()


def _wgrad_ref(x_nhwc, dy_nhwc):
    """dW[tap][ci][co] = sum_px X[px + off(tap)][ci] dY[px][co] with zero padding (float64)."""
    n, H, W, Ci = x_nhwc.shape
    xp = np.zeros((n, H + 2, W + 2, Ci), np.float64)
    xp[:, 1:H + 1, 1:W + 1] = x_nhwc
    dy = dy_nhwc.astype(np.float64)
    out = np.zeros((9, Ci, dy.shape[-1]))
    for t in range(9):
        ky, kx = t // 3, t % 3
        out[t] = np.einsum('nyxi,nyxo->io', xp[:, ky:ky + H, kx:kx + W], dy)
    return out


@pytest.mark.parametrize('shape', [(4, 32, 32), (128, 32, 32), (3, 16, 24), (2, 40, 8), (4, 32, 32, 256), (3, 16, 24, 256)])
def test_wgrad_nhwc_mn_major(env, shape):
    """Weight gradient straight from the NHWC tensors (MN-major tcgen05 operands, halo-box taps, bulk fp32 reduction);
    256 channels = four 128 x 128 blocks of the gradient."""
    torch, _capi, lib = env
    n, H, W = shape[:3]
    C = shape[3] if len(shape) == 4 else 128
    rng = np.random.RandomState(n + H)
    x = rng.randn(n, H, W, C).astype(np.float16)
    dy = (rng.randn(n, H, W, C) * 0.1).astype(np.float16)
    tx, tdy = torch.from_numpy(x).cuda(), torch.from_numpy(dy).cuda()
    dw = torch.full((9, C, C), 1.0, device='cuda')                          # accumulates on top of what is there
    db = torch.full((C,), 2.0, device='cuda')                               # ... and so does the fused bias gradient
    _capi.check(lib.dsen2_wgrad_nhwc(_capi.ptr(tx), _capi.ptr(tdy), n, H, W, C, 0.5, _capi.ptr(dw), _capi.ptr(db),
                                     _capi.stream_ptr()), 'wgrad nhwc')
    dw2 = torch.full((9, C, C), 1.0, device='cuda')
    _capi.check(lib.dsen2_wgrad_nhwc(_capi.ptr(tx), _capi.ptr(tdy), n, H, W, C, 0.5, _capi.ptr(dw2), None, _capi.stream_ptr()),
                'wgrad nhwc, no bias gradient')
    torch.cuda.synchronize()
    ref = 1.0 + 0.5 * _wgrad_ref(x.astype(np.float64), dy)
    for got in (dw, dw2):
        np.testing.assert_allclose(got.cpu().numpy(), ref, rtol=1e-3, atol=1e-3 * np.abs(ref).max())
    ref_b = 2.0 + 0.5 * dy.astype(np.float64).reshape(-1, C).sum(0)
    np.testing.assert_allclose(db.cpu().numpy(), ref_b, rtol=1e-4, atol=1e-4 * max(1.0, np.abs(ref_b).max()))


@pytest.mark.parametrize('C', [128, 256])
def test_relu_mask(env, C):
    torch, _capi, lib = env
    rng = np.random.RandomState(2)
    g = rng.randn(3, 16, 8, C).astype(np.float16)
    a = rng.randn(3, 16, 8, C).astype(np.float16)
    tg, ta = torch.from_numpy(g).cuda(), torch.from_numpy(a).cuda()
    out = torch.empty_like(tg)
    _capi.check(lib.dsen2_relu_mask(_capi.ptr(tg), _capi.ptr(ta), g.size, _capi.ptr(out), _capi.stream_ptr()), 'mask')
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy().view(np.uint16), np.where(a.astype(np.float32) > 0, g, np.float16(0)).view(np.uint16))


@pytest.mark.parametrize('C,shape', [pytest.param(C, (2, 32, 32), id=str(C)) for C in (128, 256)] +
                         [pytest.param(C, s, id='%d-%s' % (C, name)) for name, s in (('patch', ts.PATCH), ('batch128', ts.BATCH128))
                          for C in (128, 256)])
def test_conv_relu_bwd_is_the_transposed_convolution(env, C, shape):
    """ts.BATCH128 is DSen2's training batch: seven tiles on the busiest CTA pair."""
    torch, _capi, lib = env
    import torch.nn.functional as F
    n, H, W = shape
    rng = np.random.RandomState(3)
    dy = (rng.randn(n, H, W, C) * 0.1).astype(np.float16)
    act = np.maximum(rng.randn(n, H, W, C), 0).astype(np.float16)
    lim = np.sqrt(6.0 / (9 * C))
    w = rng.uniform(-lim, lim, size=(3, 3, C, C)).astype(np.float32)
    tw = torch.empty((9, C, C), dtype=torch.float16, device='cuda')
    _capi.check(lib.dsen2_pack_dgrad_weights(_capi.ptr(torch.from_numpy(w).cuda()), C, C, C, C, 0.1, _capi.ptr(tw),
                                             _capi.stream_ptr()), 'pack dgrad')
    zero = torch.zeros(C, device='cuda')
    out = torch.zeros((n, H, W, C), dtype=torch.float16, device='cuda')
    tdy, tact = torch.from_numpy(dy).cuda(), torch.from_numpy(act).cuda()      # keep both alive across the launch
    _capi.check(lib.dsen2_conv_relu_bwd(_capi.ptr(tdy), _capi.ptr(tw), _capi.ptr(zero), _capi.ptr(tact), n, H, W, C,
                                        _capi.ptr(out), _capi.stream_ptr()), 'relu bwd')
    torch.cuda.synchronize()
    # reference: gradient of y = conv(x, w) w.r.t. x, times 0.1, masked by the forward activation
    wq = (np.float32(0.1) * w).astype(np.float16).astype(np.float64)           # operand as packed (scale folded, fp16)
    wt = torch.from_numpy(wq).permute(3, 2, 0, 1).contiguous()                     # (Cout, Cin, 3, 3)
    g = F.conv_transpose2d(torch.from_numpy(dy.astype(np.float64)).permute(0, 3, 1, 2), wt, padding=1)
    ref = np.where(act.astype(np.float32) > 0, g.permute(0, 2, 3, 1).numpy(), 0)
    got = out.cpu().numpy().astype(np.float64)
    ts.check(ts.pair_schedule(n, H, W), 'conv_relu_bwd C=%d' % C, np.abs(got - ref).max() / np.abs(ref).max())
    np.testing.assert_allclose(got, ref, rtol=2e-3, atol=2e-3 * np.abs(ref).max())


@pytest.mark.parametrize('F', [128, 256])
def test_pack_trunk_layers_equals_per_layer_packing(env, F):
    """One launch for all F -> F layers == dsen2_pack_conv_weights / dsen2_pack_dgrad_weights layer by layer (bit-exact)."""
    torch, _capi, lib = env
    L = 5
    rng = np.random.RandomState(F)
    stride = 9 * F * F + F                                  # kernels lie a kernel + a bias apart in the flat parameter vector
    flat = torch.from_numpy(rng.randn(L * stride).astype(np.float32)).cuda()
    fwd = torch.zeros((L, 9, F, F), dtype=torch.float16, device='cuda')
    bwd = torch.zeros_like(fwd)
    st = _capi.stream_ptr()
    _capi.check(lib.dsen2_pack_trunk_layers(_capi.ptr(flat), stride, L, F, 0.1, _capi.ptr(fwd), _capi.ptr(bwd), st), 'pack trunk')
    one_f = torch.zeros((9, F, F), dtype=torch.float16, device='cuda')
    one_b = torch.zeros_like(one_f)
    for l in range(L):
        k = flat[l * stride:l * stride + 9 * F * F]
        _capi.check(lib.dsen2_pack_conv_weights(_capi.ptr(k), F, F, F, F, _capi.ptr(one_f), st), 'pack')
        _capi.check(lib.dsen2_pack_dgrad_weights(_capi.ptr(k), F, F, F, F, 0.1 if l & 1 else 1.0, _capi.ptr(one_b), st), 'pack dgrad')
        torch.cuda.synchronize()
        assert torch.equal(fwd[l], one_f) and torch.equal(bwd[l], one_b)


def _setup(L=2, n=4, P=32, run_60=False, seed=0, F=128):
    from dsen2_b200.DSen2Net import s2model
    chans = (4, 6, 2) if run_60 else (4, 6)
    rng = np.random.RandomState(seed)
    model = s2model(tuple((c, None, None) for c in chans), num_layers=L, feature_size=F, seed=7)
    ws = model.get_weights()
    for i in range(1, len(ws), 2):
        ws[i] = (rng.randn(*ws[i].shape) * 0.05).astype(np.float32)
    model.set_weights(ws)
    xs = [(0.8 + 0.4 * rng.randn(n, c, P, P)).clip(0, 5).astype(np.float32) for c in chans]
    y = (xs[-1] + 0.1 * rng.randn(*xs[-1].shape)).astype(np.float32)
    return model, ws, xs, y


@pytest.mark.parametrize('cfg', [dict(L=2, n=4, P=32), dict(L=6, n=8, P=32), dict(L=1, n=2, P=32, run_60=True),
                                 dict(L=0, n=2, P=16), dict(L=2, n=4, P=32, F=256), dict(L=1, n=2, P=32, run_60=True, F=256),
                                 dict(L=4, n=8, P=32, F=256), dict(L=32, n=2, P=32, F=256), dict(L=2, n=128, P=32),
                                 dict(L=1, n=64, P=32, F=256)])
def test_gradients_vs_autograd(env, cfg):
    """n = 128 is DSen2's training batch (supres_train.py), n = 64 at F = 256 the benchmark's VDSen2 training step: there
    every convolution of the step runs several tiles per CTA (pair)."""
    torch, _capi, lib = env
    from dsen2_b200.train import Trainer
    from oracle import train_oracle as to
    model, ws, xs, y = _setup(**cfg)
    tr = Trainer(model)
    loss, mse = tr.train_step([torch.from_numpy(a).cuda() for a in xs], torch.from_numpy(y).cuda(), apply=False)
    ref_loss, ref_mse, ref_g = to.loss_and_grads(xs, y, [(ws[2 * i], ws[2 * i + 1]) for i in range(len(ws) // 2)])
    assert abs(float(loss) - ref_loss) <= 2e-3 * ref_loss + 1e-5
    assert abs(float(mse) - ref_mse) <= 5e-3 * ref_mse + 1e-6
    g = tr.grads.cpu().numpy()
    worst = 0.0
    for i, (gk, gb) in enumerate(ref_g):
        for ref, (o0, o1) in ((gk, (tr.offsets[2 * i], tr.offsets[2 * i + 1])), (gb, (tr.offsets[2 * i + 1], tr.offsets[2 * i + 2]))):
            got = g[o0:o1].reshape(ref.shape)
            err = np.abs(got - ref).max() / (np.abs(ref).max() + 1e-12)
            worst = max(worst, err)
            assert err <= 2e-2, "layer %d %s: relative gradient error %.3e" % (i, ref.shape, err)
    n, P = cfg['n'], cfg['P']
    label = 'training step %s, relative gradient' % cfg
    ts.check(ts.pair_schedule(n, P, P), label, worst)
    if cfg.get('F', 128) == 256:                     # the 256-feature step's last layer is the swapped tail
        ts.check(ts.tail_schedule(n, P, P), label, worst)


def test_mae_grad_at_the_training_batch(env):
    """dsen2_mae_grad over DSen2's batch (128 x 6 x 32 x 32 = 786,432 elements), where its grid-stride loop runs several
    times per thread: dpred = gscale * sign(fp32(pred - y)) bit for bit, +0 on exact ties; both double sums against float64
    numpy, accumulated on top of what the buffer holds."""
    torch, _capi, lib = env
    total = 128 * 6 * 32 * 32
    threads = min(-(-total // 256), 4 * ts.sm_count()) * 256      # grid_for(total, 256, 4)
    loops = -(-total // threads)
    print('mae_grad: %d elements over %d threads, %d iterations on the busiest thread' % (total, threads, loops))
    assert loops >= 3
    rng = np.random.RandomState(128)
    pred = (0.8 + 0.4 * rng.randn(total)).astype(np.float32)
    y = (pred + 0.1 * rng.randn(total)).astype(np.float32)
    tie = rng.rand(total) < 0.01
    y[tie] = pred[tie]
    gscale = np.float32(3.0 / 7.0)
    sums0 = np.array([123.5, -7.25])
    tp, ty = torch.from_numpy(pred).cuda(), torch.from_numpy(y).cuda()
    dpred = torch.full((total,), float('nan'), device='cuda')
    sums = torch.from_numpy(sums0).cuda()
    _capi.check(lib.dsen2_mae_grad(_capi.ptr(tp), _capi.ptr(ty), total, float(gscale), _capi.ptr(dpred), _capi.ptr(sums),
                                   _capi.stream_ptr()), 'mae')
    torch.cuda.synchronize()
    d = pred - y                                                     # float32, as the kernel subtracts
    got = dpred.cpu().numpy()
    assert np.array_equal(got.view(np.uint32), (gscale * np.sign(d)).view(np.uint32))
    assert tie.sum() > 1000 and not got[tie].view(np.uint32).any()   # +0, not -0
    d64 = d.astype(np.float64)
    ref = sums0 + np.array([np.abs(d64).sum(), (d64 * d64).sum()])
    got_s = sums.cpu().numpy()
    print('mae_grad sums: relative error %.3e %.3e' % tuple(np.abs(got_s - ref) / np.abs(ref)))
    np.testing.assert_allclose(got_s, ref, rtol=1e-10, atol=0)


@pytest.mark.parametrize('F', [128, 256])
def test_nadam_steps_vs_oracle(env, F):
    torch, _capi, lib = env
    from dsen2_b200.train import Nadam, Trainer
    from oracle import train_oracle as to
    model, ws, xs, y = _setup(L=2, n=4, P=32, F=F)
    lr = 1e-3
    tr = Trainer(model, Nadam(lr=lr))
    dx, dy = [torch.from_numpy(a).cuda() for a in xs], torch.from_numpy(y).cuda()
    losses = [float(tr.train_step(dx, dy)[0]) for _ in range(4)]
    ref_losses, ref_w = to.train_steps([(xs, y)] * 4, [(ws[2 * i], ws[2 * i + 1]) for i in range(len(ws) // 2)], lr=lr)
    np.testing.assert_allclose(losses, ref_losses, rtol=5e-3)
    assert losses[-1] < losses[0]
    got = tr.get_weights()
    # Nadam steps are ~lr per element and sign-like (an element whose tiny gradient flips sign under fp16 rounding moves
    # the other way), so compare the UPDATES statistically, in units of lr * steps
    d = np.concatenate([np.abs((got[2 * i + j] - ws[2 * i + j]) - (kb[j] - ws[2 * i + j])).ravel()
                        for i, kb in enumerate(ref_w) for j in (0, 1)]) / (lr * 4)
    print('update error / (lr*steps): median %.4f  p99 %.4f  max %.4f' % (np.median(d), np.percentile(d, 99), d.max()))
    assert np.median(d) < 0.02 and np.mean(d > 0.25) < 0.02
    # the exact Nadam arithmetic: feed the oracle's gradient through the kernel
    ref_loss, _, ref_g = to.loss_and_grads(xs, y, [(ws[2 * i], ws[2 * i + 1]) for i in range(len(ws) // 2)])
    tr2 = Trainer(model, Nadam(lr=lr))
    flat_g = np.concatenate([a.ravel() for kb in ref_g for a in kb]).astype(np.float32)
    p0 = tr2.params.cpu().numpy().astype(np.float64)
    m = np.zeros_like(p0); v = np.zeros_like(p0); ms = 1.0
    for t in range(1, 4):
        tr2.grads.copy_(torch.from_numpy(flat_g).cuda())
        tr2.apply_gradients(1.0)
        p0, m, v, ms = to.nadam_reference(p0, flat_g.astype(np.float64), m, v, t, ms, lr=lr)
        np.testing.assert_allclose(tr2.params.cpu().numpy(), p0, rtol=0, atol=5e-6)


def test_keras_like_compile_fit(env):
    model, ws, xs, y = _setup(L=1, n=8, P=32)
    with pytest.raises(RuntimeError):
        model.train_on_batch(xs, y)
    model.compile(optimizer='nadam', loss='mean_absolute_error', metrics=['mean_squared_error'])
    hist = model.fit(xs, y, batch_size=4, epochs=3, shuffle=True, seed=0)
    assert len(hist['loss']) == 3 and hist['loss'][-1] < hist['loss'][0]
    assert any(np.abs(a - b).max() > 0 for a, b in zip(model.get_weights(), ws))   # synced back into the model
    pred = model.predict(xs)                       # ... and the inference path runs on the trained weights
    assert abs(np.abs(pred - y).mean() - model.train_on_batch(xs, y)[0]) < 5e-3


@pytest.mark.parametrize('F', [128, 256])
def test_graph_replay_equals_eager_steps(env, F):
    """The CUDA-graph replay of the step (third call on) performs the same updates as the eager path."""
    torch, _capi, lib = env
    from dsen2_b200.train import Nadam, Trainer
    model, ws, xs, y = _setup(L=2, n=4, P=32, F=F)
    dx, dy = [torch.from_numpy(a).cuda() for a in xs], torch.from_numpy(y).cuda()
    runs = []
    for use_graph in (False, True):
        model.set_weights(ws)
        tr = Trainer(model, Nadam(lr=1e-3))
        tr.use_graph = use_graph
        losses = [float(tr.train_step(dx, dy)[0]) for _ in range(5)]
        assert tr.iterations == 5
        runs.append((losses, tr.params.cpu().numpy()))
    np.testing.assert_allclose(runs[0][0], runs[1][0], rtol=2e-3)   # fp32 reduction order differs run to run
    # fp32 atomics in the weight-gradient reduction make the two runs differ in the last bits only
    d = np.abs(runs[0][1] - runs[1][1]) / (1e-3 * 5)
    assert np.median(d) < 1e-3 and np.mean(d > 0.25) < 0.01


def test_fit_with_validation_and_callbacks(env, tmp_path):
    """model.fit as supres_train.py:218-230 uses it: validation_data, best-only checkpoints, LR reduction; evaluate()
    agrees with the oracle's loss; the checkpoint is a Keras-style weight file the model can load again."""
    from dsen2_b200.callbacks import LossLog, ModelCheckpoint, ReduceLROnPlateau
    from dsen2_b200.train import Nadam
    from oracle import train_oracle as to
    model, ws, xs, y = _setup(L=1, n=12, P=32)
    model.compile(optimizer=Nadam(lr=2e-3), loss='mean_absolute_error', metrics=['mean_squared_error'])
    ref_loss, ref_mse, _ = to.loss_and_grads([a[8:] for a in xs], y[8:], [(ws[2 * i], ws[2 * i + 1]) for i in range(len(ws) // 2)])
    ev = model.evaluate([a[8:] for a in xs], y[8:], batch_size=4)
    assert abs(ev[0] - ref_loss) <= 2e-3 * ref_loss and abs(ev[1] - ref_mse) <= 5e-3 * ref_mse
    ck = str(tmp_path / 'ck.hdf5')
    cbs = [ModelCheckpoint(ck, monitor='val_loss', save_best_only=True),
           ReduceLROnPlateau(monitor='val_loss', factor=0.5, patience=1, epsilon=10.0, cooldown=0, min_lr=1e-4),
           LossLog(str(tmp_path / 'log.txt'))]
    hist = model.fit([a[:8] for a in xs], y[:8], batch_size=4, epochs=4, callbacks=cbs,
                     validation_data=([a[8:] for a in xs], y[8:]), seed=0)
    assert len(hist['val_loss']) == 4 and hist['loss'][-1] < hist['loss'][0]
    assert model.optimizer.lr < 2e-3                      # epsilon = 10 makes every epoch a "plateau": the LR was cut
    assert open(str(tmp_path / 'log.txt')).read().count('Finished epoch') == 4
    from dsen2_b200.DSen2Net import s2model
    again = s2model(((4, None, None), (6, None, None)), num_layers=1, feature_size=128)
    again.load_weights(ck)
    best = int(np.argmin(hist['val_loss']))
    if best == 3:                                          # the last epoch was the best: the file holds the final weights
        for a, b in zip(again.get_weights(), model.get_weights()):
            assert np.array_equal(a, b)


@pytest.mark.parametrize('deep', [False, True])
def test_supres_train_cli_trains_and_predicts(env, tmp_path, deep):
    """python -m dsen2_b200.supres_train [--deep] on a tiny synthetic data set laid out like the reference's ../data/."""
    import json
    from dsen2_b200 import supres_train
    rng = np.random.RandomState(3)
    root = str(tmp_path) + '/'
    d = tmp_path / 'train' / 'S2A_X.SAFE'
    d.mkdir(parents=True)
    x10 = (0.8 + 0.3 * rng.randn(16, 4, 32, 32)).clip(0, 4).astype(np.float32) * 2000
    x20 = (0.8 + 0.3 * rng.randn(16, 6, 32, 32)).clip(0, 4).astype(np.float32) * 2000
    np.save(d / 'data10.npy', x10); np.save(d / 'data20.npy', x20)
    np.save(d / 'data20_gt.npy', (x20 + 50 * rng.randn(*x20.shape)).astype(np.float32))
    val = np.zeros(16, bool); val[::4] = True
    np.save(tmp_path / 'train' / 'val_index.npy', val)
    flags = ['--deep'] if deep else []
    assert supres_train.main(['--path', root, '--epochs', '2'] + flags) == 0
    ck = root + 'network_data/' + supres_train.model_nr + 'lr_1e-04.hdf5'
    import os
    assert os.path.exists(ck) and 'Finished epoch' in open(root + 'network_data/' + supres_train.model_nr + '_lr_1.0e-04.txt').read()
    t = tmp_path / 'test' / 'S2A_Y.SAFE'
    t.mkdir(parents=True)
    np.save(t / 'data10.npy', x10[:4]); np.save(t / 'data20.npy', x20[:4])
    json.dump([0, 0, 48, 48], open(t / 'roi.json', 'w'))
    assert supres_train.main(['--path', root, '--predict', ck] + flags) == 0
    out = np.load(str(t / (ck[-20:-13] + '-predict.npy')))
    assert out.shape == (48, 48, 6) and np.isfinite(out).all()


def test_model_and_trainer_weights_stay_in_sync(env, tmp_path):
    """Keras semantics around compile(): load_weights AFTER compile trains from the loaded weights (supres_train.py:143,183),
    and predict / get_weights / save_weights after train_on_batch see the UPDATED weights."""
    torch, _capi, lib = env
    from dsen2_b200.DSen2Net import s2model
    from dsen2_b200.train import Nadam
    model, ws, xs, y = _setup(L=1, n=4, P=32)
    other = s2model(((4, None, None), (6, None, None)), num_layers=1, feature_size=128, seed=77)
    wf = str(tmp_path / 'w.hdf5')
    other.save_weights(wf)
    model.compile(optimizer=Nadam(lr=1e-3), loss='mean_absolute_error', metrics=['mean_squared_error'])
    model.load_weights(wf)                                  # compile, THEN load: the trainer must pick the new weights up
    for a, b in zip(model._trainer.get_weights(), other.get_weights()):
        assert np.array_equal(a, b)
    before = model.predict(xs)
    assert np.array_equal(before, other.predict(xs))
    for _ in range(3):
        model.train_on_batch(xs, y)
    after_w = model.get_weights()                           # no explicit sync call
    assert not np.array_equal(after_w[0], other.get_weights()[0])
    for a, b in zip(after_w, model._trainer.get_weights()):
        assert np.array_equal(a, b)
    after = model.predict(xs)
    assert not np.array_equal(after, before)
    model.save_weights(wf)
    again = s2model(((4, None, None), (6, None, None)), num_layers=1, feature_size=128)
    again.load_weights(wf)
    assert np.array_equal(again.predict(xs), after)


def test_back_to_back_graph_steps_use_their_own_nadam_scalars(env):
    """train_step returns without synchronising: the step-dependent scalars (mu_t, bias correction ...) must not be
    overwritten on the host before their upload has run.  Unsynchronised back-to-back steps == synchronised steps."""
    torch, _capi, lib = env
    from dsen2_b200.train import Nadam, Trainer
    model, ws, xs, y = _setup(L=1, n=4, P=32)
    dx, dy = [torch.from_numpy(a).cuda() for a in xs], torch.from_numpy(y).cuda()
    outs = []
    for sync in (True, False):
        model.set_weights(ws)
        tr = Trainer(model, Nadam(lr=1e-3))
        for _ in range(12):
            tr.train_step(dx, dy)
            if sync:
                torch.cuda.synchronize()
        torch.cuda.synchronize()
        outs.append(tr.params.cpu().numpy())
    d = np.abs(outs[0] - outs[1]) / (1e-3 * 12)
    assert np.median(d) < 1e-3 and np.mean(d > 0.25) < 0.01     # fp32 atomics in the weight gradients: last-bit noise only


def test_capture_while_a_dropped_trainer_awaits_collection(env):
    """A dropped model and its trainer form a reference cycle that keeps the trainer's CUDA graph until the cyclic collector
    runs.  Destroying a graph while another stream captures invalidates that capture, so the collector must not run
    during a capture: with collections due on every allocation, another model still captures and replays its steps, the
    collector is off inside the capture and on again afterwards, and the dropped trainer is collected after it."""
    import gc
    import weakref
    torch, _capi, lib = env
    from dsen2_b200.train import Nadam
    model, ws, xs, y = _setup(L=1, n=4, P=32)
    model.compile(optimizer=Nadam(lr=1e-3), loss='mean_absolute_error')
    for _ in range(3):
        model.train_on_batch(xs, y)                             # the second step captures the graph
    assert model._trainer._graphs
    dropped = weakref.ref(model._trainer)
    del model
    again = _setup(L=1, n=4, P=32)[0]
    again.compile(optimizer=Nadam(lr=1e-3), loss='mean_absolute_error')
    tr = again._trainer
    collector_on = []
    repack = tr.repack
    tr.repack = lambda: (collector_on.append(gc.isenabled()), repack())[1]
    threshold = gc.get_threshold()
    gc.set_threshold(1, 1, 1)
    try:
        losses = [float(np.asarray(again.train_on_batch(xs, y)).ravel()[0]) for _ in range(3)]
    finally:
        gc.set_threshold(*threshold)
    torch.cuda.synchronize()
    assert tr._graphs and np.isfinite(losses).all()
    assert collector_on[:2] == [True, False] and gc.isenabled()  # eager first step, then the capture
    gc.collect()
    assert dropped() is None


def test_full_model_checkpoint_resumes_training(env, tmp_path):
    """model.save (ModelCheckpoint(save_weights_only=False), supres_train.py:195-201) carries the Nadam state: a model rebuilt
    from the file continues exactly like the one that kept training."""
    torch, _capi, lib = env
    from dsen2_b200.DSen2Net import s2model
    from dsen2_b200.hdf5 import File
    from dsen2_b200.train import Nadam
    model, ws, xs, y = _setup(L=1, n=4, P=32)
    model.compile(optimizer=Nadam(lr=1e-3), loss='mean_absolute_error', metrics=['mean_squared_error'])
    for _ in range(5):
        model.train_on_batch(xs, y)
    ck = str(tmp_path / 'full.hdf5')
    model.save(ck)
    f = File(ck)
    assert sorted(f.keys()) == ['model_weights', 'optimizer_weights']
    names = [bytes(n).decode() for n in f['optimizer_weights'].attrs['weight_names']]
    assert names[0] == 'Nadam/iterations:0' and len(names) == 1 + 2 * 2 * len(model.layer_shapes)
    assert int(np.asarray(f['optimizer_weights/Nadam/iterations:0'][()]).reshape(-1)[0]) == 5
    k0 = model.get_weights()[0]
    assert f['optimizer_weights/training/Nadam/m_0:0'].shape == (k0.size,)
    for _ in range(4):
        model.train_on_batch(xs, y)
    want = np.concatenate([a.ravel() for a in model.get_weights()])

    again = s2model(((4, None, None), (6, None, None)), num_layers=1, feature_size=128, seed=99)
    again.compile(optimizer=Nadam(lr=1e-3), loss='mean_absolute_error', metrics=['mean_squared_error'])
    again.load_weights(ck)
    assert again.load_optimizer_weights(ck)
    assert again._trainer.iterations == 5 and again._trainer.m_schedule == pytest.approx(model_schedule(5))
    for _ in range(4):
        again.train_on_batch(xs, y)
    got = np.concatenate([a.ravel() for a in again.get_weights()])
    d = np.abs(got - want) / (1e-3 * 4)
    assert np.median(d) < 1e-3 and np.mean(d > 0.25) < 0.01     # fp32 atomics in the weight gradients: last-bit noise only

    cold = s2model(((4, None, None), (6, None, None)), num_layers=1, feature_size=128, seed=99)
    cold.compile(optimizer=Nadam(lr=1e-3), loss='mean_absolute_error', metrics=['mean_squared_error'])
    cold.load_weights(ck)                                       # weights only: the moments restart from zero
    for _ in range(4):
        cold.train_on_batch(xs, y)
    dc = np.abs(np.concatenate([a.ravel() for a in cold.get_weights()]) - want) / (1e-3 * 4)
    assert np.mean(dc > 0.25) > 0.2                             # ...which is visibly a different trajectory


def model_schedule(t, opt=None):
    from dsen2_b200.train import Nadam, nadam_schedule
    prod, opt = 1.0, opt or Nadam()
    for i in range(1, t + 1):
        prod = nadam_schedule(i, prod, opt)['sched_new']
    return prod


def test_vdsen2_training_step_at_depth_32(env):
    """supres_train.py:129-131 (--deep): 32 resBlocks x 256 features, batch size 8.  The step runs, the loss follows the
    fp32 oracle and decreases; predict() afterwards sees the trained weights."""
    torch, _capi, lib = env
    from dsen2_b200.train import Nadam
    from oracle import train_oracle as to
    model, ws, xs, y = _setup(L=32, n=8, P=32, F=256)
    model.compile(optimizer=Nadam(lr=1e-4), loss='mean_absolute_error', metrics=['mean_squared_error'])
    losses = [model.train_on_batch(xs, y)[0] for _ in range(6)]
    with torch.no_grad():                             # the oracle's forward pass only (66 layers x 256 features on the CPU)
        pred = to.forward([torch.from_numpy(a) for a in xs], to._params([(ws[2 * i], ws[2 * i + 1]) for i in range(len(ws) // 2)]))
    ref_loss = float((pred - torch.from_numpy(y)).abs().mean())
    assert np.isfinite(losses).all()
    assert abs(losses[0] - ref_loss) <= 5e-3 * ref_loss
    assert losses[-1] < losses[0]
    pred = model.predict(xs)
    assert abs(np.abs(pred - y).mean() - model.train_on_batch(xs, y)[0]) < 5e-3
