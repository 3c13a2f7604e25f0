"""The training step (Trainer._step_body, ~65 launches) layer by layer against float64 on its own operands
(train_reference.py), for DSen2, VDSen2 and both input sets.

Bounds.  Every operand the kernels multiply is fp16, so each product is exact and only the fp32 accumulation differs
from float64.  A tensor-core step adds up to 16 exact products to the fp32 accumulator with an error of at most
2u (|acc| + sum |products|) (u = 2^-24; the products are aligned and truncated before they are added), and a plain fp32
addition adds at most u |sum|.  A chain of m tensor-core steps and r further fp32 operations therefore stays within
(2m + r) u S, where S is the float64 sum of |terms| of that entry.  Per kernel:
  - weight gradient (dsen2_wgrad_nhwc): a CTA sums `per` tiles of 128 pixels in 8 steps each, the result is scaled and
    reduced over `splits` CTAs: m = 8 per, r = splits + 2;
    bias gradient: a drain thread adds ceil(64 / nshare) values per tile, then 2 nshare splits partial sums meet in fp32
    atomics: r = per ceil(64 / nshare) + 2 nshare splits + 2 (nshare = 3 F / 128);
  - forward convolutions: m = 9 F / 16 (fp16 trunk operands) or 4 x that (the hi / lo split of the first and last layer),
    r = 4 for the bias, the residual scale and update and the final rounding.
Gradients below the last layer are also computed from the trainer's fp16 dx_hi and g2, which differ from the
reference's where a sum lands next to a rounding boundary.  These flips are not rare and they do grow: a flipped g2 moves
dx32, which flips more of the next dx_hi.  Measured on a B200, 3 % (one resBlock) to 21 % (six) of the final dx_hi differ,
up to 100 ulps where the value is near zero.  Their effect on an entry has no bound in terms of that entry's own |terms| (an
entry whose terms are nearly all masked can be moved by more than its S), so it is charged to the tensor: DRIFT times the
largest |gradient| of that tensor, 3.5x the worst drift measured (1.75e-5).  The last layer's gradient has no such term:
its operands dpred and x_hi[L] are the trainer's own.  An fp16 forward tensor must lie within half an fp16 ulp of its
float64 value plus the accumulation bound, which allows one ulp where the value is large and more only where it is
within that bound of zero.
"""
import math

import numpy as np
import pytest

import tile_schedule as ts
import train_reference as tref

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
DRIFT = 2.0 ** -14          # divergence of the two fp16 backward chains, relative to a tensor's largest |gradient|
FLIPS = 0.3                 # fraction of the final dx_hi that may differ from the reference's (21 % measured at L = 6)
FWD_FLIPS = 2.0 ** -6       # the same for the forward fp16 tensors, which are compared layer by layer (0.7 % measured)

CASES = {
    'dsen2-batch128': dict(L=6, F=128, n=128, P=32, chans=(4, 6)),   # the bench's training line: 7 tiles per CTA pair
    '60m': dict(L=2, F=128, n=16, P=32, chans=(4, 6, 2)),            # 12 inputs, 2 outputs, skip channel 10
    'no-resblocks': dict(L=0, F=128, n=4, P=32, chans=(4, 6)),       # dsen2_conv_head writes x_hi and x_lo for the tail
    'vdsen2': dict(L=4, F=256, n=8, P=32, chans=(4, 6)),             # 16-channel head and tail, 128 x 128 gradient blocks
    'vdsen2-60m': dict(L=1, F=256, n=4, P=32, chans=(4, 6, 2)),
    'patch40': dict(L=2, F=128, n=4, P=40, chans=(4, 6)),            # 40 = 2.5 tile rows: partial tiles in every kernel
}


def _sms():
    return ts.sm_count()


def wgrad_tol(n, P, F, bias=False):
    """(2m + r) u of dsen2_wgrad_nhwc's entry point and kernel (see the module docstring)."""
    tiles = n * -(-P // 8) * -(-P // 16)
    blocks = (F // 128) ** 2
    splits = min(_sms() // (3 * blocks), tiles)
    per = -(-tiles // splits)
    splits = -(-tiles // per)
    if bias:
        nshare = 3 * (F // 128)
        return (per * -(-64 // nshare) + 2 * nshare * splits + 2) * U
    return (2 * 8 * per + splits + 2) * U


def conv_tol(F, split=False):
    return (2 * 9 * F // 16 * (4 if split else 1) + 4) * U


def _ulp16(v):
    """Spacing of the fp16 numbers at |v| (2^-24 among the subnormals and at zero)."""
    _, e = np.frexp(np.abs(v))
    return np.where(v == 0, 2.0 ** -24, np.maximum(np.ldexp(1.0, e - 11), 2.0 ** -24))


def _check_f16(got, ref, bound, label, fails):
    """got: fp16 tensor (any layout, as numpy float64), ref: float64, bound: the accumulation bound per element."""
    err = np.abs(got - ref)
    allowed = 0.5 * _ulp16(got) + bound
    flips = float(np.mean(got.astype(np.float16) != ref.astype(np.float16)))
    print('  %-22s flips %.2e  max err %.2e  max err / (ulp/2 + bound) %.3f' % (label, flips, err.max(), (err / allowed).max()))
    if (err > allowed).any() or flips > FWD_FLIPS:
        fails.append('%s: %d elements outside the bound, %.2e flipped' % (label, int((err > allowed).sum()), flips))


def _setup(L, F, n, P, chans, seed=0):
    from dsen2_b200.DSen2Net import s2model
    rng = np.random.RandomState(seed + n + L)
    model = s2model(tuple((c, None, None) for c in chans), num_layers=L, feature_size=F, seed=7)
    ws = model.get_weights()
    for i in range(1, len(ws), 2):
        ws[i] = (rng.randn(*ws[i].shape) * 0.05).astype(np.float32)
    model.set_weights(ws)
    xs = [(0.8 + 0.4 * rng.randn(n, c, P, P)).clip(0, 5).astype(np.float32) for c in chans]
    y = (xs[-1] + 0.1 * rng.randn(*xs[-1].shape)).astype(np.float32)
    return model, xs, y


def _snapshot(tr, n, P):
    b = tr._bufs[(n, P)]
    keep = ('x_hi', 't', 'x_lo', 'xin_hi', 'xin_lo', 'pred', 'dx_hi')
    return {k: ([a.clone() for a in b[k]] if isinstance(b[k], list) else b[k].clone()) for k in keep}


def _keras(tr, flat):
    """Flat fp32 parameter (or gradient) vector -> Keras order list of arrays."""
    host = flat.cpu().numpy()
    out = []
    for i, (cin, cout) in enumerate(tr.model.layer_shapes):
        out.append(host[tr.offsets[2 * i]:tr.offsets[2 * i + 1]].reshape(3, 3, cin, cout))
        out.append(host[tr.offsets[2 * i + 1]:tr.offsets[2 * i + 2]])
    return out


@pytest.fixture(scope='module', params=sorted(CASES))
def step(request):
    """One case: an eager step without update (its forward tensors and gradient kept), then three steps with the update --
    eager, captured and replayed, replayed -- with the state before the third kept."""
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from dsen2_b200.train import Nadam, Trainer
    cfg = CASES[request.param]
    n, P = cfg['n'], cfg['P']
    model, xs, y = _setup(**cfg)
    tr = Trainer(model, Nadam(lr=1e-3))
    tr.use_graph = True
    dx, dy = [torch.from_numpy(a).cuda() for a in xs], torch.from_numpy(y).cuda()
    weights = tr.get_weights()
    loss, mse = tr.train_step(dx, dy, apply=False)
    torch.cuda.synchronize()
    eager = dict(bufs=_snapshot(tr, n, P), grads=tr.grads.clone(), loss=float(loss), mse=float(mse), weights=weights)
    tr.train_step(dx, dy)
    tr.train_step(dx, dy)
    torch.cuda.synchronize()
    before = dict(params=tr.params.clone(), m=tr.m.clone(), v=tr.v.clone(), iterations=tr.iterations,
                  m_schedule=tr.m_schedule, weights=tr.get_weights())
    tr.train_step(dx, dy)
    torch.cuda.synchronize()
    assert (n, P, len(xs)) in tr._graphs
    replay = dict(bufs=_snapshot(tr, n, P), grads=tr.grads.clone(), params=tr.params.clone(), m=tr.m.clone(), v=tr.v.clone())
    return dict(name=request.param, cfg=cfg, tr=tr, xs=dx, y=dy, eager=eager, before=before, replay=replay)


def _schedule(st, label, worst):
    n, P, F = st['cfg']['n'], st['cfg']['P'], st['cfg']['F']
    ts.check(ts.pair_schedule(n, P, P), '%s %s' % (st['name'], label), worst)
    if F == 256:
        ts.check(ts.tail_schedule(n, P, P), '%s %s' % (st['name'], label), worst)


def test_forward_layers_teacher_forced(step):
    """Each forward tensor against float64 of its layer on the trainer's own previous tensors; the prepared input bit for
    bit against the split of the inputs."""
    import torch
    cfg, bufs = step['cfg'], step['eager']['bufs']
    F, L = cfg['F'], cfg['L']
    fails = []
    # prepared input: hi = f16(x), lo = f16(x - hi) of the concatenated inputs (centre tap of the 64-channel form)
    xcat = torch.cat(step['xs'], 1).permute(0, 2, 3, 1)
    c0 = 16 if bufs['xin_hi'].shape[-1] == 64 else 0
    ctot = xcat.shape[-1]
    hi = xcat.half()
    assert torch.equal(bufs['xin_hi'][..., c0:c0 + ctot], hi)
    assert torch.equal(bufs['xin_lo'][..., c0:c0 + ctot], (xcat - hi.float()).half())
    r = tref.layer_references(bufs, step['eager']['weights'])
    npy = lambda a: a.cpu().numpy()
    nhwc = lambda a: npy(a.permute(0, 2, 3, 1))
    f16 = lambda a: npy(a).astype(np.float64)
    print('\n%s forward:' % step['name'])
    tol_head = conv_tol(16 if F == 256 else 64, split=True)
    _check_f16(f16(bufs['x_hi'][0]), nhwc(r['head']), tol_head * nhwc(r['head_mag']), 'x_hi[0] (head)', fails)
    trunk_err = tol_head * nhwc(r['head_mag'])
    for l in range(L):
        _check_f16(f16(bufs['t'][l]), nhwc(r['t'][l]), conv_tol(F) * nhwc(r['t_mag'][l]), 't[%d]' % l, fails)
        trunk_err = trunk_err + conv_tol(F) * (0.1 * nhwc(r['c2_mag'][l]) + np.abs(nhwc(r['trunk'][l])))
        _check_f16(f16(bufs['x_hi'][l + 1]), nhwc(r['trunk'][l + 1]), trunk_err, 'x_hi[%d] (trunk)' % (l + 1), fails)
    # x_lo = f16(trunk32 - x_hi[L]): the pair carries the fp32 trunk to the last layer
    pair = f16(bufs['x_hi'][L]) + f16(bufs['x_lo'])
    err = np.abs(pair - nhwc(r['trunk'][L]))
    bound = trunk_err + 2.0 ** -11 * np.abs(f16(bufs['x_lo'])) + 2.0 ** -24
    print('  %-22s max err %.2e  max err / bound %.3f' % ('x_hi[L] + x_lo', err.max(), (err / bound).max()))
    if (err > bound).any():
        fails.append('x_hi[L] + x_lo: %d elements outside the bound' % int((err > bound).sum()))
    got = npy(bufs['pred']).astype(np.float64)
    err = np.abs(got - npy(r['pred']))
    bound = conv_tol(F, split=True) * npy(r['pred_mag'])
    worst = float((err / bound).max())
    print('  %-22s max err %.2e  max err / bound %.3f' % ('pred', err.max(), worst))
    if (err > bound).any():
        fails.append('pred: %d elements outside the bound' % int((err > bound).sum()))
    _schedule(step, 'forward, worst pred error / bound', worst)
    assert not fails, fails


def test_loss_equals_float64_sums(step):
    import torch
    pred, y = step['eager']['bufs']['pred'], step['y']
    d = (pred - y).double()                                  # fp32 difference, as dsen2_mae_grad takes it
    loss, mse = d.abs().mean().item(), (d * d).mean().item()
    print('\n%s loss %.6e (rel err %.1e)  mse %.6e (rel err %.1e)' % (
        step['name'], loss, abs(step['eager']['loss'] - loss) / loss, mse, abs(step['eager']['mse'] - mse) / mse))
    assert abs(step['eager']['loss'] - loss) <= 1e-10 * loss
    assert abs(step['eager']['mse'] - mse) <= 1e-10 * mse
    assert torch.isfinite(pred).all()


def _layer_names(L):
    return ['head'] + ['conv1[%d]' % l if i == 0 else 'conv2[%d]' % l for l in range(L) for i in range(2)] + ['tail']


def _check_gradients(st, run, weights, label):
    """tr.grads of one step against train_reference.step_gradients on that step's forward tensors and weights."""
    cfg, tr = st['cfg'], st['tr']
    n, P, F, L = cfg['n'], cfg['P'], cfg['F'], cfg['L']
    ref = tref.step_gradients(run['bufs'], st['xs'], st['y'], weights, magnitudes=True)
    got = [a.astype(np.float64) for a in _keras(tr, run['grads'])]
    # the final dx_hi: the fp16 gradient after the whole backward-data chain
    dxg = run['bufs']['dx_hi'].double().cpu().numpy()
    dxr = ref['dx_hi'].cpu().numpy()
    flips = float(np.mean(dxg.astype(np.float16) != dxr.astype(np.float16)))
    ulps = float((np.abs(dxg - dxr) / _ulp16(dxr)).max())
    print('\n%s %s: final dx_hi flips %.2e, max %.1f ulp' % (st['name'], label, flips, ulps))
    fails = [] if flips <= FLIPS else ['final dx_hi: %.2e of the elements flipped' % flips]
    names = _layer_names(L)
    worst = 0.0
    classes = {}
    for i, (g, r, mag) in enumerate(zip(got, ref['grads'], ref['mags'])):
        r, mag = r.cpu().numpy(), mag.cpu().numpy()
        layer, kind = names[i // 2], 'bias' if i % 2 else 'kernel'
        tail = i // 2 == 2 * L + 1
        tol = wgrad_tol(n, P, F, bias=i % 2 == 1)
        err = np.abs(g - r)
        bound = tol * mag + (U * mag.max() if tail else DRIFT * np.abs(r).max())
        rel_s = float((err / (mag + 1e-300)).max())
        rel_max = float(err.max() / np.abs(r).max())
        ratio = float((err / bound).max())
        worst = max(worst, ratio)
        print('  %-10s %-6s err/S %.2e  (%.2e)  err/max|g| %.2e  (%s, old 2e-2)  err/bound %.2f' % (
            layer, kind, rel_s, tol, rel_max, 'none' if tail else '%.1e' % DRIFT, ratio))
        cls = (layer.split('[')[0], kind)
        c = classes.setdefault(cls, [0.0, 0.0, tol])
        c[0], c[1] = max(c[0], rel_s), max(c[1], rel_max)
        if (err > bound).any():
            fails.append('%s %s: %d entries outside the bound, worst %.2e of S' % (layer, kind, int((err > bound).sum()), rel_s))
    for (layer, kind), (rs, rm, tol) in sorted(classes.items()):
        print('  class %-6s %-6s worst err/S %.2e  (%.2e)  worst err/max|g| %.2e' % (layer, kind, rs, tol, rm))
    _schedule(st, '%s, worst gradient error / bound' % label, worst)
    return fails


def test_gradients_vs_float64_reference(step):
    """Every gradient tensor of the eager step (kernels and biases) against the reference on the step's own forward
    tensors, to the accumulation bound of its entries (module docstring)."""
    fails = _check_gradients(step, step['eager'], step['eager']['weights'], 'eager step')
    assert not fails, fails


def test_graph_replay_gradients_and_nadam_update(step):
    """The third step replays the captured graph: its gradient against the reference on the replay's forward tensors and
    the weights before it; params, m and v against oracle.nadam_reference of the GPU's own gradient at that iteration.
    Update tolerances: fp32 evaluation of Keras-2 Nadam, ~15 roundings (< 2^-20 relative to the terms), plus 1 - beta_2
    taken from the fp32 beta_2 (1.3e-5 relative on the g^2 term of v, half that on the step).  The step is measured
    against its two terms lr (|(1 - mu_t) g'| + |mu_next m'|) / (sqrt(v') + eps), which can cancel."""
    from dsen2_b200.train import nadam_schedule
    from oracle import train_oracle as to
    tr, before, run = step['tr'], step['before'], step['replay']
    fails = _check_gradients(step, run, before['weights'], 'graph replay')
    t = before['iterations'] + 1
    assert tr.iterations == t
    p0, m0, v0 = (before[k].double().cpu().numpy() for k in ('params', 'm', 'v'))
    g = run['grads'].double().cpu().numpy()
    o = tr.opt
    p, m, v, ms = to.nadam_reference(p0, g, m0, v0, t, before['m_schedule'], lr=o.lr, b1=o.beta_1, b2=o.beta_2,
                                     eps=o.epsilon, decay=o.schedule_decay)
    assert math.isclose(tr.m_schedule, ms, rel_tol=1e-12)
    got = {k: run[k].double().cpu().numpy() for k in ('params', 'm', 'v')}
    sc = nadam_schedule(t, before['m_schedule'], o)
    terms = o.lr * ((1 - sc['mu_t']) * np.abs(g) / (1 - sc['sched_new']) + sc['mu_next'] * np.abs(m) / (1 - sc['sched_next'])) / (
        np.sqrt(v / sc['bias2']) + o.epsilon)
    bounds = dict(params=2.0 ** -23 * np.abs(p) + 2.0 ** -16 * terms,
                  m=2.0 ** -20 * (np.abs(o.beta_1 * m0) + np.abs((1 - o.beta_1) * g)),
                  v=2.0 ** -20 * o.beta_2 * v0 + 2.0 ** -15 * (1 - o.beta_2) * g * g)
    for k, want in (('params', p), ('m', m), ('v', v)):
        err = np.abs(got[k] - want)
        print('  nadam %-6s max err %.2e  max err / bound %.3f' % (k, err.max(), (err / (bounds[k] + 1e-300)).max()))
        if (err > bounds[k]).any():
            fails.append('nadam %s: %d elements outside the bound' % (k, int((err > bounds[k]).sum())))
    assert np.abs(p - p0).max() > 0
    assert not fails, fails
