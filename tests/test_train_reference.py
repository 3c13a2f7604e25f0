"""The float64 restatement of the training step (train_reference.py) on CPU: with its roundings switched off it must
compute the gradient of the exact graph, so that the GPU tests may use it to judge the kernels."""
import numpy as np
import pytest
import torch

import train_reference as tref
from emulate import forward_exact


def _net(L, chans, F=128, P=12, n=2, seed=0):
    rng = np.random.RandomState(seed + 10 * L + len(chans))
    ctot, cout = sum(chans), chans[-1]
    shapes = [(ctot, F)] + [(F, F)] * (2 * L) + [(F, cout)]
    ws = []
    for cin, co in shapes:
        lim = np.sqrt(6.0 / (9 * cin))
        ws += [rng.uniform(-lim, lim, size=(3, 3, cin, co)).astype(np.float32), (rng.randn(co) * 0.05).astype(np.float32)]
    xs = [(0.8 + 0.4 * rng.randn(n, c, P, P)).clip(0, 5).astype(np.float32) for c in chans]
    y = (xs[-1] + 0.1 * rng.randn(*xs[-1].shape)).astype(np.float32)
    return ws, xs, y


def _autograd(ws, xs, y, scale=0.1):
    """torch.autograd of the graph emulate.forward_exact evaluates (DSen2Net.py:18-43), float64, loss mean |pred - y|."""
    from oracle import train_oracle as to
    ps = [torch.tensor(np.ascontiguousarray(a.transpose(3, 2, 0, 1) if a.ndim == 4 else a), dtype=torch.float64,
                       requires_grad=True) for a in ws]
    pred = to.forward([torch.tensor(a, dtype=torch.float64) for a in xs], ps, scale)
    exact = forward_exact(xs, [(ws[2 * i], ws[2 * i + 1]) for i in range(len(ws) // 2)], scale)
    assert np.abs(pred.detach().numpy() - exact).max() <= 1e-12 * np.abs(exact).max()
    (pred - torch.tensor(y, dtype=torch.float64)).abs().mean().backward()
    return [p.grad.permute(2, 3, 1, 0) if p.ndim == 4 else p.grad for p in ps]


@pytest.mark.parametrize('chans', [(4, 6), (4, 6, 2)], ids=['20m', '60m'])
@pytest.mark.parametrize('L', [0, 2])
def test_reference_gradients_without_rounding_equal_autograd(L, chans):
    ws, xs, y = _net(L, chans)
    bufs = tref.exact_buffers(xs, ws)
    out = tref.step_gradients(bufs, xs, y, ws, rounding=False, magnitudes=True)
    ref = _autograd(ws, xs, y)
    assert len(out['grads']) == len(ref) == 4 * L + 4
    for i, (got, want, mag) in enumerate(zip(out['grads'], ref, out['mags'])):
        assert got.shape == want.shape, i
        err = (got - want).abs().max().item()
        assert err <= 1e-12 * want.abs().max().item(), (i, err)
        assert (mag >= got.abs() * (1 - 1e-12)).all(), i         # |sum| <= sum |products|
    # with the roundings on, the gradients move by the fp16 rounding of the operands, and only by that
    rounded = tref.step_gradients(bufs, xs, y, ws)['grads']
    moved = [(got - want).abs().max().item() / want.abs().max().item() for got, want in zip(rounded, ref)]
    assert 1e-5 < max(moved) <= 2e-2, moved


@pytest.mark.parametrize('chans', [(4, 6), (4, 6, 2)], ids=['20m', '60m'])
@pytest.mark.parametrize('L', [0, 2])
def test_layer_references_reproduce_the_exact_forward(L, chans):
    """Teacher-forced on the exact forward tensors, every layer restatement returns the next tensor."""
    ws, xs, y = _net(L, chans)
    bufs = tref.exact_buffers(xs, ws)
    r = tref.layer_references(bufs, ws, rounding=False)
    close = lambda a, b: (a - b).abs().max().item() <= 1e-12 * max(1.0, b.abs().max().item())
    assert close(r['head'], tref.nchw(bufs['x_hi'][0], 'cpu'))
    for l in range(L):
        assert close(r['t'][l], tref.nchw(bufs['t'][l], 'cpu'))
        assert close(r['trunk'][l + 1], tref.nchw(bufs['x_hi'][l + 1], 'cpu'))
    assert close(r['pred'], bufs['pred'])
    exact = forward_exact(xs, [(ws[2 * i], ws[2 * i + 1]) for i in range(len(ws) // 2)])
    assert np.abs(r['pred'].numpy() - exact).max() <= 1e-12 * np.abs(exact).max()
    assert (r['pred_mag'] >= r['pred'].abs() * (1 - 1e-12)).all()
