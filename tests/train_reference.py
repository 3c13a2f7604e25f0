"""float64 restatement of one training step of ``dsen2_b200.train.Trainer`` (tests only).

``step_gradients`` is the backward pass of ``Trainer._step_body`` fed with the forward tensors the trainer keeps
(``tr._bufs[(n, P)]``).  It rounds to fp16 exactly where the step rounds and nowhere else:

    dpred = 2^-4 sign(fl32(pred - y)), +0 on ties                      (exact in fp16)
    tail:      dW = inv sum x_hi[L] (x) dpred,  db = inv sum dpred,  dx32 = convT(dpred, f16(W)),  dx_hi = f16(dx32)
    resBlock l = L-1 .. 0:
               conv2  dW = 0.1 inv sum t[l] (x) dx_hi,  db = 0.1 inv sum dx_hi
                      g2 = f16([t[l] > 0] convT(dx_hi, f16(fl32(0.1) W2)))
               conv1  dW = inv sum x_hi[l] (x) g2,  db = inv sum g2
                      dx32 += convT(g2, f16(W1)),  dx_hi = f16(dx32)
    head:      g = [x_hi[0] > 0] dx_hi,  dW = inv sum f16(x) (x) g,  db = inv sum g      (x: the concatenated inputs)
    inv = 1 / (2^-4 * pred.numel())

The ReLU masks come from the trainer's own tensors, and the backward pass is linear once they are fixed, so the
kernels and this restatement differ only in the order of the fp32 accumulation and in rare one-ulp flips of the fp16
gradients dx_hi and g2 (a sum that lands next to a rounding boundary).  ``layer_references`` restates each forward layer
of ``Trainer.forward`` on the trainer's own previous tensors.

Plain torch.nn.functional in float64: the same code runs on CPU tensors and on CUDA tensors (cuDNN / ATen, not this
library).  ``rounding=False`` drops every rounding; the gradients are then those of the exact graph.
"""
import numpy as np
import torch
import torch.nn.functional as F

GSCALE = 2.0 ** -4          # Trainer.GSCALE: the scaled MAE gradient entering the fp16 backward path


def _oihw(k):
    return k.permute(3, 2, 0, 1)


def conv(x, k, b=None):
    """3x3 'same' convolution, NCHW activations, HWIO kernel."""
    return F.conv2d(x, _oihw(k), b, padding=1)


def conv_t(dy, k):
    """Gradient of conv(., k) with respect to its input."""
    return F.conv_transpose2d(dy, _oihw(k), padding=1)


def wgrad(x, dy, shape):
    """HWIO (3, 3, cin, cout) kernel gradient: sum over pixels of x[px + tap] (x) dy[px]."""
    return torch.nn.grad.conv2d_weight(x, (shape[3], shape[2], 3, 3), dy, padding=1).permute(2, 3, 1, 0)


def _rounding(on):
    if not on:
        return (lambda a: a), (lambda a: a)
    return (lambda a: a.to(torch.float16).double()), (lambda a: a.to(torch.float32).double())


def nchw(a, dev):
    """A trainer buffer (NHWC) -> float64 NCHW on `dev`."""
    return torch.as_tensor(a).to(dev).double().permute(0, 3, 1, 2)


def _f64(a, dev):
    return torch.as_tensor(np.asarray(a) if not torch.is_tensor(a) else a).to(dev).double()


def step_gradients(bufs, xs, y, weights, rounding=True, magnitudes=False):
    """bufs: 'x_hi' (L+1 NHWC tensors), 't' (L NHWC tensors), 'pred' (n, cout, P, P); xs: the inputs (n, c_i, P, P);
    y: the labels; weights: Keras order [kernel HWIO, bias, ...].  Returns a dict:
      grads  the gradient tensors in Keras order (float64, on the device of pred),
      mags   with `magnitudes`: for every entry, inv * sum |products| (0.1 inv for conv2) -- the size of the terms the fp32
             accumulation of that entry carries,
      dx_hi  NHWC: the gradient reaching the first layer's output before its ReLU mask, the last dx_hi of the step."""
    dev = torch.as_tensor(bufs['pred']).device
    q16, q32 = _rounding(rounding)
    w = [_f64(a, dev) for a in weights]
    L = len(bufs['t'])
    x_hi = [nchw(a, dev) for a in bufs['x_hi']]
    t = [nchw(a, dev) for a in bufs['t']]
    pred = _f64(bufs['pred'], dev)
    # fl32(pred - y) is zero exactly when pred == y and has the sign of the exact difference otherwise
    dpred = GSCALE * torch.sign(pred - _f64(y, dev))
    inv = 1.0 / (GSCALE * pred.numel())
    grads, mags = [None] * len(w), [None] * len(w)

    def record(layer, x, dy, scale):
        k = w[2 * layer]
        grads[2 * layer] = scale * wgrad(x, dy, k.shape)
        grads[2 * layer + 1] = scale * dy.sum((0, 2, 3))
        if magnitudes:
            mags[2 * layer] = scale * wgrad(x.abs(), dy.abs(), k.shape)
            mags[2 * layer + 1] = scale * dy.abs().sum((0, 2, 3))

    nl = 2 * L + 2
    record(nl - 1, x_hi[L], dpred, inv)
    dx32 = conv_t(dpred, q16(w[-2]))
    dx = q16(dx32)
    s = float(np.float32(0.1)) if rounding else 0.1          # Lambda(x * 0.1) folded into the operand in fp32
    for l in range(L - 1, -1, -1):
        i1, i2 = 1 + 2 * l, 2 + 2 * l
        record(i2, t[l], dx, 0.1 * inv)
        g2 = q16(torch.where(t[l] > 0, conv_t(dx, q16(q32(s * w[2 * i2]))), 0.0))
        record(i1, x_hi[l], g2, inv)
        dx32 = dx32 + conv_t(g2, q16(w[2 * i1]))
        dx = q16(dx32)
    g = torch.where(x_hi[0] > 0, dx, 0.0)
    xin = q16(torch.cat([_f64(a, dev) for a in xs], dim=1))
    record(0, xin, g, inv)
    out = dict(grads=grads, dx_hi=dx.permute(0, 2, 3, 1))
    if magnitudes:
        out['mags'] = mags
    return out


def _split_weight(k, q16):
    """First / last layer operands as dsen2_pack_head*/tail*_weights split them: (W_hi, W_lo), W_lo = f16(W - W_hi)."""
    hi = q16(k)
    return hi, q16(k - hi)


def layer_references(bufs, weights, rounding=True):
    """Each layer of Trainer.forward in float64 on the trainer's OWN previous tensors (NCHW results):
      head, head_mag    relu(conv(xin_hi + xin_lo, W_hi + W_lo) + b) and the sum of |terms| (every hi / lo product);
      t[l], t_mag[l]    relu(conv(x_hi[l], f16 W1) + b1) and its sum of |terms|;
      trunk[l]          the float64 running trunk: trunk[0] = head, trunk[l+1] = trunk[l] + 0.1 (conv(t[l], f16 W2) + b2),
                        on the trainer's t[l]; c2_mag[l] the sum of |terms| of that convolution;
      pred, pred_mag    conv(x_hi[L] + x_lo, W_hi + W_lo) + b + skip, the skip read from xin_hi + xin_lo (bands
                        sum(c) - cout ..), and the sum of |terms| including |skip|.
    bufs also needs 'x_lo', 'xin_hi', 'xin_lo' (the 64-channel prepared input of the 128-feature step, whose centre
    horizontal tap is channels 16..31, or the 16-channel one of the 256-feature step)."""
    dev = torch.as_tensor(bufs['x_hi'][0]).device
    q16, _ = _rounding(rounding)
    w = [_f64(a, dev) for a in weights]
    L = len(bufs['t'])
    ctot, cout = w[0].shape[2], w[-2].shape[3]
    xin_hi, xin_lo = nchw(bufs['xin_hi'], dev), nchw(bufs['xin_lo'], dev)
    c0 = 16 if xin_hi.shape[1] == 64 else 0
    xin_hi, xin_lo = xin_hi[:, c0:c0 + ctot], xin_lo[:, c0:c0 + ctot]
    wh, wl = _split_weight(w[0], q16)
    b0 = w[1]
    r = dict(head=torch.relu(conv(xin_hi + xin_lo, wh + wl, b0)),
             head_mag=conv(xin_hi.abs() + xin_lo.abs(), wh.abs() + wl.abs(), b0.abs()), t=[], t_mag=[], c2_mag=[])
    trunk = [r['head']]
    for l in range(L):
        x = nchw(bufs['x_hi'][l], dev)
        k1, b1 = q16(w[2 + 4 * l]), w[3 + 4 * l]
        r['t'].append(torch.relu(conv(x, k1, b1)))
        r['t_mag'].append(conv(x.abs(), k1.abs(), b1.abs()))
        tl = nchw(bufs['t'][l], dev)
        k2, b2 = q16(w[4 + 4 * l]), w[5 + 4 * l]
        trunk.append(trunk[-1] + 0.1 * conv(tl, k2, b2))
        r['c2_mag'].append(conv(tl.abs(), k2.abs(), b2.abs()))
    r['trunk'] = trunk
    xh, xl = nchw(bufs['x_hi'][L], dev), nchw(bufs['x_lo'], dev)
    wh, wl = _split_weight(w[-2], q16)
    skip = (xin_hi + xin_lo)[:, ctot - cout:ctot]
    r['pred'] = conv(xh + xl, wh + wl, w[-1]) + skip
    r['pred_mag'] = conv(xh.abs() + xl.abs(), wh.abs() + wl.abs(), w[-1].abs()) + skip.abs()
    return r


def exact_buffers(xs, weights):
    """The forward tensors of the exact graph (float64, no rounding) in the trainer's buffer layout: x_hi[l] = trunk,
    t[l], x_lo = 0, xin_hi = the concatenated inputs in the 16-channel layout, xin_lo = 0, pred."""
    w = [_f64(a, 'cpu') for a in weights]
    L = (len(w) - 4) // 4
    x_in = torch.cat([_f64(a, 'cpu') for a in xs], dim=1)
    nhwc = lambda a: a.permute(0, 2, 3, 1).contiguous()
    x = torch.relu(conv(x_in, w[0], w[1]))
    x_hi, ts = [nhwc(x)], []
    for l in range(L):
        tl = torch.relu(conv(x, w[2 + 4 * l], w[3 + 4 * l]))
        x = x + 0.1 * conv(tl, w[4 + 4 * l], w[5 + 4 * l])
        ts.append(nhwc(tl))
        x_hi.append(nhwc(x))
    pred = conv(x, w[-2], w[-1]) + _f64(xs[-1], 'cpu')
    n, c, H, W = x_in.shape
    xin = torch.zeros((n, H, W, 16), dtype=torch.float64)
    xin[..., :c] = nhwc(x_in)
    return dict(x_hi=x_hi, t=ts, x_lo=torch.zeros_like(x_hi[-1]), xin_hi=xin, xin_lo=torch.zeros_like(xin), pred=pred)
