"""Host-side mirror of the reference ``utils/DSen2Net.py``: ``s2model(input_shape, num_layers, feature_size)``.

The reference builds a Keras graph (DSen2Net.py:18-43):
    concat(inputs) -> Conv3x3+ReLU -> num_layers x [Conv3x3, ReLU, Conv3x3, x0.1, +skip] -> Conv3x3 -> + last input
Here ``s2model`` returns an ``S2Model`` exposing the Keras ``Model`` methods the reference's callers use
(``load_weights``, ``predict``, ``count_params``; supres.py:63,65, supres_train.py:146,161,169) whose
forward pass is the tcgen05 implicit-GEMM path behind ``dsen2_s2model_forward`` (include/dsen2_b200.h).
"""
import ctypes
import math
import os

import numpy as np

from . import _capi
from .hdf5 import File, write_hdf5


def resBlock(*_a, **_k):  # pragma: no cover - graph-construction helper of the reference, no standalone equivalent
    raise NotImplementedError("resBlock is fused into the conv epilogues; build the network with s2model()")


class S2Model:
    def __init__(self, input_shape, num_layers=32, feature_size=256, seed=None):
        if len(input_shape) not in (2, 3):
            raise ValueError("s2model takes 2 or 3 inputs (10 m, 20 m[, 60 m])")
        if feature_size not in (128, 256):
            raise ValueError("feature_size must be 128 (DSen2) or 256 (VDSen2); got %r" % (feature_size,))
        if int(num_layers) > 0 and int(input_shape[-1][0]) > 7:
            raise ValueError("at most 7 output bands (the last input's channel count); got %d" % int(input_shape[-1][0]))
        self.input_shape = tuple(tuple(s) for s in input_shape)
        self.in_channels = [int(s[0]) for s in self.input_shape]
        self.out_channels = self.in_channels[-1]                 # DSen2Net.py:35
        self.num_layers, self.feature_size = int(num_layers), int(feature_size)
        ctot, F = sum(self.in_channels), self.feature_size
        self.layer_shapes = [(ctot, F)] + [(F, F)] * (2 * self.num_layers) + [(F, self.out_channels)]
        rng = np.random.RandomState(seed)
        self._weights = []
        for cin, cout in self.layer_shapes:                      # he_uniform kernels, zero bias (:10,12,29,35)
            lim = math.sqrt(6.0 / (9 * cin))
            self._weights.append((rng.uniform(-lim, lim, size=(3, 3, cin, cout)).astype(np.float32),
                                  np.zeros((cout,), np.float32)))
        self._packed = {}        # device index -> (weights tensors, bias tensors, pointer arrays)
        self._workspace = {}
        self._trainer = None     # set by compile(); owns the fp32 master weights while training
        self._weights_stale = False   # the trainer's weights are newer than self._weights

    # ---- Keras-like weight access -------------------------------------------------------- #
    def count_params(self):
        return int(sum(k.size + b.size for k, b in self._weights))

    def get_weights(self):
        self._pull_trained_weights()
        return [a for kb in self._weights for a in kb]

    def _pull_trained_weights(self):
        """After ``train_on_batch`` the current weights live in the trainer; Keras' predict / get_weights / save_weights see
        them, so pull them back before any of those."""
        if self._weights_stale and self._trainer is not None:
            self._weights_stale = False
            self._set_weights_local(self._trainer.get_weights())

    def set_weights(self, arrays):
        self._set_weights_local(arrays)
        self._weights_stale = False
        if self._trainer is not None:            # compile() then load_weights() (supres_train.py:143,183): train from them
            self._trainer.set_weights(self.get_weights())

    def _set_weights_local(self, arrays):
        arrays = list(arrays)
        if len(arrays) != 2 * len(self.layer_shapes):
            raise ValueError("expected %d arrays (kernel, bias per conv layer), got %d"
                             % (2 * len(self.layer_shapes), len(arrays)))
        new = []
        for i, (cin, cout) in enumerate(self.layer_shapes):
            k = np.ascontiguousarray(arrays[2 * i], dtype=np.float32)
            b = np.ascontiguousarray(arrays[2 * i + 1], dtype=np.float32)
            if k.shape != (3, 3, cin, cout) or b.shape != (cout,):
                raise ValueError("layer %d: expected kernel %s / bias %s, got %s / %s"
                                 % (i, (3, 3, cin, cout), (cout,), k.shape, b.shape))
            new.append((k, b))
        self._weights = new
        self._packed.clear()

    def load_weights(self, filepath):
        """Keras 2.x HDF5 weights or full-model file (``model.load_weights``, supres.py:63).

        Layers are matched in ``layer_names`` order, restricted to layers that own weights (Keras'
        topological load); auto-generated layer names differ between sessions and are ignored.
        """
        f = File(filepath)                                   # OSError if missing / not HDF5, like h5py
        g = f
        if 'layer_names' not in f.attrs and 'model_weights' in f.keys():
            g = f['model_weights']                               # full-model save (supres_train.py:195-201)
        if 'layer_names' not in g.attrs:
            raise ValueError("%s is not a Keras weight file (no layer_names attribute)" % filepath)
        arrays = []
        for lname in np.atleast_1d(g.attrs['layer_names']):
            lname = lname.decode('utf8') if isinstance(lname, bytes) else str(lname)
            lg = g[lname]
            wnames = np.atleast_1d(lg.attrs['weight_names']) if 'weight_names' in lg.attrs else []
            for wn in wnames:
                wn = wn.decode('utf8') if isinstance(wn, bytes) else str(wn)
                arrays.append(np.asarray(lg[wn][()]))
        if len(arrays) != 2 * len(self.layer_shapes):
            raise ValueError("You are trying to load a weight file containing %d weight arrays into a model with %d"
                             % (len(arrays), 2 * len(self.layer_shapes)))
        self.set_weights(arrays)

    def _weights_tree(self, prefix=''):
        """(tree, attrs) of the Keras-2 weight layout: one group per layer, layer_names / weight_names attributes."""
        self._pull_trained_weights()
        tree, attrs, names = {}, {}, []
        for i, (k, b) in enumerate(self._weights):
            n = 'conv2d_%d' % (i + 1)
            names.append(n.encode())
            tree[n] = {n: {'kernel:0': k, 'bias:0': b}}
            attrs[prefix + '/' + n] = {'weight_names': np.array([('%s/kernel:0' % n).encode(), ('%s/bias:0' % n).encode()])}
        attrs[prefix or '/'] = {'layer_names': np.array(names), 'backend': np.bytes_(b'dsen2_b200'),
                                'keras_version': np.bytes_(b'2.2.4')}
        return tree, attrs

    def save_weights(self, filepath):
        """Write a Keras-2-style weight file (layer_names / weight_names attributes, kernel:0 / bias:0)."""
        tree, attrs = self._weights_tree()
        write_hdf5(filepath, tree, attrs)

    def save(self, filepath):
        """``model.save(filepath)`` -- what ``ModelCheckpoint(save_weights_only=False)`` writes (supres_train.py:195-201):
        the Keras-2 full-model layout, ``/model_weights`` (as ``save_weights``), ``/optimizer_weights`` (Nadam: iterations,
        first moments, second moments -- Keras' ``optimizer.weights`` order) and the ``model_config`` / ``training_config``
        attributes.  ``load_weights`` reads the file back; ``load_optimizer_weights`` restores the optimizer."""
        import json
        wtree, attrs = self._weights_tree('/model_weights')
        tree = {'model_weights': wtree}
        root = {'keras_version': np.bytes_(b'2.2.4'), 'backend': np.bytes_(b'dsen2_b200'),
                'model_config': np.bytes_(json.dumps({'class_name': 'Model', 'config': {
                    'name': 's2model', 'input_shape': [[c, None, None] for c in self.in_channels],
                    'num_layers': self.num_layers, 'feature_size': self.feature_size}}).encode())}
        tr = self._trainer
        if tr is not None:
            o = tr.opt
            root['training_config'] = np.bytes_(json.dumps({
                'optimizer_config': {'class_name': 'Nadam', 'config': {'lr': o.lr, 'beta_1': o.beta_1, 'beta_2': o.beta_2,
                                                                       'epsilon': o.epsilon, 'schedule_decay': o.schedule_decay}},
                'loss': 'mean_absolute_error', 'metrics': ['mean_squared_error']}).encode())
            m, v = tr.m.cpu().numpy(), tr.v.cpu().numpy()
            opt, names = {'Nadam': {'iterations:0': np.array(tr.iterations, np.int64)}}, [b'Nadam/iterations:0']
            grp = {}
            for kind, flat in (('m', m), ('v', v)):
                for i in range(2 * len(self.layer_shapes)):
                    name = '%s_%d:0' % (kind, i)
                    grp[name] = flat[int(tr.offsets[i]):int(tr.offsets[i + 1])].copy()
                    names.append(('training/Nadam/' + name).encode())
            opt['training'] = {'Nadam': grp}
            tree['optimizer_weights'] = opt
            # Keras does not store Nadam's running product of the momentum schedule; kept here so that a resume is exact
            attrs['/optimizer_weights'] = {'weight_names': np.array(names), 'm_schedule': np.array(tr.m_schedule, np.float64)}
        attrs['/'] = root
        write_hdf5(filepath, tree, attrs)

    def load_optimizer_weights(self, filepath):
        """Restore the Nadam state a ``save()`` file carries (after ``compile``); returns False if the file has none."""
        if self._trainer is None:
            raise RuntimeError("You must compile a model before restoring its optimizer state.")
        f = File(filepath)
        if 'optimizer_weights' not in f.keys():
            return False
        g = f['optimizer_weights']
        tr, torch = self._trainer, _capi.require_cuda()
        flat = {}
        for kind in ('m', 'v'):
            parts = [np.asarray(g['training/Nadam/%s_%d:0' % (kind, i)][()], np.float32).ravel()
                     for i in range(2 * len(self.layer_shapes))]
            flat[kind] = np.concatenate(parts)
        tr.m.copy_(torch.from_numpy(flat['m']).to(tr.dev))
        tr.v.copy_(torch.from_numpy(flat['v']).to(tr.dev))
        tr.iterations = int(np.asarray(g['Nadam/iterations:0'][()]).reshape(-1)[0])
        ms = g.attrs['m_schedule'] if 'm_schedule' in g.attrs else None
        if ms is None:                       # a file written by Keras: rebuild the product from the schedule
            from .train import nadam_schedule
            prod = 1.0
            for t in range(1, tr.iterations + 1):
                prod = nadam_schedule(t, prod, tr.opt)['sched_new']
            ms = prod
        tr.m_schedule = float(np.asarray(ms).reshape(-1)[0])
        return True

    # ---- device side ------------------------------------------------------------------- #
    @property
    def xin16(self):
        """Networks with resblocks (DSen2, VDSen2) prepare the input un-gathered (16 channels, ``dsen2_prep16_*``), run
        the first layer with nine taps (``dsen2_conv_head16_q``) and keep the residual trunk as fp16 + 8 bits (include/
        dsen2_b200.h).  A network WITHOUT resblocks (128 features only) keeps the 64-channel form with the three
        horizontal taps pre-gathered, whose first layer hands the last one an fp16 hi + lo pair."""
        return self.num_layers > 0

    def _ensure_packed(self, device):
        torch = _capi.require_cuda()
        self._pull_trained_weights()
        key = device.index if device.index is not None else torch.cuda.current_device()
        if key in self._packed:
            return self._packed[key]
        lib = _capi.lib()
        F = self.feature_size
        wts, biases = [], []
        with torch.cuda.device(device):
            st = _capi.stream_ptr()
            for i, (k, b) in enumerate(self._weights):
                cin, cout = self.layer_shapes[i]
                head, tail = i == 0, i == len(self._weights) - 1
                src = torch.from_numpy(k).to(device)
                if head and self.xin16:
                    dst = torch.empty((9, 2 * F, 16), dtype=torch.float16, device=device)
                    _capi.check(lib.dsen2_pack_head16_weights(_capi.ptr(src), cin, F, _capi.ptr(dst), st),
                                "dsen2_pack_head16_weights")
                    cout_pad = F
                elif head:
                    dst = torch.empty((3, 2 * F, 64), dtype=torch.float16, device=device)
                    _capi.check(lib.dsen2_pack_head_weights(_capi.ptr(src), cin, F, _capi.ptr(dst), st),
                                "dsen2_pack_head_weights")
                    cout_pad = F
                elif tail and self.xin16:
                    dst = torch.empty((128, F), dtype=torch.float16, device=device)
                    _capi.check(lib.dsen2_pack_tail16_weights(_capi.ptr(src), F, cout, _capi.ptr(dst), st),
                                "dsen2_pack_tail16_weights")
                    cout_pad = 16
                elif tail:
                    dst = torch.empty((9, 32, F), dtype=torch.float16, device=device)
                    _capi.check(lib.dsen2_pack_tail_weights(_capi.ptr(src), F, cout, _capi.ptr(dst), st),
                                "dsen2_pack_tail_weights")
                    cout_pad = 16
                else:
                    cout_pad = F
                    dst = torch.empty((9, F, F), dtype=torch.float16, device=device)
                    _capi.check(lib.dsen2_pack_conv_weights(_capi.ptr(src), cin, cout, F, F, _capi.ptr(dst), st),
                                "dsen2_pack_conv_weights")
                bp = torch.zeros((max(cout_pad, 16),), dtype=torch.float32, device=device)
                bp[:cout] = torch.from_numpy(b).to(device)
                wts.append(dst)
                biases.append(bp)
            torch.cuda.current_stream().synchronize()
        nl = len(wts)
        wp = (ctypes.c_void_p * nl)(*[t.data_ptr() for t in wts])
        bp_ = (ctypes.c_void_p * nl)(*[t.data_ptr() for t in biases])
        self._packed[key] = (wts, biases, wp, bp_)
        return self._packed[key]

    def workspace_bytes(self, n, P):
        return int(_capi.lib().dsen2_s2model_workspace_bytes(n, P, sum(self.in_channels), self.feature_size))

    def _buffers(self, dev, n, P, reuse_larger=False):
        """Activation buffers for n patches of P x P.  ``reuse_larger``: views of the smallest cached set that holds n
        patches, if there is one -- batches of active patches have arbitrary sizes, and a set per size would pile up."""
        torch = _capi.require_cuda()
        key = (dev.index, torch.cuda.current_stream().cuda_stream, n, P)
        if reuse_larger and key not in self._workspace:
            fits = [k for k in self._workspace if k[:2] == key[:2] and k[3] == P and k[2] >= n]
            if fits:
                return {name: t[:n] for name, t in self._workspace[min(fits, key=lambda k: k[2])].items()}
        buf = self._workspace.get(key)
        if buf is None:
            if len(self._workspace) > 8:
                self._workspace.clear()
            F = self.feature_size
            mk = lambda c: torch.empty((n, P, P, c), dtype=torch.float16, device=dev)
            cx = 16 if self.xin16 else 64                                    # prepared input: un-gathered / 3 taps gathered
            buf = dict(xin_hi=mk(cx), xin_lo=mk(cx), x_hi=mk(F), x_lo=mk(F), t=mk(F))
            if self.xin16:                                                   # low bytes of the fp16 + 8 bit trunk
                buf['xq'] = torch.empty((n, P, (P + 7) // 8, F // 16, 8, 16), dtype=torch.uint8, device=dev)
            self._workspace[key] = buf
        return buf

    @staticmethod
    def _timed(timers, kind, n, fn):
        if timers is None:
            return fn()
        import torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        timers.setdefault(kind, []).append((e0, e1, n))

    def _trunk(self, buf, wts, biases, n, P, st, timers):
        """First layer + resblocks on the buffers; shared by the patch-stack and the image form of the input."""
        lib, ptr, F, L = _capi.lib(), _capi.ptr, self.feature_size, self.num_layers
        x_hi, x_lo, t = buf['x_hi'], buf['x_lo'], buf['t']
        if L == 0:
            # no resblocks: the 64-channel first layer writes the fp16 hi + lo pair the last layer reads
            self._timed(timers, 'conv_head', n, lambda: _capi.check(lib.dsen2_conv_head(
                ptr(buf['xin_hi']), ptr(buf['xin_lo']), ptr(wts[0]), ptr(biases[0]), n, P, P, F, ptr(x_hi), ptr(x_lo), None,
                st), "dsen2_conv_head"))
            return
        # fp16 + 8 bit trunk: x_hi (NHWC, what the next convolution reads) updated in place + one byte per element
        # (include/dsen2_b200.h, dsen2_conv_resq); the last block hands the last layer x_hi, x_lo
        xq = buf['xq']
        resq = lib.dsen2_conv_resq256 if F == 256 else lib.dsen2_conv_resq
        self._timed(timers, 'conv_head', n, lambda: _capi.check(lib.dsen2_conv_head16_q(
            ptr(buf['xin_hi']), ptr(buf['xin_lo']), ptr(wts[0]), ptr(biases[0]), n, P, P, F, ptr(x_hi), ptr(xq), st),
            "dsen2_conv_head16_q"))
        for l in range(L):
            self._timed(timers, 'conv_res1', n, lambda: _capi.check(lib.dsen2_conv_relu(
                ptr(x_hi), ptr(wts[1 + 2 * l]), ptr(biases[1 + 2 * l]), n, P, P, F, ptr(t), st), "dsen2_conv_relu"))
            self._timed(timers, 'conv_res2', n, lambda: _capi.check(resq(
                ptr(t), ptr(wts[2 + 2 * l]), ptr(biases[2 + 2 * l]), n, P, P, 0.1, ptr(x_hi), ptr(xq),
                ptr(x_lo) if l == L - 1 else None, st), "dsen2_conv_resq"))

    def _tail_args(self, buf, wts, biases):
        ptr = _capi.ptr
        return (ptr(buf['x_hi']), ptr(buf['x_lo']), ptr(wts[-1]), ptr(biases[-1]), ptr(buf['xin_hi']), ptr(buf['xin_lo']),
                sum(self.in_channels) - self.out_channels, self.out_channels)

    def forward_device(self, xs, out=None, timers=None):
        """xs: list of CUDA float32 (n, C_i, P, P) contiguous tensors -> CUDA float32 (n, Cout, P, P).

        One launch per layer on the current stream (input preparation + 2*num_layers+2 tcgen05
        convolutions).  ``timers`` (optional dict) collects CUDA-event pairs per kernel kind for bench.py.
        The same sequence is available to C callers as ``dsen2_s2model_forward``."""
        torch = _capi.require_cuda()
        if len(xs) != len(self.in_channels):
            raise ValueError("model expects %d inputs, got %d" % (len(self.in_channels), len(xs)))
        n, _, P, P2 = xs[0].shape
        for x, c in zip(xs, self.in_channels):
            if not (x.is_cuda and x.dtype == torch.float32 and x.is_contiguous()):
                raise ValueError("inputs must be contiguous CUDA float32 tensors")
            if tuple(x.shape) != (n, c, P, P) or P != P2:
                raise ValueError("expected input of shape %s, got %s" % ((n, c, P, P), tuple(x.shape)))
        dev = xs[0].device
        wts, biases, _wp, _bp = self._ensure_packed(dev)
        if out is None:
            out = torch.empty((n, self.out_channels, P, P), dtype=torch.float32, device=dev)
        if n == 0:
            return out
        lib, ptr = _capi.lib(), _capi.ptr
        buf = self._buffers(dev, n, P)
        with torch.cuda.device(dev):
            st = _capi.stream_ptr()
            x2, c2 = (xs[2], self.in_channels[2]) if len(xs) == 3 else (None, 0)
            prep = lib.dsen2_prep16_from_patches if self.xin16 else lib.dsen2_prep_from_patches
            self._timed(timers, 'prep', n, lambda: _capi.check(prep(
                ptr(xs[0]), self.in_channels[0], ptr(xs[1]), self.in_channels[1], ptr(x2), c2, n, P,
                ptr(buf['xin_hi']), ptr(buf['xin_lo']), st), "dsen2_prep_from_patches"))
            self._trunk(buf, wts, biases, n, P, st, timers)
            if self.xin16:
                self._timed(timers, 'conv_tail', n, lambda: _capi.check(lib.dsen2_conv_tail16(
                    *self._tail_args(buf, wts, biases), self.feature_size, n, P, P, ptr(out), st), "dsen2_conv_tail16"))
            else:
                self._timed(timers, 'conv_tail', n, lambda: _capi.check(lib.dsen2_conv_tail(
                    *self._tail_args(buf, wts, biases), n, P, P, ptr(out), st), "dsen2_conv_tail"))
        return out

    def forward_c(self, xs, out=None):
        """Same as ``forward_device`` through the single C entry point ``dsen2_s2model_forward`` (what a C caller of
        ``include/dsen2_b200.h`` uses): one call, workspace supplied by the caller."""
        torch = _capi.require_cuda()
        n, _, P, _ = xs[0].shape
        dev = xs[0].device
        _wts, _biases, wp, bp = self._ensure_packed(dev)
        if out is None:
            out = torch.empty((n, self.out_channels, P, P), dtype=torch.float32, device=dev)
        nbytes = self.workspace_bytes(n, P)
        ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
        xp = (ctypes.c_void_p * len(xs))(*[x.data_ptr() for x in xs])
        ch = (ctypes.c_int * len(xs))(*self.in_channels)
        with torch.cuda.device(dev):
            _capi.check(_capi.lib().dsen2_s2model_forward(xp, ch, len(xs), n, P, self.num_layers, self.feature_size, wp, bp,
                                                          _capi.ptr(ws), nbytes, _capi.ptr(out), _capi.stream_ptr()),
                        "dsen2_s2model_forward")
        return out

    def forward_images(self, d10, d20, d60, patch, border, first_patch, n, canvas, mul, timers=None, patch_ids=None,
                       avoid=None, add_offset=None):
        """Fused tile pipeline of the fast path: patches [first_patch, first_patch+n) are gathered straight
        from the HWC images (extract + bilinear + /mul), run through the network, and the pixels they own
        are written x mul into ``canvas`` (H, W, Cout).  No patch stack or prediction stack exists.  The images are
        float32 or uint16 (digital numbers) HWC CUDA tensors.  ``patch_ids``: a CUDA int32 tensor of n patch indices to
        run instead of the range (``first_patch`` is then ignored).  ``canvas`` is a contiguous float32 or uint16 tensor;
        a uint16 canvas receives the float values rounded half to even and clipped to [0, 65535] (NaN: 0), and a value
        equal to ``avoid`` (an int in [0, 65535], the nodata value) is written one step away from it
        (``dsen2_conv_tail16_stitch_u16`` in include/dsen2_b200.h).  ``add_offset``: a finite float (None: none) added to
        every band value before the preparation and subtracted from every output value before it is stored
        (``dsen2_prep16_from_images_offset``, ``dsen2_conv_tail16_stitch_offset``).

        Chip stacks: 4-D images (N, H, W, C) of N same-size chips and an (N, H, W, Cout) canvas.  [first_patch,
        first_patch+n) is then a range of the flat list chip * ppc + patch (ppc = the filled patches of one chip), which
        may straddle chips; each chip is prepared and stitched as the 3-D call on that chip does it
        (``dsen2_prep16_from_chips``, ``dsen2_conv_tail16_stitch_chips``).  No ``patch_ids`` with stacks."""
        torch = _capi.require_cuda()
        if not self.xin16:
            raise _capi.DSen2Error("forward_images needs a network with resblocks (num_layers > 0)")
        dev = d10.device
        chips = d10.dim() == 4
        lead = (int(d10.shape[0]),) if chips else ()
        H, W = int(d10.shape[len(lead)]), int(d10.shape[len(lead) + 1])
        imgs = [t for t in (d10, d20, d60) if t is not None]
        if any(t.dtype != d10.dtype for t in imgs) or d10.dtype not in (torch.float32, torch.uint16):
            raise ValueError("images must all be float32 or all be uint16")
        if chips:
            for t, div, c in zip(imgs, (1, 2, 6), self.in_channels):
                if not (t.is_cuda and t.is_contiguous() and tuple(t.shape) == lead + (H // div, W // div, c)):
                    raise ValueError("chip stack images must be contiguous CUDA tensors of shape %s, got %s"
                                     % (lead + (H // div, W // div, c), tuple(t.shape)))
            if patch_ids is not None:
                raise ValueError("patch_ids are not supported with chip stacks")
        if patch_ids is not None and not (patch_ids.is_cuda and patch_ids.dtype == torch.int32 and patch_ids.is_contiguous()
                                          and tuple(patch_ids.shape) == (n,)):
            raise ValueError("patch_ids must be a contiguous CUDA int32 tensor of %d ids" % n)
        if not (canvas.is_cuda and canvas.dtype in (torch.float32, torch.uint16) and canvas.is_contiguous()
                and tuple(canvas.shape) == lead + (H, W, self.out_channels)):
            raise ValueError("canvas must be a contiguous CUDA float32 or uint16 tensor of shape %s"
                             % (lead + (H, W, self.out_channels),))
        u16 = canvas.dtype == torch.uint16
        if avoid is not None and not u16:
            raise ValueError("avoid applies to a uint16 canvas only")
        avoid = -1 if avoid is None else int(avoid)
        if not -1 <= avoid <= 65535:
            raise ValueError("avoid %d is not a uint16 value" % avoid)
        img_dtype = _capi.IMG_U16 if d10.dtype == torch.uint16 else _capi.IMG_F32
        wts, biases, _wp, _bp = self._ensure_packed(dev)
        if n == 0:
            return canvas
        lib, ptr = _capi.lib(), _capi.ptr
        buf = self._buffers(dev, n, patch, reuse_larger=patch_ids is not None)
        with torch.cuda.device(dev):
            st = _capi.stream_ptr()
            if chips:
                add, a = (0, 0.0) if add_offset is None else (1, float(add_offset))
                self._timed(timers, 'prep', n, lambda: _capi.check(lib.dsen2_prep16_from_chips(
                    ptr(d10), ptr(d20), ptr(d60), img_dtype, lead[0], H, W, patch, border, first_patch, n, float(mul), add,
                    a, ptr(buf['xin_hi']), ptr(buf['xin_lo']), st), "dsen2_prep16_from_chips"))
                self._trunk(buf, wts, biases, n, patch, st, timers)
                self._timed(timers, 'conv_tail', n, lambda: _capi.check(lib.dsen2_conv_tail16_stitch_chips(
                    *self._tail_args(buf, wts, biases), self.feature_size, n, patch, first_patch, border, lead[0], H, W,
                    float(mul), add, a, _capi.IMG_U16 if u16 else _capi.IMG_F32, avoid, ptr(canvas), st),
                    "dsen2_conv_tail16_stitch_chips"))
                return canvas
            if add_offset is not None:
                self._timed(timers, 'prep', n, lambda: _capi.check(lib.dsen2_prep16_from_images_offset(
                    ptr(d10), ptr(d20), ptr(d60), img_dtype, H, W, patch, border, first_patch, ptr(patch_ids), n,
                    float(mul), float(add_offset), ptr(buf['xin_hi']), ptr(buf['xin_lo']), st),
                    "dsen2_prep16_from_images_offset"))
            elif patch_ids is None:
                self._timed(timers, 'prep', n, lambda: _capi.check(lib.dsen2_prep16_from_images(
                    ptr(d10), ptr(d20), ptr(d60), img_dtype, H, W, patch, border, first_patch, n, float(mul),
                    ptr(buf['xin_hi']), ptr(buf['xin_lo']), st), "dsen2_prep16_from_images"))
            else:
                self._timed(timers, 'prep', n, lambda: _capi.check(lib.dsen2_prep16_from_images_ids(
                    ptr(d10), ptr(d20), ptr(d60), img_dtype, H, W, patch, border, ptr(patch_ids), n, float(mul),
                    ptr(buf['xin_hi']), ptr(buf['xin_lo']), st), "dsen2_prep16_from_images_ids"))
            self._trunk(buf, wts, biases, n, patch, st, timers)
            if add_offset is not None:
                self._timed(timers, 'conv_tail', n, lambda: _capi.check(lib.dsen2_conv_tail16_stitch_offset(
                    *self._tail_args(buf, wts, biases), self.feature_size, n, patch, first_patch, ptr(patch_ids), border,
                    H, W, float(mul), float(add_offset), _capi.IMG_U16 if u16 else _capi.IMG_F32, avoid, ptr(canvas), st),
                    "dsen2_conv_tail16_stitch_offset"))
                return canvas
            # the canvas type picks the entry point; the uint16 ones take the value to avoid after the scale
            which = (ptr(patch_ids),) if patch_ids is not None else (first_patch,)
            name = 'dsen2_conv_tail16_stitch' + ('_ids' if patch_ids is not None else '') + ('_u16' if u16 else '')
            tail = getattr(lib, name)
            extra = (float(mul), avoid) if u16 else (float(mul),)
            self._timed(timers, 'conv_tail', n, lambda: _capi.check(tail(
                *self._tail_args(buf, wts, biases), self.feature_size, n, patch, *which, border, H, W, *extra,
                ptr(canvas), st), name))
        return canvas

    def forward_scenes(self, table, patch_scene, num_scenes, total, run_60, img_dtype, u16, patch, border, first_patch, n,
                       mul, timers=None, add_offset=None):
        """Fused tile pipeline over a scene list (scenes of any sizes): patches [first_patch, first_patch+n) of the flat
        list first_i + p are prepared, run through the network and stitched into their scenes' canvases.  ``table``: the
        device copy of a ``dsen2_scene_table`` (uint8 CUDA tensor), ``patch_scene`` its patch -> scene map (int32 CUDA
        tensor of ``total`` entries), ``num_scenes`` / ``total`` / ``run_60`` as the table was built.  ``img_dtype``:
        ``_capi.IMG_F32`` / ``IMG_U16`` of every scene's images; ``u16``: the canvases are uint16.  ``add_offset`` as for
        ``forward_images`` (``dsen2_prep16_from_scenes``, ``dsen2_conv_tail16_stitch_scenes``)."""
        torch = _capi.require_cuda()
        if not self.xin16:
            raise _capi.DSen2Error("forward_scenes needs a network with resblocks (num_layers > 0)")
        if not (patch_scene.is_cuda and patch_scene.dtype == torch.int32 and patch_scene.is_contiguous()
                and patch_scene.numel() >= total and table.is_cuda):
            raise ValueError("table and patch_scene must be CUDA tensors (patch_scene: contiguous int32, %d entries)" % total)
        dev = table.device
        wts, biases, _wp, _bp = self._ensure_packed(dev)
        if n == 0:
            return
        lib, ptr = _capi.lib(), _capi.ptr
        buf = self._buffers(dev, n, patch, reuse_larger=True)      # chunks of a scene list have any patch count
        add, a = (0, 0.0) if add_offset is None else (1, float(add_offset))
        with torch.cuda.device(dev):
            st = _capi.stream_ptr()
            self._timed(timers, 'prep', n, lambda: _capi.check(lib.dsen2_prep16_from_scenes(
                ptr(table), ptr(patch_scene), num_scenes, total, img_dtype, int(run_60), patch, border, first_patch, n,
                float(mul), add, a, ptr(buf['xin_hi']), ptr(buf['xin_lo']), st), "dsen2_prep16_from_scenes"))
            self._trunk(buf, wts, biases, n, patch, st, timers)
            self._timed(timers, 'conv_tail', n, lambda: _capi.check(lib.dsen2_conv_tail16_stitch_scenes(
                *self._tail_args(buf, wts, biases), self.feature_size, n, patch, first_patch, border, ptr(table),
                ptr(patch_scene), num_scenes, total, float(mul), add, a, _capi.IMG_U16 if u16 else _capi.IMG_F32, -1, st),
                "dsen2_conv_tail16_stitch_scenes"))

    def launches_per_forward(self):
        return 2 * self.num_layers + 3             # input preparation + first layer + 2 per resblock + last layer

    def predict(self, x, batch_size=32, verbose=0, device_batch=None):
        """``model.predict([x10, x20(, x60)])`` -> (N, Cout, P, P) float32 numpy (supres.py:65).

        Patches are independent, so the result does not depend on ``batch_size``; the device batch is
        chosen for occupancy (``device_batch``, default 64 patches of 128x128).
        """
        torch = _capi.require_cuda()
        xs = [np.ascontiguousarray(a, dtype=np.float32) for a in (x if isinstance(x, (list, tuple)) else [x])]
        N, P = xs[0].shape[0], xs[0].shape[2]
        if device_batch is None:
            device_batch = max(1, (64 * 128 * 128) // (P * P))
        out = np.empty((N, self.out_channels, P, P), np.float32)
        for i in range(0, N, device_batch):
            dx = [torch.from_numpy(a[i:i + device_batch]).cuda() for a in xs]
            out[i:i + device_batch] = self.forward_device(dx).cpu().numpy()
            if verbose:
                print("%d/%d" % (min(i + device_batch, N), N))
        return out

    # ---- training (supres_train.py:137-144, 218-230) ------------------------------------------------------ #
    def compile(self, optimizer=None, loss='mean_absolute_error', metrics=None):
        """``model.compile(optimizer=Nadam(...), loss='mean_absolute_error', metrics=['mean_squared_error'])``."""
        from .train import Nadam, Trainer
        if loss != 'mean_absolute_error':
            raise ValueError("only loss='mean_absolute_error' (the reference's) is implemented")
        if optimizer is None or optimizer == 'nadam':
            optimizer = Nadam()
        self._trainer = Trainer(self, optimizer)
        self.metrics_names = ['loss', 'mean_squared_error']
        return self._trainer

    def train_on_batch(self, x, y):
        """One optimisation step on numpy (or CUDA tensor) inputs; returns [loss, mean_squared_error] like Keras."""
        torch = _capi.require_cuda()
        if self._trainer is None:
            raise RuntimeError("You must compile a model before training/testing. Use `model.compile(optimizer, loss)`.")
        tr = self._trainer
        to_dev = lambda a: a if torch.is_tensor(a) else torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(tr.dev)
        loss, mse = tr.train_step([to_dev(a) for a in (x if isinstance(x, (list, tuple)) else [x])], to_dev(y))
        self._weights_stale = True
        return [float(loss), float(mse)]

    @property
    def optimizer(self):
        """``model.optimizer.lr`` as the reference's callbacks read / set it (supres_train.py:47)."""
        if self._trainer is None:
            raise RuntimeError("You must compile a model before training/testing. Use `model.compile(optimizer, loss)`.")
        return self._trainer.opt

    def evaluate(self, x, y, batch_size=128, verbose=0):
        """``model.evaluate`` -> [loss, mean_squared_error] (sample-weighted mean over the batches)."""
        torch = _capi.require_cuda()
        tr = self.optimizer and self._trainer
        xs = [np.asarray(a) for a in (x if isinstance(x, (list, tuple)) else [x])]
        y = np.asarray(y)
        n = y.shape[0]
        to_dev = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(tr.dev)
        tot = np.zeros(2)
        for i in range(0, n, batch_size):
            l, q = tr.evaluate([to_dev(a[i:i + batch_size]) for a in xs], to_dev(y[i:i + batch_size]))
            m = min(batch_size, n - i)
            tot += np.array([float(l), float(q)]) * m
        return list(tot / n)

    def fit(self, x, y, batch_size=128, epochs=1, verbose=0, callbacks=None, validation_data=None, shuffle=True,
            initial_epoch=0, seed=None, **_ignored):
        """``model.fit`` as supres_train.py:218-230 calls it: shuffled mini-batches, optional ``validation_data`` and
        ``callbacks`` (dsen2_b200.callbacks).  Returns the history dict {'loss', 'mean_squared_error'[, 'val_*']}."""
        xs = [np.asarray(a) for a in (x if isinstance(x, (list, tuple)) else [x])]
        y = np.asarray(y)
        n = y.shape[0]
        rng = np.random.RandomState(seed)
        hist = {'loss': [], 'mean_squared_error': []}
        callbacks = list(callbacks or [])
        for cb in callbacks:
            cb.set_model(self)
            cb.on_train_begin()
        for ep in range(initial_epoch, epochs):
            order = rng.permutation(n) if shuffle else np.arange(n)
            tot, tot_mse, cnt = 0.0, 0.0, 0
            for i in range(0, n, batch_size):
                idx = np.sort(order[i:i + batch_size])
                l, q = self.train_on_batch([a[idx] for a in xs], y[idx])
                tot, tot_mse, cnt = tot + l * len(idx), tot_mse + q * len(idx), cnt + len(idx)
            logs = {'loss': tot / cnt, 'mean_squared_error': tot_mse / cnt}
            if validation_data is not None:
                vl, vq = self.evaluate(validation_data[0], validation_data[1], batch_size=batch_size)
                logs.update(val_loss=vl, val_mean_squared_error=vq)
            for k, v in logs.items():
                hist.setdefault(k, []).append(v)
            if verbose:
                print("Epoch %d/%d - " % (ep + 1, epochs) + " - ".join("%s: %.6f" % kv for kv in logs.items()))
            if callbacks:
                self.sync_weights_from_trainer()          # checkpoints see the current weights
                for cb in callbacks:
                    cb.on_epoch_end(ep, logs)
        self.sync_weights_from_trainer()
        return hist

    def sync_weights_from_trainer(self):
        """Pull the trained fp32 master weights back into the model (predict / get_weights / save_weights do it lazily)."""
        self._pull_trained_weights()

    def to_yaml(self):
        """``model.to_yaml()`` (supres_train.py:191-193 writes it next to the checkpoints): the architecture as YAML -- the
        arguments ``s2model`` was built with and the layer list of DSen2Net.py:18-43, enough to rebuild the network."""
        lines = ['backend: dsen2_b200', 'class_name: Model', 'config:', '  name: s2model',
                 '  input_shape: [%s]' % ', '.join('[%d, null, null]' % c for c in self.in_channels),
                 '  num_layers: %d' % self.num_layers, '  feature_size: %d' % self.feature_size,
                 '  data_format: channels_first', '  layers:']
        F = self.feature_size
        add = lambda name, **kw: lines.append('  - {name: %s, %s}' % (name, ', '.join('%s: %s' % kv for kv in kw.items())))
        add('concatenate_1', class_name='Concatenate', axis=1)
        add('conv2d_1', class_name='Conv2D', filters=F, kernel_size='[3, 3]', padding='same', activation='relu',
            kernel_initializer='he_uniform')
        for l in range(self.num_layers):
            add('conv2d_%d' % (2 * l + 2), class_name='Conv2D', filters=F, kernel_size='[3, 3]', padding='same', activation='relu',
                kernel_initializer='he_uniform')
            add('conv2d_%d' % (2 * l + 3), class_name='Conv2D', filters=F, kernel_size='[3, 3]', padding='same',
                activation='linear', kernel_initializer='he_uniform')
            add('lambda_%d' % (l + 1), class_name='Lambda', scale=0.1)
            add('add_%d' % (l + 1), class_name='Add')
        add('conv2d_%d' % (2 * self.num_layers + 2), class_name='Conv2D', filters=self.out_channels, kernel_size='[3, 3]',
            padding='same', activation='linear', kernel_initializer='he_uniform')
        add('add_%d' % (self.num_layers + 1), class_name='Add', skip='last input')
        return '\n'.join(lines) + '\n'


def s2model(input_shape, num_layers=32, feature_size=256, seed=None):
    """Same signature as DSen2Net.py:18 (plus an optional ``seed`` for the he_uniform initialiser)."""
    return S2Model(input_shape, num_layers=num_layers, feature_size=feature_size, seed=seed)
