"""Training step of the DSen2 network -- mirror of ``training/supres_train.py:137-144, 218-230``:

    nadam = Nadam(lr=1e-4, beta_1=0.9, beta_2=0.999, epsilon=1e-8, schedule_decay=0.004)
    model.compile(optimizer=nadam, loss='mean_absolute_error', metrics=['mean_squared_error'])
    model.fit(x=train, y=label, batch_size=128, ...)

One ``Trainer.train_step`` = forward + MAE loss + backward + (NCCL all-reduce of the flat gradient when the process
group has more than one rank) + Keras-2 Nadam update, all in the CUDA kernels behind ``include/dsen2_b200.h``:
the forward and backward-data convolutions are the CTA-pair tcgen05 kernels (``csrc/conv_pair.cu``; backward uses
flipped / transposed operands), weight gradients are tcgen05 GEMMs over the pixel dimension
(``csrc/train_kernels.cu``).  Activations and gradients are fp16 operands with fp32 accumulation; gradients carry a
power-of-two loss scale so that the MAE gradient sign(pred-y)/N enters the fp16 data path as exactly +-2^-4.
Master weights, gradients and the Nadam moments are fp32.  DSen2 (feature_size 128) and VDSen2 (256; ``--deep``,
``supres_train.py:129-131``: the 256-channel layers stream their weights, weight gradients run per 128 x 128 block).
"""
import gc
import math
import os

import numpy as np

from . import _capi


class Nadam:
    """Hyper-parameters of ``keras.optimizers.Nadam`` as the reference configures it (supres_train.py:137-141)."""

    def __init__(self, lr=1e-4, beta_1=0.9, beta_2=0.999, epsilon=1e-8, schedule_decay=0.004):
        self.lr, self.beta_1, self.beta_2, self.epsilon, self.schedule_decay = lr, beta_1, beta_2, epsilon, schedule_decay


def nadam_schedule(t, m_schedule, opt):
    """Keras-2 Nadam momentum schedule at (1-based) iteration t -> dict of the scalars the update kernel needs."""
    mu_t = opt.beta_1 * (1.0 - 0.5 * 0.96 ** (t * opt.schedule_decay))
    mu_next = opt.beta_1 * (1.0 - 0.5 * 0.96 ** ((t + 1) * opt.schedule_decay))
    sched_new = m_schedule * mu_t
    return dict(mu_t=mu_t, mu_next=mu_next, sched_new=sched_new, sched_next=sched_new * mu_next,
                bias2=1.0 - opt.beta_2 ** t)


def dist_setup(backend=None):
    """One process per GPU under ``torch.distributed.run``: pick this rank's device and join the process group BEFORE any
    model / trainer state is created (a Trainer lives on the current CUDA device).  Returns (rank, world).  Without the
    launcher's environment: (0, 1) and nothing is initialised."""
    if 'RANK' not in os.environ or int(os.environ.get('WORLD_SIZE', '1')) <= 1:
        return 0, 1
    import torch
    import torch.distributed as dist
    if backend is None:
        backend = 'nccl' if torch.cuda.is_available() else 'gloo'
    if torch.cuda.is_available():
        torch.cuda.set_device(int(os.environ.get('LOCAL_RANK', '0')))
    if not dist.is_initialized():
        dist.init_process_group(backend)
    return dist.get_rank(), dist.get_world_size()


def broadcast_weights(model, src=0, group=None):
    """Replicas must start from the same parameters (he_uniform draws differ per process): rank ``src``'s weights replace
    everybody's.  Works on the model's host arrays, so it runs under NCCL and gloo alike."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return model
    ws = model.get_weights()
    flat = torch.from_numpy(np.concatenate([a.ravel() for a in ws]).astype(np.float32))
    if dist.get_backend(group) == 'nccl':
        flat = flat.cuda()
    dist.broadcast(flat, src=src, group=group)
    flat = flat.cpu().numpy()
    out, o = [], 0
    for a in ws:
        out.append(flat[o:o + a.size].reshape(a.shape).copy())
        o += a.size
    model.set_weights(out)
    return model


def shard_training_set(arrays, label, rank, world):
    """Strided shares of the (identically ordered) training set, truncated to the SAME length on every rank: all ranks then
    run the same number of steps per epoch, so every gradient all-reduce has all its participants."""
    n = (label.shape[0] // world) * world
    return [a[rank:n:world] for a in arrays], label[rank:n:world]


def allreduce_gradients(flat, group=None, async_op=False):
    """Sum the flat gradient over the ranks (NCCL on GPUs, gloo in the CPU tests); returns the world size to divide by
    (``async_op``: the pending work handle instead -- the collective then runs beside whatever is launched next)."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return None if async_op else 1
    world = dist.get_world_size(group)
    if async_op:
        return dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group, async_op=True) if world > 1 else None
    if world > 1:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    return world


class Trainer:
    GSCALE = 2.0 ** -4          # value of the scaled MAE gradient entering the fp16 backward path

    def __init__(self, model, optimizer=None, device=None, group=None):
        torch = _capi.require_cuda()
        if model.feature_size not in (128, 256):
            raise _capi.DSen2Error("training is implemented for feature_size 128 (DSen2) and 256 (VDSen2)")
        if model.feature_size == 256 and model.out_channels > 7:
            raise _capi.DSen2Error("feature_size 256: at most 7 output bands (dsen2_conv_tail16)")
        self.torch, self.model, self.opt, self.group = torch, model, optimizer or Nadam(), group
        self.dev = torch.device('cuda', torch.cuda.current_device()) if device is None else device
        self.F, self.L = model.feature_size, model.num_layers
        self.ctot, self.cout = sum(model.in_channels), model.out_channels
        shapes = model.layer_shapes
        self.sizes = []
        for cin, cout in shapes:
            self.sizes += [9 * cin * cout, cout]
        self.offsets = np.concatenate([[0], np.cumsum(self.sizes)]).astype(np.int64)
        total = int(self.offsets[-1])
        flat = np.concatenate([a.ravel() for a in model.get_weights()]).astype(np.float32)
        assert flat.size == total
        self.params = torch.from_numpy(flat).to(self.dev)
        self.grads = torch.zeros(total, dtype=torch.float32, device=self.dev)
        self.m = torch.zeros_like(self.grads)
        self.v = torch.zeros_like(self.grads)
        self.iterations, self.m_schedule = 0, 1.0
        self.sums = torch.zeros(2, dtype=torch.float64, device=self.dev)
        self.zero_bias = torch.zeros(model.feature_size, dtype=torch.float32, device=self.dev)
        # 128 features: first / last layer on the 64-channel prepared input (dsen2_conv_head / dsen2_conv_tail); 256: the
        # inference path's 16-channel forms (dsen2_conv_head16_relu / dsen2_conv_tail16), whose N = 512 stacked head does not
        # fit the tensor memory
        self.in16 = model.feature_size == 256
        self._bufs = {}
        # replay the whole step as one CUDA graph from the third call of a shape on (DSEN2_TRAIN_NO_GRAPH=1: eager, for ncu)
        self.use_graph = not os.environ.get('DSEN2_TRAIN_NO_GRAPH')
        self._graphs, self._calls = {}, {}
        # Data parallel: the gradient of the LATER layers (the tail of the flat vector; their backward pass runs first) is
        # all-reduced while the backward pass of the first `split_l` resBlocks and the first layer still runs -- see
        # `_overlap_allreduce`.  DSEN2_TRAIN_NO_OVERLAP=1 forces the single all-reduce after the whole backward pass.
        self.split_l = max(1, model.num_layers // 4) if model.num_layers > 0 else 0
        self.no_overlap = bool(os.environ.get('DSEN2_TRAIN_NO_OVERLAP'))
        # step-dependent Nadam scalars travel through a ring of pinned staging buffers: a slot is rewritten only after the
        # asynchronous upload that last used it has completed (train_step returns without synchronising)
        self.hp_ring = [[torch.zeros(10, dtype=torch.float32).pin_memory(), None] for _ in range(8)]
        self.hp_dev = torch.zeros(10, dtype=torch.float32, device=self.dev)
        self.loss_out = torch.zeros(2, dtype=torch.float64, device=self.dev)
        f16 = lambda *s: torch.empty(s, dtype=torch.float16, device=self.dev)
        F, L = self.F, self.L
        # the 2L trunk layers' operands are stacked so that ONE launch repacks them all after every update
        self.w_fwd_trunk, self.w_bwd_trunk = f16(max(2 * L, 1), 9, F, F), f16(max(2 * L, 1), 9, F, F)
        self.w_fwd = ([f16(9, 2 * F, 16) if self.in16 else f16(3, 2 * F, 64)] + [self.w_fwd_trunk[i] for i in range(2 * L)] +
                      [f16(128, F) if self.in16 else f16(9, 32, F)])
        self.w_bwd = [None] + [self.w_bwd_trunk[i] for i in range(2 * L)] + [f16(9, F, F)]
        # biases: the F-channel layers read theirs straight from the flat parameter vector (a view, nothing to copy after an
        # update); the last layer's is padded to 16
        self.b_fwd = [self.bias(i) if c == self.F else torch.zeros(max(c, 16), dtype=torch.float32, device=self.dev)
                      for i, (_, c) in enumerate(shapes)]
        self.gw_head = torch.zeros((9, F, F), dtype=torch.float32, device=self.dev)
        self.gw_tail = torch.zeros((9, F, F), dtype=torch.float32, device=self.dev)
        self.gb_tail = torch.zeros(F, dtype=torch.float32, device=self.dev)
        self.repack()

    # ---- parameter views -------------------------------------------------------------------------------------
    def _view(self, flat, i):
        return flat[int(self.offsets[i]):int(self.offsets[i + 1])]

    def kernel(self, layer, flat=None):
        return self._view(self.params if flat is None else flat, 2 * layer)

    def bias(self, layer, flat=None):
        return self._view(self.params if flat is None else flat, 2 * layer + 1)

    def get_weights(self):
        """Keras order [kernel, bias, ...] as numpy arrays (HWIO kernels)."""
        host = self.params.cpu().numpy()
        out = []
        for i, (cin, cout) in enumerate(self.model.layer_shapes):
            out.append(host[self.offsets[2 * i]:self.offsets[2 * i + 1]].reshape(3, 3, cin, cout).copy())
            out.append(host[self.offsets[2 * i + 1]:self.offsets[2 * i + 2]].copy())
        return out

    def set_weights(self, arrays):
        """New master weights (``model.load_weights`` / ``set_weights`` after ``compile``); the optimizer state is kept, as
        Keras keeps it."""
        flat = np.concatenate([np.asarray(a, np.float32).ravel() for a in arrays])
        if flat.size != self.params.numel():
            raise ValueError("expected %d parameters, got %d" % (self.params.numel(), flat.size))
        self.params.copy_(self.torch.from_numpy(flat).to(self.dev))
        self.repack()

    def repack(self):
        """fp32 master weights -> fp16 operands of the forward and backward-data convolutions."""
        lib, ptr, st = _capi.lib(), _capi.ptr, _capi.stream_ptr()
        F, L, nl = self.F, self.L, 2 * self.L + 2
        with self.torch.cuda.device(self.dev):
            pack_head = lib.dsen2_pack_head16_weights if self.in16 else lib.dsen2_pack_head_weights
            pack_tail = lib.dsen2_pack_tail16_weights if self.in16 else lib.dsen2_pack_tail_weights
            _capi.check(pack_head(ptr(self.kernel(0)), self.ctot, F, ptr(self.w_fwd[0]), st), "pack head")
            if L > 0:
                # the second conv of a resBlock is followed by Lambda(x * 0.1) (DSen2Net.py:13): folded into its
                # backward operand; consecutive F -> F kernels lie 9*F*F + F floats apart in the flat parameter vector
                _capi.check(lib.dsen2_pack_trunk_layers(ptr(self.kernel(1)), 9 * F * F + F, 2 * L, F, 0.1,
                                                        ptr(self.w_fwd_trunk), ptr(self.w_bwd_trunk), st), "pack trunk layers")
            _capi.check(pack_tail(ptr(self.kernel(nl - 1)), F, self.cout, ptr(self.w_fwd[-1]), st), "pack tail")
            _capi.check(lib.dsen2_pack_dgrad_weights(ptr(self.kernel(nl - 1)), F, self.cout, F, F, 1.0, ptr(self.w_bwd[-1]), st),
                        "pack dgrad tail")
            for i in range(nl):
                c = self.model.layer_shapes[i][1]
                if c != F:
                    self.b_fwd[i][:c].copy_(self.bias(i))

    def _buffers(self, n, P):
        key = (n, P)
        b = self._bufs.get(key)
        if b is None:
            torch, F, L = self.torch, self.F, self.L
            f16 = lambda *s: torch.empty(s, dtype=torch.float16, device=self.dev)
            cin = 16 if self.in16 else 64
            b = dict(xin_hi=f16(n, P, P, cin), xin_lo=f16(n, P, P, cin), x_hi=[f16(n, P, P, F) for _ in range(L + 1)],
                     t=[f16(n, P, P, F) for _ in range(L)], x_lo=f16(n, P, P, F),
                     x32=torch.empty((n, P, (P + 7) // 8, F // 4, 8, 4), dtype=torch.float32, device=self.dev),
                     dx32=torch.empty((n, P, (P + 7) // 8, F // 4, 8, 4), dtype=torch.float32, device=self.dev),
                     dx_hi=f16(n, P, P, F), g2=f16(n, P, P, F), dy_nhwc=f16(n, P, P, F),
                     pred=torch.empty((n, self.cout, P, P), dtype=torch.float32, device=self.dev),
                     dpred=torch.empty((n, self.cout, P, P), dtype=torch.float32, device=self.dev),
                     )
            self._bufs[key] = b          # kept for the lifetime of the trainer: captured graphs point into them
        return b

    # ---- forward ---------------------------------------------------------------------------------------------
    def forward(self, xs, b, n, P):
        lib, ptr, st = _capi.lib(), _capi.ptr, _capi.stream_ptr()
        F, L, ch = self.F, self.L, self.model.in_channels
        x2, c2 = (xs[2], ch[2]) if len(xs) == 3 else (None, 0)
        prep = lib.dsen2_prep16_from_patches if self.in16 else lib.dsen2_prep_from_patches
        _capi.check(prep(ptr(xs[0]), ch[0], ptr(xs[1]), ch[1], ptr(x2), c2, n, P, ptr(b['xin_hi']), ptr(b['xin_lo']), st), "prep")
        if self.in16:
            if L == 0:
                raise _capi.DSen2Error("feature_size 256: training needs at least one resBlock")
            _capi.check(lib.dsen2_conv_head16_relu(ptr(b['xin_hi']), ptr(b['xin_lo']), ptr(self.w_fwd[0]), ptr(self.b_fwd[0]), n, P, P,
                                                   F, ptr(b['x_hi'][0]), ptr(b['x32']), st), "head")
        else:
            _capi.check(lib.dsen2_conv_head(ptr(b['xin_hi']), ptr(b['xin_lo']), ptr(self.w_fwd[0]), ptr(self.b_fwd[0]), n, P, P, F,
                                            ptr(b['x_hi'][0]), ptr(b['x_lo']) if L == 0 else None,
                                            ptr(b['x32']) if L > 0 else None, st), "head")
        for l in range(L):
            _capi.check(lib.dsen2_conv_relu(ptr(b['x_hi'][l]), ptr(self.w_fwd[1 + 2 * l]), ptr(self.b_fwd[1 + 2 * l]), n, P, P, F,
                                            ptr(b['t'][l]), st), "conv1")
            _capi.check(lib.dsen2_conv_res32(ptr(b['t'][l]), ptr(self.w_fwd[2 + 2 * l]), ptr(self.b_fwd[2 + 2 * l]), n, P, P, F, 0.1,
                                             ptr(b['x32']), ptr(b['x_hi'][l + 1]), ptr(b['x_lo']) if l == L - 1 else None, st),
                        "conv2")
        if self.in16:
            _capi.check(lib.dsen2_conv_tail16(ptr(b['x_hi'][L]), ptr(b['x_lo']), ptr(self.w_fwd[-1]), ptr(self.b_fwd[-1]),
                                              ptr(b['xin_hi']), ptr(b['xin_lo']), self.ctot - self.cout, self.cout, F, n, P, P,
                                              ptr(b['pred']), st), "tail")
        else:
            _capi.check(lib.dsen2_conv_tail(ptr(b['x_hi'][L]), ptr(b['x_lo']), ptr(self.w_fwd[-1]), ptr(self.b_fwd[-1]),
                                            ptr(b['xin_hi']), ptr(b['xin_lo']), self.ctot - self.cout, self.cout, n, P, P,
                                            ptr(b['pred']), st), "tail")
        return b['pred']

    # ---- one optimisation step ----------------------------------------------------------------------------------
    def train_step(self, xs, y, apply=True):
        """One optimisation step (see ``_step_body``).  The first call of a batch shape runs eagerly (it also performs the
        one-time kernel attribute set-up), the second is captured into a CUDA graph (~65 launches, an NCCL all-reduce
        and the repacking of the weights), later calls copy the batch into the graph's static buffers, upload the ten
        step-dependent Nadam scalars and replay it."""
        torch = self.torch
        n, P = int(xs[0].shape[0]), int(xs[0].shape[2])
        key = (n, P, len(xs))
        if not (apply and self.use_graph):
            return self._step_body(xs, y, apply)
        calls = self._calls.get(key, 0)
        self._calls[key] = calls + 1
        if calls == 0:
            return self._step_body(xs, y, True)
        b = self._buffers(n, P)
        if 'in_x' not in b:
            b['in_x'] = [torch.empty_like(x) for x in xs]
            b['in_y'] = torch.empty_like(y)
        with torch.cuda.device(self.dev):
            for d, s_ in zip(b['in_x'], xs):
                d.copy_(s_, non_blocking=True)
            b['in_y'].copy_(y, non_blocking=True)
            self._advance_schedule(1.0 / self._world())
            multi = self._world() > 1
            overlap = multi and self._overlap_allreduce(n, P)
            if key not in self._graphs:
                # one graph on a single GPU; with several ranks the NCCL all-reduce stays an eager call between
                # "gradient" graphs and an "update" graph (a collective inside the capture deadlocked in testing).
                # The cyclic garbage collector stays off while capturing: a dropped model and its trainer form a cycle, and
                # collecting it there would destroy that trainer's graphs, which a capturing stream does not permit (it
                # invalidates this capture).
                gc_was_enabled = gc.isenabled()
                gc.disable()
                try:
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        loss, mse = self._step_body(b['in_x'], b['in_y'], not multi, dev_hp=True,
                                                    part='a' if overlap else None)
                        self.loss_out[0].copy_(loss)
                        self.loss_out[1].copy_(mse)
                    gb = g2 = None
                    if overlap:
                        gb = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(gb):
                            self._step_body(b['in_x'], b['in_y'], False, part='b')
                    if multi:
                        g2 = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(g2):
                            self._update_dev()
                finally:
                    if gc_was_enabled:
                        gc.enable()
                self._graphs[key] = (g, gb, g2)
            g, gb, g2 = self._graphs[key]
            g.replay()
            if overlap:
                off = int(self.offsets[2 * (1 + 2 * self.split_l)])     # first element of resBlock `split_l`'s first kernel
                late = allreduce_gradients(self.grads[off:], self.group, async_op=True)
                gb.replay()                                             # ... runs beside the collective
                early = allreduce_gradients(self.grads[:off], self.group, async_op=True)
                late.wait()
                early.wait()
                g2.replay()
            elif multi:
                allreduce_gradients(self.grads, self.group)
                g2.replay()
            return self.loss_out[0].clone(), self.loss_out[1].clone()

    def _overlap_allreduce(self, n, P):
        """Two buckets: the all-reduce of the later layers' gradients runs beside the backward pass of the first `split_l`
        resBlocks and the first layer.  Measured piece by piece on two B200s (tools/gpu_overlap_probe.py) for VDSen2
        (151 MB of gradients, batch 8): the 241 us all-reduce of the late bucket disappears behind the concurrent part of
        the backward pass, which slows from 621 to 702 us; step 4.40 -> 4.24 ms (8 GPUs: 4.45 -> 4.35 ms).  DSen2's 7 MB
        gradient is a latency-bound collective (44 us on two GPUs, 74 us on eight): two of them cost as much as they hide
        (8 GPUs: 1.72 ms with one bucket, 1.82 ms with two on another box), so small gradients keep the single all-reduce."""
        return not self.no_overlap and self.L > 0 and self.grads.numel() * 4 >= (32 << 20)

    def _update_dev(self):
        """Nadam update with the scalars published in ``hp_dev`` + operand repacking (capturable)."""
        lib, ptr, st = _capi.lib(), _capi.ptr, _capi.stream_ptr()
        _capi.check(lib.dsen2_nadam_step_dev(ptr(self.params), ptr(self.grads), ptr(self.m), ptr(self.v), self.params.numel(),
                                             ptr(self.hp_dev), st), "nadam")
        self.repack()

    def _world(self):
        import torch.distributed as dist
        return dist.get_world_size(self.group) if (dist.is_available() and dist.is_initialized()) else 1

    def _advance_schedule(self, grad_mul):
        """Host side of one Nadam iteration: advance t and the momentum schedule, publish the scalars to the device."""
        self.iterations += 1
        s = nadam_schedule(self.iterations, self.m_schedule, self.opt)
        self.m_schedule = s['sched_new']
        o = self.opt
        vals = [grad_mul, o.lr, o.beta_1, o.beta_2, o.epsilon, s['mu_t'], s['mu_next'], s['sched_new'], s['sched_next'], s['bias2']]
        slot = self.hp_ring[self.iterations % len(self.hp_ring)]
        if slot[1] is not None:
            slot[1].synchronize()
        for i, v_ in enumerate(vals):
            slot[0][i] = float(v_)
        self.hp_dev.copy_(slot[0], non_blocking=True)
        slot[1] = self.torch.cuda.Event()
        slot[1].record()
        return s

    def _step_body(self, xs, y, apply=True, dev_hp=False, part=None):
        """xs: list of CUDA float32 (n,C_i,P,P); y: CUDA float32 (n,Cout,P,P).  Returns (loss, mse) device scalars
        of THIS rank's batch (Keras reports the same quantities per batch).  ``apply=False`` stops after the gradient
        (``self.grads``, flat fp32 in Keras weight order) for inspection.  ``part``: 'a' = forward, loss and the backward
        pass down to resBlock ``split_l`` (the later layers' gradients are then final), 'b' = the rest of the backward
        pass; None = both."""
        torch = self.torch
        lib, ptr = _capi.lib(), _capi.ptr
        n, P = int(xs[0].shape[0]), int(xs[0].shape[2])
        F, L = self.F, self.L
        b = self._buffers(n, P)
        do_a, do_b = part in (None, 'a'), part in (None, 'b')
        split = self.split_l if part is not None else 0     # resBlocks >= split belong to part 'a'
        nl = 2 * L + 2
        npix = n * P * P
        total = b['pred'].numel()
        inv = 1.0 / (self.GSCALE * total)                   # loss scale: d(pred) = GSCALE * sign instead of sign / total
        loss = mse = None
        with torch.cuda.device(self.dev):
            st = _capi.stream_ptr()

            def wgrad(x_nhwc, dy_nhwc, scale, out_w, out_b):
                # out_w (9,F,F) fp32 += scale * sum_px X[px+tap] (x) dY[px];  out_b (F,) fp32 += scale * sum_px dY[px]
                _capi.check(lib.dsen2_wgrad_nhwc(ptr(x_nhwc), ptr(dy_nhwc), n, P, P, F, scale, ptr(out_w), ptr(out_b), st), "wgrad")

            def resblock_bwd(l):                            # DSen2Net.py:9-15, gradient arriving in dx_hi / dx32
                i1, i2 = 1 + 2 * l, 2 + 2 * l
                wgrad(b['t'][l], b['dx_hi'], 0.1 * inv, self.kernel(i2, self.grads), self.bias(i2, self.grads))   # conv2 (x 0.1)
                _capi.check(lib.dsen2_conv_relu_bwd(ptr(b['dx_hi']), ptr(self.w_bwd[i2]), ptr(self.zero_bias), ptr(b['t'][l]),
                                                    n, P, P, F, ptr(b['g2']), st), "dgrad conv2 + relu")
                wgrad(b['x_hi'][l], b['g2'], inv, self.kernel(i1, self.grads), self.bias(i1, self.grads))
                _capi.check(lib.dsen2_conv_res32(ptr(b['g2']), ptr(self.w_bwd[i1]), ptr(self.zero_bias), n, P, P, F, 1.0,
                                                 ptr(b['dx32']), ptr(b['dx_hi']), None, st), "dgrad conv1 + skip")

            if do_a:
                pred = self.forward(xs, b, n, P)
                self.sums.zero_()
                self.grads.zero_()
                self.gw_head.zero_()
                self.gw_tail.zero_()
                self.gb_tail.zero_()
                _capi.check(lib.dsen2_mae_grad(ptr(pred), ptr(y), total, self.GSCALE, ptr(b['dpred']), ptr(self.sums), st), "mae")
                # ---- last layer: Conv2D(cout) (DSen2Net.py:35); the Add of the global skip passes the gradient through
                _capi.check(lib.dsen2_nchw_to_nhwc_f16(ptr(b['dpred']), self.cout, None, 0, None, 0, n, P, P, F, ptr(b['dy_nhwc']),
                                                       st), "dpred nhwc")
                wgrad(b['x_hi'][L], b['dy_nhwc'], inv, self.gw_tail, self.gb_tail)
                self.kernel(nl - 1, self.grads).view(9, F, self.cout).copy_(self.gw_tail[:, :, :self.cout])
                self.bias(nl - 1, self.grads).copy_(self.gb_tail[:self.cout])
                b['dx32'].zero_()
                _capi.check(lib.dsen2_conv_res32(ptr(b['dy_nhwc']), ptr(self.w_bwd[-1]), ptr(self.zero_bias), n, P, P, F, 1.0,
                                                 ptr(b['dx32']), ptr(b['dx_hi']), None, st), "dgrad tail")
                # ---- resBlocks, last to first
                for l in range(L - 1, split - 1, -1):
                    resblock_bwd(l)
                loss = self.sums[0] / total
                mse = self.sums[1] / total
            if do_b:
                for l in range(split - 1, -1, -1):
                    resblock_bwd(l)
                # ---- first layer: Conv2D(F, relu) on the concatenated inputs (DSen2Net.py:24-29)
                _capi.check(lib.dsen2_relu_mask(ptr(b['dx_hi']), ptr(b['x_hi'][0]), npix * F, ptr(b['g2']), st), "relu mask")
                x2, c2 = (xs[2], self.model.in_channels[2]) if len(xs) == 3 else (None, 0)
                _capi.check(lib.dsen2_nchw_to_nhwc_f16(ptr(xs[0]), self.model.in_channels[0], ptr(xs[1]), self.model.in_channels[1],
                                                       ptr(x2), c2, n, P, P, F, ptr(b['dy_nhwc']), st), "input nhwc")
                wgrad(b['dy_nhwc'], b['g2'], inv, self.gw_head, self.bias(0, self.grads))
                self.kernel(0, self.grads).view(9, self.ctot, F).copy_(self.gw_head[:, :self.ctot, :])
            # ---- data-parallel exchange + Nadam (the two-part form leaves both to train_step)
            if part is None and apply and dev_hp:           # single-GPU graph capture: scalars come from hp_dev
                self._update_dev()
            elif part is None and apply:
                world = allreduce_gradients(self.grads, self.group)
                self.apply_gradients(1.0 / world)
        return loss, mse

    def evaluate(self, xs, y):
        """Forward + loss only: (mean_absolute_error, mean_squared_error) of one batch as device scalars."""
        lib, ptr = _capi.lib(), _capi.ptr
        n, P = int(xs[0].shape[0]), int(xs[0].shape[2])
        b = self._buffers(n, P)
        with self.torch.cuda.device(self.dev):
            pred = self.forward(xs, b, n, P)
            total = pred.numel()
            self.sums.zero_()
            _capi.check(lib.dsen2_mae_grad(ptr(pred), ptr(y), total, self.GSCALE, ptr(b['dpred']), ptr(self.sums),
                                           _capi.stream_ptr()), "mae")
            return self.sums[0] / total, self.sums[1] / total

    def apply_gradients(self, grad_mul=1.0):
        lib, ptr, st = _capi.lib(), _capi.ptr, _capi.stream_ptr()
        self.iterations += 1
        s = nadam_schedule(self.iterations, self.m_schedule, self.opt)
        self.m_schedule = s['sched_new']
        o = self.opt
        _capi.check(lib.dsen2_nadam_step(ptr(self.params), ptr(self.grads), ptr(self.m), ptr(self.v), self.params.numel(),
                                         grad_mul, o.lr, o.beta_1, o.beta_2, o.epsilon, s['mu_t'], s['mu_next'], s['sched_new'],
                                         s['sched_next'], s['bias2'], st), "nadam")
        self.repack()

    def launches_per_step(self):
        """Kernels of THIS library per step: forward, loss, backward (dgrad + wgrad with the bias gradients), Nadam, repacking."""
        L = self.L
        fwd = 1 + 1 + 2 * L + 1
        bwd = 1 + 1 + 2 + L * 4 + 3
        return fwd + bwd + 1 + 3 + (1 if L > 0 else 0)        # ... Nadam, first / last layer operand packing, one launch for the trunk
