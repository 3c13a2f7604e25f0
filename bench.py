#!/usr/bin/env python
"""Headline benchmark: output Mpixel/s of DSen2 20 m -> 10 m super-resolution of a synthetic full
10980 x 10980 Sentinel-2 tile (BASELINE.json configs[2]), patches sharded across N B200s of one node.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (oracle port)
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/*.npy

One "step" = one pass of the hot path over the whole tile: extract(/2000) -> bilinear(/2000) -> 14 tcgen05
convolutions -> stitch(x2000) for every patch the rank owns.  Rank 0 prints ONE JSON line.
  value  : device-resident inputs/outputs, CUDA-event timed, max over ranks.
  e2e    : same step through pinned HOST buffers (H2D of the rank's input rows + D2H of its output rows).
  roofline: the resblock convolution kernel (12 of the 14 convs), CUDA events inside the timed region.
  cpu_baseline: the CPU oracle (torch-CPU restatement of the Keras graph + numpy patch ops) on a bounded crop.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_PIXEL = {('dsen2', 20): 3575808, ('vdsen2', 20): 75571200, ('dsen2', 60): 3571200,
                  ('vdsen2', 60): 75561984}                                                      # SURVEY 2.3 / 8(d)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


DTYPE_Q8 = ("fp16 operands, fp32 accumulate (TMEM), residual trunk fp16 + 8 bits (19 significant bits); first/last layer split "
            "hi+lo (fp32-equivalent)")


def peaks():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as fh:
            p = json.load(fh)
        return dict(hbm=p['hbm_gbs'], tf_burst=p['bf16_tflops'], tf_sust=p.get('bf16_tflops_sustained', p['bf16_tflops']),
                    source='measured (MEASURED_PEAKS.json)')
    except Exception:
        return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, source='fallback (B200_PROFILING.md)')


def synth_tile(torch, H, W, device, seed=20170928, with_60=False):
    """SURVEY 8(d) config 3: integer DN, 1600 + 900*smooth + 150*noise clipped to [0, 12000]."""
    g = torch.Generator(device=device).manual_seed(seed)
    F = torch.nn.functional

    def field(h, w, c):
        lo = torch.randn((1, c, h // 64 + 2, w // 64 + 2), generator=g, device=device)
        smooth = F.interpolate(lo, size=(h, w), mode='bilinear', align_corners=False)[0]
        out = torch.empty((h, w, c), device=device)
        for k in range(c):                         # band by band to bound the temporaries
            noise = torch.randn((h, w), generator=g, device=device)
            out[:, :, k] = (1600 + 900 * smooth[k] + 150 * noise).clamp_(0, 12000).round_()
        return out
    return (field(H, W, 4), field(H // 2, W // 2, 6)) + ((field(H // 6, W // 6, 2),) if with_60 else ())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, uuid):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', uuid, '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '200'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception as e:                      # pragma: no cover
            log('clock sampler unavailable:', e)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
                for nme, v in zip(names, r[3:7]):
                    if v.lower().startswith('active'):
                        reasons.add(nme)
            except Exception:
                continue
        loaded = [s for s, p in zip(sm, pw) if p > 0.5 * max(pw)] if pw else sm
        return {"sm_mhz": float(np.median(loaded)) if loaded else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------- #
# CPU oracle legs
# ---------------------------------------------------------------------------------------------- #
def cpu_sample(deep):
    """The bounded sample BOTH CPU legs time (the `--impl reference` arm and the GPU arm's `cpu_baseline`): a crop of the
    synthetic scene whose patch count is a whole number of the reference's predict batches (32 for DSen2, 8 for VDSen2,
    supres.py:65) and whose allocated patch stack has no surplus zero patches (H/2, W/2 not multiples of 56).
    DSen2: 892 x 1340 = 8 x 12 = 96 patches (3 batches, ~5 s per pass on 16 cores); VDSen2: 444 x 444 = 16 patches."""
    return (444, 444) if deep else (892, 1340)


DUMP_SAMPLE = 1 << 20          # rows (output pixels, parameters) kept by --dump-outputs from a larger array


def sample_rows(n, limit=DUMP_SAMPLE, seed=20170928):
    """A fixed, sorted set of at most `limit` row indices out of n, the same from run to run (numpy int64)."""
    if n <= limit:
        return np.arange(n)
    return np.unique(np.random.RandomState(seed).randint(0, n, size=limit, dtype=np.int64))


def dump_outputs(dirname, arrays):
    """--dump-outputs: write each array as dirname/<name>.npy (float32 / float64 only), at most 64 MB in all, so that two
    builds can be compared output for output on the same seeded inputs."""
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values()), {k: a.dtype for k, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= 64 << 20, total
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + '.npy'), np.ascontiguousarray(a))
    log('dumped %d arrays (%.1f MB) to %s' % (len(arrays), total / 2 ** 20, dirname))


def cpu_oracle_run(shape, steps, warmup, deep=False):
    """Time the CPU oracle end to end on an (H, W) 10 m synthetic scene; returns (Mpixel/s, s/step, threads, patches)."""
    import torch
    from oracle import dsen2net_oracle as no
    torch.set_num_threads(os.cpu_count() or 1)
    H, W = shape
    rng = np.random.RandomState(20170928)
    d10 = rng.randint(200, 6000, size=(H, W, 4)).astype(np.float32)
    d20 = rng.randint(200, 6000, size=(H // 2, W // 2, 6)).astype(np.float32)
    w = no.he_uniform_weights(10, 6, 32 if deep else 6, 256 if deep else 128, seed=0)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        out = no.DSen2_20(d10, d20, w)
        dt = time.perf_counter() - t0
        assert out.shape == (H, W, 6)
        if i >= warmup:
            times.append(dt)
    per = float(np.mean(times))
    patches = (-(-H // 112)) * (-(-W // 112))
    return H * W / per / 1e6, per, torch.get_num_threads(), patches


def cpu_sample_text(shape, patches, per):
    return ("%dx%d crop (%d patches = whole predict batches) of the synthetic scene through the CPU oracle port (numpy "
            "extract/bilinear/stitch + torch-CPU fp32 conv graph; TensorFlow/Keras not installable), %.1f s per pass; "
            "extrapolates linearly to the tile" % (shape[0], shape[1], patches, per))


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    deep = args.model == 'vdsen2'
    shape = cpu_sample(deep)
    mpx, per, threads, patches = cpu_oracle_run(shape, args.steps, args.warmup, deep=deep)
    line = {"impl": "reference", "metric": "output_Mpixel_per_s", "value": mpx, "unit": "Mpixel/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": per * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": workload_config(args, cpu=True),
            "cpu_baseline": {"value": mpx, "unit": "Mpixel/s", "cores": threads, "kind": "port",
                             "sample": cpu_sample_text(shape, patches, per)},
            "e2e": {"value": mpx, "unit": "Mpixel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def cpu_train_run(deep, steps, warmup, n):
    """Time the CPU oracle's training step (torch-CPU fp32 autograd of the same graph + NAdam, oracle/train_oracle.py) on n
    patches of 32 x 32; returns (samples/s, s/step, threads)."""
    import torch
    from oracle import dsen2net_oracle as no
    from oracle import train_oracle as to
    torch.set_num_threads(os.cpu_count() or 1)
    g = torch.Generator().manual_seed(1234)                              # SURVEY 8(d) config 5
    xs = [torch.rand((n, c, 32, 32), generator=g).mul_(2.5).numpy() for c in (4, 6)]
    y = torch.rand((n, 6, 32, 32), generator=g).mul_(2.5).numpy()
    w = no.he_uniform_weights(10, 6, 32 if deep else 6, 256 if deep else 128, seed=0)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        to.train_steps([(xs, y)], w, lr=1e-4)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    per = float(np.mean(times))
    return n / per, per, torch.get_num_threads()


def run_reference_train(args):
    """`--impl reference --workload train`: the CPU oracle's training step on the host cores, rank 0 only."""
    if int(os.environ.get('RANK', '0')) != 0:
        return
    deep = args.model == 'vdsen2'
    n = 8 if deep else 32                                                # a bounded sample: one quarter of the DSen2 batch
    sps, per, threads = cpu_train_run(deep, args.steps, args.warmup, n)
    sample = ("%d patches of 32x32 (the GPU arm: %d per GPU) through the CPU oracle's step: torch-CPU fp32 autograd of the same "
              "graph, MAE, torch NAdam(momentum_decay=0.004) = the Keras-2 Nadam recurrence; %.2f s per step; TensorFlow/Keras "
              "not installable" % (n, 8 if deep else 128, per))
    line = {"impl": "reference", "metric": "train_samples_per_s", "value": sps, "unit": "samples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": per * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": {"workload": "%s training step, MAE + Keras-2 Nadam, CPU sample of %d patches 32x32" % (
                'VDSen2 (32x256)' if deep else 'DSen2 (6x128)', n), "batch_per_gpu": n, "cpu_sample_only": True},
            "cpu_baseline": {"value": sps, "unit": "samples/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": sps, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def workload_config(args, cpu=False):
    T = args.tile
    P, B = (192, 12) if args.path == 60 else (128, 8)
    n = (-(-T // (P - 2 * B))) ** 2
    return {"workload": "%s %dm->10m, synthetic %dx%d Sentinel-2 tile, %d patches %dx%d (border %d), "
                        "he_uniform weights seed 0 (shipped hdf5 absent)" % ('VDSen2 (32x256)' if args.model == 'vdsen2'
                                                                             else 'DSen2 (6x128)', args.path, T, T, n, P, P, B),
            "tile": T, "patches": n, "device_batch": args.batch, "sharding": "contiguous patch ranges, no collective",
            "l2": "inputs (2.6 GB) and activations larger than L2; no flush needed",
            "cpu_sample_only": bool(cpu)}


# ---------------------------------------------------------------------------------------------- #
# GPU arm
# ---------------------------------------------------------------------------------------------- #
# DRAM bytes per patch and launch of the trunk convolutions, dram__bytes_read.sum + dram__bytes_write.sum of an
# `ncu --set full` capture (a CONSTANT taken from the named file, not measured in the bench run): mean of the RELU layer
# (619 + 571 MB per 147 patches) and the RESIDUALQ layer (1544 + 877 MB per 147 patches).
NCU_TRAFFIC = {128: dict(bytes_per_patch=(1.190e9 + 2.421e9) / 2 / 147, source="profiles/r02_whole_batch_final_ncu_full.txt")}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from dsen2_b200 import sharding, supres
    from dsen2_b200.DSen2Net import s2model
    from dsen2_b200.patches import patch_counts

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    run_60 = args.path == 60
    T, P, B, r = (args.tile, 192, 12, 6) if run_60 else (args.tile, 128, 8, 2)
    if args.batch <= 0:
        args.batch = supres.default_device_batch(T, P, B)
    if T % r:
        raise SystemExit("--tile must be a multiple of %d for the %d m path" % (r, args.path))
    deep = args.model == 'vdsen2'
    shape = ((4, None, None), (6, None, None)) + (((2, None, None),) if run_60 else ())
    model = s2model(shape, num_layers=32 if deep else 6, feature_size=256 if deep else 128, seed=0)
    tile = synth_tile(torch, T, T, dev, with_60=run_60)
    d10, d20 = tile[0], tile[1]
    d60 = tile[2] if run_60 else None
    _, filled = patch_counts(T // r, T // r, P // r, B // r)
    first, count = sharding.shard_range(filled, rank, world)
    cout = model.out_channels
    out = torch.zeros((T, T, cout), dtype=torch.float32, device=dev)
    n_batches = -(-count // args.batch)
    # per batch: 1 input-preparation kernel + 2 + 2 * num_layers convolutions (extract / bilinear / stitch are fused into them)
    launches_per_step = n_batches * model.launches_per_forward()

    def step(timers=None):
        supres.super_resolve_device(model, d10, d20, d60, first_patch=first, num_patches=count, out=out,
                                    device_batch=args.batch, timers=timers)

    # ---- value: device-resident ---------------------------------------------------------------
    for _ in range(args.warmup):
        step()
    timers = {}
    barrier()
    uuid = str(torch.cuda.get_device_properties(dev).uuid)
    sampler = ClockSampler(uuid if uuid.startswith('GPU-') else 'GPU-' + uuid) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step(timers)
    e1.record()
    barrier()
    clocks = sampler.stop() if sampler else None
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    ms_step = ms_total / args.steps
    value = T * T / (ms_step * 1e-3) / 1e6
    if args.dump_outputs:
        # the super-resolved tile of the last timed step: a seeded sample of its pixels (all bands) and the full-resolution
        # top-left corner, which spans several patch seams.  Each rank wrote only the pixels its patches own into a
        # zero-filled canvas, so a sum over ranks assembles the whole tile's values.
        idx = torch.from_numpy(sample_rows(T * T)).to(dev)
        c = min(T, 512)
        parts = [out.view(T * T, cout).index_select(0, idx), out[:c, :c].contiguous()]
        if world > 1:
            for t in parts:
                dist.all_reduce(t)
        if rank == 0:
            dump_outputs(args.dump_outputs, {"sr_pixel_sample": parts[0].cpu().numpy(), "sr_corner": parts[1].cpu().numpy()})
        del parts

    # roofline of the dominant kernel (resblock convolutions), from the events recorded in the timed region
    pk = peaks()
    F = model.feature_size
    conv_ms, conv_n = [], []
    for kind in ('conv_res1', 'conv_res2'):
        for a, b, n in timers.get(kind, []):
            conv_ms.append(a.elapsed_time(b)); conv_n.append(n)
    kernel_ms = float(np.mean(conv_ms))
    per_kind = {k: float(np.sum([a.elapsed_time(b) for a, b, _ in v])) / args.steps for k, v in timers.items()}
    exec_flop = 2.0 * 9 * F * F * P * P * float(np.mean(conv_n))                 # executed per launch
    # algorithmic work = output pixels only (SURVEY 8(d)): the reference tiling recomputes the patch overlap
    algo_flop = exec_flop * (float(T) * T) / (float(filled) * P * P)
    by_epi = {}
    for kind, label in (('conv_res1', 'relu'), ('conv_res2', 'residual')):
        ms = [a.elapsed_time(b) for a, b, _ in timers.get(kind, [])]
        if ms:
            by_epi[label] = {"avg_launch_ms": float(np.mean(ms)), "tflops_executed": exec_flop / float(np.mean(ms)) / 1e9,
                             "frac_executed": exec_flop / float(np.mean(ms)) / 1e9 / pk['tf_sust']}
    ncu = NCU_TRAFFIC.get(F)
    traffic = ncu['bytes_per_patch'] * float(np.mean(conv_n)) if ncu else None
    traffic_src = ("CONSTANT, not measured in this run: ncu --set full dram__bytes_read+write per launch of %s, scaled "
                   "per patch" % ncu['source']) if ncu else "no ncu capture for this shape"
    kname = ("conv_pair_kernel<N=%d> (CTA-pair tcgen05 3x3 conv %d->%d, %s weights, RELU / RESIDUALQ epilogues; %d of %d convs)"
             % (F, F, F, 'shared-memory resident' if F == 128 else 'streamed', 2 * model.num_layers, 2 * model.num_layers + 2))
    roofline = {"bound": "tensor", "kernel": kname,
                "achieved": algo_flop / kernel_ms / 1e9, "achieved_executed": exec_flop / kernel_ms / 1e9,
                "peak": pk['tf_sust'], "peak_burst": pk['tf_burst'], "peak_source": pk['source'] + ", sustained figure (kernel timed inside a long step)",
                "unit": "TFLOP/s", "frac": algo_flop / kernel_ms / 1e9 / pk['tf_sust'],
                "frac_executed": exec_flop / kernel_ms / 1e9 / pk['tf_sust'],
                "avg_launch_ms": kernel_ms, "patches_per_launch": float(np.mean(conv_n)),
                "algorithmic_flop_per_launch": algo_flop, "executed_flop_per_launch": exec_flop, "traffic": traffic,
                "traffic_source": traffic_src, "by_epilogue": by_epi, "ms_per_step_by_kernel": per_kind}

    # ---- e2e: pinned host -> device -> pinned host every step, through the public host-buffer pipeline --------
    # supres.HostPipeline is what supres.DSen2_20 runs: chunked uploads / compute / downloads overlapped on three
    # streams.  Host inputs are uint16 digital numbers (what Sentinel-2 L1C holds and GDAL delivers,
    # s2_tiles_supres.py:311-315; the synthetic DN are integers), the output float32 as the reference returns it.
    # Each rank moves only the input rows its patches read and the output pixels they own.
    y0, y1 = sharding.output_rows(first, count, T, T, P, B)
    dev_rows = out[y0:y1].clone()                       # device-resident result, to check the e2e result against
    h10 = torch.empty((T, T, 4), dtype=torch.uint16).pin_memory()
    h20 = torch.empty((T // 2, T // 2, 6), dtype=torch.uint16).pin_memory()
    h60 = torch.empty((T // 6, T // 6, 2), dtype=torch.uint16).pin_memory() if run_60 else None
    hout = torch.zeros((T, T, cout), dtype=torch.float32).pin_memory()
    h10.numpy()[...] = d10.cpu().numpy()                # integer-valued float32 -> uint16, exact
    h20.numpy()[...] = d20.cpu().numpy()
    if run_60:
        h60.numpy()[...] = d60.cpu().numpy()
    torch.cuda.synchronize()
    del d10, d20, d60, tile, out
    torch.cuda.empty_cache()
    pipe = supres.HostPipeline(model, T, T, run_60=run_60, device=dev, device_batch=args.batch, dtype=torch.uint16)

    def step_e2e():
        pipe.run(h10, h20, h60, hout=hout, first_patch=first, num_patches=count)

    for _ in range(max(1, args.warmup // 2)):
        step_e2e()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step_e2e()
    e1.record()
    barrier()
    e2e_ms = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    h2d, d2h = pipe.h2d_bytes, pipe.d2h_bytes
    if world > 1:
        tb = torch.tensor([h2d, d2h], dtype=torch.float64, device=dev)
        dist.all_reduce(tb)
        h2d, d2h = int(tb[0].item()), int(tb[1].item())
    # the rows this rank owns completely: host-pipeline result (uint16 in, chunked) == device-resident result (float32 in)
    rects = [rc for rc in sharding.owned_rects(first, count, T, T, P, B) if rc[2] == 0 and rc[3] == T]
    same = all(bool(torch.equal(hout[a:b].to(dev), dev_rows[a - y0:b - y0])) for a, b, _, _ in rects)
    checksum = float(hout[y0:y1:97, ::89].double().sum())
    del dev_rows

    # ---- e2e through the facade itself: supres.DSen2_20(numpy, numpy, model=) -> numpy, pageable host arrays -----------
    facade = None
    if world == 1 and not args.no_facade:
        n10, n20 = h10.numpy().copy(), h20.numpy().copy()          # ordinary (pageable) numpy arrays, uint16 DN
        n60 = h60.numpy().copy() if run_60 else None
        del pipe
        torch.cuda.empty_cache()
        call = (lambda **kw: supres.DSen2_60(n10, n20, n60, model=model, **kw)) if run_60 else \
            (lambda **kw: supres.DSen2_20(n10, n20, model=model, **kw))
        res = call()                                               # first call: allocates the pipeline + staging ring
        fresh, reuse = [], []
        for _ in range(2):
            t0 = time.perf_counter(); res = call(); fresh.append(time.perf_counter() - t0)
        for _ in range(2):
            t0 = time.perf_counter(); call(out=res); reuse.append(time.perf_counter() - t0)
        ok = bool(np.array_equal(res[y0:y1:97, ::89], hout[y0:y1:97, ::89].numpy()))
        facade = {"call": "supres.DSen2_%d(numpy uint16 ..., model=) -> numpy float32, pageable host arrays" % args.path,
                  "ms_fresh_output": float(np.mean(fresh)) * 1e3, "ms_reused_output": float(np.mean(reuse)) * 1e3,
                  "value_fresh_output": T * T / float(np.mean(fresh)) / 1e6, "value_reused_output": T * T / float(np.mean(reuse)) / 1e6,
                  "unit": "Mpixel/s", "timing": "host wall clock around the call (it synchronises), mean of 2",
                  "matches_pinned_pipeline": ok}

    if rank == 0:
        line = {"metric": "output_Mpixel_per_s", "value": value, "unit": "Mpixel/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": DTYPE_Q8,
                "data": "synthetic", "config": workload_config(args), "clocks": clocks,
                "e2e": {"value": T * T / (e2e_ms * 1e-3) / 1e6, "unit": "Mpixel/s", "ms_per_step": e2e_ms,
                        "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "host_buffers": "pinned; inputs uint16 DN, output float32",
                        "matches_device_resident": same},
                "gpu_launches": launches_per_step * args.steps, "roofline": roofline,
                "tflops_executed_whole_step": FLOP_PER_PIXEL[(args.model, args.path)] * float(filled) * P * P / (ms_step * 1e-3) / 1e12,
                "checksum": checksum}
        if facade:
            line["e2e_facade"] = facade
        if world == 1 and not args.no_cpu_baseline:
            shp = cpu_sample(deep)                   # the same sample the `--impl reference` arm times
            mpx, per, threads, patches = cpu_oracle_run(shp, 1, 1, deep=deep)     # one untimed pass first, as the reference arm does
            line["cpu_baseline"] = {"value": mpx, "unit": "Mpixel/s", "cores": threads, "kind": "port",
                                    "sample": cpu_sample_text(shp, patches, per)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------- #
# config 5: data-parallel training step (supres_train.py:137-144,218-230), batch 128 per GPU of 32x32 patches
# ---------------------------------------------------------------------------------------------- #
def run_train(args):
    import torch
    import torch.distributed as dist
    from dsen2_b200.DSen2Net import s2model
    from dsen2_b200.train import Nadam, Trainer

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    deep = args.model == 'vdsen2'                                        # supres_train.py:129-131: 32 x 256, batch size 8
    n, P = (args.train_batch or (8 if deep else 128)), 32
    L, F = (32, 256) if deep else (6, 128)
    model = s2model(((4, None, None), (6, None, None)), num_layers=L, feature_size=F, seed=0)
    tr = Trainer(model, Nadam(lr=1e-4), device=dev)
    g = torch.Generator().manual_seed(1234 + rank)                       # SURVEY 8(d) config 5
    host = [torch.rand((n, c, P, P), generator=g).mul_(2.5).pin_memory() for c in (4, 6, 6)]
    devb = [torch.empty((n, c, P, P), device=dev) for c in (4, 6, 6)]
    for d, h in zip(devb, host):
        d.copy_(h)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1) / args.steps
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    losses, last = [], [None]

    def step_dev():
        last[0] = tr.train_step(devb[:2], devb[2])

    def step_e2e():
        for d, h in zip(devb, host):
            d.copy_(h, non_blocking=True)
        loss, _ = tr.train_step(devb[:2], devb[2])
        losses.append(float(loss))                                      # device -> host read of the step's result

    ms = timed(step_dev)
    if args.dump_outputs and rank == 0:
        # what a caller of the step receives after the last timed step: its loss / MSE and the updated fp32 master
        # weights (a seeded sample of them when they exceed the dump budget, as VDSen2's 37.8 M do)
        loss, mse = last[0]
        idx = torch.from_numpy(sample_rows(tr.params.numel(), 4 * DUMP_SAMPLE)).to(dev)
        dump_outputs(args.dump_outputs, {"loss": loss.double().cpu().numpy().reshape(1),
                                         "mse": mse.double().cpu().numpy().reshape(1),
                                         "params_sample": tr.params.index_select(0, idx).cpu().numpy()})
    ms_e2e = timed(step_e2e)
    # the one exchange step of the path: all-reduce of the flat fp32 gradient (1.79 M elements), timed on its own
    allreduce_us = None
    if world > 1:
        from dsen2_b200.train import allreduce_gradients
        g = torch.zeros_like(tr.grads)
        for _ in range(5):
            allreduce_gradients(g)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            allreduce_gradients(g)
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1) / 20 * 1e3], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        allreduce_us = float(t.item())
    flop = 3.0 * FLOP_PER_PIXEL[(args.model, 20)] * n * P * P            # forward + backward-data + weight-gradient
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:            # the oracle's step on the host cores, bounded sample
        ncpu = 8 if deep else 32
        sps, per, threads = cpu_train_run(deep, 3, 1, ncpu)
        cpu = {"value": sps, "unit": "samples/s", "cores": threads, "kind": "port",
               "sample": "%d patches of 32x32 through the CPU oracle's step (torch-CPU fp32 autograd + NAdam), %.2f s per step, "
                         "3 steps after 1 warm-up" % (ncpu, per)}
    if rank == 0:
        pk = peaks()
        line = {"metric": "train_samples_per_s", "value": world * n / (ms * 1e-3), "unit": "samples/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "fp16 operands / gradients (loss-scaled), fp32 accumulate, fp32 master weights + Nadam",
                "data": "synthetic",
                "config": {"workload": "%s training step, %d patches 32x32 per GPU, MAE + Keras-2 Nadam, "
                                       "NCCL all-reduce of %.2f M fp32 gradients" % ('VDSen2 (32x256)' if deep else 'DSen2 (6x128)', n,
                                                                                    tr.grads.numel() / 1e6), "batch_per_gpu": n,
                           "l2": "activations kept for the backward pass: %.2f GB per step%s" % (
                               (2 * L + 1) * n * P * P * F * 2 / 1e9, " > L2" if (2 * L + 1) * n * P * P * F * 2 > 126e6 else
                               " (L2-resident: the reference's batch size; weights %.0f MB stream from HBM)" % (tr.grads.numel() * 2 / 1e6))},
                "e2e": {"value": world * n / (ms_e2e * 1e-3), "unit": "samples/s", "ms_per_step": ms_e2e,
                        "h2d_bytes_per_step": world * sum(h.numel() * 4 for h in host), "d2h_bytes_per_step": world * 8},
                "gpu_launches": tr.launches_per_step() * args.steps,
                "roofline": {"bound": "tensor", "kernel": "whole step (conv_pair_kernel fwd/dgrad + wgrad_kernel)",
                             "achieved": flop / ms / 1e9, "peak": pk['tf_burst'], "unit": "TFLOP/s",
                             "frac": flop / ms / 1e9 / pk['tf_burst'], "traffic": None,
                             "peak_source": pk['source'] + ", burst figure (millisecond-scale step)"},
                "kernel_shares_ncu": dict(
                    {"note": "CONSTANTS from an ncu gpu__time_duration launch list of this workload (profiles/%s), not measured "
                             "in this run" % ("r02_train_vdsen2_launch_list.txt" if deep else "r02_train_launch_list.txt")},
                    **({"forward + backward-data convolutions (conv_pair_kernel, conv_tail_swapped_kernel)": 0.648,
                        "weight + bias gradients (wgrad_direct_kernel)": 0.273, "Nadam": 0.038, "operand repacking": 0.024,
                        "loss, layout, fills": 0.017} if deep else
                       {"forward + backward-data convolutions (conv_pair_kernel)": 0.615,
                        "weight + bias gradients (wgrad_direct_kernel)": 0.316, "Nadam": 0.006, "operand repacking": 0.012,
                        "loss, layout, fills": 0.051})),
                "allreduce": {"us": allreduce_us, "bytes": int(tr.grads.numel()) * 4, "algo": ("NCCL all_reduce(SUM) in two buckets between the gradient graphs and the update "
                                       "graph: the later layers' bucket runs beside the rest of the backward pass" if tr._overlap_allreduce(n, P)
                                       else "NCCL all_reduce(SUM), one bucket, between the gradient graph and the update graph") +
                              "; `us` is ONE all-reduce of the whole gradient, timed alone"} if world > 1 else None,
                "cpu_baseline": cpu,
                "last_loss": losses[-1] if losses else None}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None, help='timed steps (default 3; 50 for the GPU training step)')
    ap.add_argument('--warmup', type=int, default=None, help='untimed steps first (default 3; 10 for the GPU training step)')
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--model', default='dsen2', choices=['dsen2', 'vdsen2'])
    ap.add_argument('--tile', type=int, default=10980)
    ap.add_argument('--path', type=int, default=20, choices=[20, 60], help='20 m -> 10 m (DSen2_20) or 60 m -> 10 m (DSen2_60)')
    ap.add_argument('--batch', type=int, default=0, help='patches per device batch (0 = whole patch rows, see supres.default_device_batch)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-facade', action='store_true', help='skip the e2e_facade leg (numpy -> supres.DSen2_20 -> numpy)')
    ap.add_argument('--workload', default='tile', choices=['tile', 'train'],
                    help="'tile' = the headline inference benchmark; 'train' = BASELINE.json configs[4] (training step)")
    ap.add_argument('--train-batch', type=int, default=0, help='patches per GPU and step (0 = the reference\'s: 128, or 8 with --model vdsen2)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step computed as DIR/<name>.npy (float32 / float64, at most 64 MB)')
    args = ap.parse_args()
    gpu_train = args.workload == 'train' and args.impl == 'ours'
    if args.steps is None:
        args.steps = 50 if gpu_train else 3
    if args.warmup is None:
        args.warmup = 10 if gpu_train else 3
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes the outputs of the CUDA path (--impl ours)')
    if gpu_train:
        run_train(args)
    elif args.impl == 'reference' and args.workload == 'train':
        run_reference_train(args)
    elif args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
