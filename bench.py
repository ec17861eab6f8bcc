#!/usr/bin/env python
"""Benchmark of the B200 fusion-loss hot path (contract: see the task statement / DESIGN.md §6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[4], the configuration the headline metric is quoted on):
fused loss forward+backward (SSIM + 0.01*pixel-max-L1 + 0.1*Sobel-max-L1, train.py:302-317) on
synthetic 4096x3072 pairs, global batch 64 sharded by batch over the N ranks (strong scaling, the
partition of train.py:209); one step = the three drop-in loss modules + total.backward() on the rank's shard
(ONE launch of the warp-specialised single-pass loss + gradient kernel and the in-place rescale) + one 16-byte
all-reduce of the loss scalars (N > 1).  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

H, W, GLOBAL_B = 3072, 4096, 64            # "4096x3072" is WxH (README.md:67 convention), batch 64
METRIC, UNIT = 'fused_loss_fwd_bwd_throughput', 'Mpix/s'
WORKLOAD = 'fusion loss fwd+bwd, 4096x3072 pairs, global batch 64 (BASELINE configs[4])'
ALG_BYTES_FWD, ALG_BYTES_BWD = 12, 16      # SURVEY.md 8(d): read 3 images; read 3 + write dIf


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--no-extras', action='store_true', help='skip the e2e / metric-suite / cpu legs (profiling runs)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed step returned to DIR/<name>.npy (see dump_outputs), to compare two builds')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs applies to --impl ours')
    return args


def measured_peak():
    """HBM GB/s of this pool's B200s from the driver-written MEASURED_PEAKS.json (the sustained figure when the file
    distinguishes burst / sustained: the kernel is timed inside a long step), else the recipe's fallback."""
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as fh:
            d = json.load(fh)
        flat = {}

        def walk(prefix, obj):
            if isinstance(obj, dict):
                for k, v in obj.items():
                    walk(f'{prefix}.{k}' if prefix else str(k), v)
            elif isinstance(obj, (int, float)) and not isinstance(obj, bool):
                flat[prefix.lower()] = float(obj)

        walk('', d)
        if 'hbm_gbs' in flat:
            return flat['hbm_gbs'], 'measured (MEASURED_PEAKS.json hbm_gbs)'
        cand = [(k, v) for k, v in flat.items() if 'hbm' in k and 1000.0 < v < 20000.0]
        for want in ('sustain', 'gbs', 'gb'):
            for k, v in cand:
                if want in k:
                    return v, f'measured (MEASURED_PEAKS.json {k})'
        if cand:
            return cand[0][1], f'measured (MEASURED_PEAKS.json {cand[0][0]})'
    except Exception:
        pass
    return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU with NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self._halt = index, [], set(), None, threading.Event()

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksThrottleReasonHwSlowdown: 'hw_slowdown',
                     nv.nvmlClocksThrottleReasonHwThermalSlowdown: 'hw_thermal_slowdown',
                     nv.nvmlClocksThrottleReasonSwThermalSlowdown: 'sw_thermal_slowdown',
                     nv.nvmlClocksThrottleReasonSwPowerCap: 'sw_power_cap',
                     nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: 'hw_power_brake'}
            while not self._halt.is_set():
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
                time.sleep(0.02)
        except Exception as e:  # pragma: no cover
            self.reasons.add(f'nvml_unavailable:{type(e).__name__}')

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {'sm_mhz': s[len(s) // 2] if s else None, 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons),
                'samples': len(s)}


def physical_gpu_index(local):
    vis = os.environ.get('CUDA_VISIBLE_DEVICES')
    if vis:
        try:
            return int(vis.split(',')[local])
        except Exception:
            return local
    return local


# ------------------------------------------------------------------------------------ reference arm
def reference_objective():
    """-> (fn(a, b, f) running loss fwd+bwd on the host and returning the gradient, kind, description).
    kind "reference": the reference's OWN core/loss.py modules (byte-compiled artefact oracle/_ref, built by
    oracle/build_ref.py where /root/reference exists); kind "port": the oracle restatement (bit-pinned to it)."""
    try:
        from oracle import build_ref
        RL, _, _ = build_ref.load()
        f1, f2, f3 = RL.SSIMLoss('ssim', weight=1.0), RL.PixelLoss('l1', weight=0.01), RL.GradLoss('l1', weight=0.1)   # train.py:302-308

        def run(a, b, f):
            y = f.detach().requires_grad_(True)
            (f1(a, b, y) + f2(a, b, y, mode='max') + f3(a, b, y, mode='max')).backward()       # train.py:64-71
            return y.grad
        return run, 'reference', "cpu torch, the reference's own core/loss.py (oracle/_ref)"
    except ImportError:
        from oracle import fusion_loss as OL

        def run(a, b, f):
            return OL.train_objective_grad(a, b, f)[1]
        return run, 'port', 'cpu torch, oracle port of core/loss.py (oracle/_ref not built)'


def run_reference(args, rank):
    """The reference's own CPU implementation of the path, all host threads, one bounded sample per
    step: loss fwd+bwd on ONE 4096x3072 pair of the same workload."""
    if rank != 0:
        return
    run, kind, host = reference_objective()
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    g = torch.Generator().manual_seed(0)
    a, b, f = (torch.rand(1, 1, H, W, generator=g) for _ in range(3))

    def step():
        run(a, b, f)

    nwarm = min(args.warmup, 3)            # each step is ~4.5 s of host time on the GPU box
    for _ in range(nwarm):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    val = H * W / 1e6 / dt
    sample = f'1 of {GLOBAL_B} pairs (one 4096x3072 pair, fwd+bwd) per step'
    print(json.dumps({
        'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': nwarm, 'ms_per_step': dt * 1e3, 'higher_is_better': True, 'scaling': 'strong',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': WORKLOAD, 'sample': sample, 'host': host},
        'cpu_baseline': {'value': val, 'unit': UNIT, 'cores': torch.get_num_threads(), 'kind': kind, 'sample': sample},
        'e2e': {'value': val, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0}))


# ------------------------------------------------------------------------------------ our arm
def main():
    args = parse()
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    if args.impl == 'reference':
        run_reference(args, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit('bench.py --impl ours needs a CUDA device (no CPU fallback exists)')
    import torch.distributed as dist
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    import mmif_b200  # noqa: F401
    from mmif_b200 import _lib as L
    from mmif_b200.core import loss as ML
    from mmif_b200.core import metric as MM
    import ctypes

    if GLOBAL_B % world:
        raise SystemExit(f'global batch {GLOBAL_B} not divisible by {world} ranks')
    from mmif_b200 import dist_utils as DU
    B = GLOBAL_B // world
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    a, b, f = (torch.rand(B, 1, H, W, device=dev, generator=g) for _ in range(3))
    lib = L.load()
    L.ensure_device(dev)
    # ---- the timed step IS the reference's call sequence (train.py:64-71) on the drop-in modules -------------------
    fn1, fn2, fn3 = ML.SSIMLoss('ssim', weight=1.0), ML.PixelLoss('l1', weight=0.01), ML.GradLoss('l1', weight=0.1)   # train.py:302-308

    def step(ev=None):
        y = f.detach().requires_grad_(True)              # a fresh imgf every step, as the network produces one
        if ev:
            ev[0].record()
        l1 = fn1(a, b, y)                                # launches fusion_loss_ws_kernel<11,1,2>: loss values + d(total)/d imgf
        if ev:
            ev[1].record()
        l2, l3 = fn2(a, b, y, mode='max'), fn3(a, b, y, mode='max')      # the other two read the same launch
        total = l1 + l2 + l3
        total.backward()                                 # rescale_unit_kernel: in place, exits at once for unit upstream
        if ev:
            ev[2].record()
        if world > 1:                                    # the path's only collective: ONE 16-byte all-reduce, in place on the
            DU.reduce_loss_vector(ML.last_loss_vector(), world)      # kernel's own output vector (train.py:92-96 does four)
        return y.grad, (l1, l2, l3, total)

    # ---- the same work straight through the C ABI: two-kernel path (forward, then recomputing backward) --------------
    cfg = ML._cfg(1.0, 'max', 'max', 'l1', 'l1', 1.0, 0.01, 0.1)
    out = torch.empty(lib.mmif_loss_out_doubles(B), dtype=torch.float64, device=dev)
    ws = torch.zeros(lib.mmif_loss_workspace_bytes(B, H, W), dtype=torch.uint8, device=dev)
    gout = torch.ones(3, device=dev)
    dF = torch.empty_like(f)
    st = L.stream_ptr(dev)

    def fwd():        # two-kernel path, kernel 1: loss values only (12 B/px)
        L.check(lib.mmif_fusion_loss_fwd(a.data_ptr(), b.data_ptr(), f.data_ptr(), B, H, W, ctypes.byref(cfg),
                                         out.data_ptr(), None, ws.data_ptr(), ws.numel(), st))

    def bwd():        # two-kernel path, kernel 2: recomputing backward (16 B/px)
        L.check(lib.mmif_fusion_loss_bwd(a.data_ptr(), b.data_ptr(), f.data_ptr(), B, H, W, ctypes.byref(cfg),
                                         gout.data_ptr(), None, dF.data_ptr(), ws.data_ptr(), ws.numel(), st))

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(run, steps):
        """run(ev) records ev[0..2] around its two phases; returns (ms per step = max over ranks, mean ms of each phase,
        what the last run returned)."""
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
        t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        t_begin.record()
        for k in range(steps):
            last = run(ev[k])
            if k + 1 < steps:
                del last            # freed before the next step allocates its gradient, as a discarded result would be
        t_end.record()
        sync_all()
        ms_total = t_begin.elapsed_time(t_end)
        ms_a = sum(e[0].elapsed_time(e[1]) for e in ev) / steps
        ms_b = sum(e[1].elapsed_time(e[2]) for e in ev) / steps
        tmax = torch.tensor([ms_total], device=dev)
        if world > 1:
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        return tmax.item() / steps, ms_a, ms_b, last

    def two_kernel_step(ev):
        ev[0].record(); fwd(); ev[1].record(); bwd(); ev[2].record()

    for _ in range(max(args.warmup, 3)):
        step()
    sync_all()
    sampler = ClockSampler(physical_gpu_index(local))
    sampler.start()
    c0 = L.launch_counts()
    ms_step, ms_z, ms_rest, last = timed(step, args.steps)
    c1 = L.launch_counts()
    clocks = sampler.stop()
    launches = {k: c1[k] - c0[k] for k in c1}
    assert launches['loss_single_pass'] == args.steps and launches['loss_fwd'] == 0 and launches['loss_bwd'] == 0, launches
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last)
    del last
    grad_modules = step()[0]
    vec = ML.last_loss_vector().double().cpu()
    for _ in range(3):
        fwd(); bwd()
    ms_step2, ms_fwd, ms_bwd, _ = timed(two_kernel_step, args.steps)
    total_mpix = GLOBAL_B * H * W / 1e6
    value = total_mpix / (ms_step * 1e-3)

    # ---- output checks on the timed path (a fast kernel with wrong results is not done) -----------------------------------
    torch.cuda.synchronize()
    ref_blk = out[:4].cpu()
    gscale = dF.abs().max().item()
    checks = {'single_pass_vs_two_kernel_grad_maxnorm': (grad_modules - dF).abs().max().item() / gscale,
              'single_pass_vs_two_kernel_loss_rel': max(abs(vec[k].item() - ref_blk[k].item()) / abs(ref_blk[k].item()) for k in range(3))
              if world == 1 else None}
    assert checks['single_pass_vs_two_kernel_grad_maxnorm'] <= 2e-6, checks
    del grad_modules
    if rank == 0:
        checks.update(crop_parity_check(dev, ML, a, b, f))

    # ---- roofline of the dominant kernel (single-pass loss+gradient: 16 algorithmic bytes per pixel) ----
    peak, peak_src = measured_peak()
    local_pix = B * H * W
    gbs = lambda bpp, ms: bpp * local_pix / (ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, 'profiles', 'traffic.json')) as fh:
            tj = json.load(fh)
        ent = tj.get('fusion_loss_ws_kernel<FAST,ZMODE>') or tj['fusion_loss_bwd_kernel<FAST,ZMODE>']
        traffic = ent['dram_bytes_per_pixel'] * local_pix
        traffic_src = 'stored constant: ncu --set full dram__bytes_read.sum + dram__bytes_write.sum of this kernel (%s), per pixel x the pixels of one launch; not measured in this run' % ent.get('capture', 'profiles/traffic.json')
    except Exception:
        pass
    roofline = {'bound': 'hbm', 'kernel': 'fusion_loss_ws_kernel<11, FAST=1, ZMODE=2> (warp-specialised: the three loss values + dIf, one launch) as launched by core.loss.SSIMLoss',
                'achieved': gbs(ALG_BYTES_BWD, ms_z), 'peak': peak, 'unit': 'GB/s', 'frac': gbs(ALG_BYTES_BWD, ms_z) / peak,
                'traffic': traffic, 'traffic_source': traffic_src, 'peak_source': peak_src, 'algorithmic_bytes_per_pixel': ALG_BYTES_BWD,
                'ms_per_launch': ms_z,
                'note': 'FP32-FMA-pipe bound, not HBM bound (DESIGN.md section 4): 264 FMA/px of exact-fp32 separable blurs alone cap the '
                        'kernel at 27% of the HBM roof; see roofline_fp32 for the roof that binds'}
    # secondary roof, the one that binds: ALGORITHMIC fp32 FMAs (12 blurred maps x 2 passes x 11 taps = 264 FMA/px, the
    # irreducible part; epilogue / Sobel / products excluded) against the measured packed-FMA issue rate of B200
    # (tools/microbench/pipes.cu, profiles/pipes_r1.txt: 58.4 FFMA2/clk/SM = 116.8 FMA/clk/SM at 1965 MHz x 148 SMs)
    fma_peak = 116.8 * 148 * 1.965e9 / 1e12
    fma_ach = 264.0 * local_pix / (ms_z * 1e-3) / 1e12
    roofline_fp32 = {'bound': 'fp32 FMA pipe', 'achieved': fma_ach, 'peak': fma_peak, 'unit': 'TFMA/s', 'frac': fma_ach / fma_peak,
                     'algorithmic_fma_per_pixel': 264, 'peak_source': 'measured FFMA2 issue rate (profiles/pipes_r1.txt)'}
    two_kernel = {'value': total_mpix / (ms_step2 * 1e-3), 'unit': UNIT, 'ms_per_step': ms_step2,
                  'fwd': {'kernel': 'moment_fwd_kernel<11,EPI_SSIM>', 'ms_per_launch': ms_fwd, 'achieved': gbs(ALG_BYTES_FWD, ms_fwd),
                          'frac': gbs(ALG_BYTES_FWD, ms_fwd) / peak, 'algorithmic_bytes_per_pixel': ALG_BYTES_FWD},
                  'bwd': {'kernel': 'fusion_loss_ws_kernel<FAST=1,ZMODE=0>', 'ms_per_launch': ms_bwd, 'achieved': gbs(ALG_BYTES_BWD, ms_bwd),
                          'frac': gbs(ALG_BYTES_BWD, ms_bwd) / peak, 'algorithmic_bytes_per_pixel': ALG_BYTES_BWD},
                  'combined_28B': {'achieved': gbs(ALG_BYTES_FWD + ALG_BYTES_BWD, ms_fwd + ms_bwd),
                                   'frac': gbs(ALG_BYTES_FWD + ALG_BYTES_BWD, ms_fwd + ms_bwd) / peak},
                  'note': 'C-ABI calls (mmif_fusion_loss_fwd without want_grad, then mmif_fusion_loss_bwd): what backward costs when the '
                          'upstream gradients differ or a graph is retained; not the path the timed step takes'}

    result = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
        'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic',
        'config': {'workload': WORKLOAD, 'per_rank_batch': B, 'parallelism': f'batch sharded over {world} rank(s)',
                   'path': 'core.loss.SSIMLoss + PixelLoss + GradLoss on device-resident tensors, total.backward() (train.py:64-71): '
                           'ONE single-pass launch (loss + gradient) + the in-place rescale; launch counters asserted in-run',
                   'l2': 'inputs larger than L2 (per-rank tensors %.0f MB each)' % (B * H * W * 4 / 1e6),
                   'collective': 'one 16-byte all-reduce (AVG) in place on the kernel\'s loss vector per step' if world > 1 else 'none'},
        'roofline': roofline, 'roofline_fp32': roofline_fp32, 'ms_after_kernel': ms_rest, 'two_kernel': two_kernel, 'clocks': clocks,
        'checks': checks, 'gpu_launches': L.kernel_launches(c0, c1), 'launch_counts': launches,
    }

    if not args.no_extras:
        result['e2e'] = e2e_leg(args, dev, world, rank, ML, B)
        result['train_step_c2'] = train_step_leg(dev, world, rank, ML)
        sharded = metric_suite_sharded_leg(dev, world, rank, MM) if world > 1 else None
        if rank == 0:
            result['torch_cuda_eager'] = torch_eager_leg(dev, ML, value)
            result['metric_suite'] = metric_suite_leg(dev, MM, world)
            if sharded is not None:
                result['metric_suite']['sharded_by_pair'] = sharded
        if world == 1:
            result['cpu_baseline'] = cpu_baseline_leg()
    else:
        result['e2e'] = None
    if world > 1:
        dist.barrier()
    if rank == 0:
        print(json.dumps(result))
    if world > 1:
        dist.destroy_process_group()


DUMP_SAMPLE, DUMP_SEED, DUMP_CORNER = 1 << 22, 0, 512


def dump_outputs(out_dir, grad, losses):
    """What the last timed step handed its caller (rank 0's shard when N > 1), as float32 .npy files in `out_dir`:
    loss.npy      [ssim, pixel, grad, total]: the three module outputs and their sum;
    grad.npy      d(total)/d imgf at DUMP_SAMPLE flat indices drawn with numpy's default_rng(DUMP_SEED), sorted and
                  de-duplicated (the whole gradient is 3.2 GB);
    grad_corners.npy  the top-left DUMP_CORNER^2 block of the first image and the bottom-right one of the last, where the
                  Sobel term's reflect padding and the SSIM window's valid region end.
    The inputs come from a seeded generator, so two builds run with the same arguments can be compared file by file."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    flat = grad.reshape(-1)
    idx = np.unique(np.random.default_rng(DUMP_SEED).integers(0, flat.numel(), DUMP_SAMPLE))
    c = DUMP_CORNER
    arrays = {'loss': torch.stack([t.detach() for t in losses]),
              'grad': flat[torch.from_numpy(idx).to(flat.device)],
              'grad_corners': torch.stack([grad[0, 0, :c, :c], grad[-1, 0, -c:, -c:]])}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), t.float().cpu().numpy())


def crop_parity_check(dev, ML, a, b, f):
    """Parity of the timed path on a crop of the timed tensors: sample 0, rows/cols 0..383 x 0..511 of the bench inputs
    through the same modules, against the fp64 oracle on the host (gates of tests/gates.py)."""
    from oracle import fusion_loss as OL
    ca, cb, cf = (t[:1, :, :384, :512].contiguous() for t in (a, b, f))
    y = cf.clone().requires_grad_(True)
    l1 = ML.SSIMLoss('ssim', weight=1.0)(ca, cb, y)
    l2 = ML.PixelLoss('l1', weight=0.01)(ca, cb, y, mode='max')
    l3 = ML.GradLoss('l1', weight=0.1)(ca, cb, y, mode='max')
    (l1 + l2 + l3).backward()
    (r1, r2, r3), g64 = OL.train_objective_grad(ca.cpu().double(), cb.cpu().double(), cf.cpu().double())
    rel = [abs(x.item() - r.item()) / abs(r.item()) for x, r in zip((l1, l2, l3), (r1, r2, r3))]
    diff = (y.grad.cpu().double() - g64).abs() / g64.abs().max().item()
    frac = (diff > 1e-5).double().mean().item()          # L1 sign ties (SURVEY 8(c)) are counted, not hidden: <= 1e-4 of the elements
    assert max(rel) <= 1e-5 and frac <= 1e-4, (rel, frac)
    return {'crop_1x384x512_loss_rel_vs_fp64_oracle': max(rel), 'crop_1x384x512_grad_frac_beyond_1e-5_vs_fp64_oracle': frac,
            'crop_1x384x512_grad_median_rel_err': diff.median().item()}


def e2e_leg(args, dev, world, rank, ML, B):
    """Same metric through the public drop-in modules with HOST buffers, as a training step sees them (train.py:57-71):
    every step copies the rank's shard of the SOURCES I1 / I2 from pinned host memory (chunked, double-buffered against
    the compute) — float32 as the reference's DataLoader delivers them, and, second figure, uint8 widened to
    float32 / 255 on the device (core.loss.ingest_u8, bit-identical to the host-side scaling) — while imgf is where
    train.py:63 leaves it, on the device (it is the network's output); runs SSIMLoss + PixelLoss + GradLoss forward and
    backward per chunk and reads the loss back."""
    import torch.distributed as dist
    chunk = 8 if B % 8 == 0 else B
    nchunk = B // chunk
    steps = max(1, min(args.steps, 3))
    g = torch.Generator(device=dev).manual_seed(99 + rank)
    imgf = torch.rand(B, 1, H, W, device=dev, generator=g)
    fn1, fn2, fn3 = ML.SSIMLoss('ssim', weight=1.0), ML.PixelLoss('l1', weight=0.01), ML.GradLoss('l1', weight=0.1)
    copy_stream = torch.cuda.Stream(device=dev)
    comp = torch.cuda.current_stream(dev)
    loss_host = torch.empty(1, pin_memory=True)
    out = {}
    for tag, dtype in (('f32', torch.float32), ('u8', torch.uint8)):
        host = [torch.empty(B, 1, H, W, dtype=dtype, pin_memory=True) for _ in range(2)]
        for t in host:
            if dtype == torch.uint8:
                t.random_(0, 256)
            else:
                t.uniform_(0, 1)
        stage = [[torch.empty(chunk, 1, H, W, dtype=dtype, device=dev) for _ in range(2)] for _ in range(2)]
        wide = [[torch.empty(chunk, 1, H, W, device=dev) for _ in range(2)] for _ in range(2)] if dtype == torch.uint8 else stage
        ready = [torch.cuda.Event() for _ in range(2)]
        free = [torch.cuda.Event() for _ in range(2)]

        def step():
            acc = torch.zeros((), device=dev)
            for c in range(nchunk):
                s = c & 1
                with torch.cuda.stream(copy_stream):
                    copy_stream.wait_event(free[s])
                    for k in range(2):
                        stage[s][k].copy_(host[k][c * chunk:(c + 1) * chunk], non_blocking=True)
                    ready[s].record(copy_stream)
                comp.wait_event(ready[s])
                if dtype == torch.uint8:
                    for k in range(2):
                        ML.ingest_u8(stage[s][k], out=wide[s][k])
                x1, x2 = wide[s][0], wide[s][1]
                y = imgf[c * chunk:(c + 1) * chunk].detach().requires_grad_(True)
                tot = (fn1(x1, x2, y) + fn2(x1, x2, y, mode='max') + fn3(x1, x2, y, mode='max')) / nchunk
                tot.backward()
                acc = acc + tot.detach()
                free[s].record(comp)
            loss_host.copy_(acc.reshape(1), non_blocking=True)
            torch.cuda.synchronize()
            return loss_host.item()

        for s_ in range(2):
            free[s_].record(comp)
        step()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        torch.cuda.synchronize()
        dt = torch.tensor([(time.perf_counter() - t0) / steps], device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        out[tag] = (GLOBAL_B * H * W / 1e6 / dt.item(), 2 * GLOBAL_B * H * W * host[0].element_size())
        del host, stage, wide
    return {'value': out['f32'][0], 'unit': UNIT, 'h2d_bytes_per_step': out['f32'][1], 'd2h_bytes_per_step': 4 * world, 'steps': steps,
            'gpu_launches_per_step': 2 * nchunk * world,
            'api': 'core.loss.SSIMLoss/PixelLoss/GradLoss + backward; sources I1, I2 float32 from pinned host memory every step (chunks of %d), '
                   'imgf device-resident as train.py:63 produces it' % chunk,
            'u8_sources': {'value': out['u8'][0], 'unit': UNIT, 'h2d_bytes_per_step': out['u8'][1],
                           'api': 'the same with 8-bit sources widened to float32 / 255 on the device (core.loss.ingest_u8)'}}


# ------------------------------------------------------------------------ library baselines (torch CUDA eager)
def eager_objective(x1, x2, f, w_ssim=1.0, w_pixel=0.01, w_grad=0.1):
    """What train.py runs on the GPU today (train.py:64-69,302-317 through core/loss.py:42-110,240-344): the same three
    terms as ~250 stock torch CUDA kernels (depthwise conv2d blurs, reflect pads, elementwise, reductions).  Written
    out here as the LIBRARY baseline of the path (SURVEY.md 8(d)); it is not the product and not the parity checker."""
    import math
    import torch.nn.functional as F
    t = torch.tensor([math.exp(-(i - 5) ** 2 / (2.0 * 1.5 ** 2)) for i in range(11)], dtype=torch.float32)
    t = (t / t.sum()).unsqueeze(1)
    win = torch.mm(t, t.t())[None, None].to(f)
    c1, c2 = 0.01 ** 2, 0.03 ** 2

    def blur(u):
        return F.conv2d(u, win, groups=1)

    def ssim_mean(x, y):
        mx, my = blur(x), blur(y)
        mxx, myy, mxy = mx * mx, my * my, mx * my
        vx = (blur(x * x) - mxx).clamp(min=0)
        vy = (blur(y * y) - myy).clamp(min=0)
        cov = blur(x * y) - mxy
        m = ((2.0 * mxy + c1) * (2.0 * cov + c2)) / ((mxx + myy + c1) * (vx + vy + c2))
        return m.mean(dim=(1, 2, 3)).mean()

    kx = torch.tensor([[-1., 0., 1.], [-2., 0., 2.], [-1., 0., 1.]]).reshape(1, 1, 3, 3).to(f)
    ky = torch.tensor([[-1., -2., -1.], [0., 0., 0.], [1., 2., 1.]]).reshape(1, 1, 3, 3).to(f)

    def sobel(u):
        q = F.pad(u, (1, 1, 1, 1), 'reflect')
        return torch.abs(F.conv2d(q, kx)) + torch.abs(F.conv2d(q, ky))

    l1 = w_ssim * (1.0 - 0.5 * (ssim_mean(x1, f) + ssim_mean(x2, f)))
    l2 = w_pixel * torch.abs(f - torch.max(x1, x2)).mean()
    l3 = w_grad * torch.abs(sobel(f) - torch.max(sobel(x1), sobel(x2))).mean()
    return l1, l2, l3


def _cuda_time(fn, iters, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def torch_eager_leg(dev, ML, our_value):
    """The library baseline on the same B200: torch CUDA eager loss fwd+bwd (what train.py does now) on a bounded sample
    of the workload (2 of the 64 pairs: the eager graph keeps ~600 B/pixel of intermediates), next to the drop-in
    modules on the same tensors; and the small-image latency case BASELINE configs[0] (one 1224x1024 pair)."""
    out = {}
    fn1, fn2, fn3 = ML.SSIMLoss('ssim', weight=1.0), ML.PixelLoss('l1', weight=0.01), ML.GradLoss('l1', weight=0.1)
    for name, (b, h, w), iters in (('2x3072x4096', (2, H, W), 3), ('1x1024x1224', (1, 1024, 1224), 20)):
        g = torch.Generator(device=dev).manual_seed(5)
        x1, x2, y = (torch.rand(b, 1, h, w, device=dev, generator=g) for _ in range(3))

        def eager():
            f = y.detach().requires_grad_(True)
            l1, l2, l3 = eager_objective(x1, x2, f)
            (l1 + l2 + l3).backward()
            return f.grad

        def ours():
            f = y.detach().requires_grad_(True)
            (fn1(x1, x2, f) + fn2(x1, x2, f, mode='max') + fn3(x1, x2, f, mode='max')).backward()
            return f.grad

        go, ge = ours(), eager()            # torch's default lets cuDNN run these fp32 convolutions in TF32 (what train.py gets)
        err_tf32 = ((ge - go).abs().max() / ge.abs().max()).item()
        keep = torch.backends.cudnn.allow_tf32
        torch.backends.cudnn.allow_tf32 = False
        ge = eager()
        err = ((ge - go).abs().max() / ge.abs().max()).item()
        ms_e32 = _cuda_time(eager, iters)
        torch.backends.cudnn.allow_tf32 = keep
        ms_e, ms_o = _cuda_time(eager, iters), _cuda_time(ours, iters)
        del ge, go
        torch.cuda.empty_cache()
        mp = b * h * w / 1e6
        out[name] = {'torch_eager_mpix_per_s': mp / (ms_e * 1e-3), 'torch_eager_ms': ms_e, 'dropin_modules_mpix_per_s': mp / (ms_o * 1e-3),
                     'dropin_modules_ms': ms_o, 'speedup': ms_e / ms_o, 'torch_eager_ms_tf32_off': ms_e32,
                     'grad_maxnorm_diff_vs_eager_tf32_default': err_tf32, 'grad_maxnorm_diff_vs_eager_tf32_off': err}
    out['note'] = ('torch eager = stock torch CUDA kernels of the same objective (library baseline, SURVEY 8(d)); drop-in = '
                   'core.loss modules + backward() incl. their Python/ctypes overhead; headline value (device-resident C-ABI) %.0f Mpix/s' % our_value)
    return out


class _FusionNetStandIn(torch.nn.Module):
    """A DenseFuse-SHAPED encoder / dense block / decoder (1 -> 16 -> 64 channels, 3x3 convolutions, four decoder
    convolutions, last one linear) written for this benchmark only: the reference's models stay the reference's
    (out of scope, /root/reference is not on the GPU box); what matters here is a network of the same size and
    activation footprint in front of the loss, so that the step-time share of the loss is realistic."""

    def __init__(self):
        super().__init__()
        C = torch.nn.Conv2d
        self.stem = C(1, 16, 3, padding=1, padding_mode='reflect')
        self.dense = torch.nn.ModuleList([C(16 * (k + 1), 16, 3, padding=1, padding_mode='reflect') for k in range(3)])
        self.dec = torch.nn.ModuleList([C(64, 64, 3, padding=1, padding_mode='reflect'), C(64, 32, 3, padding=1, padding_mode='reflect'),
                                        C(32, 16, 3, padding=1, padding_mode='reflect'), C(16, 1, 3, padding=1, padding_mode='reflect')])

    def encode(self, x):
        x = torch.relu(self.stem(x))
        for conv in self.dense:
            x = torch.cat([x, torch.relu(conv(x))], dim=1)
        return x

    def forward(self, x1, x2):
        z = 0.5 * (self.encode(x1) + self.encode(x2))
        for k, conv in enumerate(self.dec):
            z = conv(z)
            if k < 3:
                z = torch.relu(z)
        return z


def train_step_leg(dev, world, rank, ML):
    """BASELINE configs[1] (SURVEY 8(d) C2): one training step on 256x256 patches, per-rank batch 8 (global 64 at 8
    GPUs), DDP when world > 1, Adam 1e-4, grad-norm clip 5 (train.py:64-71), with the torch-eager loss and with the
    drop-in loss modules; plus the loss-only (forward + backward to imgf) time of each.  Max over ranks."""
    import torch.distributed as dist
    torch.manual_seed(0)
    try:            # the reference's own DenseFuse (core/model.py:165-187) from the byte-compiled artefact oracle/_ref
        from oracle import build_ref
        net = build_ref.load()[2].DenseFuse().to(dev)
        net_name = "the reference's DenseFuse (core/model.py:165-187, oracle/_ref)"
    except ImportError:
        net = _FusionNetStandIn().to(dev)
        net_name = 'DenseFuse-shaped stand-in network (oracle/_ref not built)'
    model = torch.nn.parallel.DistributedDataParallel(net, device_ids=[dev.index]) if world > 1 else net
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)
    g = torch.Generator(device=dev).manual_seed(100 + rank)
    x1, x2 = (torch.rand(8, 1, 256, 256, device=dev, generator=g) for _ in range(2))
    fn1, fn2, fn3 = ML.SSIMLoss('ssim', weight=1.0), ML.PixelLoss('l1', weight=0.01), ML.GradLoss('l1', weight=0.1)

    def loss_ours(f):
        return fn1(x1, x2, f) + fn2(x1, x2, f, mode='max') + fn3(x1, x2, f, mode='max')

    def loss_eager(f):
        l1, l2, l3 = eager_objective(x1, x2, f)
        return l1 + l2 + l3

    def make_step(loss_fn):
        def step():
            opt.zero_grad(set_to_none=True)
            loss_fn(model(x1, x2)).backward()
            torch.nn.utils.clip_grad_norm_(model.parameters(), 5.0)
            opt.step()
        return step

    with torch.no_grad():
        f0 = net(x1, x2)

    def make_loss_only(loss_fn):
        def run():
            f = f0.detach().requires_grad_(True)
            loss_fn(f).backward()
        return run

    class _Floor(torch.autograd.Function):
        """PyTorch's own cost of this call pattern: a custom Function with three scalar outputs whose forward / backward do
        nothing but allocate (no kernel of ours) — what remains of loss_only_ms_dropin above this is the drop-in's host code."""

        @staticmethod
        def forward(ctx, f):
            ctx.shape = f.shape
            o = torch.empty(4, device=f.device)
            return o[0], o[1], o[2]

        @staticmethod
        def backward(ctx, g0, g1, g2):
            return torch.empty(ctx.shape, device=g0.device)

    def loss_floor(f):
        l1, l2, l3 = _Floor.apply(f)
        return l1 + l2 + l3

    # the same loss-only step captured once into a CUDA graph and replayed (what a latency-sensitive training loop does at
    # this size: 8 x 256 x 256 is a 40 us kernel under ~150 us of eager-mode host work)
    sf = f0.detach().clone().requires_grad_(True)
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        for _ in range(3):
            sf.grad = None
            loss_ours(sf).backward()
    torch.cuda.current_stream(dev).wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    sf.grad = None
    with torch.cuda.graph(graph):
        loss_ours(sf).backward()

    res = {}
    for key, fn in (('step_ms_torch_eager_loss', make_step(loss_eager)), ('step_ms_dropin_loss', make_step(loss_ours)),
                    ('loss_only_ms_torch_eager', make_loss_only(loss_eager)), ('loss_only_ms_dropin', make_loss_only(loss_ours)),
                    ('loss_only_ms_autograd_floor', make_loss_only(loss_floor)), ('loss_only_ms_dropin_cuda_graph', graph.replay)):
        ms = torch.tensor([_cuda_time(fn, 20, warm=5)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        res[key] = ms.item()
    del graph
    res['config'] = '%s, per-rank batch 8 x 256x256 (global %d), Adam 1e-4, clip 5 (train.py:64-71), %s' % (
        net_name, 8 * world, 'DDP over NCCL' if world > 1 else 'single process')
    res['global_mpix_per_step'] = 8 * world * 65536 / 1e6
    return res


def metric_suite_sharded_leg(dev, world, rank, MM):
    """BASELINE configs[3] / configs[2] over N GPUs (SURVEY 8(e)): pairs i = rank (mod world) on each rank, one launch
    per kernel family per rank, ONE all-gather of the (pairs/rank, 16) float64 rows; images resident in HBM.
    Time per evaluation = max over ranks (device events around K evaluations, barrier on both sides)."""
    import torch.distributed as dist
    out = {}
    for name, (n, h, w) in (('polar_32x1224x1024', (32, 1024, 1224)), ('tno_21x640x480', (21, 480, 640))):
        g = torch.Generator(device=dev).manual_seed(7)              # same pairs on every rank, then this rank's shard
        a = torch.randint(0, 256, (n, 1, h, w), device=dev, generator=g).float()
        b = torch.randint(0, 256, (n, 1, h, w), device=dev, generator=g).float()
        f = torch.floor((a + b) / 2)
        mine = list(range(rank, n, world))
        sa, sb, sf = (t[mine].contiguous() for t in (a, b, f))
        del a, b, f
        per = (n + world - 1) // world
        pad = torch.zeros(per, 16, dtype=torch.float64, device=dev)
        table = torch.empty(world * per, 16, dtype=torch.float64, device=dev)

        def evaluate():
            if mine:
                pad[:len(mine)] = MM.eval_metrics_batch(sa, sb, sf)
            dist.all_gather_into_tensor(table, pad)

        for _ in range(3):
            evaluate()
        iters = 10
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            evaluate()
        e1.record()
        dist.barrier()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1) / iters], device=dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        out[name] = {'pairs_per_s': n / (ms.item() * 1e-3), 'ms_per_evaluation': ms.item(), 'pairs': n, 'pairs_per_rank': per,
                     'collective': 'one all-gather of %d x 16 float64 rows per rank' % per}
    return out


def eval_py_row(MM, a, b, f):
    """The calls eval.py:29-75 makes for one pair, on the drop-in functions (CPU tensors in, python floats out: every
    value is pulled with .item() like eval.py:52-68 does)."""
    m = (MM.calc_mse(a, f) + MM.calc_mse(b, f)) * 0.5
    q, n, l = MM.calc_Qabf(a, b, f, L=1.5, full=True)
    vals = [MM.calc_std(f), MM.calc_ag(f), MM.calc_sf(f), m, MM.calc_psnr(m), (MM.calc_cc(a, f) + MM.calc_cc(b, f)) * 0.5,
            MM.calc_scd(a, b, f), MM.calc_entropy(f), MM.calc_cross_ent(a, f) + MM.calc_cross_ent(b, f),
            MM.calc_mul_info(a, f, normalized=True) + MM.calc_mul_info(b, f, normalized=True), q, n, l,
            (MM.calc_ssim(a, f) + MM.calc_ssim(b, f)) * 0.5, (MM.calc_msssim(a, f) + MM.calc_msssim(b, f)) * 0.5,
            MM.calc_viff(a, b, f, simple=False)]
    return [v.item() for v in vals]


def metric_suite_leg(dev, MM, world=1):
    """Second headline metric: full 16-metric suite, pairs/s (BASELINE configs[2] and configs[3] shapes).
    `pairs_per_s`: images resident in HBM (float32, as the reference's functions take them);
    `e2e_*`: through the public batched entry with HOST buffers, H2D of the images and D2H of the rows inside
    the timed region — float32 host images (what eval.py builds, eval.py:189-194) and uint8 host images
    (what cv2 decodes, eval.py:182-187; widened on the device);
    `cpu_reference_pairs_per_s`: the oracle port of eval.py:29-75 on the host cores, one pair."""
    from oracle import fusion_metric as OM
    out = {}
    peak = measured_peak()[0]
    for name, (n, h, w) in (('tno_21x640x480', (21, 480, 640)), ('polar_32x1224x1024', (32, 1024, 1224))):
        g = torch.Generator(device=dev).manual_seed(7)
        a = torch.randint(0, 256, (n, 1, h, w), device=dev, generator=g).float()
        b = torch.randint(0, 256, (n, 1, h, w), device=dev, generator=g).float()
        f = torch.floor((a + b) / 2)

        def timeit(fn, iters):
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / iters

        ms = timeit(lambda: MM.eval_metrics_batch(a, b, f), 10)
        ms_sub = timeit(lambda: MM.eval_subset_batch(a, b, f), 10) if name.startswith('polar') else None
        # value-distribution check (SURVEY 8(d)): uniform noise is the best case for the shared-memory histogram
        # atomics and the SSIM/VIF branches; smooth 8-bit fields with exactly flat patches are the worst
        import torch.nn.functional as F

        def smooth(seed):
            gg = torch.Generator(device=dev).manual_seed(seed)
            lo = torch.rand(n, 1, h // 32 + 2, w // 32 + 2, device=dev, generator=gg)
            u = F.interpolate(lo, size=(h, w), mode='bicubic', align_corners=False).clamp_(0, 1)
            u = torch.round(u * 255)
            u[:, :, : h // 3, : w // 4] = 17.0
            u[:, :, h // 2:, w // 2:] = torch.round(u[:, :, h // 2:, w // 2:] / 32) * 32
            return u.contiguous()

        na, nb_ = smooth(11), smooth(12)
        nf = torch.floor((na + nb_) / 2)
        ms_nat = timeit(lambda: MM.eval_metrics_batch(na, nb_, nf), 10)
        del na, nb_, nf
        hf = [t.cpu().pin_memory() for t in (a, b, f)]
        hu = [t.to(torch.uint8).cpu().pin_memory() for t in (a, b, f)]
        rows_host = torch.empty(n, 16, dtype=torch.float64).pin_memory()

        def e2e_f32():      # pinned host images in, rows back on the host: upload pipelined against the suite
            rows_host.copy_(MM.eval_metrics_batch_host(*hf), non_blocking=True)
            torch.cuda.synchronize()

        def e2e_u8():
            rows_host.copy_(MM.eval_metrics_batch_host(*hu), non_blocking=True)
            torch.cuda.synchronize()

        ms_f32, ms_u8 = timeit(e2e_f32, 5), timeit(e2e_u8, 5)
        ca, cb, cf_ = (t[:1].cpu() for t in (a, b, f))
        # per-pair latency of the UNMODIFIED eval.py call pattern on the drop-in functions: CPU tensors in (uploaded once
        # per image), ~25 separate calc_* calls, one .item() sync per metric
        eval_py_row(MM, ca, cb, cf_)
        host_pairs = [tuple(t[k % n:k % n + 1].cpu() for t in (a, b, f)) for k in range(1, 6)]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for pa, pb, pf in host_pairs:
            eval_py_row(MM, pa, pb, pf)
        per_pair_ms = (time.perf_counter() - t0) / len(host_pairs) * 1e3
        t0 = time.perf_counter()               # of which: the three host->device copies eval.py's CPU tensors need, as the
        for pa, pb, pf in host_pairs:          # drop-ins do them (pageable memory through a pinned staging ring)
            ups = [MM._staged_upload(t, dev) for t in (pa, pb, pf)]
        torch.cuda.synchronize()
        upload_ms = (time.perf_counter() - t0) / len(host_pairs) * 1e3
        t0 = time.perf_counter()               # and what plain tensor.cuda() from pageable memory would cost
        for pa, pb, pf in host_pairs:
            ups = [t.cuda() for t in (pa, pb, pf)]
        torch.cuda.synchronize()
        upload_plain_ms = (time.perf_counter() - t0) / len(host_pairs) * 1e3
        del ups
        cpu_s = None
        if world == 1:          # under torchrun the other ranks spin on the host cores: a CPU timing there is not a baseline
            torch.set_num_threads(os.cpu_count() or 1)
            try:                # the reference's own core/metric.py (oracle/_ref) when the artefact is present, else the oracle port
                from oracle import build_ref
                RM = build_ref.load()[1]

                def cpu_row():
                    m_ = (RM.calc_mse(ca, cf_) + RM.calc_mse(cb, cf_)) * 0.5
                    RM.calc_Qabf(ca, cb, cf_, L=1.5, full=True)
                    for v_ in (RM.calc_std(cf_), RM.calc_ag(cf_), RM.calc_sf(cf_), RM.calc_psnr(m_), RM.calc_cc(ca, cf_), RM.calc_cc(cb, cf_),
                               RM.calc_scd(ca, cb, cf_), RM.calc_entropy(cf_), RM.calc_cross_ent(ca, cf_), RM.calc_cross_ent(cb, cf_),
                               RM.calc_mul_info(ca, cf_, normalized=True), RM.calc_mul_info(cb, cf_, normalized=True), RM.calc_ssim(ca, cf_),
                               RM.calc_ssim(cb, cf_), RM.calc_msssim(ca, cf_), RM.calc_msssim(cb, cf_), RM.calc_viff(ca, cb, cf_, simple=False)):
                        v_.item()
                cpu_kind = "the reference's own core/metric.py (oracle/_ref), eval.py:29-75 call sequence"
            except ImportError:
                cpu_row = lambda: OM.eval_pair(ca, cb, cf_)
                cpu_kind = 'oracle port of eval.py:29-75'
            t0 = time.perf_counter()
            cpu_row()
            cpu_s = time.perf_counter() - t0
        out[name] = {'pairs_per_s': n / (ms * 1e-3), 'ms_per_batch': ms, 'pairs': n,
                     'pairs_per_s_smooth_flat_images': n / (ms_nat * 1e-3),
                     'hbm_frac_87.6B_per_pixel': 87.6 * n * h * w / (ms * 1e-3) / 1e9 / peak,
                     'e2e_f32_host_pairs_per_s': n / (ms_f32 * 1e-3), 'e2e_u8_host_pairs_per_s': n / (ms_u8 * 1e-3),
                     'h2d_bytes_f32': 12 * n * h * w, 'h2d_bytes_u8': 3 * n * h * w, 'd2h_bytes': n * 16 * 8,
                     'eval_py_call_pattern_ms_per_pair': per_pair_ms, 'eval_py_upload_share_ms_per_pair': upload_ms,
                     'eval_py_upload_plain_cuda_ms_per_pair': upload_plain_ms,
                     'cpu_reference_pairs_per_s': (1.0 / cpu_s) if cpu_s else None, 'cpu_cores': torch.get_num_threads() if cpu_s else None,
                     'cpu_sample': ('1 pair, single run: ' + cpu_kind) if cpu_s else 'not timed under torchrun (N > 1)'}
        if ms_sub is not None:      # BASELINE configs[3]: MS-SSIM + VIFF + Qabf only (51.6 algorithmic B/px, SURVEY 8(d))
            out[name]['configs3_subset_msssim_viff_qabf'] = {
                'pairs_per_s': n / (ms_sub * 1e-3), 'ms_per_batch': ms_sub,
                'hbm_frac_51.6B_per_pixel': 51.6 * n * h * w / (ms_sub * 1e-3) / 1e9 / peak}
    return out


def cpu_baseline_leg():
    """The reference's CPU path on the host cores (rank 0, N = 1): a bounded sample of the workload (one 4096x3072 pair)
    and BASELINE configs[0] as named (one 1224x1024 pair, batch 1, CPU torch: SURVEY 8(d) C1, best of 5 after 1 warm-up)."""
    run, kind, host = reference_objective()
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    g = torch.Generator().manual_seed(0)
    a, b, f = (torch.rand(1, 1, H, W, generator=g) for _ in range(3))
    run(a, b, f)
    best = 1e30
    for _ in range(3):
        t0 = time.perf_counter()
        run(a, b, f)
        best = min(best, time.perf_counter() - t0)
    a, b, f = (torch.rand(1, 1, 1024, 1224, generator=g) for _ in range(3))
    run(a, b, f)
    best0 = 1e30
    for _ in range(5):
        t0 = time.perf_counter()
        run(a, b, f)
        best0 = min(best0, time.perf_counter() - t0)
    return {'value': H * W / 1e6 / best, 'unit': UNIT, 'cores': torch.get_num_threads(), 'kind': kind, 'host': host,
            'sample': '1 of 64 pairs (one 4096x3072 pair, fwd+bwd), best of 3 after 1 warm-up',
            'configs0_1x1024x1224': {'ms': best0 * 1e3, 'mpix_per_s': 1024 * 1224 / 1e6 / best0,
                                     'sample': 'BASELINE configs[0]: one 1224x1024 pair, batch 1, loss fwd+bwd, best of 5 after 1 warm-up'}}


if __name__ == '__main__':
    main()
