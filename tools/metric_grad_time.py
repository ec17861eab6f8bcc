"""Cost of the metric gradients.

Times mmif_stats_bwd alone with device events, with every statistics column active (mean, sd, ag, sf, both mse, both cc,
scd: the AG and SF stencil terms included), once with df only and once with da, db and df requested.  The kernel reads
a, b and f (12 B/pixel) and writes 4 B/pixel per requested gradient; the rate is reported against that traffic and
against 6463.3 GB/s, the device-to-device copy rate measured on this GPU model.  Shapes whose working set fits the
126 MB L2 are read from there after the first pass; the largest shape (8x3072x4096, 2.4 GB) is not.
Then times calc_ssim(a, f) forward + backward at 1x1024x1224 (fresh tensor objects per step, so the metric memo
recomputes the forward every time).

    python tools/metric_grad_time.py [--reps 50] [--shapes 21x480x640,1x1024x1224,8x3072x4096]
"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import mmif_b200  # noqa: E402,F401
from mmif_b200 import _lib as L  # noqa: E402
from mmif_b200.core import metric as MM  # noqa: E402

PEAK_GBS = 6463.3


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.sm,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30)
        return q.stdout.strip() or name
    except Exception as exc:  # pragma: no cover - no nvidia-smi on the host
        return f'{name} (power limit unknown: {exc})'


def time_ms(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(reps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=50)
    ap.add_argument('--shapes', default='21x480x640,1x1024x1224,8x3072x4096')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('metric_grad_time.py needs a CUDA device')
    lib = L.load()
    dev = torch.device('cuda:0')
    print('card:', card())
    g = torch.Generator(device=dev).manual_seed(0)
    for spec in args.shapes.split(','):
        n, h, w = (int(x) for x in spec.split('x'))
        a, b, f = (torch.rand(n, h, w, generator=g, device=dev) * 255.0 for _ in range(3))
        row = MM._dev_rows(MM._stats(a, b, f))
        gout = torch.zeros(L.ST_COUNT, dtype=torch.float32, device=dev)
        gout[:9] = 1.0
        outs = [torch.empty(n, h, w, device=dev) for _ in range(3)]
        for ngrad in (1, 3):
            ptrs = [o.data_ptr() if k >= 3 - ngrad else None for k, o in enumerate(outs)]

            def run():
                L.check(lib.mmif_stats_bwd(a.data_ptr(), b.data_ptr(), f.data_ptr(), n, h, w, row.data_ptr(), gout.data_ptr(),
                                           *ptrs, L.stream_int(dev)))
            ms = time_ms(run, args.reps)
            nbytes = n * h * w * (12 + 4 * ngrad)
            gbs = nbytes / ms / 1e6
            print(f'mmif_stats_bwd {spec} grads={ngrad}: {ms:.4f} ms  {gbs:.1f} GB/s  {100.0 * gbs / PEAK_GBS:.1f} % of {PEAK_GBS} GB/s'
                  f'  (working set {nbytes / 1e6:.0f} MB)')
        del a, b, f, outs
        torch.cuda.empty_cache()

    a, f = (torch.rand(1, 1, 1024, 1224, generator=g, device=dev) * 255.0 for _ in range(2))

    def ssim_step():
        x, y = a.detach().requires_grad_(True), f.detach().requires_grad_(True)
        MM.calc_ssim(x, y).backward()
    fwd = time_ms(lambda: MM.calc_ssim(a.detach(), f.detach()), args.reps)
    both = time_ms(ssim_step, args.reps)
    print(f'calc_ssim 1x1024x1224: forward {fwd:.4f} ms, forward + backward (both images) {both:.4f} ms per call')


if __name__ == '__main__':
    main()
