"""Cost of bfloat16 / float16 fused images in the drop-in training objective.

Times the step an autocast training loop runs — SSIMLoss('ssim') + PixelLoss('l1', 'max') + GradLoss('l1', 'max') and
total.backward() — with a float32, bfloat16 and float16 `imgf` (float32 sources, as autocast leaves them), alternating the
three in one process, with device events after a warm-up.  A half-precision step adds one widen launch in front of the
single-pass loss + gradient kernel and one narrow launch behind it (12 B/pixel of HBM traffic: read 2 + write 4, read 4 +
write 2) and drops the float32 step's in-place rescale, which exits at once for a unit upstream gradient.  A separate
torch.profiler run then reports, per dtype, the widen, loss + gradient, rescale and narrow kernel times by name and
the total of every other kernel in the step.

    python tools/precision_step.py [--rounds 5] [--steps 10] [--shapes 8x3072x4096,1x1024x1224]
"""
import argparse
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import mmif_b200  # noqa: E402,F401
from mmif_b200.core import loss as ML  # noqa: E402

L2_BYTES = 126 * 10 ** 6
KERNELS = (('widen', 'widen_kernel'), ('loss + gradient', 'fusion_loss'), ('rescale', 'rescale_unit_kernel'),
           ('narrow', 'narrow_kernel'))
DTYPES = (('fp32', torch.float32), ('bf16', torch.bfloat16), ('fp16', torch.float16))


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30)
        return q.stdout.strip() or name
    except Exception as exc:  # pragma: no cover - no nvidia-smi on the host
        return f'{name} (power limit unknown: {exc})'


def working_set_bytes(B, H, W, dtype):
    """Bytes one step touches: the two float32 sources, imgf, the float32 unit gradient; for a half imgf also its float32
    widening and the narrowed gradient."""
    n = B * H * W
    b = n * (4 + 4 + 4)
    if dtype != torch.float32:
        b += n * (2 + 4 + 2)
    return b


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--shapes', default='8x3072x4096,1x1024x1224')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('precision_step.py needs a CUDA device')
    print('card:', card())
    mods = (ML.SSIMLoss('ssim', weight=1.0), ML.PixelLoss('l1', weight=0.01), ML.GradLoss('l1', weight=0.1))

    def step(a, b, f):
        f.grad = None
        tot = mods[0](a, b, f) + mods[1](a, b, f, mode='max') + mods[2](a, b, f, mode='max')
        tot.backward()

    for shape in args.shapes.split(','):
        B, H, W = (int(v) for v in shape.split('x'))
        g = torch.Generator(device='cuda').manual_seed(B * H + W)
        a, b, f32 = (torch.rand(B, 1, H, W, device='cuda', generator=g) for _ in range(3))
        # detached leaves: otherwise .to(float32) returns f32 itself and the half tensors would backpropagate into it
        fs = {nm: f32.to(dt).detach().requires_grad_(True) for nm, dt in DTYPES}
        for nm, dt in DTYPES:
            ws = working_set_bytes(B, H, W, dt)
            print(f'{B}x{H}x{W} {nm}: working set {ws / 1e6:.0f} MB, {"fits" if ws <= L2_BYTES else "does not fit"} '
                  f'in the 126 MB L2')
        for nm, _ in DTYPES:
            for _ in range(args.warmup):
                step(a, b, fs[nm])
        torch.cuda.synchronize()
        times = {nm: [] for nm, _ in DTYPES}
        for r in range(args.rounds):
            order = DTYPES if r % 2 == 0 else DTYPES[::-1]
            for nm, _ in order:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.steps):
                    step(a, b, fs[nm])
                e1.record()
                e1.synchronize()
                times[nm].append(e0.elapsed_time(e1) / args.steps)
        base = statistics.median(times['fp32'])
        for nm, _ in DTYPES:
            med = statistics.median(times[nm])
            print(f'{B}x{H}x{W} {nm}: step {med:.3f} ms median of {args.rounds} rounds x {args.steps} steps '
                  f'(min {min(times[nm]):.3f}, max {max(times[nm]):.3f}); vs fp32 {med - base:+.3f} ms ({(med / base - 1) * 100:+.1f} %)')

        # kernel times from a profiled run of its own (the profiler slows the host, so the step times above are taken without it)
        from torch.profiler import ProfilerActivity, profile
        for nm, _ in DTYPES:
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(args.steps):
                    step(a, b, fs[nm])
                torch.cuda.synchronize()
            named, other = {}, []
            for ev in prof.key_averages():
                total = getattr(ev, 'device_time_total', None)
                if total is None:
                    total = ev.cuda_time_total
                if not ev.count or not total:
                    continue
                label = next((lab for lab, pat in KERNELS if pat in ev.key), None)
                if label is None:
                    other.append((total / args.steps, ev.key))
                else:
                    named[label] = (total / ev.count, ev.count / args.steps)
            for label, _ in KERNELS:
                if label in named:
                    us, per = named[label]
                    print(f'  {B}x{H}x{W} {nm} kernel {label}: {us / 1e3:.3f} ms per launch, {per:g} per step')
            ot = sum(us for us, _ in other)
            big = ', '.join(f'{k[:60]} {us / 1e3:.3f} ms' for us, k in sorted(other, reverse=True)[:3] if us > 5.0)
            print(f'  {B}x{H}x{W} {nm} other kernels: {ot / 1e3:.3f} ms per step' + (f' ({big})' if big else ''))
        del a, b, f32, fs
        torch.cuda.empty_cache()


if __name__ == '__main__':
    main()
