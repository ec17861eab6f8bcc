"""Cost of the window-based quality indices (Q, Q_W, Q_E, Q_Y).

Times one mmif_quality_index launch with device events after a warm-up, on uint8-valued images, and reports the kernel
time and its share of the 12 B/pixel HBM roof (a, b and f read once) against 6463.3 GB/s, the device-to-device copy
rate measured on this GPU model.  Next to it: the float32 oracle (oracle/quality_index.py) on the host, per pair, which
is what a CPU evaluation script of these indices costs.  The card name and power limit are read in the same run.

    python tools/quality_index_time.py [--reps 20] [--shapes 32x1024x1224,21x480x640] [--oracle-pairs 2]
"""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import mmif_b200  # noqa: E402,F401
from mmif_b200 import _lib as L  # noqa: E402
from oracle import quality_index as QI  # noqa: E402

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
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--shapes', default='32x1024x1224,21x480x640')
    ap.add_argument('--oracle-pairs', type=int, default=2, help='pairs timed on the host with the float32 oracle (0: skip)')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('quality_index_time.py needs a CUDA device')
    lib = L.load()
    dev = torch.device('cuda:0')
    print('card:', card())
    g = torch.Generator(device=dev).manual_seed(0)
    for spec in args.shapes.split(','):
        n, h, w = (int(x) for x in spec.split('x'))
        a, b, f = (torch.randint(0, 256, (n, h, w), generator=g, device=dev).float() for _ in range(3))
        nbytes = lib.mmif_quality_index_workspace_bytes(n, h, w)
        ws = torch.zeros(nbytes, dtype=torch.uint8, device=dev)
        out = torch.empty(n * L.QIDX_DOUBLES, dtype=torch.float64, device=dev)

        def run():
            L.check(lib.mmif_quality_index(a.data_ptr(), b.data_ptr(), f.data_ptr(), n, h, w, out.data_ptr(), ws.data_ptr(),
                                           nbytes, L.stream_int(dev)))
        ms = time_ms(run, args.reps)
        traffic = 12.0 * n * h * w
        gbs = traffic / ms / 1e6
        line = (f'mmif_quality_index {spec}: {ms:.4f} ms  ({ms / n:.4f} ms per pair)  {gbs:.1f} GB/s = '
                f'{100.0 * gbs / PEAK_GBS:.1f} % of the 12 B/pixel roof at {PEAK_GBS} GB/s')
        if args.oracle_pairs > 0:
            k = min(args.oracle_pairs, n)
            ha, hb, hf = (x[:k].unsqueeze(1).cpu() for x in (a, b, f))
            t0 = time.perf_counter()
            for i in range(k):
                QI.quality_indices(ha[i:i + 1], hb[i:i + 1], hf[i:i + 1])
            host = (time.perf_counter() - t0) / k * 1e3
            line += f'; float32 oracle on the host: {host:.1f} ms per pair ({torch.get_num_threads()} threads)'
        print(line)
        del a, b, f, ws, out
        torch.cuda.empty_cache()


if __name__ == '__main__':
    main()
