"""CUDA-event timing of the weight-gradient product ops.gemm_planes_mn (split-K launch + reduction), one product per call:
   python scripts/mn_time.py [--fmt f16x2|bf16x3] [--iters N] [--repeats R]
Shapes: the four products of the Envelope update's backward pass over 65,536 pair rows (three 256 x 256 hidden layers, and the
24-wide output layer whose G planes are 64 wide), and one smaller product (5,000 rows, 256 x 256).  At 65,536 rows the operands of one
product (134 MB of f16x2 planes) exceed the 126 MB L2; the small shape runs from L2.  Prints the card and its power limit with the numbers."""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch as th

from morl_baselines_b200 import ops

SHAPES = [  # (label, M, g_cols, ldg, h_cols)
    ("hidden 256x256", 65536, 256, 256, 256),
    ("output 24(ld 64)x256", 65536, 24, 64, 256),
    ("small 5000 rows 256x256", 5000, 256, 256, 256),
]


def card():
    name = th.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "power limit unknown"
    return f"{name}, {q}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--fmt", default="f16x2", choices=["f16x2", "bf16x3"])
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    assert th.cuda.is_available(), "mn_time.py needs a CUDA device"
    fmt = ops.FMT_F16X2 if args.fmt == "f16x2" else ops.FMT_BF16X3
    dev = th.device("cuda:0")
    g = th.Generator(device=dev).manual_seed(0)
    sg = ops.scale_tensor(2.0**20, dev) if fmt == ops.FMT_F16X2 else None
    sh = ops.scale_tensor(2.0, dev) if fmt == ops.FMT_F16X2 else None
    print(f"# {card()}; fmt {args.fmt}; {args.iters} calls per window, median of {args.repeats} windows")
    for label, M, gc, ldg, hc in SHAPES:
        Gp = ops.split_planes(th.randn(M, gc, device=dev, generator=g) * 1e-4, fmt, ldp=ldg, scale=sg)
        Hp = ops.split_planes(th.randn(M, hc, device=dev, generator=g).clamp_min(0), fmt, ldp=hc, scale=sh)
        out = th.empty(gc, hc, device=dev)
        cs = th.empty(gc, device=dev)
        ws = ops.gemm_mn_workspace(M, gc, hc, dev)

        def call():
            ops.gemm_planes_mn(Gp, gc, Hp, hc, out=out, workspace=ws, colsum=cs, g_scale=sg, h_scale=sh)

        for _ in range(20):
            call()
        th.cuda.synchronize()
        times = []
        for _ in range(args.repeats):
            t0, t1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
            t0.record()
            for _ in range(args.iters):
                call()
            t1.record()
            t1.synchronize()
            times.append(t0.elapsed_time(t1) * 1e3 / args.iters)
        times.sort()
        print(f"{label:26s} {times[len(times) // 2]:8.2f} us/call  (min {times[0]:.2f}, max {times[-1]:.2f})")


if __name__ == "__main__":
    main()
