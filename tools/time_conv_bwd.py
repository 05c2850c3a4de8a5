"""Per-call time of riqn_conv_bwd_strip (ReLU mask + bias sums, data gradient, weight gradient) for conv2 and conv3 at the
learner's batch, CUDA events around a graph of back-to-back calls.  The working set (< 40 MB) stays in L2 between calls,
as it largely does inside a learner step.  `--no-din` times the call without the data gradient (conv1's form).

    python tools/time_conv_bwd.py [--batch 512] [--reps 200]
"""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rainbow_iqn_apex_b200._lib import ConvGeom, call, ptr  # noqa: E402
from rainbow_iqn_apex_b200.model import _strip_perm  # noqa: E402

LAYERS = {"conv2": (32, 20, 64, 4, 2), "conv3": (64, 9, 64, 3, 1)}   # (Cin, H, Cout, k, stride), pad 0


def time_layer(name, batch, reps, with_din):
    dev = torch.device("cuda")
    cin, h, cout, k, s = LAYERS[name]
    oh = (h - k) // s + 1
    G, K = oh + k // s - 1, cin * k * k
    geom = ConvGeom(batch, cin, h, h, cout, k, k, s, 0, oh, oh, cin * h * h)
    dout = torch.randn(batch, cout, oh, oh, device=dev)
    out = torch.randn(batch, cout, oh, oh, device=dev)
    a_hi = torch.randn(batch * G * G, s * s * cin, device=dev).to(torch.bfloat16)
    w_hi = (torch.randn(cout, K, device=dev) / K ** 0.5).to(torch.bfloat16)
    perm = _strip_perm(cin, k, s, False).to(torch.int32).to(dev)
    dYg = torch.empty(batch * G * G, cout, dtype=torch.bfloat16, device=dev)
    dwp, dw, db = torch.empty(cout, K, device=dev), torch.zeros(cout, K, device=dev), torch.zeros(cout, device=dev)
    din = torch.empty(batch, cin, h, h, device=dev) if with_din else None
    go = lambda: call("riqn_conv_bwd_strip", geom, ptr(dout), ptr(out), ptr(a_hi), ptr(w_hi), ptr(perm), ptr(dYg), ptr(dwp),
                      ptr(dw), ptr(db), ptr(din), 1.0)
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        for _ in range(5):
            go()
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for _ in range(reps):
                go()
    torch.cuda.synchronize()
    graph.replay()
    torch.cuda.synchronize()
    best = []
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        graph.replay()
        e1.record()
        torch.cuda.synchronize()
        best.append(e0.elapsed_time(e1) * 1e3 / reps)
    best.sort()
    print(f"riqn_conv_bwd_strip {name} B={batch}{'' if with_din else ' (no din)'}: median {best[2]:7.2f} us/call "
          f"(min {best[0]:.2f}, max {best[-1]:.2f}; 5 graphs of {reps} calls)")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--no-din", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("no CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    print("device:", q.stdout.strip() or torch.cuda.get_device_name(0))
    for name in LAYERS:
        time_layer(name, args.batch, args.reps, not args.no_din)


if __name__ == "__main__":
    main()
