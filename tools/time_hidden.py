"""Step time and dueling-kernel throughput per hidden width (B=512, N=N'=64, K=32, 18 actions).

For every width: one CUDA-graph learner step (Learner.enable_cuda_graph, synthetic 84x84x4 replay as in bench.py), CUDA
events around blocks of steps, median over blocks; then the three z-layer + dueling entry points alone at R = 32768
rows, CUDA events around a graph of back-to-back calls.  The kernels' inputs rotate over enough buffers (>= 384 MB) that
no call finds its rows in L2.  Bytes per call, counted from the shapes:
  riqn_dueling_fwd       reads h (R, 2*hid) fp32                          4*R*2*hid
  riqn_dueling_bwd       reads h fp32, writes dh (R, 2*hid) fp32          8*R*2*hid
  riqn_dueling_bwd_bf16  reads the bf16 image of h, writes dh_hi bf16     4*R*2*hid   (the learner's default path)
(the z-weights, q, dz and the column sums are < 1 % of that and not counted).

    python tools/time_hidden.py [--widths 256,512,1024] [--steps 20] [--blocks 5] [--reps 50]
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rainbow_iqn_apex_b200 import Learner, ReplayMemory  # noqa: E402
from rainbow_iqn_apex_b200._lib import call, ptr  # noqa: E402

B, ACTIONS, ROWS, CAPACITY = 512, 18, 32768, 200_000
L2_ROTATE_BYTES = 384 << 20


def step_ms(hidden, steps, blocks):
    import bench                                       # the benchmark's argument set and synthetic replay fill
    dev = torch.device("cuda")
    torch.manual_seed(123)
    a = bench.make_args(dev, CAPACITY)
    a.hidden_size = hidden
    learner = Learner(a, ACTIONS, None)
    learner.train()
    mem = ReplayMemory(a, None)
    bench.fill_replay(mem, CAPACITY, dev, 1000)
    learner.enable_cuda_graph(mem)
    for _ in range(5):
        learner.learn_and_update(mem)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    per = []
    for _ in range(blocks):
        e0.record()
        for _ in range(steps):
            _, loss = learner.learn_and_update(mem)
        e1.record()
        torch.cuda.synchronize()
        per.append(e0.elapsed_time(e1) / steps)
    assert torch.isfinite(loss).all()
    del learner, mem
    torch.cuda.empty_cache()
    return float(np.median(per)), min(per), max(per)


def time_graph(go, nbuf, reps):
    """us per call: median of 5 replays of a graph of `reps` calls cycling over nbuf input sets."""
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        for i in range(nbuf):
            go(i)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for i in range(reps):
                go(i % nbuf)
    torch.cuda.synchronize()
    graph.replay()
    torch.cuda.synchronize()
    t = []
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        graph.replay()
        e1.record()
        torch.cuda.synchronize()
        t.append(e0.elapsed_time(e1) * 1e3 / reps)
    return float(np.median(t))


def dueling_us(hidden, reps):
    dev = torch.device("cuda")
    R, W, A = ROWS, 2 * hidden, ACTIONS
    g = torch.Generator(device=dev).manual_seed(hidden)
    nbuf = max(2, -(-L2_ROTATE_BYTES // (4 * R * W)))
    hs = [torch.randn(R, W, device=dev, generator=g).clamp_(min=0) for _ in range(nbuf)]
    hbs = [h.to(torch.bfloat16) for h in hs]
    wz = torch.randn(1 + A, hidden, device=dev, generator=g) * 0.05
    bz = torch.randn(1 + A, device=dev, generator=g)
    q = torch.empty(R, A, device=dev)
    dtheta = torch.randn(R, device=dev, generator=g)
    gscale = torch.rand(B, device=dev, generator=g)
    actions = torch.randint(0, A, (B,), device=dev, generator=g)
    dzs = [torch.empty(R, 32, device=dev) for _ in range(nbuf)]
    dzb = [torch.empty(R, 32, dtype=torch.bfloat16, device=dev) for _ in range(nbuf)]
    cs = torch.empty(W, device=dev)
    out = {}
    out["riqn_dueling_fwd"] = (time_graph(lambda i: call("riqn_dueling_fwd", R, B, hidden, A, ptr(hs[i]), ptr(wz), ptr(bz),
                                                         ptr(q)), nbuf, reps), 4.0 * R * W)
    dh = [torch.empty(R, W, device=dev) for _ in range(nbuf)]
    out["riqn_dueling_bwd"] = (time_graph(lambda i: call("riqn_dueling_bwd", R, B, hidden, A, ptr(hs[i]), ptr(wz), ptr(dtheta),
                                                         ptr(gscale), 1.0 / B, ptr(actions), ptr(dh[i]), ptr(dzs[i]),
                                                         ptr(dzb[i])), nbuf, reps), 8.0 * R * W)
    del dh
    dhb = [torch.empty(R, W, dtype=torch.bfloat16, device=dev) for _ in range(nbuf)]
    out["riqn_dueling_bwd_bf16"] = (time_graph(lambda i: call("riqn_dueling_bwd_bf16", R, B, hidden, A, ptr(hs[i]), ptr(hbs[i]),
                                                              ptr(wz), ptr(dtheta), ptr(gscale), 1.0 / B, ptr(actions),
                                                              ptr(dhb[i]), None, ptr(cs), ptr(dzs[i]), ptr(dzb[i])),
                                               nbuf, reps), 4.0 * R * W)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--widths", default="256,512,1024")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--reps", type=int, default=50)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("no CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    print("device:", q.stdout.strip() or torch.cuda.get_device_name(0))
    widths = [int(w) for w in args.widths.split(",")]
    for hid in widths:
        med, lo, hi = step_ms(hid, args.steps, args.blocks)
        print(f"hidden {hid:4d}: learner step (CUDA graph) median {med:.3f} ms (min {lo:.3f}, max {hi:.3f}; "
              f"{args.blocks} blocks of {args.steps} steps)")
    for hid in widths:
        for name, (us, nbytes) in dueling_us(hid, args.reps).items():
            print(f"hidden {hid:4d}: {name:22s} R={ROWS}: {us:8.2f} us/call  {nbytes / (us * 1e-6) / 1e9:7.1f} GB/s")
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
