#!/usr/bin/env python
"""Learner hot-path benchmark (BASELINE.json metric: learner grad-steps/sec at batch=512, N=N'=64).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host CPU cores

One "step" = one full `Learner.learn` of BASELINE config 2 on every rank: prioritized sample from the
device-resident replay shard (sum-tree descent + IS weights + 7-frame window gather), three network passes,
fused IQN loss, backward, (gradient all-reduce when N > 1), Adam, priority update of the sampled leaves.
N > 1 is the data-parallel learner of config 5 (512 transitions per GPU, weak scaling).

Timing: W untimed warm-up steps, then ONE region of exactly K timed steps, bracketed by barrier +
torch.cuda.synchronize(), CUDA events on the launching stream, max over ranks (`--blocks R` times R such regions and
reports the median).  The last timed step starts from the seeded network, optimiser and replay state (restored untimed),
and `--dump-outputs DIR` writes what it returned (sampled tree indices and per-transition losses, rank 0) as
DIR/<name>.npy, so two builds run with the same arguments can be compared output for output.  An optional
`--sustained-seconds` leg (clocks sampled) and the end-to-end leg (K steps, pinned host batches, H2D / D2H inside the
timed region) follow.  Inputs are larger than L2: every step draws a fresh prioritized minibatch from a multi-GB replay
shard and streams > 1 GB of activations.  Also in the line: rooflines of the hidden products (tensor), the embedding producer,
the conv trunk and the loss kernel (HBM), the Rainbow-only (C51, configs[2]) leg, and the CPU port timed on the host cores.
`--topology apex` (N >= 2) runs configs[3] instead: 1 learner rank + N-1 actor GPUs with sharded replay.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

METRIC = "learner grad-steps/sec (batch=512, N=N'=64)"
B, N_TAU, N_TAU_P, K_Q, ACTIONS = 512, 64, 64, 32, 18
FEAT, HID = 3136, 512


def make_args(device, capacity, rainbow_only=0):
    return SimpleNamespace(
        multi_step=3, history_length=4, discount=0.99, device=device, batch_size=B, length_actor_buffer=1000,
        model=None, lr=5e-5, adam_eps=3.125e-4, rainbow_only=rainbow_only, atoms=51, V_min=-10.0, V_max=10.0, kappa=1.0,
        num_tau_samples=N_TAU, num_tau_prime_samples=N_TAU_P, num_quantile_samples=K_Q, quantile_embedding_dim=64,
        hidden_size=HID, noisy_std=0.1, disable_cuda=False, nb_actor=1, actor_capacity=capacity, priority_weight=0.4,
        priority_exponent=0.2)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


def ncu_traffic(key="dominant_kernel_dram_bytes_per_launch"):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of a kernel, from the committed `ncu --set full` capture
    (profiles/r02_traffic.json, else round 1's); None if absent."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            return json.load(open(p)).get(key)
    return None


def config_dict(world, capacity):
    """The workload description shared by both arms (the driver compares them key by key)."""
    return {"workload": "configs[1]: 1xB200 learner, synthetic 84x84x4 replay, batch=512/GPU, N=N'=64, K=32, n-step=3",
            "batch_per_gpu": B, "global_batch": B * world, "n_tau": N_TAU, "n_tau_prime": N_TAU_P, "n_quantile": K_Q,
            "replay_capacity_per_gpu": capacity, "parallelism": f"dp{world}" if world > 1 else "single",
            "l2": "inputs larger than L2 (fresh prioritized minibatch from a %.1f GB replay shard each step; "
                  ">1 GB of activations streamed per step)" % (capacity * 7056 / 1e9)}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v == "Active":
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------ our arm
def fill_replay(mem, capacity, device, seed):
    """Synthetic 84x84 uint8 frames + metadata written straight into the shard (setup, not timed)."""
    tr = mem.transitions
    g = torch.Generator(device=device).manual_seed(seed)
    chunk = 1 << 16
    for lo in range(0, capacity, chunk):
        hi = min(capacity, lo + chunk)
        tr.frames[lo:hi] = torch.randint(0, 256, (hi - lo, 7056), dtype=torch.uint8, device=device, generator=g)
    pos = torch.arange(capacity, device=device)
    tr.timestep.copy_((pos % 1000).to(torch.int32))
    tr.nonterminal.copy_(((pos % 1000) != 999).to(torch.uint8))
    tr.action.copy_(torch.randint(0, ACTIONS, (capacity,), device=device, generator=g).to(torch.int32))
    tr.reward.copy_((torch.randint(0, 3, (capacity,), device=device, generator=g) - 1).float())
    for lo in range(0, capacity, 4096):                     # priorities U(0,1)^0.2 through the update kernel
        hi = min(capacity, lo + 4096)
        pri = torch.rand(hi - lo, device=device, generator=g).clamp_(min=1e-3).pow_(0.2)
        tr.update_multiple_value(torch.arange(lo, hi, device=device) + capacity - 1, pri)
    head = int(torch.randint(0, capacity, (1,), generator=torch.Generator().manual_seed(seed)).item())
    tr.index_actor[0] = head
    tr.index_actor_host[0] = head
    tr.is_full_actor[0] = 1


def run_ours(args):
    from rainbow_iqn_apex_b200 import Learner, ReplayMemory, _lib, parallel
    rank, world, local = parallel.init_from_env()
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    _lib.require_device()
    torch.manual_seed(123 + rank)
    a = make_args(dev, args.replay_capacity)
    learner = Learner(a, ACTIONS, None)
    learner.train()
    parallel.make_data_parallel(learner)
    mem = ReplayMemory(a, None)
    fill_replay(mem, args.replay_capacity, dev, 1000 + rank)
    # the device state one step leaves for the next (noise and sampling draws follow the step count), as seeded; it is
    # restored before the last timed step because the gradients' fp32 atomics make trajectories drift apart run to run
    # and prioritized sampling turns that drift into different minibatches
    seeded = (learner.online_net._flat, learner.optimiser._exp_avg, learner.optimiser._exp_avg_sq,
              mem.transitions.tree, mem.transitions.max_priority)
    seeded = [(t, t.clone()) for t in seeded]

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def step():
        return learner.learn_and_update(mem)

    # ---- pass 1 (eager, not the headline): per-entry-point device times for the roofline section
    for _ in range(3):
        step()
    barrier()
    timed_names = ("riqn_gemm_bf16_tc", "riqn_gemm_bf16_tc_mn", "riqn_noisy_linear_fwd", "riqn_iqn_loss_fwd_bwd", "riqn_split_bf16",
                   "riqn_quantile_embed_fwd_tc", "riqn_quantile_embed_bwd_tc", "riqn_conv_fwd_tc", "riqn_conv_bwd_tc",
                   "riqn_conv_fwd_tc_u8", "riqn_conv_fwd_strip", "riqn_conv_bwd_strip", "riqn_s2d_u8", "riqn_im2col_bf16_t", "riqn_dueling_fwd", "riqn_dueling_bwd", "riqn_dueling_bwd_bf16", "riqn_z_wgrad",
                   "riqn_z_wgrad_tc", "riqn_noisy_bias_grad", "riqn_adam_step", "riqn_frame_gather", "riqn_sumtree_sample",
                   "riqn_sumtree_update", "riqn_sumtree_is_weights", "riqn_noisy_compose", "riqn_noisy_reset_net",
                   "riqn_argmax_mean")
    prof_steps = 5
    timers = _lib.time_entry_points(timed_names)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = _lib.launch_count()
    e0.record()
    t_host0 = time.perf_counter()
    for _ in range(prof_steps):
        step()
    host_issue_ms = (time.perf_counter() - t_host0) * 1e3 / prof_steps     # CPU time to enqueue one eager step
    e1.record()
    barrier()
    _lib.time_entry_points(None)
    launches_per_step = (_lib.launch_count() - launches0) // prof_steps
    eager_ms = e0.elapsed_time(e1) / prof_steps

    # ---- pass 2 (headline): the whole step captured once in a CUDA graph and replayed
    if not args.no_graph:
        learner.enable_cuda_graph(mem, capture_collectives=not args.dp_eager_allreduce)
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    clocks = ClockSampler(local)
    clocks.start()
    # `blocks` timed regions of EXACTLY args.steps steps each (barrier + synchronize on both sides, CUDA events on the
    # launching stream, max over ranks); the headline is the MEDIAN block, the spread is reported beside it.  The last
    # step of a region starts from the seeded state, so what it returns is the same in every run with these arguments;
    # the restoring copies lie between two event pairs and are not timed.
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    block_ms = []
    for _ in range(max(1, args.blocks)):
        barrier()
        e0.record()
        for _ in range(args.steps - 1):
            step()
        e1.record()
        for t, t0 in seeded:
            t.copy_(t0)
        e2.record()
        idxs, loss = step()
        e3.record()
        barrier()
        block_ms.append(parallel.allreduce_max(e0.elapsed_time(e1) + e2.elapsed_time(e3), dev))
    launches = launches_per_step * args.steps          # kernels executed in ONE timed region (graph replays them)
    clk = clocks.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"tree_idxs": idxs.cpu().double().numpy(), "loss": loss.cpu().float().numpy()})
    ms = float(np.median(block_ms))
    ms_per_step = ms / args.steps
    value = world * 1000.0 / ms_per_step
    assert torch.isfinite(loss).all()
    # sustained leg: the same step for >= args.sustained_seconds, clocks and power sampled (what a long run delivers)
    sustained = None
    if args.sustained_seconds > 0:
        n_sus = max(args.steps, int(args.sustained_seconds * 1000.0 / ms_per_step))
        sclk = ClockSampler(local)
        sclk.start()
        barrier()
        e0.record()
        for _ in range(n_sus):
            step()
        e1.record()
        barrier()
        sus_ms = parallel.allreduce_max(e0.elapsed_time(e1), dev)
        sustained = {"steps": n_sus, "seconds": sus_ms / 1e3, "ms_per_step": sus_ms / n_sus,
                     "value": world * 1000.0 * n_sus / sus_ms, "unit": "grad-steps/s", "clocks": sclk.stop()}

    # per-entry-point device time from the CUDA events recorded on the launching stream (eager pass)
    per = {}
    for name, evs in timers.items():
        per[name] = dict(ms_total=sum(a_.elapsed_time(b_) for a_, b_, _ in evs), calls=len(evs))
    pk = peaks()
    from rainbow_iqn_apex_b200 import model as _model
    # dominant kernel: the hidden NoisyLinear products.  Algorithmic FLOPs = 2*M*N*K per launch (SURVEY 8d); the
    # split-bf16x3 mode issues 3 MMAs per algorithmic multiply-add, reported as mma_passes.
    def _is_head(a_):
        return min(a_[0], a_[1]) >= 1024 and a_[2] >= 1024
    evs = [e for e in timers["riqn_gemm_bf16_tc"] if _is_head(e[2])]
    # the weight gradient runs through the MN-major entry point (single-bf16 product): mark it as one MMA pass
    evs += [(a_, b_, tuple(g_[:4]) + (None,)) for a_, b_, g_ in timers["riqn_gemm_bf16_tc_mn"] if _is_head(g_)]
    label = "gemm_tc_kernel (tcgen05.mma + TMA; NoisyLinear fwd x3 / dgrad / wgrad, %d launches/step)" % (len(evs) // prof_steps)
    flops = sum(2.0 * a_[0] * a_[1] * a_[2] for _, _, a_ in evs)
    passes = sum((3 if a_[4] else 1) * 2.0 * a_[0] * a_[1] * a_[2] for _, _, a_ in evs) / max(flops, 1.0)
    hms = sum(a_.elapsed_time(b_) for a_, b_, _ in evs)
    head_tf = flops / (hms * 1e-3) / 1e12 if hms > 0 else 0.0
    # denominator: the timed blocks are tens of ms at full clocks -> the BURST cuBLAS figure (VERDICT r1 item 11); the
    # fraction against the seconds-long sustained figure is reported beside it, with the sustained leg's own clocks
    roof = {"kernel": label, "bound": "tensor", "achieved": head_tf, "peak": pk["tf_burst"], "unit": "TFLOP/s",
            "frac": head_tf / pk["tf_burst"], "frac_of_sustained_peak": head_tf / pk["tf_sust"], "traffic": ncu_traffic(),
            "peak_source": pk["src"] + " bf16 burst (cuBLAS best-of-10; fp16 and bf16 share the tensor rate)",
            "share_of_step": hms / (eager_ms * prof_steps), "mma_passes": passes,
            "tensor_pipe_frac": passes * head_tf / pk["tf_burst"], "precision": dict(_model.PRECISION),
            "us_per_launch": hms * 1e3 / max(len(evs), 1), "timed": "CUDA events around each launch, eager pass"}
    # HBM-bound producers (VERDICT r1 missing 6): algorithmic bytes per SURVEY 8d / measured launch time
    ek = timers["riqn_quantile_embed_fwd_tc"]
    emb_bytes = emb_ms = 0.0
    for a_, b_, g_ in ek:
        bsz, nq = g_[0], g_[1]
        images = (1 if g_[13] else 0) + (1 if g_[14] else 0)            # x_hi, x_lo / bf16 image
        emb_bytes += 2.0 * images * nq * bsz * FEAT + 4.0 * nq * bsz + 4.0 * bsz * FEAT + 4.0 * (64 * FEAT + FEAT)
        emb_ms += a_.elapsed_time(b_)
    emb_gbs = emb_bytes / (emb_ms * 1e-3) / 1e9 if emb_ms > 0 else 0.0
    roof_embed = {"kernel": "riqn_quantile_embed_fwd_tc (cos + tcgen05 product + Hadamard epilogue writing the head's operand "
                            "images; 3 launches/step)", "bound": "hbm", "achieved": emb_gbs, "peak": pk["hbm"], "unit": "GB/s",
                  "frac": emb_gbs / pk["hbm"], "traffic": ncu_traffic("embed_kernel_dram_bytes_per_launch"),
                  "algorithmic_bytes_per_step": emb_bytes / prof_steps, "ms_per_step": emb_ms / prof_steps,
                  "formula": "2*images*Nq*B*F + 4*Nq*B + 4*B*F + 4*(E*F+F)  (SURVEY 8d, materialised output)"}
    cv_ms = sum(a_.elapsed_time(b_) for a_, b_, _ in timers["riqn_conv_fwd_strip"]) + \
        sum(a_.elapsed_time(b_) for a_, b_, _ in timers["riqn_s2d_u8"])
    n_trunks = 3 * prof_steps              # three network passes per step (the two no-grad trunks share their launches)
    cv_bytes = n_trunks * (B * 4 * 7056 + 4.0 * B * FEAT)                # uint8 frame stack in, fp32 features out
    cv_gbs = cv_bytes / (cv_ms * 1e-3) / 1e9 if cv_ms > 0 else 0.0
    roof_conv = {"kernel": "conv trunk forward (riqn_s2d_u8 + riqn_conv_fwd_strip: 3 network passes in 6 launches per step)", "bound": "hbm",
                 "achieved": cv_gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": cv_gbs / pk["hbm"], "traffic": None,
                 "algorithmic_bytes_per_step": cv_bytes / prof_steps, "ms_per_step": cv_ms / prof_steps,
                 "formula": "B*4*7056 (uint8 frames) + 4*B*3136 (features) per pass: intermediates are not algorithmic"}
    lk = per["riqn_iqn_loss_fwd_bwd"]
    loss_bytes = 4 * B * (N_TAU + N_TAU_P + N_TAU) + 4 * B * N_TAU + B * (4 + 4 + 8 + 8 + 4)   # SURVEY 8d gathered form
    loss_us = lk["ms_total"] * 1e3 / max(lk["calls"], 1)
    roof_loss = {"kernel": "riqn_iqn_loss_fwd_bwd", "bound": "hbm", "achieved": loss_bytes / (loss_us * 1e-6) / 1e9,
                 "peak": pk["hbm"], "unit": "GB/s", "frac": loss_bytes / (loss_us * 1e-6) / 1e9 / pk["hbm"],
                 "traffic": None, "us_per_launch": loss_us, "algorithmic_bytes": loss_bytes,
                 "note": "0.54 MB per launch: latency-bound at B=512 (SURVEY 8d note)"}
    roof_loss_4096 = loss_kernel_point(dev, 4096, pk) if rank == 0 else None

    # ---- end-to-end through the reference-facing API with HOST buffers (pinned), H2D/D2H inside the timed region
    pool = []
    for _ in range(4):
        smp = mem.sample(B)
        pool.append(tuple(t.contiguous().cpu().pin_memory() for t in smp))
    h2d = sum(t.numel() * t.element_size() for t in pool[0])
    d2h = B * 4
    if not args.no_graph:
        learner.enable_batch_graph(mem, tuple(t.contiguous() for t in mem.sample(B)))

    if not args.no_graph:
        learner.prefetch_host_batch(pool[0])

    def e2e_step(i):
        host = pool[i % len(pool)]
        if not args.no_graph:
            loss = learner.learn_on_host_batch()                   # consumes the prefetched batch: D2D + graph replay
            learner.prefetch_host_batch(pool[(i + 1) % len(pool)])  # H2D of the NEXT batch overlaps this step
        else:
            idxs, st, ac, rt, nx, nt, w = (t.to(dev, non_blocking=True) for t in host)
            loss = learner.learn_on_batch(st, ac, rt, nx, nt, w)
            mem.update_priorities(idxs, loss)
        return loss.cpu()                                          # D2H + sync: the result the caller consumes

    for i in range(3):
        e2e_step(i)
    barrier()
    e0.record()
    for i in range(args.steps):
        e2e_step(i)
    e1.record()
    barrier()
    e2e_ms = parallel.allreduce_max(e0.elapsed_time(e1), dev) / args.steps
    e2e = {"value": world * 1000.0 / e2e_ms, "unit": "grad-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "ms_per_step": e2e_ms}

    out = {
        "metric": METRIC, "value": value, "unit": "grad-steps/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "%s fwd / %s bwd tensor-core products, fp32 accumulate in TMEM; fp32 elsewhere" % (_model.PRECISION["fwd"], _model.PRECISION["bwd"]), "data": "synthetic", "impl": "ours",
        "config": config_dict(world, args.replay_capacity),
        "blocks": {"n": len(block_ms), "steps_per_block": args.steps, "ms": block_ms, "min_ms_per_step": min(block_ms) / args.steps,
                   "max_ms_per_step": max(block_ms) / args.steps, "headline": "median block"},
        "sustained": sustained,
        "dp_allreduce": (None if world == 1 else ("eager, between two graphs" if args.dp_eager_allreduce else
                                                    "captured in the step graph; NoisyLinear bucket overlapped with the backward")),
        "frames_per_s": value * B * 4, "transitions_per_s": value * B,
        "clocks": clk, "e2e": e2e, "gpu_launches": launches, "cuda_graph": not args.no_graph,
        "eager": {"ms_per_step": eager_ms, "host_issue_ms_per_step": host_issue_ms},
        "roofline": roof, "roofline_iqn_loss": roof_loss, "roofline_iqn_loss_b4096": roof_loss_4096,
        "roofline_embed": roof_embed, "roofline_conv": roof_conv,
        "kernel_ms_per_step": {k: v["ms_total"] / prof_steps for k, v in per.items()},
    }
    if rank == 0 and world == 1 and not args.no_c51:
        del learner, mem
        torch.cuda.empty_cache()
        try:
            out["config3_c51"] = c51_leg(dev, args)
        except Exception as exc:                     # reported, never hidden: the headline line must still print
            out["config3_c51"] = {"error": repr(exc)[:300]}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(max_seconds=25.0)
    if rank == 0:
        print(json.dumps(out))
    finish(world)


def dump_outputs(directory, arrays):
    """Write each host array as `directory`/<name>.npy (float32 or float64; tree indices are exact in float64)."""
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(directory, name + ".npy"), a)


def finish(world):
    """End of a run: all ranks meet once more, then leave WITHOUT tearing NCCL down.  destroy_process_group() (and the
    interpreter's own teardown) can block forever when CUDA graphs that captured collectives are still alive (seen on
    2 GPUs in round 2: the result line was out, the process never exited).  A benchmark process has nothing to clean up."""
    sys.stdout.flush()
    sys.stderr.flush()
    if world > 1:
        torch.cuda.synchronize()
        torch.distributed.barrier()
        torch.cuda.synchronize()
        os._exit(0)


def loss_kernel_point(dev, batch, pk):
    """SURVEY 8d option (i): the fused IQN loss kernel at a size where bandwidth means something (B = 4096 = config 5's
    global batch).  Bytes = the FULL-ROW form (the kernel reads whole (N*B, A) q tensors and gathers in-kernel):
    4*A*B*(N + N') [q_on, q_tgt] + 4*B*N [tau] + 4*B*N [dtheta] + B*28.  Four input sets (> L2) are rotated."""
    from rainbow_iqn_apex_b200._lib import call, ptr
    sets = []
    for i in range(4):
        g = torch.Generator(device=dev).manual_seed(50 + i)
        sets.append(dict(q_on=torch.randn(N_TAU * batch, ACTIONS, device=dev, generator=g),
                         q_tg=torch.randn(N_TAU_P * batch, ACTIONS, device=dev, generator=g),
                         tau=torch.rand(N_TAU * batch, 1, device=dev, generator=g),
                         act=torch.randint(0, ACTIONS, (batch,), device=dev, generator=g),
                         ast=torch.randint(0, ACTIONS, (batch,), device=dev, generator=g),
                         ret=torch.randn(batch, device=dev, generator=g), nt=torch.ones(batch, device=dev)))
    loss, dth = torch.empty(batch, device=dev), torch.empty(N_TAU * batch, device=dev)

    def go(s):
        call("riqn_iqn_loss_fwd_bwd", batch, N_TAU, N_TAU_P, ACTIONS, ptr(s["q_on"]), ptr(s["q_tg"]), ptr(s["tau"]), ptr(s["act"]),
             ptr(s["ast"]), ptr(s["ret"]), ptr(s["nt"]), 0.99 ** 3, 1.0, ptr(loss), ptr(dth), None, None)
    for s in sets:
        go(s)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 40
    e0.record()
    for i in range(reps):
        go(sets[i % 4])
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / reps
    nbytes = 4.0 * ACTIONS * batch * (N_TAU + N_TAU_P) + 4.0 * batch * N_TAU * 2 + batch * 28
    gbs = nbytes / (us * 1e-6) / 1e9
    return {"kernel": "riqn_iqn_loss_fwd_bwd", "batch": batch, "bound": "hbm", "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s",
            "frac": gbs / pk["hbm"], "us_per_launch": us, "algorithmic_bytes": nbytes,
            "note": "back-to-back launches (includes launch gaps); full-row bytes, 4 rotating input sets > L2"}


def c51_leg(dev, args):
    """BASELINE configs[2]: Rainbow-only (C51 categorical loss, no IQN) learner step at batch 512 on the same replay path
    (sample -> 3 passes -> projection loss -> backward -> Adam -> priority update), CUDA events over `steps` steps."""
    from rainbow_iqn_apex_b200 import Learner, ReplayMemory
    cap = 1 << 16
    a = make_args(dev, cap, rainbow_only=1)
    a.lr, a.adam_eps = 6.25e-5, 1.5e-4
    learner = Learner(a, ACTIONS, None)
    learner.train()
    mem = ReplayMemory(a, None)
    fill_replay(mem, cap, dev, 77)
    mode = "eager"
    for _ in range(3):
        learner.learn_and_update(mem)
    if not args.no_graph:
        learner.enable_cuda_graph(mem)
        mode = "cuda graph"
        for _ in range(3):
            learner.learn_and_update(mem)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = args.steps
    e0.record()
    for _ in range(n):
        loss = learner.learn_and_update(mem)[1]
    e1.record()
    torch.cuda.synchronize()
    assert torch.isfinite(loss).all()
    ms = e0.elapsed_time(e1) / n
    return {"workload": "configs[2]: 1xB200 Rainbow-only (C51, 51 atoms), batch=512, n-step=3", "ms_per_step": ms,
            "value": 1000.0 / ms, "unit": "grad-steps/s", "steps": n, "mode": mode, "replay_capacity": cap}


def run_apex(args):
    """BASELINE configs[3] (`--topology apex`, N >= 2 ranks): rank 0 = learner (B = 512 per step), every other rank an actor
    GPU that owns a prioritized replay shard (2^19 transitions by default, one segment per environment), steps
    `--actor-envs` synthetic environments with batched greedy actions, computes initial priorities for each
    `--actor-buffer`-step buffer and appends it to its shard.  Per learner step, all ranks in lock step: shard sampling
    on the actor GPUs -> gather to the learner -> learn -> broadcast of the new losses -> priority update on the owning
    shards; parameter broadcast every 100 learner steps.  Reports learner grad-steps/s and actor frames/s."""
    from rainbow_iqn_apex_b200 import Actor, Learner, ReplayMemory, _lib, apex, parallel
    rank, world, local = parallel.init_from_env()
    if world < 2:
        raise SystemExit("--topology apex needs >= 2 ranks (torch.distributed.run --nproc-per-node N)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    _lib.require_device()
    torch.manual_seed(123 + rank)
    topo = apex.ApexTopology(B, publish_every=100)
    E, L = args.actor_envs, args.actor_buffer
    if topo.is_learner:
        agent = Learner(make_args(dev, 1), ACTIONS, None)
        mem = pool = None
    else:
        a = make_args(dev, args.replay_capacity // E)
        a.nb_actor = E
        agent = Actor(a, ACTIONS, None)
        mem = ReplayMemory(a, None)
        fill_replay_segments(mem, dev, 1000 + rank)
        pool = apex.ActorPool(agent, mem, E, L)
        pool.write_index[:] = mem.transitions.index_actor_host          # continue behind the synthetic pre-fill
        g = torch.Generator(device=dev).manual_seed(9000 + rank)
        states = torch.randint(0, 256, (E, 4, 84, 84), dtype=torch.uint8, device=dev, generator=g)
    agent.train()
    parallel.publish_parameters(agent, src=0)                  # everyone starts from the learner's weights
    flushed = [0]
    graphed = [False]
    def step():
        nonlocal states
        # all ranks: ONE gather of the shards' (pre-sampled, packed) parts; the GPUs are otherwise idle at this point, so the
        # collective does not compete with the persistent GEMMs for SMs (a side-stream prefetch under the learner's step
        # measured 7.5 ms/step on 8 GPUs: NCCL's CTAs wait for the 148-CTA kernels to end)
        batch = topo.sample(mem, beta=0.4, device=dev)
        if topo.is_learner:
            _, _, st, ac, rt, nx, nt, w = batch
            if not args.no_graph and not graphed[0]:       # capture learn_on_batch once the first gathered batch fixes the shapes
                agent.enable_learn_graph((st, ac, rt, nx, nt, w))
                graphed[0] = True
            if graphed[0]:
                loss = agent.learn_on_graph((st, ac, rt, nx, nt, w)).detach()
            else:
                loss = agent.learn_on_batch(st, ac, rt, nx, nt, w).detach()
        else:
            loss = torch.empty(B, dtype=torch.float32, device=dev)
            for _ in range(args.acts_per_step):                # acting overlaps the learner's step
                act = pool.act(states)
                nxt = torch.randint(0, 256, (E, 1, 84, 84), dtype=torch.uint8, device=dev, generator=g)
                rew = (torch.randint(0, 3, (E,), device=dev, generator=g) - 1).float()
                done = torch.rand(E, device=dev, generator=g) < 0.01
                if pool.observe(states, act, rew, done):
                    flushed[0] += pool.flush()
                states = torch.cat([states[:, 1:], nxt], 1)
        if not topo.is_learner:
            # the shard's part of the NEXT batch is drawn before this step's losses arrive (one step of priority staleness;
            # the reference's sampler queue holds five batches), so the next all-gather never waits for the actors
            topo.presample(mem)
        topo.route(loss, mem, None if topo.is_learner else batch)
        topo.maybe_publish(agent)

    def barrier():
        torch.distributed.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    clocks = ClockSampler(local)
    clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0 = flushed[0]
    barrier()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    clk = clocks.stop()
    ms = parallel.allreduce_max(e0.elapsed_time(e1), dev)
    appended = parallel.allreduce_sum(float(flushed[0] - f0), dev)
    ms_per_step = ms / args.steps
    env_steps = (world - 1) * E * args.acts_per_step * args.steps
    out = {"metric": "Ape-X topology: learner grad-steps/sec (batch=512, N=N'=64) with %d actor GPUs" % (world - 1),
           "value": 1000.0 / ms_per_step, "unit": "grad-steps/s", "n_gpus": world, "steps": args.steps,
           "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "n/a", "vs_baseline": None,
           "dtype": "fp16 fwd / bf16 bwd tensor-core products", "data": "synthetic", "impl": "ours",
           "config": {"workload": "configs[3]: 1 learner + %d actor GPUs, sharded prioritized replay %d transitions, "
                                  "NCCL parameter broadcast every 100 steps" % (world - 1, (world - 1) * args.replay_capacity),
                      "batch": B, "shard_counts": topo.counts, "replay_capacity_per_shard": args.replay_capacity,
                      "envs_per_actor_gpu": E, "actor_buffer": L, "acts_per_learner_step": args.acts_per_step},
           "actor_env_steps_per_s": env_steps / (ms * 1e-3), "actor_frames_per_s": 4.0 * env_steps / (ms * 1e-3),
           "transitions_appended_in_region": appended, "clocks": clk,
           "exchange_bytes_per_step": {"windows_to_learner": B * 7 * 7056, "losses_broadcast": 4 * B, "parameters_every_100": 26903576}}
    if rank == 0:
        print(json.dumps(out))
    finish(world)


def fill_replay_segments(mem, device, seed):
    """fill_replay for a shard with one segment per environment (setup, not timed)."""
    tr = mem.transitions
    cap = tr.full_capacity
    fill_replay(mem, cap, device, seed)
    heads = torch.randint(0, tr.actor_capacity, (tr.nb_actor,), generator=torch.Generator().manual_seed(seed))
    for a in range(tr.nb_actor):
        tr.index_actor_host[a] = int(heads[a])
        tr.is_full_actor[a] = 1
    tr.index_actor.copy_(heads.to(device))


# ------------------------------------------------------------------------------------------ CPU arms
def oracle_learner(batch, threads=None):
    """The oracle port of Learner.learn (oracle/losses.py) on the host CPU cores."""
    from oracle import cases, losses, network as net
    torch.set_num_threads(threads or os.cpu_count())
    params = net.make_params(123)
    p_on, p_tg = net.to_torch(params, requires_grad=True), net.to_torch(params)
    adam = losses.Adam([k for k in p_on if net.is_trainable(k)], lr=5e-5, eps=3.125e-4)
    cfg = cases.iqn_cfg(N_TAU, N_TAU_P, K_Q)
    b = cases.make_batch(7, batch)
    tb = cases.batch_to_torch(b)
    w = torch.from_numpy(b["weights"])
    noise_shapes = cases.make_noises(0)

    def step(i):
        noises = tuple({k: (net.scale_noise(torch.randn_like(v[0])), net.scale_noise(torch.randn_like(v[1])))
                        for k, v in n.items()} for n in noise_shapes)
        taus = tuple(torch.rand(nq * batch, 1) for nq in (K_Q, N_TAU_P, N_TAU))
        losses.learn_step(p_on, p_tg, adam, tb, w, noises, taus, cfg)

    return step


def best_threads():
    """torch's intra-op scaling on many-core hosts is not monotonic (128 threads were 10x slower than 32 on the GPU
    box): probe a small step at a few thread counts and keep the fastest, so the CPU arm is not handicapped."""
    n = os.cpu_count() or 8
    cands = sorted({c for c in (n, n // 2, 64, 32, 16, 8) if 1 <= c <= n}, reverse=True)
    best, best_t = cands[0], float("inf")
    for c in cands:
        step = oracle_learner(64, c)                    # probed at B=64 (a B=16 step is too small to rank thread counts)
        step(0)
        t0 = time.perf_counter()
        step(1)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    return best


def cpu_baseline(max_seconds=25.0):
    threads = best_threads()
    step = oracle_learner(B, threads)
    t0 = time.perf_counter()
    step(0)                                     # warm-up (also sizes the sample)
    t1 = time.perf_counter() - t0
    n = int(max(2, min(5, max_seconds // max(t1, 1e-3) - 1)))
    t0 = time.perf_counter()
    for i in range(n):
        step(i)
    dt = (time.perf_counter() - t0) / n
    return {"value": 1.0 / dt, "unit": "grad-steps/s", "cores": os.cpu_count(), "threads": torch.get_num_threads(),
            "kind": "port", "sample": f"{n} full learner steps at batch=512, N=N'=64, K=32 (oracle port, torch CPU fp32)",
            "ms_per_step": dt * 1e3}


def run_reference(args):
    """Reference arm: the reference's own algorithm (pure Python/PyTorch, cannot travel to the GPU box) restated in
    oracle/ and timed on the host cores with every thread torch can use.  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = args.gpus
    # bound the run: each step is a sample of `bs` of the 512 transitions, scaled linearly to a full step
    threads = best_threads()
    probe = oracle_learner(64, threads)
    probe(0)
    t0 = time.perf_counter()
    probe(1)
    t64 = time.perf_counter() - t0
    budget = 150.0
    total_steps = args.steps + max(args.warmup, 1)
    bs = B
    while bs > 32 and (t64 * bs / 64) * total_steps > budget:
        bs //= 2
    step = oracle_learner(bs, threads)
    for i in range(max(args.warmup, 1)):
        step(i)
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(i)
    dt = (time.perf_counter() - t0) / args.steps
    full = dt * (B / bs)                                    # time of one full 512-transition learner step
    value = 1.0 / full
    out = {"metric": METRIC, "value": value, "unit": "grad-steps/s", "n_gpus": world, "steps": args.steps,
           "warmup": max(args.warmup, 1), "ms_per_step": full * 1e3, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "fp32", "data": "synthetic", "impl": "reference",
           "config": config_dict(world, args.replay_capacity), "sample_batch": bs,
           "cpu_baseline": {"value": value, "unit": "grad-steps/s", "cores": os.cpu_count(),
                            "threads": torch.get_num_threads(), "kind": "port",
                            "sample": f"each step = {bs} of the 512 transitions of one learner step, time scaled x{B // bs}"},
           "e2e": {"value": value, "unit": "grad-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))


def watchdog(seconds):
    """Hard stop: a benchmark must never hang a GPU box (e.g. a collective waiting for a dead rank)."""
    def run():
        time.sleep(seconds)
        sys.stderr.write(f"bench.py watchdog: no result after {seconds}s, aborting\n")
        sys.stderr.flush()
        os._exit(3)
    threading.Thread(target=run, daemon=True).start()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--replay-capacity", type=int, default=1 << 19)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c51", action="store_true", help="skip the configs[2] (Rainbow-only) leg")
    ap.add_argument("--dp-eager-allreduce", action="store_true",
                    help="N > 1: keep the gradient all-reduce eager between two CUDA graphs (round-1 scheme) instead of capturing it")
    ap.add_argument("--topology", default="dp", choices=["dp", "apex"],
                    help="dp: data-parallel learner (configs[1]/[4], the headline); apex: 1 learner + N-1 actor GPUs (configs[3])")
    ap.add_argument("--actor-envs", type=int, default=128, help="apex: environments per actor GPU")
    ap.add_argument("--actor-buffer", type=int, default=200, help="apex: steps per actor buffer flush (reference: 1000)")
    ap.add_argument("--acts-per-step", type=int, default=1, help="apex: batched acting iterations per learner step")
    ap.add_argument("--blocks", type=int, default=1, help="timed regions of --steps steps each; the median is the headline")
    ap.add_argument("--sustained-seconds", type=float, default=0.0, help="length of the sustained leg (0 = skip)")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of CUDA-graph replay")
    ap.add_argument("--max-seconds", type=int, default=900, help="watchdog: abort the process after this long")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed learner step (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and (args.impl != "ours" or args.topology != "dp"):
        ap.error("--dump-outputs applies to the data-parallel learner (--impl ours --topology dp)")
    watchdog(args.max_seconds)
    if args.impl == "reference":
        run_reference(args)
    elif args.topology == "apex":
        run_apex(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
