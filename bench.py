#!/usr/bin/env python
"""bench.py -- learner-side PPO throughput (GAE + normalisation + full update) of rlgym_ppo_b200 on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c2|c3]
                    [--precision bf16|fp32] [--device cpu|cuda] [--no-cpu] [--no-sub] [--dump-outputs DIR]

One "step" = one learner iteration at steady state on synthetic rollouts of the example shape (SURVEY.md 8d):
Learner.add_new_experience on N_new fresh timesteps (value inference on N_new+1 states, GAE + reward normalisation,
Welford update, ring append) followed by PPOLearner.learn on the full buffer (ppo_epochs x floor(buffer/B) optimiser
steps: permutation gather, fwd/bwd, clip, Adam).

  value     device-timed (CUDA events per step, L2 flushed between steps), rollout arrays already resident in HBM
  e2e       the same iteration through the public API with HOST (pinned) rollout arrays: H2D of the 7 arrays and the D2H
            read of the report scalars inside the timed region.  THIS is SURVEY.md 8(d)'s t_device ("from rollout arrays
            resident in pinned host memory to weights updated + report scalars on host") and the headline against the
            reference arm; `value` and the roofline explain it.
  roofline  per-kernel CUDA-event timing of one more (eager) step; work per launch = SURVEY.md 8(d)'s ALGORITHMIC figures
            (un-padded flops for the MLP kernels -> tensor roof; 28 B/step GAE, 744 B/sample gather, 28 B/param optimiser,
            1480 B/step append -> HBM roof), traffic = DRAM bytes per launch from the committed ncu --set full capture.
  sub       the other BASELINE.json configs, each with its own roofline: precision_fp32 (the same C2 step in the mode that
            meets the 1e-3 parity bar), c3 (large nets), c4 (4096-slot batched inference + 1M-step GAE), c5 (GAE sweep);
            at N > 1 also `strong` (dp_mode="replicated": fixed global batch, the reference's minibatch slices).
  cpu_baseline  the UNMODIFIED reference (baseline/_ref, pip-installed by build()) on this box's host cores, bounded
            sample (rank 0, N=1 only).

The headline and the precision_fp32, c3 and strong sub-records time exactly --steps learner iterations each (c4 times its
245 ticks, c5 its sweep).  `--dump-outputs DIR` writes what the last
device-timed step handed its caller (see dump_outputs) as DIR/<name>.npy; the inputs depend on the arguments only, so two
builds can be compared output for output.  The benchmark writes nothing into the source tree.

`--impl reference` times that reference alone (all host threads; `--device cuda`: PyTorch eager on the B200, the same-box
GPU comparator of BASELINE.md section 3) on this arm's config and prints the same JSON line.
Multi-GPU (torchrun, one rank per GPU): weak scaling -- every rank contributes N_new timesteps and takes 1/R of every
batch; the global batch, rollout and buffer grow with R (config.global_*); the reference arm runs that global config.
"""
import argparse
import contextlib
import io
import json
import os
import sys
import time
from types import SimpleNamespace

import numpy as np

sys.dont_write_bytecode = True      # the source tree may be read-only, and a run leaves nothing in it
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.benchlib import (ClockSampler, host_threads, import_reference, load_peaks, run_reference,  # noqa: E402
                            synth_rollout)

WORKLOADS = {
    # BASELINE.json configs[1]: example.py shape on 1xB200
    "c2": dict(name="example.py shape (configs[1]): 50k-step rollout, obs 89, 90 actions, 256x3 MLPs, buffer 150k, "
                    "batch 50k, 1 epoch", n_new=50000, obs=89, act=90, layers=(256, 256, 256), buffer=150000,
               batch=50000, epochs=1, ent=0.001),
    # BASELINE.json configs[2] (per-GPU share of it)
    "c3": dict(name="large nets (configs[2]): 2048-2048-1024-1024 policy/value, buffer 150k, batch 50k, 3 epochs",
               n_new=50000, obs=89, act=90, layers=(2048, 2048, 1024, 1024), buffer=150000, batch=50000, epochs=3,
               ent=0.001),
}
FLOP_PER_SAMPLE_UPDATE = {"c2": 1894912.0, "c3": 90097664.0}     # SURVEY.md 8(d), fwd+bwd both nets, un-padded
FLOP_PER_STATE_VALUE = {"c2": 308224.0, "c3": 15046656.0}
FLOP_PER_OBS_POLICY = {"c2": 353792.0, "c3": 15228928.0}

# ---- SURVEY.md 8(d): which roof bounds a C-ABI entry point, and its algorithmic bytes where ops.py counts real ones ----
TENSOR_BOUND = ("rlppo_policy_value_train_fused", "rlppo_policy_train_fused", "rlppo_value_train_fused", "rlppo_policy_infer_fused",
                "rlppo_value_infer_fused", "rlppo_wgrad_multi", "rlppo_linear_fwd", "rlppo_linear_dgrad",
                "rlppo_linear_dgrad_db", "rlppo_linear_wgrad", "rlppo_policy_head_train", "rlppo_policy_head_sample",
                "rlppo_linear_fwd_split", "rlppo_linear_dgrad_split", "rlppo_linear_wgrad_split",
                "rlppo_policy_head_train_split", "rlppo_policy_head_sample_split")
# C-ABI entry point -> kernel name in the ncu reports (profiles/ncu_traffic.json is keyed by kernel name)
KERNEL_OF = {"rlppo_wgrad_multi": "wgrad_multi_kernel", "rlppo_policy_value_train_fused": "fused_duo_kernel",
             "rlppo_policy_train_fused": "fused_duo_kernel",
             "rlppo_value_train_fused": "fused_duo_kernel", "rlppo_value_infer_fused": "fused_mlp_kernel<0, 0>",
             "rlppo_policy_infer_fused": "fused_mlp_kernel<0, 0>",
             "rlppo_gather_batch": "gather_kernel", "rlppo_gae_f32": "gae_scan3_kernel<1, 1>",
             "rlppo_linear_wgrad": "wgrad_kernel<256>", "rlppo_linear_fwd": "rowgemm_kernel<256, 0>",
             "rlppo_linear_dgrad": "rowgemm_kernel<256, 1>", "rlppo_linear_dgrad_db": "rowgemm_kernel<256, 1>",
             "rlppo_linear_wgrad_split": "wgrad_kernel<256>", "rlppo_linear_fwd_split": "rowgemm_kernel<256, 0>",
             "rlppo_linear_dgrad_split": "rowgemm_kernel<256, 1>",
             "rlppo_norm_clip_adam": "norm_clip_adam_kernel<0>", "rlppo_ring_append_fields_dev": "ring_append_fields_kernel",
             "rlppo_welford_update": "welford_kernel<1>", "rlppo_rows_to_bf16": "rows_to_bf16_kernel<0>"}
# ties in time are broken in this order, so the reported kernel does not flip between runs (VERDICT r1, weak #4)
DOMINANT_ORDER = ("rlppo_policy_value_train_fused", "rlppo_policy_train_fused", "rlppo_linear_fwd_split", "rlppo_linear_fwd", "rlppo_wgrad_multi",
                  "rlppo_value_train_fused")


def algorithmic(name, v, ctx):
    """(bound, work per ALL launches of this entry point in one step) from SURVEY.md 8(d).  ctx: rows per optimiser
    step, new timesteps, parameter count."""
    if name in TENSOR_BOUND:
        return "tensor", v["flop"]                       # ops.py counts 2*M*N*K with the true (un-padded) extents
    b = v["byte"]
    if name == "rlppo_gather_batch":
        b = 744.0 * ctx["rows_per_update"] * v["calls"]  # 372 B/sample read + 372 B written (materialised)
    elif name in ("rlppo_norm_clip_adam", "rlppo_norm_clip_adam_peers", "rlppo_norm_clip_adam_peers2"):
        b = 28.0 * ctx["n_params"] * v["calls"]          # p, g, m, v read; p, m, v written
    elif name == "rlppo_ring_append_fields_dev":
        b = 1480.0 * ctx["n_new"] * v["calls"]
    elif name == "rlppo_welford_update":
        b = 4.0 * 150 * v["calls"]
    return "hbm", b


def roofline_table(per, peaks, ctx, workload):
    """Per entry point: share of the step, achieved algorithmic rate, roof, fraction, DRAM traffic per launch."""
    try:
        tbl = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    except Exception:
        tbl = {}
    total = sum(v["ms"] for v in per.values()) or 1.0
    rows = {}
    for name, v in per.items():
        bound, work = algorithmic(name, v, ctx)
        if bound == "tensor":
            ach, peak, unit = work / v["ms"] / 1e9, peaks["tc"], "TFLOP/s"
        else:
            ach, peak, unit = work / v["ms"] / 1e6, peaks["hbm"], "GB/s"
        traffic = tbl.get(workload, {}).get(KERNEL_OF.get(name, name))
        row = {"kernel": name, "bound": bound, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak,
               "traffic": traffic, "launches": v["calls"], "avg_launch_ms": v["ms"] / v["calls"], "ms": v["ms"],
               "share": v["ms"] / total,
               "algorithmic_per_launch": work / v["calls"], "algorithmic_unit": "flop" if bound == "tensor" else "byte"}
        if bound == "tensor":
            row["frac_of_burst_peak"] = ach / peaks["tc_burst"]
            if v.get("mma_flop"):
                row["issued_mma_tflops"] = v["mma_flop"] / v["ms"] / 1e9      # split operands: 3-6 MMAs per algorithmic one
        if traffic and bound == "hbm":
            row["traffic_over_algorithmic"] = traffic / (work / v["calls"])
        elif traffic and v["byte"]:
            row["dram_bytes_per_launch_vs_min_io"] = traffic / (v["byte"] / v["calls"])
        rows[name] = row
    return rows


def dominant(rows):
    top = max(r["ms"] for r in rows.values())
    for name in DOMINANT_ORDER:
        if name in rows and rows[name]["ms"] >= 0.9 * top:
            return name
    return max(rows, key=lambda k: rows[k]["ms"])


# ------------------------------------------------------------------------------------------------------------------
# reference arm
# ------------------------------------------------------------------------------------------------------------------
def reference_arm(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    R = max(1, args.gpus)
    # the config of OUR arm at this N (weak scaling: global rollout / batch / buffer grow with N)
    glob = dict(wl, n_new=wl["n_new"] * R, batch=wl["batch"] * R, buffer=wl["buffer"] * R)
    steps, warmup = max(1, min(args.steps, 5)), max(0, min(args.warmup, 1))
    if args.workload == "c3":
        steps, warmup = 1, 0          # one c3 iteration is minutes of CPU work
    if R >= 4:
        steps = min(steps, 2)
    device = "cuda:0" if args.device == "cuda" else "cpu"
    tput, sec, threads, kind = run_reference(glob, steps, warmup, device=device)
    sample = (f"{steps} steady-state iteration(s) of the full workload after {warmup} warm-up: the unmodified reference's "
              f"Learner.add_new_experience + PPOLearner.learn on {device}" if kind == "reference" else
              f"{steps} iteration(s), oracle port of the reference (baseline/_ref missing)")
    line = {"impl": "reference", "metric": "learner_timesteps_per_sec", "value": tput, "unit": "timesteps/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": sec * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["name"], "global_new_timesteps": glob["n_new"], "global_batch": glob["batch"],
                       "global_buffer": glob["buffer"], "device": device},
            "cpu_baseline": {"value": tput, "unit": "timesteps/s", "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": tput, "unit": "timesteps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------------------------
class Rig:
    """A learner (PPOLearner + the namespace Learner.add_new_experience runs on) with a pool of synthetic rollouts,
    pinned on the host and resident on the device."""

    def __init__(self, wl, dev, rank, world, precision, dp_mode="sharded", n_pool=3, quiet=True):
        import torch
        from rlgym_ppo_b200.learner import Learner
        from rlgym_ppo_b200.ppo import ExperienceBuffer, PPOLearner
        from rlgym_ppo_b200.util import WelfordRunningStat
        self.torch, self.Learner, self.wl, self.dev, self.world, self.rank = torch, Learner, wl, dev, world, rank
        torch.manual_seed(123)        # identical initial weights on every rank
        replicated = dp_mode == "replicated"
        # sharded (weak scaling): every rank owns its rollout / buffer / shuffle, per-rank batch = the workload's batch.
        # replicated (strong scaling): the SAME rollout, buffer and permutation on every rank, the workload's batch is global.
        with contextlib.redirect_stdout(io.StringIO()) if quiet else contextlib.nullcontext():
            self.ppo = PPOLearner(wl["obs"], wl["act"], 0, wl["layers"], wl["layers"], (0.1, 1.0), wl["batch"],
                                  wl["epochs"], 3e-4, 3e-4, 0.2, wl["ent"], wl["batch"], dev, dp_mode=dp_mode,
                                  precision=precision)
        self.ns = SimpleNamespace(ppo_learner=self.ppo, return_stats=WelfordRunningStat(1, device=dev),
                                  standardize_returns=True, gae_gamma=0.99, gae_lambda=0.95,
                                  max_returns_per_stats_increment=150,
                                  experience_buffer=ExperienceBuffer(wl["buffer"], 123 + (0 if replicated else rank), dev))
        rng = np.random.RandomState(0 if replicated else rank)
        self.pool_host, self.pool_dev = [], []
        for _ in range(n_pool):
            states, rewards, next_states, dones, truncated = synth_rollout(rng, wl["n_new"], wl["obs"])
            acts, logp = self.ppo.policy.get_action_device(torch.from_numpy(states).to(dev))
            host = [torch.from_numpy(a).pin_memory() for a in
                    (states, acts.float().cpu().numpy(), logp.cpu().numpy(), rewards, next_states, dones, truncated)]
            self.pool_host.append((tuple(t.numpy() for t in host), host))   # numpy views of pinned memory (+ keep-alive)
            self.pool_dev.append(tuple(t.to(dev) for t in host))
        self.h2d_bytes = sum(t.numel() * t.element_size() for t in self.pool_host[0][1])
        self.d2h_bytes = self.ppo._tail_host.numel() * 4
        self.it = 0
        self.n_pool = n_pool

    def step(self, exp):
        self.Learner.add_new_experience(self.ns, exp)
        return self.ppo.learn(self.ns.experience_buffer)

    def next_dev(self):
        e = self.pool_dev[self.it % self.n_pool]
        self.it += 1
        return e

    def next_host(self):
        e = self.pool_host[self.it % self.n_pool][0]
        self.it += 1
        return e

    def barrier(self):
        if self.world > 1:
            self.torch.distributed.barrier()
        self.torch.cuda.synchronize()

    def fill_and_warm(self, n_warm):
        wl = self.wl
        while len(self.ns.experience_buffer) + wl["n_new"] < wl["buffer"]:
            self.Learner.add_new_experience(self.ns, self.next_dev())
        self.barrier()                                # ranks reach their first data-parallel step together
        for _ in range(max(n_warm, 2 * self.n_pool)):  # every pooled rollout at least twice: its CUDA graph exists
            self.step(self.next_dev())

    def timed_device(self, K, flush_buf):
        torch = self.torch
        self.barrier()
        evs = []
        for _ in range(K):
            flush_buf.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            report = self.step(self.next_dev())
            e1.record()
            evs.append((e0, e1))
        self.barrier()
        return sum(a.elapsed_time(b) for a, b in evs), report

    def timed_e2e(self, K, n_warm):
        for _ in range(n_warm):                       # the host-input path has its own staging slots and graph
            self.step(self.next_host())
        self.barrier()
        t0 = time.perf_counter()
        for _ in range(K):
            report = self.step(self.next_host())
            _ = report["Policy Entropy"]
        self.barrier()
        return (time.perf_counter() - t0) * 1e3

    def phase_pass(self, K, flush_buf):
        """Device time of the two halves of a step (events around each), K steps: where a multi-GPU step waits."""
        torch = self.torch
        self.barrier()
        a = b = 0.0
        for _ in range(K):
            flush_buf.zero_()
            e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            exp = self.next_dev()
            e0.record()
            self.Learner.add_new_experience(self.ns, exp)
            e1.record()
            self.ppo.learn(self.ns.experience_buffer)
            e2.record()
            torch.cuda.synchronize()
            a += e0.elapsed_time(e1)
            b += e1.elapsed_time(e2)
        self.barrier()
        return a / K, b / K

    def max_over_ranks(self, *vals):
        if self.world == 1:
            return vals
        t = self.torch.tensor(vals, dtype=self.torch.float64, device=self.dev)
        self.torch.distributed.all_reduce(t, op=self.torch.distributed.ReduceOp.MAX)
        return tuple(float(x) for x in t)

    def kernel_pass(self, flush_buf):
        """One eager step with CUDA events around every C-ABI call (rlgym_ppo_b200._lib.timing_begin)."""
        from rlgym_ppo_b200 import _lib
        flush_buf.zero_()
        self.torch.cuda.synchronize()
        _lib.timing_begin()
        self.step(self.next_dev())
        return _lib.timing_end()

    def ctx(self):
        wl = self.wl
        n_params = int(self.ppo._params.numel())
        return {"rows_per_update": wl["batch"], "n_new": wl["n_new"], "n_params": n_params}


def dump_outputs(rig, report, out_dir):
    """What one step hands its caller, as out_dir/<name>.npy: the report's metrics (float64; the wall-clock
    "PPO Batch Consumption Time" is not a result and is left out), both networks' updated parameters (float32) and the
    value targets and advantages add_new_experience computed for the step's rollout (the newest n_new buffer rows).
    The inputs are the same from run to run, the outputs are not bit-identical: weight gradients are summed with float
    atomics, and Adam carries those last-bit differences forward.  Two runs of one build with --steps 20 --warmup 3
    (26 learner iterations; B200 at its 1000 W power limit) differed by up to 1.1e-2 relative L2 on a weight tensor,
    2.2e-3 on the advantages and 6.4e-3 relative on a report metric (the clip fraction)."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"report." + k.lower().replace(" ", "_"): np.float64(v) for k, v in report.items()
              if k != "PPO Batch Consumption Time"}
    for net, module in (("policy", rig.ppo.policy), ("value_net", rig.ppo.value_net)):
        for k, t in module.state_dict().items():
            arrays[f"{net}.{k}"] = t.detach().float().cpu().numpy()
    buf = rig.ns.experience_buffer
    for field in ("values", "advantages"):
        arrays["buffer." + field] = getattr(buf, field)[-rig.wl["n_new"]:].cpu().numpy()
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def gae_sweep(dev, peaks, log2s=(20, 22, 24, 26, 28), reps=5):
    """BASELINE configs[4] (C5): flat rollouts with random done masks, 28 algorithmic bytes per step, CUDA events around
    the C-ABI call, median of `reps`; inputs of 2^24 steps and more exceed the 126 MB L2."""
    import torch
    from rlgym_ppo_b200 import ops
    out = []
    for log2n in log2s:
        n = 1 << log2n
        g = torch.Generator(device=dev)
        g.manual_seed(5)
        rew = torch.randn(n, device=dev, generator=g) * 0.1
        done = (torch.rand(n, device=dev, generator=g) < 1 / 300).float()
        tr32 = ((torch.rand(n, device=dev, generator=g) < 1 / 1500).float() * (1 - done))
        tr32[-1] = 1 - done[-1]
        val = torch.randn(n + 1, device=dev, generator=g)
        std = torch.tensor([0.7], device=dev)
        bufs = tuple(torch.empty(n, device=dev) for _ in range(3))
        row = {"timesteps": n}
        for label, tr, real in (("f64_truncated", tr32.double(), 32), ("f32_truncated", tr32, 28)):
            for _ in range(2):
                ops.gae(rew, done, tr, val, 0.99, 0.95, std, out=bufs)
            ts = []
            for _ in range(reps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                ops.gae(rew, done, tr, val, 0.99, 0.95, std, out=bufs)
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
            ms = float(np.median(ts))
            row[label] = {"ms": ms, "algorithmic_GBps": 28 * n / ms / 1e6, "frac": 28 * n / ms / 1e6 / peaks["hbm"],
                          "real_bytes_per_step": real, "timesteps_per_sec": n / ms * 1e3}
        del rew, done, tr32, val, bufs
        out.append(row)
    return out


def sub_fp32(args, dev, rank, world, flush_buf, peaks):
    """The same C2 step with precision="fp32" (split operands): the mode the 1e-3 parity tests run."""
    wl = WORKLOADS["c2"]
    rig = Rig(wl, dev, rank, world, "fp32")
    rig.fill_and_warm(3)
    K = args.steps
    dev_ms, _ = rig.timed_device(K, flush_buf)
    e2e_ms = rig.timed_e2e(K, 3)
    dev_ms, e2e_ms = rig.max_over_ranks(dev_ms, e2e_ms)
    out = {"precision": "fp32 (hi/mid/lo bf16 split: 6 products forward, 3 backward)",
           "value": wl["n_new"] * world * K / (dev_ms / 1e3), "ms_per_step": dev_ms / K,
           "e2e": {"value": wl["n_new"] * world * K / (e2e_ms / 1e3), "ms_per_step": e2e_ms / K}, "unit": "timesteps/s"}
    if rank == 0:
        rows = roofline_table(rig.kernel_pass(flush_buf), peaks, rig.ctx(), "c2_fp32")
        top = dominant(rows)
        out["roofline"] = rows[top]
        out["kernels"] = {k.replace("rlppo_", ""): {"ms": round(r["ms"], 4), "share": round(r["share"], 3),
                                                    "frac": round(r["frac"], 3), "bound": r["bound"]}
                          for k, r in sorted(rows.items(), key=lambda kv: -kv[1]["ms"])}
    elif world > 1:
        flush_buf.zero_()
        rig.step(rig.next_dev())
    return out


def sub_c3(args, dev, rank, world, flush_buf, peaks):
    """BASELINE configs[2]: 2048-2048-1024-1024 nets, 3 epochs x 3 batches per iteration (per-GPU share; weak scaling)."""
    wl = WORKLOADS["c3"]
    rig = Rig(wl, dev, rank, world, "bf16", n_pool=2)
    rig.fill_and_warm(2)
    K = args.steps
    dev_ms, _ = rig.timed_device(K, flush_buf)
    (dev_ms,) = rig.max_over_ranks(dev_ms)
    n_updates = wl["epochs"] * (wl["buffer"] // wl["batch"])
    flop = wl["n_new"] * FLOP_PER_STATE_VALUE["c3"] + n_updates * wl["batch"] * FLOP_PER_SAMPLE_UPDATE["c3"]
    out = {"workload": wl["name"], "value": wl["n_new"] * world * K / (dev_ms / 1e3), "unit": "timesteps/s",
           "ms_per_step": dev_ms / K, "steps": K, "algorithmic_tflop_per_step_per_gpu": flop / 1e12,
           "achieved_tflops_per_gpu": flop / (dev_ms / K / 1e3) / 1e12,
           "frac_of_sustained_bf16_peak": flop / (dev_ms / K / 1e3) / 1e12 / peaks["tc"],
           "gradient_exchange": rig.ppo.dp_collective}
    if rank == 0:
        rows = roofline_table(rig.kernel_pass(flush_buf), peaks, rig.ctx(), "c3")
        top = dominant(rows)
        out["roofline"] = rows[top]
        out["kernels"] = {k.replace("rlppo_", ""): {"ms": round(r["ms"], 3), "share": round(r["share"], 3),
                                                    "frac": round(r["frac"], 3), "bound": r["bound"]}
                          for k, r in sorted(rows.items(), key=lambda kv: -kv[1]["ms"])}
    elif world > 1:
        flush_buf.zero_()
        rig.step(rig.next_dev())
    return out


def sub_c4(args, dev, rank, world, peaks):
    """BASELINE configs[3]: batched policy inference over 4096 env slots (sharded across ranks) for 245 ticks -- the
    observations of every tick go pinned host -> HBM, the sampled actions come back to the host -- then value inference and
    GAE over the 1 003 520-step iteration (this rank's slots), through the collection classes' own tick path."""
    import torch
    from rlgym_ppo_b200 import ops
    from rlgym_ppo_b200.batched_agents.tick import TickInference
    from rlgym_ppo_b200.ppo import DiscreteFF, ValueEstimator
    wl = WORKLOADS["c2"]
    slots, ticks = 4096 // world, 245
    torch.manual_seed(123)
    pol = DiscreteFF(wl["obs"], wl["act"], wl["layers"], dev)
    val = ValueEstimator(wl["obs"], wl["layers"], dev)
    tick = TickInference(pol, slots, wl["obs"])
    rng = np.random.RandomState(rank)
    tick.obs_host.copy_(torch.from_numpy(rng.randn(slots, wl["obs"]).astype(np.float32)))
    for _ in range(5):
        tick.run()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(ticks):
        tick.run()                       # returns after the actions of this tick are in pinned host memory
    infer_s = time.perf_counter() - t0
    n = slots * ticks
    g = torch.Generator(device=dev)
    g.manual_seed(7)
    states = torch.randn(n + 1, wl["obs"], device=dev, generator=g)
    rew = torch.randn(n, device=dev, generator=g) * 0.1
    done = (torch.rand(n, device=dev, generator=g) < 1 / 300).float()
    tr = ((torch.rand(n, device=dev, generator=g) < 1 / 1500).float() * (1 - done)).double()
    std = torch.tensor([0.7], device=dev)
    ws = val._stack.workspace(n + 1)
    out3 = tuple(torch.empty(n, device=dev) for _ in range(3))
    values = torch.empty(n + 1, device=dev)

    def learner_half():
        val._stack.stage_rows(states, ws["x"])
        val.values_from_bf16(ws["x"], n + 1, out=values)
        ops.gae(rew, done, tr, values, 0.99, 0.95, std, out=out3)
    for _ in range(2):
        learner_half()
    e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    torch.cuda.synchronize()
    e0.record()
    val._stack.stage_rows(states, ws["x"])
    val.values_from_bf16(ws["x"], n + 1, out=values)
    e1.record()
    ops.gae(rew, done, tr, values, 0.99, 0.95, std, out=out3)
    e2.record()
    torch.cuda.synchronize()
    v_ms, g_ms = e0.elapsed_time(e1), e1.elapsed_time(e2)
    t = torch.tensor([infer_s, v_ms, g_ms], dtype=torch.float64, device=dev)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    infer_s, v_ms, g_ms = (float(x) for x in t)
    total_steps = slots * world * ticks
    flop_tick = slots * FLOP_PER_OBS_POLICY["c2"]
    return {"workload": "configs[3]: 4096 env slots x 245 ticks = 1 003 520 steps per iteration",
            "slots_per_gpu": slots, "ticks": ticks,
            "inference_tick_us": infer_s / ticks * 1e6,
            "inference_rows_per_sec": slots * world * ticks / infer_s,
            "inference_tflops_per_gpu": flop_tick * ticks / infer_s / 1e12,
            "tick_path": "pinned obs -> H2D -> rows_to_bf16 -> fused policy kernel (MLP + sample) -> actions D2H, one CUDA "
                         "graph per tick, host waits on one event",
            "value_inference_ms": v_ms, "gae_ms": g_ms,
            "gae_algorithmic_GBps": 28 * n / g_ms / 1e6, "gae_frac_of_hbm": 28 * n / g_ms / 1e6 / peaks["hbm"],
            "iteration_timesteps_per_sec_no_env": total_steps / (infer_s + (v_ms + g_ms) / 1e3),
            "note": "environment stepping excluded (host processes; not part of the learner-side path)"}


def sub_strong(args, dev, rank, world, flush_buf):
    """Strong scaling: the reference's semantics -- ONE 50k rollout, global batch 50k split into `world` minibatch slices
    (ppo_learner.py:134-193), replicated buffers, identical optimiser step on every rank."""
    wl = WORKLOADS["c2"]
    rig = Rig(wl, dev, rank, world, args.precision, dp_mode="replicated")
    rig.fill_and_warm(3)
    K = args.steps
    dev_ms, _ = rig.timed_device(K, flush_buf)
    e2e_ms = rig.timed_e2e(K, 3)
    dev_ms, e2e_ms = rig.max_over_ranks(dev_ms, e2e_ms)
    return {"scaling": "strong", "dp_mode": "replicated", "global_new_timesteps": wl["n_new"], "global_batch": wl["batch"],
            "value": wl["n_new"] * K / (dev_ms / 1e3), "ms_per_step": dev_ms / K, "unit": "timesteps/s",
            "e2e": {"value": wl["n_new"] * K / (e2e_ms / 1e3), "ms_per_step": e2e_ms / K},
            "gae": "sharded across ranks by contiguous chunks" if getattr(rig.ppo, "gae_sharded", False) else "replicated",
            "gradient_exchange": rig.ppo.dp_collective}


def b200_arm(args, wl):
    import torch

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    dev = f"cuda:{local_rank}"
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device(dev))

    from rlgym_ppo_b200 import _lib
    _lib.require_device()
    peaks = load_peaks()

    R = world
    n_glob, batch, cap = wl["n_new"] * R, wl["batch"] * R, wl["buffer"] * R
    rig = Rig(wl, dev, rank, world, args.precision)
    ppo = rig.ppo
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
    n_warm = max(args.warmup, 3)
    rig.fill_and_warm(n_warm)

    # ---- (1) device-resident timing: K steps, one event pair per step, L2 flushed between steps --------------------
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    calls0 = _lib.CALLS
    dev_ms, report = rig.timed_device(args.steps, flush_buf)
    calls = _lib.CALLS - calls0
    if args.dump_outputs and rank == 0:
        dump_outputs(rig, report, args.dump_outputs)
    # ---- (2) end to end through the public API with host buffers ---------------------------------------------------
    e2e_ms = rig.timed_e2e(args.steps, n_warm)
    clocks = sampler.stop() if sampler else None
    dev_ms, e2e_ms = rig.max_over_ranks(dev_ms, e2e_ms)
    phases = rig.max_over_ranks(*rig.phase_pass(5, flush_buf))

    # ---- (3) per-kernel pass for the roofline object (rank 0; not part of the timed numbers) --------------------------
    roofline, kernels = None, None
    if rank != 0 and world > 1:
        flush_buf.zero_()
        rig.step(rig.next_dev())      # the collectives of rank 0's instrumented step need their peers
    if rank == 0:
        rows = roofline_table(rig.kernel_pass(flush_buf), peaks, rig.ctx(), args.workload)
        top = dominant(rows)
        roofline = dict(rows[top], peak_source=peaks["src"],
                        why_this_kernel="largest share of the step among the kernels (ties within 10 % resolved in a "
                                        "fixed order so the name is stable across runs)")
        kernels = {k.replace("rlppo_", ""): {"calls": r["launches"], "ms": round(r["ms"], 4), "share": round(r["share"], 4),
                                             "bound": r["bound"], r["unit"]: round(r["achieved"], 2),
                                             "frac": round(r["frac"], 4),
                                             **({"traffic_over_algorithmic": round(r["traffic_over_algorithmic"], 2)}
                                                if "traffic_over_algorithmic" in r else {})}
                   for k, r in sorted(rows.items(), key=lambda kv: -kv[1]["ms"])}

    # ---- (4) the other configs (every rank takes part; rank 0 reports) --------------------------------------------
    sub = {}
    rig_bytes[0], rig_bytes[1] = rig.h2d_bytes, rig.d2h_bytes
    if not args.no_sub and args.workload == "c2":
        del rig
        torch.cuda.empty_cache()
        for name, fn in (("precision_fp32", lambda: sub_fp32(args, dev, rank, world, flush_buf, peaks)),
                         ("c3", lambda: sub_c3(args, dev, rank, world, flush_buf, peaks)),
                         ("c4", lambda: sub_c4(args, dev, rank, world, peaks)),
                         ("strong", (lambda: sub_strong(args, dev, rank, world, flush_buf)) if world > 1 else None)):
            if fn is None:
                continue
            try:
                sub[name] = fn()
            except Exception as e:  # noqa: BLE001  (a failing sub-benchmark must not lose the headline line)
                if world > 1:
                    raise           # ranks would desynchronise: fail loudly instead
                sub[name] = {"error": f"{type(e).__name__}: {e}"}
            torch.cuda.empty_cache()
        try:
            sweep = gae_sweep(dev, peaks)
            if world > 1:
                ms = torch.tensor([r["f64_truncated"]["ms"] for r in sweep] + [r["f32_truncated"]["ms"] for r in sweep],
                                  dtype=torch.float64, device=dev)
                torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
                k = len(sweep)
                for i, r in enumerate(sweep):       # every rank scans its own 2^k-step rollout: aggregate = world x
                    for j, label in enumerate(("f64_truncated", "f32_truncated")):
                        t = float(ms[j * k + i])
                        r[label].update(ms=t, aggregate_GBps=28 * r["timesteps"] * world / t / 1e6,
                                        aggregate_timesteps_per_sec=r["timesteps"] * world / t * 1e3)
            sub["c5"] = {"workload": "configs[4]: flat GAE sweep, random done masks (p=1/300), one rollout per GPU",
                         "peak_GBps": peaks["hbm"], "sweep": sweep}
        except Exception as e:  # noqa: BLE001
            if world > 1:
                raise
            sub["c5"] = {"error": f"{type(e).__name__}: {e}"}

    # ---- (5) CPU baseline: the reference itself on this box's host cores (rank 0, single-GPU run only) -----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        if args.workload == "c2":
            tput, sec, threads, kind = run_reference(wl, 3, 1)
            cpu = {"value": tput, "unit": "timesteps/s", "cores": threads, "kind": kind,
                   "sample": "3 steady-state iterations of the full workload after 1 warm-up: the unmodified reference "
                             "(baseline/_ref) Learner.add_new_experience + PPOLearner.learn, device='cpu'",
                   "sec_per_step": sec}
        else:
            small = dict(wl, n_new=5000, batch=5000, buffer=15000)
            tput, sec, threads, kind = run_reference(small, 1, 0)
            cpu = {"value": tput, "unit": "timesteps/s", "cores": threads, "kind": kind,
                   "sample": "1 iteration at 1/10 of the rows (5k new, batch 5k, buffer 15k), same nets and epochs",
                   "sec_per_step": sec}

    if rank == 0:
        K = args.steps
        n_updates = wl["epochs"] * (cap // batch)
        flop_step = n_glob * FLOP_PER_STATE_VALUE[args.workload] + n_updates * batch * FLOP_PER_SAMPLE_UPDATE[args.workload]
        exact = args.precision == "fp32"
        line = {
            "metric": "learner_timesteps_per_sec", "value": n_glob * K / (dev_ms / 1e3), "unit": "timesteps/s",
            "n_gpus": world, "steps": K, "warmup": n_warm, "ms_per_step": dev_ms / K,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16x3 (fp32-equivalent split operands)" if exact else "bf16", "data": "synthetic",
            "config": {"workload": wl["name"], "global_new_timesteps": n_glob, "global_batch": batch,
                       "global_buffer": cap, "optimizer_steps_per_step": n_updates,
                       "consumed_samples_per_step": n_updates * batch,
                       "precision": args.precision,
                       "headline": "e2e (SURVEY.md 8(d) t_device: pinned host arrays in, report scalars out); `value` "
                                   "starts with the rollout resident in HBM",
                       "parallelism": (f"dp{world} (per-rank experience shards; gradient exchange per optimiser step: "
                                       + ("summed inside the optimiser launch from the peers' arenas over NVLink)"
                                          if ppo.dp_collective == "p2p" else "NCCL allreduce of the flat gradient arena)"))
                       if world > 1 else "dp1",
                       "gradient_exchange": ppo.dp_collective,
                       "l2": "flushed between timed steps (256 MiB write); working set > L2",
                       "algorithmic_tflop_per_step": flop_step / 1e12,
                       "achieved_tflops": flop_step / (dev_ms / K / 1e3) / 1e12,
                       "step_frac_of_sustained_bf16_peak": flop_step / (dev_ms / K / 1e3) / 1e12 / (peaks["tc"] * world)},
            "e2e": {"value": n_glob * K / (e2e_ms / 1e3), "unit": "timesteps/s", "ms_per_step": e2e_ms / K,
                    "h2d_bytes_per_step": rig_bytes[0] * world, "d2h_bytes_per_step": rig_bytes[1] * world},
            "gpu_launches": calls,
            "phases_ms": {"add_new_experience": phases[0], "learn": phases[1],
                          "note": "device time of the two halves of a step, max over ranks (5 extra steps)"},
            "clocks": clocks,
            "roofline": roofline,
            "cpu_baseline": cpu,
            "kernels": kernels,
            "sub": sub,
            "report": {k: (float(v) if isinstance(v, (int, float, np.floating)) else v) for k, v in report.items()},
        }
        print(json.dumps(line))
    if world > 1:
        torch.distributed.destroy_process_group()


rig_bytes = [0, 0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default=os.environ.get("RLPPO_PRECISION", "bf16"), choices=["bf16", "fp32"])
    ap.add_argument("--device", default="cpu", choices=["cpu", "cuda"], help="--impl reference: where the reference runs")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-sub", action="store_true", help="skip the sub-records (other configs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last device-timed step as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of this project's timed path (--impl b200)")
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        reference_arm(args, wl)
    else:
        b200_arm(args, wl)


if __name__ == "__main__":
    main()
