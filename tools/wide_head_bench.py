"""Wide discrete head (rlppo_head_discrete_*): kernel times and achieved HBM bandwidth at M = 50 000 rows, and the
learn() step time of a 256x3 PPOLearner with 90 actions (the fused path) against 300 / 1024 actions (logits + per-row
head), run alternately in one process.

    python tools/wide_head_bench.py [--out profiles/wide_head_bench.json] [--launches 50] [--steps 5]

Kernel times: CUDA events around R launches replayed from one CUDA graph (so host-side launch preparation is not
counted), after warm-up.  Each launch reads a different copy of the inputs, the copies together more than twice the
126 MB L2, so every launch reads its logits from HBM.  Achieved bytes/s = the algorithmic bytes (2 * 3 * A of split logits
+ 12 B of scalars in; train: 2 * pad8(A) of bf16 d(logits) out; sample: 12 B out) over kernel time, compared with the
6459 GB/s copy bandwidth measured on B200 (DESIGN.md section 5)."""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

COPY_GBPS = 6459.0
L2_BYTES = 126 << 20
M = 50_000


def pad8(n):
    return (n + 7) // 8 * 8


def pad64(n):
    return (n + 63) // 64 * 64


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # noqa: BLE001
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"not read ({e})"}


def graph_time_ms(launch, n_launch, repeats=5):
    """Per-launch device time of `launch(i)` for i in range(n_launch), replayed from one CUDA graph."""
    for i in range(n_launch):                  # warm-up: module load, attribute setup, first-touch of every copy
        launch(i)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            for i in range(n_launch):
                launch(i)
    torch.cuda.current_stream().wait_stream(side)
    g.replay()
    torch.cuda.synchronize()
    times = []
    for _ in range(repeats):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1) / n_launch)
    return float(np.median(times)), float(min(times)), float(max(times))


def kernel_bench(A, n_launch):
    from rlgym_ppo_b200 import ops
    P = pad64(A)
    per_copy = M * 3 * P * 2
    copies = max(2, int(np.ceil(2 * L2_BYTES / (M * 3 * A * 2))))
    z = [torch.randn(M, 3 * P, device="cuda").mul_(0.5).to(torch.bfloat16) for _ in range(copies)]
    for t in z:                      # the low parts an order of magnitude below the high part, as a split fp32 value
        t[:, P:].mul_(2 ** -8)
    dz = [torch.empty(M, pad8(A), dtype=torch.bfloat16, device="cuda") for _ in range(copies)]
    acts = torch.randint(0, A, (M,), device="cuda").float()
    old = torch.full((M,), -np.log(A), device="cuda")
    adv = torch.randn(M, device="cuda")
    metrics = torch.zeros(8, device="cuda")
    a_out = torch.empty(M, dtype=torch.int64, device="cuda")
    lp_out = torch.empty(M, device="cuda")

    def train(i):
        k = i % copies
        ops.head_discrete_train(z[k], 3, P, M, A, acts, old, adv, 1.0 / M, 0.2, 0.01, dz[k], 1, 0, pad8(A), metrics)

    def sample(i):
        ops.head_discrete_sample(z[i % copies], 3, P, M, A, seed=1, offset=i * M, actions_i64_out=a_out, logp_out=lp_out)

    out = {"A": A, "rows": M, "input_copies": copies, "input_bytes_total": copies * per_copy}
    for name, fn, nbytes in (("train", train, M * (6 * A + 12 + 2 * pad8(A))), ("sample", sample, M * (6 * A + 12))):
        med, lo, hi = graph_time_ms(fn, n_launch)
        gbps = nbytes / (med * 1e-3) / 1e9
        out[name] = {"us_median": med * 1e3, "us_min": lo * 1e3, "us_max": hi * 1e3, "bytes": nbytes,
                     "GBps": gbps, "fraction_of_copy_bw": gbps / COPY_GBPS}
    del z, dz
    torch.cuda.empty_cache()
    return out


def make_learner(A):
    from rlgym_ppo_b200.ppo import ExperienceBuffer, PPOLearner
    obs = 89
    torch.manual_seed(A)
    with contextlib.redirect_stdout(io.StringIO()):
        lr = PPOLearner(obs, A, 0, (256,) * 3, (256,) * 3, (0.1, 1.0), M, 1, 3e-4, 3e-4, 0.2, 0.01, M, "cuda:0")
    rng = np.random.RandomState(A)
    buf = ExperienceBuffer(M, 1, "cuda:0")
    buf.submit_experience(rng.randn(M, obs).astype(np.float32), rng.randint(0, A, M).astype(np.float32),
                          np.full(M, -np.log(A), np.float32), np.zeros(M, np.float32), np.zeros((M, obs), np.float32),
                          np.zeros(M, np.float32), np.zeros(M), rng.randn(M).astype(np.float32),
                          rng.randn(M).astype(np.float32))
    return lr, buf


def learn_bench(actions, steps, rounds=3):
    nets = {A: make_learner(A) for A in actions}
    for lr, buf in nets.values():          # warm-up: workspaces, graph capture, kernel configuration
        for _ in range(2):
            lr.learn(buf)
    torch.cuda.synchronize()
    times = {A: [] for A in actions}
    for _ in range(rounds):                # alternate the shapes so that drift on a shared host hits all of them
        for A, (lr, buf) in nets.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                lr.learn(buf)
            torch.cuda.synchronize()
            times[A].append((time.perf_counter() - t0) / steps * 1e3)
    return {str(A): {"ms_per_learn_median": float(np.median(v)), "ms_rounds": v, "fused": nets[A][0].policy._stack.fused_ok,
                     "wide_head": nets[A][0].policy.wide} for A, v in times.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "wide_head_bench.json"))
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--steps", type=int, default=5)
    args = ap.parse_args()
    from rlgym_ppo_b200 import _lib
    _lib.require_device()
    res = {"gpu": gpu_info(), "copy_bandwidth_GBps": COPY_GBPS,
           "method": "CUDA events around graph-replayed launches; inputs rotated over copies totalling > 2x L2",
           "kernels": [kernel_bench(A, args.launches) for A in (257, 1024, 4096)],
           "learn": {"rows": M, "nets": "256x3 policy and critic, obs 89, one epoch, batch = minibatch = 50 000",
                     "steps_per_round": args.steps, "by_actions": learn_bench((90, 300, 1024), args.steps)}}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
