"""Hidden widths that are not multiples of 8, and the value head above 2048 inputs: what they cost.

    python tools/width_bench.py [--out profiles/width_bench.json] [--steps 5] [--launches 20]

1. PPOLearner.learn() step time with both nets at hidden widths (300,)*3, (304,)*3 and (296,)*3, Discrete(90), obs 89,
   one epoch of a 50 000-row batch (bench.py's C2 shape apart from the widths), the three shapes alternated in rounds.
   A 300-wide layer runs as 304 units on the device, so it should cost what 304 costs.
2. rlppo_value_head (training mode: v, dv, dH, dw) at K = 1000, 2048 (the last register form), 2049, 3000 and 4096, at
   50 000 and 1 000 000 rows.  CUDA events around R launches replayed from one CUDA graph; between timed launches a
   256 MB buffer is overwritten, so every launch reads H from HBM (the overwrite is timed separately and subtracted).
   Bytes are the real ones: H read once (2 pad8(K) per row), dH written once (2 pad8(K)), targets in and values out
   (8 per row); w / dw are negligible.
The card name and power limit are read in the same process."""
import argparse
import contextlib
import io
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from wide_head_bench import gpu_info  # noqa: E402

M_LEARN = 50_000
FLUSH_BYTES = 256 << 20


def pad8(n):
    return (n + 7) // 8 * 8


def make_learner(width):
    from rlgym_ppo_b200.ppo import ExperienceBuffer, PPOLearner
    obs, A, M = 89, 90, M_LEARN
    torch.manual_seed(width)
    layers = (width,) * 3
    with contextlib.redirect_stdout(io.StringIO()):
        lr = PPOLearner(obs, A, 0, layers, layers, (0.1, 1.0), M, 1, 3e-4, 3e-4, 0.2, 0.001, M, "cuda:0")
    rng = np.random.RandomState(width)
    buf = ExperienceBuffer(M, 1, "cuda:0")
    buf.submit_experience(rng.randn(M, obs).astype(np.float32), rng.randint(0, A, M).astype(np.float32),
                          np.full(M, -np.log(A), np.float32), np.zeros(M, np.float32), np.zeros((M, obs), np.float32),
                          np.zeros(M, np.float32), np.zeros(M), rng.randn(M).astype(np.float32),
                          rng.randn(M).astype(np.float32))
    return lr, buf


def learn_bench(widths, steps, rounds=5):
    nets = {w: make_learner(w) for w in widths}
    for lr, buf in nets.values():          # warm-up: workspaces, graph capture, kernel configuration
        for _ in range(2):
            lr.learn(buf)
    torch.cuda.synchronize()
    times = {w: [] for w in widths}
    for _ in range(rounds):                # alternate the shapes so that drift on a shared host hits all of them
        for w, (lr, buf) in nets.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                lr.learn(buf)
            torch.cuda.synchronize()
            times[w].append((time.perf_counter() - t0) / steps * 1e3)
    return {str(w): {"ms_per_learn_median": float(np.median(v)), "ms_min": float(min(v)), "ms_max": float(max(v)),
                     "ms_rounds": v, "fused": nets[w][0].policy._stack.fused_ok} for w, v in times.items()}


def timed(fn, n, flush):
    """Median over 5 repeats of (n x [flush; fn] - n x [flush]) / n, each replayed from a CUDA graph, in ms."""
    def graph(body):
        body()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            with torch.cuda.graph(g, stream=side):
                body()
        torch.cuda.current_stream().wait_stream(side)
        return g

    def run(g):
        g.replay()
        torch.cuda.synchronize()
        out = []
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            g.replay()
            e1.record()
            torch.cuda.synchronize()
            out.append(e0.elapsed_time(e1))
        return float(np.median(out))

    def with_fn():
        for _ in range(n):
            flush.add_(1)
            fn()

    def flush_only():
        for _ in range(n):
            flush.add_(1)

    t_both, t_flush = run(graph(with_fn)), run(graph(flush_only))
    return (t_both - t_flush) / n, t_flush / n


def value_head_bench(Ks, rows_list, n_launch):
    from rlgym_ppo_b200 import ops
    flush = torch.zeros(FLUSH_BYTES // 4, device="cuda")
    out = []
    for M in rows_list:
        for K in Ks:
            k8 = pad8(K)
            h = torch.relu(torch.randn(M, k8, device="cuda")).to(torch.bfloat16)
            h[:, K:] = 0
            dh = torch.empty(M, k8, dtype=torch.bfloat16, device="cuda")
            w = torch.randn(K, device="cuda") * 0.05
            b = torch.zeros(1, device="cuda")
            tgt = torch.randn(M, device="cuda")
            v = torch.empty(M, device="cuda")
            dw = torch.zeros(K, device="cuda")
            db = torch.zeros(1, device="cuda")
            metrics = torch.zeros(8, device="cuda")

            def fn():
                ops.value_head(h, w, b, K, values_out=v, targets=tgt, inv_batch=1.0 / M, dh=dh, dw=dw, db=db,
                               metrics=metrics)

            ms, flush_ms = timed(fn, n_launch, flush)
            nbytes = M * (4 * k8 + 8)
            out.append({"K": K, "rows": M, "form": "registers" if K <= 2048 else "shared-memory (wide)",
                        "us": ms * 1e3, "bytes": nbytes, "GBps": nbytes / (ms * 1e-3) / 1e9,
                        "flush_us_subtracted": flush_ms * 1e3})
            print(json.dumps(out[-1]), flush=True)
            del h, dh
            torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "width_bench.json"))
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--launches", type=int, default=20)
    args = ap.parse_args()
    from rlgym_ppo_b200 import _lib
    _lib.require_device()
    res = {"gpu": gpu_info(),
           "value_head": {"method": "CUDA events, graph replay, 256 MB overwritten before each launch (its time "
                                    "subtracted); training mode; bytes = H in + dH out + 8 B/row",
                          "results": value_head_bench((1000, 2048, 2049, 3000, 4096), (50_000, 1_000_000),
                                                      args.launches)},
           "learn": {"rows": M_LEARN, "nets": "policy and critic both 3 hidden layers of the given width, obs 89, "
                                               "Discrete(90), one epoch, batch = minibatch = 50 000",
                     "steps_per_round": args.steps, "by_width": learn_bench((300, 304, 296), args.steps)}}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
