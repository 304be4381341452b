"""`Learner(..., data_parallel=True).learn()` under torchrun (one rank per GPU): python -m torch.distributed.run
--standalone --nproc-per-node N tests/dp_learner_check.py OUT_DIR.  OUT_DIR is shared by the ranks.

For a Discrete and a MultiDiscrete policy with standardize_obs=True it checks that
  * the ranks' first rollouts differ (per-rank environment and sampler seeds);
  * after every iteration the parameter arena, Adam m / v and step counters are the same bits on every rank;
  * the merged observation statistics are the same on every rank and equal a host replay
    (increment_from_serialized_other) of the gathered deltas onto the previous base;
  * Cumulative Timesteps is the sum of the ranks' collected steps, and every rank runs the same number of iterations under
    the global timestep_limit;
  * only rank 0 printed iteration reports and wrote a checkpoint folder;
  * a Learner resuming from "latest" starts, on every rank, from the weights, Adam state and counters saved.
At world size 1 it also checks that the first rollout is byte-identical to that of a data_parallel=False Learner.
The first Learner initialises the process group itself; the last one destroys it in cleanup()."""
import contextlib
import io
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

REPORT = "BEGIN ITERATION REPORT"


def kwargs(folder, world, n_proc=2):
    return dict(n_proc=n_proc, min_inference_size=n_proc, ts_per_iteration=400, exp_buffer_size=1200, ppo_batch_size=400,
                ppo_epochs=2, policy_layer_sizes=(64, 64), critic_layer_sizes=(64, 64), standardize_obs=True,
                standardize_returns=True, checkpoints_save_folder=folder, add_unix_timestamp=True, log_to_wandb=False,
                timestep_limit=1000 * world, save_every_ts=1000 * world, ppo_ent_coef=0.01)


def gather(t):
    t = t.contiguous()
    out = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(out, t)
    return out


def all_same(t):
    return all(torch.equal(g, gather(t)[0]) for g in gather(t))


def state(lrn):
    p = lrn.ppo_learner
    return [p._params, p._m, p._v, p._steps]


def saved_state(lrn):
    """What a checkpoint holds of state(): the two nets' segments (the data-parallel arenas carry a metric segment)."""
    p, n = lrn.ppo_learner, lrn.ppo_learner._n_net
    return [p._params[:n], p._m[:n], p._v[:n], p._steps[:2]]


def host_stats(st):
    """(count, mean, m2) host copies of a WelfordRunningStat."""
    return int(st.count), np.array(st.running_mean, np.float32).ravel(), np.array(st.running_variance, np.float32).ravel()


def replay(base, blocks, stride, world, dim):
    """The host merge of every rank's gathered delta block onto `base` (count, mean, m2), in rank order."""
    from rlgym_ppo_b200.util import WelfordRunningStat
    ref = WelfordRunningStat(dim)
    ref.count, ref.running_mean, ref.running_variance = base[0], base[1].copy(), base[2].copy()
    raw = blocks.cpu().numpy()
    for r in range(world):
        b = raw[r * stride:(r + 1) * stride]
        count = int(b[0:8].view(np.int64)[0])
        f = b[8:8 + 8 * dim].view(np.float32)
        ref.increment_from_serialized_other(f[:dim].tolist() + f[dim:].tolist() + [count])
    return host_stats(ref)


def instrument(lrn, log):
    """Wrap one Learner's collection, exchange and iteration with the cross-rank checks."""
    from rlgym_ppo_b200 import parallel
    world, dev = dist.get_world_size(), torch.device(lrn.device)
    collect, iteration, exchange = lrn.agent.collect_timesteps, lrn._iteration, parallel.exchange
    seen = {}

    def collect_hook(n):
        out = collect(n)
        seen["n_steps"] = out[2]
        if "first" not in log:
            log["first"] = [x.detach().cpu().clone() for x in out[0]]
        return out

    def exchange_hook(block, tail, group=None):
        blocks, stride, tails = exchange(block, tail, group)
        seen["gathered"] = (blocks.clone(), stride)
        return blocks, stride, tails

    def iteration_hook():
        base = host_stats(lrn._obs_base)
        cum0 = lrn.agent.cumulative_timesteps
        parallel.exchange = exchange_hook
        try:
            steps = iteration()
        finally:
            parallel.exchange = exchange
        own = torch.tensor([seen["n_steps"]], dtype=torch.int64, device=dev)
        per_rank = [int(x) for x in gather(own)]
        assert steps == sum(per_rank) and lrn.agent.cumulative_timesteps == cum0 + sum(per_rank), (steps, per_rank)
        for t in state(lrn):
            assert all_same(t), "replicas diverged"
        merged = lrn._obs_base.device_block()
        dim = lrn._obs_base._dim
        assert torch.equal(lrn.agent.obs_stats.device_block()[:8 + 8 * dim], merged[:8 + 8 * dim])
        assert all_same(merged[:8 + 8 * dim]), "merged observation statistics differ between ranks"
        blocks, stride = seen["gathered"]
        want, got = replay(base, blocks, stride, world, dim), host_stats(lrn._obs_base)
        assert want[0] == got[0] and np.array_equal(want[1].view(np.uint32), got[1].view(np.uint32)) \
            and np.array_equal(want[2].view(np.uint32), got[2].view(np.uint32)), "merge differs from the host replay"
        assert lrn.agent.obs_delta.count == 0
        log.setdefault("t_exchange", []).append(lrn._t_exchange)
        log["iterations"] = log.get("iterations", 0) + 1
        return steps

    lrn.agent.collect_timesteps = collect_hook
    lrn._iteration = iteration_hook


def run(kind, make_env, out_dir, first_learner, last_learner):
    from rlgym_ppo_b200 import Learner
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    base = os.path.join(out_dir, kind, "run")
    text = io.StringIO()
    log = {}
    with contextlib.redirect_stdout(text):
        lrn = Learner(make_env, checkpoint_load_folder=None, data_parallel=True, **kwargs(base, world))
    if first_learner:
        assert lrn._owns_group and dist.is_initialized()
        lrn._owns_group = False         # the checks below keep using the group
    assert lrn.world_size == world and lrn.rank == rank and lrn.data_parallel == (world > 1)
    assert lrn.device == f"cuda:{int(os.environ['LOCAL_RANK'])}"
    if world == 1:
        with contextlib.redirect_stdout(text):
            lrn.learn()
        out = text.getvalue()
        assert "LEARNING LOOP ENCOUNTERED AN ERROR" not in out and out.count(REPORT) >= 2, out[-3000:]
        return lrn, log, out
    assert lrn.ppo_learner.dp_mode == "sharded" and lrn.ppo_learner.world_size == world
    instrument(lrn, log)
    with contextlib.redirect_stdout(text):
        lrn.learn()
    out = text.getvalue()
    assert "LEARNING LOOP ENCOUNTERED AN ERROR" not in out, out[-3000:]
    first = log["first"][0][:16].to(lrn.device)
    firsts = gather(first)
    assert not any(torch.equal(firsts[0], f) for f in firsts[1:]), "ranks collected the same first rollout"
    its = gather(torch.tensor([log["iterations"]], device=lrn.device))
    assert all(int(i) == int(its[0]) for i in its) and int(its[0]) >= 2
    assert lrn.agent.cumulative_timesteps >= lrn.timestep_limit
    reports = [int(x) for x in gather(torch.tensor([out.count(REPORT)], device=lrn.device))]
    assert reports == [log["iterations"]] + [0] * (world - 1), reports
    dist.barrier()
    runs = [d for d in os.listdir(os.path.dirname(base)) if d.startswith("run-")]
    assert runs == [os.path.basename(lrn.checkpoints_save_folder)], runs        # rank 0's folder, and only that one
    final = [t.clone() for t in saved_state(lrn)]
    counters = (lrn.agent.cumulative_timesteps, lrn.ppo_learner.cumulative_model_updates)
    assert all_same(torch.tensor(counters, device=lrn.device))
    base_stats = host_stats(lrn._obs_base)
    dist.barrier()

    # ---- resume from "latest": every rank loads the folder rank 0 resolved ----
    text2 = io.StringIO()
    with contextlib.redirect_stdout(text2):
        res = Learner(make_env, checkpoint_load_folder="latest", data_parallel=True,
                      **dict(kwargs(base, world), timestep_limit=counters[0] + 1))
    for a, b in zip(saved_state(res), final):
        assert torch.equal(a, b), "resumed state differs from the saved one"
    for t in state(res):
        assert all_same(t)
    assert (res.agent.cumulative_timesteps, res.ppo_learner.cumulative_model_updates) == counters
    with open(os.path.join(lrn.checkpoints_save_folder, str(counters[0]), "BOOK_KEEPING_VARS.json")) as f:
        book = json.load(f)
    assert book["cumulative_timesteps"] == counters[0] and res.return_stats.count == book["reward_running_stats"]["count"]
    assert res.epoch == book["epoch"] == lrn.epoch - 1          # saved before the loop counts the iteration
    assert book["obs_running_stats"]["count"] == base_stats[0]
    got = host_stats(res._obs_base)
    assert got[0] == base_stats[0] and np.array_equal(got[1], base_stats[1]) and np.array_equal(got[2], base_stats[2])
    assert res.agent.obs_delta.count == 0
    if last_learner:
        res._owns_group = True          # its cleanup() destroys the group
        instrument(res, {})
        with contextlib.redirect_stdout(text2):
            res.learn()
        assert not dist.is_initialized()
    else:
        res.cleanup()
    return lrn, log, out


def first_rollout_matches_plain(out_dir):
    """World size 1: data_parallel=True is the data_parallel=False path (same seeds, same first rollout)."""
    from rlgym_ppo_b200 import Learner
    from tests.seeded_env import make_env
    rollouts = []
    for dp in (True, False):
        with contextlib.redirect_stdout(io.StringIO()):
            lrn = Learner(make_env, checkpoint_load_folder=None, data_parallel=dp,
                          **kwargs(os.path.join(out_dir, f"plain{int(dp)}", "run"), 1, n_proc=1))
        try:
            rollouts.append([x.detach().cpu().clone() for x in lrn.agent.collect_timesteps(400)[0]])
        finally:
            lrn.cleanup()
    for a, b in zip(*rollouts):
        assert a.dtype == b.dtype and a.shape == b.shape and torch.equal(a.view(torch.uint8), b.view(torch.uint8))


def main():
    from tests.seeded_env import make_env, make_env_md
    out_dir = sys.argv[1]
    world = int(os.environ["WORLD_SIZE"])
    rank = int(os.environ["RANK"])
    assert not dist.is_initialized()
    _, log_d, _ = run("discrete", make_env, out_dir, first_learner=True, last_learner=False)
    if world == 1:
        first_rollout_matches_plain(out_dir)
    _, log_md, _ = run("multi_discrete", make_env_md, out_dir, first_learner=False, last_learner=world > 1)
    if world == 1:
        dist.destroy_process_group()
    if rank == 0:
        t = sorted(log_d.get("t_exchange", []) + log_md.get("t_exchange", []))
        med = f"{1e3 * t[len(t) // 2]:.3f} ms over {len(t)} iterations" if t else "n/a"
        print(f"dp_learner_check OK world={world} collective={os.environ.get('RLPPO_DP_COLLECTIVE', 'auto')} "
              f"exchange+merge (host clock, synchronised) median {med}", flush=True)


if __name__ == "__main__":
    main()
