"""Host-side data-parallel bookkeeping (one process per GPU; torch.distributed carries the collectives: NCCL on the
GPUs, gloo in the CPU tests).  No tensor math here beyond the collectives themselves.

The reference has no distributed mode (SURVEY.md 2.2); the seam is its gradient accumulation over minibatch slices
(ppo_learner.py:134-193), which sums (mb/B)-scaled minibatch gradients before ONE clip + Adam step.
"""
import os

import numpy as np
import torch
import torch.distributed as dist


def world(group=None):
    """(world_size, rank) of the initialised process group, (1, 0) without one."""
    if dist.is_available() and dist.is_initialized():
        return dist.get_world_size(group), dist.get_rank(group)
    return 1, 0


def rank_rows(k, batch_size, rank, world_size, mode):
    """Rows of the epoch's permutation that `rank` consumes for optimiser step k: (first, count).

    replicated: every rank holds the same buffer and the same permutation; batch k = perm[k*B : (k+1)*B] is cut into
                world_size consecutive slices -- the reference's minibatch slices with mini_batch_size = B / world_size.
    sharded:    every rank holds its own buffer and permutation and consumes a whole per-rank batch."""
    if mode == "sharded" or world_size == 1:
        return k * batch_size, batch_size
    assert batch_size % world_size == 0, "batch_size must be a multiple of the number of ranks"
    local = batch_size // world_size
    return k * batch_size + rank * local, local


def gae_chunk(n, rank, world_size, align=64):
    """Contiguous chunk [lo, hi) of an n-step flat rollout that `rank` scans when GAE is sharded (SURVEY.md 8e: the
    recurrence is an associative affine scan, so the step axis can be cut anywhere).  Chunks are `m` steps long (a
    multiple of `align`, so every chunk starts 16-byte aligned in f32 and f64 arrays), the last ones may be short or
    empty.  Returns (lo, hi, m)."""
    m = -(-int(n) // int(world_size))
    m = -(-m // align) * align
    lo = min(int(n), rank * m)
    hi = min(int(n), lo + m)
    return lo, hi, m


def samples_per_step(batch_size, world_size, mode):
    """Number of samples one optimiser step averages over (the B of the 1/B gradient weight)."""
    return batch_size * world_size if (mode == "sharded" and world_size > 1) else batch_size


ONE_SHOT_BYTES = 16 << 20


def choose_collective(world_size, n_params, requested=None, env=None):
    """How data-parallel ranks exchange gradients: "none" (one rank), "p2p" (summed inside the optimiser launch from the
    peers' symmetric-memory arenas: rlppo_norm_clip_adam_peers) or "nccl" (all_reduce on the flat arena).

    The one-shot peer exchange makes every rank read all (R-1) peer arenas, (R-1) * 4 * n bytes over NVLink per step:
    latency-optimal for the example-size nets.  Big arenas take the two-shot form "p2p2" (rlppo_norm_clip_adam_peers2:
    every rank reduces 1/R of the arena from all peers, then reads the reduced slices -- 2 * 4 * n bytes however many ranks
    there are), still inside the optimiser launch, so a whole learn() stays one CUDA graph.  Round 2 on 8 x B200 with the
    60 MB arena of the 2048-2048-1024-1024 nets: 52.4 ms/step against 54.1 ms with the NCCL all-reduce between two graphs;
    validated by tests/dp_check.py (sum equal to NCCL's to rounding, same bits on every rank, 1500 launches under random
    per-rank skew).  Peer mappings exist inside one box only (at most 8 ranks): beyond that, and whenever the mappings
    cannot be set up, NCCL.  `requested` (constructor argument) wins over `env` (RLPPO_DP_COLLECTIVE) which wins over the
    size rule."""
    if world_size <= 1:
        return "none"
    auto = "p2p" if (world_size - 1) * 4 * int(n_params) <= ONE_SHOT_BYTES else "p2p2"
    choice = requested or env or auto
    if choice not in ("p2p", "nccl", "p2p2"):
        raise ValueError(f"dp_collective must be 'p2p', 'nccl' or 'p2p2', got {choice!r}")
    if choice in ("p2p", "p2p2") and world_size > 8:
        choice = "nccl"
    return choice


def allreduce_sum_(t, group=None):
    """In-place sum over ranks (flat gradient arena, metric sums); identity without a process group."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t


def report_from_sums(sums):
    """sums: the 8 metric accumulators of rlppo_policy_head_train / rlppo_value_head summed over ranks and minibatches
    -> the four averaged report entries of ppo_learner.py:204-210 (equal-size minibatches: mean of means = total mean)."""
    s = [float(x) for x in sums]
    rows_p = s[4] if s[4] > 0 else 1.0
    rows_v = s[6] if s[6] > 0 else 1.0
    return {"Policy Entropy": s[0] / rows_p, "Mean KL Divergence": s[1] / rows_p, "SB3 Clip Fraction": s[2] / rows_p,
            "Value Function Loss": s[5] / rows_v}


# ---- Learner(data_parallel=True): one learner on every GPU of a box, one process per GPU under torchrun -----------------
# Each rank collects its own rollouts (weak scaling, dp_mode="sharded").  Once per iteration the ranks exchange, in ONE
# all-gather, their observation-statistics increments (a Welford device block) and a small f64 tail:
TAIL = ("steps", "collect_time", "average_reward", "has_reward", "error")


def init_torchrun():
    """(created, local_rank): joins the process group of a torchrun launch.  An initialised group is used as it is
    (created = False); without one, NCCL is initialised from the torchrun environment.  Without a torchrun environment
    there is one process: (False, None).  The current CUDA device becomes cuda:LOCAL_RANK whenever LOCAL_RANK is set."""
    local = os.environ.get("LOCAL_RANK")
    local = None if local is None else int(local)
    if local is not None:
        torch.cuda.set_device(local)
    if dist.is_available() and dist.is_initialized():
        return False, local
    if local is None or "WORLD_SIZE" not in os.environ:
        return False, None
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return True, local


def rank_seeds(random_seed, rank, n_proc):
    """(environment seed base, experience-buffer seed) of `rank`: its workers are seeded base + proc_id, i.e.
    random_seed + rank * n_proc + proc_id, and its buffer random_seed + rank.  Rank 0 keeps the single-process seeds."""
    return random_seed + rank * n_proc, random_seed + rank


def sampler_seed(seed, rank):
    """Key of `rank`'s policy sampler (Philox) from the key every rank drew: rank 0 keeps it, the others mix in their
    rank so that no two ranks sample the same action stream."""
    if rank == 0:
        return seed
    return (seed ^ (rank * 0x9E3779B97F4A7C15)) % (1 << 62)


def pack_tail(steps, collect_time, average_reward, error):
    """This rank's f64 tail (TAIL order); average_reward None (no episode finished yet) is sent as has_reward = 0."""
    has = average_reward is not None
    return np.array([steps, collect_time, average_reward if has else 0.0, float(has), float(bool(error))], np.float64)


def combine_tails(tails):
    """tails f64 [world, len(TAIL)] in rank order -> what every rank acts on: the global step count, the slowest
    collection, the mean of the ranks' average rewards (None when no rank has one), the ranks that failed."""
    t = np.asarray(tails, np.float64).reshape(-1, len(TAIL))
    rew = t[t[:, 3] != 0, 2]
    return {"steps": int(round(t[:, 0].sum())), "collect_time": float(t[:, 1].max()),
            "average_reward": float(rew.mean()) if len(rew) else None,
            "failed": [int(r) for r in np.flatnonzero(t[:, 4] != 0)]}


def collection_report(agg, total_time):
    """The collection entries of the iteration report (learner.py:275-296) over all ranks: global steps over the slowest
    rank's collection time, and over this rank's iteration time."""
    steps, t_collect = agg["steps"], agg["collect_time"]
    return {"Timesteps Collected": steps, "Timestep Collection Time": t_collect,
            "Timestep Consumption Time": total_time - t_collect,
            "Collected Steps per Second": steps / t_collect if t_collect > 0 else float("nan"),
            "Overall Steps per Second": steps / total_time if total_time > 0 else float("nan"),
            "Policy Reward": np.nan if agg["average_reward"] is None else agg["average_reward"]}


def exchange(block, tail, group=None):
    """ONE all-gather of [block bytes | tail f64] from every rank.  block: uint8 tensor (8-byte multiple; may be empty) on
    the collective's device; tail: f64 array.  Returns (gathered uint8 [world * stride], stride in bytes, tails f64
    [world, len(tail)] on the host)."""
    nb = int(block.numel())
    assert block.dtype == torch.uint8 and nb % 8 == 0
    tail = torch.from_numpy(np.ascontiguousarray(tail, np.float64))
    stride = nb + 8 * int(tail.numel())
    world = dist.get_world_size(group)
    send = torch.empty(stride, dtype=torch.uint8, device=block.device)
    send[:nb].copy_(block)
    send[nb:].view(torch.float64).copy_(tail)
    out = torch.empty(world * stride, dtype=torch.uint8, device=block.device)
    dist.all_gather_into_tensor(out, send, group=group)
    tails = out.view(world, stride)[:, nb:].contiguous().view(torch.float64).cpu().numpy()
    return out, stride, tails


def agree_on_folders(save_folder, load_folder, resolve_latest, group=None):
    """Rank 0's checkpoint folders on every rank: its (time-stamped) save folder, and the folder to load, with "latest"
    resolved by rank 0 (resolve_latest(); None when there is nothing to load)."""
    if dist.get_rank(group) == 0 and load_folder == "latest":
        load_folder = resolve_latest()
    obj = [save_folder, load_folder]
    dist.broadcast_object_list(obj, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
    return obj[0], obj[1]


def gather_metrics(metrics, group=None):
    """Every rank's collected metrics, concatenated in rank order, on rank 0 (None on the others)."""
    rank = dist.get_rank(group)
    out = [None] * dist.get_world_size(group) if rank == 0 else None
    dist.gather_object(metrics, out, dst=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
    return [m for ms in out for m in ms] if rank == 0 else None
