"""The host protocol of Learner(data_parallel=True) on CPU: world size 2 over gloo (spawned processes, 127.0.0.1
rendezvous).  Seeds per rank, the per-iteration exchange tail, the aggregated report, the loop decision and the
checkpoint folders every rank agrees on."""
import os
import socket
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_rank_seeds_keep_rank_zero():
    from rlgym_ppo_b200 import parallel
    assert parallel.rank_seeds(123, 0, 8) == (123, 123)                  # rank 0: the single-process seeds
    assert parallel.rank_seeds(123, 1, 8) == (131, 124)
    assert parallel.rank_seeds(123, 3, 4) == (135, 126)
    # environment seeds random_seed + r * n_proc + proc_id: disjoint over ranks and processes
    env = [parallel.rank_seeds(7, r, 5)[0] + p for r in range(4) for p in range(5)]
    assert sorted(env) == list(range(7, 27))
    key = 0x1234_5678_9ABC_DEF
    keys = [parallel.sampler_seed(key, r) for r in range(8)]
    assert keys[0] == key and len(set(keys)) == 8 and all(0 <= k < 1 << 62 for k in keys)


def test_tail_pack_and_combine():
    from rlgym_ppo_b200 import parallel
    t0 = parallel.pack_tail(600, 0.25, 1.5, False)
    t1 = parallel.pack_tail(612, 0.5, None, False)
    assert t0.dtype == np.float64 and len(t0) == len(parallel.TAIL)
    assert list(t1) == [612, 0.5, 0.0, 0.0, 0.0]
    agg = parallel.combine_tails(np.stack([t0, t1]))
    assert agg == {"steps": 1212, "collect_time": 0.5, "average_reward": 1.5, "failed": []}
    agg = parallel.combine_tails(np.stack([parallel.pack_tail(0, 0.1, None, False), parallel.pack_tail(0, 0.1, None, True)]))
    assert agg["average_reward"] is None and agg["failed"] == [1]
    rep = parallel.collection_report({"steps": 1212, "collect_time": 0.5, "average_reward": 2.0, "failed": []}, 2.0)
    assert rep == {"Timesteps Collected": 1212, "Timestep Collection Time": 0.5, "Timestep Consumption Time": 1.5,
                   "Collected Steps per Second": 2424.0, "Overall Steps per Second": 606.0, "Policy Reward": 2.0}
    assert np.isnan(parallel.collection_report(dict(agg, steps=5, collect_time=1.0), 2.0)["Policy Reward"])


def _learner_stub(folder, stamp):
    return SimpleNamespace(checkpoints_save_folder=f"{folder}-{stamp}", add_unix_timestamp=True)


def _worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from rlgym_ppo_b200 import parallel
        from rlgym_ppo_b200.learner import Learner
        res = {}
        # ---- the exchange: one all-gather of [Welford block | f64 tail] -------------------------------------------------
        dim = 3
        block = torch.zeros(8 + 16 * dim, dtype=torch.uint8)
        block[0:8].view(torch.int64).fill_(10 + rank)
        block[8:].view(torch.float32)[:dim] = torch.arange(dim, dtype=torch.float32) + rank
        reward = 1.0 + rank if rank == 0 else None
        tail = parallel.pack_tail(100 + rank, 0.1 * (rank + 1), reward, error=(rank == 1 and out_dir.endswith("fail")))
        blocks, stride, tails = parallel.exchange(block, tail)
        assert stride == block.numel() + 8 * len(parallel.TAIL) and blocks.numel() == world * stride
        res["counts"] = [int(blocks[r * stride:r * stride + 8].view(torch.int64)) for r in range(world)]
        res["means"] = [blocks[r * stride + 8:r * stride + 8 + 4 * dim].view(torch.float32).tolist() for r in range(world)]
        res["agg"] = parallel.combine_tails(tails)
        # tails only (no observation statistics): an empty block
        _, s2, t2 = parallel.exchange(torch.empty(0, dtype=torch.uint8), parallel.pack_tail(7, 1.0, None, False))
        res["empty"] = (s2, t2.tolist())
        # ---- Learner._learn's loop on the exchanged numbers: the global timestep_limit, and a failure on one rank ------
        cum, its = 0, 0
        fail = out_dir.endswith("fail")
        while True:
            _, _, t = parallel.exchange(torch.empty(0, dtype=torch.uint8),
                                        parallel.pack_tail(300 + 50 * rank, 0.1, None, fail and rank == 1 and its == 1))
            agg = parallel.combine_tails(t)
            cum += agg["steps"]
            its += 1
            if agg["failed"] or cum >= 2000:      # _iteration_dp raises on a failure; the while condition is the limit
                break
        res["loop"] = (cum, its)
        # ---- checkpoint folders: rank 0's save folder and its resolution of "latest" ----------------------------------
        base = os.path.join(out_dir, "ckpt", "run")
        for stamp, steps in ((111, (500, 1000)), (222, (700,))):
            for st in steps:
                os.makedirs(f"{base}-{stamp}/{st}", exist_ok=True)
        dist.barrier()
        me = _learner_stub(base, 1000 + rank)
        res["folders"] = parallel.agree_on_folders(me.checkpoints_save_folder, "latest",
                                                   lambda: Learner._latest_checkpoint(me))
        res["explicit"] = parallel.agree_on_folders(me.checkpoints_save_folder, "/some/folder" if rank == 0 else None,
                                                    lambda: None)
        # ---- metrics of every rank on rank 0, in rank order --------------------------------------------------------
        res["metrics"] = parallel.gather_metrics([np.full(2, rank, np.float32)] * (rank + 1))
        torch.save(res, os.path.join(out_dir, f"r{rank}.pt"))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("case", ["ok", "fail"])
def test_protocol_world_two(tmp_path, case):
    world = 2
    out = str(tmp_path / case)
    os.makedirs(out)
    mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    r = [torch.load(os.path.join(out, f"r{i}.pt"), weights_only=False) for i in range(world)]
    for i in range(world):
        assert r[i]["counts"] == [10, 11] and r[i]["means"] == [[0.0, 1.0, 2.0], [1.0, 2.0, 3.0]]
        assert r[i]["agg"] == r[0]["agg"]
        assert r[i]["agg"]["steps"] == 201 and r[i]["agg"]["collect_time"] == pytest.approx(0.2)
        assert r[i]["agg"]["average_reward"] == 1.0                      # only rank 0 has a value
        assert r[i]["agg"]["failed"] == ([1] if case == "fail" else [])
        assert r[i]["empty"] == (40, [[7.0, 1.0, 0.0, 0.0, 0.0]] * 2)
        # 650 steps per iteration over both ranks: the global limit of 2000 ends every rank's loop after 4 iterations;
        # rank 1 failing in the second iteration ends both loops there
        assert r[i]["loop"] == ((1300, 2) if case == "fail" else (2600, 4))
        save, load = r[i]["folders"]
        assert save == str(tmp_path / case / "ckpt" / "run") + "-1000"          # rank 0's time-stamped folder
        assert load == str(tmp_path / case / "ckpt" / "run") + "-222/700"       # newest run, most steps
        assert r[i]["explicit"] == (save, "/some/folder")
    metrics = r[0]["metrics"]
    assert [float(m[0]) for m in metrics] == [0.0, 1.0, 1.0] and r[1]["metrics"] is None
