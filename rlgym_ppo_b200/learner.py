"""Learner: the `Learner(env_fn).learn()` surface of rlgym_ppo/learner.py over the B200 learner path.

Constructor keywords, defaults, public attributes, report keys and checkpoint files are the reference's
(learner.py:29-78, 169-189, 275-296, 387-564).  Environment stepping stays on host processes
(batched_agents.BatchedAgentManager); everything between "rollout arrays are on the host" and "weights updated"
runs on the device without a host round trip:

  add_new_experience (learner.py:330-385)
    7 rollout arrays --one async H2D each--> HBM
    [states ; next_states[-1]] -> bf16 rows -> value net (tcgen05 GEMMs + fused value head) -> V[N+1]
    rlppo_gae_f32: segmented reverse scan, reward / return_std clip fused, std read from the device Welford state
    rlppo_welford_update on the first min(150, N) returns (f64, as the reference's Python floats)
    rlppo_ring_append x9 into the ExperienceBuffer rings
  PPOLearner.learn: see ppo/ppo_learner.py
"""
import json
import os
import random
import shutil
import time
from typing import Tuple, Union

import numpy as np
import torch

from . import _lib, ops, parallel
from ._graphs import GraphCache
from ._staging import Stager
from .ppo import ExperienceBuffer, PPOLearner
from .util import WelfordRunningStat

_EXP_FIELDS = ("states", "actions", "log_probs", "rewards", "next_states", "dones", "truncated")


def _f32(t):
    return t if t.dtype == torch.float32 else t.to(torch.float32)


def _staged_dtype(x):
    """dtype a rollout array keeps on the device: f32/f64 as given (the kernels cast f64 like torch.as_tensor(...,
    dtype=float32) does), anything else is converted to f32 on the host first (see Stager.to_device)."""
    dt = x.dtype if hasattr(x, "dtype") else np.asarray(x).dtype
    if dt in (torch.float64, np.float64) or str(dt) in ("float64", "torch.float64"):
        return torch.float64
    return torch.float32


class Learner(object):
    def __init__(
            # fmt: off
            self,
            env_create_function,
            metrics_logger=None,
            n_proc: int = 8,
            min_inference_size: int = 80,
            render: bool = False,
            render_delay: float = 0,
            timestep_limit: int = 5_000_000_000,
            exp_buffer_size: int = 100000,
            ts_per_iteration: int = 50000,
            standardize_returns: bool = True,
            standardize_obs: bool = True,
            max_returns_per_stats_increment: int = 150,
            steps_per_obs_stats_increment: int = 5,
            policy_layer_sizes: Tuple[int, ...] = (256, 256, 256),
            critic_layer_sizes: Tuple[int, ...] = (256, 256, 256),
            continuous_var_range: Tuple[float, ...] = (0.1, 1.0),
            ppo_epochs: int = 10,
            ppo_batch_size: int = 50000,
            ppo_minibatch_size: Union[int, None] = None,
            ppo_ent_coef: float = 0.005,
            ppo_clip_range: float = 0.2,
            gae_lambda: float = 0.95,
            gae_gamma: float = 0.99,
            policy_lr: float = 3e-4,
            critic_lr: float = 3e-4,
            log_to_wandb: bool = False,
            load_wandb: bool = True,
            wandb_run=None,
            wandb_project_name: Union[str, None] = None,
            wandb_group_name: Union[str, None] = None,
            wandb_run_name: Union[str, None] = None,
            checkpoints_save_folder: Union[str, None] = None,
            add_unix_timestamp: bool = True,
            checkpoint_load_folder: Union[str, None] = "latest",  # "latest" loads latest checkpoint
            save_every_ts: int = 1_000_000,
            instance_launch_delay: Union[float, None] = None,
            random_seed: int = 123,
            n_checkpoints_to_keep: int = 5,
            shm_buffer_size: int = 8192,
            device: str = "auto",
            data_parallel: bool = False):
        assert (
                env_create_function is not None
        ), "MUST PROVIDE A FUNCTION TO CREATE RLGYM FUNCTIONS TO INITIALIZE RLGYM-PPO"

        # data_parallel: one Learner per GPU under torchrun, trained as one (weak scaling, see INTEGRATION.md).  At world
        # size 1 nothing below differs from data_parallel=False.
        self._owns_group, local_rank = parallel.init_torchrun() if data_parallel else (False, None)
        self.world_size, self.rank = parallel.world() if data_parallel else (1, 0)
        self.data_parallel = self.world_size > 1
        if checkpoints_save_folder is None:
            checkpoints_save_folder = os.path.join("data", "checkpoints", "rlgym-ppo-run")
        self.add_unix_timestamp = add_unix_timestamp
        if add_unix_timestamp:
            checkpoints_save_folder = f"{checkpoints_save_folder}-{time.time_ns()}"

        torch.manual_seed(random_seed)
        np.random.seed(random_seed)
        random.seed(random_seed)

        self.n_checkpoints_to_keep = n_checkpoints_to_keep
        self.checkpoints_save_folder = checkpoints_save_folder
        self.max_returns_per_stats_increment = max_returns_per_stats_increment
        self.metrics_logger = metrics_logger
        self.standardize_returns = standardize_returns
        self.save_every_ts = save_every_ts
        self.ts_since_last_save = 0
        if self.data_parallel:
            # one run: rank 0's save folder, and the checkpoint rank 0 resolves "latest" to, on every rank
            self.checkpoints_save_folder, checkpoint_load_folder = parallel.agree_on_folders(
                checkpoints_save_folder, checkpoint_load_folder, self._latest_checkpoint)

        # There is no CPU learner here: "auto"/"gpu" pick the current CUDA device, anything else must name one.
        _lib.require_device()
        if device in {"auto", "gpu"}:
            self.device = "cuda:%d" % torch.cuda.current_device()
        elif "cuda" in str(device):
            self.device = device
        else:
            raise _lib.RlppoError(f"device {device!r}: rlgym_ppo_b200 runs on a B200 only (no CPU fallback)")
        if local_rank is not None and torch.device(self.device).index not in (None, local_rank):
            raise _lib.RlppoError(f"device {device!r}: a data-parallel rank runs on its torchrun GPU, cuda:{local_rank}")
        print(f"Using device {self.device}")

        self.exp_buffer_size = exp_buffer_size
        self.timestep_limit = timestep_limit
        self.ts_per_epoch = ts_per_iteration
        self.gae_lambda = gae_lambda
        self.gae_gamma = gae_gamma
        self.return_stats = WelfordRunningStat(1, device=self.device)
        self.epoch = 0

        env_seed, buffer_seed = (parallel.rank_seeds(random_seed, self.rank, n_proc) if self.data_parallel
                                 else (random_seed, random_seed))
        self.experience_buffer = ExperienceBuffer(self.exp_buffer_size, seed=buffer_seed, device=self.device)

        print("Initializing processes...")
        from .batched_agents import BatchedAgentManager
        collect_metrics_fn = None if metrics_logger is None else self.metrics_logger.collect_metrics
        self.agent = BatchedAgentManager(
            None, min_inference_size=min_inference_size,
            seed=env_seed,
            standardize_obs=standardize_obs,
            steps_per_obs_stats_increment=steps_per_obs_stats_increment,
            device=self.device,
            keep_obs_delta=self.data_parallel,
        )
        obs_space_size, act_space_size, action_space_type = self.agent.init_processes(
            n_processes=n_proc,
            build_env_fn=env_create_function,
            collect_metrics_fn=collect_metrics_fn,
            spawn_delay=instance_launch_delay,
            render=render,
            render_delay=render_delay,
            shm_buffer_size=shm_buffer_size,
        )
        obs_space_size = np.prod(obs_space_size)
        print("Initializing PPO...")
        if ppo_minibatch_size is None:
            ppo_minibatch_size = ppo_batch_size

        self.ppo_learner = PPOLearner(
            obs_space_size,
            act_space_size,
            device=self.device,
            batch_size=ppo_batch_size,
            mini_batch_size=ppo_minibatch_size,
            n_epochs=ppo_epochs,
            continuous_var_range=continuous_var_range,
            policy_type=action_space_type,
            policy_layer_sizes=policy_layer_sizes,
            critic_layer_sizes=critic_layer_sizes,
            policy_lr=policy_lr,
            critic_lr=critic_lr,
            clip_range=ppo_clip_range,
            ent_coef=ppo_ent_coef,
            **(dict(process_group=torch.distributed.group.WORLD, dp_mode="sharded") if self.data_parallel else {}),
        )
        if self.data_parallel:
            # after the nets are built, so that the initial weights do not depend on the rank
            policy = self.ppo_learner.policy
            policy._seed = parallel.sampler_seed(policy._seed, self.rank)

        self.agent.policy = self.ppo_learner.policy

        # hyper-parameters the reference records (and hands to wandb), learner.py:169-189
        hp = locals()
        self.config = {k: hp[k] for k in (
            "n_proc", "min_inference_size", "timestep_limit", "exp_buffer_size", "ts_per_iteration",
            "standardize_returns", "standardize_obs", "policy_layer_sizes", "critic_layer_sizes", "ppo_epochs",
            "ppo_batch_size", "ppo_minibatch_size", "ppo_ent_coef", "ppo_clip_range", "gae_lambda", "gae_gamma",
            "policy_lr", "critic_lr", "shm_buffer_size")}

        self.wandb_run = wandb_run if self.rank == 0 else None
        self._obs_loaded = False
        wandb_loaded = checkpoint_load_folder is not None and self.load(checkpoint_load_folder,
                                                                        load_wandb and self.rank == 0, policy_lr,
                                                                        critic_lr)
        if self.data_parallel:
            self._start_replicas()

        if log_to_wandb and self.rank == 0 and self.wandb_run is None and not wandb_loaded:
            import wandb
            print("Attempting to create new wandb run...")
            self.wandb_run = wandb.init(project=wandb_project_name or "rlgym-ppo",
                                        group=wandb_group_name or "unnamed-runs",
                                        name=wandb_run_name or "rlgym-ppo-run", config=self.config, reinit=True)
            print("Created new wandb run!", self.wandb_run.id)
        print("Learner successfully initialized!")

    def update_learning_rate(self, new_policy_lr=None, new_critic_lr=None):
        """Set the learning rate of either optimiser (learner.py:205-216).  The device copy of the rates is refreshed by
        PPOLearner._sync_lr at the next learn()."""
        targets = (("policy", "policy_lr", new_policy_lr, self.ppo_learner.policy_optimizer),
                   ("critic", "critic_lr", new_critic_lr, self.ppo_learner.value_optimizer))
        for label, attr, lr, optimizer in targets:
            if lr is None:
                continue
            setattr(self, attr, lr)
            for group in optimizer.param_groups:
                group["lr"] = lr
            print(f"New {label} learning rate: {lr}")

    def _start_replicas(self):
        """Data parallel: every rank starts from rank 0's parameter arena, Adam moments and step counters (after any
        checkpoint load), and from the same observation statistics: the loaded ones, else none (the increments each rank
        made so far, its reset observations, are in its delta and enter the first merge)."""
        import torch.distributed as dist
        ppo = self.ppo_learner
        for t in (ppo._params, ppo._m, ppo._v, ppo._steps):
            dist.broadcast(t, src=0)
        ppo.policy._stack.refresh_operands(force=True)
        ppo.value_net._stack.refresh_operands(force=True)
        self._obs_base = None
        if self.agent.standardize_obs:
            self._obs_base = WelfordRunningStat(self.agent.obs_stats.shape, device=self.device)
            if self._obs_loaded:
                self._obs_base.copy_device_(self.agent.obs_stats)
                self.agent.obs_delta.reset()
        self._t_exchange = None

    def learn(self):
        """Run iterations until the timestep limit; on an exception print it, try to checkpoint, and always release the
        workers (the contract of learner.py:218-238)."""
        try:
            self._learn()
        except Exception:
            import traceback
            print("\n\nLEARNING LOOP ENCOUNTERED AN ERROR\n")
            traceback.print_exc()
            try:
                self.save(self.agent.cumulative_timesteps)
            except Exception:  # noqa: BLE001
                print("FAILED TO SAVE ON EXIT")
        finally:
            self.cleanup()

    def _iteration(self):
        """collect -> add_new_experience -> PPOLearner.learn -> report.  Returns the number of steps collected."""
        from .util import reporting
        if self.data_parallel:
            return self._iteration_dp()
        t_start = time.perf_counter()
        experience, env_metrics, n_steps, t_collect = self.agent.collect_timesteps(self.ts_per_epoch)
        if self.metrics_logger is not None:
            self.metrics_logger.report_metrics(env_metrics, self.wandb_run, self.agent.cumulative_timesteps)
        self.add_new_experience(experience)
        report = dict(self.ppo_learner.learn(self.experience_buffer))
        t_total = time.perf_counter() - t_start
        if self.epoch < 1:
            report["Value Function Loss"] = np.nan      # the first iteration's critic loss is not reported (:273-274)
        avg_rew = self.agent.average_reward
        report.update({
            "Cumulative Timesteps": self.agent.cumulative_timesteps,
            "Total Iteration Time": t_total,
            "Timesteps Collected": n_steps,
            "Timestep Collection Time": t_collect,
            "Timestep Consumption Time": t_total - t_collect,
            "Collected Steps per Second": n_steps / t_collect,
            "Overall Steps per Second": n_steps / t_total,
            "Policy Reward": np.nan if avg_rew is None else avg_rew,
        })
        reporting.report_metrics(loggable_metrics=report, debug_metrics=None, wandb_run=self.wandb_run)
        return n_steps

    def _iteration_dp(self):
        """collect -> exchange -> merge of the observation statistics -> add_new_experience -> learn -> report (rank 0).
        Returns the number of steps collected by all ranks.

        The exchange is one all-gather of every rank's observation-statistics delta and collection tail.  It comes before
        add_new_experience, whose first call holds a collective of its own, and a rank whose collection raised still takes
        part (with its error flag set): every rank issues the same collectives in the same order, and all of them leave
        the loop together when any rank failed."""
        from .util import reporting
        t_start = time.perf_counter()
        cum0 = self.agent.cumulative_timesteps
        error, experience, env_metrics, n_steps, t_collect = None, None, [], 0, 0.0
        try:
            experience, env_metrics, n_steps, t_collect = self.agent.collect_timesteps(self.ts_per_epoch)
        except Exception as e:  # noqa: BLE001  (re-raised below, after the exchange)
            error, t_collect = e, time.perf_counter() - t_start
        t_x = time.perf_counter()
        delta = self.agent.obs_delta
        block = delta.device_block() if delta is not None else torch.empty(0, dtype=torch.uint8, device=self.device)
        blocks, stride, tails = parallel.exchange(
            block, parallel.pack_tail(n_steps, t_collect, self.agent.average_reward, error is not None))
        agg = parallel.combine_tails(tails)
        if agg["failed"]:
            self.agent.cumulative_timesteps = cum0
            if error is not None:
                raise error
            raise RuntimeError(f"environment collection failed on data-parallel rank(s) {agg['failed']}")
        if delta is not None:
            # base <- base + every rank's increments, in rank order; the base becomes every rank's working statistics
            self._obs_base.merge_device(blocks, self.world_size, stride)
            self.agent.obs_stats.copy_device_(self._obs_base)
            delta.reset()
        torch.cuda.current_stream().synchronize()
        self._t_exchange = time.perf_counter() - t_x
        self.agent.cumulative_timesteps = cum0 + agg["steps"]
        if self.metrics_logger is not None:
            metrics = parallel.gather_metrics(env_metrics)
            if self.rank == 0:
                self.metrics_logger.report_metrics(metrics, self.wandb_run, self.agent.cumulative_timesteps)
        self.add_new_experience(experience)
        report = dict(self.ppo_learner.learn(self.experience_buffer))
        if self.rank == 0:
            if self.epoch < 1:
                report["Value Function Loss"] = np.nan
            report["Cumulative Timesteps"] = self.agent.cumulative_timesteps
            report["Total Iteration Time"] = t_total = time.perf_counter() - t_start
            report.update(parallel.collection_report(agg, t_total))
            reporting.report_metrics(loggable_metrics=report, debug_metrics=None, wandb_run=self.wandb_run)
        return agg["steps"]

    def _poll_keys(self, kb):
        """p = pause until a key, c = checkpoint, q = checkpoint and stop.  Returns True when the loop should end."""
        if not kb.kbhit():
            return False
        key = kb.getch()
        if key == "p":
            print("Paused, press any key to resume")
            while not kb.kbhit():
                time.sleep(0.05)
        if key in ("c", "q"):
            self.save(self.agent.cumulative_timesteps)
        if key == "q":
            return True
        if key in ("c", "p"):
            print("Resuming...\n")
        return False

    def _learn(self):
        from .util.kbhit import KBHit
        kb = None
        if not self.data_parallel:     # data parallel: the ranks take every loop decision together, so no keys
            kb = KBHit()   # guarded: no-op without a TTY (gpurun / CI)
            print("Press (p) to pause (c) to checkpoint, (q) to checkpoint and quit (after next iteration)\n")
        # data parallel: cumulative_timesteps, timestep_limit and save_every_ts count the steps of all ranks
        while self.agent.cumulative_timesteps < self.timestep_limit:
            self.ts_since_last_save += self._iteration()
            if kb is not None and self._poll_keys(kb):
                return
            if self.ts_since_last_save >= self.save_every_ts:
                self.save(self.agent.cumulative_timesteps)
                self.ts_since_last_save = 0
            self.epoch += 1

    # ---- the learner-side hot path, first half (learner.py:330-385) ------------------------------------------------
    def add_new_experience(self, experience):
        """
        Add timesteps to the experience buffer and compute advantages, value targets and returns for them.
        `experience`: (states, actions, log_probs, rewards, next_states, dones, truncated) as NumPy arrays (any float
        dtype; pinned memory is copied without a bounce), torch CPU tensors or device tensors.
        Everything after the H2D copies runs on the device; nothing is read back.  Also callable unbound on any
        object carrying ppo_learner, return_stats, standardize_returns, gae_gamma, gae_lambda,
        max_returns_per_stats_increment and experience_buffer.
        """
        buf = self.experience_buffer
        ppo = self.ppo_learner
        value_net = ppo.value_net
        vst = value_net._stack
        dev = vst.device
        stager = getattr(self, "_stager", None)
        if stager is None:
            stager = self._stager = Stager(dev)
        n = int(experience[0].shape[0]) if hasattr(experience[0], "shape") else len(experience[0])
        if n == 0:
            return
        # ---- the 7 arrays in HBM at addresses a graph can bake in: host arrays are copied (one async H2D each) into
        # persistent device slots; arrays that already live on the device are used where they are ---------------------
        shapes = tuple((tuple(np.shape(x)), _staged_dtype(x)) for x in experience)
        # "sharded" data parallelism over peer memory: one rollout per rank, the return statistics are rank 0's (the
        # reference updates them from the head of ONE rollout, learner.py:368-372).  Rank 0 publishes its std in a
        # symmetric-memory slot (double buffered by iteration parity) and every rank's scan reads that slot directly over
        # NVLink: no broadcast, no NCCL call in the iteration.
        peer_std = (getattr(ppo, "world_size", 1) > 1 and getattr(ppo, "dp_mode", "") == "sharded"
                    and getattr(ppo, "_std_slots_rank0", None) is not None and self.standardize_returns)
        stats_here = (not peer_std) or ppo.rank == 0
        stage = getattr(self, "_exp_stage", None)
        if stage is None or stage["shapes"] != shapes:
            stage = {"shapes": shapes, "gen": (0 if stage is None else stage["gen"] + 1)}
            n_inc = min(int(self.max_returns_per_stats_increment), n) if (self.standardize_returns and stats_here) else 0
            stage["values"] = torch.empty(n + 1, dtype=torch.float32, device=dev)
            stage["out"] = tuple(torch.empty(n, dtype=torch.float32, device=dev) for _ in range(3))
            stage["head"] = torch.empty(n_inc, dtype=torch.float64, device=dev) if n_inc else None
            stage["gae_ws"] = ops.gae_workspace(n, dev)
            self._exp_stage = stage
        # next_states arriving from the HOST take the late path: nothing on the learner path reads that ring (only its last
        # row feeds the value net, learner.py:349), so the 17.8 MB block -- half of the PCIe traffic of an example-size
        # iteration -- is copied and appended on a second stream while this call's device work and the whole of
        # PPOLearner.learn run; only the last row crosses on the main stream.  Readers (the `next_states` attribute, the
        # next call) wait for it through ExperienceBuffer.sync_late().
        ns_in = experience[4]
        late_ns = (not (isinstance(ns_in, torch.Tensor) and ns_in.is_cuda) and n >= 2
                   and os.environ.get("RLPPO_LATE_NEXT_STATES", "1") == "1")
        buf.sync_late()      # the previous call's late block is in its ring (and out of its staging slot) before we go on
        d, ptrs = {}, []
        for name, arr, (shape, dt) in zip(_EXP_FIELDS, experience, shapes):
            if name == "next_states" and late_ns:
                if "ns_last" not in stage:
                    stage["ns_last"] = torch.empty((1, shape[1]), dtype=dt, device=dev)
                    stage[name] = torch.empty(shape, dtype=dt, device=dev)
                d["ns_last"] = stager.to_device(arr[n - 1:n], "exp.ns_last", out=stage["ns_last"])
                ptrs.append(d["ns_last"].data_ptr())
                continue
            if isinstance(arr, torch.Tensor) and arr.is_cuda and arr.dtype == dt and arr.is_contiguous():
                d[name] = arr
            else:
                if name not in stage:
                    stage[name] = torch.empty(shape, dtype=dt, device=dev)
                d[name] = stager.to_device(arr, "exp." + name, out=stage[name])
            ptrs.append(d[name].data_ptr())
        if late_ns:
            late = getattr(self, "_late_stream", None)
            if late is None:
                late = self._late_stream = torch.cuda.Stream(device=dev)
            late.wait_stream(torch.cuda.current_stream())     # after whatever the main stream still has queued on these blocks
            with torch.cuda.stream(late):
                ns_dev = stager.to_device(ns_in, "exp.next_states", out=stage["next_states"])
            stage["next_states"].record_stream(late)
        obs = int(d["states"].shape[1])
        if buf._rings is None:
            a_shape = tuple(d["actions"].shape)
            buf._allocate(obs, int(a_shape[1]) if len(a_shape) == 2 else 1)
        vst.workspace(n + 1)
        vst.refresh_operands()
        ret_std = self.return_stats.device_std() if self.standardize_returns else None     # learner.py:356
        n_inc = 0 if stage["head"] is None else stage["head"].numel()
        par = 0
        if peer_std:
            par = getattr(self, "_std_parity", None)
            if par is None:
                # first call: rank 0's current std (1, or whatever a loaded checkpoint holds) into slot 0, once, for everyone
                import torch.distributed as dist
                par = 0
                if ppo.rank == 0:
                    ppo._std_slots_local[0:1].copy_(ret_std)
                torch.cuda.synchronize(dev)
                dist.barrier(getattr(ppo, "_pg", None))
            ret_std = ppo._std_slots_rank0[par:par + 1]
            self._std_parity = 1 - par

        # GAE shards by trajectory (BASELINE north_star; SURVEY.md 8e): when every rank holds the SAME rollout
        # (dp_mode="replicated"), rank r runs the value net and the scan on its contiguous chunk only.
        world, rank = getattr(ppo, "world_size", 1), getattr(ppo, "rank", 0)
        shard = (world > 1 and getattr(ppo, "dp_mode", "") == "replicated" and n >= 2048 * world
                 and os.environ.get("RLPPO_GAE_SHARD", "1") == "1")
        if hasattr(ppo, "world_size"):
            ppo.gae_sharded = shard

        def values_and_gae_sharded():
            """Chunk [lo, hi) of the flat step axis: value net on its rows + 1 halo row, the chunk's affine summary
            (rlppo_gae_chunk_summary), all-gather of the 4-double summaries, carry = the chunks to the right composed onto 0
            (rlppo_gae_compose_carry), the scan with that carry, all-gather of advantages / value targets; the first
            returns (Welford input, learner.py:368-372) come from rank 0's chunk.  Exact: composition of affine maps."""
            import torch.distributed as dist
            from . import parallel
            group = getattr(ppo, "_pg", None)
            lo, hi, m = parallel.gae_chunk(n, rank, world)
            cnt = hi - lo
            sh = stage.get("shard")
            if sh is None or sh["m"] != m:
                f64 = lambda k: torch.zeros(k, dtype=torch.float64, device=dev)  # noqa: E731
                sh = stage["shard"] = {"m": m, "summ": f64(4), "all": f64(4 * world), "carry": f64(2),
                                       "loc": torch.zeros((2, m), dtype=torch.float32, device=dev),
                                       "ret": torch.empty(m, dtype=torch.float32, device=dev),
                                       "full": [torch.empty(world * m, dtype=torch.float32, device=dev) for _ in range(2)],
                                       "values": torch.empty(m + 1, dtype=torch.float32, device=dev),
                                       "ws": ops.gae_workspace(m, dev)}
            states = _f32(d["states"])
            x = vst.workspace(n + 1)["x"]
            sh["summ"].zero_()
            sh["summ"][0] = 1.0       # an empty chunk is the identity map (a = 1, b = 0)
            sh["summ"][2] = 1.0
            if cnt > 0:
                vst.stage_rows(states[lo:hi], x)
                halo = states[hi:hi + 1] if hi < n else (_f32(d["ns_last"]) if late_ns else _f32(d["next_states"])[n - 1:n])
                vst.stage_rows(halo, x[cnt:cnt + 1])
                values = value_net.values_from_bf16(x, cnt + 1, out=sh["values"][:cnt + 1])
                rew, done, trunc = _f32(d["rewards"])[lo:hi], _f32(d["dones"])[lo:hi], d["truncated"][lo:hi]
                ops.gae_chunk_summary(rew, done, trunc, values, self.gae_gamma, self.gae_lambda, ret_std, out=sh["summ"])
            dist.all_gather_into_tensor(sh["all"], sh["summ"], group=group)
            ops.gae_compose_carry(sh["all"], rank, world, out=sh["carry"])
            if cnt > 0:
                head = stage["head"] if (rank == 0 and n_inc) else None
                ops.gae(rew, done, trunc, values, self.gae_gamma, self.gae_lambda, ret_std,
                        out=(sh["loc"][0, :cnt], sh["loc"][1, :cnt], sh["ret"][:cnt]), ret_head64=head,
                        carry_in=sh["carry"], ws=sh["ws"])
            dist.all_gather_into_tensor(sh["full"][0], sh["loc"][0], group=group)
            dist.all_gather_into_tensor(sh["full"][1], sh["loc"][1], group=group)
            if n_inc:
                assert n_inc <= m, "the returns that feed the running statistics must lie in rank 0's chunk"
                dist.broadcast(stage["head"], src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
            return sh["full"][0][:n], sh["full"][1][:n]

        def body():
            """Device work only (what the CUDA graph captures): value net on [states ; next_states[-1]]
            (learner.py:347-352), GAE (:358-366), return statistics (:368-372), the nine ring appends (:375-385)."""
            if shard:
                vt, adv = values_and_gae_sharded()
            else:
                states = _f32(d["states"])
                x = vst.workspace(n + 1)["x"]
                vst.stage_rows(states, x)
                vst.stage_rows(_f32(d["ns_last"]) if late_ns else _f32(d["next_states"])[n - 1:n], x[n:n + 1])
                values = value_net.values_from_bf16(x, n + 1, out=stage["values"])      # stays on the device
                vt, adv, _ = ops.gae(_f32(d["rewards"]), _f32(d["dones"]), d["truncated"], values, self.gae_gamma,
                                     self.gae_lambda, ret_std, out=stage["out"], ret_head64=stage["head"],
                                     ws=stage["gae_ws"])
            fields = {k: v for k, v in d.items() if k != "ns_last"}
            fields["values"], fields["advantages"] = vt, adv
            if n_inc:
                # The Welford update (150 strictly sequential f64 steps on one thread: ~22 us of pure latency) only
                # gates the NEXT call's scan, so it runs beside the ring appends on a second stream -- a parallel branch
                # of the captured graph -- after the scan has read std.
                main = torch.cuda.current_stream()
                side = getattr(self, "_side_stream", None)
                if side is None:
                    side = self._side_stream = torch.cuda.Stream(device=dev)
                fork, join = torch.cuda.Event(), torch.cuda.Event()
                fork.record(main)
                side.wait_event(fork)
                with torch.cuda.stream(side):
                    self.return_stats.increment_device(stage["head"], n_inc)
                    if peer_std:     # the scale the NEXT iteration's scans read (every rank, out of this rank's memory)
                        ppo._std_slots_local[1 - par:2 - par].copy_(self.return_stats.device_std())
                    join.record(side)
                buf.append_device(fields)
                main.wait_event(join)
            else:
                buf.append_device(fields)

        graphs = getattr(self, "_add_graphs", None)
        if graphs is None:
            graphs = self._add_graphs = GraphCache()
        key = (n, obs, stage["gen"], tuple(ptrs), late_ns, buf.uid, getattr(vst, "ws_gen", 0), id(self.return_stats._d), n_inc,
               peer_std, par,
               float(self.gae_gamma), float(self.gae_lambda), bool(self.standardize_returns), vst.fused_ok, vst.precision)
        # (the sharded scan has NCCL exchanges in it and runs eagerly; everything else replays as one graph)
        if shard or not (getattr(ppo, "use_cuda_graph", False) and _lib._TIMING is None and graphs.replay(key, body)):
            body()
        if late_ns:
            buf.append_next_states_late(ns_dev, late)      # position from the host mirrors, BEFORE they advance
        # host mirrors of what the device work did
        buf.advance_host(min(n, buf.capacity))
        if n_inc:
            self.return_stats._dev_is_newer = True
            if getattr(ppo, "world_size", 1) > 1 and getattr(ppo, "dp_mode", "") == "sharded" and not peer_std:
                # one rollout per rank (NCCL gradient exchange: no peer mappings): the statistics follow rank 0's
                self.return_stats.broadcast_(src=0, group=getattr(ppo, "_pg", None))

    # ---- checkpoints: the reference's directory layout and file formats (learner.py:387-564) ---------------------
    # <save folder>/<cumulative timesteps>/{PPO_POLICY.pt, PPO_VALUE_NET.pt, PPO_POLICY_OPTIMIZER.pt,
    # PPO_VALUE_NET_OPTIMIZER.pt, BOOK_KEEPING_VARS.json}; at most n_checkpoints_to_keep numbered folders are kept.
    def _book_keeping(self):
        bk = {
            "cumulative_timesteps": self.agent.cumulative_timesteps,
            "cumulative_model_updates": self.ppo_learner.cumulative_model_updates,
            "policy_average_reward": self.agent.average_reward,
            "epoch": self.epoch,
            "ts_since_last_save": self.ts_since_last_save,
            "reward_running_stats": self.return_stats.to_json(),
        }
        if self.agent.standardize_obs:
            # data parallel: the merged statistics of all ranks
            obs_stats = self._obs_base if self.data_parallel else self.agent.obs_stats
            bk["obs_running_stats"] = obs_stats.to_json()
        run = self.wandb_run
        if run is not None:
            bk.update(wandb_run_id=run.id, wandb_project=run.project, wandb_entity=run.entity, wandb_group=run.group,
                      wandb_config=run.config.as_dict())
        return bk

    def save(self, cumulative_timesteps):
        if self.rank != 0:       # data parallel: rank 0 writes the run's checkpoints
            return
        root = self.checkpoints_save_folder
        target = os.path.join(root, str(cumulative_timesteps))
        os.makedirs(target, exist_ok=True)
        print(f"Saving checkpoint {cumulative_timesteps}...")
        # prune: the reference compares with ">" after creating the new folder, i.e. keeps the newest n (+ the new one)
        numbered = sorted(int(name) for name in os.listdir(root) if name.isdigit())
        if len(numbered) > self.n_checkpoints_to_keep:
            for stale in numbered[:-self.n_checkpoints_to_keep]:
                shutil.rmtree(os.path.join(root, str(stale)), ignore_errors=True)
        os.makedirs(target, exist_ok=True)
        self.ppo_learner.save_to(target)
        with open(os.path.join(target, "BOOK_KEEPING_VARS.json"), "w") as f:
            json.dump(self._book_keeping(), f, indent=4)
        print(f"Checkpoint {cumulative_timesteps} saved!\n")

    def _latest_checkpoint(self):
        """The numbered folder with the most timesteps inside the newest run folder, or None.  With add_unix_timestamp the
        run folders are `<base>-<time_ns>` siblings and the newest stamp wins (learner.py:452-499)."""
        run_dir = self.checkpoints_save_folder
        if run_dir is None:
            return None
        if self.add_unix_timestamp:
            base = run_dir[:run_dir.rfind("-")]
            parent = os.path.dirname(base)
            if not os.path.isdir(parent):
                return None
            stamped = []
            for name in os.listdir(parent):
                full = os.path.join(parent, name)
                stamp = full[full.rfind("-") + 1:]
                if os.path.isdir(full) and full.startswith(base) and stamp.isdigit():
                    stamped.append((int(stamp), full))
            if not stamped:
                return None
            run_dir = max(stamped)[1]
        elif not os.path.isdir(run_dir):
            return None
        steps = [int(name) for name in os.listdir(run_dir)
                 if name.isdigit() and os.path.isdir(os.path.join(run_dir, name))]
        return os.path.join(run_dir, str(max(steps))) if steps else None

    def load(self, folder_path, load_wandb, new_policy_lr=None, new_critic_lr=None):
        """Load a checkpoint written by this implementation or by the reference.  Returns True when a wandb run was
        resumed, None when `folder_path == "latest"` finds nothing."""
        if folder_path == "latest":
            folder_path = self._latest_checkpoint()
            if folder_path is None:
                return None
            print(f"Auto-load path: {folder_path}")
        assert os.path.exists(folder_path), f"UNABLE TO LOCATE FOLDER {folder_path}"
        print(f"Loading from checkpoint at {folder_path}")
        self.ppo_learner.load_from(folder_path)
        with open(os.path.join(folder_path, "BOOK_KEEPING_VARS.json"), "r") as f:
            bk = dict(json.load(f))
        self.agent.cumulative_timesteps = bk["cumulative_timesteps"]
        self.agent.average_reward = bk["policy_average_reward"]
        self.ppo_learner.cumulative_model_updates = bk["cumulative_model_updates"]
        self.epoch = bk["epoch"]
        self.return_stats.from_json(bk["reward_running_stats"])
        if self.agent.standardize_obs and "obs_running_stats" in bk:
            self.agent.obs_stats = WelfordRunningStat(1, device=self.device)
            self.agent.obs_stats.from_json(bk["obs_running_stats"])
            self._obs_loaded = True
        if new_policy_lr is not None or new_critic_lr is not None:
            self.update_learning_rate(new_policy_lr, new_critic_lr)
        resumed = False
        if load_wandb and "wandb_run_id" in bk:
            import wandb
            self.wandb_run = wandb.init(settings=wandb.Settings(start_method="spawn"), entity=bk["wandb_entity"],
                                        project=bk["wandb_project"], group=bk["wandb_group"], id=bk["wandb_run_id"],
                                        config=bk["wandb_config"], resume="allow", reinit=True)
            resumed = True
        print("Checkpoint loaded!")
        return resumed

    def cleanup(self):
        if self.wandb_run is not None:
            self.wandb_run.finish()
        agent = getattr(self, "agent", None)
        if agent is not None and hasattr(agent, "cleanup"):
            agent.cleanup()
        self.experience_buffer.clear()
        if self._owns_group:
            import torch.distributed as dist
            dist.destroy_process_group()
            self._owns_group = False
