"""BatchedAgentManager: the learner side of timestep collection (replaces
rlgym_ppo/batched_agents/batched_agent_manager.py for the data path; process plumbing is deliberately simple).

What the reference does per environment step (batched_agent_manager.py:180-350): np.concatenate the ready
observations, one small torch forward + multinomial + .cpu(), per-message NumPy parsing, Python lists of per-agent
timesteps that are flattened with np.asarray at the end (:125-172).

Here every observation crosses PCIe exactly once and stays in HBM:
  * the reference's asynchronous loop (actions to whoever is waiting, then responses as they arrive until at least
    min_inference_size observations are in); every worker's observation lands in one PINNED slab row [slots, obs];
  * one async H2D of that row, then on the device: optional standardisation (clip((x-mean)/std, +-5)) fused with
    the bf16 conversion, the policy MLP on tcgen05, softmax/clamp/categorical sample/log-prob in the head epilogue;
  * actions come back in one small D2H; observations, actions and log-probs stay in time-major device slabs;
  * a tick is ONE CUDA-graph launch (tick.TickInference) ending in the action D2H; the host waits on one event;
  * at the end of collect_timesteps the flat per-trajectory layout the learner expects (SURVEY.md A.1: completed
    trajectories in completion order, then open ones by process id; each agent's steps in time order; last step of
    every run forced truncated unless done) is produced by ONE index gather on the device.
collect_timesteps therefore returns DEVICE tensors; Learner.add_new_experience consumes them without a copy.

An environment may return a different number of agents after each reset.  Process p owns `capacity[p]` slots (its
largest count so far) starting at slot0[p]; only the first n_agents[p] of them are live: sent as actions, recorded and
counted.  A count above the capacity re-lays the slots out once (_grow).
"""
import multiprocessing as mp
import multiprocessing.sharedctypes
import os
import time

import numpy as np
import torch

from .. import _lib, ops
from ..util import WelfordRunningStat
from .batched_agent import batched_agent_process
from .env_worker import env_worker
from .wire import WireConn


class BatchedAgentManager(object):
    def __init__(self, policy, min_inference_size=8, seed=123, standardize_obs=True, steps_per_obs_stats_increment=5,
                 device=None, keep_obs_delta=False):
        self.policy = policy
        self.seed = seed
        self.processes = []
        self.average_reward = None
        self.cumulative_timesteps = 0
        self.min_inference_size = min_inference_size   # observations that must have arrived before the next inference
        self.standardize_obs = standardize_obs
        self.steps_per_obs_stats_increment = steps_per_obs_stats_increment
        self.steps_since_obs_stats_update = 0
        self.obs_stats = None
        # data-parallel Learner: obs_delta is a second Welford state fed the same samples as obs_stats, holding the
        # increments since the ranks last merged their statistics (Learner resets it after every merge)
        self.keep_obs_delta = keep_obs_delta
        self.obs_delta = None
        self.ep_rews = []
        self.n_procs = 0
        self.device = device
        self._current_obs = None     # pinned [slots, obs]: the observation every slot will act on next

    # ---- processes -------------------------------------------------------------------------------------------
    def init_processes(self, n_processes, build_env_fn, collect_metrics_fn=None, spawn_delay=None, render=False,
                       render_delay=None, shm_buffer_size=8192, transport=None):
        """transport: "pipe" (default; multiprocessing pipes, env_worker.py) or "wire" -- the reference's own worker
        protocol (UDP datagrams + a shared float32 slab of shm_buffer_size bytes per worker, batched_agent.py /
        comm_consts.py), so workers written for the reference plug in unchanged.  RLPPO_WORKER_TRANSPORT overrides."""
        _lib.require_device()
        if self.device is None:
            self.device = "cuda:%d" % torch.cuda.current_device()
        methods = mp.get_all_start_methods()
        ctx = mp.get_context("forkserver" if "forkserver" in methods else "spawn")
        self.n_procs = n_processes
        transport = os.environ.get("RLPPO_WORKER_TRANSPORT", transport or "pipe")
        assert transport in ("pipe", "wire"), transport
        self.transport = transport
        if transport == "wire":
            self.shm_size = shm_buffer_size // 4                         # floats per worker (batched_agent_manager.py:437)
            self.shm_buffer = multiprocessing.sharedctypes.RawArray("f", n_processes * self.shm_size)
        for proc_id in range(n_processes):
            if transport == "wire":
                parent = WireConn(self.shm_buffer, proc_id * self.shm_size * 4, self.shm_size)
                p = ctx.Process(target=batched_agent_process,
                                args=(proc_id, parent.endpoint, self.shm_buffer, proc_id * self.shm_size * 4, self.shm_size,
                                      self.seed + proc_id, render and proc_id == 0, render_delay), daemon=True)
                p.start()
            else:
                parent, child = ctx.Pipe(duplex=True)
                p = ctx.Process(target=env_worker, args=(child, proc_id, self.seed + proc_id, render and proc_id == 0,
                                                         render_delay), daemon=True)
                p.start()
                child.close()
            self.processes.append((p, parent))
        if transport == "wire":
            for _, conn in self.processes:
                conn.accept()
        for _, conn in self.processes:
            if spawn_delay is not None:
                time.sleep(spawn_delay)
            conn.send(("init", build_env_fn, collect_metrics_fn))
        first = [self._recv(conn, "reset")[1] for _, conn in self.processes]
        for p, o in enumerate(first):
            if o.shape[0] == 0:
                raise RuntimeError(f"environment process {p} returned an observation with no agents")
        self._n = [int(o.shape[0]) for o in first]     # agents in each process's current observation
        self._cap = list(self._n)                      # slots each process owns: its largest count so far
        self._slot0 = np.concatenate([[0], np.cumsum(self._cap)]).astype(np.int64)
        self.n_slots = int(self._slot0[-1])
        self.obs_dim = int(first[0].shape[1])
        self.ep_rews = [np.zeros(a, np.float64) for a in self._n]
        self._current_obs = torch.empty((self.n_slots, self.obs_dim), dtype=torch.float32).pin_memory()
        cur = self._current_obs.numpy()
        for p, o in enumerate(first):
            cur[self._slot0[p]:self._slot0[p + 1]] = o
        if self.standardize_obs:
            # NB the reference builds WelfordRunningStat(shape=obs) and seeds it with the reset observations (:377-380)
            self.obs_stats = WelfordRunningStat(self.obs_dim, device=self.device)
            if self.keep_obs_delta:
                self.obs_delta = WelfordRunningStat(self.obs_dim, device=self.device)
            for o in first:
                self._increment_obs_stats(o)
        self.processes[0][1].send(("shapes",))
        _, obs_size, n_acts, space_type = self._recv(self.processes[0][1], "shapes")
        return obs_size, n_acts, space_type

    def _increment_obs_stats(self, o):
        self.obs_stats.increment(o, o.shape[0])
        if self.obs_delta is not None:
            self.obs_delta.increment(o, o.shape[0])

    @staticmethod
    def _recv(conn, expect):
        msg = conn.recv()
        if msg[0] == "error":
            raise RuntimeError("environment worker failed:\n" + msg[1])
        assert msg[0] == expect, f"expected {expect!r} from worker, got {msg[0]!r}"
        return msg

    # ---- collection ------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def collect_timesteps(self, n):
        """Collect at least n timesteps.  Returns ((states, actions, log_probs, rewards, next_states, dones,
        truncated) as DEVICE tensors in the reference's flat layout, collected_metrics, n_collected, elapsed).

        The loop is the reference's (batched_agent_manager.py:98-123): actions go out to the processes whose observation
        is waiting, then responses are taken as they arrive until at least min(min_inference_size, n_procs) new
        observations are in, and the next inference runs on whatever arrived -- a slow environment never holds the others
        up.  The inference itself is one fixed-shape CUDA graph over ALL slots (a tick costs the same 50-70 us for 8 or
        4096 rows); only the live rows of the processes that were waiting are used, sent and recorded."""
        import selectors
        from .tick import TickInference
        t1 = time.perf_counter()
        S, D, P, dev = self.n_slots, self.obs_dim, self.n_procs, torch.device(self.device)
        tick = getattr(self, "_tick", None)
        if tick is None or tick.policy is not self.policy:
            tick = self._tick = TickInference(self.policy, S, D, standardize=self.standardize_obs)
            tick.obs_host = self._current_obs          # the workers' observations land in the tick's pinned row
        act_w = tick.act_w
        need = max(1, min(int(self.min_inference_size), P))      # :101-102
        agents_min = max(1, min(self._n))
        cap = (int(n) + need * agents_min - 1) // (need * agents_min) + P + 8      # ticks; grown if the estimate is short

        def alloc(T):
            return (torch.empty((T + 1, S, D), dtype=torch.float32, device=dev),
                    torch.empty((T, S) if act_w == 1 else (T, S, act_w), dtype=torch.float32, device=dev),
                    torch.empty((T, S), dtype=torch.float32, device=dev))
        obs_slab, act_slab, logp_slab = alloc(cap)
        collected_metrics = []
        cur = self._current_obs.numpy()
        # per process: the tick at which each of its steps was inferred, how many agents acted, and what the environment
        # answered
        seq = [dict(tick=[], n=[], rew=[], done=[], trunc=[], order=[]) for _ in range(P)]
        sel = getattr(self, "_selector", None)
        if sel is None:
            sel = self._selector = selectors.DefaultSelector()
            for pid, (_, conn) in enumerate(self.processes):
                sel.register(conn.fileno() if hasattr(conn, "fileno") else conn.sock.fileno(), selectors.EVENT_READ, pid)

        def push_stats():
            # the reference standardises EVERY feature with the statistics of feature 0
            # (`self.obs_stats.mean[0]`, `.std[0]`, batched_agent_manager.py:233-235): reproduced as is
            if self.standardize_obs:
                tick.set_obs_stats(self.obs_stats.device_mean()[0:1].expand(D), self.obs_stats.device_std()[0:1].expand(D))

        push_stats()
        waiting = getattr(self, "_waiting", None)          # processes whose observation awaits an action
        if waiting is None:
            waiting = list(range(P))
        in_flight = set()
        n_collected, tk, completion = 0, 0, 0

        def take_response(pid):
            nonlocal n_collected, completion, tick, S, cur, obs_slab, act_slab, logp_slab
            _, o, r, d, tr, metrics = self._recv(self.processes[pid][1], "step")
            n_act, n_next = self._n[pid], int(o.shape[0])      # the agents that acted; those of the new observation
            r = np.asarray(r, np.float32).reshape(-1)
            if r.shape[0] != n_act:
                raise RuntimeError(f"environment process {pid} returned {r.shape[0]} rewards for {n_act} agents")
            if n_next != n_act and not (d or tr):
                raise RuntimeError(f"environment process {pid} changed its agent count from {n_act} to {n_next} "
                                   "without ending the episode")
            if n_next == 0:
                raise RuntimeError(f"environment process {pid} returned an observation with no agents")
            if n_next > self._cap[pid]:
                tick, (obs_slab, act_slab, logp_slab) = self._grow(pid, n_next, (obs_slab, act_slab, logp_slab))
                S, cur = self.n_slots, self._current_obs.numpy()
                self._stats_dirty = True
            lo = self._slot0[pid]
            cur[lo:lo + n_next] = o
            self._n[pid] = n_next
            q = seq[pid]
            q["n"].append(n_act)
            q["rew"].append(r)
            q["done"].append(bool(d))
            q["trunc"].append(bool(tr))
            q["order"].append(completion)
            completion += 1
            if metrics is not None:
                collected_metrics.append(metrics)
            self.ep_rews[pid] += r
            if d or tr:                                   # :327-335
                if self.average_reward is None:
                    self.average_reward = float(self.ep_rews[pid][0])
                else:
                    for ep_rew in self.ep_rews[pid]:
                        self.average_reward = self.average_reward * 0.9 + float(ep_rew) * 0.1
                self.ep_rews[pid] = np.zeros(n_next, np.float64)
            if self.standardize_obs:                      # :303-315 (per response)
                self.steps_since_obs_stats_update += 1
                if self.steps_since_obs_stats_update > self.steps_per_obs_stats_increment:
                    self._increment_obs_stats(o)
                    self.steps_since_obs_stats_update = 0
                    self._stats_dirty = True
            in_flight.discard(pid)
            n_collected += n_act
            return n_act

        while n_collected < n:
            if tk >= cap:                                 # the estimate was short (many single-response passes): grow
                cap2 = cap + cap // 2 + 8
                o2, a2, l2 = alloc(cap2)
                o2[:cap + 1].copy_(obs_slab)
                a2[:cap].copy_(act_slab)
                l2[:cap].copy_(logp_slab)
                obs_slab, act_slab, logp_slab, cap = o2, a2, l2, cap2
            if getattr(self, "_stats_dirty", False):
                push_stats()
                self._stats_dirty = False
            # one CUDA-graph launch: H2D obs -> standardise/stage -> fused MLP + sample -> D2H actions; then the slab rows
            # (device-to-device, behind the event the host waits on: they never delay the workers)
            tick.enqueue()
            obs_slab[tk].copy_(tick.obs_seen, non_blocking=True)
            act_slab[tk].copy_(tick.act_dev, non_blocking=True)
            logp_slab[tk].copy_(tick.logp_dev, non_blocking=True)
            tick.done_ev.synchronize()
            a = tick.act_host.numpy()
            for pid in waiting:                           # :181-221 _send_actions
                lo = self._slot0[pid]
                self.processes[pid][1].send(("act", a[lo:lo + self._n[pid]].copy()))
                seq[pid]["tick"].append(tk)
                in_flight.add(pid)
            waiting = []
            got = 0
            while got < need and in_flight:               # :223-252 _collect_responses
                for key, _ in sel.select():
                    if key.data in in_flight:
                        got += take_response(key.data)
                        waiting.append(key.data)
            tk += 1
        # every action that was sent is answered before the call returns (the reference leaves such steps to its next
        # call; here the slabs are per call), then the observation every process will act on next is staged as row `tk`
        while in_flight:
            for key, _ in sel.select():
                if key.data in in_flight:
                    take_response(key.data)
                    waiting.append(key.data)
        self._waiting = sorted(set(waiting) | (set(range(P)) - set(waiting) - in_flight))
        if getattr(self, "_stats_dirty", False):
            push_stats()
            self._stats_dirty = False
        self._stage_only(tick, obs_slab[tk])
        for p in range(P):
            seq[p]["n_end"] = self._n[p]
        out = self.flatten_steps(obs_slab, act_slab, logp_slab, seq, self._slot0, tk)
        n_out = int(out[3].shape[0])
        self.cumulative_timesteps += n_out
        return out, collected_metrics, n_out, time.perf_counter() - t1

    def _stage_only(self, tick, dst):
        tick.obs_raw.copy_(tick.obs_host, non_blocking=True)
        if self.standardize_obs:
            ops.rows_to_bf16(tick.obs_raw, tick._scratch(), tick.mean_dev, tick.std_dev, tick.clip, dst_f32=dst)
        else:
            dst.copy_(tick.obs_raw, non_blocking=True)
        torch.cuda.current_stream().synchronize()      # obs_host may be rewritten by the next collect_timesteps

    def _grow(self, pid, n_agents, slabs):
        """Raise process pid's capacity to n_agents: a new slot layout, pinned observation row and tick (its graph is
        captured again on its second use), and this call's time-major slabs remapped to the new slots with one device
        index_select each.  Returns (tick, slabs).  Happens once per new maximum count."""
        from .tick import TickInference
        old0, old_cap = self._slot0, list(self._cap)
        self._cap[pid] = n_agents
        self._slot0 = np.concatenate([[0], np.cumsum(self._cap)]).astype(np.int64)
        self.n_slots = int(self._slot0[-1])
        src = np.zeros(self.n_slots, np.int64)       # new slot -> old slot; the added slots are stale until written
        old_obs = self._current_obs.numpy()
        self._current_obs = torch.zeros((self.n_slots, self.obs_dim), dtype=torch.float32).pin_memory()
        new_obs = self._current_obs.numpy()
        for p in range(self.n_procs):
            lo, w = int(self._slot0[p]), old_cap[p]
            src[lo:lo + w] = np.arange(old0[p], old0[p] + w)
            new_obs[lo:lo + w] = old_obs[old0[p]:old0[p] + w]
        old = self._tick
        tick = self._tick = TickInference(self.policy, self.n_slots, self.obs_dim, standardize=self.standardize_obs)
        tick.obs_host = self._current_obs
        tick.offset_dev.copy_(old.offset_dev)        # the sampler's counter stream goes on where it was
        idx = torch.from_numpy(src).to(self.device)
        return tick, tuple(x.index_select(1, idx) for x in slabs)

    @staticmethod
    def flatten(obs_slab, act_slab, logp_slab, rew, done, trunc, env_done, slot0):
        """Lock-step form (every process steps at every tick) of flatten_steps, kept for the fixture the reference's own
        collect_timesteps produced (tests/golden/collect.npz):
          obs_slab [T+1, S, D], act_slab [T, S] or [T, S, A], logp_slab [T, S] device f32;
          rew / done / trunc [T, S] host f32; env_done [T, procs] bool; slot0 [procs+1] first slot of every process."""
        T, n_procs = act_slab.shape[0], env_done.shape[1]
        seq = []
        for p in range(n_procs):
            lo, hi = int(slot0[p]), int(slot0[p + 1])
            seq.append(dict(tick=list(range(T)), rew=[rew[t, lo:hi] for t in range(T)],
                            done=[bool(done[t, lo]) for t in range(T)], trunc=[bool(trunc[t, lo]) for t in range(T)],
                            order=[t * n_procs + p for t in range(T)], ends=[bool(env_done[t, p]) for t in range(T)]))
        return BatchedAgentManager.flatten_steps(obs_slab, act_slab, logp_slab, seq, slot0, T)

    @staticmethod
    def flatten_steps(obs_slab, act_slab, logp_slab, seq, slot0, t_end):
        """Device slabs + per-process step lists -> the reference's flat rollout (batched_agent_manager.py:125-172 +
        BatchedTrajectory.get_all, batched_trajectory.py:58-105; SURVEY.md A.1): completed trajectories in completion
        order, then the still-open ones by process id; inside a trajectory agent after agent, each agent's steps in time
        order; the last step of every run is truncated iff it is not done (:145).
          seq[p]: tick[k] = slab row in which step k of process p was inferred; n[k] (optional, default: the slot width
          slot0[p+1]-slot0[p]) = agents that acted, in slots slot0[p]..; rew[k] [n[k]], done[k], trunc[k] what the
          environment answered; order[k] = global arrival number of that answer; ends[k] (optional) = the run ends here
          (default: done[k]); n_end (optional, default: the slot width) = agents after the last step.  The state after
          a process's last step is slab row t_end.
        A run also ends at a step after which the agent count changes (a run's agent set is constant).  At such a step
        an agent whose index no longer exists has no successor row: its next_states row is its own state.
        The index lists are built on the host (O(steps)); the data moves in device gathers."""
        dev = obs_slab.device
        S, D = obs_slab.shape[1], obs_slab.shape[2]
        runs = []           # (completion key, proc, k0, k1) with k1 inclusive
        n_open = 0
        n_after = []        # per process: agents of the observation each step produced
        for p, q in enumerate(seq):
            K = len(q["rew"])
            width = int(slot0[p + 1] - slot0[p])
            n = q.get("n", [width] * K)
            n_after.append(list(n[1:K]) + [q.get("n_end", width)])
            ends = q.get("ends", q["done"])
            k0 = 0
            for k in range(K):
                if ends[k] or n_after[p][k] != n[k]:
                    runs.append((0, q["order"][k], p, k0, k))
                    k0 = k + 1
            if k0 < K:
                runs.append((1, p, p, k0, K - 1))       # still open: after the completed ones, by process id
                n_open += 1
        runs.sort()
        row, nxt, rw, dn, tr, last_rows, pos = [], [], [], [], [], [], 0
        for _, _, p, k0, k1 in runs:
            q = seq[p]
            ticks = np.asarray(q["tick"][k0:k1 + 1], np.int64)
            nticks = np.asarray([q["tick"][k + 1] if k + 1 < len(q["tick"]) and k + 1 < len(q["rew"]) else t_end
                                 for k in range(k0, k1 + 1)], np.int64)
            after = np.asarray(n_after[p][k0:k1 + 1], np.int64)
            r = np.stack(q["rew"][k0:k1 + 1]).astype(np.float32)            # [steps, agents]
            d = np.asarray(q["done"][k0:k1 + 1], np.float32)
            t = np.asarray(q["trunc"][k0:k1 + 1], np.float32)
            for ai in range(r.shape[1]):
                s = int(slot0[p]) + ai
                row.append(ticks * S + s)
                nxt.append(np.where(ai < after, nticks, ticks) * S + s)
                rw.append(r[:, ai])
                dn.append(d)
                tr.append(t)
                pos += len(ticks)
                last_rows.append(pos - 1)
        cat = lambda xs, dt: np.concatenate(xs).astype(dt) if xs else np.zeros(0, dt)  # noqa: E731
        row, nxt = cat(row, np.int64), cat(nxt, np.int64)
        rw, dn, tr = cat(rw, np.float32), cat(dn, np.float32), cat(tr, np.float32)
        n_collected = int(row.shape[0])
        # f32 flags: the reference's list mixes np.float32 and Python ints and so comes out float64; the values are the same
        # 0/1 and the scan reads 4 instead of 8 bytes per step
        last_rows = np.asarray(last_rows, np.int64)
        tr[last_rows] = np.where(dn[last_rows] == 0, 1.0, 0.0)       # :145

        idx = torch.from_numpy(row).to(dev)
        states = torch.empty((n_collected, D), dtype=torch.float32, device=dev)
        next_states = torch.empty_like(states)
        log_probs = torch.empty(n_collected, dtype=torch.float32, device=dev)
        wide = act_slab.dim() == 3
        T = act_slab.shape[0]
        actions = torch.empty((n_collected, act_slab.shape[2]) if wide else (n_collected,), dtype=torch.float32, device=dev)
        src = _Slab(obs_slab.view(-1, D), None if wide else act_slab.view(-1), logp_slab.view(-1), None, None)
        ops.gather_batch(src, idx, out_actions=None if wide else actions, out_logp=log_probs, out_states=states)
        if wide:
            ops.gather_batch(_Slab(act_slab.view(T * S, -1), None, None, None, None), idx, out_states=actions)
        ops.gather_batch(_Slab(obs_slab.view(-1, D), None, None, None, None), torch.from_numpy(nxt).to(dev),
                         out_states=next_states)
        rewards, dones, truncated = (torch.from_numpy(x).to(dev) for x in (rw, dn, tr))
        return states, actions, log_probs, rewards, next_states, dones, truncated

    def cleanup(self):
        import traceback
        sel = getattr(self, "_selector", None)
        if sel is not None:
            sel.close()
            self._selector = None
        self._waiting = None
        for p, conn in self.processes:
            try:
                conn.send(("stop",))
            except Exception:
                pass
        for p, conn in self.processes:
            try:
                p.join(timeout=5)
                if p.is_alive():
                    p.terminate()
            except Exception:
                print("Unable to join process")
                traceback.print_exc()
            try:
                conn.close()
            except Exception:
                pass
        self.processes = []


class _Slab:
    """Adapter so ops.gather_batch (written for the experience ring) reads the time-major rollout slabs."""

    def __init__(self, states, actions, log_probs, values, advantages):
        self.states, self.actions, self.log_probs = states, actions, log_probs
        self.values, self.advantages = values, advantages
        self.states_bf16 = None
        self.obs_dim = states.shape[1]
        self.capacity = states.shape[0]
        self.start = 0
