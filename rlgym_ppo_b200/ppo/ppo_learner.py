"""PPOLearner on the B200 kernels (replaces rlgym_ppo/ppo/ppo_learner.py).

Same constructor, attributes, `learn(exp) -> report`, `save_to` / `load_from` (same four .pt files) as the
reference.  What changes is how an optimiser step is executed (ppo_learner.py:119-195):

  reference                                           here
  ---------                                           ----
  CPU fancy-index + 5 H2D copies per minibatch        one device permutation-gather kernel (bf16 obs rows)
  nn.Sequential forward, autograd backward (fp32)     bf16 tcgen05 GEMMs, fp32 TMEM accumulators; the softmax /
                                                      clamp / log-prob / entropy / ratio / clip / KL / clip-fraction
                                                      / MSE math and its analytic backward (SURVEY.md A.3) fused
                                                      into the head kernels
  4 x .item() per minibatch, 2 x all params D2H       8 metric sums + 2 update norms accumulated on the device,
                                                      ONE readback per learn()
  clip_grad_norm_ x2 + Adam.step x2                   one norm kernel + one fused clip+Adam kernel over the flat
                                                      [policy | value] arena (separate norms, lrs, step counters)
  single device                                       data parallel: rank r takes slice r of every batch (exactly the
                                                      reference's minibatch slices), flat-arena NCCL allreduce,
                                                      identical optimiser step on every rank

Gradient accumulation over minibatches is a memory knob in the reference (sum of (mb/B)-scaled minibatch
gradients == full-batch gradient).  Here a rank's share of the batch is processed in chunks of at most
`max_chunk_rows` rows (activations for 131072 rows of the 2048-wide nets are ~3 GB of 180 GB), with the same
1/batch_size weighting, so `mini_batch_size` keeps its meaning for the result and stops costing launches.
"""
import os
import sys
import time

import numpy as np
import torch

from .. import _lib, ops, parallel
from .continuous_policy import ContinuousPolicy
from .discrete_policy import DiscreteFF
from .fused_adam import FusedAdam
from .multi_discrete_policy import MultiDiscreteFF
from .value_estimator import ValueEstimator


class PPOLearner(object):
    def __init__(
        self,
        obs_space_size,
        act_space_size,
        policy_type,
        policy_layer_sizes,
        critic_layer_sizes,
        continuous_var_range,
        batch_size,
        n_epochs,
        policy_lr,
        critic_lr,
        clip_range,
        ent_coef,
        mini_batch_size,
        device,
        max_chunk_rows=131072,
        process_group=None,
        dp_mode="replicated",
        dp_collective=None,
        precision=None,
    ):
        _lib.require_device()
        if device in (None, "auto", "gpu"):
            device = "cuda:%d" % torch.cuda.current_device()
        if "cuda" not in str(device):
            raise _lib.RlppoError(f"PPOLearner device must be a CUDA device (got {device!r}); there is no CPU path")
        self.device = device
        dev = torch.device(device)

        assert (
            batch_size % mini_batch_size == 0
        ), "MINIBATCH SIZE MUST BE AN INTEGER MULTIPLE OF BATCH SIZE"
        # precision of the Linear layers: "bf16" (throughput) or "fp32" (split operands, reference-grade gradients);
        # None = the package default (RLPPO_PRECISION / set_default_precision)
        obs_space_size = int(obs_space_size)
        self.policy_type = int(policy_type)
        if self.policy_type == 2:            # ppo_learner.py:34-50
            self.policy = ContinuousPolicy(obs_space_size, int(act_space_size) * 2, policy_layer_sizes, device,
                                           var_min=continuous_var_range[0], var_max=continuous_var_range[1],
                                           precision=precision)
        elif self.policy_type == 1:
            self.policy = MultiDiscreteFF(obs_space_size, policy_layer_sizes, device, precision=precision)
        else:
            self.policy = DiscreteFF(obs_space_size, act_space_size, policy_layer_sizes, device, precision)
        self._act_w = int(getattr(self.policy, "act_width", 1))
        self.value_net = ValueEstimator(obs_space_size, critic_layer_sizes, device, precision)
        self.precision = self.policy._stack.precision
        self.mini_batch_size = mini_batch_size

        # ---- one flat arena [policy | value] for params, grads and both Adam moments -------------------------
        ps, vs = self.policy._stack, self.value_net._stack
        n_p, n_v = ps.n_params, vs.n_params
        self._pg = process_group
        self.world_size, self.rank = parallel.world(process_group)
        # Data parallel: the 8 metric sums of an optimiser step ride at the end of the gradient arena as a third segment
        # with learning rate 0, so the gradient exchange (peer loads inside the optimiser launch, or the NCCL all-reduce)
        # sums them over the ranks too -- no separate metric collective, nothing NCCL inside an iteration on the p2p path.
        n_x = 8 if self.world_size > 1 else 0
        self._n_net = n_p + n_v
        self._seg = np.asarray([0, n_p, n_p + n_v] + ([n_p + n_v + n_x] if n_x else []), dtype=np.int64)
        n_seg = len(self._seg) - 1
        self._params = torch.zeros(n_p + n_v + n_x, dtype=torch.float32, device=dev)
        # Gradient exchange between data-parallel ranks (world_size > 1):
        #  "p2p"  (default): the gradient arena lives in symmetric memory every GPU of the box has mapped; the optimiser
        #         kernel itself sums the peers' arenas over NVLink in rank order (rlppo_norm_clip_adam_peers) -- no
        #         separate collective launch, and nothing NCCL inside the step, so a whole learn() stays ONE CUDA graph.
        #         `.grad` then holds this rank's own contribution; the summed gradient is `self._gsum`.
        #  "nccl": torch.distributed all_reduce on the flat arena between the backward and the optimiser launch.
        self.dp_collective = "none"
        self._grads = None
        if self.world_size > 1:
            self.dp_collective = parallel.choose_collective(self.world_size, n_p + n_v, dp_collective,
                                                            os.environ.get("RLPPO_DP_COLLECTIVE"))
            if self.dp_collective in ("p2p", "p2p2"):
                # Peer mappings need NVLink / P2P between all ranks' GPUs.  If the rendezvous fails on ANY rank, every rank
                # switches to the NCCL exchange (agreed through one all-reduce, so no rank is left waiting on flags).
                import torch.distributed as dist
                err = None
                try:
                    self._setup_peers(dev, n_p + n_v + n_x)
                except Exception as e:  # noqa: BLE001
                    err = e
                ok = torch.tensor([0 if err is not None else 1], dtype=torch.int32, device=dev)
                dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self._pg)
                if int(ok.item()) == 0:
                    if dp_collective in ("p2p", "p2p2"):
                        raise _lib.RlppoError(f"dp_collective='p2p' requested but peer mappings are unavailable: {err}")
                    print(f"[rlgym_ppo_b200] rank {self.rank}: symmetric-memory peer mappings unavailable ({err}); "
                          "gradients go through NCCL all_reduce", file=sys.stderr, flush=True)
                    self.dp_collective = "nccl"
                    self._grads = None
        if self._grads is None:
            self._grads = torch.zeros_like(self._params)
        self._m = torch.zeros_like(self._params)
        self._v = torch.zeros_like(self._params)
        self._before = torch.zeros_like(self._params)
        ps.bind(self._params[:n_p], self._grads[:n_p])
        vs.bind(self._params[n_p:n_p + n_v], self._grads[n_p:n_p + n_v])
        self._steps = torch.zeros(n_seg, dtype=torch.int64, device=dev)
        self._lr_dev = torch.zeros(n_seg, dtype=torch.float32, device=dev)
        self._lr_host = None
        self._sqnorm = torch.zeros(n_seg, dtype=torch.float32, device=dev)
        self._tail = torch.zeros(12, dtype=torch.float32, device=dev)   # metrics[0:8] | update sq-norms [8:10]
        self._tail_host = torch.zeros(12, dtype=torch.float32).pin_memory()

        self.policy_optimizer = FusedAdam(ps, policy_lr, self._m[:n_p], self._v[:n_p], self._steps[0:1])
        self.value_optimizer = FusedAdam(vs, critic_lr, self._m[n_p:n_p + n_v], self._v[n_p:n_p + n_v], self._steps[1:2])

        policy_params_count, critic_params_count = n_p, n_v
        total_parameters = policy_params_count + critic_params_count
        print("Trainable Parameters:")
        print(f"{'Component':<10} {'Count':<10}")
        print("-" * 20)
        print(f"{'Policy':<10} {policy_params_count:<10}")
        print(f"{'Critic':<10} {critic_params_count:<10}")
        print("-" * 20)
        print(f"{'Total':<10} {total_parameters:<10}")
        print(f"Current Policy Learning Rate: {policy_lr}")
        print(f"Current Critic Learning Rate: {critic_lr}")

        self.n_epochs = n_epochs
        self.batch_size = batch_size
        self.clip_range = clip_range
        self.ent_coef = ent_coef
        self.cumulative_model_updates = 0
        self.max_chunk_rows = int(max_chunk_rows)

        # ---- data parallelism ---------------------------------------------------------------------------------
        # Data-parallel modes (world_size > 1; one process per GPU, NCCL through torch.distributed):
        #  "replicated": every rank holds the SAME experience buffer and draws the same global permutation; rank r takes
        #                slice r of every batch -- exactly the reference's minibatch slices (ppo_learner.py:134-143), so the
        #                result equals the single-process one.  batch_size is the GLOBAL batch.
        #  "sharded":    every rank holds its OWN experience (its own env workers) and shuffles it with its own stream;
        #                batch_size is the PER-RANK batch, the optimiser step averages over world_size * batch_size
        #                samples.  Nothing but gradients (and a few scalars) crosses NVLink: this is the weak-scaling mode.
        assert dp_mode in ("replicated", "sharded")
        self.dp_mode = dp_mode
        if dp_mode == "replicated":
            assert batch_size % self.world_size == 0, "batch_size must be a multiple of the number of ranks"
        self._mb = None
        self.launches = 0   # kernels enqueued by the last learn() (bench.py reports it)
        self._views_sig = None
        self._sync_operand_views()
        # CUDA graphs: one optimiser step (gather -> fwd/bwd -> clip+Adam) is ~25 launches of 2-170 us kernels; replaying
        # a captured graph removes the Python/ctypes/driver launch cost that otherwise dominates the example-size nets
        self.use_cuda_graph = True
        self._nb_final = None
        self._graphs = {}
        self.max_graphs = 16        # captured graphs kept (each owns a private memory pool); the oldest is dropped beyond
        self._graph_warm = set()
        self._idx_cur = None
        self._perm_dev = None

    def _setup_peers(self, dev, n):
        """Gradient arena + flag block in symmetric memory (torch.distributed._symmetric_memory: CUDA peer mappings over
        NVLink); a collective call -- every rank constructs its learners in the same order."""
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm_mem
        group = self._pg if self._pg is not None else dist.group.WORLD
        grads = symm_mem.empty(n, dtype=torch.float32, device=dev)
        grads.zero_()
        gh = symm_mem.rendezvous(grads, group)
        flags = symm_mem.empty(int(_lib._lib.rlppo_peer_flag_bytes()) // 4, dtype=torch.int32, device=dev)
        flags.zero_()
        fh = symm_mem.rendezvous(flags, group)
        torch.cuda.synchronize(dev)
        dist.barrier(group)                         # every rank's flag block is zero before anyone launches
        self._grads = grads
        self._peer_grad_ptrs = [int(x) for x in gh.buffer_ptrs]
        self._peer_flag_ptrs = [int(x) for x in fh.buffer_ptrs]
        self._symm = (grads, gh, flags, fh)         # keep the mappings alive
        # Return-normalisation scale of rank 0, double buffered by iteration parity: in "sharded" mode every rank's GAE
        # kernel reads it straight out of rank 0's memory (a peer load), so the per-iteration Welford broadcast disappears
        # (Learner.add_new_experience).  Both slots start at 1 (the std of an empty WelfordRunningStat).
        slots = symm_mem.empty(4, dtype=torch.float32, device=dev)
        slots.fill_(1.0)
        sh = symm_mem.rendezvous(slots, group)
        self._std_slots_local = slots
        self._std_slots_rank0 = sh.get_buffer(0, (4,), torch.float32) if self.rank != 0 else slots
        self._symm += (slots, sh)
        torch.cuda.synchronize(dev)
        dist.barrier(group)
        if self.dp_collective == "p2p2":
            # two-shot form (experimental): the reduced gradient lives in symmetric memory too, peers read its slices
            gsum = symm_mem.empty(n, dtype=torch.float32, device=dev)
            gsum.zero_()
            rh = symm_mem.rendezvous(gsum, group)
            torch.cuda.synchronize(dev)
            dist.barrier(group)
            self._gsum = gsum
            self._peer_red_ptrs = [int(x) for x in rh.buffer_ptrs]
            self._symm += (gsum, rh)
        else:
            self._gsum = torch.zeros(n, dtype=torch.float32, device=dev)

    # ---- workspaces ----------------------------------------------------------------------------------------
    def _minibatch_buffers(self, rows):
        """The gathered minibatch (bf16 observation rows + the per-sample scalars)."""
        cur = self._mb
        if cur is None or cur["rows"] < rows:
            dev = self._params.device
            f = lambda: torch.empty(rows, dtype=torch.float32, device=dev)  # noqa: E731
            self._mb_gen = getattr(self, "_mb_gen", 0) + 1
            ps = self.policy._stack
            cur = {"rows": rows, "actions": f(), "old_logp": f(), "targets": f(), "adv": f()}
            if self._act_w > 1:      # action rows (batch_acts.view(batch_size, -1), ppo_learner.py:131)
                cur["actions"] = torch.empty((rows, self._act_w), dtype=torch.float32, device=dev)
            if ps.exact:
                # "fp32" mode: the f32 observation rows are gathered and split into 3 bf16 parts (both nets read them)
                cur["x32"] = torch.empty((rows, ps.in_dim), dtype=torch.float32, device=dev)
                cur["x"] = torch.zeros((rows, 3 * ps.in_ps), dtype=torch.bfloat16, device=dev)
            else:
                cur["x"] = torch.zeros((rows, ps.in_pad), dtype=torch.bfloat16, device=dev)
            self._mb = cur
        return cur

    def _gather(self, exp, idx, M, mb):
        """Rows idx[0:M] of the experience rings into a minibatch buffer set, on the current stream."""
        if self.policy._stack.exact:
            exp.gather(idx, out_actions=mb["actions"], out_logp=mb["old_logp"], out_values=mb["targets"],
                       out_adv=mb["adv"], out_states=mb["x32"])
            self.policy._stack.stage_rows(mb["x32"][:M], mb["x"])
            self.launches += 1
        else:
            exp.gather(idx, out_actions=mb["actions"], out_logp=mb["old_logp"], out_values=mb["targets"],
                       out_adv=mb["adv"], out_states_bf16=mb["x"])

    def _sync_lr(self):
        lr = (float(self.policy_optimizer.param_groups[0]["lr"]), float(self.value_optimizer.param_groups[0]["lr"]))
        if lr != self._lr_host:
            pad = (0.0,) * (self._lr_dev.numel() - 2)          # the metric segment never moves
            self._lr_dev.copy_(torch.tensor(lr + pad, dtype=torch.float32))
            self._lr_host = lr

    def _sync_operand_views(self):
        """Which bf16 operands the optimiser launch refreshes.  A stack that runs on the fused kernels needs no transposed
        weight copies (its backward data GEMMs read W itself as an MN-major operand); the layer-wise kernels do.  Re-checked
        before every batch: tests and experiments switch paths on a live learner (force_layerwise)."""
        ps, vs = self.policy._stack, self.value_net._stack
        sig = (ps.fused_ok and self.policy_type == 0, vs.fused_ok)
        if sig == self._views_sig:
            return
        for st, fused in zip((ps, vs), sig):
            was = st.need_wt
            st.need_wt = not fused
            if st.need_wt and not was and st.params is not None:
                st.refresh_operands(force=True)
        views = ps.bf16_views(0) + vs.bf16_views(ps.n_params)
        self._views = (_lib.Bf16View * len(views))(*views)
        self._views_sig = sig

    # ---- one chunk of one batch: gather -> fwd -> fused heads -> bwd (grads accumulate) -------------------------
    def _train_chunk(self, exp, idx, M):
        self._sync_operand_views()
        mb = self._minibatch_buffers(M)
        self._gather(exp, idx, M, mb)
        x = mb["x"]
        # (1/mb) * (mb/B), ppo_learner.py:172-177; B = the number of samples one optimiser step averages over
        inv_b = 1.0 / float(parallel.samples_per_step(self.batch_size, self.world_size, self.dp_mode))
        metrics = self._step_metrics()
        n = 1
        if self.policy_type == 0 and self.policy._stack.fused_ok and self.value_net._stack.fused_ok:
            # Both nets in ONE persistent launch: 2 x ceil(M/128) work items (policy tiles first) dealt out over
            # one CTA per SM, then every weight (and bias) gradient of both nets in one launch.  Two launches, one per
            # net, would each end on a partly filled round of tiles: 391 tiles over 148 CTAs.
            ps, vs = self.policy._stack, self.value_net._stack
            wp, wv = ps.workspace(M), vs.workspace(M)
            ops.policy_value_train_fused(ps.fused_net(x.stride(0), wp, policy_head=True), vs.fused_net(x.stride(0), wv), x, M,
                                         self.policy.n_actions, mb["actions"], mb["old_logp"], mb["adv"], inv_b,
                                         float(self.clip_range), float(self.ent_coef), vs.w[-1], mb["targets"], vs.gw[-1],
                                         metrics)
            ops.wgrad_multi(ps.fused_wgrad_items(x, wp, head_dy=wp["dz"]) + vs.fused_wgrad_items(x, wv), M)
            self.launches += 3
            return
        wg_items = []
        for net, is_policy in ((self.policy, True), (self.value_net, False)):
            st = net._stack
            ws = st.workspace(M)
            if st.fused_ok and (not is_policy or self.policy_type == 0):
                # one persistent kernel: forward, fused head, backward data path, bias gradients (mlp_fused.cu)
                if is_policy:
                    fnet = st.fused_net(x.stride(0), ws, policy_head=True)
                    ops.policy_train_fused(fnet, x, M, net.n_actions, mb["actions"], mb["old_logp"], mb["adv"], inv_b,
                                           float(self.clip_range), float(self.ent_coef), metrics)
                    wg_items += st.fused_wgrad_items(x, ws, head_dy=ws["dz"])
                else:
                    fnet = st.fused_net(x.stride(0), ws)
                    ops.value_train_fused(fnet, x, M, st.w[-1], mb["targets"], inv_b, st.gw[-1], metrics)
                    wg_items += st.fused_wgrad_items(x, ws)
                n += 1
                continue
            h = st.forward_hidden(x, M, ws)
            if is_policy and self.policy_type != 0:
                # MultiDiscrete / Continuous: last Linear -> per-row head kernel -> head wgrad / dgrad
                dh = net.train_head(h, M, ws, mb["actions"], mb["old_logp"], mb["adv"], inv_b, float(self.clip_range),
                                    float(self.ent_coef), metrics)
                n += 5 + (1 if st.exact else 0)
            elif is_policy:
                dh = st.policy_head_train(h, M, ws, net.n_actions, mb["actions"], mb["old_logp"], mb["adv"], inv_b,
                                          float(self.clip_range), float(self.ent_coef), metrics)
                n += 4 + (1 if st.exact else 0)      # head GEMM, wgrad, colsum (per dz part), dgrad
            else:
                dh = st.value_head_train(h, M, ws, mb["targets"], inv_b, metrics)
                n += 1
            st.backward_hidden(x, M, ws, dh)
            L = len(st.hidden)
            n += L + 2 * L + (L - 1)   # fwd GEMMs, wgrad + colsum per layer, dgrad for all but the first
        if wg_items:
            ops.wgrad_multi(wg_items, M)       # every weight gradient of both nets: one persistent launch
            n += (len(wg_items) + 7) // 8
        self.launches += n

    def _step_metrics(self):
        """Where the kernels of the current optimiser step accumulate their 8 metric sums: the running totals directly
        (one rank), or the tail of the gradient arena (data parallel: summed over ranks with the gradients, then added to
        the totals by _collect_step_metrics)."""
        if self.world_size > 1:
            return self._grads[self._n_net:self._n_net + 8]
        return self._tail[0:8]

    def _collect_step_metrics(self, summed):
        if self.world_size > 1:
            self._tail[0:8].add_(summed[self._n_net:self._n_net + 8])

    def _optimizer_step(self):
        if self.dp_collective == "p2p2":
            ops.norm_clip_adam_peers2(self._params, self._peer_grad_ptrs, self._peer_flag_ptrs, self._peer_red_ptrs,
                                      self.rank, self._m, self._v, self._seg, self._sqnorm, self._lr_dev, self._steps,
                                      max_norm=0.5, views=self._views if len(self._views) else None)
            self._collect_step_metrics(self._gsum)
            self._operands_after_step()
            self.launches += 1
            return
        if self.dp_collective == "p2p":
            # the all-reduce happens inside the optimiser launch (peer loads over NVLink, rank-order sum)
            ops.norm_clip_adam_peers(self._params, self._peer_grad_ptrs, self._peer_flag_ptrs, self.rank, self._gsum,
                                     self._m, self._v, self._seg, self._sqnorm, self._lr_dev, self._steps, max_norm=0.5,
                                     views=self._views if len(self._views) else None)
            self._collect_step_metrics(self._gsum)
            self._operands_after_step()
            self.launches += 1
            return
        parallel.allreduce_sum_(self._grads, self._pg)   # NCCL sum over NVLink; the gradients carry the global 1/B
        self._apply_step()

    def _operands_after_step(self):
        """bf16 mode: the optimiser launch has rewritten the bf16 operands itself (views).  "fp32" mode: the split
        operands are rebuilt here (one small launch per Linear, inside the same graph)."""
        for st in (self.policy._stack, self.value_net._stack):
            if st.exact:
                st.refresh_operands(force=True)
                self.launches += len(st.linears)
            else:
                st.mark_operands_fresh()

    def _apply_step(self):
        # ppo_learner.py:187-193 in one launch: fixed-order (deterministic) norms -> clip -> Adam -> bf16 operand refresh
        ops.norm_clip_adam(self._params, self._grads, self._m, self._v, self._seg, self._sqnorm, self._lr_dev,
                           self._steps, max_norm=0.5, views=self._views if len(self._views) else None)
        self._collect_step_metrics(self._grads)
        self._operands_after_step()
        self.launches += 1

    def _backward_body(self, exp, idx, local, chunk):
        self._grads.zero_()                                     # ppo_learner.py:131-132
        for c0 in range(0, local, chunk):
            rows = min(chunk, local - c0)
            self._train_chunk(exp, idx[c0:c0 + rows], rows)

    def _batch_body(self, exp, idx, local, chunk):
        self._backward_body(exp, idx, local, chunk)
        self._optimizer_step()

    def _captured(self, key, fn):
        """Replay `fn` as a CUDA graph (captured on its second use: the first run allocates workspaces and configures
        kernel attributes eagerly).  Returns False when the caller has to run `fn` eagerly itself."""
        entry = self._graphs.get(key)
        if entry is None:
            if key not in self._graph_warm:
                self._graph_warm.add(key)
                return False
            calls0, launches0 = _lib.CALLS, self.launches
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                fn()
            entry = (graph, _lib.CALLS - calls0, self.launches - launches0)
            self.launches = launches0
            _lib.CALLS = calls0
            while len(self._graphs) >= self.max_graphs:      # oldest first: dicts keep insertion order
                old = next(iter(self._graphs))
                del self._graphs[old]
                self._graph_warm.discard(old)
            self._graphs[key] = entry
        graph, n_calls, n_launch = entry
        graph.replay()
        _lib.CALLS += n_calls
        self.launches += n_launch
        return True

    def _batch_step(self, exp, idx, local, chunk):
        """One optimiser step on this rank's share `idx` of a batch: eager, or as replayed CUDA graphs.  With several
        ranks the step is two graphs (forward/backward, clip+Adam) with the NCCL allreduce between them."""
        if not self.use_cuda_graph or _lib._TIMING is not None:
            self._batch_body(exp, idx, local, chunk)
            return
        if self._idx_cur is None or self._idx_cur.numel() < local:
            self._idx_cur = torch.empty(local, dtype=torch.int64, device=self._params.device)
        cur = self._idx_cur[:local]
        cur.copy_(idx)      # the graph reads its indices from a fixed buffer; the ring origin from exp.start_dev
        key = self._graph_key(exp, local, chunk) + (self._idx_cur.data_ptr(),)
        if self.world_size == 1 or self.dp_collective in ("p2p", "p2p2"):
            if not self._captured(("step",) + key, lambda: self._batch_body(exp, cur, local, chunk)):
                self._batch_body(exp, cur, local, chunk)
        else:
            if not self._captured(("bwd",) + key, lambda: self._backward_body(exp, cur, local, chunk)):
                self._backward_body(exp, cur, local, chunk)
            parallel.allreduce_sum_(self._grads, self._pg)
            if not self._captured(("opt",) + key, self._apply_step):
                self._apply_step()
        self.policy._stack.mark_operands_fresh()
        self.value_net._stack.mark_operands_fresh()

    def _graph_key(self, exp, local, chunk):
        """Everything a captured graph bakes in: buffer identity, workspace generations (addresses), scalar arguments."""
        return (exp.uid, local, chunk, float(self.clip_range), float(self.ent_coef), self.batch_size, self.world_size,
                self.dp_mode, self.dp_collective, self.precision, self.policy_type, self.policy._stack.fused_ok, self.value_net._stack.fused_ok, getattr(self, "_mb_gen", 0),
                getattr(self.policy._stack, "ws_gen", 0), getattr(self.value_net._stack, "ws_gen", 0))

    def _learn_body(self, exp, n_batches, local, chunk, tail=True):
        """Device work of one learn() call (ppo_learner.py:110-220): update-magnitude baseline, every optimiser step of
        every epoch (indices from self._perm_dev, one row per epoch), update magnitudes, the report scalars to pinned
        host memory.  Enqueue only -- this is what the whole-call CUDA graph captures."""
        B, R = self.batch_size, self.world_size
        self._before.copy_(self._params)          # update-magnitude baseline (:110-116), stays on the device
        self._tail.zero_()
        steps = [(epoch, parallel.rank_rows(k, B, self.rank, R, self.dp_mode)[0])
                 for epoch in range(self.n_epochs) for k in range(n_batches)]
        idx_of = lambda i: self._perm_dev[steps[i][0], steps[i][1]:steps[i][1] + local]  # noqa: E731
        for i in range(len(steps)):
            self._batch_body(exp, idx_of(i), local, chunk)
        ops.sqdiff(self._before, self._params, self._seg, self._tail[8:8 + len(self._seg) - 1])
        if tail:
            self._tail_host.copy_(self._tail, non_blocking=True)      # metric sums are global already (see __init__)

    def learn(self, exp):
        """
        Compute PPO updates with an experience buffer (ppo_learner.py:92-238).
        Returns the reference's report dictionary (same keys).
        """
        self.launches = 0
        self.policy._stack.refresh_operands()
        self.value_net._stack.refresh_operands()
        self._sync_lr()

        t1 = time.time()
        B, R, E = self.batch_size, self.world_size, self.n_epochs
        local = parallel.rank_rows(0, B, self.rank, R, self.dp_mode)[1]
        chunk = min(local, self.max_chunk_rows)
        total = len(exp)
        n_batches = total // B                                  # experience_buffer.py:100, remainder dropped
        if R > 1 and self.dp_mode == "sharded":
            # Every rank must run the same number of optimiser steps (each one is a rendezvous): agree on the minimum over
            # the ranks' own buffers -- a host collective outside the iteration's graph, needed only while buffers are still
            # filling: once EVERY rank reports a full ring (its length can no longer change) the agreed count is final and
            # the steady state has no collective outside the optimiser launch.
            full = int(total >= getattr(exp, "max_size", total + 1))
            if not (self._nb_final is not None and full):
                nb = torch.tensor([n_batches, full], dtype=torch.int64, device=self._params.device)
                torch.distributed.all_reduce(nb, op=torch.distributed.ReduceOp.MIN)
                n_batches = int(nb[0].item())
                self._nb_final = n_batches if int(nb[1].item()) == 1 else None
            else:
                n_batches = self._nb_final
        # One `rng.permutation(total)` per epoch (experience_buffer.py:98), drawn in the reference's order, uploaded into
        # one [epochs, total] device buffer before any device work: the whole call is then a single graph replay.
        fresh = self._perm_dev is None or self._perm_dev.shape[0] != E or self._perm_dev.shape[1] < total
        if fresh:
            self._perm_dev = torch.empty((E, max(total, 1)), dtype=torch.int64, device=self._params.device)
        for epoch in range(E):
            exp.next_permutation_into(self._perm_dev[epoch, :total], fresh_alloc=fresh)
        n_iterations = E * n_batches

        p2p = R > 1 and self.dp_collective in ("p2p", "p2p2")
        whole = self.use_cuda_graph and _lib._TIMING is None and n_batches > 0 and (R == 1 or p2p)
        if whole:
            # data parallel over peer memory: the graph holds the WHOLE call, the report readback included
            tail = True
            key = ("learn", total, E, n_batches, tail, self._perm_dev.data_ptr()) + self._graph_key(exp, local, chunk)
            if not self._captured(key, lambda: self._learn_body(exp, n_batches, local, chunk, tail)):
                self._learn_body(exp, n_batches, local, chunk, tail)
            self.policy._stack.mark_operands_fresh()
            self.value_net._stack.mark_operands_fresh()
        else:
            self._before.copy_(self._params)
            self._tail.zero_()
            for epoch in range(E):
                for k in range(n_batches):
                    base = parallel.rank_rows(k, B, self.rank, R, self.dp_mode)[0]
                    self._batch_step(exp, self._perm_dev[epoch, base:base + local], local, chunk)
            # ---- report: one device -> host readback for the whole call ---------------------------------------
            ops.sqdiff(self._before, self._params, self._seg, self._tail[8:8 + len(self._seg) - 1])
            self._tail_host.copy_(self._tail, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        t = self._tail_host.double().numpy()
        avg = parallel.report_from_sums(t[0:8])

        if n_iterations == 0:
            n_iterations = 1
        self.cumulative_model_updates += n_iterations

        report = {
            "PPO Batch Consumption Time": (time.time() - t1) / n_iterations,
            "Cumulative Model Updates": self.cumulative_model_updates,
            "Policy Entropy": avg["Policy Entropy"],
            "Mean KL Divergence": avg["Mean KL Divergence"],
            "Value Function Loss": avg["Value Function Loss"],
            "SB3 Clip Fraction": avg["SB3 Clip Fraction"],
            "Policy Update Magnitude": float(np.sqrt(t[8])),
            "Value Function Update Magnitude": float(np.sqrt(t[9])),
        }
        return report

    # ---- checkpoints: the reference's four files, stock torch formats (ppo_learner.py:240-271) -------------------
    def save_to(self, folder_path):
        os.makedirs(folder_path, exist_ok=True)
        cpu = lambda sd: {k: v.detach().cpu().clone() for k, v in sd.items()}  # noqa: E731
        torch.save(cpu(self.policy.state_dict()), os.path.join(folder_path, "PPO_POLICY.pt"))
        torch.save(cpu(self.value_net.state_dict()), os.path.join(folder_path, "PPO_VALUE_NET.pt"))
        torch.save(_optim_to_cpu(self.policy_optimizer.state_dict()),
                   os.path.join(folder_path, "PPO_POLICY_OPTIMIZER.pt"))
        torch.save(_optim_to_cpu(self.value_optimizer.state_dict()),
                   os.path.join(folder_path, "PPO_VALUE_NET_OPTIMIZER.pt"))

    def load_from(self, folder_path):
        assert os.path.exists(folder_path), "PPO LEARNER CANNOT FIND FOLDER {}".format(folder_path)
        dev = self._params.device
        self.policy.load_state_dict(torch.load(os.path.join(folder_path, "PPO_POLICY.pt"), map_location=dev))
        self.value_net.load_state_dict(torch.load(os.path.join(folder_path, "PPO_VALUE_NET.pt"), map_location=dev))
        self.policy_optimizer.load_state_dict(
            torch.load(os.path.join(folder_path, "PPO_POLICY_OPTIMIZER.pt"), map_location=dev))
        self.value_optimizer.load_state_dict(
            torch.load(os.path.join(folder_path, "PPO_VALUE_NET_OPTIMIZER.pt"), map_location=dev))
        self._lr_host = None


def _optim_to_cpu(sd):
    state = {i: {k: (v.detach().cpu() if isinstance(v, torch.Tensor) else v) for k, v in s.items()}
             for i, s in sd["state"].items()}
    return {"state": state, "param_groups": sd["param_groups"]}
