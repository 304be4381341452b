"""One environment tick of batched policy inference for ALL env slots (replaces BatchedAgentManager._send_actions,
batched_agent_manager.py:180-221: np.concatenate of the ready observations, a small torch forward, multinomial,
`.cpu()`): the observations of every slot sit in one PINNED slab row, and a tick is

    H2D of the row -> [standardise + bf16 staging] -> fused policy kernel (MLP + categorical sample + log-prob)
                   -> D2H of the actions into pinned memory

captured ONCE as a CUDA graph and replayed per tick: one graph launch, one event wait on the host, no stream
synchronisation, no allocation.  The sampler's Philox offset lives in device memory (advanced inside the graph), the
standardisation statistics in fixed device buffers, so nothing a tick needs is baked into the graph.
Policies the fused kernel does not cover (other heads, very wide nets, precision="fp32") run the same sequence eagerly.
"""
import torch

from .. import _lib, ops


class TickInference(object):
    def __init__(self, policy, n_slots, obs_dim, standardize=False, clip=5.0):
        _lib.require_device()
        self.policy = policy
        st = policy._stack
        dev = st.device
        self.S, self.D = int(n_slots), int(obs_dim)
        self.standardize, self.clip = bool(standardize), float(clip)
        self.act_w = int(getattr(policy, "act_width", 1))
        self.obs_host = torch.empty((self.S, self.D), dtype=torch.float32).pin_memory()
        self.obs_raw = torch.empty((self.S, self.D), dtype=torch.float32, device=dev)
        # what the policy actually saw (standardised when enabled): the trajectory stores these rows
        self.obs_seen = torch.empty((self.S, self.D), dtype=torch.float32, device=dev) if self.standardize else self.obs_raw
        shape = (self.S,) if self.act_w == 1 else (self.S, self.act_w)
        self.act_dev = torch.empty(shape, dtype=torch.float32, device=dev)
        self.logp_dev = torch.empty(self.S, dtype=torch.float32, device=dev)
        self.act_host = torch.empty(shape, dtype=torch.float32).pin_memory()
        self.mean_dev = torch.zeros(self.D, dtype=torch.float32, device=dev)
        self.std_dev = torch.ones(self.D, dtype=torch.float32, device=dev)
        self.offset_dev = torch.zeros(1, dtype=torch.int64, device=dev)
        self.done_ev = torch.cuda.Event()
        self._graph = None
        self._warm = 0
        self._sig = None
        self.use_cuda_graph = True
        self.ticks = 0

    def set_obs_stats(self, mean, std):
        """mean / std: f32 [obs_dim] device tensors (enqueued copies into the fixed buffers the graph reads)."""
        self.mean_dev.copy_(mean, non_blocking=True)
        self.std_dev.copy_(std, non_blocking=True)

    @property
    def graphable(self):
        st = self.policy._stack
        return (self.use_cuda_graph and hasattr(self.policy, "n_actions") and st.fused_ok and _lib._TIMING is None)

    def _body(self, graph_mode):
        pol, st = self.policy, self.policy._stack
        self.obs_raw.copy_(self.obs_host, non_blocking=True)
        ws = st.workspace(self.S)
        if self.standardize:
            if st.exact:
                ops.rows_to_bf16(self.obs_raw, self._scratch(), self.mean_dev, self.std_dev, self.clip, dst_f32=self.obs_seen)
                st.stage_rows(self.obs_seen, ws["x"])
            else:
                ops.rows_to_bf16(self.obs_raw, ws["x"], self.mean_dev, self.std_dev, self.clip, dst_f32=self.obs_seen)
        else:
            st.stage_rows(self.obs_raw, ws["x"])
        if graph_mode:
            ops.policy_infer_fused(st.fused_net(ws["x"].stride(0), policy_head=True), ws["x"], self.S, pol.n_actions,
                                   seed=pol._seed, offset=0, offset_dev=self.offset_dev, actions_out=self.act_dev,
                                   logp_out=self.logp_dev)
            ops.u64_add(self.offset_dev, self.S)
        elif hasattr(pol, "n_actions"):                 # DiscreteFF, layer by layer
            h = st.forward_hidden(ws["x"], self.S, ws)
            if pol.wide:                                # above 256 actions: logits + per-row sampling kernel
                z, parts, ps = st.logits(h, self.S, ws)
                ops.head_discrete_sample(z, parts, ps, self.S, pol.n_actions, seed=pol._seed, offset=pol._offset,
                                         actions_out=self.act_dev, logp_out=self.logp_dev)
            else:
                st.policy_head_sample(h, self.S, pol.n_actions, seed=pol._seed, offset=pol._offset,
                                      actions_out=self.act_dev, logp_out=self.logp_dev)
            pol._offset += self.S
        else:                                           # MultiDiscreteFF / ContinuousPolicy: logits + per-row head kernel
            h = st.forward_hidden(ws["x"], self.S, ws)
            z, parts, ps = st.logits(h, self.S, ws)
            if hasattr(pol, "n_act"):
                ops.head_continuous_sample(z, parts, ps, self.S, pol.n_act, pol.var_min, pol.var_max, self.act_dev,
                                           self.logp_dev, seed=pol._seed, offset=pol._offset)
            else:
                ops.head_multi_discrete_sample(z, parts, ps, self.S, self.act_dev, self.logp_dev, seed=pol._seed,
                                               offset=pol._offset)
            pol._offset += self.S
        self.act_host.copy_(self.act_dev, non_blocking=True)

    def _scratch(self):
        sc = getattr(self, "_sc", None)
        if sc is None:
            sc = self._sc = torch.empty((self.S, ops.pad8(self.D)), dtype=torch.bfloat16, device=self.obs_raw.device)
        return sc

    def enqueue(self):
        """Enqueue one tick on the current stream (reads self.obs_host, fills act_dev / logp_dev / obs_seen / act_host)
        and record done_ev behind it.  Returns without waiting."""
        st = self.policy._stack
        st.refresh_operands()
        if self.graphable:
            sig = (getattr(st, "ws_gen", 0), id(self.policy), st.precision)
            if self._graph is not None and self._sig != sig:
                self._graph, self._warm = None, 0      # workspaces moved: re-capture
            if self._graph is None:
                if self._warm < 1:                     # first use eagerly: allocates workspaces, configures kernels
                    self._warm += 1
                    st.workspace(self.S)
                    self._sig = (getattr(st, "ws_gen", 0), id(self.policy), st.precision)
                    self._body(True)
                else:
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        self._body(True)
                    self._graph, self._sig = g, sig
                    g.replay()
            else:
                self._graph.replay()
        else:
            self._body(False)
        self.done_ev.record()
        self.ticks += 1

    def run(self):
        """One tick; returns the pinned action tensor once this tick's actions have landed in it."""
        self.enqueue()
        self.done_ev.synchronize()
        return self.act_host
