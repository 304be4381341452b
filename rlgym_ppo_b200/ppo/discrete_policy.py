"""DiscreteFF on the B200 kernels (replaces rlgym_ppo/ppo/discrete_policy.py).

Same constructor, attributes (`.model`, `.n_actions`, `.device`) and state-dict as the reference; the arithmetic
runs in hand-written sm_100a kernels: bf16 tcgen05 GEMMs with fp32 TMEM accumulation for the Linear/ReLU stack,
and the softmax -> clamp(1e-11, 1) -> {multinomial sample | log-prob gather + entropy} tail fused into the
epilogue of the last GEMM (rlppo_policy_head_sample / rlppo_policy_head_train).

Up to 256 actions a row's logits fit the epilogue's tile.  Wider action spaces (257..4096, `wide`) run the last Linear
on its own (Stack.logits, fp32-exact split logits) followed by the per-row kernels rlppo_head_discrete_{sample,train,
backward}, with the same arithmetic.
"""
import numpy as np
import torch
import torch.nn as nn

from .. import ops
from ._mlp import BF16, Stack, StackFunction, autograd_wanted, build_sequential, grad_f32

EPILOGUE_MAX_ACTIONS = 256     # widest head the fused epilogue of the head GEMM serves
MAX_ACTIONS = 4096             # widest head the per-row kernels serve


class DiscreteFF(nn.Module):
    autograd = False    # True: differentiable get_output / forward / get_backprop_data (_mlp.autograd_wanted)

    def __init__(self, input_shape, n_actions, layer_sizes, device, precision=None):
        super().__init__()
        if int(n_actions) > MAX_ACTIONS:
            raise ValueError(f"DiscreteFF supports at most {MAX_ACTIONS} actions (got {int(n_actions)})")
        self.device = device
        self.model = build_sequential(input_shape, layer_sizes, n_actions, softmax=True)   # :22-31
        self.n_actions = int(n_actions)
        self.wide = self.n_actions > EPILOGUE_MAX_ACTIONS
        self._stack = Stack(self.model, device, precision)
        dev = self._stack.device
        # standalone arenas; PPOLearner re-binds both nets into one shared arena
        self._stack.bind(torch.zeros(self._stack.n_params, device=dev), torch.zeros(self._stack.n_params, device=dev))
        # Philox stream of the sampler: seeded from torch's generator at construction (Learner seeds torch first,
        # learner.py:95-97), advanced by the number of rows sampled
        self._seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        self._offset = 0
        self._obs_stats = None  # optional (mean, std, clip) device tensors: standardisation fused into staging

    def load_state_dict(self, state_dict, strict=True, assign=False):
        """Stock nn.Module.load_state_dict into the arena views, then the bf16 GEMM operands are rebuilt at once."""
        if assign:
            raise RuntimeError("assign=True would detach the parameters from the flat arena the kernels read")
        out = super().load_state_dict(state_dict, strict=strict)
        self._stack.refresh_operands(force=True)
        return out

    # nn.Module.to()/cuda()/cpu() would re-allocate parameters and silently break the arena views
    def _apply(self, fn, recurse=True):
        probe = fn(torch.empty(0, device=self._stack.device))
        if probe.device != self._stack.device or probe.dtype != torch.float32:
            raise RuntimeError("DiscreteFF lives on its CUDA device in fp32; it cannot be moved or cast")
        return self

    # ---- staging -------------------------------------------------------------------------------------------
    def _stage_obs(self, obs):
        """numpy / list / tensor -> bf16 [n, in_pad] device rows (the reference's as_tensor(float32), :35-41)."""
        st = self._stack
        if not isinstance(obs, torch.Tensor):
            obs = torch.as_tensor(np.asarray(obs))
        if obs.dtype not in (torch.float32,):
            obs = obs.to(torch.float32)
        obs = obs.reshape(-1, st.in_dim)
        if not obs.is_cuda:
            obs = obs.to(st.device, non_blocking=True)
        obs = obs.contiguous()
        n = obs.shape[0]
        ws = st.workspace(n)
        if self._obs_stats is not None:
            mean, std, clip = self._obs_stats
            st.stage_rows(obs, ws["x"], mean, std, clip)
        else:
            st.stage_rows(obs, ws["x"])
        return ws["x"], n, ws

    def _head_sample(self, obs, deterministic, want_probs):
        st = self._stack
        st.refresh_operands()
        x, n, ws = self._stage_obs(obs)
        dev = st.device
        acts = torch.empty(n, dtype=torch.int64, device=dev)
        logp = torch.empty(n, dtype=torch.float32, device=dev)
        if n and st.fused_ok and not want_probs:
            ops.policy_infer_fused(st.fused_net(x.stride(0), policy_head=True), x, n, self.n_actions, seed=self._seed,
                                   offset=self._offset, deterministic=deterministic, actions_i64_out=acts,
                                   logp_out=logp)
            self._offset += n
            return acts, logp, None
        h = st.forward_hidden(x, n, ws)
        probs = torch.empty((n, self.n_actions), dtype=torch.float32, device=dev) if want_probs else None
        if n and self.wide:
            z, parts, ps = st.logits(h, n, ws)
            ops.head_discrete_sample(z, parts, ps, n, self.n_actions, seed=self._seed, offset=self._offset,
                                     deterministic=deterministic, actions_i64_out=acts, logp_out=logp, probs_out=probs)
            self._offset += n
        elif n:
            st.policy_head_sample(h, n, self.n_actions, seed=self._seed, offset=self._offset,
                                  deterministic=deterministic, actions_i64_out=acts, logp_out=logp, probs_out=probs)
            self._offset += n
        return acts, logp, probs

    # ---- wide heads: last Linear -> per-row kernel -> the head's weight / data gradients ----------------------------
    def _wide_head_backward(self, h, M, ws, actions, d_logp, d_ent, d_probs, gw, gb):
        st = self._stack
        z, parts, ps = st.logits(h, M, ws)
        dz, dparts, dps, dcols = st.dz_view(ws)
        ops.head_discrete_backward(z, parts, ps, M, self.n_actions, actions, d_logp, d_ent, d_probs, dz, dparts, dps,
                                   dcols)
        return st.head_backward(h, M, ws, gw, gb)

    def _head_backward(self, h, M, ws, actions, d_logp, d_ent, d_probs, gw, gb):
        """Head backward for upstream gradients of (log-prob, mean entropy, probabilities).  Returns dL/dH_last."""
        if self.wide:
            return self._wide_head_backward(h, M, ws, actions, d_logp, d_ent, d_probs, gw, gb)
        return self._stack.policy_head_backward(h, M, ws, self.n_actions, actions, d_logp, d_ent, d_probs, gw, gb)

    def train_head(self, h, M, ws, actions, old_logp, adv, inv_b, clip, ent_coef, metrics, logp_out=None):
        """PPOLearner._train_chunk for wide heads: logits, the PPO block and its backward into d(logits), then the head's
        weight / bias gradients.  Returns dL/dH_last."""
        st = self._stack
        z, parts, ps = st.logits(h, M, ws)
        dz, dparts, dps, dcols = st.dz_view(ws)
        ops.head_discrete_train(z, parts, ps, M, self.n_actions, actions, old_logp, adv, inv_b, clip, ent_coef, dz, dparts,
                                dps, dcols, metrics, logp_out=logp_out)
        return st.head_backward(h, M, ws)

    # ---- reference surface -------------------------------------------------------------------------------------
    def get_output(self, obs):
        """Softmax probabilities [.., n_actions] (discrete_policy.py:35-42).  Differentiable with respect to the
        parameters when `autograd` is set and grad mode is on (_mlp.StackFunction)."""
        shape = tuple(obs.shape[:-1]) if hasattr(obs, "shape") else tuple(np.asarray(obs).shape[:-1])
        if autograd_wanted(self, obs):
            def run():
                probs = self._head_sample(obs, True, True)[2]
                return probs, probs.shape[0], None

            def head_backward(h, M, ws, grads, gw, gb, saved):
                return self._head_backward(h, M, ws, None, None, None, grad_f32(grads[0], M, self.n_actions), gw, gb)
            probs = StackFunction.apply(self._stack, run, head_backward, *self.parameters())
        else:
            _, _, probs = self._head_sample(obs, True, True)
        return probs.view(*shape, self.n_actions)

    def forward(self, obs):
        return self.get_output(obs)

    def get_action(self, obs, deterministic=False):
        """(action, log_prob) as CPU tensors (discrete_policy.py:44-62).  Sampling is an inverse-CDF draw over the
        clamped probabilities from a Philox4x32-10 stream (torch.multinomial's own stream is not reproducible
        outside torch; the distribution is the same)."""
        acts, logp, _ = self._head_sample(obs, bool(deterministic), False)
        if deterministic:
            # the reference returns `probs.cpu().numpy().argmax(), 0`: ONE flat argmax over the whole [n, A] array
            # (:56-57), meaningful for a batch of one.  Reproduce that contract from the per-row winners.
            a = acts.cpu().numpy()
            if a.shape[0] == 1:
                return a[0], 0
            lp = logp.cpu().numpy()
            row = int(np.argmax(lp))          # the largest clamped probability is the flat argmax's row
            return np.int64(row * self.n_actions + a[row]), 0
        return acts.cpu(), logp.cpu()

    def get_action_device(self, obs):
        """Same as get_action(deterministic=False) but leaves (actions int64, log_probs f32) on the device."""
        acts, logp, _ = self._head_sample(obs, False, False)
        return acts, logp

    def get_backprop_data(self, obs, acts):
        """(log-prob of `acts` [n,1], mean entropy) (discrete_policy.py:64-80).  Differentiable with respect to the
        parameters when `autograd` is set and grad mode is on (_mlp.StackFunction); PPOLearner.learn runs its own
        fused backward."""
        if autograd_wanted(self, obs):
            def run():
                logp, ent, acts_f = self._backprop_forward(obs, acts)
                return (logp, ent), logp.shape[0], acts_f.clone()

            def head_backward(h, M, ws, grads, gw, gb, acts_f):
                return self._head_backward(h, M, ws, acts_f, grad_f32(grads[0], M), grad_f32(grads[1], 1), None, gw, gb)
            return StackFunction.apply(self._stack, run, head_backward, *self.parameters())
        logp, ent, _ = self._backprop_forward(obs, acts)
        return logp, ent

    def _backprop_forward(self, obs, acts):
        st = self._stack
        st.refresh_operands()
        x, n, ws = self._stage_obs(obs)
        h = st.forward_hidden(x, n, ws)
        dev = st.device
        acts_f = torch.as_tensor(acts).to(device=dev, dtype=torch.float32).reshape(-1).contiguous()
        assert acts_f.numel() == n
        zeros = torch.zeros(n, dtype=torch.float32, device=dev)
        logp = torch.empty(n, dtype=torch.float32, device=dev)
        metrics = torch.zeros(8, dtype=torch.float32, device=dev)
        if self.wide:
            z, parts, ps = st.logits(h, n, ws)
            dz, dparts, dps, dcols = st.dz_view(ws)
            ops.head_discrete_train(z, parts, ps, n, self.n_actions, acts_f, zeros, zeros, 0.0, 0.2, 0.0, dz, dparts, dps,
                                    dcols, metrics, logp_out=logp)
            return logp.view(-1, 1), metrics[0] / metrics[4], acts_f
        hl = st.hidden[-1]
        sp = ops.make_split(3, 3, 3, 2, ops.pad64(hl), ops.pad64(hl), ops.pad64(st.out_dim)) if st.exact else None
        ops.policy_head_train(h, st.wq[-1], st.b[-1], self.n_actions, hl, acts_f, zeros, zeros, 0.0, 0.2,
                              0.0, ws["dz"], metrics, logp_out=logp, M=n, split=sp)
        entropy = metrics[0] / metrics[4]
        return logp.view(-1, 1), entropy, acts_f
