"""ContinuousPolicy on the B200 kernels (replaces rlgym_ppo/ppo/continuous_policy.py).

For N actions the network outputs 2N values through Tanh; the first half is the mean, the second half is mapped
linearly onto [var_min, var_max] and used as the standard deviation of a diagonal Gaussian (torch_functions.py:15-33).
Same constructor, `.model` state-dict (the Sequential ends in nn.Tanh like the reference's) and methods; the tail runs in
rlppo_head_continuous_{sample,train}.
"""
import torch

from .. import ops
from ._head_policy import HeadPolicy
from ._mlp import build_sequential, grad_f32

MAX_ACTIONS = 32     # widest action space rlppo_head_continuous_* serve (2 * 32 network outputs)


class ContinuousPolicy(HeadPolicy):
    def __init__(self, input_shape, output_shape, layer_sizes, device, var_min=0.1, var_max=1.0, precision=None):
        super().__init__()
        self.device = device
        assert int(output_shape) % 2 == 0, "ContinuousPolicy outputs a mean and a std per action"
        if not 1 <= int(output_shape) // 2 <= MAX_ACTIONS:
            raise ValueError(f"ContinuousPolicy supports 1 to {MAX_ACTIONS} actions, i.e. output_shape 2 to "
                             f"{2 * MAX_ACTIONS} (got {int(output_shape)})")
        self.n_act = int(output_shape) // 2
        self.act_width = self.n_act
        self.var_min, self.var_max = float(var_min), float(var_max)
        self.model = build_sequential(input_shape, layer_sizes, int(output_shape), softmax=False, tanh=True)   # :27-38
        self._init_stack(device, precision)

    def get_output(self, obs):
        """(mean, std) [.., N] each (:61-68): tanh, then the affine map of the second half.  Differentiable when `autograd` is
        set and grad mode is on."""
        def run():
            zview, n, _, lead = self._logits(obs)
            t = torch.tanh(self._logits_f32(zview, n)).view(*lead, 2 * self.n_act)
            m = (self.var_max - self.var_min) / 2.0              # torch_functions.py:27-28
            return (t[..., :self.n_act], t[..., self.n_act:] * m + (self.var_min + m)), n, None

        def head_kernel(logits, M, ws, grads, saved):
            self._head_bwd_kernel(logits(), M, None, None, None, grad_f32(grads[0], M, self.n_act),
                                  grad_f32(grads[1], M, self.n_act), self._stack.dz_view(ws))
        return self._with_autograd(obs, run, head_kernel)

    def forward(self, obs):
        return self.get_output(obs)

    def get_action_device(self, obs, deterministic=False):
        st = self._stack
        zview, n, _, lead = self._logits(obs)
        acts = torch.empty((n, self.n_act), dtype=torch.float32, device=st.device)
        logp = torch.empty(n, dtype=torch.float32, device=st.device)
        if n:
            z, parts, ps = zview
            ops.head_continuous_sample(z, parts, ps, n, self.n_act, self.var_min, self.var_max, acts, logp,
                                       seed=self._seed, offset=self._offset, deterministic=deterministic)
            self._offset += n
        return acts, logp, lead

    def get_action(self, obs, summed_probs=True, deterministic=False):
        """(action [.., N], summed log-prob [..]) as CPU tensors (:70-104); deterministic: (mean on the device, 0)."""
        if not summed_probs:
            raise NotImplementedError("summed_probs=False is not used anywhere on the reference's learner path")
        acts, logp, lead = self.get_action_device(obs, bool(deterministic))
        if deterministic:
            return acts.view(*lead, self.n_act), 0
        return acts.view(*lead, self.n_act).cpu(), logp.view(*lead).cpu()

    def _head_train_kernel(self, zview, M, actions, old_logp, adv, inv_b, clip, ent_coef, dzview, metrics, logp_out):
        z, parts, ps = zview
        dz, dparts, dps, dcols = dzview
        ops.head_continuous_train(z, parts, ps, M, self.n_act, self.var_min, self.var_max, actions, old_logp, adv, inv_b,
                                  clip, ent_coef, dz, dparts, dps, dcols, metrics, logp_out=logp_out)

    def _head_bwd_kernel(self, zview, M, actions, d_logp, d_ent, d_mean, d_std, dzview):
        z, parts, ps = zview
        dz, dparts, dps, dcols = dzview
        ops.head_continuous_backward(z, parts, ps, M, self.n_act, self.var_min, self.var_max, actions, d_logp, d_ent,
                                     d_mean, d_std, dz, dparts, dps, dcols)

    def get_backprop_data(self, obs, acts, summed_probs=True):
        """(summed log-pdf of `acts` [n], mean entropy over all n*N elements) (:106-120); differentiable when `autograd` is set and grad
        mode is on."""
        if not summed_probs:
            raise NotImplementedError("summed_probs=False is not used anywhere on the reference's learner path")
        return self._backprop_grad(obs, acts)
