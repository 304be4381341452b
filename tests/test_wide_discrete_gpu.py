"""DiscreteFF with 257..4096 actions: the per-row head kernels (rlppo_head_discrete_*) against fp64 references applied
to the kernels' own logits, the bias-gradient column sums of heads wider than 2048, one PPOLearner.learn step against
the oracle in both precision modes, torch autograd, and two Learner iterations with collection on a scripted env."""
import os

import numpy as np
import pytest
import torch

from oracle import ref_oracle as O
from parity_helpers import capture_steps, close, philox_rows, philox_uniform, rel_l2, unflatten

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
WIDE = [257, 300, 1000, 2048, 2049, 4096]
NAMES = ("states", "actions", "log_probs", "rewards", "next_states", "dones", "truncated", "values", "advantages")
BF16 = torch.bfloat16


def pad8(n):
    return (n + 7) // 8 * 8


def pad64(n):
    return (n + 63) // 64 * 64


def logits(M, A, seed):
    """fp64 logits; every third row scaled up so that most of its probabilities fall below the 1e-11 clamp."""
    rng = np.random.RandomState(seed)
    z = rng.randn(M, A)
    z[::3] *= 12.0
    return torch.from_numpy(z)


def split3(z64):
    """fp64 [M, A] -> (bf16 [M, 3 * pad64(A)] with the fp32 value as hi | mid | lo parts, the parts' sum in fp64)."""
    M, A = z64.shape
    P = pad64(A)
    z32 = z64.float()
    hi = z32.to(BF16)
    r = z32 - hi.float()
    mid = r.to(BF16)
    lo = (r - mid.float()).to(BF16)
    buf = torch.zeros(M, 3 * P, dtype=BF16)
    buf[:, :A], buf[:, P:P + A], buf[:, 2 * P:2 * P + A] = hi, mid, lo
    return buf.to(DEV), hi.double() + mid.double() + lo.double(), P


def dz_buffer(M, A, parts):
    """d(logits) as Stack.dz_view lays it out: bf16 mode one part of pad8(A) columns, fp32 mode two parts pad64(A) apart.
    Pre-filled with ones so that the zeroed padding columns are checked too."""
    ps = pad64(A) if parts == 2 else 0
    buf = torch.ones(M, parts * pad64(A) if parts == 2 else pad8(A), dtype=BF16, device=DEV)
    return buf, ps, pad8(A)


def dz_value(buf, parts, ps, A):
    b = buf.double().cpu()
    out = b[:, :A].clone()
    for q in range(1, parts):
        out += b[:, q * ps:q * ps + A]
    return out, [b[:, q * ps + A:q * ps + pad8(A)] for q in range(parts)]


def assert_dz(got, want, parts):
    rtol = 4e-3 if parts == 1 else 1e-4
    atol = 1e-5 * float(want.abs().max())
    err = (got - want).abs()
    assert bool((err <= rtol * want.abs() + atol).all()), float((err - rtol * want.abs()).max())


@pytest.fixture(scope="module")
def ops():
    from rlgym_ppo_b200 import _lib, ops as o
    _lib.require_device()
    return o


# ---- 1. kernels against fp64 ------------------------------------------------------------------------------------
@pytest.mark.parametrize("A", WIDE)
def test_sample_probs_argmax_and_inverse_cdf(ops, A):
    M = 413
    zbuf, z, P = split3(logits(M, A, A))
    s = torch.softmax(z, -1)
    # probabilities (deterministic call) and the per-row argmax with its log-prob
    probs = torch.empty(M, A, device=DEV)
    acts = torch.empty(M, dtype=torch.int64, device=DEV)
    logp = torch.empty(M, device=DEV)
    ops.head_discrete_sample(zbuf, 3, P, M, A, deterministic=True, actions_i64_out=acts, logp_out=logp, probs_out=probs)
    torch.cuda.synchronize()
    assert torch.allclose(probs.double().cpu(), s, rtol=1e-4, atol=1e-7)
    assert torch.equal(acts.cpu(), z.argmax(-1))
    want_lp = torch.log(torch.clamp(1.0 / torch.exp(z - z.max(-1, keepdim=True).values).sum(-1), 1e-11, 1.0))
    assert torch.allclose(logp.double().cpu(), want_lp, rtol=0, atol=2e-5)
    # inverse CDF over the clamped probabilities with injected uniforms away from the bucket edges
    rng = np.random.RandomState(A + 1)
    u = torch.from_numpy(rng.rand(M))
    p = torch.clamp(s, 1e-11, 1.0)
    c = torch.cumsum(p, -1) / p.sum(-1, keepdim=True)
    keep = ((c - u[:, None]).abs().min(-1).values > 1e-5)
    want = (c > u[:, None]).double().argmax(-1)
    u_dev = u.float().to(DEV)
    acts_f = torch.empty(M, device=DEV)
    ops.head_discrete_sample(zbuf, 3, P, M, A, u=u_dev, actions_out=acts_f, actions_i64_out=acts, logp_out=logp)
    torch.cuda.synchronize()
    assert int(keep.sum()) > M // 2
    assert torch.equal(acts.cpu()[keep], want[keep])
    assert torch.equal(acts_f.cpu().long(), acts.cpu())
    got_lp = logp.double().cpu()[keep]
    want_lp = torch.log(p.gather(-1, want[:, None]).flatten())[keep]
    assert torch.allclose(got_lp, want_lp, rtol=0, atol=2e-5 * max(1.0, float(want_lp.abs().max())))
    # the Philox stream (counter (offset + row, high word, 0, 0), key (seed lo, seed hi)): a launch whose rows cross the
    # carry into the counter's high word draws exactly what the host restatement's uniforms draw when injected
    seed, off = 0x0123456789ABCDEF, 2 ** 32 - M // 2
    u_host = torch.from_numpy(philox_uniform(philox_rows(seed, off, M)[:, 0])).float().to(DEV)
    draws = []
    for kw in (dict(seed=seed, offset=off), dict(u=u_host)):
        a_, l_ = torch.empty(M, dtype=torch.int64, device=DEV), torch.empty(M, device=DEV)
        ops.head_discrete_sample(zbuf, 3, P, M, A, actions_i64_out=a_, logp_out=l_, **kw)
        draws.append((a_, l_))
    torch.cuda.synchronize()
    assert torch.equal(draws[0][0], draws[1][0]) and torch.equal(draws[0][1].view(torch.int32), draws[1][1].view(torch.int32))


def _ppo_reference(z, a, old, adv, inv_b, clip, ent_coef):
    """fp64 autograd of the PPO loss block (ppo_learner.py:146-180) over softmax -> clamp -> log (discrete_policy.py:64-80)."""
    zt = z.clone().requires_grad_(True)
    p = torch.clamp(torch.softmax(zt, -1), 1e-11, 1.0)
    lp_all = torch.log(p)
    logp = lp_all.gather(-1, a[:, None]).flatten()
    ent_rows = -(lp_all * p).sum(-1)
    ratio = torch.exp(logp - old)
    s1, s2 = ratio * adv, torch.clamp(ratio, 1.0 - clip, 1.0 + clip) * adv
    loss = (-torch.min(s1, s2).sum() - ent_coef * ent_rows.sum()) * inv_b
    loss.backward()
    with torch.no_grad():
        lr = logp - old
        kl = ((ratio - 1.0) - lr).sum()
        clipc = ((ratio - 1.0).abs() > clip).double().sum()
        surr = torch.min(s1, s2).sum()
    return logp.detach(), zt.grad, [float(ent_rows.detach().sum()), float(kl), float(clipc), float(surr),
                                    float(z.shape[0])]


@pytest.mark.parametrize("dz_parts", [1, 2])
@pytest.mark.parametrize("A", WIDE)
def test_train_logp_metrics_and_dz(ops, A, dz_parts):
    M = 413
    zbuf, z, P = split3(logits(M, A, 7 * A))
    rng = np.random.RandomState(A)
    a = rng.randint(0, A, M)
    a[5], a[6] = A + 7, -3                                 # stored actions outside the range are clamped
    a_ref = torch.from_numpy(np.clip(a, 0, A - 1))
    lp0 = torch.log(torch.clamp(torch.softmax(z, -1), 1e-11, 1.0)).gather(-1, a_ref[:, None]).flatten()
    old = lp0 + torch.from_numpy(rng.randn(M) * 0.3).float().double()
    adv = torch.from_numpy(rng.randn(M)).float().double()
    inv_b, clip, ent_coef = 1.0 / (2 * M), 0.2, 0.01
    want_lp, want_dz, want_m = _ppo_reference(z, a_ref, old, adv, inv_b, clip, ent_coef)
    dz, ps, cols = dz_buffer(M, A, dz_parts)
    metrics = torch.zeros(8, device=DEV)
    logp = torch.empty(M, device=DEV)
    ops.head_discrete_train(zbuf, 3, P, M, A, torch.from_numpy(a.astype(np.float32)).to(DEV), old.float().to(DEV),
                            adv.float().to(DEV), inv_b, clip, ent_coef, dz, dz_parts, ps, cols, metrics, logp_out=logp)
    torch.cuda.synchronize()
    assert torch.allclose(logp.double().cpu(), want_lp, rtol=0, atol=2e-5 * max(1.0, float(want_lp.abs().max())))
    m = metrics.double().cpu().tolist()
    assert abs(m[0] - want_m[0]) <= 1e-4 * abs(want_m[0]) + 1e-3, (m[0], want_m[0])
    assert abs(m[1] - want_m[1]) <= 1e-4 * abs(want_m[1]) + 1e-5 * M, (m[1], want_m[1])
    assert abs(m[2] - want_m[2]) <= 1.0, (m[2], want_m[2])
    assert abs(m[3] - want_m[3]) <= 1e-4 * abs(want_m[3]) + 1e-5 * M, (m[3], want_m[3])
    assert m[4] == M and m[5] == m[6] == m[7] == 0.0
    got, pads = dz_value(dz, dz_parts, ps, A)
    assert all(bool((t == 0).all()) for t in pads)
    assert_dz(got, want_dz, dz_parts)


@pytest.mark.parametrize("which", ["logp", "ent", "probs", "all"])
@pytest.mark.parametrize("A", [257, 1000, 2049, 4096])
def test_upstream_backward(ops, A, which):
    M = 333
    zbuf, z, P = split3(logits(M, A, 3 * A))
    rng = np.random.RandomState(A + 5)
    a = torch.from_numpy(rng.randint(0, A, M))
    zt = z.clone().requires_grad_(True)
    s = torch.softmax(zt, -1)
    p = torch.clamp(s, 1e-11, 1.0)
    lp = torch.log(p)
    outs = {"logp": lp.gather(-1, a[:, None]).flatten(), "ent": -(lp * p).sum(-1).mean(), "probs": s}
    grads = {"logp": torch.from_numpy(rng.randn(M)), "ent": torch.tensor(float(rng.randn())),
             "probs": torch.from_numpy(rng.randn(M, A))}
    keys = ["logp", "ent", "probs"] if which == "all" else [which]
    # the kernels read f32 upstream gradients: the reference takes the same rounded values
    grads = {k: v.float().double() for k, v in grads.items()}
    (want,) = torch.autograd.grad([outs[k] for k in keys], [zt], [grads[k] for k in keys])
    dev = {k: (grads[k].float().reshape(-1 if k == "ent" else grads[k].shape).to(DEV) if k in keys else None)
           for k in grads}
    if dev["ent"] is not None:
        dev["ent"] = dev["ent"].reshape(1)
    dz, ps, cols = dz_buffer(M, A, 2)
    ops.head_discrete_backward(zbuf, 3, P, M, A, a.float().to(DEV), dev["logp"], dev["ent"], dev["probs"], dz, 2, ps, cols)
    torch.cuda.synchronize()
    got, pads = dz_value(dz, 2, ps, A)
    assert all(bool((t == 0).all()) for t in pads)
    assert_dz(got, want, 2)


def test_philox_stream_chi_square(ops):
    """2^20 draws from one row of 300 logits with a fixed seed: the histogram against the probabilities (deterministic)."""
    from scipy.stats import chi2
    A, N = 300, 1 << 20
    row = torch.from_numpy(np.random.RandomState(0).randn(A)).float().to(BF16)
    zbuf = torch.zeros(N, pad8(A), dtype=BF16, device=DEV)
    zbuf[:, :A] = row.to(DEV)
    acts = torch.empty(N, dtype=torch.int64, device=DEV)
    ops.head_discrete_sample(zbuf, 1, 0, N, A, seed=0x5EED1234, offset=0, actions_i64_out=acts)
    again = torch.empty_like(acts)
    ops.head_discrete_sample(zbuf, 1, 0, N, A, seed=0x5EED1234, offset=0, actions_i64_out=again)
    moved = torch.empty_like(acts)
    ops.head_discrete_sample(zbuf, 1, 0, N, A, seed=0x5EED1234, offset=N, actions_i64_out=moved)
    torch.cuda.synchronize()
    assert torch.equal(acts, again) and not torch.equal(acts, moved)
    counts = np.bincount(acts.cpu().numpy(), minlength=A)
    assert counts.shape[0] == A
    p = torch.clamp(torch.softmax(row.double(), -1), 1e-11, 1.0)
    expected = (p / p.sum()).numpy() * N
    assert expected.min() > 5
    stat = float(((counts - expected) ** 2 / expected).sum())
    pval = float(chi2.sf(stat, A - 1))
    print(f"chi-square {stat:.1f} on {A - 1} dof, p = {pval:.3f}")
    assert pval > 1e-3, (stat, pval)


def test_argument_checks(ops):
    from rlgym_ppo_b200._lib import RlppoError
    zbuf, _, P = split3(logits(4, 256, 1))
    with pytest.raises(RlppoError, match="4096"):
        ops.head_discrete_sample(zbuf, 3, P, 4, 256, deterministic=True, logp_out=torch.empty(4, device=DEV))
    zbuf, _, P = split3(logits(4, 300, 1))
    with pytest.raises(RlppoError, match="logits view"):
        ops.head_discrete_sample(zbuf[:, 1:], 3, P, 4, 300, deterministic=True, logp_out=torch.empty(4, device=DEV))


# ---- 2. bias-gradient column sums wider than 2048 ----------------------------------------------------------------
@pytest.mark.parametrize("N", [2049, 3000, 4096])
def test_linear_wgrad_wide_column_sums(ops, N):
    M, K = 1000, 64
    rng = np.random.RandomState(N)
    dy = torch.zeros(M, pad8(N), dtype=BF16)
    dy[:, :N] = torch.from_numpy(rng.randn(M, N)).to(BF16)
    x = torch.from_numpy(rng.randn(M, K)).to(BF16)
    dw = torch.zeros(N, K, device=DEV)
    db = torch.zeros(N, device=DEV)
    ops.linear_wgrad(dy.to(DEV), x.to(DEV), dw, db, N, K, M=M)
    torch.cuda.synchronize()
    want_db = dy[:, :N].double().sum(0)
    want_dw = dy[:, :N].double().t() @ x.double()
    assert torch.allclose(db.double().cpu(), want_db, rtol=1e-5, atol=1e-3)
    assert torch.allclose(dw.double().cpu(), want_dw, rtol=1e-5, atol=1e-3)


# ---- 3. one PPOLearner.learn step against the oracle -----------------------------------------------------------------
def _problem(A, n, obs):
    rng = np.random.RandomState(A)
    states = rng.randn(n, obs).astype(np.float32)
    return dict(states=states, actions=rng.randint(0, A, n).astype(np.float32),
                log_probs=(-np.log(A) + rng.randn(n) * 0.3).astype(np.float32), rewards=np.zeros(n, np.float32),
                next_states=np.roll(states, -1, 0).copy(), dones=np.zeros(n, np.float32),
                truncated=np.zeros(n, np.float64), values=rng.randn(n).astype(np.float32),
                advantages=rng.randn(n).astype(np.float32))


def _learner(A, n, obs, layers, precision):
    import contextlib
    import io
    from rlgym_ppo_b200.ppo import PPOLearner
    torch.manual_seed(A)
    with contextlib.redirect_stdout(io.StringIO()):
        lr = PPOLearner(obs, A, 0, layers, layers, (0.1, 1.0), n, 1, 3e-4, 3e-4, 0.2, 0.01, n, DEV, precision=precision)
    assert lr.policy.wide
    return lr


SCALARS = ("Policy Entropy", "Mean KL Divergence", "Value Function Loss", "SB3 Clip Fraction")


@pytest.mark.parametrize("A", [300, 1000])
def test_learn_step_bf16_vs_oracle(A):
    from rlgym_ppo_b200.ppo import ExperienceBuffer
    n, obs, layers = 2000, 40, (64, 64)
    fields = _problem(A, n, obs)
    lr = _learner(A, n, obs, layers, "bf16")
    pol0 = [p.detach().cpu().clone() for p in lr.policy.parameters()]
    val0 = [p.detach().cpu().clone() for p in lr.value_net.parameters()]
    buf = ExperienceBuffer(n, 123, DEV)
    buf.submit_experience(*[fields[k] for k in NAMES])
    ob = O.BufferOracle(n, 123)
    ob.submit(**fields)
    orc = O.PPOLearnerOracle(pol0, val0, n, 1, 3e-4, 3e-4, 0.2, 0.01, n, quant=O.quant_bf16)
    want = orc.learn(ob)
    got = lr.learn(buf)
    for k in SCALARS:
        assert abs(got[k] - want[k]) <= 1e-3 * max(1.0, abs(want[k])), (k, got[k], want[k])
    for i, p in enumerate(lr.policy.parameters()):
        assert close(p.detach().cpu().numpy(), orc.pol[i].numpy(), 1e-3), ("pol", i)
        assert rel_l2(p.detach().cpu().numpy(), orc.pol[i].numpy()) < 1e-3, ("pol", i)
    for i, p in enumerate(lr.value_net.parameters()):
        assert close(p.detach().cpu().numpy(), orc.val[i].numpy(), 1e-3), ("val", i)
        assert rel_l2(p.detach().cpu().numpy(), orc.val[i].numpy()) < 1e-3, ("val", i)


@pytest.mark.parametrize("A", [300, 1000])
def test_learn_step_fp32_vs_fp64(A):
    from rlgym_ppo_b200.ppo import ExperienceBuffer
    n, obs, layers = 2000, 40, (64, 64)
    fields = _problem(A, n, obs)
    lr = _learner(A, n, obs, layers, "fp32")
    pol = [p.detach().cpu().double() for p in lr.policy.parameters()]
    val = [p.detach().cpu().double() for p in lr.value_net.parameters()]
    buf = ExperienceBuffer(n, 123, DEV)
    buf.submit_experience(*[fields[k] for k in NAMES])
    captured = capture_steps(lr)
    got = lr.learn(buf)
    assert len(captured) == 1
    grads = unflatten(lr, captured[0])
    ob = O.BufferOracle(n, 123)
    ob.submit(**fields)
    ((_, (b_acts, b_old, b_obs, b_tgt, b_adv)),) = list(ob.batches(n))
    t = lambda a: torch.from_numpy(a).double()      # noqa: E731
    pg, vg, mt = O.ppo_minibatch(pol, val, t(b_obs), torch.from_numpy(b_acts), t(b_old), t(b_tgt), t(b_adv), 0.2, 0.01, n)
    pg, vg = O.clip_grad_norm(pg, 0.5)[0], O.clip_grad_norm(vg, 0.5)[0]
    errs = [rel_l2(a, b.numpy()) for a, b in zip(grads, pg + vg)]
    print(f"A={A} fp32 post-clip gradient rel-L2 vs fp64 per tensor", [float(f"{e:.2e}") for e in errs])
    assert max(errs) < 1e-3, errs
    new_pol = O.AdamOracle(pol, 3e-4).step(list(pol), pg)
    new_val = O.AdamOracle(val, 3e-4).step(list(val), vg)
    for p, w in zip(list(lr.policy.parameters()) + list(lr.value_net.parameters()), new_pol + new_val):
        assert close(p.detach().cpu().numpy(), w.numpy(), 1e-3)
        assert rel_l2(p.detach().cpu().numpy(), w.numpy()) < 1e-3
    want = {"Policy Entropy": mt["entropy"], "Mean KL Divergence": mt["kl"], "Value Function Loss": mt["value_loss"],
            "SB3 Clip Fraction": mt["clip_fraction"]}
    for k in SCALARS:
        assert abs(got[k] - want[k]) <= 1e-3 * max(1.0, abs(want[k])), (k, got[k], want[k])


# ---- 4. torch autograd --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("method", ["get_output", "get_backprop_data"])
@pytest.mark.parametrize("A", [300, 2049])
def test_autograd_vs_cpu(A, method, precision):
    from rlgym_ppo_b200.ppo import DiscreteFF
    from rlgym_ppo_b200.ppo._mlp import build_sequential
    obs_dim, layers, n = 20, (64, 64), 129
    torch.manual_seed(3)
    rng = np.random.RandomState(4)
    m = DiscreteFF(obs_dim, A, layers, DEV, precision=precision)
    m.autograd = True
    obs = torch.from_numpy(rng.randn(n, obs_dim).astype(np.float32))
    acts = torch.from_numpy(rng.randint(0, A, (n, 1)).astype(np.float32))
    outs = m.get_output(obs.to(DEV)) if method == "get_output" else m.get_backprop_data(obs.to(DEV), acts)
    outs = outs if isinstance(outs, tuple) else (outs,)
    grads = [torch.from_numpy(np.asarray(rng.randn(*o.shape), dtype=np.float32)) for o in outs]
    for p in m.parameters():
        p.grad.zero_()
    torch.autograd.backward(outs, [g.to(DEV) for g in grads])
    got = [p.grad.detach().cpu().numpy().copy() for p in m.parameters()]

    def head(z):
        if method == "get_output":
            return (torch.softmax(z, -1),)
        p = torch.clamp(torch.softmax(z, -1), 1e-11, 1.0)
        lp = torch.log(p)
        return lp.gather(-1, acts.view(-1, 1).long()), -(lp * p).sum(-1).mean()

    sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    if precision == "fp32":
        seq = build_sequential(obs_dim, layers, A, softmax=False).double()
        seq.load_state_dict({k[len("model."):]: v.double() for k, v in sd.items()})
        torch.autograd.backward(head(seq(obs.double())), [g.double() for g in grads])
        want = [p.grad.numpy() for p in seq.parameters()]
    else:
        params = [v.float() for v in sd.values()]
        z, layer_in = O.mlp_forward(params, obs.float(), O.quant_bf16)
        zl = z.detach().requires_grad_(True)
        (dz,) = torch.autograd.grad(head(zl), [zl], grads)
        want = [g.numpy() for g in O.mlp_backward(params, layer_in, dz, O.quant_bf16)]
    errs = [rel_l2(a, b) for a, b in zip(got, want)]
    print(f"A={A} {method} {precision}: grad rel-L2 per tensor", [float(f"{e:.2e}") for e in errs])
    assert max(errs) <= (1e-3 if precision == "fp32" else 2e-3), errs


# ---- 5. Learner end to end --------------------------------------------------------------------------------------
class _Discrete:
    def __init__(self, n):
        self.n = n

    def seed(self, s):
        pass


class _Box:
    def __init__(self, shape):
        self.shape = shape


class WideEnv:
    """Two agents, 16-dim observations, Discrete(300), episodes of 23 steps; reward for action == argmax(obs) * 17."""
    N_AGENTS, OBS, ACT, LEN = 2, 16, 300, 23

    def __init__(self):
        self.action_space = _Discrete(self.ACT)
        self.observation_space = _Box((self.OBS,))
        self.rng = np.random.RandomState(os.getpid() % 1000)
        self.t = 0
        self.obs = None

    def reset(self):
        self.t = 0
        self.obs = self.rng.randn(self.N_AGENTS, self.OBS).astype(np.float32)
        return self.obs

    def step(self, actions):
        a = np.asarray(actions).reshape(self.N_AGENTS).astype(np.int64)
        assert a.min() >= 0 and a.max() < self.ACT
        rew = (a == self.obs.argmax(-1) * 17).astype(np.float32)
        self.t += 1
        self.obs = self.rng.randn(self.N_AGENTS, self.OBS).astype(np.float32)
        return self.obs, list(rew), self.t >= self.LEN, {"state": None}

    def close(self):
        pass


def make_wide_env():
    return WideEnv()


def test_learner_collects_and_learns_discrete_300(tmp_path):
    import contextlib
    import io
    from rlgym_ppo_b200 import Learner
    from rlgym_ppo_b200.ppo import PPOLearner
    folder = str(tmp_path / "ckpt")
    kw = dict(n_proc=2, min_inference_size=2, ts_per_iteration=600, exp_buffer_size=10000, ppo_batch_size=600,
              ppo_epochs=1, policy_layer_sizes=(64, 64), critic_layer_sizes=(64, 64), standardize_obs=False,
              standardize_returns=True, checkpoints_save_folder=folder, add_unix_timestamp=False,
              save_every_ts=10 ** 9, log_to_wandb=False, ppo_ent_coef=0.01)
    learner = Learner(make_wide_env, timestep_limit=1200, **kw)
    pol = learner.ppo_learner.policy
    assert pol.n_actions == WideEnv.ACT and pol.wide
    checked = []
    orig = learner.ppo_learner.learn

    def learn(buf):
        # the rows collected since the last update were sampled by the current policy: their stored log-probs are
        # get_backprop_data of the stored states and actions
        seen = sum(checked)
        states, actions, logp = buf.states[seen:], buf.actions[seen:], buf.log_probs[seen:]
        a = actions.cpu().numpy()
        assert a.min() >= 0 and a.max() < WideEnv.ACT and np.array_equal(a, np.round(a))
        with torch.no_grad():
            lp, ent = pol.get_backprop_data(states, actions)
        assert torch.allclose(lp.flatten(), logp.flatten(), rtol=0, atol=1e-5)
        assert 0.0 < float(ent) <= np.log(WideEnv.ACT) + 1e-4
        checked.append(states.shape[0])
        return orig(buf)

    learner.ppo_learner.learn = learn
    with contextlib.redirect_stdout(io.StringIO()):
        learner.learn()
    assert len(checked) == 2 and all(c >= 600 for c in checked)
    # checkpoint round trip
    with contextlib.redirect_stdout(io.StringIO()):
        learner.save(learner.agent.cumulative_timesteps)
        target = os.path.join(folder, str(learner.agent.cumulative_timesteps))
        lr2 = PPOLearner(WideEnv.OBS, WideEnv.ACT, 0, (64, 64), (64, 64), (0.1, 1.0), 600, 1, 3e-4, 3e-4, 0.2, 0.01, 600,
                         DEV)
        lr2.load_from(target)
    for k, v in pol.state_dict().items():
        assert torch.equal(v.cpu(), lr2.policy.state_dict()[k].cpu()), k
    x = torch.from_numpy(np.random.RandomState(9).randn(77, WideEnv.OBS).astype(np.float32))
    acts = torch.from_numpy(np.random.RandomState(10).randint(0, WideEnv.ACT, 77).astype(np.float32))
    with torch.no_grad():
        assert torch.equal(pol.get_backprop_data(x, acts)[0], lr2.policy.get_backprop_data(x, acts)[0])


# ---- 6. errors -------------------------------------------------------------------------------------------------------
def test_too_many_actions_raises_at_construction():
    from rlgym_ppo_b200.ppo import DiscreteFF
    with pytest.raises(ValueError, match="4096"):
        DiscreteFF(10, 4097, (64,), DEV)
    assert DiscreteFF(10, 4096, (64,), DEV).wide
    assert not DiscreteFF(10, 256, (64,), DEV).wide
