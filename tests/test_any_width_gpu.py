"""GPU tests: networks whose hidden widths are not multiples of 8, and the value head above 2048 inputs.

A hidden layer of width h runs on the device as pad8(h) units whose extra units are inert (Stack in ppo/_mlp.py).
Covered here:
  1. rlppo_value_head / rlppo_value_head_backward at any K (register form up to 2048, shared-memory form above) against
     fp64, with guard regions after dw / db and the padding columns of dH;
  2. rlppo_linear_dgrad's fused bias gradient at widths 300 and 4: exactly K entries change;
  3. zero extension: a (300, 100) net and a (304, 104) net holding the same function give bit-identical outputs, and
     train to the same parameters while the extra units stay exactly zero;
  4. one PPOLearner.learn step against the oracle for all three policy types, in both precision modes, and a
     (256, 3000) critic;
  5. torch autograd through a (300, 100) DiscreteFF and ValueEstimator;
  6. a Learner with (500, 500) / (300, 3000) nets collecting and learning, with a checkpoint round trip.

Run with `pytest -m gpu` on a B200."""
import contextlib
import io
import os

import numpy as np
import pytest
import torch

from oracle import ref_oracle as O
from parity_helpers import DEV, SENTINEL, bits, capture_steps, close, recon, rel_l2, sentinel, split_rows, unflatten

pytestmark = pytest.mark.gpu

U = 2.0 ** -24


@pytest.fixture(scope="module")
def ops():
    from rlgym_ppo_b200 import _lib, ops as _ops
    _lib.require_device()
    return _ops


def pad8(n):
    return (n + 7) // 8 * 8


def pad64(n):
    return (n + 63) // 64 * 64


def _hprev(M, K, seed):
    """A ReLU output with tiny positives and -0.0 among ordinary values."""
    g = torch.Generator().manual_seed(seed)
    h = torch.relu(torch.randn(M, K, generator=g))
    pick = torch.randint(0, 6, (M, K), generator=g)
    h[pick == 0] = 1e-30
    h[pick == 1] = -0.0
    return h


def _guarded(vals, dev=DEV):
    """f32 device buffer: `vals` followed by 16 NaN sentinels; returns (buffer, view of the first len(vals))."""
    n = vals.numel()
    buf = torch.full((n + 16,), float("nan"), dtype=torch.float32)
    buf[:n] = vals
    buf = buf.to(dev)
    return buf, buf[:n]


def _guard_intact(buf, n):
    return bool((buf[n:].cpu().view(torch.int32) == torch.full((16,), float("nan")).view(torch.int32)).all())


# ---- 1. value head at any K ----------------------------------------------------------------------------------------
KS = [1, 3, 7, 12, 100, 300, 2047, 2049, 3000, 4096]


@pytest.mark.parametrize("split", [False, True], ids=["bf16", "split"])
@pytest.mark.parametrize("mode", ["infer", "train", "upstream"])
@pytest.mark.parametrize("K", KS)
def test_value_head_any_k(ops, K, mode, split):
    """Bounds as test_split_kernels_gpu.py::test_value_head_split / test_value_head_backward, with the summation depth
    of either kernel form: (8 ceil(K/256) + 14) u (sum_k |h w| + |b|) for v; dH one product rounded to its parts; dw, db
    sums of M terms.  H rows span pad8(K) columns (padding zero); dH's padding columns must come out +0, the columns
    past pad8(K) (and every column past each part's pad8(K) in the split layout) keep their sentinel, and nothing after
    dw[K-1] or db[0] changes."""
    M = 2600                      # > 296 wide-form tiles of 8 rows: the grid-stride loop takes a second round
    k8 = pad8(K)
    g = torch.Generator().manual_seed(K)
    h = _hprev(M, K, 7 + K)
    w = torch.randn(K, generator=g) * 0.1
    b = torch.tensor([0.3])
    if split:
        kp = pad64(K)
        hbuf = split_rows(ops, h, 3, kp)
        hkw = dict(h_parts=3, h_pstride=kp)
        hd = recon(hbuf, 3, kp, K)
        assert bool((bits(hbuf.cpu()).view(M, 3, kp)[:, :, K:] == 0).all())
        d_ps = k8 + 8
        dh = sentinel(M, 2 * d_ps)
        dkw = dict(dh_parts=2, dh_pstride=d_ps)
        rnd = 2.0 ** -16 + U
    else:
        hb = torch.zeros((M, k8), dtype=torch.bfloat16)
        hb[:, :K] = h.bfloat16()
        hbuf, hkw, hd = hb.to(DEV), {}, hb[:, :K].double()
        d_ps = 0
        dh = sentinel(M, k8 + 8)
        dkw = {}
        rnd = 2.0 ** -8 + U
    wd = w.double()
    dw0 = torch.randn(K, generator=g)
    dwbuf, dw = _guarded(dw0)
    dbbuf, db = _guarded(torch.tensor([0.5]))
    mask = (hd > 0).double()
    if mode == "upstream":
        d_v = torch.randn(M, generator=g)
        ops.value_head_backward(hbuf, w.to(DEV), K, d_v.to(DEV), dh, dw, db, **hkw, **dkw)
        torch.cuda.synchronize()
        d64, ddv = d_v.double(), torch.zeros(M, dtype=torch.float64)
    else:
        tgt = torch.randn(M, generator=g)
        v = torch.empty(M, device=DEV)
        metrics = torch.zeros(8, device=DEV)
        inv_b = 1.0 / (3 * M)
        if mode == "train":
            ops.value_head(hbuf, w.to(DEV), b.to(DEV), K, values_out=v, targets=tgt.to(DEV), inv_batch=inv_b, dh=dh,
                           dw=dw, db=db, metrics=metrics, **hkw, **dkw)
        else:
            ops.value_head(hbuf, w.to(DEV), b.to(DEV), K, values_out=v, **hkw)
        torch.cuda.synchronize()
        v64 = hd @ wd + 0.3
        v_err = (8 * ((K + 255) // 256) + 14) * U * (hd.abs() @ wd.abs() + 0.3)
        assert bool(((v.cpu().double() - v64).abs() <= v_err).all())
        if mode == "infer":
            assert bool((bits(dh.cpu()) == SENTINEL).all())
            assert torch.equal(dw.cpu(), dw0) and float(db.cpu()) == 0.5
            assert _guard_intact(dwbuf, K) and _guard_intact(dbbuf, 1)
            return
        d64 = 2 * inv_b * (v64 - tgt.double())
        ddv = 2 * inv_b * (v_err + U * (v64 - tgt.double()).abs()) + 2 * U * d64.abs()
        m = metrics.cpu().double()
        sq = float(((v64 - tgt.double()) ** 2).sum())
        assert m[6] == M
        assert abs(m[5] - sq) <= 1e-5 * sq
    dh_ref = d64[:, None] * wd[None, :] * mask
    dh_bound = (wd.abs()[None, :] * ddv[:, None] + rnd * dh_ref.abs()) * mask
    got = recon(dh, 2, d_ps, K) if split else dh.cpu()[:, :K].double()
    assert bool(((got - dh_ref).abs() <= dh_bound + 1e-300).all())
    xb = bits(dh.cpu())
    for q in range(2 if split else 1):
        blk = xb[:, q * d_ps:q * d_ps + k8]
        assert bool((blk[:, :K][mask == 0] == 0).all())
        assert bool((blk[:, K:k8] == 0).all()), "dH padding columns must be +0"
        assert bool((xb[:, q * d_ps + k8:(q + 1) * d_ps if split else None] == SENTINEL).all())
    dw_ref = (d64[:, None] * hd).sum(0) + dw0.double()
    dw_bound = (hd.abs() * ddv[:, None]).sum(0) + (M + 1) * U * ((d64.abs()[:, None] * hd).sum(0) + dw0.double().abs())
    assert bool(((dw.cpu().double() - dw_ref).abs() <= dw_bound).all())
    db_ref = float(d64.sum()) + 0.5
    assert abs(float(db.cpu()) - db_ref) <= float(ddv.sum()) + (M + 1) * U * (float(d64.abs().sum()) + 0.5)
    assert _guard_intact(dwbuf, K) and _guard_intact(dbbuf, 1)


def test_value_head_argument_checks(ops):
    from rlgym_ppo_b200._lib import RlppoError
    h = torch.zeros((4, 16), dtype=torch.bfloat16, device=DEV)
    w = torch.zeros(16, device=DEV)
    with pytest.raises(RlppoError, match="covering pad8"):       # ldh 8 < pad8(9)
        ops.value_head(h[:, :8].contiguous(), w, None, 9, values_out=torch.empty(4, device=DEV))
    with pytest.raises(RlppoError, match=r"K must be in \[1,"):
        ops.value_head(h, w, None, 0, values_out=torch.empty(4, device=DEV))


# ---- 2. linear_dgrad's fused bias gradient bounded by the true width -------------------------------------------------
@pytest.mark.parametrize("split", [False, True], ids=["bf16", "split"])
@pytest.mark.parametrize("K", [300, 4])
def test_linear_dgrad_db_below_true_width(ops, K, split):
    """dX over pad8(K) columns (padding columns +0), db_below += column sums of the stored dX over exactly K entries:
    the 16 floats after them (the next parameter, in the arena) stay bit-identical."""
    M, N = 1000, 64
    k8 = pad8(K)
    g = torch.Generator().manual_seed(K)
    dy = torch.randn(M, N, generator=g)
    w = torch.randn(N, K, generator=g) * 0.1
    h = _hprev(M, K, 30 + K)
    db0 = torch.randn(K, generator=g)
    dbbuf, db = _guarded(db0)
    if split:
        d_ps = pad64(max(N, K))
        dys = split_rows(ops, dy, 2, d_ps)
        hs = split_rows(ops, h, 3, pad64(K))
        wt = torch.zeros((k8, 2 * pad64(N)), dtype=torch.bfloat16, device=DEV)
        ops.weight_split(w.to(DEV).contiguous(), None, 0, 0, wt, 2, pad64(N))
        dx = sentinel(M, 2 * d_ps)
        ops.linear_dgrad(dys, wt, hs, dx, N, K, M=M, db_below=db,
                         split=ops.make_split(2, 2, 2, 2, d_ps, pad64(N), d_ps))
        torch.cuda.synchronize()
        mask = (recon(hs, 3, pad64(K), K) > 0).double()
        got = recon(dx, 2, d_ps, K)
        ref = (dy.double() @ w.double()) * mask
        assert rel_l2(got, ref) < 1e-4
        xb = bits(dx.cpu())
        for q in range(2):
            assert bool((xb[:, q * d_ps + K:q * d_ps + k8] == 0).all())
            assert bool((xb[:, q * d_ps + k8:(q + 1) * d_ps] == SENTINEL).all())
        want = db0.double() + got.sum(0)
        assert float((db.cpu().double() - want).abs().max()) <= 1e-4 * max(1.0, float(want.abs().max()))
    else:
        hb = torch.zeros((M, k8), dtype=torch.bfloat16)
        hb[:, :K] = h.bfloat16()
        wt = torch.zeros((k8, N), dtype=torch.bfloat16)
        wt[:K] = w.t().bfloat16()
        dx = sentinel(M, k8 + 8)
        ops.linear_dgrad(dy.bfloat16().to(DEV), wt.to(DEV), hb.to(DEV), dx, N, K, db_below=db)
        torch.cuda.synchronize()
        mask = (hb[:, :K].double() > 0).double()
        ref = (dy.bfloat16().double() @ w.bfloat16().double()) * mask
        got = dx.cpu()[:, :K].double()
        assert rel_l2(got, ref) < 4e-3
        xb = bits(dx.cpu())
        assert bool((xb[:, K:k8] == 0).all())
        assert bool((xb[:, k8:] == SENTINEL).all())
        want = db0.double() + got.sum(0)
        assert float((db.cpu().double() - want).abs().max()) <= 1e-4 * max(1.0, float(want.abs().max()))
    assert _guard_intact(dbbuf, K)


# ---- 3. zero extension: (300, 100) and (304, 104) hold the same function ---------------------------------------------
ACT = {0: 9, 1: 8, 2: 3}      # Discrete(9); MultiDiscrete (its own 21 logits); Continuous with 3 actions


def _ppo(ptype, pol_layers, crit_layers, precision, B, seed=5):
    from rlgym_ppo_b200.ppo import PPOLearner
    torch.manual_seed(seed)
    with contextlib.redirect_stdout(io.StringIO()):
        return PPOLearner(23, ACT[ptype], ptype, pol_layers, crit_layers, (0.1, 1.0), B, 1, 3e-4, 3e-4, 0.2, 0.01, B, DEV,
                          precision=precision)


def _zero_extend(src, dst):
    sd = {}
    for k, v in src.state_dict().items():
        z = torch.zeros_like(dst.state_dict()[k])
        z[tuple(slice(0, s) for s in v.shape)] = v
        sd[k] = z
    dst.load_state_dict(sd)


def _outputs(ptype, pol, obs):
    outs = []
    with torch.no_grad():
        for o in (pol.get_output(obs), pol.forward(obs)):
            outs += list(o) if isinstance(o, tuple) else [o]
    outs += [torch.as_tensor(t) for t in pol.get_action(obs.cpu().numpy(), deterministic=True)]
    outs += [torch.as_tensor(t) for t in pol.get_action(obs.cpu().numpy())]
    return outs


def _buffer(ptype, lr, states, rng):
    from rlgym_ppo_b200.ppo import ExperienceBuffer
    B = states.shape[0]
    acts, logp = lr.policy.get_action(states)
    acts = np.asarray(acts, dtype=np.float32).reshape(B, -1)
    old = (np.asarray(logp, dtype=np.float32).reshape(B) + rng.randn(B) * 0.3).astype(np.float32)
    fields = (states, acts if acts.shape[1] > 1 else acts.reshape(B), old, (rng.randn(B) * 0.1).astype(np.float32),
              np.roll(states, -1, 0).copy(), np.zeros(B, np.float32), np.zeros(B, np.float64),
              rng.randn(B).astype(np.float32), rng.randn(B).astype(np.float32))
    return fields


def _arena_views(lr, flat, net):
    """Per-parameter views of a flat learner arena (params / grads / Adam moments) for `net` (policy or value_net)."""
    off = 0 if net is lr.policy else lr.policy._stack.n_params
    out = []
    for p in net.parameters():
        out.append(flat[off:off + p.numel()].view(p.shape))
        off += p.numel()
    return out


def _pad_is_zero(t, true_shape):
    """Every entry of t outside the leading block of true_shape is exactly +0 (bit pattern)."""
    t = t.detach().cpu()
    keep = torch.zeros(t.shape, dtype=torch.bool)
    keep[tuple(slice(0, s) for s in true_shape)] = True
    raw = t.view(torch.int16) if t.dtype == torch.bfloat16 else t.view(torch.int32)
    return bool((raw[~keep] == 0).all())


def _operand_padding_zero(st):
    """wq / wt (and their split parts) of stack `st`: rows and columns past the true [out, in] block are +0."""
    for i, lin in enumerate(st.linears):
        o, n = lin.out_features, lin.in_features
        if st.exact:
            ps = pad64(n)
            for q in range(3):
                if not _pad_is_zero(st.wq[i][:, q * ps:(q + 1) * ps], (o, n)):
                    return False
            if st.wt[i] is not None:
                pt = pad64(o)
                for q in range(2):
                    if not _pad_is_zero(st.wt[i][:, q * pt:(q + 1) * pt], (n, o)):
                        return False
        else:
            if not _pad_is_zero(st.wq[i], (o, n)):
                return False
            if st.wt[i] is not None and not _pad_is_zero(st.wt[i], (n, o)):
                return False
    return True


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("ptype", [0, 1, 2])
def test_zero_extension_equivalence(ptype, precision):
    B = 512
    a = _ppo(ptype, (300, 100), (300, 100), precision, B)
    b = _ppo(ptype, (304, 104), (304, 104), precision, B)
    for na, nb in ((a.policy, b.policy), (a.value_net, b.value_net)):
        _zero_extend(na, nb)
    b.policy._seed, b.policy._offset = a.policy._seed, a.policy._offset
    assert not a.policy._stack.fused_ok and not b.policy._stack.fused_ok
    rng = np.random.RandomState(ptype)
    obs = torch.from_numpy(rng.randn(300, 23).astype(np.float32)).to(DEV)
    for x, y in zip(_outputs(ptype, a.policy, obs), _outputs(ptype, b.policy, obs)):
        assert torch.equal(x.cpu(), y.cpu())
    with torch.no_grad():
        assert torch.equal(a.value_net(obs).cpu(), b.value_net(obs).cpu())
    states = rng.randn(B, 23).astype(np.float32)
    fields = _buffer(ptype, a, states, rng)
    from rlgym_ppo_b200.ppo import ExperienceBuffer
    bufs = []
    for _ in range(2):
        buf = ExperienceBuffer(B, 123, DEV)
        buf.submit_experience(*fields)
        bufs.append(buf)
    for _ in range(3):
        ra, rb = a.learn(bufs[0]), b.learn(bufs[1])
    for k in ("Policy Entropy", "Mean KL Divergence", "Value Function Loss", "SB3 Clip Fraction"):
        assert abs(ra[k] - rb[k]) <= 1e-5 * max(1.0, abs(ra[k])), (k, ra[k], rb[k])
    for na, nb in ((a.policy, b.policy), (a.value_net, b.value_net)):
        for pa, pb, gb, mb, vb in zip(na.parameters(), nb.parameters(), _arena_views(b, b._grads, nb),
                                      _arena_views(b, b._m, nb), _arena_views(b, b._v, nb)):
            for t in (pb, gb, mb, vb):
                assert _pad_is_zero(t, pa.shape), "extra units must stay exactly zero"
            shared = pb.detach()[tuple(slice(0, s) for s in pa.shape)].cpu()
            ref = pa.detach().cpu()
            # not bit for bit: the weight-gradient kernels add with fp32 atomics in no fixed order, and the gradient
            # norm's fixed summation order depends on the arena length.  Adam turns a last-bit change of a gradient
            # near eps into up to ~1e-7 of weight change; 2e-6 is test_learner_gpu.py's chunk-invariance bound.
            assert float((shared - ref).abs().max()) <= 2e-6, float((shared - ref).abs().max())
        assert _operand_padding_zero(na._stack)


# ---- 4. one learn step against the oracle --------------------------------------------------------------------------
def _problem(ptype, lr, B, rng):
    states = rng.randn(B, 23).astype(np.float32)
    return _buffer(ptype, lr, states, rng)


FIELD_NAMES = ("states", "actions", "log_probs", "rewards", "next_states", "dones", "truncated", "values", "advantages")


def _fp32_step_vs_fp64(ptype, pol_layers, crit_layers):
    from rlgym_ppo_b200.ppo import ExperienceBuffer
    B = 512
    lr = _ppo(ptype, pol_layers, crit_layers, "fp32", B, seed=60 + ptype)
    pol0 = [p.detach().cpu().double() for p in lr.policy.parameters()]
    val0 = [p.detach().cpu().double() for p in lr.value_net.parameters()]
    rng = np.random.RandomState(70 + ptype)
    fields = _problem(ptype, lr, B, rng)
    buf = ExperienceBuffer(B, 123, DEV)
    buf.submit_experience(*fields)
    captured = capture_steps(lr)
    got = lr.learn(buf)
    assert len(captured) == 1
    grads = unflatten(lr, captured[0])
    ob = O.BufferOracle(B, 123)
    ob.submit(**dict(zip(FIELD_NAMES, fields)))
    ((_, (b_acts, b_old, b_obs, b_tgt, b_adv)),) = list(ob.batches(B))
    t = lambda a: torch.from_numpy(a).double()      # noqa: E731
    if ptype == 0:
        pg, vg, mt = O.ppo_minibatch(pol0, val0, t(b_obs), torch.from_numpy(b_acts), t(b_old), t(b_tgt), t(b_adv), 0.2,
                                     0.01, B)
    else:
        pg, vg, mt = O.ppo_minibatch_head(ptype, pol0, val0, t(b_obs), t(b_acts), t(b_old), t(b_tgt), t(b_adv), 0.2,
                                          0.01, B, (0.1, 1.0))
    pg, vg = O.clip_grad_norm(pg, 0.5)[0], O.clip_grad_norm(vg, 0.5)[0]
    wants = [w.numpy() for w in pg + vg]
    n_pol = len(pg)
    norms = [np.sqrt(sum(float((w ** 2).sum()) for w in wants[:n_pol])),
             np.sqrt(sum(float((w ** 2).sum()) for w in wants[n_pol:]))]
    errs = [float(np.abs(a - w).max()) / norms[0 if i < n_pol else 1] if w.size == 1 else rel_l2(a, w)
            for i, (a, w) in enumerate(zip(grads, wants))]
    print(f"ptype {ptype} {pol_layers}/{crit_layers} fp32: grad rel-L2 per tensor", [float(f"{e:.2e}") for e in errs])
    assert max(errs) < 1e-3, errs
    new_pol = O.AdamOracle(pol0, 3e-4).step(list(pol0), pg)
    new_val = O.AdamOracle(val0, 3e-4).step(list(val0), vg)
    for p, w in zip(list(lr.policy.parameters()) + list(lr.value_net.parameters()), new_pol + new_val):
        assert close(p.detach().cpu().numpy(), w.numpy(), 1e-3)
        assert rel_l2(p.detach().cpu().numpy(), w.numpy()) < 1e-3
    want = {"Policy Entropy": mt["entropy"], "Mean KL Divergence": mt["kl"], "Value Function Loss": mt["value_loss"],
            "SB3 Clip Fraction": mt["clip_fraction"]}
    for k, v in want.items():
        assert abs(got[k] - v) <= 1e-3 * max(1.0, abs(v)), (k, got[k], v)


@pytest.mark.parametrize("ptype", [0, 1, 2])
def test_learn_step_fp32_vs_fp64(ptype):
    _fp32_step_vs_fp64(ptype, (300, 12), (4,))


def test_wide_critic_learn_step_fp32_vs_fp64():
    """(256, 3000) critic: the value head's K > 2048 form inside a training step."""
    _fp32_step_vs_fp64(0, (64, 64), (256, 3000))


@pytest.mark.parametrize("ptype", [0, 1, 2])
def test_learn_step_bf16_vs_oracle(ptype):
    """bf16 mode against the oracle's bf16 rounding model, at the tolerance of test_wide_discrete_gpu.py's bf16 step."""
    from rlgym_ppo_b200.ppo import ExperienceBuffer
    B = 512
    lr = _ppo(ptype, (300, 12), (4,), "bf16", B, seed=80 + ptype)
    pol0 = [p.detach().cpu().clone() for p in lr.policy.parameters()]
    val0 = [p.detach().cpu().clone() for p in lr.value_net.parameters()]
    fields = _problem(ptype, lr, B, np.random.RandomState(90 + ptype))
    buf = ExperienceBuffer(B, 123, DEV)
    buf.submit_experience(*fields)
    ob = O.BufferOracle(B, 123)
    ob.submit(**dict(zip(FIELD_NAMES, fields)))
    orc = O.PPOLearnerOracle(pol0, val0, B, 1, 3e-4, 3e-4, 0.2, 0.01, B, quant=O.quant_bf16, policy_type=ptype)
    want = orc.learn(ob)
    got = lr.learn(buf)
    for k in ("Policy Entropy", "Mean KL Divergence", "Value Function Loss", "SB3 Clip Fraction"):
        assert abs(got[k] - want[k]) <= 1e-3 * max(1.0, abs(want[k])), (k, got[k], want[k])
    for mine, ref in ((lr.policy.parameters(), orc.pol), (lr.value_net.parameters(), orc.val)):
        for i, p in enumerate(mine):
            assert close(p.detach().cpu().numpy(), ref[i].numpy(), 1e-3), i
            assert rel_l2(p.detach().cpu().numpy(), ref[i].numpy()) < 1e-3, i


# ---- 5. torch autograd ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("kind", ["discrete", "value"])
def test_autograd_300_100(kind, precision):
    from rlgym_ppo_b200.ppo import DiscreteFF, ValueEstimator
    from rlgym_ppo_b200.ppo._mlp import build_sequential
    obs_dim, layers, n, A = 20, (300, 100), 129, 9
    torch.manual_seed(3)
    rng = np.random.RandomState(4)
    m = DiscreteFF(obs_dim, A, layers, DEV, precision=precision) if kind == "discrete" else \
        ValueEstimator(obs_dim, layers, DEV, precision=precision)
    obs = torch.from_numpy(rng.randn(n, obs_dim).astype(np.float32))
    call = m.get_output if kind == "discrete" else m.forward
    with torch.no_grad():
        plain = call(obs.to(DEV)).clone()
    m.autograd = True
    out = call(obs.to(DEV))
    assert torch.equal(out.detach(), plain)
    grad = torch.from_numpy(rng.randn(*out.shape).astype(np.float32))
    for p in m.parameters():
        p.grad = None if p.grad is None else p.grad.zero_()
    torch.autograd.backward(out, grad.to(DEV))
    got = [p.grad.detach().cpu().numpy().copy() for p in m.parameters()]
    head = (lambda z: torch.softmax(z, -1)) if kind == "discrete" else (lambda z: z)
    sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    n_out = A if kind == "discrete" else 1
    if precision == "fp32":
        seq = build_sequential(obs_dim, layers, n_out, softmax=False).double()
        seq.load_state_dict({k[len("model."):]: v.double() for k, v in sd.items()})
        torch.autograd.backward(head(seq(obs.double())), grad.double())
        want = [p.grad.numpy() for p in seq.parameters()]
    else:
        params = [v.float() for v in sd.values()]
        z, layer_in = O.mlp_forward(params, obs.float(), O.quant_bf16)
        zl = z.detach().requires_grad_(True)
        (dz,) = torch.autograd.grad(head(zl), [zl], grad)
        if kind == "discrete":
            want = [g.numpy() for g in O.mlp_backward(params, layer_in, dz, O.quant_bf16)]
        else:
            # as test_autograd_gpu.py::reference_grads: the value head is an f32 SIMT pass (dv and w not rounded)
            h = layer_in[-1]
            dh = (dz @ params[-2]) * (h > 0).to(dz.dtype)
            hidden = O.mlp_backward(params[:-2], layer_in[:-1], dh, O.quant_bf16)
            want = [g.numpy() for g in hidden + [dz.t() @ h, dz.sum(0)]]
    errs = [rel_l2(a, b) for a, b in zip(got, want)]
    print(f"{kind} {precision}: grad rel-L2 per tensor", [float(f"{e:.2e}") for e in errs])
    assert max(errs) <= (1e-3 if precision == "fp32" else 2e-3), errs


# ---- 6. Learner end to end -------------------------------------------------------------------------------------------
class _Discrete:
    def __init__(self, n):
        self.n = n

    def seed(self, s):
        pass


class _Box:
    def __init__(self, shape):
        self.shape = shape


class ScriptedEnv:
    """Two agents, 16-dim observations, Discrete(6), episodes of 23 steps; reward for action == argmax(obs) % 6."""
    N_AGENTS, OBS, ACT, LEN = 2, 16, 6, 23

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
        rew = (a == self.obs.argmax(-1) % self.ACT).astype(np.float32)
        self.t += 1
        self.obs = self.rng.randn(self.N_AGENTS, self.OBS).astype(np.float32)
        return self.obs, list(rew), self.t >= self.LEN, {"state": None}

    def close(self):
        pass


def make_scripted_env():
    return ScriptedEnv()


def test_learner_any_width(tmp_path):
    from rlgym_ppo_b200 import Learner
    from rlgym_ppo_b200.ppo import PPOLearner
    folder = str(tmp_path / "ckpt")
    pl, cl = (500, 500), (300, 3000)
    kw = dict(n_proc=2, min_inference_size=2, ts_per_iteration=600, exp_buffer_size=10000, ppo_batch_size=600,
              ppo_epochs=1, policy_layer_sizes=pl, critic_layer_sizes=cl, standardize_obs=False,
              standardize_returns=True, checkpoints_save_folder=folder, add_unix_timestamp=False,
              save_every_ts=10 ** 9, log_to_wandb=False, ppo_ent_coef=0.01)
    learner = Learner(make_scripted_env, timestep_limit=1200, **kw)
    ppo = learner.ppo_learner
    before = [p.detach().clone() for p in list(ppo.policy.parameters()) + list(ppo.value_net.parameters())]
    calls = []
    orig = ppo.learn

    def learn(buf):
        calls.append(1)
        return orig(buf)

    ppo.learn = learn
    with contextlib.redirect_stdout(io.StringIO()):
        learner.learn()
    assert len(calls) == 2
    after = list(ppo.policy.parameters()) + list(ppo.value_net.parameters())
    for p0, p in zip(before, after):
        assert torch.isfinite(p).all()
        assert not torch.equal(p0, p.detach())
    with contextlib.redirect_stdout(io.StringIO()):
        learner.save(learner.agent.cumulative_timesteps)
    target = os.path.join(folder, str(learner.agent.cumulative_timesteps))
    saved_pol = torch.load(os.path.join(target, "PPO_POLICY.pt"), map_location="cpu")
    saved_val = torch.load(os.path.join(target, "PPO_VALUE_NET.pt"), map_location="cpu")
    assert tuple(saved_pol["model.0.weight"].shape) == (500, ScriptedEnv.OBS)
    assert tuple(saved_pol["model.2.weight"].shape) == (500, 500)
    assert tuple(saved_pol["model.4.weight"].shape) == (ScriptedEnv.ACT, 500)
    assert tuple(saved_val["model.2.weight"].shape) == (3000, 300)
    assert tuple(saved_val["model.4.weight"].shape) == (1, 3000)
    with contextlib.redirect_stdout(io.StringIO()):
        lr2 = PPOLearner(ScriptedEnv.OBS, ScriptedEnv.ACT, 0, pl, cl, (0.1, 1.0), 600, 1, 3e-4, 3e-4, 0.2, 0.01, 600, DEV)
        lr2.load_from(target)
    for net, net2 in ((ppo.policy, lr2.policy), (ppo.value_net, lr2.value_net)):
        for k, v in net.state_dict().items():
            assert torch.equal(v.cpu(), net2.state_dict()[k].cpu()), k
    x = torch.from_numpy(np.random.RandomState(9).randn(77, ScriptedEnv.OBS).astype(np.float32)).to(DEV)
    with torch.no_grad():
        assert torch.equal(ppo.policy.get_output(x), lr2.policy.get_output(x))
        assert torch.equal(ppo.value_net(x), lr2.value_net(x))
