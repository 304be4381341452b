"""GPU parity of the MultiDiscrete (21-logit Rolv) and Continuous (tanh-Gaussian) heads -- SURVEY.md 8(f)-4 -- against
the fixtures the unmodified reference produced (tests/golden/make_golden_heads.py -> heads.npz: get_backprop_data on a
minibatch, one PPOLearner.learn with the post-clip gradients of every optimiser step, updated weights, report) and
against the oracle's restated heads on injected random numbers.  multi_discrete_policy.py:16-89,
continuous_policy.py:23-120, torch_functions.py:15-33, 81-122, ppo_learner.py:34-50."""
import numpy as np
import pytest
import torch

from oracle import ref_oracle as O
from parity_helpers import (SENTINEL, bits, capture_steps, close, philox_rows, philox_uniform, recon, rel_l2, sentinel,
                            split_rows, unflatten)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
NAMES = ("states", "actions", "log_probs", "rewards", "next_states", "dones", "truncated", "values", "advantages")


def _learner(g, tag, ptype, precision):
    import contextlib
    import io
    from rlgym_ppo_b200.ppo import PPOLearner
    obs_dim, B, mb, epochs, total, n_cont, l0, l1 = [int(x) for x in g["cfg"]]
    plr, clr, clip, ent, vmin, vmax = [float(x) for x in g["hyper"]]
    with contextlib.redirect_stdout(io.StringIO()):
        lr = PPOLearner(obs_dim, n_cont, ptype, (l0, l1), (l0, l1), (vmin, vmax), B, epochs, plr, clr, clip, ent, mb, DEV,
                        precision=precision)
    for net, pre in ((lr.policy, f"{tag}.pol0"), (lr.value_net, f"{tag}.val0")):
        keys = list(net.state_dict().keys())
        net.load_state_dict({k: torch.from_numpy(g[f"{pre}.{i}"]) for i, k in enumerate(keys)})
    return lr, mb


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("tag,ptype", [("md", 1), ("ct", 2)])
def test_head_learn_matches_reference(golden, tag, ptype, precision):
    from rlgym_ppo_b200.ppo import ContinuousPolicy, ExperienceBuffer, MultiDiscreteFF
    g = golden("heads")
    lr, mb = _learner(g, tag, ptype, precision)
    assert isinstance(lr.policy, MultiDiscreteFF if ptype == 1 else ContinuousPolicy)
    exact = precision == "fp32"
    # state-dict layout = the reference's (continuous: the Sequential ends in Tanh, no extra keys)
    assert [tuple(v.shape) for v in lr.policy.state_dict().values()][-1] == ((21,) if ptype == 1 else (16,))
    # get_backprop_data on the first minibatch of the rollout
    obs = torch.from_numpy(g[f"{tag}.buf.states"][:mb])
    acts = torch.from_numpy(g[f"{tag}.buf.actions"][:mb])
    logp, ent = lr.policy.get_backprop_data(obs, acts)
    tol = 1e-4 if exact else 1e-2
    assert close(logp.cpu().numpy().reshape(-1), g[f"{tag}.bp_logp"].reshape(-1), tol)
    assert abs(float(ent) - float(g[f"{tag}.bp_entropy"][0])) < tol
    # PPOLearner.learn
    buf = ExperienceBuffer(1000, 123, DEV)
    buf.submit_experience(*[g[f"{tag}.buf.{n}"] for n in NAMES])
    assert np.array_equal(buf.actions.cpu().numpy(), g[f"{tag}.buf.actions"])           # action ROWS, byte-exact
    captured = capture_steps(lr)
    report = lr.learn(buf)
    n_steps = int(g[f"{tag}.n_steps"][0])
    assert len(captured) == n_steps
    ref_rep = dict(zip([str(k) for k in g[f"{tag}.report.keys"]], g[f"{tag}.report.vals"]))
    mtol = 1e-3 if exact else 3e-3
    for k in ("Policy Entropy", "Mean KL Divergence", "Value Function Loss", "SB3 Clip Fraction"):
        assert abs(report[k] - ref_rep[k]) <= mtol * max(1.0, abs(ref_rep[k])), (k, report[k], ref_rep[k])
    n_pol = len(list(lr.policy.parameters()))
    errs = []
    for s, flat in enumerate(captured):
        tensors = unflatten(lr, flat)
        wants = [g[f"{tag}.pgrad{s}.{i}"] if i < n_pol else g[f"{tag}.vgrad{s}.{i - n_pol}"] for i in range(len(tensors))]
        # a 1-element tensor (the value head's bias gradient, a sum that nearly cancels) has no meaningful relative error
        # of its own: it is measured against the norm of its network's whole gradient
        net_norm = [np.sqrt(sum(float((w.astype(np.float64) ** 2).sum()) for w in wants[:n_pol])),
                    np.sqrt(sum(float((w.astype(np.float64) ** 2).sum()) for w in wants[n_pol:]))]
        for i, (got, want) in enumerate(zip(tensors, wants)):
            if want.size == 1:
                errs.append((s, i, float(np.abs(got - want).max()) / net_norm[0 if i < n_pol else 1]))
            else:
                errs.append((s, i, rel_l2(got, want)))
    worst = max(e for _, _, e in errs)
    print(tag, precision, "max grad rel-L2 vs reference:", worst, [(s, i, float(f"{e:.1e}")) for s, i, e in errs if e > 1e-4])
    # Step 0 starts from the reference's weights: pure kernel error, held to the north-star 1e-3 in fp32 mode (measured
    # ~7e-6).  Later steps start from OUR step-0 weights: Adam normalises every gradient element to a +-lr move, so an
    # element whose gradient is ~0 (the value head's scalar bias gradient is a sum that nearly cancels) can move by +lr here
    # and -lr in the reference; that one weight shifts every value prediction and the NEXT gradient by a few per cent
    # (measured on B200: one element off by lr after step 0 -> 2-3.5e-2 on the md value net at step 1; the same happens
    # between two fp32 evaluations of the reference with different summation orders).
    assert max(e for s, _, e in errs if s == 0) < (1e-3 if exact else 0.25), errs
    assert worst < (6e-2 if exact else 0.25), errs
    for name, net in (("pol1", lr.policy), ("val1", lr.value_net)):
        for i, p in enumerate(net.parameters()):
            got, want = p.detach().cpu().numpy(), g[f"{tag}.{name}.{i}"]
            if exact:
                assert close(got, want, 1e-3), (name, i, np.abs(got - want).max())
                assert rel_l2(got, want) < 1e-3, (name, i)
            else:
                # bf16 operands: an element whose tiny gradient changes sign moves by up to 2 * lr per Adam step
                plr = float(g["hyper"][0])
                assert np.abs(got - want).max() <= 2 * plr * n_steps + 1e-6, (name, i, np.abs(got - want).max())


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_multi_discrete_sampling(golden, precision):
    """Inverse-CDF draws per distribution on injected uniforms equal the oracle's; log-probs are consistent with
    get_backprop_data; the deterministic branch returns the reference's [8, n] argmax layout."""
    from rlgym_ppo_b200 import ops
    g = golden("heads")
    lr, _ = _learner(g, "md", 1, precision)
    pol = lr.policy
    rng = np.random.RandomState(3)
    obs = g["md.buf.states"][:300]
    z = pol.get_output(obs).cpu()
    assert z.shape == (300, 21)
    zref, _ = O.mlp_forward([torch.from_numpy(g[f"md.pol0.{i}"]) for i in range(6)], torch.from_numpy(obs))
    assert close(z.numpy(), zref.numpy(), 1e-4 if precision == "fp32" else 2e-2)
    u = torch.from_numpy(rng.rand(300, 8).astype(np.float32)).to(DEV)
    zview, n, ws, _ = pol._logits(obs)
    acts = torch.empty((300, 8), device=DEV)
    logp = torch.empty(300, device=DEV)
    ops.head_multi_discrete_sample(zview[0], zview[1], zview[2], 300, acts, logp, u=u)
    # oracle draw from the DEVICE logits (so ties in the CDF do not depend on GEMM rounding)
    zd = z.double()
    start, want_a, want_lp = 0, [], torch.zeros(300, dtype=torch.float64)
    for gi, nb in enumerate(O.ROLV_BINS):
        lsm = zd[:, start:start + nb] - torch.logsumexp(zd[:, start:start + nb], -1, keepdim=True)
        c = torch.cumsum(lsm.exp().float(), -1)          # the kernel accumulates the CDF in f32
        a = (c > u[:, gi:gi + 1].cpu()).float().argmax(-1)
        a = torch.where((c > u[:, gi:gi + 1].cpu()).any(-1), a, torch.full_like(a, nb - 1))
        want_a.append(a)
        want_lp += lsm.gather(-1, a.view(-1, 1)).flatten()
        start += nb
    want_a = torch.stack(want_a, -1).float()
    mism = (acts.cpu() != want_a).float().mean()
    assert mism < 0.01, float(mism)         # CDF ties within one f32 ulp may land on the neighbouring bin
    same = (acts.cpu() == want_a).all(-1)
    assert close(logp.cpu().numpy()[same.numpy()], want_lp.numpy()[same.numpy()], 1e-4)
    lp2, _ = pol.get_backprop_data(obs, acts)
    assert close(lp2.cpu().numpy(), logp.cpu().numpy(), 1e-5)
    a_cpu, lp_cpu = pol.get_action(obs)
    assert a_cpu.shape == (300, 8) and a_cpu.dtype == torch.int64 and not a_cpu.is_cuda and lp_cpu.shape == (300,)
    assert int(a_cpu[:, :5].max()) <= 2 and int(a_cpu[:, 5:].max()) <= 1 and int(a_cpu.min()) >= 0
    det, zero = pol.get_action(obs, deterministic=True)
    assert det.shape == (8, 300) and zero == 0
    assert np.array_equal(det[0], z[:, 0:3].argmax(-1).numpy()) and np.array_equal(det[7], z[:, 19:21].argmax(-1).numpy())


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_continuous_sampling(golden, precision):
    from rlgym_ppo_b200 import ops
    g = golden("heads")
    lr, _ = _learner(g, "ct", 2, precision)
    pol = lr.policy
    obs = g["ct.buf.states"][:257]
    mean, std = pol.get_output(obs)
    assert mean.shape == (257, 8) and std.shape == (257, 8)
    assert float(std.min()) >= 0.1 - 1e-6 and float(std.max()) <= 1.0 + 1e-6 and float(mean.abs().max()) <= 1.0
    uref, _ = O.mlp_forward([torch.from_numpy(g[f"ct.pol0.{i}"]) for i in range(6)], torch.from_numpy(obs))
    assert close(mean.cpu().numpy(), torch.tanh(uref)[:, :8].numpy(), 1e-4 if precision == "fp32" else 2e-2)
    nrm = torch.randn(257, 8, generator=torch.Generator().manual_seed(1)).to(DEV)
    zview, n, ws, _ = pol._logits(obs)
    acts = torch.empty((257, 8), device=DEV)
    logp = torch.empty(257, device=DEV)
    ops.head_continuous_sample(zview[0], zview[1], zview[2], 257, 8, 0.1, 1.0, acts, logp, normals=nrm)
    want = (mean + std * nrm).clamp(-1, 1)
    assert close(acts.cpu().numpy(), want.cpu().numpy(), 1e-5)
    lp2, ent = pol.get_backprop_data(obs, acts)
    assert close(lp2.cpu().numpy(), logp.cpu().numpy(), 1e-4)
    want_ent = (0.5 + 0.5 * np.log(2 * np.pi) + torch.log(std)).mean()
    assert abs(float(ent) - float(want_ent)) < 1e-4
    a_cpu, lp_cpu = pol.get_action(obs)
    assert a_cpu.shape == (257, 8) and not a_cpu.is_cuda and float(a_cpu.abs().max()) <= 1.0
    # the Philox Box-Muller normals are standard normal: moments of (a - mean) / std over unclamped samples
    zs = ((a_cpu.to(DEV) - mean) / std)[(a_cpu.to(DEV).abs() < 1.0)]
    assert abs(float(zs.mean())) < 0.1
    det, zero = pol.get_action(obs, deterministic=True)
    assert zero == 0 and close(det.cpu().numpy(), mean.cpu().numpy(), 1e-6)


# =====================================================================================================================
# kernel level: rlppo_head_{multi_discrete,continuous}_{train,sample} called directly, against fp64 references.
# The logits are f32 masters staged with ops.rows_split; the references take the fp64 sum of the staged parts (exactly
# the f32 value the kernel's zload forms, for 1, 2 or 3 parts).  u = 2^-24.  Every bound below is a first-order
# propagation of the kernel's own roundings (no fast-math in this build: expf, tanhf, sinf, cosf within 2 ulp = 4u
# relative, logf within 1 ulp, sqrtf and divisions IEEE), doubled to cover the second-order terms and the compiler's
# choice of fused multiply-adds.
# =====================================================================================================================
U = 2.0 ** -24
RATIOS = (0.5, 0.79, 0.95, 1.0, 1.05, 1.21, 2.0)
MIXES = [(0.2, 0.01), (0.2, 0.0), (0.1, 0.05)]
ROWS = [1, 31, 129, 50001]
METRICS0 = [1.5, -0.25, 3.0, 0.75, 7.0, 11.0, 13.0, 17.0]      # the kernels accumulate into metrics
SEED = 0x0123456789ABCDEF                                        # both 32-bit halves non-zero
ZPS = 64                                                         # part stride of the staged logits


@pytest.fixture(scope="module")
def ops():
    from rlgym_ppo_b200 import _lib, ops as _ops
    _lib.require_device()
    return _ops


def f32(x):
    return float(np.float32(x))


def _stage(ops, z32, parts):
    """f32 logits [M, out] -> (split bf16 device buffer, fp64 value the kernel sees)."""
    buf = split_rows(ops, z32, parts, ZPS)
    return buf, recon(buf, parts, ZPS, z32.shape[1])


def _ppo_inputs(logp64, M, seed):
    """old_logp and adv built so that every clip regime appears: row i has ratio RATIOS[i % 7] (exact in fp64 up to the
    f32 rounding of old_logp), the sign of adv alternates every 7 rows and every 5th row has adv = 0.  With clip 0.2 or
    0.1 no target ratio lies within 0.01 of 1 +- clip, far beyond the kernels' log-prob error."""
    g = torch.Generator().manual_seed(seed)
    i = torch.arange(M)
    r = torch.tensor(RATIOS, dtype=torch.float64)[i % 7]
    sign = 1.0 - 2.0 * ((i // 7) % 2).double()
    adv = (0.1 + torch.rand(M, generator=g, dtype=torch.float64)) * sign
    adv[i % 5 == 4] = 0.0
    return (logp64 - torch.log(r)).float(), adv.float()


def _ppo64(logp, ent_sum, old, adv, inv_b, clip, ent_coef):
    """ppo_learner.py:153-177 in fp64: torch.min splits ties 0.5 / 0.5 and the clamp passes the gradient inside the range
    inclusively (autograd's rules, the kernels' ppo_row)."""
    log_ratio = logp - old.double()
    ratio = torch.exp(log_ratio)
    a = adv.double()
    s1, s2 = ratio * a, torch.clamp(ratio, 1 - clip, 1 + clip) * a
    surr = torch.min(s1, s2)
    loss = (-surr.sum() - ent_coef * ent_sum) * inv_b
    with torch.no_grad():
        in_range = ((ratio >= 1 - clip) & (ratio <= 1 + clip)).double()
        d1 = (s1 < s2).double() + 0.5 * (s1 == s2).double()
        d2 = (s1 > s2).double() + 0.5 * (s1 == s2).double()
        d_logp = -inv_b * a * (d1 + d2 * in_range) * ratio
        kl = (ratio - 1) - log_ratio
        clipc = ((ratio - 1).abs() > clip).double()
    return loss, dict(ratio=ratio.detach(), log_ratio=log_ratio.detach(), d_logp=d_logp, kl=kl.detach(), clipc=clipc,
                      surr=surr.detach())


def _metrics_check(m, M, ent_rows, d_ent_rows, p, eps_r, d_logp_err):
    """metrics [0] entropy, [1] KL, [3] surrogate against the fp64 sums, [2] clip count and [4] rows exact.  Each kernel
    row term t_i carries its own error e_i (propagated below); the sums are a 5-level warp tree and one atomicAdd per
    warp onto the pre-filled value, so |sum - fp64| <= sum e_i + (W + 6) u (sum |t_i| + |pre|), W = ceil(M / 32)."""
    W = (M + 31) // 32
    pre = torch.tensor(METRICS0[:5], dtype=torch.float64)
    ratio, lr = p["ratio"], p["log_ratio"]
    kl_err = ratio.abs() * eps_r + d_logp_err + 2 * U * (ratio - 1).abs() + U * (lr.abs() + p["kl"].abs())
    surr_err = p["surr"].abs() * (eps_r + 2 * U)
    worst = 0.0
    for k, t, e in ((0, ent_rows, d_ent_rows), (1, p["kl"], kl_err), (3, p["surr"], surr_err)):
        want = float(pre[k] + t.sum())
        bound = 2 * float(e.sum()) + (W + 6) * U * (float(t.abs().sum()) + abs(float(pre[k])))
        err = abs(float(m[k]) - want)
        worst = max(worst, err / bound)
        assert err <= bound, (k, float(m[k]), want, bound)
    assert float(m[2]) == float(pre[2] + p["clipc"].sum())
    assert float(m[4]) == float(pre[4]) + M
    assert [float(x) for x in m[5:8]] == METRICS0[5:8]
    return worst


def _check_dz_layout(dz, M, parts, ps, cols, out):
    """Columns [out, dz_cols) of every part are +0, everything outside the parts' [0, dz_cols) and every row >= M keeps
    the sentinel."""
    b = bits(dz.cpu())
    written = torch.zeros(b.shape[1], dtype=torch.bool)
    for q in range(parts):
        assert bool((b[:M, q * ps + out:q * ps + cols] == 0).all()), "padding columns of d(logits) not zero"
        written[q * ps:q * ps + cols] = True
    assert bool((b[:M][:, ~written] == SENTINEL).all()), "written outside the d(logits) view"
    assert bool((b[M:] == SENTINEL).all()), "written below row M"


# ---- MultiDiscrete ---------------------------------------------------------------------------------------------------
MD_STARTS = (0, 3, 6, 9, 12, 15, 17, 19)
# (z_parts, dz_parts, dz_cols, dz part stride, dz ld, ld_act): bf16 mode (1 part, pstride 0, pad8(21) = 24 columns),
# fp32 mode (2 parts) with a gap between dz_cols and the part stride, a dz_cols wider than pad8, strided actions
MD_VIEWS = [(1, 1, 24, 0, 24, 8), (2, 2, 24, 32, 64, 11), (3, 2, 40, 48, 96, 8), (3, 1, 32, 0, 40, 11)]


def _md64(z):
    """Per-column fp64 quantities of the eight categoricals: lsm, p, the group's H, and the kernel's log-softmax error
    dl = u (R + |lse| + |lsm| + 11) (R = max - min of the group's logits): z_j - max rounds by u R, the <= 3 expf (4u
    each) and their sum give se to u R + 6u relative, logf adds 1 ulp of log se <= log 3 (u 9 in all), mx + log se and
    z_j - lse round once each."""
    M = z.shape[0]
    lsm, dl, Hc = torch.empty_like(z), torch.empty_like(z), torch.empty_like(z)
    H = torch.empty(M, 8, dtype=torch.float64)
    for g, (s, nb) in enumerate(zip(MD_STARTS, O.ROLV_BINS)):
        zg = z[:, s:s + nb]
        lse = torch.logsumexp(zg, -1, keepdim=True)
        lsm[:, s:s + nb] = zg - lse
        R = zg.max(-1, keepdim=True).values - zg.min(-1, keepdim=True).values
        dl[:, s:s + nb] = U * (R + lse.abs() + lsm[:, s:s + nb].abs() + 11)
        H[:, g] = -(lsm[:, s:s + nb] * lsm[:, s:s + nb].exp()).sum(-1)
        Hc[:, s:s + nb] = H[:, g:g + 1]
    return lsm, lsm.exp(), H, Hc, dl


def _md_logp_err(lsm, dl, acts):
    """logp = sum of 8 lsm[a_g]: their errors plus 8 u sum |lsm[a_g]| for the f32 sum."""
    idx = torch.tensor(MD_STARTS) + acts.long()
    la = lsm.gather(-1, idx)
    return dl.gather(-1, idx).sum(-1) + 8 * U * la.abs().sum(-1), la.sum(-1)


MD_TRAIN = [(M, v, mx, sat) for M in ROWS for v in range(len(MD_VIEWS)) for mx in range(len(MIXES)) for sat in (0, 1)]


@pytest.mark.parametrize("M,view,mix,saturated", MD_TRAIN,
                         ids=[f"M{M}-v{v}-mix{mx}-{'sat' if s else 'normal'}" for M, v, mx, s in MD_TRAIN])
def test_head_multi_discrete_train_kernel(ops, M, view, mix, saturated):
    """rlppo_head_multi_discrete_train against fp64 autograd through O.head_multi_discrete and the PPO block.

    dz per element, d = d(loss)/d(logp), ce = ent_coef inv_batch, dz_j = d (onehot_j - p_j) + ce p_j (lsm_j + H_g):
      lsm_j to dl_j (_md64); p_j = expf(lsm_j) to ep_j = dl_j + 4u relative; H_g = -sum lsm p to
      dH = sum_k p_k (dl_k + |lsm_k| ep_k) + 3u sum_k p_k |lsm_k|;
      logp = sum_g lsm[a_g] to dlp (_md_logp_err); ratio = expf(logp - old) to er = dlp + u |log ratio| + 4u relative,
      d to ed = er + 3u (three products);
      |err_j| <= |d| (ed |onehot - p| + p ep + 2u |onehot - p|) + |ce| p ((ep + 3u) |lsm + H| + dl + dH + u |lsm + H|)
                 + u |dz| + 2^-126 (|d| + |ce| (|lsm| + |H| + 1))     [expf underflow below 2^-126]
      plus the output rounding 2^-8 (one bf16 part) or 2^-16 (two) of |dz| and 2^-134 (bf16 subnormal spacing);
    the whole doubled.  Every term is absolute (in |d|, |ce|, p), so a row whose dz cancels is still held to the size of
    its terms, and an adv = 0 row (d = 0) to its entropy term alone.
    logp_out within 2 dlp; metrics by _metrics_check with the entropy row error sum_g dH_g + 8u sum_g |H_g|.
    A launch with logp_out and metrics NULL writes bit-identical dz.
    Measured on a B200: dz error / bound at most 0.57 up to M = 129.  At M = 50001 with saturated logits it reaches
    0.97-0.998: inv_batch = 1e-5 puts some dz entries at bf16's subnormal floor, where the bound's 2^-134 term is the
    whole allowance (the largest, 4.592e-41 = 2^-134 (1 + 5e-6), is stored as 2^-133).  Rounding to nearest cannot
    exceed that floor, so these are the output format's limit, not slack taken by the kernel.  logp_out at most 0.16 of
    its bound, metrics at most 0.054."""
    zp, dzp, cols, dps, dld, ld_act = MD_VIEWS[view]
    clip, ent_coef = (f32(x) for x in MIXES[mix])
    inv_b = f32(1.0 / (2 * M))
    g = torch.Generator().manual_seed(1000 * view + 10 * mix + saturated + M)
    z32 = torch.randn(M, 21, generator=g) * (30.0 if saturated else 1.5)
    zbuf, z = _stage(ops, z32, zp)
    acts = torch.stack([torch.randint(0, nb, (M,), generator=g) for nb in O.ROLV_BINS], -1).float()
    lsm, p, H, Hc, dl = _md64(z)
    dlp, lp64 = _md_logp_err(lsm, dl, acts)
    old, adv = _ppo_inputs(lp64, M, 7 + M)
    a_buf = torch.full((M, ld_act), 99.0)
    a_buf[:, :8] = acts
    a_dev, old_dev, adv_dev = a_buf.to(DEV), old.to(DEV), adv.to(DEV)
    dz = sentinel(M + 2, dld)
    logp = torch.full((M,), float("nan"), device=DEV)
    metrics = torch.tensor(METRICS0, device=DEV)
    ops.head_multi_discrete_train(zbuf, zp, ZPS, M, a_dev, old_dev, adv_dev, inv_b, clip, ent_coef, dz, dzp, dps, cols,
                                  metrics, logp_out=logp)
    dz2 = sentinel(M + 2, dld)
    ops.head_multi_discrete_train(zbuf, zp, ZPS, M, a_dev, old_dev, adv_dev, inv_b, clip, ent_coef, dz2, dzp, dps, cols,
                                  None, logp_out=None)
    torch.cuda.synchronize()
    assert torch.equal(bits(dz), bits(dz2))
    _check_dz_layout(dz, M, dzp, dps, cols, 21)
    # fp64 reference
    zt = z.clone().requires_grad_(True)
    lp_t, ent_mean, _ = O.head_multi_discrete(zt, acts)
    loss, pp = _ppo64(lp_t, ent_mean * M, old, adv, inv_b, clip, ent_coef)
    (ref,) = torch.autograd.grad(loss, [zt])
    got = recon(dz, dzp, dps, 21, rows=slice(0, M))
    # bound
    d = pp["d_logp"][:, None]
    ce = ent_coef * inv_b
    onehot = torch.zeros(M, 21, dtype=torch.float64).scatter_(-1, torch.tensor(MD_STARTS) + acts.long(), 1.0)
    ep = dl + 4 * U
    dHg = torch.stack([(p[:, s:s + nb] * (dl[:, s:s + nb] + lsm[:, s:s + nb].abs() * ep[:, s:s + nb])).sum(-1)
                       + 3 * U * (p[:, s:s + nb] * lsm[:, s:s + nb].abs()).sum(-1)
                       for s, nb in zip(MD_STARTS, O.ROLV_BINS)], -1)
    dH = dHg[:, torch.tensor([gi for gi, nb in enumerate(O.ROLV_BINS) for _ in range(nb)])]
    eps_r = dlp + U * pp["log_ratio"].abs() + 4 * U
    ed = (eps_r + 3 * U)[:, None]
    om, lh = (onehot - p).abs(), (lsm + Hc).abs()
    err = (d.abs() * (ed * om + p * ep + 2 * U * om) + abs(ce) * p * ((ep + 3 * U) * lh + dl + dH + U * lh)
           + U * ref.abs() + 2.0 ** -126 * (d.abs() + abs(ce) * (lsm.abs() + Hc.abs() + 1)))
    bound = 2 * (err + (2.0 ** -8 if dzp == 1 else 2.0 ** -16) * (ref.abs() + err)) + 2.0 ** -134
    ratio_dz = float(((got - ref).abs() / bound).max())
    lp_ratio = float(((logp.cpu().double() - lp64).abs() / (2 * dlp)).max())
    ent_err = dHg.sum(-1) + 8 * U * H.abs().sum(-1)
    m_ratio = _metrics_check(metrics.cpu().double(), M, H.sum(-1), ent_err, pp, eps_r, dlp)
    print(f"md train M={M} view={view} mix={mix} sat={saturated}: dz err/bound {ratio_dz:.3g}, logp {lp_ratio:.3g}, "
          f"metrics {m_ratio:.3g}")
    assert ratio_dz <= 1.0, ratio_dz
    assert lp_ratio <= 1.0, lp_ratio
    # every clip regime is present (M >= 31): in range, clipped without gradient, outside the range with gradient
    if M >= 31:
        out = pp["clipc"] > 0
        assert bool((out & (pp["d_logp"] == 0) & (adv != 0)).any()) and bool((out & (pp["d_logp"] != 0)).any())
        assert bool((~out & (adv != 0)).any())


def _rlppo_error():
    from rlgym_ppo_b200._lib import RlppoError
    return RlppoError


def test_head_train_argument_errors(ops):
    """Argument errors raise before any launch: n_act 0 and 33 (continuous, train and sample), dz_cols below the head's
    width, a MultiDiscrete ld_act below its 8 actions."""
    M = 4
    err = _rlppo_error()
    zbuf = split_rows(ops, torch.zeros(M, 64), 1, 64)
    old, adv, metrics = torch.zeros(M, device=DEV), torch.zeros(M, device=DEV), torch.zeros(8, device=DEV)
    dz = torch.zeros(M, 128, dtype=torch.bfloat16, device=DEV)
    for n in (0, 33):
        with pytest.raises(err):
            ops.head_continuous_train(zbuf, 1, 0, M, n, 0.1, 1.0, torch.zeros(M, 40, device=DEV), old, adv, 0.1, 0.2,
                                      0.01, dz, 1, 0, 128, metrics)
        with pytest.raises(err):
            ops.head_continuous_sample(zbuf, 1, 0, M, n, 0.1, 1.0, torch.zeros(M, 40, device=DEV), old)
    with pytest.raises(err):
        ops.head_continuous_train(zbuf, 1, 0, M, 3, 0.1, 1.0, torch.zeros(M, 3, device=DEV), old, adv, 0.1, 0.2, 0.01,
                                  dz, 1, 0, 5, metrics)
    acts = torch.zeros(M, 8, device=DEV)
    with pytest.raises(err):
        ops.head_multi_discrete_train(zbuf, 1, 0, M, acts, old, adv, 0.1, 0.2, 0.01, dz, 1, 0, 20, metrics)
    with pytest.raises(err):
        ops.head_multi_discrete_train(zbuf, 1, 0, M, torch.zeros(M, 7, device=DEV), old, adv, 0.1, 0.2, 0.01, dz, 1, 0,
                                      24, metrics)
    # the same calls with valid arguments go through
    ops.head_multi_discrete_train(zbuf, 1, 0, M, acts, old, adv, 0.1, 0.2, 0.01, dz, 1, 0, 24, metrics)
    ops.head_continuous_train(zbuf, 1, 0, M, 3, 0.1, 1.0, torch.zeros(M, 3, device=DEV), old, adv, 0.1, 0.2, 0.01,
                              dz, 1, 0, 6, metrics)
    torch.cuda.synchronize()


# ---- Continuous ------------------------------------------------------------------------------------------------------
# (z_parts, dz_parts, dz_cols extra over pad8(2n), dz part-stride gap, ld_act extra over n)
CT_VIEWS = [(1, 1, 0, 0, 0), (2, 2, 0, 8, 3), (3, 2, 16, 8, 0), (3, 1, 8, 0, 3)]
VAR_RANGES = [(0.1, 1.0), (0.5, 2.0)]
CT_TRAIN = [(M, n, mx, sat) for M in ROWS for n in (1, 3, 8, 32) for mx in range(len(MIXES)) for sat in (0, 1)]


class _Ct64:
    """fp64 quantities of the tanh-Gaussian head at actions x, with the kernel's error terms:
      mean = tanhf to 4u relative; sd = ts m + b to esd = u (6 (m |ts| + b) / sd + 1) relative (tanhf, the product,
      m and b formed in f32, the sum);
      the four log-pdf terms t1 = -mean^2 / 2sd^2, t2 = mean x / sd^2, t3 = -x^2 / 2sd^2 (relative errors <= 12u + 2 esd)
      and t4 = log(1 / sqrt(2 pi sd^2)) (absolute esd + 4u + 2u |t4|), summed as ((t1 + t2) + t3) + t4 (3u sum |t|)
      and over the n actions (n u sum |t|): dlp = sum_j ((2 esd + 15u) S_j + esd + 4u) + n u sum_j S_j, S_j = sum |t|;
      the row entropy, mean over j of 0.5 + 0.5 log 2 pi + log sd, to
      dent = (sum_j (esd + 4u + 2u |log sd|) + (n + 2) u sum_j |e_j|) / n + u |ent|."""

    def __init__(self, z, x, var_min, var_max):
        n = z.shape[1] // 2
        self.n, self.x = n, x
        self.m = (var_max - var_min) / 2.0
        self.b = var_min + self.m
        self.tm, self.ts = torch.tanh(z[:, :n]), torch.tanh(z[:, n:])
        self.sd = self.ts * self.m + self.b
        self.esd = U * (6 * (self.m * self.ts.abs() + self.b) / self.sd + 1)
        ssq = self.sd ** 2
        t = [-(self.tm ** 2) / (2 * ssq), self.tm * x / ssq, -(x ** 2) / (2 * ssq), torch.log(1 / torch.sqrt(2 * np.pi * ssq))]
        S = sum(a.abs() for a in t)
        self.logp = sum(t).sum(-1)
        self.dlp = ((2 * self.esd + 15 * U) * S + self.esd + 4 * U).sum(-1) + n * U * S.sum(-1)
        e = 0.5 + 0.5 * np.log(2 * np.pi) + torch.log(self.sd)
        self.ent = e.mean(-1)
        self.dent = ((self.esd + 4 * U + 2 * U * torch.log(self.sd).abs()).sum(-1) + (n + 2) * U * e.abs().sum(-1)) / n \
            + U * self.ent.abs()


@pytest.mark.parametrize("M,n,mix,saturated", CT_TRAIN,
                         ids=[f"M{M}-n{n}-mix{mx}-{'sat' if s else 'normal'}" for M, n, mx, s in CT_TRAIN])
def test_head_continuous_train_kernel(ops, M, n, mix, saturated):
    """rlppo_head_continuous_train against fp64 autograd through O.head_continuous and the PPO block.  The view and the
    (var_min, var_max) range cycle with the case index over CT_VIEWS and VAR_RANGES.

    dz per element, d = d(loss)/d(logp) with ed as in the MultiDiscrete test (dlp from _Ct64), ce = -ent_coef inv / n:
      diff = x - mean to Dd = 4u |mean| + u |diff| (absolute: x and mean may cancel);
      d_mean = d diff / sd^2 to |d_mean| (ed + 2 esd + 3u) + |d| Dd / sd^2;
      q = diff^2 / sd^3 - 1 / sd to Dq = 2 |diff| Dd / sd^3 + diff^2 / sd^3 (3 esd + 4u) + (esd + u) / sd
                                         + u (diff^2 / sd^3 + 1 / sd)   (absolute: the two terms cancel);
      d_std = d q + ce / sd to |d| Dq + |q d| ed + |ce| / sd (esd + 3u) + 2u (|d q| + |ce| / sd);
      dz_mean = d_mean (1 - tm^2): + |d_mean| (8u tm^2 + 2u) + u |dz| (1 - tm^2 cancels where tanh saturates);
      dz_std = d_std m (1 - ts^2): + |d_std| m (8u ts^2 + 3u) + 2u |dz|;
    plus the output rounding 2^-8 / 2^-16 and 2^-134, doubled.  logp_out within 2 dlp; metrics by _metrics_check with
    the row entropy error dent.  A launch with logp_out and metrics NULL writes bit-identical dz.
    Measured on a B200: dz error / bound at most 0.498 (one bf16 part: the rounding of an entry just above a power of
    two is 2^-8 relative, half the doubled allowance), logp_out at most 0.088, metrics at most 0.05."""
    case = CT_TRAIN.index((M, n, mix, saturated))
    zp, dzp, extra, gap, act_extra = CT_VIEWS[case % len(CT_VIEWS)]
    var_min, var_max = (f32(v) for v in VAR_RANGES[case % len(VAR_RANGES)])
    out = 2 * n
    cols = (out + 7) // 8 * 8 + extra
    dps = cols + gap if dzp == 2 else 0
    dld = (dzp - 1) * dps + cols + 8
    ld_act = n + act_extra
    clip, ent_coef = (f32(x) for x in MIXES[mix])
    inv_b = f32(1.0 / (2 * M))
    g = torch.Generator().manual_seed(3000 + 7 * n + 10 * mix + saturated + M)
    z32 = torch.randn(M, out, generator=g)
    if saturated:
        big = torch.rand(M, out, generator=g) < 0.5
        z32[big] = torch.sign(z32[big]) * (10.5 + 5 * torch.rand(int(big.sum()), generator=g))
    zbuf, z = _stage(ops, z32, zp)
    t = torch.tanh(z)
    sd0 = t[:, n:] * (var_max - var_min) / 2 + (var_max + var_min) / 2
    x = (t[:, :n] + sd0 * torch.randn(M, n, generator=g, dtype=torch.float64)).clamp(-1, 1).float()
    c = _Ct64(z, x.double(), var_min, var_max)
    old, adv = _ppo_inputs(c.logp, M, 11 + M)
    a_buf = torch.full((M, ld_act), 7.0)
    a_buf[:, :n] = x
    a_dev, old_dev, adv_dev = a_buf.to(DEV), old.to(DEV), adv.to(DEV)
    dz = sentinel(M + 2, dld)
    logp = torch.full((M,), float("nan"), device=DEV)
    metrics = torch.tensor(METRICS0, device=DEV)
    ops.head_continuous_train(zbuf, zp, ZPS, M, n, var_min, var_max, a_dev, old_dev, adv_dev, inv_b, clip, ent_coef, dz,
                              dzp, dps, cols, metrics, logp_out=logp)
    dz2 = sentinel(M + 2, dld)
    ops.head_continuous_train(zbuf, zp, ZPS, M, n, var_min, var_max, a_dev, old_dev, adv_dev, inv_b, clip, ent_coef, dz2,
                              dzp, dps, cols, None, logp_out=None)
    torch.cuda.synchronize()
    assert torch.equal(bits(dz), bits(dz2))
    _check_dz_layout(dz, M, dzp, dps, cols, out)
    zt = z.clone().requires_grad_(True)
    lp_t, ent_mean, _ = O.head_continuous(zt, x.double(), var_min, var_max)
    loss, pp = _ppo64(lp_t, ent_mean * M, old, adv, inv_b, clip, ent_coef)
    (ref,) = torch.autograd.grad(loss, [zt])
    got = recon(dz, dzp, dps, out, rows=slice(0, M))
    # bound
    d = pp["d_logp"][:, None]
    ce = abs(ent_coef * inv_b / n)
    eps_r = c.dlp + U * pp["log_ratio"].abs() + 4 * U
    ed = (eps_r + 3 * U)[:, None]
    sd, esd, tm, ts = c.sd, c.esd, c.tm, c.ts
    diff = x.double() - tm
    Dd = 4 * U * tm.abs() + U * diff.abs()
    d_mean = d * diff / sd ** 2
    e_mean = d_mean.abs() * (ed + 2 * esd + 3 * U) + d.abs() * Dd / sd ** 2
    q = diff ** 2 / sd ** 3 - 1 / sd
    Dq = (2 * diff.abs() * Dd / sd ** 3 + diff ** 2 / sd ** 3 * (3 * esd + 4 * U) + (esd + U) / sd
          + U * (diff ** 2 / sd ** 3 + 1 / sd))
    d_std = d * q - ce / sd
    e_std = d.abs() * Dq + (q * d).abs() * ed + ce / sd * (esd + 3 * U) + 2 * U * ((d * q).abs() + ce / sd)
    dzm, dzs = ref[:, :n], ref[:, n:]
    err = torch.cat([e_mean * (1 - tm ** 2) + d_mean.abs() * (8 * U * tm ** 2 + 2 * U) + U * dzm.abs(),
                     e_std * c.m * (1 - ts ** 2) + d_std.abs() * c.m * (8 * U * ts ** 2 + 3 * U) + 2 * U * dzs.abs()], -1)
    bound = 2 * (err + (2.0 ** -8 if dzp == 1 else 2.0 ** -16) * (ref.abs() + err)) + 2.0 ** -134
    ratio_dz = float(((got - ref).abs() / bound).max())
    lp_ratio = float(((logp.cpu().double() - c.logp).abs() / (2 * c.dlp)).max())
    m_ratio = _metrics_check(metrics.cpu().double(), M, c.ent, c.dent, pp, eps_r, c.dlp)
    print(f"ct train M={M} n={n} mix={mix} sat={saturated} view={case % len(CT_VIEWS)}: dz err/bound {ratio_dz:.3g}, "
          f"logp {lp_ratio:.3g}, metrics {m_ratio:.3g}")
    assert ratio_dz <= 1.0, ratio_dz
    assert lp_ratio <= 1.0, lp_ratio


# ---- sampling kernels ------------------------------------------------------------------------------------------------
def _md_rows(M, seed):
    """Random logits followed by the edge rows: E0 (u = 0, first bin 120 below the others: expf(lsm) underflows to 0 in
    f32, so that bin has probability 0), E1 (u = 1 - 2^-24), T (exact ties: all bins equal, or the last two equal and
    largest)."""
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(M, 21, generator=g) * 2
    u = torch.rand(M, 8, generator=g, dtype=torch.float64).float()
    e0 = torch.randn(16, 21, generator=g)
    for s, nb in zip(MD_STARTS, O.ROLV_BINS):
        e0[:, s + 1:s + nb] = e0[:, s + 1:s + 2]
        e0[:, s] = e0[:, s + 1] - 120.0
    e1 = torch.randn(16, 21, generator=g) * 2
    tie = torch.full((16, 21), 0.25)
    for s, nb in zip(MD_STARTS, O.ROLV_BINS):
        tie[8:, s + nb - 2:s + nb] = 0.75
    z = torch.cat([z, e0, e1, tie])
    u = torch.cat([u, torch.zeros(16, 8), torch.full((16, 8), 1.0 - 2.0 ** -24), torch.rand(16, 8, generator=g)])
    return z, u, (M, M + 16, M + 32)


def test_head_multi_discrete_sample_kernel(ops):
    """rlppo_head_multi_discrete_sample on injected uniforms u [M, 8], all eight groups against the fp64 inverse CDF (first
    j with cdf_j > u): a differing entry must have u within the f32 CDF's error of a bucket edge, sum_k p_k ep_k + 3u
    (ep from _md64).  Edge rows (_md_rows): a zero-probability first bin is never drawn at u = 0; u = 1 - 2^-24 stays in
    range; deterministic draws return the first of exactly tied logits in every group.  logp_out within 2 dlp of the
    fp64 sum of lsm[a]; the train kernel's logp_out on the returned actions is bit-identical (both run the same
    log-softmax sum; measured on a B200: identical on every row)."""
    z32, u, (e0, e1, tie) = _md_rows(3000, 5)
    M = z32.shape[0]
    zbuf, z = _stage(ops, z32, 3)
    lsm, p, _, _, dl = _md64(z)
    acts = torch.full((M, 11), float("nan"), device=DEV)          # ld_aout 11: columns 8..10 untouched
    logp = torch.empty(M, device=DEV)
    ops.head_multi_discrete_sample(zbuf, 3, ZPS, M, acts, logp, u=u.to(DEV))
    torch.cuda.synchronize()
    assert bool(acts[:, 8:].isnan().all())
    a = acts[:, :8].cpu()
    ep = dl + 4 * U
    near_rows = torch.zeros(M, dtype=torch.bool)
    for gi, (s, nb) in enumerate(zip(MD_STARTS, O.ROLV_BINS)):
        cdf = p[:, s:s + nb].cumsum(-1)
        hit = cdf > u[:, gi:gi + 1].double()
        want = torch.where(hit.any(-1), hit.double().argmax(-1), torch.full((M,), nb - 1))
        slack = (p[:, s:s + nb] * ep[:, s:s + nb]).sum(-1) + 3 * U
        ag = a[:, gi].long()
        assert bool(((ag >= 0) & (ag < nb)).all())
        bad = (ag != want).nonzero().flatten()
        for r in bad.tolist():
            j = min(int(ag[r]), int(want[r]))
            assert abs(float(cdf[r, j]) - float(u[r, gi])) <= float(slack[r]), (r, gi, int(ag[r]), int(want[r]))
        near_rows |= ((cdf - u[:, gi:gi + 1].double()).abs() <= slack[:, None]).any(-1)
        assert bad.numel() <= int(near_rows.sum())
    assert bool((a[e0:e1] == 1).all()), "a zero-probability bin was drawn at u = 0"
    assert float(np.exp(np.float32(-120.0))) == 0.0
    dlp, lp64 = _md_logp_err(lsm, dl, a)
    assert bool(((logp.cpu().double() - lp64).abs() <= 2 * dlp).all())
    # the train kernel's log-prob of the drawn actions
    lp_train = torch.empty(M, device=DEV)
    dz = torch.empty(M, 24, dtype=torch.bfloat16, device=DEV)
    ops.head_multi_discrete_train(zbuf, 3, ZPS, M, acts, torch.zeros(M, device=DEV), torch.zeros(M, device=DEV), 1.0 / M,
                                  0.2, 0.01, dz, 1, 0, 24, None, logp_out=lp_train)
    # deterministic: the first maximum of every group, exact ties included
    det = torch.empty(M, 8, device=DEV)
    lp_det = torch.empty(M, device=DEV)
    ops.head_multi_discrete_sample(zbuf, 3, ZPS, M, det, lp_det, deterministic=True)
    torch.cuda.synchronize()
    assert torch.equal(lp_train.view(torch.int32), logp.view(torch.int32))
    want_det = torch.stack([z[:, s:s + nb].argmax(-1) for s, nb in zip(MD_STARTS, O.ROLV_BINS)], -1)
    assert torch.equal(det.cpu().long(), want_det)
    assert bool((det.cpu()[tie:tie + 8] == 0).all()) and bool((det.cpu()[tie + 8:] == torch.tensor(O.ROLV_BINS) - 2).all())
    dlp, lp64 = _md_logp_err(lsm, dl, det.cpu())
    assert bool(((lp_det.cpu().double() - lp64).abs() <= 2 * dlp).all())


def test_head_multi_discrete_philox_stream(ops):
    """rlppo_head_multi_discrete_sample from (seed, offset) draws exactly what the host restatement's uniforms draw when
    injected: groups 0-3 take the words (x, y, z, w) of the counter (offset + row, high word, 0, 0), groups 4-7 those of
    (offset + row, high word, 1, 0).  The offset 2^32 - M/2 makes the launch cross the carry into the high word."""
    M = 4001
    g = torch.Generator().manual_seed(21)
    zbuf, _ = _stage(ops, torch.randn(M, 21, generator=g) * 2, 3)
    off = 2 ** 32 - M // 2
    uh = np.concatenate([philox_uniform(philox_rows(SEED, off, M, word2=w)) for w in (0, 1)], -1)
    draws = []
    for kw in (dict(seed=SEED, offset=off), dict(u=torch.from_numpy(uh).float().to(DEV))):
        a_, l_ = torch.empty(M, 8, device=DEV), torch.empty(M, device=DEV)
        ops.head_multi_discrete_sample(zbuf, 3, ZPS, M, a_, l_, **kw)
        draws.append((a_, l_))
    torch.cuda.synchronize()
    assert torch.equal(draws[0][0], draws[1][0])
    assert torch.equal(draws[0][1].view(torch.int32), draws[1][1].view(torch.int32))
    assert float(draws[0][0][:, :5].std(0).min()) > 0.5       # a real draw, not a constant


def _ct_logits(M, n, seed):
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(M, 2 * n, generator=g)
    z[::7] *= 12.0                                            # saturated rows: tanh +-1, std at var_min / var_max
    return z, g


def _ct_action_err(c, nrm):
    """|x - x64| for x = mean + sd n in f32: 4u |mean| + |n| sd esd + 2u (|mean| + sd |n|)."""
    return 4 * U * c.tm.abs() + nrm.abs() * c.sd * c.esd + 2 * U * (c.tm.abs() + c.sd * nrm.abs())


@pytest.mark.parametrize("n", [1, 3, 8, 32])
def test_head_continuous_sample_kernel(ops, n):
    """rlppo_head_continuous_sample on injected normals, ld_aout = n + 5: actions = clamp(tanh z_mean + sd n, -1, 1)
    within twice _ct_action_err, entries clamped with margin exactly +-1; logp_out within 2 dlp of the fp64 log-pdf of
    the clamped action the kernel returned; deterministic draws return tanh z_mean within 4u and log-prob 0; the train
    kernel's logp_out on the returned actions is bit-identical (the same four-term expression on the same f32 action;
    measured on a B200: identical on every row for every n)."""
    M = 3001
    var_min, var_max = 0.1, 1.0
    z32, g = _ct_logits(M, n, 40 + n)
    zbuf, z = _stage(ops, z32, 3)
    nrm = torch.randn(M, n, generator=g) * 1.5
    acts = torch.full((M, n + 5), float("nan"), device=DEV)
    logp = torch.empty(M, device=DEV)
    ops.head_continuous_sample(zbuf, 3, ZPS, M, n, var_min, var_max, acts, logp, normals=nrm.to(DEV))
    torch.cuda.synchronize()
    assert bool(acts[:, n:].isnan().all())
    a = acts[:, :n].cpu().double()
    c = _Ct64(z, a, f32(var_min), f32(var_max))
    x64 = c.tm + c.sd * nrm.double()
    xerr = 2 * _ct_action_err(c, nrm.double())
    assert bool(((a - x64.clamp(-1, 1)).abs() <= xerr).all())
    out = x64.abs() > 1 + xerr
    assert bool(out.any()) and torch.equal(a[out], torch.sign(x64[out]))
    assert bool(((logp.cpu().double() - c.logp).abs() <= 2 * c.dlp).all())
    lp_train = torch.empty(M, device=DEV)
    dz = torch.empty(M, 2 * n + 8, dtype=torch.bfloat16, device=DEV)
    ops.head_continuous_train(zbuf, 3, ZPS, M, n, var_min, var_max, acts, torch.zeros(M, device=DEV),
                              torch.zeros(M, device=DEV), 1.0 / M, 0.2, 0.01, dz, 1, 0, 2 * n, None, logp_out=lp_train)
    det = torch.full((M, n + 5), float("nan"), device=DEV)
    lp_det = torch.full((M,), float("nan"), device=DEV)
    ops.head_continuous_sample(zbuf, 3, ZPS, M, n, var_min, var_max, det, lp_det, deterministic=True)
    torch.cuda.synchronize()
    assert torch.equal(lp_train.view(torch.int32), logp.view(torch.int32))
    assert bool(((det[:, :n].cpu().double() - c.tm).abs() <= 4 * U * c.tm.abs()).all())
    assert bool(det[:, n:].isnan().all()) and bool((lp_det == 0).all())


@pytest.mark.parametrize("n", [1, 3, 8, 32])
def test_head_continuous_philox_stream(ops, n):
    """rlppo_head_continuous_sample from (seed, offset) against the host restatement of its Box-Muller normals, injected:
    action j of a row takes the words x, y of the counter (offset + row, high word, j >> 1, 0), u1 = max(x-uniform,
    2^-24), u2 = y-uniform, n_j = sqrt(-2 log u1) (cos 2 pi u2 for even j, sin for odd j), computed in fp64.  The kernel's
    f32 normal is within rad (4 pi u + 4u) + 4u |n| of it (2 pi u2 rounded, sinf / cosf and logf / sqrtf to a few
    ulp), so the two launches' actions agree within twice sd (that + u |n|) + 2u (|mean| + sd |n|).  The offset 2^32 -
    M/2 makes the launch cross the carry into the counter's high word.  Measured on a B200: at most 0.33 of the bound."""
    M = 2001
    z32, _ = _ct_logits(M, n, 60 + n)
    zbuf, z = _stage(ops, z32, 3)
    off = 2 ** 32 - M // 2
    nrm = np.empty((M, n))
    rad_all = np.empty((M, n))
    for j in range(n):
        q = philox_rows(SEED, off, M, word2=j >> 1)
        u1 = np.maximum(philox_uniform(q[:, 0]), 2.0 ** -24)
        u2 = philox_uniform(q[:, 1])
        rad = np.sqrt(-2.0 * np.log(u1))
        nrm[:, j] = rad * (np.cos(2 * np.pi * u2) if j % 2 == 0 else np.sin(2 * np.pi * u2))
        rad_all[:, j] = rad
    draws = []
    for kw in (dict(seed=SEED, offset=off), dict(normals=torch.from_numpy(nrm).float().to(DEV))):
        a_, l_ = torch.empty(M, n, device=DEV), torch.empty(M, device=DEV)
        ops.head_continuous_sample(zbuf, 3, ZPS, M, n, 0.1, 1.0, a_, l_, **kw)
        draws.append(a_.cpu().double())
    c = _Ct64(z, draws[1], f32(0.1), f32(1.0))
    nt = torch.from_numpy(nrm)
    dn = torch.from_numpy(rad_all) * (4 * np.pi * U + 4 * U) + 5 * U * nt.abs()
    bound = 2 * (c.sd * dn + 2 * U * (c.tm.abs() + c.sd * nt.abs()))
    diff = (draws[0] - draws[1]).abs()
    print(f"ct philox n={n}: max |a - a_host| / bound {float((diff / bound).max()):.3g}")
    assert bool((diff <= bound).all())
    assert abs(float(nt.mean())) < 0.1 and abs(float(nt.std()) - 1) < 0.1


@pytest.mark.parametrize("n_act", [1, 32])
def test_continuous_learn_step0_matches_oracle(n_act):
    """One PPOLearner.learn minibatch of a ContinuousPolicy with 1 and 32 actions in fp32 mode (widths the golden run
    does not have, so the class wiring -- dz_view, act_width, the padded head width -- is exercised where its padding
    differs): the post-clip gradients of the one optimiser step against O.ppo_minibatch_head in fp64 plus
    O.clip_grad_norm per network, 1e-3 rel-L2 per tensor as test_head_learn_matches_reference's step 0 (a 1-element
    tensor against its network's whole gradient norm).  Measured on a B200: at most 7.9e-6."""
    import contextlib
    import io
    from rlgym_ppo_b200.ppo import ExperienceBuffer, PPOLearner
    obs_dim, B, layers, clip, ent, vr = 23, 256, (64, 64), 0.2, 0.01, (0.1, 1.0)
    torch.manual_seed(50 + n_act)
    with contextlib.redirect_stdout(io.StringIO()):
        lr = PPOLearner(obs_dim, n_act, 2, layers, layers, vr, B, 1, 3e-4, 3e-4, clip, ent, B, DEV, precision="fp32")
    pol0 = [p.detach().cpu().double() for p in lr.policy.parameters()]
    val0 = [p.detach().cpu().double() for p in lr.value_net.parameters()]
    rng = np.random.RandomState(n_act)
    states = rng.randn(B, obs_dim).astype(np.float32)
    acts, logp = lr.policy.get_action(states)
    acts = acts.numpy().astype(np.float32)
    old = (logp.numpy() + rng.randn(B) * 0.3).astype(np.float32)
    values = rng.randn(B).astype(np.float32)
    adv = rng.randn(B).astype(np.float32)
    buf = ExperienceBuffer(B, 123, DEV)
    buf.submit_experience(states, acts, old, (rng.randn(B) * 0.1).astype(np.float32), np.roll(states, -1, 0).copy(),
                          np.zeros(B, np.float32), np.zeros(B, np.float64), values, adv)
    captured = capture_steps(lr)
    lr.learn(buf)
    assert len(captured) == 1
    got = unflatten(lr, captured[0])
    f64 = lambda a: torch.from_numpy(a).double()      # noqa: E731
    pg, vg, _ = O.ppo_minibatch_head(2, pol0, val0, f64(states), f64(acts), f64(old), f64(values), f64(adv), clip, ent, B,
                                     vr)
    pg, _ = O.clip_grad_norm(pg)
    vg, _ = O.clip_grad_norm(vg)
    wants = [w.numpy() for w in pg + vg]
    n_pol = len(pg)
    norms = [np.sqrt(sum(float((w ** 2).sum()) for w in wants[:n_pol])), np.sqrt(sum(float((w ** 2).sum()) for w in wants[n_pol:]))]
    errs = [float(np.abs(a - w).max()) / norms[0 if i < n_pol else 1] if w.size == 1 else rel_l2(a, w)
            for i, (a, w) in enumerate(zip(got, wants))]
    print(f"ct learn n_act={n_act}: grad rel-L2 per tensor", [float(f"{e:.2e}") for e in errs])
    assert max(errs) < 1e-3, errs
