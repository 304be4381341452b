"""GPU parity tests, kernel level: every C-ABI entry point of include/rlppo.h against the CPU oracle
(oracle/ref_oracle.py, itself pinned to the reference by tests/test_oracle_vs_golden.py) and against the
golden vectors produced by the reference.  Run with `pytest -m gpu` on a B200."""
import numpy as np
import pytest
import torch

from oracle import ref_oracle as O

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


@pytest.fixture(scope="module")
def ops():
    from rlgym_ppo_b200 import _lib, ops as _ops
    _lib.require_device()
    return _ops


def dev(a, dtype=None):
    t = torch.as_tensor(a)
    if dtype is not None:
        t = t.to(dtype)
    return t.to(DEV).contiguous()


def bf16_round(t):
    return t.to(torch.bfloat16).to(torch.float32)


def rel_l2(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float((a - b).norm() / max(float(b.norm()), 1e-30))


# ------------------------------------------------------------------------------------------------------------
# GAE
# ------------------------------------------------------------------------------------------------------------
def _run_gae(ops, rew, done, trunc, val, gamma, lam, std, head=0):
    std_t = None if std is None else dev(np.asarray([std], np.float32))
    head_t = torch.zeros(head, dtype=torch.float64, device=DEV) if head else None
    vt, adv, ret = ops.gae(dev(rew), dev(done), dev(trunc), dev(val), gamma, lam, std_t, ret_head64=head_t)
    torch.cuda.synchronize()
    return vt.cpu().numpy(), adv.cpu().numpy(), ret.cpu().numpy(), (head_t.cpu().numpy() if head else None)


def test_gae_golden_bit_exact(ops, golden):
    """CUDA scan vs the reference's own outputs: bit-exact advantages / value targets (f32), returns equal to
    the f32 rounding of the reference's f64 list, first-150 returns exact in f64 up to scan re-association."""
    g = golden("gae")
    gamma, lam = g["gamma_lambda"]
    for c in g["cases"]:
        std = g[f"{c}.std"][0]
        std = None if np.isnan(std) else np.float32(std)
        for trunc_dtype in (np.float64, np.float32):
            n = len(g[f"{c}.rew"])
            vt, adv, ret, head = _run_gae(ops, g[f"{c}.rew"], g[f"{c}.done"], g[f"{c}.trunc"].astype(trunc_dtype),
                                          g[f"{c}.val"], gamma, lam, std, head=min(150, n))
            # tolerance 1e-5 scale-aware is the contract; we also count exact matches (expected: all)
            for name, got, want in (("adv", adv, g[f"{c}.adv"]), ("vt", vt, g[f"{c}.vt"]),
                                    ("ret", ret, g[f"{c}.ret"].astype(np.float32))):
                assert np.all(np.abs(got - want) <= 1e-5 * np.maximum(np.abs(want), 1.0)), (c, name)
                mism = int((got != want).sum())
                assert mism <= max(1, n // 1000), (c, name, "bit mismatches", mism, "of", n)
            assert np.allclose(head, g[f"{c}.ret"][:len(head)], rtol=1e-12, atol=1e-14), c


@pytest.mark.parametrize("n,p_done", [(1, 0.0), (2047, 0.01), (2048, 0.0), (2049, 1 / 300), (50000, 1 / 300),
                                      (300001, 0.1), (1 << 20, 0.0), (1 << 20, 1.0)])
def test_gae_vs_oracle_sizes(ops, n, p_done):
    rng = np.random.RandomState(n % 9973)
    rew = (rng.randn(n) * 0.1).astype(np.float32)
    done = (rng.rand(n) < p_done).astype(np.float32)
    trunc = ((rng.rand(n) < 1 / 1500) * (1 - done)).astype(np.float64)
    trunc[-1] = 1 - done[-1]
    val = rng.randn(n + 1).astype(np.float32)
    std = np.float32(0.7)
    vt0, adv0, ret0 = O.gae_nep50_c(rew, done, trunc, val, 0.99, 0.95, std)
    vt, adv, ret, _ = _run_gae(ops, rew, done, trunc, val, 0.99, 0.95, std)
    for name, got, want in (("adv", adv, adv0), ("vt", vt, vt0), ("ret", ret, ret0.astype(np.float32))):
        err = np.abs(got - want) / np.maximum(np.abs(want), 1.0)
        assert err.max() <= 1e-5, (name, float(err.max()))
        assert (got != want).mean() < 1e-3, (name, "bit mismatch rate", float((got != want).mean()))


@pytest.mark.parametrize("trunc_dtype", [np.float64, np.float32])
def test_gae_fractional_and_negative_zero_flags(ops, trunc_dtype):
    """Flags that are not exactly +0 / 1 (fractional, -0.0, 2.0) leave the staged kernel's 0/1 fast path and must be
    evaluated as the reference writes them (torch_functions.py:59-60): aligned full tiles, mixed with ordinary steps."""
    rng = np.random.RandomState(11)
    n = 3 * 2048 + 77
    rew = (rng.randn(n) * 0.1).astype(np.float32)
    done = (rng.rand(n) < 0.01).astype(np.float32)
    trunc = ((rng.rand(n) < 0.005) * (1 - done)).astype(trunc_dtype)
    odd = rng.choice(n, 64, replace=False)
    done[odd[:16]] = 0.5
    done[odd[16:24]] = -0.0
    done[odd[24:32]] = 2.0
    trunc[odd[32:48]] = 0.25
    trunc[odd[48:56]] = -0.0
    trunc[odd[56:]] = 1.5
    val = rng.randn(n + 1).astype(np.float32)
    for std in (np.float32(0.7), None):
        vt0, adv0, ret0 = O.gae_nep50_c(rew, done, trunc.astype(np.float64), val, 0.99, 0.95, std)
        vt, adv, ret, _ = _run_gae(ops, rew, done, trunc, val, 0.99, 0.95, std)
        for name, got, want in (("adv", adv, adv0), ("vt", vt, vt0), ("ret", ret, ret0.astype(np.float32))):
            err = np.abs(got - want) / np.maximum(np.abs(want), 1.0)
            assert err.max() <= 1e-5, (name, float(err.max()))
            assert (got != want).mean() < 1e-3, (name, "bit mismatch rate", float((got != want).mean()))


def _assert_vs_oracle(outs, want, case):
    """(vt, adv, ret) device tensors against the oracle's (vt, adv, ret): 1e-5 scale-aware, bit mismatches < 1e-3."""
    for name, got, w in zip(("vt", "adv", "ret"), outs, want):
        got, w = got.cpu().numpy(), w.astype(np.float32)
        err = np.abs(got - w) / np.maximum(np.abs(w), 1.0)
        assert err.max() <= 1e-5, (case, name, float(err.max()))
        assert (got != w).mean() < 1e-3, (case, name, "bit mismatch rate", float((got != w).mean()))


def test_gae_unaligned_views_and_carry(ops):
    """Misaligned inputs, misaligned `out=` buffers and chunk summaries of misaligned views take the bounds-checked path
    on every tile; carry_in + chunk summaries reproduce the unsharded scan.  600001 steps > 444 CTAs x 1024: CTAs take
    several tiles."""
    for n, cut in ((10007, 6000), (600001, 360000)):
        for trunc_dtype in (np.float32, np.float64):
            case = (n, trunc_dtype.__name__)
            rng = np.random.RandomState(3)
            rew = (rng.randn(n) * 0.1).astype(np.float32)
            done = (rng.rand(n) < 0.002).astype(np.float32)
            val = rng.randn(n + 1).astype(np.float32)
            trunc = ((rng.rand(n) < 1 / 1500) * (1 - done)).astype(trunc_dtype)
            vt0, adv0, ret0 = O.gae_nep50_c(rew, done, trunc, val, 0.99, 0.95, None)
            pad = lambda a: dev(np.concatenate([[0], a]).astype(a.dtype))[1:]  # noqa: E731  4-byte-offset views
            vt, adv, ret = ops.gae(pad(rew), pad(done), pad(trunc), pad(val), 0.99, 0.95, None)
            assert np.allclose(adv.cpu().numpy(), adv0, rtol=1e-6, atol=1e-6), case
            assert np.allclose(ret.cpu().numpy(), ret0, rtol=1e-6, atol=1e-6), case
            _assert_vs_oracle((vt, adv, ret), (vt0, adv0, ret0), case)
            # aligned inputs, outputs at a 4-byte offset
            out = tuple(torch.zeros(n + 1, dtype=torch.float32, device=DEV)[1:] for _ in range(3))
            ops.gae(dev(rew), dev(done), dev(trunc), dev(val), 0.99, 0.95, None, out=out)
            _assert_vs_oracle(out, (vt0, adv0, ret0), case)
            # two shards: right shard first, its first values are the left shard's carry
            r, d, t, v = dev(rew), dev(done), dev(trunc), dev(val)
            vt_r, adv_r, ret_r = ops.gae(r[cut:].clone(), d[cut:].clone(), t[cut:].clone(), v[cut:].clone(), 0.99, 0.95,
                                         None)
            _assert_vs_oracle((vt_r, adv_r, ret_r), (vt0[cut:], adv0[cut:], ret0[cut:]), case)
            summ = ops.gae_chunk_summary(r[cut:].clone(), d[cut:].clone(), t[cut:].clone(), v[cut:].clone(), 0.99, 0.95,
                                         None)
            s = summ.cpu().numpy()
            assert abs(s[1] - float(adv0[cut])) < 1e-5 and abs(s[3] - float(ret0[cut])) < 1e-5, case
            summ_u = ops.gae_chunk_summary(pad(rew[cut:]), pad(done[cut:]), pad(trunc[cut:]), pad(val[cut:]), 0.99, 0.95,
                                           None)
            s_u = summ_u.cpu().numpy()
            assert abs(s_u[1] - float(adv0[cut])) < 1e-5 and abs(s_u[3] - float(ret0[cut])) < 1e-5, case
            assert np.allclose(s_u, s, rtol=1e-12, atol=1e-12), case
            # carry = the right shard's values at its first step: bA and bR of its summary
            carry = dev(np.asarray([s[1], s[3]], np.float64))
            vt_l, adv_l, ret_l = ops.gae(r[:cut].clone(), d[:cut].clone(), t[:cut].clone(), v[:cut + 1].clone(), 0.99,
                                         0.95, None, carry_in=carry)
            assert np.allclose(adv_l.cpu().numpy(), adv0[:cut], rtol=1e-6, atol=1e-6), case
            assert np.allclose(ret_l.cpu().numpy(), ret0[:cut], rtol=1e-6, atol=1e-6), case
            assert np.allclose(adv_r.cpu().numpy(), adv0[cut:], rtol=1e-6, atol=1e-6), case
            _assert_vs_oracle((vt_l, adv_l, ret_l), (vt0[:cut], adv0[:cut], ret0[:cut]), case)
            # the left shard again from misaligned views, with the same carry
            _assert_vs_oracle(ops.gae(pad(rew[:cut]), pad(done[:cut]), pad(trunc[:cut]), pad(val[:cut + 1]), 0.99, 0.95,
                                      None, carry_in=carry), (vt0[:cut], adv0[:cut], ret0[:cut]), case)


def test_gae_linearity_full_size(ops):
    """Size-independent property at a bench size (2^24 steps): with std=None the returns are linear in the
    rewards, R(a*r1 + r2) = a*R(r1) + R(r2), and all-done rollouts give R = r, A = r - V."""
    n = 1 << 24
    g = torch.Generator(device=DEV).manual_seed(0)
    r1 = torch.randn(n, device=DEV, generator=g) * 0.1
    r2 = torch.randn(n, device=DEV, generator=g) * 0.1
    done = (torch.rand(n, device=DEV, generator=g) < 1 / 300).float()
    trunc = torch.zeros(n, device=DEV)
    val = torch.zeros(n + 1, device=DEV)
    _, _, R1 = ops.gae(r1, done, trunc, val, 0.99, 0.95, None)
    _, _, R2 = ops.gae(r2, done, trunc, val, 0.99, 0.95, None)
    _, _, R3 = ops.gae(2.0 * r1 + r2, done, trunc, val, 0.99, 0.95, None)
    assert float((R3 - (2.0 * R1 + R2)).abs().max()) < 2e-5
    ones = torch.ones(n, device=DEV)
    v = torch.randn(n + 1, device=DEV, generator=g)
    vt, adv, ret = ops.gae(r1, ones, trunc, v, 0.99, 0.95, None)
    assert torch.equal(ret, r1) and torch.equal(adv, r1 - v[:-1])


# ------------------------------------------------------------------------------------------------------------
# Welford
# ------------------------------------------------------------------------------------------------------------
def test_welford_golden(ops, golden):
    g = golden("welford")
    mean = torch.zeros(1, device=DEV)
    m2 = torch.zeros(1, device=DEV)
    cnt = torch.zeros(1, dtype=torch.int64, device=DEV)
    std = torch.zeros(1, device=DEV)
    mu = torch.zeros(1, device=DEV)
    s = dev(g["samples"])
    ops.welford_update(mean, m2, cnt, s, 0, std, mu)
    assert std.item() == 1.0 and mu.item() == 0.0
    ops.welford_update(mean, m2, cnt, s, 150, std, mu)
    assert np.array_equal(mean.cpu().numpy(), g["s150.mean"]) and np.array_equal(m2.cpu().numpy(), g["s150.m2"])
    assert cnt.item() == 150 and np.array_equal(std.cpu().numpy(), g["s150.std"])
    ops.welford_update(mean, m2, cnt, s[150:], 1, std, mu)
    assert np.array_equal(mean.cpu().numpy(), g["s151.mean"]) and np.array_equal(m2.cpu().numpy(), g["s151.m2"])
    ops.welford_update(mean, m2, cnt, s[151:], 249, std, mu)
    assert np.array_equal(mean.cpu().numpy(), g["s400.mean"]) and np.array_equal(m2.cpu().numpy(), g["s400.m2"])
    assert np.array_equal(std.cpu().numpy(), g["s400.std"])
    # zero variance guard
    mean.zero_(); m2.zero_(); cnt.zero_()
    ops.welford_update(mean, m2, cnt, dev(np.full(5, 2.0)), 5, std, mu)
    assert np.array_equal(std.cpu().numpy(), g["const.std"]) and np.array_equal(mu.cpu().numpy(), g["const.mean"])
    # vector f32 stats
    xs = g["vec.samples"]
    mean5 = torch.zeros(5, device=DEV); m25 = torch.zeros(5, device=DEV); c5 = torch.zeros(1, dtype=torch.int64, device=DEV)
    ops.welford_update(mean5, m25, c5, dev(xs[:40]), 40)
    assert np.array_equal(mean5.cpu().numpy(), g["vec.a.mean"]) and np.array_equal(m25.cpu().numpy(), g["vec.a.m2"])


# ------------------------------------------------------------------------------------------------------------
# ring + gather
# ------------------------------------------------------------------------------------------------------------
def test_ring_append_and_gather_vs_oracle(ops):
    rng = np.random.RandomState(5)
    cap, obs = 1000, 89

    class Buf:
        pass

    b = Buf()
    b.capacity, b.obs_dim, b.start = cap, obs, 0
    b.states = torch.zeros(cap, obs, device=DEV)
    b.states_bf16 = torch.zeros(cap, 96, dtype=torch.bfloat16, device=DEV)
    for f in ("actions", "log_probs", "values", "advantages"):
        setattr(b, f, torch.zeros(cap, device=DEV))
    size = 0
    ob = O.BufferOracle(cap, 123)
    for n in (300, 500, 450, 1000, 70):
        f = {k: rng.randn(n).astype(np.float32) for k in O.FIELDS}
        f["states"] = rng.randn(n, obs).astype(np.float32)
        f["next_states"] = rng.randn(n, obs).astype(np.float32)
        f["truncated"] = (rng.rand(n) < 0.1).astype(np.float64)
        ob.submit(**f)
        first = (b.start + size) % cap
        ops.ring_append(b.states, first, dev(f["states"]), n, ring_bf16=b.states_bf16)
        ops.ring_append(b.actions, first, dev(f["actions"]), n)
        ops.ring_append(b.log_probs, first, dev(f["log_probs"]), n)
        ops.ring_append(b.values, first, dev(f["values"]), n)
        ops.ring_append(b.advantages, first, dev(f["truncated"]), n)  # f64 source path
        over = max(0, size + n - cap)
        b.start = (b.start + over) % cap
        size = min(cap, size + n)
        total = ob.f["rewards"].shape[0]
        assert total == size
        idx = ob.rng.permutation(total)
        B = 256
        outs = dict(out_actions=torch.empty(B, device=DEV), out_logp=torch.empty(B, device=DEV),
                    out_values=torch.empty(B, device=DEV), out_adv=torch.empty(B, device=DEV),
                    out_states=torch.empty(B, obs, device=DEV),
                    out_states_bf16=torch.empty(B, 96, dtype=torch.bfloat16, device=DEV))
        ii = idx[:B]
        ops.gather_batch(b, dev(ii), **outs)
        torch.cuda.synchronize()
        assert np.array_equal(outs["out_actions"].cpu().numpy(), ob.f["actions"][ii])
        assert np.array_equal(outs["out_logp"].cpu().numpy(), ob.f["log_probs"][ii])
        assert np.array_equal(outs["out_values"].cpu().numpy(), ob.f["values"][ii])
        assert np.array_equal(outs["out_adv"].cpu().numpy(), ob.f["truncated"][ii])  # the f64-cast field
        assert np.array_equal(outs["out_states"].cpu().numpy(), ob.f["states"][ii])
        want = torch.from_numpy(ob.f["states"][ii]).to(torch.bfloat16)
        got = outs["out_states_bf16"].cpu()
        assert torch.equal(got[:, :obs], want) and float(got[:, obs:].float().abs().max()) == 0.0


def test_ring_append_fields_device_state_vs_oracle(ops):
    """All nine rings in one launch with the ring position kept on the device (rlppo_ring_append_fields_dev): every
    logical field equals the FIFO oracle (`_cat`, experience_buffer.py:17-37) after appends that fill, wrap inside a
    64-row block, exactly fill and overfill the ring; f64 sources are cast like torch.as_tensor(..., float32)."""
    rng = np.random.RandomState(9)
    cap, obs, pad = 777, 89, 96
    rings = {k: torch.zeros((cap, obs) if k in ("states", "next_states") else (cap,), device=DEV) for k in O.FIELDS}
    rings_bf16 = torch.full((cap, pad), 7.0, dtype=torch.bfloat16, device=DEV)   # padding must come out as zeros
    state = torch.zeros(2, dtype=torch.int64, device=DEV)
    ob = O.BufferOracle(cap, 123)
    start = size = 0
    for n in (300, 100, 450, 777, 70, 5, 776):
        f = {k: rng.randn(n).astype(np.float32) for k in O.FIELDS}
        f["states"] = rng.randn(n, obs).astype(np.float32)
        f["next_states"] = rng.randn(n, obs).astype(np.float32)
        f["truncated"] = (rng.rand(n) < 0.1).astype(np.float64)
        ob.submit(**f)
        fields = [(rings[k], dev(f[k]), rings_bf16 if k == "states" else None) for k in O.FIELDS]
        ops.ring_append_fields(fields, cap, 0, n, state_dev=state)
        over = max(0, size + n - cap)
        start, size = (start + over) % cap, min(cap, size + n)
        assert state.cpu().tolist() == [start, size]
        order = (start + np.arange(size)) % cap
        for k in O.FIELDS:
            assert np.array_equal(rings[k].cpu().numpy()[order], ob.f[k].astype(np.float32)), k
        got = rings_bf16.cpu()[order]
        assert torch.equal(got[:, :obs], torch.from_numpy(ob.f["states"]).to(torch.bfloat16))
        assert float(got[:, obs:].float().abs().max()) == 0.0


# ------------------------------------------------------------------------------------------------------------
# tensor-core layers
# ------------------------------------------------------------------------------------------------------------
def _mk(shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return bf16_round(torch.randn(*shape, generator=g) * scale)


def _head_setup(M, K, A, seed):
    h = torch.relu(_mk((M, K), seed))
    w = _mk((A, K), seed + 1, 0.2)
    b = torch.randn(A, generator=torch.Generator().manual_seed(seed + 2)) * 0.1
    Ap = (A + 7) // 8 * 8
    wq = torch.zeros(Ap, K)
    wq[:A] = w
    return h, w, b, wq


@pytest.mark.parametrize("M,K,A", [(1000, 256, 90), (50000, 256, 90), (333, 64, 90), (500, 256, 21), (700, 128, 200)])
def test_policy_head_sample(ops, M, K, A):
    h, w, b, wq = _head_setup(M, K, A, 10)
    u = torch.rand(M, generator=torch.Generator().manual_seed(1))
    acts = torch.empty(M, device=DEV)
    acts64 = torch.empty(M, dtype=torch.int64, device=DEV)
    logp = torch.empty(M, device=DEV)
    probs = torch.empty(M, A, device=DEV)
    ops.policy_head_sample(dev(h, torch.bfloat16), dev(wq, torch.bfloat16), dev(b), A, K, u=dev(u),
                           actions_out=acts, actions_i64_out=acts64, logp_out=logp, probs_out=probs)
    torch.cuda.synchronize()
    z = h.double() @ w.double().t() + b.double()
    p_ref = torch.softmax(z, -1)
    assert float((probs.cpu().double() - p_ref).abs().max()) < 2e-5
    a = acts64.cpu()
    assert torch.equal(acts.cpu().long(), a) and int(a.min()) >= 0 and int(a.max()) < A
    # inverse-CDF contract on the kernel's own probabilities: cdf[a-1] <= u*P < cdf[a] (up to fp32 summation slack)
    pc = probs.cpu().double().clamp(1e-11, 1.0)
    cdf = pc.cumsum(-1)
    thr = u.double() * cdf[:, -1]
    hi = cdf.gather(-1, a.view(-1, 1)).flatten()
    lo = torch.where(a > 0, cdf.gather(-1, (a - 1).clamp(min=0).view(-1, 1)).flatten(), torch.zeros(M, dtype=torch.double))
    assert bool(((thr < hi + 1e-5) & (thr >= lo - 1e-5)).all())
    agree = (O.sample_inverse_cdf(p_ref.float(), u) == a).float().mean()
    assert agree > 0.999, float(agree)
    lp_ref = torch.log(p_ref.clamp(1e-11, 1.0)).gather(-1, a.view(-1, 1)).flatten()
    assert float((logp.cpu().double() - lp_ref).abs().max()) < 1e-4
    # deterministic branch = per-row argmax
    ops.policy_head_sample(dev(h, torch.bfloat16), dev(wq, torch.bfloat16), dev(b), A, K, deterministic=True,
                           actions_i64_out=acts64, logp_out=logp)
    assert (acts64.cpu() == z.argmax(-1)).float().mean() > 0.999


def test_policy_head_sample_philox_distribution(ops):
    """Chi-square of the Philox-driven sampler against the softmax probabilities (same row repeated)."""
    M, K, A = 200000, 64, 90
    h1, w, b, wq = _head_setup(1, K, A, 20)
    h = h1.expand(M, K).contiguous()
    acts64 = torch.empty(M, dtype=torch.int64, device=DEV)
    ops.policy_head_sample(dev(h, torch.bfloat16), dev(wq, torch.bfloat16), dev(b), A, K, seed=1234, offset=0,
                           actions_i64_out=acts64)
    p = torch.softmax(h1.double() @ w.double().t() + b.double(), -1).flatten()
    counts = torch.bincount(acts64.cpu(), minlength=A).double()
    chi2 = float((((counts - M * p) ** 2) / (M * p)).sum())
    assert chi2 < 160.0, chi2   # 89 dof: mean 89, 99.99th percentile ~ 146
    acts_b = torch.empty(M, dtype=torch.int64, device=DEV)
    ops.policy_head_sample(dev(h, torch.bfloat16), dev(wq, torch.bfloat16), dev(b), A, K, seed=1234, offset=0,
                           actions_i64_out=acts_b)
    assert torch.equal(acts_b, acts64)          # counter-based: reproducible
    ops.policy_head_sample(dev(h, torch.bfloat16), dev(wq, torch.bfloat16), dev(b), A, K, seed=1234, offset=M,
                           actions_i64_out=acts_b)
    assert not torch.equal(acts_b, acts64)      # a new offset is a new stream


@pytest.mark.parametrize("M,K,A", [(1000, 256, 90), (50000, 256, 90), (300, 64, 90), (640, 128, 200)])
def test_policy_head_train(ops, M, K, A):
    h, w, b, wq = _head_setup(M, K, A, 30)
    g = torch.Generator().manual_seed(7)
    acts = torch.randint(0, A, (M,), generator=g).float()
    z = (h @ w.t() + b)
    lp_all = torch.log(torch.softmax(z, -1).clamp(1e-11, 1))
    old = lp_all.gather(-1, acts.long().view(-1, 1)).flatten() + torch.randn(M, generator=g) * 0.3
    adv = torch.randn(M, generator=g) * 0.5
    Ap = (A + 7) // 8 * 8
    dz = torch.full((M, Ap), 3.0, dtype=torch.bfloat16, device=DEV)
    metrics = torch.zeros(8, device=DEV)
    logp = torch.empty(M, device=DEV)
    B_total = 2 * M   # pretend this is half a batch: inv_batch = 1/(2M)
    ops.policy_head_train(dev(h, torch.bfloat16), dev(wq, torch.bfloat16), dev(b), A, K, dev(acts), dev(old), dev(adv),
                          1.0 / B_total, 0.2, 0.01, dz, metrics, logp_out=logp)
    torch.cuda.synchronize()
    # oracle: policy = single Linear on h; reuse ppo_minibatch with an identity value net of the same width
    zt = z.double().clone().requires_grad_(True)
    s = torch.softmax(zt, -1)
    p = s.clamp(1e-11, 1.0)
    lpa = torch.log(p)
    lp = lpa.gather(-1, acts.long().view(-1, 1)).flatten()
    ent = -(lpa * p).sum(-1)
    ratio = torch.exp(lp - old.double())
    surr = torch.min(ratio * adv.double(), ratio.clamp(0.8, 1.2) * adv.double())
    loss = (-surr.sum() - 0.01 * ent.sum()) / B_total
    loss.backward()
    m = metrics.cpu().double()
    assert m[4] == M
    assert abs(m[0] / M - float(ent.mean())) < 1e-4 * max(1, abs(float(ent.mean())))
    kl = ((ratio - 1) - (lp - old.double())).mean()
    assert abs(m[1] / M - float(kl)) < 1e-4
    assert abs(m[2] / M - float(((ratio - 1).abs() > 0.2).double().mean())) < 2e-3
    assert abs(m[3] / M - float(surr.mean())) < 1e-4
    assert float((logp.cpu().double() - lp.detach()).abs().max()) < 1e-4
    got = dz.float().cpu()
    assert float(got[:, A:].abs().max()) == 0.0 if Ap > A else True
    assert rel_l2(got[:, :A], zt.grad.float()) < 6e-3, rel_l2(got[:, :A], zt.grad.float())  # bf16 output rounding


@pytest.mark.parametrize("M,K", [(1000, 256), (50001, 256), (333, 64), (2000, 1024), (512, 2048)])
def test_value_head(ops, M, K):
    h = torch.relu(_mk((M, K), 40))
    w = torch.randn(K, generator=torch.Generator().manual_seed(41)) * 0.1
    b = torch.tensor([0.3])
    tgt = torch.randn(M, generator=torch.Generator().manual_seed(42))
    v = torch.empty(M, device=DEV)
    ops.value_head(dev(h, torch.bfloat16), dev(w), dev(b), K, values_out=v)
    ref_v = (h.double() @ w.double() + 0.3)
    assert float((v.cpu().double() - ref_v).abs().max()) < 1e-4
    dh = torch.empty(M, K, dtype=torch.bfloat16, device=DEV)
    dw = torch.full((K,), 0.5, device=DEV)
    db = torch.zeros(1, device=DEV)
    metrics = torch.zeros(8, device=DEV)
    inv_b = 1.0 / (3 * M)
    ops.value_head(dev(h, torch.bfloat16), dev(w), dev(b), K, values_out=v, targets=dev(tgt), inv_batch=inv_b, dh=dh,
                   dw=dw, db=db, metrics=metrics)
    torch.cuda.synchronize()
    dv = 2 * inv_b * (ref_v - tgt.double())
    assert rel_l2(dh.float().cpu(), (dv[:, None] * w.double()[None, :] * (h > 0).double()).float()) < 4e-3
    assert rel_l2(dw.cpu(), (dv[:, None] * h.double()).sum(0).float() + 0.5) < 1e-4
    assert abs(db.item() - float(dv.sum())) < 1e-4 * max(1.0, abs(float(dv.sum())))
    m = metrics.cpu().double()
    assert m[6] == M and abs(m[5] / M - float(((ref_v - tgt.double()) ** 2).mean())) < 1e-4


# ------------------------------------------------------------------------------------------------------------
# optimiser
# ------------------------------------------------------------------------------------------------------------
def test_clip_adam_vs_torch(ops):
    torch.manual_seed(0)
    sizes = [177754, 154881]
    seg = [0, sizes[0], sizes[0] + sizes[1]]
    p0 = torch.randn(seg[-1]) * 0.05
    params = [torch.nn.Parameter(p0[seg[i]:seg[i + 1]].clone()) for i in range(2)]
    opts = [torch.optim.Adam([params[0]], lr=3e-4), torch.optim.Adam([params[1]], lr=1e-4)]
    p = dev(p0.clone()); m = torch.zeros_like(p); v = torch.zeros_like(p)
    sq = torch.zeros(2, device=DEV); lr = dev(torch.tensor([3e-4, 1e-4])); steps = torch.zeros(2, dtype=torch.int64, device=DEV)
    before = p.clone()
    for it in range(5):
        g = torch.randn(seg[-1]) * (0.01 if it % 2 else 1e-4)   # alternate clipped / unclipped regimes
        for i in range(2):
            params[i].grad = g[seg[i]:seg[i + 1]].clone()
            torch.nn.utils.clip_grad_norm_([params[i]], 0.5)
            opts[i].step()
        gd = dev(g)
        ops.grad_sqnorm(gd, seg, sq)
        ops.clip_adam(p, gd, m, v, seg, sq, lr, steps)
    torch.cuda.synchronize()
    ref = torch.cat([q.detach() for q in params])
    assert float((p.cpu() - ref).abs().max()) < 2e-7
    assert steps.tolist() == [5, 5]
    st = opts[0].state[params[0]]
    assert rel_l2(m[:sizes[0]].cpu(), st["exp_avg"]) < 1e-5 and rel_l2(v[:sizes[0]].cpu(), st["exp_avg_sq"]) < 1e-5
    out = torch.zeros(2, device=DEV)
    ops.sqdiff(p, before, seg, out)
    want = [float((ref[seg[i]:seg[i + 1]] - p0[seg[i]:seg[i + 1]]).norm()) for i in range(2)]
    assert np.allclose(out.sqrt().cpu().numpy(), want, rtol=1e-4)


@pytest.mark.parametrize("sizes", [[177754, 154881], [7575083, 7575088], [5, 1]])
def test_norm_clip_adam_one_launch_vs_torch_and_deterministic(ops, sizes):
    """rlppo_norm_clip_adam (norm + clip + Adam in one launch, grid barrier, fixed-order norm) against torch's
    clip_grad_norm_ + Adam, against the two-launch path, and bit-identical from run to run (what keeps data-parallel
    replicas in step); the workspace counters clean themselves (5 launches on one workspace)."""
    torch.manual_seed(1)
    seg = [0, sizes[0], sizes[0] + sizes[1]]
    p0 = torch.randn(seg[-1]) * 0.05
    params = [torch.nn.Parameter(p0[seg[i]:seg[i + 1]].clone()) for i in range(2)]
    opts = [torch.optim.Adam([params[0]], lr=3e-4), torch.optim.Adam([params[1]], lr=1e-4)]
    lr = dev(torch.tensor([3e-4, 1e-4]))
    runs = []
    for rep in range(2):
        p = dev(p0.clone()); m = torch.zeros_like(p); v = torch.zeros_like(p)
        sq = torch.zeros(2, device=DEV); steps = torch.zeros(2, dtype=torch.int64, device=DEV)
        gen = torch.Generator().manual_seed(2)
        for it in range(5):
            g = torch.randn(seg[-1], generator=gen) * (0.01 if it % 2 else 1e-4)
            if rep == 0:
                for i in range(2):
                    params[i].grad = g[seg[i]:seg[i + 1]].clone()
                    torch.nn.utils.clip_grad_norm_([params[i]], 0.5)
                    opts[i].step()
            gd = dev(g)
            ops.norm_clip_adam(p, gd, m, v, seg, sq, lr, steps)
            want_sq = [float((g[seg[i]:seg[i + 1]].double() ** 2).sum()) for i in range(2)]
            assert np.allclose(sq.cpu().numpy(), want_sq, rtol=1e-5)
        torch.cuda.synchronize()
        assert steps.tolist() == [5, 5]
        runs.append((p.clone(), m.clone(), v.clone()))
    ref = torch.cat([q.detach() for q in params])
    assert float((runs[0][0].cpu() - ref).abs().max()) < 2e-7
    for a, b in zip(runs[0], runs[1]):
        assert torch.equal(a, b), "the one-launch optimiser step is not deterministic"


def test_weight_and_rows_to_bf16(ops):
    w = torch.randn(90, 89)
    wq = torch.full((96, 96), 9.0, dtype=torch.bfloat16, device=DEV)
    wt = torch.full((96, 96), 9.0, dtype=torch.bfloat16, device=DEV)
    ops.weight_to_bf16(dev(w), wq, wt)
    ref = torch.zeros(96, 96); ref[:90, :89] = w
    assert torch.equal(wq.cpu(), ref.to(torch.bfloat16)) and torch.equal(wt.cpu(), ref.t().contiguous().to(torch.bfloat16))
    x = torch.randn(1001, 89)
    xb = torch.full((1001, 96), 9.0, dtype=torch.bfloat16, device=DEV)
    ops.rows_to_bf16(dev(x), xb)
    refx = torch.zeros(1001, 96); refx[:, :89] = x
    assert torch.equal(xb.cpu(), refx.to(torch.bfloat16))
    mean, std = torch.randn(89), torch.rand(89) + 0.5
    ops.rows_to_bf16(dev(x), xb, dev(mean), dev(std), 5.0)
    refx[:, :89] = ((x - mean) / std).clamp(-5, 5)
    assert torch.equal(xb.cpu(), refx.to(torch.bfloat16))
