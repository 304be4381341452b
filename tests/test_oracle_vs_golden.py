"""Pins oracle/ (CPU restatement) against the golden vectors produced by the reference itself
(tests/golden/make_golden.py).  CPU only."""
import numpy as np
import pytest
import torch

from oracle import ref_oracle as O


def _params(g, prefix):
    out, i = [], 0
    while f"{prefix}.{i}" in g:
        out.append(torch.from_numpy(g[f"{prefix}.{i}"]))
        i += 1
    return out


def test_gae_nep50_matches_reference_bit_exact(golden):
    g = golden("gae")
    gamma, lam = g["gamma_lambda"]
    for c in g["cases"]:
        std = g[f"{c}.std"][0]
        std = None if np.isnan(std) else np.float32(std)
        for fn in (O.gae_nep50, O.gae_nep50_c):
            vt, adv, ret = fn(g[f"{c}.rew"], g[f"{c}.done"], g[f"{c}.trunc"], g[f"{c}.val"], gamma, lam, std)
            assert np.array_equal(adv, g[f"{c}.adv"]), (c, fn.__name__)
            assert np.array_equal(vt, g[f"{c}.vt"]), (c, fn.__name__)
            assert np.array_equal(ret, g[f"{c}.ret"]), (c, fn.__name__)


def test_gae_fp64_statement_within_tolerance(golden):
    g = golden("gae")
    gamma, lam = g["gamma_lambda"]
    for c in g["cases"]:
        std = g[f"{c}.std"][0]
        std = None if np.isnan(std) else float(std)
        vt, adv, ret = O.gae_fp64(g[f"{c}.rew"], g[f"{c}.done"], g[f"{c}.trunc"], g[f"{c}.val"], gamma, lam, std)
        for a, b in ((vt, g[f"{c}.vt"]), (adv, g[f"{c}.adv"]), (ret, g[f"{c}.ret"])):
            assert np.all(np.abs(a - b) <= 1e-5 * np.maximum(np.abs(b), 1.0)), c


def test_welford(golden):
    g = golden("welford")
    st = O.WelfordOracle(1)
    assert np.array_equal(st.get_std(), g["std_empty"]) and np.array_equal(st.get_mean(), g["mean_empty"])
    s = g["samples"]
    st.increment(list(s[:150]), 150)
    assert np.array_equal(st.mean, g["s150.mean"]) and np.array_equal(st.m2, g["s150.m2"])
    assert st.count == g["s150.count"][0] and np.array_equal(st.get_std(), g["s150.std"])
    st.increment(list(s[150:151]), 1)
    assert np.array_equal(st.mean, g["s151.mean"]) and np.array_equal(st.m2, g["s151.m2"])
    st.increment(list(s[151:400]), 249)
    assert np.array_equal(st.mean, g["s400.mean"]) and np.array_equal(st.m2, g["s400.m2"])
    assert np.array_equal(st.get_std(), g["s400.std"])
    # C restatement of the same update
    lib = O._c_lib()
    mean = np.zeros(1, np.float32); m2 = np.zeros(1, np.float32); cnt = np.zeros(1, np.int64)
    lib.oracle_welford_update(mean.ctypes.data, m2.ctypes.data, cnt.ctypes.data, s.ctypes.data, 400)
    assert np.array_equal(mean, g["s400.mean"]) and np.array_equal(m2, g["s400.m2"]) and cnt[0] == 400
    z = O.WelfordOracle(1)
    z.increment([np.float64(2.0)] * 5, 5)
    assert np.array_equal(z.get_std(), g["const.std"]) and np.array_equal(z.get_mean(), g["const.mean"])
    a, b = O.WelfordOracle(5), O.WelfordOracle(5)
    xs = g["vec.samples"]
    a.increment(xs[:40], 40)
    b.increment(xs[40:], 20)
    assert np.array_equal(a.mean, g["vec.a.mean"]) and np.array_equal(a.m2, g["vec.a.m2"])
    ser = g["vec.b.ser"]
    assert np.allclose(np.concatenate([b.mean, b.m2, [b.count]]), ser, rtol=0, atol=0)
    a.merge(ser[:5], ser[5:10], int(ser[-1]))
    assert np.allclose(a.mean, g["vec.merged.mean"], rtol=1e-6, atol=1e-7)
    assert np.allclose(a.m2, g["vec.merged.m2"], rtol=1e-6, atol=1e-6)
    assert a.count == g["vec.merged.count"][0]
    assert np.allclose(a.get_std(), g["vec.merged.std"], rtol=1e-6)


def test_buffer_fifo_and_shuffle_bit_exact(golden):
    g = golden("buffer")
    obs_dim, max_size, seed = g["cfg"]
    buf = O.BufferOracle(int(max_size), int(seed))
    for k, n in enumerate(g["sizes"]):
        buf.submit(**{name: g[f"in{k}.{name}"] for name in O.FIELDS})
        for name in O.FIELDS:
            assert np.array_equal(buf.f[name], g[f"after{k}.{name}"]), (k, name)
        for ep in range(2):
            batches = list(buf.batches(32))
            assert len(batches) == g[f"after{k}.ep{ep}.nbatches"][0]
            for bi, (_, tup) in enumerate(batches):
                for name, arr in zip(("actions", "log_probs", "states", "values", "advantages"), tup):
                    assert np.array_equal(arr, g[f"after{k}.ep{ep}.b{bi}.{name}"]), (k, ep, bi, name)


def test_mt19937_permutation_restatement(golden):
    g = golden("buffer")
    for impl in (O.mt19937_permutation, O.mt19937_permutation_c):
        st = np.random.RandomState(7).get_state()
        p1, key, pos = impl(st[1], st[2], 1000)
        p2, key, pos = impl(key, pos, 1000)
        assert np.array_equal(p1, g["perm1000"]) and np.array_equal(p2, g["perm1000.b"]), impl.__name__
        r = np.random.RandomState(7)
        r.permutation(1000); r.permutation(1000)
        st2 = r.get_state()
        assert np.array_equal(key, st2[1]) and pos == st2[2]
    st = np.random.RandomState(123).get_state()
    p1, key, pos = O.mt19937_permutation_c(st[1], st[2], 150000)
    p2, key, pos = O.mt19937_permutation_c(key, pos, 150000)
    assert np.array_equal(p1[:64], g["perm150000.head"]) and np.array_equal(p2[:64], g["perm150000.second_head"])


def test_philox4x32_10_known_answers():
    """The host Philox that the samplers' stream tests draw from, pinned to the Random123 known-answer vectors
    (kat_vectors, philox4x32_10), all three evaluated in one vectorised call; the uniform is the top 24 bits."""
    from parity_helpers import philox4x32_10, philox_rows, philox_uniform
    ctr = np.array([[0, 0, 0, 0], [0xFFFFFFFF] * 4, [0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344]], np.uint32)
    key = np.array([[0, 0], [0xFFFFFFFF] * 2, [0xA4093822, 0x299F31D0]], np.uint32)
    want = np.array([[0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8],
                     [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD],
                     [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]], np.uint32)
    assert np.array_equal(philox4x32_10(ctr, key), want)
    assert np.array_equal(philox_uniform(np.array([0, 0xFF, 0x100, 0xFFFFFFFF], np.uint32)),
                          [0.0, 0.0, 2.0 ** -24, 1.0 - 2.0 ** -24])
    # the launch layout: ctr = offset + row carries into the counter's second word; the key is (seed lo, seed hi)
    r = philox_rows(0xA4093822299F31D0, (0x85A308D3 << 32) + 0x243F6A88 - 1, 2, word2=0x13198A2E)
    assert r.shape == (2, 4)
    r1 = philox4x32_10(np.array([0x243F6A88, 0x85A308D3, 0x13198A2E, 0], np.uint32),
                       np.array([0x299F31D0, 0xA4093822], np.uint32))
    assert np.array_equal(r[1], r1)
    r = philox_rows(1, 0xFFFFFFFF, 2)
    assert np.array_equal(r[1], philox4x32_10(np.array([0, 1, 0, 0], np.uint32), np.array([1, 0], np.uint32)))


def test_policy_and_value_forward(golden):
    g = golden("policy")
    pol, val = _params(g, "pol"), _params(g, "val")
    obs = torch.from_numpy(g["obs"])
    probs = O.policy_probs(pol, obs)
    assert torch.allclose(probs, torch.from_numpy(g["probs"]), rtol=1e-5, atol=1e-7)
    lp = O.action_logprob(pol, obs, torch.from_numpy(g["actions"]))
    assert torch.allclose(lp, torch.from_numpy(g["logp"]), rtol=1e-5, atol=1e-6)
    v, _ = O.mlp_forward(val, obs)
    assert torch.allclose(v, torch.from_numpy(g["values"]), rtol=1e-5, atol=1e-6)
    assert torch.allclose(lp, torch.from_numpy(g["bp_logp"]).flatten(), rtol=1e-5, atol=1e-6)
    # inverse-CDF sampler contract: u -> first index whose cumulative mass exceeds u
    u = torch.tensor([0.0, 0.55, 0.999999])
    p = torch.tensor([[0.2, 0.3, 0.5]] * 3)
    assert O.sample_inverse_cdf(p, u).tolist() == [0, 2, 2]


def test_ppo_learn_matches_reference(golden):
    """The analytic backward (SURVEY A.3) + restated clip/Adam reproduce the reference's autograd run."""
    g = golden("ppo_learn")
    obs_dim, n_act, B, mb, epochs, total = [int(x) for x in g["cfg"][:6]]
    plr, clr, clip, ent = g["hyper"]
    buf = O.BufferOracle(1000, 123)
    buf.submit(**{name: g[f"buf.{name}"] for name in O.FIELDS})
    L = O.PPOLearnerOracle(_params(g, "pol0"), _params(g, "val0"), B, epochs, plr, clr, clip, ent, mb)
    grads_seen = []
    orig = L.popt.step

    def spy(params, grads):
        grads_seen.append((L.last_grads[0], L.last_grads[1]))
        return orig(params, grads)

    L.popt.step = spy
    rep = L.learn(buf)
    n_steps = int(g["n_steps"][0])
    assert len(grads_seen) == n_steps == epochs * (total // B)
    for s in range(n_steps):
        for i, gr in enumerate(grads_seen[s][0]):
            ref = torch.from_numpy(g[f"pgrad{s}.{i}"])
            assert ((gr - ref).norm() / ref.norm()) < 2e-5, ("pgrad", s, i)
        for i, gr in enumerate(grads_seen[s][1]):
            ref = torch.from_numpy(g[f"vgrad{s}.{i}"])
            assert ((gr - ref).norm() / ref.norm()) < 2e-5, ("vgrad", s, i)
    for i, p in enumerate(L.pol):
        assert torch.allclose(p, torch.from_numpy(g[f"pol1.{i}"]), rtol=0, atol=2e-6), ("pol", i)
    for i, p in enumerate(L.val):
        assert torch.allclose(p, torch.from_numpy(g[f"val1.{i}"]), rtol=0, atol=2e-6), ("val", i)
    for i in range(len(L.pol)):
        assert torch.allclose(L.popt.m[i], torch.from_numpy(g[f"padam.{i}.m"]), rtol=1e-3, atol=1e-9)
        assert torch.allclose(L.popt.v[i], torch.from_numpy(g[f"padam.{i}.v"]), rtol=1e-3, atol=1e-12)
    assert L.popt.step_count == g["padam.step"][0]
    ref_rep = dict(zip(g["report.keys"], g["report.vals"]))
    for k, v in rep.items():
        assert abs(v - ref_rep[k]) <= 1e-4 * max(abs(ref_rep[k]), 1.0), (k, v, ref_rep[k])
    assert ref_rep["SB3 Clip Fraction"] > 0.2  # the fixture really exercises the clip


def test_add_new_experience(golden):
    g = golden("add_exp")
    val = _params(g, "val")
    buf = O.BufferOracle(int(g["cfg"][2]), 123)
    st = O.WelfordOracle(1)
    for it in range(2):
        exp = tuple(g[f"it{it}.{n}"] for n in ("states", "actions", "log_probs", "rewards", "next_states", "dones",
                                               "truncated"))
        assert np.array_equal(st.get_std(), g[f"it{it}.std_before"])
        O.add_new_experience(val, buf, st, exp, 0.99, 0.95)
        mean, m2, cnt = g[f"it{it}.stats"]
        assert abs(st.mean[0] - mean) <= 1e-6 * max(abs(mean), 1) and abs(st.m2[0] - m2) <= 1e-5 * max(abs(m2), 1)
        assert st.count == cnt
        assert buf.f["rewards"].shape[0] == g[f"it{it}.buf.len"][0]
        assert np.allclose(buf.f["values"], g[f"it{it}.buf.values"], rtol=1e-5, atol=1e-5)
        assert np.allclose(buf.f["advantages"], g[f"it{it}.buf.advantages"], rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("tag,ptype", [("md", 1), ("ct", 2)])
def test_other_heads_match_reference(golden, tag, ptype):
    """MultiDiscreteFF / ContinuousPolicy (SURVEY.md 8(f)-4, the next rows of the hot path): the restated heads and
    their analytic backward reproduce the reference's get_backprop_data and a full PPOLearner.learn (autograd)."""
    g = golden("heads")
    obs_dim, B, mb, epochs, total, n_cont = [int(x) for x in g["cfg"][:6]]
    plr, clr, clip, ent, vmin, vmax = g["hyper"]
    pol0, val0 = _params(g, f"{tag}.pol0"), _params(g, f"{tag}.val0")
    # get_backprop_data on the first minibatch of the rollout
    obs = torch.from_numpy(g[f"{tag}.buf.states"][:mb])
    acts = torch.from_numpy(g[f"{tag}.buf.actions"][:mb])
    z, _ = O.mlp_forward(pol0, obs)
    head = O.head_multi_discrete(z, acts) if ptype == 1 else O.head_continuous(z, acts, vmin, vmax)
    assert torch.allclose(head[0], torch.from_numpy(g[f"{tag}.bp_logp"]), rtol=1e-5, atol=1e-5)
    assert abs(float(head[1]) - float(g[f"{tag}.bp_entropy"][0])) < 1e-5
    # PPOLearner.learn
    buf = O.BufferOracle(1000, 123)
    buf.submit(**{name: g[f"{tag}.buf.{name}"] for name in O.FIELDS})
    L = O.PPOLearnerOracle(pol0, val0, B, epochs, plr, clr, clip, ent, mb, policy_type=ptype, var_range=(vmin, vmax))
    grads_seen = []
    orig = L.popt.step

    def spy(params, grads):
        grads_seen.append((L.last_grads[0], L.last_grads[1]))
        return orig(params, grads)

    L.popt.step = spy
    rep = L.learn(buf)
    n_steps = int(g[f"{tag}.n_steps"][0])
    assert len(grads_seen) == n_steps == epochs * (total // B)
    for s in range(n_steps):
        for i, gr in enumerate(grads_seen[s][0]):
            ref = torch.from_numpy(g[f"{tag}.pgrad{s}.{i}"])
            assert ((gr - ref).norm() / ref.norm()) < 2e-5, ("pgrad", s, i, float((gr - ref).norm() / ref.norm()))
        for i, gr in enumerate(grads_seen[s][1]):
            ref = torch.from_numpy(g[f"{tag}.vgrad{s}.{i}"])
            assert ((gr - ref).norm() / ref.norm()) < 2e-5, ("vgrad", s, i)
    for i, p in enumerate(L.pol):
        assert torch.allclose(p, torch.from_numpy(g[f"{tag}.pol1.{i}"]), rtol=0, atol=2e-6), ("pol", i)
    for i, p in enumerate(L.val):
        assert torch.allclose(p, torch.from_numpy(g[f"{tag}.val1.{i}"]), rtol=0, atol=2e-6), ("val", i)
    ref_rep = dict(zip(g[f"{tag}.report.keys"], g[f"{tag}.report.vals"]))
    for k, v in rep.items():
        assert abs(v - ref_rep[k]) <= 1e-4 * max(abs(ref_rep[k]), 1.0), (k, v, ref_rep[k])
    assert ref_rep["SB3 Clip Fraction"] > 0.2


def test_flatten_rollout_matches_reference(golden):
    """SURVEY.md 8(a) a-4: the restated flattening equals what the reference's own collect_timesteps produced for
    scripted rollouts (tests/golden/make_golden_collect.py), value for value."""
    g = golden("collect")
    for case in g["cases"]:
        ins = [g[f"{case}.in.{k}"] for k in ("obs", "acts", "logp", "rew", "done", "trunc")]
        got = O.flatten_rollout(*ins, [int(a) for a in g[f"{case}.agents"]])
        assert got[0].shape[0] == int(g[f"{case}.n"][0])
        for arr, k in zip(got, ("states", "actions", "log_probs", "rewards", "next_states", "dones", "truncated")):
            want = g[f"{case}.out.{k}"]
            assert arr.shape == want.shape, (case, k, arr.shape, want.shape)
            assert np.array_equal(arr.astype(np.float64), want.astype(np.float64)), (case, k)
