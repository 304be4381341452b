"""The one-GPU optimiser forms of csrc/optim.cu -- rlppo_norm_clip_adam (one launch) and rlppo_grad_sqnorm +
rlppo_clip_adam (two launches; with a zero norm it is FusedAdam.step) -- against a host float64 restatement of
clip_grad_norm_ + torch.optim.Adam's single-tensor step (ppo_learner.py:187-193), launch by launch, and the bf16 GEMM
operands the same launch rewrites against the new fp32 weights.

Reference of one launch, per segment, from the kernel's own fp32 inputs (p0, m0, v0 read back before the launch) and with
the step count t after the launch (coefficients in Python doubles, as torch forms them):
    c  = clamp(max_norm / (sqrt(S) + 1e-6), max=1)        S = the kernel's sum of squares; a NaN propagates
    m1 = b1 m0 + (1 - b1) g c
    v1 = b2 v0 + (1 - b2) (g c)^2
    p1 = p0 - lr / (1 - b1^t) * m1 / (sqrt(v1) / sqrt(1 - b2^t) + eps)     with the KERNEL's m1 and v1
so rounding never compounds over launches.

Bounds, u = 2^-24 (every fp32 operation and every cast of a double coefficient to fp32 errs by at most u relative):
  * c: cast of max_norm, sqrtf, the constant 1e-6f, the add, the divide: 5u relative (all operands positive), and
    g*c adds one rounding: 6u |g c|.
  * m1 = m0 + (g c - m0) * (1 - b1): the difference errs by 6u |g c| + u (|g c| + |m0|), the cast (1 - b1) and the product
    by 2u more of (1 - b1)(|g c| + |m0|), the final add by u |m1| <= u (|m0| + (1 - b1) |g c|):
    |m1 - ref| <= 14u (|m0| + (1 - b1) |g c|).
  * v1 = v0 b2 + (1 - b2) (g c)^2: (g c)^2 carries 12u + u, the cast and two products 3u, the cast of b2 and its product
    2u on b2 v0, the add u; all terms are positive: |v1 - ref| <= 20u (b2 v0 + (1 - b2) (g c)^2).
  * p1 = p0 - s (m1 / d): d = sqrtf(v1) / sqrt(bc2) + eps errs by 4u (sqrtf, the cast of sqrt(bc2), the divide, the
    cast of eps and the add; positive terms), the quotient by u more, the cast of s = lr / bc1 and the product by 2u:
    x = s m1 / d errs by 7u, and the subtraction adds u |p1|: |p1 - ref| <= 10u |x| + 2u |p0|.
    A bias correction formed at t instead of t+1 moves x by (1 - b1^(t+1)) / (1 - b1^t) - 1 (11 % at t = 8): far outside.
  * S: positive terms, so a sum whose longest chain of additions is L errs by at most L u S.  The one-launch norm is
    thread-serial (ceil(n / threads) terms), a 5-level shuffle tree, 8 warps in order, blocks added lane-strided
    (ceil(grid / 32)) and a 5-level tree; grad_sqnorm adds block partials with atomics, up to `grid` in a chain.
Segments at lr 0 must keep p bit for bit.  Boundary elements of every segment are scaled up, so an element counted in its
neighbour's segment moves that segment's sum and coefficient far outside these bounds."""
import contextlib
import io

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
U = 2.0 ** -24
HP_DEFAULT = (0.5, 0.9, 0.999, 1e-8)       # max_norm, beta1, beta2, eps of the learner
STEPS0 = (0, 1, 7, 100_000)                # initial step counts, per segment in turn (100k: a resumed checkpoint)
REGIMES = ("zero", "clipped", "unclipped", "at_norm", "huge")
LAYOUTS = {                                # segment sizes
    "1": [1],
    "5": [5],
    "1023": [1023],
    "1025": [600, 425],
    "dp": [177754, 154881, 8],            # the learner's data-parallel arena: policy | value | 8 metric floats at lr 0
    "empty_first": [0, 700, 325],
    "empty_mid": [512, 0, 511],
    "empty_last": [1000, 25, 0],
    "eight": [3, 0, 4093, 1, 777, 0, 2048, 8],
    "big": None,                          # > 2 * 4 * 1024 * SMs * 4: every thread also runs the loop past its 4 registers
}


@pytest.fixture(scope="module")
def ops():
    from rlgym_ppo_b200 import _lib, ops as _ops
    _lib.require_device()
    return _ops


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def layout(name):
    sizes = LAYOUTS[name]
    if sizes is None:
        n = 2 * 4 * 1024 * sm_count() * 4 + 5
        sizes = [n // 3, n - n // 3]
    return np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)


def base_lrs(seg):
    """Distinct learning rates per segment; the last of >= 3 segments is the learner's lr-0 metric tail."""
    k = len(seg) - 1
    lr = [3e-4 / (1 + 0.7 * j) for j in range(k)]
    if k >= 3:
        lr[-1] = 0.0
    return np.asarray(lr, np.float32)


class State:
    """One optimiser's device state over a flat arena; p, m, v, steps seeded per segment."""

    def __init__(self, seg, seed):
        rng = np.random.default_rng(seed)
        n, k = int(seg[-1]), len(seg) - 1
        steps = np.asarray([STEPS0[j % len(STEPS0)] for j in range(k)], np.int64)
        p = (rng.standard_normal(n) * 0.05).astype(np.float32)
        m = np.zeros(n, np.float32)
        v = np.zeros(n, np.float32)
        for j in range(k):
            s = slice(seg[j], seg[j + 1])
            if steps[j] > 0:      # a resumed state; a fresh segment (step 0) has m = v = 0: eps-dominated denominators
                m[s] = rng.standard_normal(s.stop - s.start) * 1e-3
                v[s] = rng.random(s.stop - s.start) * 1e-6
        self.p, self.m, self.v = (torch.from_numpy(x).to(DEV) for x in (p, m, v))
        self.steps = torch.from_numpy(steps).to(DEV)
        self.lr = torch.zeros(k, dtype=torch.float32, device=DEV)
        self.sq = torch.full((k,), -1.0, dtype=torch.float32, device=DEV)

    def host(self):
        return {a: getattr(self, a).cpu().numpy().copy() for a in ("p", "m", "v", "steps", "sq")}


def make_grads(regime, seg, rng, max_norm):
    """fp32 gradients of one launch.  clipped / unclipped / at_norm set every segment's norm to a distinct multiple of
    max_norm (> 1, < 1, = 1); the first and last element of every segment are 30x the others."""
    n = int(seg[-1])
    g = rng.standard_normal(n)
    if regime == "zero":
        return np.zeros(n, np.float32)
    if regime == "huge":
        return (g * 1e10).astype(np.float32)
    for j in range(len(seg) - 1):
        a, b = int(seg[j]), int(seg[j + 1])
        if a == b:
            continue
        g[a] *= 30
        g[b - 1] *= 30
        f = {"clipped": 2.0 + 1.5 * j, "unclipped": 0.1 + 0.08 * j, "at_norm": 1.0}[regime]
        g[a:b] *= f * max_norm / np.sqrt((g[a:b] ** 2).sum())
    return g.astype(np.float32)


def _close(got, ref, bound, what):
    """Same NaN positions; elsewhere |got - ref| <= bound element-wise."""
    got = got.astype(np.float64)
    nan_ref, nan_got = np.isnan(ref), np.isnan(got)
    assert np.array_equal(nan_ref, nan_got), f"{what}: NaN at {np.flatnonzero(nan_ref != nan_got)[:8]}"
    ok = ~nan_ref
    err = np.abs(got[ok] - ref[ok])
    bad = np.flatnonzero(~(err <= bound[ok]))
    assert bad.size == 0, (f"{what}: {bad.size} elements outside the bound, first at {np.flatnonzero(ok)[bad[0]]}: "
                           f"got {got[ok][bad[0]]!r} want {ref[ok][bad[0]]!r} bound {bound[ok][bad[0]]!r}")


def sum_chain(n, total, form):
    """Longest chain of fp32 additions in the sum of squares of an n-element segment of a `total`-element arena (module
    docstring).  The grid follows the arena: ceil(total / 1024) blocks of 256 threads, at most SMs x (1..4) blocks for the
    one-launch form (its occupancy is not known here) and SMs x 8 for grad_sqnorm."""
    want = max(-(-total // 1024), 1)
    if form == "fused":
        grid_lo, grid_hi = min(want, sm_count()), min(want, 4 * sm_count())
        return -(-n // (256 * grid_lo)) + 1 + 5 + 8 + -(-grid_hi // 32) + 5
    grid = min(want, 8 * sm_count())
    return -(-n // (256 * grid)) + 1 + 5 + 8 + grid


def check_launch(pre, post, g, seg, lr, hp, form):
    """One launch of `form` against the float64 reference (module docstring).  pre / post: State.host() dicts."""
    max_norm, b1, b2, eps = hp
    p0, m0, v0 = (pre[a].astype(np.float64) for a in ("p", "m", "v"))
    S = post["sq"]
    assert np.array_equal(post["steps"], pre["steps"] + 1), (pre["steps"], post["steps"])
    with np.errstate(all="ignore"):
        for k in range(len(seg) - 1):
            s = slice(int(seg[k]), int(seg[k + 1]))
            n = s.stop - s.start
            gk = g[s].astype(np.float64)
            S_ref = float((gk * gk).sum())
            if form != "no_clip":
                if np.isnan(S_ref) or np.isinf(S_ref):
                    assert np.isnan(S[k]) if np.isnan(S_ref) else S[k] == np.inf, (k, S[k], S_ref)
                else:
                    assert abs(float(S[k]) - S_ref) <= sum_chain(n, int(seg[-1]), form) * U * S_ref, (k, float(S[k]), S_ref)
            if n == 0:
                continue
            t = float(post["steps"][k])
            c = np.minimum(max_norm / (np.sqrt(np.float64(S[k])) + 1e-6), 1.0)       # np.minimum keeps a NaN
            gc = gk * c
            _close(post["m"][s], b1 * m0[s] + (1 - b1) * gc, 14 * U * (np.abs(m0[s]) + (1 - b1) * np.abs(gc)), f"m[seg {k}]")
            _close(post["v"][s], b2 * v0[s] + (1 - b2) * gc * gc, 20 * U * (b2 * v0[s] + (1 - b2) * gc * gc), f"v[seg {k}]")
            m1, v1 = post["m"][s].astype(np.float64), post["v"][s].astype(np.float64)
            x = float(lr[k]) / (1 - b1 ** t) * m1 / (np.sqrt(v1) / np.sqrt(1 - b2 ** t) + eps)
            _close(post["p"][s], p0[s] - x, 10 * U * np.abs(x) + 2 * U * np.abs(p0[s]), f"p[seg {k}]")
            if lr[k] == 0:
                fin = ~np.isnan(x)
                assert np.array_equal(post["p"][s][fin].view(np.uint32), pre["p"][s][fin].view(np.uint32)), \
                    f"segment {k} has lr 0 but its weights moved"


def launch(ops, form, st, g, seg, hp, views=None):
    max_norm, b1, b2, eps = hp
    if form == "fused":
        ops.norm_clip_adam(st.p, g, st.m, st.v, seg, st.sq, st.lr, st.steps, max_norm, b1, b2, eps, views=views)
    elif form == "two_launch":
        ops.grad_sqnorm(g, seg, st.sq)
        ops.clip_adam(st.p, g, st.m, st.v, seg, st.sq, st.lr, st.steps, max_norm, b1, b2, eps, views=views)
    else:      # "no_clip": FusedAdam.step's call, a zero norm (coefficient 1)
        st.sq.zero_()
        ops.clip_adam(st.p, g, st.m, st.v, seg, st.sq, st.lr, st.steps, max_norm, b1, b2, eps, views=views)


# ---- bf16 operand views ------------------------------------------------------------------------------------
SENTINEL = int(torch.tensor([-77.0], dtype=torch.bfloat16).view(torch.int16).item())
GUARD = 1 << 18      # sentinel elements after every operand buffer: a misplaced store stays inside the pool and shows


def pad8(n):
    return (n + 7) // 8 * 8


class Operands:
    """bf16 operand buffers of a list of Linears (out_f, in_f, offset in the arena, has W^T) carved from one sentinel-filled
    pool, wq [pad8(out), pad8(in)] and wt [pad8(in), pad8(out)], each followed by a guard; `order` lists the views."""

    def __init__(self, linears, order):
        self.linears = linears
        self.blocks = []
        at = 0
        for out_f, in_f, off, has_wt in linears:
            wq = (at, pad8(in_f))
            at += pad8(out_f) * pad8(in_f) + GUARD
            wt = None
            if has_wt:
                wt = (at, pad8(out_f))
                at += pad8(in_f) * pad8(out_f) + GUARD
            self.blocks.append((wq, wt))
        self.pool = torch.full((at,), SENTINEL, dtype=torch.int16, device=DEV)
        from rlgym_ppo_b200 import _lib
        views = []
        base = self.pool.data_ptr()
        for q in order:
            (out_f, in_f, off, _), (wq, wt) = linears[q], self.blocks[q]
            v = _lib.Bf16View()
            v.offset, v.out_f, v.in_f = off, out_f, in_f
            v.wq, v.wq_ld = base + 2 * wq[0], wq[1]
            v.wt, v.wt_ld = (None, 0) if wt is None else (base + 2 * wt[0], wt[1])
            views.append(v)
        self.views = (_lib.Bf16View * len(views))(*views)

    def check(self, p):
        """Every view's blocks hold bf16(p) bit for bit (a NaN weight: some NaN); everything else is still the sentinel."""
        want = np.full(self.pool.numel(), SENTINEL, np.int16)
        is_nan = np.zeros(self.pool.numel(), bool)
        for (out_f, in_f, off, _), (wq, wt) in zip(self.linears, self.blocks):
            w = p[off:off + out_f * in_f].reshape(out_f, in_f)
            wb = torch.from_numpy(w.copy()).to(torch.bfloat16).view(torch.int16).numpy()
            for (at, ld), blk, nan in [(wq, wb, np.isnan(w))] + ([] if wt is None else [(wt, wb.T, np.isnan(w).T)]):
                idx = at + np.arange(blk.shape[0])[:, None] * ld + np.arange(blk.shape[1])[None, :]
                want[idx] = blk
                is_nan[idx] = nan
        got = self.pool.cpu().numpy()
        got_nan = ((got & 0x7F80) == 0x7F80) & ((got & 0x7F) != 0)
        assert np.all(got_nan[is_nan]), "a NaN weight's bf16 operand is not NaN"
        bad = np.flatnonzero((got != want) & ~is_nan)
        assert bad.size == 0, f"{bad.size} operand elements wrong, first at pool index {bad[0]}: {got[bad[0]]} != {want[bad[0]]}"


def run_sequence(ops, form, seg, hp=HP_DEFAULT, regimes=REGIMES, seed=0, operands=None, edit=None):
    """Launches of `form`, one per regime, each checked against the reference; the per-segment lr changes every launch.
    `edit(i, g)` may alter the gradients of launch i.  Returns the device snapshots after every launch."""
    st = State(seg, seed)
    rng = np.random.default_rng(seed + 1)
    lr0 = base_lrs(seg)
    snaps = []
    for i, regime in enumerate(regimes):
        lr = (lr0 * (1.0 + 0.37 * i)).astype(np.float32)
        st.lr.copy_(torch.from_numpy(lr))
        g = make_grads(regime, seg, rng, hp[0])
        if edit is not None:
            edit(i, g)
        pre = st.host()
        launch(ops, form, st, torch.from_numpy(g).to(DEV), seg, hp, None if operands is None else operands.views)
        torch.cuda.synchronize()
        post = st.host()
        check_launch(pre, post, g, seg, lr, hp, form)
        if operands is not None:
            operands.check(post["p"])
        snaps.append(post)
    return snaps


def assert_same_bits(a, b):
    for x, y in zip(a, b):
        for key in x:
            assert np.array_equal(np.ascontiguousarray(x[key]).view(np.uint8), np.ascontiguousarray(y[key]).view(np.uint8)), \
                f"{key} differs between two runs of the same launches"


# ---- the update ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(LAYOUTS))
@pytest.mark.parametrize("form", ["fused", "two_launch"])
def test_optimiser_launch_vs_fp64(ops, form, name):
    """Every layout, every gradient regime, step counts 0 / 1 / 7 / 100k, lr changed between launches; the one-launch
    form is bit-identical from run to run."""
    seg = layout(name)
    snaps = run_sequence(ops, form, seg)
    if form == "fused":
        assert_same_bits(snaps, run_sequence(ops, form, seg))


@pytest.mark.parametrize("hp", [(2.0, 0.0, 0.0, 1e-6), (0.05, 0.5, 0.95, 1e-3), (1.0, 0.9, 0.999, 1e-8)])
@pytest.mark.parametrize("form", ["fused", "two_launch", "no_clip"])
def test_optimiser_hyperparameters(ops, form, hp):
    """Non-default max_norm, betas (0 included) and eps, which FusedAdam.step passes from param_groups; "no_clip" is
    FusedAdam.step's own call (a zero norm)."""
    for name in ("dp", "eight"):
        run_sequence(ops, form, layout(name), hp=hp, seed=3)


@pytest.mark.parametrize("form", ["fused", "two_launch"])
def test_nan_gradient_poisons_its_segment(ops, form):
    """torch: a NaN in a segment's gradient makes clip_grad_norm_ return NaN, clamp keeps it, and every gradient, moment
    and weight of that segment turns NaN; the other segments update as usual."""
    seg = layout("dp")
    nan_at = int(seg[1]) + 12345

    def edit(i, g):
        if i == 1:
            g[nan_at] = np.nan
    snaps = run_sequence(ops, form, seg, regimes=("clipped", "clipped", "unclipped"), edit=edit)
    for post in snaps[1:]:
        for key in ("p", "m", "v"):
            x = post[key]
            assert np.isnan(x[seg[1]:seg[2]]).all(), f"{key}: the NaN segment is not NaN throughout"
            assert not np.isnan(x[:seg[1]]).any() and not np.isnan(x[seg[2]:]).any(), f"{key}: NaN outside its segment"


@pytest.mark.parametrize("form", ["fused", "two_launch"])
def test_inf_gradient_zeroes_its_segment(ops, form):
    """torch: an inf gradient makes the norm inf and the coefficient 0: the inf entries become NaN (inf * 0), the finite
    gradients of that segment count as zero, the other segments update as usual."""
    seg = layout("dp")
    at = [5, 177000]

    def edit(i, g):
        if i == 0:
            g[at[0]], g[at[1]] = np.inf, -np.inf
    snaps = run_sequence(ops, form, seg, regimes=("clipped", "unclipped"), edit=edit)
    p = snaps[0]["p"]
    assert np.isnan(p[at]).all() and np.isnan(p).sum() == 2


def test_nine_segments_refused(ops):
    from rlgym_ppo_b200._lib import RlppoError
    seg = np.arange(10, dtype=np.int64) * 4
    st = State(seg, 0)
    steps = st.steps.clone()
    for form in ("fused", "two_launch"):
        with pytest.raises(RlppoError):
            launch(ops, form, st, torch.zeros(int(seg[-1]), device=DEV), seg, HP_DEFAULT)
    torch.cuda.synchronize()
    assert torch.equal(st.steps, steps)


# ---- bf16 operand refresh --------------------------------------------------------------------------------------
def arena(segments):
    """segments: per segment, a list of Linears (out_f, in_f, has W^T), each taking out*in weights then out biases, and
    plain floats (an int: that many) that no view covers.  Returns (segment offsets, [(out_f, in_f, offset, has_wt)])."""
    seg, lin, at = [0], [], 0
    for items in segments:
        for it in items:
            if isinstance(it, int):
                at += it
                continue
            out_f, in_f, has_wt = it
            lin.append((out_f, in_f, at, has_wt))
            at += out_f * in_f + out_f
        seg.append(at)
    return np.asarray(seg, np.int64), lin


TINY = [(1, 1, True), (3, 5, True), (5, 3, False), (2, 7, True), (1, 4, True), (7, 2, True), (4, 1, False), (3, 3, True)]
VIEW_CONFIGS = {
    # the 16-view maximum, 1 x 1 to 7 x 2, 50 floats apart: a thread's elements (256 apart) lie in different views
    "tiny16": [[x for t in TINY for x in (t, 50)], [x for t in TINY[::-1] for x in (t, 50)]],
    # 89 x 300 and 300 x 89 with padded leading dimensions, W^T missing for some, then the lr-0 metric tail
    "wide": [[(300, 89, True), (89, 300, True), (1, 89, False)], [(300, 89, False), (89, 300, True), (1, 89, True)], [8]],
}


@pytest.mark.parametrize("config", list(VIEW_CONFIGS))
@pytest.mark.parametrize("form", ["fused", "two_launch", "no_clip"])
def test_operand_views_refreshed(ops, form, config):
    """After every launch wq[:out, :in] and wt[:in, :out] are bf16 of the new weights bit for bit (views listed out of
    arena order; the last launch has a NaN gradient in the second segment, whose operands must then be NaN); padding,
    guards and the W^T buffers of views without one keep their sentinel."""
    seg, lin = arena(VIEW_CONFIGS[config])
    order = [int(q) for q in np.random.default_rng(7).permutation(len(lin))]
    operands = Operands(lin, order)

    def edit(i, g):
        if i == 2:
            g[int(seg[1]) + 1] = np.nan
    run_sequence(ops, form, seg, regimes=("clipped", "unclipped", "clipped"), operands=operands, edit=edit, seed=11)


def test_seventeen_views_refused(ops):
    from rlgym_ppo_b200._lib import RlppoError
    seg, lin = arena([TINY + TINY + TINY[:1]])
    operands = Operands(lin, list(range(17)))
    st = State(seg, 0)
    steps = st.steps.clone()
    for form in ("fused", "two_launch"):
        with pytest.raises(RlppoError):
            launch(ops, form, st, torch.zeros(int(seg[-1]), device=DEV), seg, HP_DEFAULT, operands.views)
    torch.cuda.synchronize()
    assert torch.equal(st.steps, steps) and bool((operands.pool == SENTINEL).all())


# ---- the learner's operands after a step ------------------------------------------------------------------------
def _buffer(n, dev, obs=89, act=90):
    from rlgym_ppo_b200.ppo import ExperienceBuffer
    r = np.random.RandomState(3)
    b = ExperienceBuffer(n, 11, dev)
    b.submit_experience(r.randn(n, obs).astype(np.float32), r.randint(0, act, n).astype(np.float32),
                        (-4.5 + 0.3 * r.randn(n)).astype(np.float32), r.randn(n).astype(np.float32),
                        r.randn(n, obs).astype(np.float32), np.zeros(n, np.float32), np.zeros(n),
                        r.randn(n).astype(np.float32), r.randn(n).astype(np.float32))
    return b


def _assert_operands_fresh(ops, lrn):
    for net in (lrn.policy, lrn.value_net):
        st = net._stack
        for i in range(len(st.linears)):
            wq = torch.zeros_like(st.wq[i])
            wt = None if st.wt[i] is None or not st.need_wt else torch.zeros_like(st.wt[i])
            ops.weight_to_bf16(st.w[i], wq, wt)
            torch.cuda.synchronize()
            assert torch.equal(st.wq[i].view(torch.int16), wq.view(torch.int16)), f"wq[{i}] is stale"
            if wt is not None:
                assert torch.equal(st.wt[i].view(torch.int16), wt.view(torch.int16)), f"wt[{i}] is stale"


@pytest.mark.parametrize("widths", [(256, 256), (300, 100)])
def test_learner_operands_equal_weights(ops, widths):
    """bf16 mode: after PPOLearner.learn (the optimiser launch refreshes the operands) and after FusedAdam.step (a
    separate refresh), every Linear's wq, and wt where the layer-wise kernels read it, is weight_to_bf16 of its weight."""
    from rlgym_ppo_b200.ppo import PPOLearner
    torch.manual_seed(5)
    B = 1024
    with contextlib.redirect_stdout(io.StringIO()):
        lrn = PPOLearner(89, 90, 0, widths, widths, (0.1, 1.0), B, 2, 3e-4, 3e-4, 0.2, 0.01, B // 2, DEV,
                         precision="bf16")
    fused = lrn.policy._stack.fused_ok and lrn.value_net._stack.fused_ok
    assert fused == (widths == (256, 256))
    before = lrn._params.clone()
    lrn.learn(_buffer(2 * B, DEV))
    torch.cuda.synchronize()
    assert not torch.equal(before, lrn._params)
    assert lrn.policy._stack.need_wt == (not fused)
    _assert_operands_fresh(ops, lrn)
    for opt in (lrn.policy_optimizer, lrn.value_optimizer):
        opt.step()
    _assert_operands_fresh(ops, lrn)
