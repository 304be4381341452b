"""GPU tests, kernel level: the whole-network fused kernels (mlp_fused.cu + fused_epilogue.inc) called directly through
rlgym_ppo_b200.ops with rlppo_fused_net descriptors built from test-owned tensors, checked stage by stage against fp64
references (computed on the device in float64).

Every reference starts from the kernel's own STORED bf16 input to that stage (x, H_{l-1}, dz, dH_{l+1}), so the bf16
rounding of one stage does not propagate into the next stage's check and every bound is per element.  Where a stage's
input is not stored (the value net's last hidden activation; every activation of the inference launches) the reference
carries an interval: each bf16 activation the kernel can have produced lies in [RN(lo), RN(hi)] (RN = bf16
round-to-nearest, monotone, so the interval follows from the fp32 error bound of the pre-activation).

Accumulation error of a tensor-core GEMM (bf16 x bf16 products are exact in fp32, sums in fp32), element (i, j):
    e_ij = (sqrt(K) + 2) u (sum_k |a_ik w_jk| + |b_j|),   u = 2^-24.
The worst case K u (sum) could not tell a bias that is one Adam step stale (3e-4) from rounding at K = 256.  The rounding
errors of a sum whose terms have random signs add like a random walk of partial sums far smaller than sum |a w|; sqrt(K) u
sum |a w| bounds it with a wide margin (the same estimate test_split_kernels_gpu.py uses), + 2u for the bias add and the
final rounding.  Each test prints the largest error it implies, in units of e ("H excess"): the distance from the fp64
value to the set of reals that round to the stored bf16 value, over e.

Measured on an NVIDIA B200 (1000 W power limit), largest over every shape as a fraction of each bound: H 0.105,
dH 0.354, dz 0.933 (its bound's 2^-8 |dz| term is the bf16 rounding itself), logp_out 0.042, values_out 0.691, gw_head
0.95 (M = 1: the value tail's one ambiguous activation sits at an end of its interval).  These maxima, and the file's
18 s run time there, were taken when the file also re-ran the duo shapes in the single-tile form and in a CTA-pair
variant of it that the library no longer has.  wgrad_multi's dW and db, per element against (sqrt(M) + 2) u of their
sums of magnitudes (check_wgrad), came to at most 0.704 of that bound on the same GPU and power limit: the policy
head's dW (90 x 256, duo 256x3 net) at M = 129, at an element whose 129 terms dz H are almost all of one sign
(|sum t| / sum |t| = 0.985: H >= 0 after the ReLU, and that logit's dz column keeps its sign).  Same-signed terms make
the partial sums grow to sum |t|, so every fp32 rounding is a fraction of the whole sum and the random walk of them
comes near the sqrt(M) u sum |t| estimate; random-signed terms keep the partial sums near sqrt(M) |t| (the random
operands of test_bf16_gemm_gpu.py reach 0.0085 on the same kernel).  The policy heads' dW at M = 127..129 give the
largest values (0.46 to 0.70); the column sums db at most 0.116.  The atomicAdd order moves only the last few
roundings (three row splits at M = 129).

Layout edges the harness sets up on purpose:
  - x has a row stride past in_dim, and 2 rows past M; both are NaN.  They are outside the x tensor map.
  - each forward weight wq[l] has NaN columns past K (outside the weight map).
  - the policy head's rows n_actions .. pad8(n_actions) ARE inside its map: they hold finite non-zero values.  No output
    may depend on them (the epilogue gives those logit columns a -1e30 bias and a zero d(logit)); every check below
    uses only rows [0, n_actions) of the head weights, so a dependence would fail it.
  - h / dh / dz have ld >= width + 8 and M + 130 rows, filled with the bf16 NaN 0x7FC1; logp_out / values_out have
    M + 1 floats; every gbias[l] the kernels must not write is an f32 NaN sentinel.  gw_head and the value net's
    gbias[n_hidden] start non-zero (accumulation).  The value net's h[n_hidden - 1] is NULL (never stored).

Weight and bias gradients: ops.wgrad_multi is enqueued on the fused outputs right after the fused launch, with no
synchronisation in between (as ppo_learner does), so the PDL hand-off between the two launches is under test too.

Launch forms (test ids start with the form the rule of duo_ok in mlp_fused.cu selects from the nets' shapes):
  duo    -- fused_duo_kernel: CTA pairs, two tiles in flight per CTA (training, widths 128/256, <= 3 layers);
  single -- fused_mlp_kernel<TRAIN>: one tile per CTA (training with other widths or 4 layers; every inference launch).

Every stage check has a negative control on the same data that must fail its bound.

Run with `pytest -m gpu` on a B200."""
import math

import pytest
import torch

from oracle import ref_oracle as O
from parity_helpers import philox_rows, philox_uniform
from test_split_kernels_gpu import _prob_bound, gemm_err

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
U = 2.0 ** -24
SENTINEL = 0x7FC1            # bf16 NaN
F32_SENTINEL = 0x7FC00ABC    # f32 NaN
CLIP, ENT = 0.2, 0.01
STALE = 3e-4                 # one Adam step at lr = 3e-4: the size of a stale-parameter read


@pytest.fixture(scope="module")
def ops():
    from rlgym_ppo_b200 import _lib, ops as _ops
    _lib.require_device()
    return _ops


# ------------------------------------------------------------------------------------------------------------
# harness
# ------------------------------------------------------------------------------------------------------------
def pad8(n):
    return (int(n) + 7) // 8 * 8


def form(*hiddens):
    """The training launch form mlp_fused.cu picks for these nets (duo_ok)."""
    if all(w in (128, 256) for h in hiddens for w in h) and all(len(h) <= 3 for h in hiddens):
        return "duo"
    return "single"


def sentinel(rows, cols):
    return torch.full((rows, cols), SENTINEL, dtype=torch.int16, device=DEV).view(torch.bfloat16)


def f32_sentinel(n):
    return torch.full((n,), F32_SENTINEL, dtype=torch.int32, device=DEV).view(torch.float32)


def bits(t):
    return t.view(torch.int16) if t.dtype == torch.bfloat16 else t.view(torch.int32)


def _down32(x):
    f = x.float()
    return torch.where(f.double() > x, torch.nextafter(f, torch.full_like(f, -math.inf)), f)


def _up32(x):
    f = x.float()
    return torch.where(f.double() < x, torch.nextafter(f, torch.full_like(f, math.inf)), f)


def rn_lo(x):
    """The least bf16 value an fp32 number >= x can round to (as fp64)."""
    return _down32(x).bfloat16().double()


def rn_hi(x):
    return _up32(x).bfloat16().double()


def in_rounding_interval(s, lo, hi):
    sv = s.double()
    return (sv >= rn_lo(lo)) & (sv <= rn_hi(hi))


def gemm_e(a, w, b=None):
    """e of module docstring for a [M, K] @ w^T [K, N] (+ b)."""
    K = a.shape[1]
    absum = a.abs() @ w.abs().t()
    if b is not None:
        absum = absum + b.abs()
    return (math.sqrt(K) + 2) * U * absum


def excess(s, z, e):
    """Largest accumulation error the stored bf16 values s imply, in units of e: distance from z to the reals that
    round to s (half a bf16 ulp either side), over e."""
    sv = s.double()
    _, ex = torch.frexp(sv)
    hu = torch.where(sv == 0, torch.zeros_like(sv), torch.ldexp(torch.ones_like(sv), ex - 9))
    d = torch.maximum((sv - hu) - z, z - (sv + hu)).clamp_min(0)
    return float((d / (e + 1e-300)).max()) if d.numel() else 0.0


class Net:
    """Parameters of one net: bf16 forward operands wq[l] [N, pad8(K) + 8] (NaN past K), the policy head's rows
    pad8(n_actions) (finite non-zero past n_actions), f32 biases, the value head's f32 w_head.  Scales keep every
    activation ~0.4 (bf16 steps ~1e-3 and below, so a 3e-4 bias error moves roundings) and logits ~1."""

    def __init__(self, in_dim, hidden, n_out, policy, seed):
        g = torch.Generator().manual_seed(seed)
        self.in_dim, self.hidden, self.policy, self.L = in_dim, tuple(hidden), policy, len(hidden)
        self.A = n_out if policy else 1
        dims = [in_dim] + list(hidden)
        self.W, self.wq, self.bias = [], [], []
        for l in range(self.L):
            K, N = dims[l], dims[l + 1]
            w = (torch.randn(N, K, generator=g) * ((0.4 if l == 0 else 1.5) / math.sqrt(K))).bfloat16()
            self._add_w(w, N, K)
            self.bias.append((torch.randn(N, generator=g) * 0.05).to(DEV))
        K = hidden[-1]
        if policy:
            rows = pad8(self.A)
            w = (torch.randn(rows, K, generator=g) * 0.5).bfloat16()       # rows past n_actions: finite, non-zero
            w[:self.A] = (torch.randn(self.A, K, generator=g) * (4.0 / math.sqrt(K))).bfloat16()
            self._add_w(w, rows, K)
            self.W[-1] = self.W[-1][:self.A]
            self.bias.append((torch.randn(self.A, generator=g) * 0.1).to(DEV))
        else:
            self.w_head = (torch.randn(K, generator=g) * (1.5 / math.sqrt(K))).to(DEV)
            self.bias.append(torch.tensor([0.3], device=DEV))

    def _add_w(self, w, rows, K):
        buf = torch.full((rows, pad8(K) + 8), float("nan"), dtype=torch.bfloat16)
        buf[:, :K] = w
        self.wq.append(buf.to(DEV))
        self.W.append(w.double().to(DEV))

    def b(self, l):
        """fp64 copy of the bias the device holds NOW (a parameter update may have rewritten it)."""
        return self.bias[l].double()

    def struct(self, x_ld, outs=None):
        from rlgym_ppo_b200 import _lib
        s = _lib.FusedNet()
        s.n_hidden, s.in_dim, s.in_ld = self.L, self.in_dim, x_ld
        for i, h in enumerate(self.hidden):
            s.hidden[i] = h
        for i, w in enumerate(self.wq):
            s.wq[i], s.wq_ld[i] = w.data_ptr(), w.stride(0)
        for i, b in enumerate(self.bias):
            s.bias[i] = b.data_ptr()
        if outs is not None:
            for i, gb in enumerate(outs.gbias):
                s.gbias[i] = gb.data_ptr()
            for l in range(self.L):
                if outs.h[l] is not None:
                    s.h[l], s.h_ld[l] = outs.h[l].data_ptr(), outs.h[l].stride(0)
                s.dh[l], s.dh_ld[l] = outs.dh[l].data_ptr(), outs.dh[l].stride(0)
            if self.policy:
                s.dz, s.dz_ld = outs.dz.data_ptr(), outs.dz.stride(0)
        return s


class Outs:
    """Training outputs of one net, sentinel-filled (see the module docstring)."""

    def __init__(self, net, M):
        R = M + 130
        self.h = [None if (not net.policy and l == net.L - 1) else sentinel(R, w + 8) for l, w in enumerate(net.hidden)]
        self.dh = [sentinel(R, w + 8) for w in net.hidden]
        self.dz = sentinel(R, pad8(net.A) + 8) if net.policy else None
        self.gbias = [f32_sentinel(w) for w in net.hidden] + [f32_sentinel(net.A) if net.policy else
                                                              torch.full((1,), 0.5, device=DEV)]
        if not net.policy:
            self.gw0 = 0.25 + 0.01 * torch.arange(net.hidden[-1], dtype=torch.float32, device=DEV)
            self.gw_head = self.gw0.clone()


class Rows:
    """Per-row inputs and outputs of a training launch."""

    def __init__(self, M, A, seed):
        g = torch.Generator().manual_seed(seed)
        self.M, self.inv = M, 1.0 / M
        self.acts = torch.randint(0, A, (M,), generator=g).float().to(DEV)
        self.old = (-math.log(A) + 0.5 * torch.randn(M, generator=g)).to(DEV)
        self.adv = (0.5 * torch.randn(M, generator=g)).to(DEV)
        self.targets = (0.3 * torch.randn(M, generator=g)).to(DEV)
        self.metrics = torch.zeros(8, device=DEV)
        self.logp = f32_sentinel(M + 1)
        self.values = f32_sentinel(M + 1)


def make_x(M, in_dim, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.full((M + 2, pad8(in_dim) + 8), float("nan"), dtype=torch.bfloat16)
    x[:M, :in_dim] = torch.randn(M, in_dim, generator=g).bfloat16()
    return x.to(DEV)


def wgrad_items(net, outs, x, M):
    """(dy, x, dW, N, K, db) per Linear, as Stack.fused_wgrad_items; dW / db start at zero."""
    z = lambda *s: torch.zeros(*s, device=DEV)  # noqa: E731
    L, items = net.L, []
    if net.policy:
        items.append((outs.dz, outs.h[L - 1], z(net.A, net.hidden[-1]), net.A, net.hidden[-1], z(net.A)))
    for l in range(L - 1, -1, -1):
        inp = outs.h[l - 1] if l > 0 else x
        K = net.hidden[l - 1] if l > 0 else net.in_dim
        items.append((outs.dh[l], inp, z(net.hidden[l], K), net.hidden[l], K, z(net.hidden[l])))
    return items


def launch_train(ops, nets, x, M, d):
    """One fused training launch ((policy, outs), (value, outs), or both in one launch), then wgrad_multi on its outputs
    with no synchronisation in between.  Returns the wgrad items."""
    by = {n.policy: (n, o) for n, o in nets}
    items = []
    if len(nets) == 2:
        (pn, po), (vn, vo) = by[True], by[False]
        ops.policy_value_train_fused(pn.struct(x.stride(0), po), vn.struct(x.stride(0), vo), x, M, pn.A, d.acts, d.old,
                                     d.adv, d.inv, CLIP, ENT, vn.w_head, d.targets, vo.gw_head, d.metrics,
                                     logp_out=d.logp, values_out=d.values)
    elif True in by:
        pn, po = by[True]
        ops.policy_train_fused(pn.struct(x.stride(0), po), x, M, pn.A, d.acts, d.old, d.adv, d.inv, CLIP, ENT,
                               d.metrics, logp_out=d.logp)
    else:
        vn, vo = by[False]
        ops.value_train_fused(vn.struct(x.stride(0), vo), x, M, vn.w_head, d.targets, d.inv, vo.gw_head, d.metrics,
                              values_out=d.values)
    for n, o in nets:
        items += wgrad_items(n, o, x, M)
    ops.wgrad_multi(items, M)
    return items


def chain_terms(M):
    """Length of the longest fp32 summation chain of a per-launch sum over rows (metrics, head gradients): a running
    sum per thread over the tiles it handles, a 5-level warp tree, then per warp a shared or global atomic add (at most
    8 epilogue warps per tile, 148 CTAs)."""
    tiles = (M + 127) // 128
    return 8 * tiles + 8 + 148


# ------------------------------------------------------------------------------------------------------------
# stage checks
# ------------------------------------------------------------------------------------------------------------
def _ppo_reference(z64, acts, old, adv, B_total, clip=CLIP, ent_coef=ENT):
    """test_split_kernels_gpu._ppo_reference, also returning d(loss)/d(softmax) (the g of the dz bound)."""
    zt = z64.clone().requires_grad_(True)
    s = torch.softmax(zt, -1)
    s.retain_grad()
    p = s.clamp(1e-11, 1.0)
    lpa = torch.log(p)
    lp = lpa.gather(-1, acts.long().view(-1, 1)).flatten()
    ent = -(lpa * p).sum(-1)
    ratio = torch.exp(lp - old.double())
    surr = torch.min(ratio * adv.double(), ratio.clamp(1 - clip, 1 + clip) * adv.double())
    loss = (-surr.sum() - ent_coef * ent.sum()) / B_total
    loss.backward()
    kl = (ratio - 1) - (lp - old.double())
    clipped = ((ratio - 1).abs() > clip).double()
    return zt.grad, s.grad, lp.detach(), ent.detach(), kl.detach(), clipped, surr.detach(), ratio.detach()


def check_hidden(net, outs, x, M, rec):
    """H_l, every stored hidden layer: the stored bf16 value is the rounding of a value within e of fp64
    relu(A Wq_l^T + b_l), A = x (layer 0) or the stored H_{l-1}; bit-zero where the pre-activation is below -e.
    Control: the same check against b_l + 3e-4 fails.  Returns the stored activations (fp64) and the value tail's
    pre-activation interval."""
    A = x[:M, :net.in_dim].double()
    Hs, worst = [], 0.0
    for l in range(net.L):
        z = A @ net.W[l].t() + net.b(l)
        e = gemm_e(A, net.W[l], net.b(l))
        if outs.h[l] is None:       # the value net's last activation: not stored
            Hs.append(None)
            rec["H excess"] = worst
            return Hs, (z, e), A
        s = outs.h[l][:M, :net.hidden[l]]
        ok = in_rounding_interval(s, (z - e).clamp_min(0), (z + e).clamp_min(0))
        assert bool(ok.all()), f"H{l}: {int((~ok).sum())} of {ok.numel()} elements outside the bound"
        assert bool((bits(s)[(z + e) < 0] == 0).all()), f"H{l}: a negative pre-activation stored as non-zero"
        ctl = in_rounding_interval(s, (z + STALE - e).clamp_min(0), (z + STALE + e).clamp_min(0))
        assert not bool(ctl.all()), f"H{l}: control (bias + {STALE}) passed"
        worst = max(worst, excess(s, z.clamp_min(0), e))
        A = s.double()
        Hs.append(A)
    rec["H excess"] = worst
    return Hs, None, A


def check_dgrad(s, dy, W, mask, wrong_mask, what, rec):
    """dH = (dy W) (.) mask: unmasked entries the rounding of a value within e of fp64; masked entries bit-zero.
    Control: the same stored dH against wrong_mask fails."""
    r = dy @ W
    e = gemm_e(dy, W.t())

    def ok_with(m):
        return torch.where(m, in_rounding_interval(s, r - e, r + e), bits(s) == 0)

    ok = ok_with(mask)
    assert bool(ok.all()), f"{what}: {int((~ok).sum())} of {ok.numel()} elements outside the bound"
    if float(r.abs().max()) == 0.0:         # a one-action head with an exactly zero dz: any mask fits
        assert bool((s == 0).all())
        return
    assert not bool(ok_with(wrong_mask).all()), f"{what}: control (wrong ReLU mask) passed"
    rec["dH excess"] = max(rec.get("dH excess", 0.0), excess(s[mask], r[mask], e[mask]))


def wrong_mask(Hs, l):
    """The ReLU mask of another hidden layer of the same width, else this layer's mask shifted by one column."""
    for k in range(len(Hs)):
        if k != l and Hs[k] is not None and Hs[k].shape == Hs[l].shape:
            return Hs[k] > 0
    return torch.roll(Hs[l] > 0, 1, dims=1)


def check_policy(net, outs, x, M, d, rec):
    """Every stage of a policy training launch; see the docstrings of the helpers and of test_fused_train."""
    L, A, K = net.L, net.A, net.hidden[-1]
    Hs, _, Hl = check_hidden(net, outs, x, M, rec)
    # ---- head: dz, logp_out, metrics [0..4] ----
    Wh, bh = net.W[L], net.b(L)
    z = Hl @ Wh.t() + bh
    ze = gemm_e(Hl, Wh, bh)
    inv32 = float(torch.tensor(d.inv, dtype=torch.float32))
    dz_ref, g_s, lp, ent, kl, clipped, surr, ratio = _ppo_reference(z, d.acts, d.old, d.adv, 1.0 / inv32)
    eps = _prob_bound(z, ze * 2.0 ** 22, A)                            # [M, 1]; logit error 2 * max_j e_j
    lp_tol = eps.flatten() + 2 * 2.0 ** -23 * lp.abs().clamp_min(1.0)
    got_lp = d.logp[:M].double()
    assert bool(((got_lp - lp).abs() <= lp_tol).all()), float(((got_lp - lp).abs() / lp_tol).max())
    rec["logp err / bound"] = float(((got_lp - lp).abs() / lp_tol).max())
    if A > 1:   # control: the odd-numbered head biases off by 3e-4
        zc = z + STALE * (torch.arange(A, device=DEV) % 2).double()
        lpc = torch.log_softmax(zc, -1).gather(-1, d.acts.long().view(-1, 1)).flatten()
        assert not bool(((got_lp - lpc).abs() <= lp_tol).all()), "logp control passed"
    else:
        assert bool((got_lp == 0).all())
    # dz, per element (rows whose ratio sits within its error of 1 +- clip are left out: the branch may go either way)
    dzs = outs.dz[:M, :pad8(A)]
    # padding columns: zero; -0.0 where the entropy factor is negative (the padding's s_j = __expf(-1e30) = 0 times it)
    assert bool((dzs[:, A:] == 0).all()), "dz padding columns must be zero"
    got = dzs[:, :A].double()
    edge = (((ratio - 1).abs() - CLIP).abs() <= 2 * (lp_tol + 8 * U) * ratio) | (d.adv == 0)
    assert int(edge.sum()) <= M // 50 + 2
    s64 = torch.softmax(z, -1)
    cw = ENT * inv32
    E = 2 * eps + 2.0 ** -21 + lp_tol[:, None] + (A + 4) * U
    scale = g_s.abs().max(-1, keepdim=True).values + (g_s.abs() * s64).sum(-1, keepdim=True) + cw
    bound = 4 * E * s64 * scale + 2.0 ** -8 * dz_ref.abs() + 2.0 ** -125 * scale + 2.0 ** -134 + 3e-10 * cw

    def dz_ok(ref):
        return ((got - ref).abs() <= bound)[~edge]

    ok = dz_ok(dz_ref)
    assert bool(ok.all()), f"dz: {int((~ok).sum())} elements outside the bound, worst {float(((got - dz_ref).abs() / bound)[~edge].max()):.3g}"
    rec["dz err / bound"] = float(((got - dz_ref).abs() / bound)[~edge].max()) if bool((~edge).any()) else 0.0
    if A > 1:   # control: the last two rows swapped (M >= 2), else the wrong action
        if M >= 2:
            perm = torch.arange(M, device=DEV)
            perm[[M - 1, M - 2]] = perm[[M - 2, M - 1]]
            zc, ac, oc, vc = z[perm], d.acts[perm], d.old[perm], d.adv[perm]
        else:
            zc, ac, oc, vc = z, (d.acts + 1) % A, d.old, d.adv
        dz_c = _ppo_reference(zc, ac, oc, vc, 1.0 / inv32)[0]
        assert not bool(dz_ok(dz_c).all()), "dz control passed"
    # metrics [0..4]: sums over rows of per-row values good to the bounds above, plus the fp32 summation chain
    m = d.metrics.double()
    ch = chain_terms(M) * U
    assert float(m[4]) == M
    e0 = float(((2 * eps.flatten() + 2.0 ** -21) * (1 + ent)).sum()) + ch * float(ent.sum())
    assert abs(float(m[0]) - float(ent.sum())) <= e0, (float(m[0]), float(ent.sum()), e0)
    e1 = float((lp_tol * (ratio + 1) + 4 * U * ((ratio - 1).abs() + (lp - d.old.double()).abs())).sum()) + ch * float(kl.abs().sum())
    assert abs(float(m[1]) - float(kl.sum())) <= e1, (float(m[1]), float(kl.sum()), e1)
    assert abs(float(m[2]) - float(clipped.sum())) <= int(edge.sum())
    e3 = float((d.adv.double().abs() * ratio * (lp_tol + 4 * U)).sum()) + ch * float(surr.abs().sum())
    assert abs(float(m[3]) - float(surr.sum())) <= e3, (float(m[3]), float(surr.sum()), e3)
    # ---- backward data path ----
    dy = got_dz = dzs[:, :A].double()
    check_dgrad(outs.dh[L - 1][:M, :K], got_dz, Wh, Hs[L - 1] > 0, wrong_mask(Hs, L - 1), f"dH{L - 1}", rec)
    for l in range(L - 1, 0, -1):
        dy = outs.dh[l][:M, :net.hidden[l]].double()
        check_dgrad(outs.dh[l - 1][:M, :net.hidden[l - 1]], dy, net.W[l], Hs[l - 1] > 0, wrong_mask(Hs, l - 1),
                    f"dH{l - 1}", rec)


def value_tail(net, z, e):
    """The value net's last hidden activation is not stored: each element is bf16 lo or hi (its rounding interval;
    lo == hi for all but ~1% of them, whose pre-activation lies within e of a rounding boundary).  v = sum H w_head + b
    then takes one of the values base + sum_{c ambiguous} b_c (hi_c - lo_c) w_c, b_c in {0, 1}: candidates enumerated
    over the 6 largest such terms of each row, the rest added to the tolerance.  v's accumulation: per thread 4 fma
    chains of N/8 terms, two pairwise adds, the two halves of the row and + b: N/8 + 5 roundings of partial sums below
    sum |H w| + |b|.  Returns lo, hi, candidates [M, 64], tolerance [M]."""
    lo, hi = rn_lo((z - e).clamp_min(0)), rn_hi((z + e).clamp_min(0))
    w, b = net.w_head.double(), net.b(net.L)
    t = (hi - lo) * w
    top = t.abs().topk(6, dim=1)
    combos = torch.tensor([[(i >> j) & 1 for j in range(6)] for i in range(64)], dtype=torch.float64, device=DEV)
    cand = (lo @ w + b)[:, None] + t.gather(1, top.indices) @ combos.t()
    tol = t.abs().sum(1) - top.values.sum(1) + (net.hidden[-1] / 8 + 5) * U * (hi @ w.abs() + b.abs())
    return lo, hi, cand, tol


def v_err(got, cand, tol):
    """Per row: distance from got to the nearest candidate, over the tolerance."""
    return (got[:, None] - cand).abs().min(1).values / tol


def check_value(net, outs, x, M, d, rec):
    """Every stage of a value training launch.
      values_out: within value_tail's tolerance of one of its candidates; control: b_head + 3e-4.
      dv = 2 inv (v - t) is recomputed in fp32 from the stored values_out (the kernel's own dv).  dH_{L-1} =
        bf16(fp32(dv w_head)) masked by the tail's ReLU: bit-exact where the tail activation is surely positive, bit-zero
        where surely zero, one of the two where its rounding interval contains 0.  Control: the mask shifted one column.
      gw_head += sum_rows dv bf16(H_L): within sum |dv| (hi - lo) / 2 plus the summation chain.
      gbias[n_hidden] += sum dv, metrics[5] = sum (v - t)^2, metrics[6] = M: within the summation chain."""
    L, N = net.L, net.hidden[-1]
    Hs, (z, e), _ = check_hidden(net, outs, x, M, rec)
    lo, hi, cand, tol = value_tail(net, z, e)
    got = d.values[:M].double()
    r = v_err(got, cand, tol)
    assert bool((r <= 1).all()), float(r.max())
    rec["v err / bound"] = float(r.max())
    assert not bool((v_err(got - STALE, cand, tol) <= 1).all()), "values control (b_head + 3e-4) passed"
    t = d.targets
    err32 = d.values[:M] - t
    dv32 = (2 * torch.tensor(d.inv, dtype=torch.float32, device=DEV)) * err32
    dvw = (dv32[:, None] * net.w_head[None, :]).bfloat16()
    s = outs.dh[L - 1][:M, :N]

    def ok_with(pos, zero):
        return torch.where(pos, bits(s) == bits(dvw),
                           torch.where(zero, bits(s) == 0, (bits(s) == 0) | (bits(s) == bits(dvw))))

    ok = ok_with(lo > 0, hi == 0)
    assert bool(ok.all()), f"value dH{L - 1}: {int((~ok).sum())} elements differ"
    assert not bool(ok_with(torch.roll(lo > 0, 1, 1), torch.roll(hi == 0, 1, 1)).all()), "value dH control passed"
    ch = chain_terms(M) * U
    dv = dv32.double()
    gw_ref = outs.gw0.double() + dv @ ((lo + hi) / 2)
    gw_b = dv.abs() @ ((hi - lo) / 2) + ch * (dv.abs() @ hi + outs.gw0.double().abs())
    gw = outs.gw_head.double()
    assert bool(((gw - gw_ref).abs() <= gw_b).all()), float(((gw - gw_ref).abs() / gw_b).max())
    rec["gw_head err / bound"] = float(((gw - gw_ref).abs() / gw_b).max())
    gb = float(outs.gbias[L])
    assert abs(gb - (0.5 + float(dv.sum()))) <= ch * (float(dv.abs().sum()) + 0.5)
    m = d.metrics.double()
    sq = float((err32.double() ** 2).sum())
    assert float(m[6]) == M
    assert abs(float(m[5]) - sq) <= (ch + 2 * U) * sq
    for l in range(L - 1, 0, -1):
        dy = outs.dh[l][:M, :net.hidden[l]].double()
        check_dgrad(outs.dh[l - 1][:M, :net.hidden[l - 1]], dy, net.W[l], Hs[l - 1] > 0, wrong_mask(Hs, l - 1),
                    f"value dH{l - 1}", rec)


def check_untouched(net, outs, M, d):
    """Rows >= M and the columns past each width keep the sentinel; logp_out[M], values_out[M] and the gbias entries
    the kernels must not write too."""
    bufs = [(h, w) for h, w in zip(outs.h, net.hidden) if h is not None] + list(zip(outs.dh, net.hidden))
    if net.policy:
        bufs.append((outs.dz, pad8(net.A)))
    for buf, w in bufs:
        b = bits(buf)
        assert bool((b[M:] == SENTINEL).all()), "write past row M"
        assert bool((b[:M, w:] == SENTINEL).all()), "write into the row-stride padding"
    for gb in (outs.gbias if net.policy else outs.gbias[:net.L]):
        assert bool((bits(gb) == F32_SENTINEL).all()), "a bias gradient the fused kernels must leave alone was written"
    assert int(bits(d.logp)[M]) == F32_SENTINEL and int(bits(d.values)[M]) == F32_SENTINEL
    if net.policy:
        assert not bool(bits(d.logp[:M]).eq(F32_SENTINEL).any())


def check_wgrad(items, M, rec):
    """rlppo_wgrad_multi on the stored fused outputs: dW = dy^T x and db = column sums of dy against the fp64
    contraction of the same stored bf16 operands, per element: |dW - ref| <= (sqrt(M) + 2) u sum_m |dy x| (the module
    docstring's e with the contraction over M rows; gemm_err), db likewise with sum_m |dy|.  Control: the reference
    without the rows of the 128-row tile holding row M / 2 (a kernel that skipped one tile) fails it."""
    bound = (math.sqrt(M) + 2) * U
    t0 = (M // 2) // 128 * 128
    keep = torch.ones(M, dtype=torch.bool, device=DEV)
    keep[t0:t0 + 128] = False
    for dy, x, dw, N, K, db in items:
        a, b = dy[:M, :N].double(), x[:M, :K].double()
        ref, ref_db = a.t() @ b, a.sum(0)
        if float(ref.abs().max()) == 0.0:        # a one-action head: dz is identically zero
            assert float(dw.abs().max()) == 0.0 and float(db.abs().max()) == 0.0
            continue
        absum = a.abs().t() @ b.abs() + 1e-300   # (+ 1e-300: an entry with no terms must come out exactly zero)
        e_w = gemm_err(dw.double(), ref, absum) / bound
        e_b = gemm_err(db.double(), ref_db, a.abs().sum(0) + 1e-300) / bound
        assert e_w <= 1.0 and e_b <= 1.0, (N, K, e_w, e_b)
        assert gemm_err(dw.double(), a[keep].t() @ b[keep], absum) > bound, "wgrad control passed"
        rec["wgrad"] = max(rec.get("wgrad", 0.0), e_w, e_b)


def run_and_check(ops, nets, x, M, d, tag):
    items = launch_train(ops, nets, x, M, d)
    torch.cuda.synchronize()
    rec = {}
    for net, outs in nets:
        r = {}
        (check_policy if net.policy else check_value)(net, outs, x, M, d, r)
        check_untouched(net, outs, M, d)
        rec["policy" if net.policy else "value"] = r
    w = {}
    check_wgrad(items, M, w)
    rec["wgrad"] = w
    print(f"{tag}: " + "; ".join(f"{k} " + ", ".join(f"{n} {v:.3g}" for n, v in r.items()) for k, r in rec.items()))
    return rec


# ------------------------------------------------------------------------------------------------------------
# training launches
# ------------------------------------------------------------------------------------------------------------
BENCH = ((256, 256, 256), 89, 90)
TRAIN_CASES = ([BENCH + (M,) for M in (1, 127, 128, 129, 257, 20480, 49999, 50000)] + [
    ((128,), 20, 7, 1100),
    ((128, 256, 128), 256, 128, 1100),
    ((256, 128), 64, 1, 1100),                   # one action: dz is identically zero
    ((128, 128), 89, 65, 1100),                  # out_kb = 2, the second k-block partial
    ((64, 64), 89, 90, 129),
    ((64, 64), 89, 90, 1100),
    ((256, 192, 128, 64), 200, 128, 1100),       # obs > 128: a 2-stage weight ring in the single-tile kernel
    ((192,), 256, 1, 1100),
    ((64, 256), 1, 16, 1100),
])


def _tid(hidden, obs, A, M):
    return f"{form(hidden)}-h{'x'.join(map(str, hidden))}-obs{obs}-A{A}-M{M}"


@pytest.mark.parametrize("hidden,obs,A,M", TRAIN_CASES, ids=[_tid(*c) for c in TRAIN_CASES])
def test_fused_train(ops, hidden, obs, A, M):
    """rlppo_policy_train_fused and rlppo_value_train_fused on the same hidden layers, each followed by wgrad_multi.

    dz bound, per element: dz_j = s_j (g_j - G), g = d(loss)/d(softmax), G = sum_k g_k s_k.  The logits carry e
    (module docstring), so s is good to eps relative (_prob_bound with logit error 2 max_j e_j) and log p to
    lp_tol = eps + 2^-22 max(1, |log p|).  g_a = d_logp / p_a carries the ratio's and p_a's errors, the entropy part
    cw (log s_j + 1) eps + 2^-21 (__logf): |dg| <= E scale, E = 2 eps + 2^-21 + lp_tol + (A + 4) u, scale =
    max|g| + sum |g| s + cw.  With the s_j and G errors, |dz_j - dz64_j| <= 4 E s_j scale + 2^-8 |dz64_j| (bf16 output)
    + 2^-125 scale + 2^-134 (range floors, see test_policy_head_backward_subsets) + 3e-10 cw (the kernel keeps the
    entropy gradient where s_j < 1e-11; the reference's clamp drops it).  Rows whose ratio lies within its error of
    1 +- clip are left out of the dz check (the clip branch can go either way), at most M / 50 + 2 of them.
    Metrics: the per-row errors above summed, plus chain_terms(M) u of the sums.
    Measured on a B200: dz at most 0.933 of its bound, logp_out 0.042, H 0.105 e, dH 0.354 e (module docstring)."""
    pnet = Net(obs, hidden, A, True, 100 + M)
    vnet = Net(obs, hidden, 1, False, 200 + M)
    x = make_x(M, obs, 300 + M)
    for net in (pnet, vnet):
        d = Rows(M, A, 400 + M)
        run_and_check(ops, [(net, Outs(net, M))], x, M, d, f"{_tid(hidden, obs, A, M)} {'policy' if net.policy else 'value'}")


JOINT_CASES = [(((256, 256, 256), (128,), 89, 90), M) for M in (129, 640, 50000)] + [
    (((64, 64), (256, 192, 128, 64), 89, 90), 1100)]


def _jid(c, M):
    ph, vh, obs, A = c
    return f"{form(ph, vh)}-p{'x'.join(map(str, ph))}-v{'x'.join(map(str, vh))}-M{M}"


@pytest.mark.parametrize("case,M", JOINT_CASES, ids=[_jid(*c) for c in JOINT_CASES])
def test_fused_train_joint(ops, case, M):
    """rlppo_policy_value_train_fused with two different nets (one launch whose CTAs run phase lists of different
    lengths side by side; at M = 129 one cluster runs a policy tile beside a value tile): every per-net check of
    test_fused_train on each net, and the per-row outputs (stored H / dH / dz with their padding, logp_out,
    values_out) bit-identical to the two single-net launches of the same form.  Only the atomically summed outputs
    (metrics, gw_head, gbias) may differ between the two."""
    ph, vh, obs, A = case
    assert form(ph, vh) == form(ph) == form(vh)
    pnet, vnet = Net(obs, ph, A, True, 500 + M), Net(obs, vh, 1, False, 600 + M)
    x = make_x(M, obs, 700 + M)
    d = Rows(M, A, 800 + M)
    po, vo = Outs(pnet, M), Outs(vnet, M)
    run_and_check(ops, [(pnet, po), (vnet, vo)], x, M, d, _jid(case, M))
    d1, d2 = Rows(M, A, 800 + M), Rows(M, A, 800 + M)
    po1, vo1 = Outs(pnet, M), Outs(vnet, M)
    launch_train(ops, [(pnet, po1)], x, M, d1)
    launch_train(ops, [(vnet, vo1)], x, M, d2)
    torch.cuda.synchronize()
    for a, b in [(po.dz, po1.dz)] + list(zip(po.h + po.dh, po1.h + po1.dh)) + list(zip(vo.h + vo.dh, vo1.h + vo1.dh)):
        if a is not None:
            assert torch.equal(bits(a), bits(b))
    assert torch.equal(bits(d.logp), bits(d1.logp)) and torch.equal(bits(d.values), bits(d2.values))


def test_fused_train_after_parameter_update(ops):
    """The learner's order: an optimiser launch (rlppo_norm_clip_adam) rewrites the biases and w_head in a flat arena,
    and the fused training launch follows on the same stream with no synchronisation (a PDL launch: its prologue
    overlaps the optimiser).  lr = 1e-2 moves every parameter by ~1e-2 (Adam's first step is lr sign(g)), 30x the
    3e-4 shift each stage's control already shows to fail: outputs computed from stale biases or w_head fail by a
    wide margin.  Every stage is checked against references built from the UPDATED parameters."""
    M = 1100
    pnet, vnet = Net(89, (256, 256, 256), 90, True, 900), Net(89, (128,), 1, False, 901)
    pieces = pnet.bias + vnet.bias + [vnet.w_head]
    sizes = [p.numel() for p in pieces]
    arena = torch.cat([p.float() for p in pieces])
    offs = [0]
    for n in sizes:
        offs.append(offs[-1] + n)
    views = [arena[offs[i]:offs[i + 1]] for i in range(len(pieces))]
    npb = len(pnet.bias)
    pnet.bias, vnet.bias, vnet.w_head = views[:npb], views[npb:-1], views[-1]
    g = torch.Generator().manual_seed(902)
    grads = ((torch.randint(0, 2, (offs[-1],), generator=g) * 2 - 1) * (0.5 + torch.rand(offs[-1], generator=g))).to(DEV)
    m, v = torch.zeros_like(arena), torch.zeros_like(arena)
    lr = torch.full((2,), 1e-2, device=DEV)
    step = torch.zeros(2, dtype=torch.int64, device=DEV)
    sq = torch.zeros(2, device=DEV)
    seg = [0, offs[npb], offs[-1]]
    x = make_x(M, 89, 903)
    d = Rows(M, 90, 904)
    po, vo = Outs(pnet, M), Outs(vnet, M)
    before = arena.clone()
    torch.cuda.synchronize()
    ops.norm_clip_adam(arena, grads, m, v, seg, sq, lr, step, max_norm=1e9)
    run_and_check(ops, [(pnet, po), (vnet, vo)], x, M, d, f"{form((256,) * 3, (128,))} after update")
    assert bool(((arena - before).abs() > 0.9e-2).all())


# ------------------------------------------------------------------------------------------------------------
# inference launches (always the single-tile kernel; nothing but the outputs is stored)
# ------------------------------------------------------------------------------------------------------------
def interval_chain(net, x, M):
    """Interval [lo, hi] holding every bf16 activation of the last hidden layer the kernel can produce: per layer
    z in [lo W+ + hi W- + b - e, hi W+ + lo W- + b + e] (W+ / W- the positive / negative parts, e with hi as the
    activations' magnitude), each end rounded outwards to bf16 after the ReLU."""
    lo = hi = x[:M, :net.in_dim].double()
    for l in range(net.L):
        W, b = net.W[l], net.b(l)
        Wp, Wn = W.clamp_min(0), W.clamp_max(0)
        e = gemm_e(hi, W, b)
        zl = lo @ Wp.t() + hi @ Wn.t() + b - e
        zh = hi @ Wp.t() + lo @ Wn.t() + b + e
        lo, hi = rn_lo(zl.clamp_min(0)), rn_hi(zh.clamp_min(0))
    return lo, hi


def head_interval(net, lo, hi):
    W, b = net.W[net.L], net.b(net.L)
    Wp, Wn = W.clamp_min(0), W.clamp_max(0)
    zl = lo @ Wp.t() + hi @ Wn.t() + b
    zh = hi @ Wp.t() + lo @ Wn.t() + b
    return (zl + zh) / 2, (zh - zl) / 2 + gemm_e(hi, W, b)


INFER_CASES = [BENCH + (M,) for M in (1, 129, 3000)] + [((64, 64), 89, 90, 3000), ((128, 128), 89, 65, 3000),
                                                        ((192,), 256, 1, 129)]


def _iid(hidden, obs, A, M):
    return f"h{'x'.join(map(str, hidden))}-obs{obs}-A{A}-M{M}"


@pytest.mark.parametrize("hidden,obs,A,M", INFER_CASES, ids=[_iid(*c) for c in INFER_CASES])
def test_policy_infer_fused(ops, hidden, obs, A, M):
    """rlppo_policy_infer_fused.  Logits: the midpoint of head_interval, error zerr (half-width + e); probabilities
    within _prob_bound of them.
      injected uniforms: actions against O.sample_inverse_cdf on the fp64 probabilities; a differing row must have
        u * P within its slack (the fp32 CDF's rounding + the probability bound) of a CDF boundary, so the mismatch
        count is bounded by the number of such rows.  The slack follows the logit interval: on the bench shape some
        rows carry logit errors of a few 1e-2 from activations whose rounding is ambiguous, and their share of
        mismatches is larger than the per-layer kernel test's (test_split_kernels_gpu) fixed M / 500.  actions_out ==
        actions_i64_out; logp_out within lp_tol of log clamp(p[a]).  Control: logits with the odd-numbered biases off
        by 3e-4 fail the logp bound (asserted for M > 1: the logit interval of a single row can be as wide as the
        shift, since every activation whose rounding is ambiguous widens the next layer's interval).
      deterministic: the argmax wherever the top-2 gap exceeds 2 zerr, log-prob of the row maximum.
      d_offset: a launch with offset o and a device counter advanced by rlppo_u64_add(c) draws exactly what a launch
        with offset o + c draws, and not what offset o alone draws.
      Philox stream: with seed 0x0123456789ABCDEF and offset + device counter = 2^32 - M/2, the actions and log-probs
        equal those drawn from the host restatement's uniforms (tests/parity_helpers.py), bit for bit.
    Nothing is written at row M.
    Measured on a B200: logp_out at most 0.287 of lp_tol; logit intervals up to 0.094 wide on the bench shape at
    M = 3000, where 16 of 1788 boundary rows sample differently from the fp64 reference (1 of 257 for (64, 64), 4 of 387
    for (128, 128) with 65 actions)."""
    net = Net(obs, hidden, A, True, 1000 + M)
    x = make_x(M, obs, 1100 + M)
    lo, hi = interval_chain(net, x, M)
    z, zerr = head_interval(net, lo, hi)
    eps = _prob_bound(z, zerr * 2.0 ** 22, A)
    p64 = torch.softmax(z, -1)
    u = torch.rand(M, generator=torch.Generator().manual_seed(1200 + M), dtype=torch.float64).float().to(DEV)
    af, a64, lp = f32_sentinel(M + 1), torch.full((M + 1,), -7, dtype=torch.int64, device=DEV), f32_sentinel(M + 1)
    s = net.struct(x.stride(0))
    ops.policy_infer_fused(s, x, M, A, u=u, actions_out=af, actions_i64_out=a64, logp_out=lp)
    torch.cuda.synchronize()
    assert int(a64[M]) == -7 and int(bits(af)[M]) == F32_SENTINEL and int(bits(lp)[M]) == F32_SENTINEL
    a = a64[:M]
    assert torch.equal(af[:M].long(), a) and bool((a >= 0).all()) and bool((a < A).all())
    a_ref = O.sample_inverse_cdf(p64, u.double())
    pc = p64.clamp(1e-11, 1.0)
    cdf = pc.cumsum(-1)
    thr = u.double() * cdf[:, -1]
    slack = (A + 2) * 2.0 ** -23 + eps.flatten()
    diff = (a != a_ref).nonzero().flatten()
    for r in diff.tolist():
        j = min(int(a[r]), int(a_ref[r]))
        assert abs(float(cdf[r, j] - thr[r])) <= float(slack[r]) * float(cdf[r, -1]), (r, int(a[r]), int(a_ref[r]))
    near = ((cdf - thr[:, None]).abs() <= (slack * cdf[:, -1])[:, None]).any(-1)
    assert diff.numel() <= max(2, int(near.sum()))
    lp_ref = torch.log(pc.gather(-1, a.view(-1, 1))).flatten()
    lp_tol = eps.flatten() + 2 * 2.0 ** -23 * lp_ref.abs().clamp_min(1.0)
    got = lp[:M].double()
    assert bool(((got - lp_ref).abs() <= lp_tol).all()), float(((got - lp_ref).abs() / lp_tol).max())
    if A > 1 and M > 1:
        zc = z + STALE * (torch.arange(A, device=DEV) % 2).double()
        lpc = torch.log_softmax(zc, -1).gather(-1, a.view(-1, 1)).flatten()
        assert not bool(((got - lpc).abs() <= lp_tol).all()), "logp control passed"
    print(f"infer {_iid(hidden, obs, A, M)}: {diff.numel()} mismatches of {int(near.sum())} boundary rows, logp err / bound "
          f"{float(((got - lp_ref).abs() / lp_tol).max()):.3g}, max logit error {float(zerr.max()):.3g}")
    # deterministic
    ops.policy_infer_fused(s, x, M, A, deterministic=True, actions_i64_out=a64, logp_out=lp)
    torch.cuda.synchronize()
    top2 = z.topk(min(2, A), -1).values
    clear = (top2[:, 0] - top2[:, -1] > 2 * zerr.max(-1).values) if A > 1 else torch.ones(M, dtype=torch.bool, device=DEV)
    assert torch.equal(a64[:M][clear], z.argmax(-1)[clear])
    lp_det = torch.log(p64.max(-1).values.clamp(1e-11, 1.0))
    tol_det = eps.flatten() + 2 * 2.0 ** -23 * lp_det.abs().clamp_min(1.0)
    assert bool(((lp[:M].double() - lp_det).abs() <= tol_det).all())
    # d_offset
    ctr = torch.zeros(1, dtype=torch.int64, device=DEV)
    ops.u64_add(ctr, 12345)
    out = []
    for off, dev_off in ((1000, ctr), (13345, None), (1000, None)):
        a_, l_ = torch.empty(M, dtype=torch.int64, device=DEV), torch.empty(M, device=DEV)
        ops.policy_infer_fused(s, x, M, A, seed=77, offset=off, offset_dev=dev_off, actions_i64_out=a_, logp_out=l_)
        out.append((a_, l_))
    torch.cuda.synchronize()
    assert int(ctr) == 12345
    assert torch.equal(out[0][0], out[1][0]) and torch.equal(bits(out[0][1]), bits(out[1][1]))
    if A > 1 and M > 1:
        assert not torch.equal(out[0][0], out[2][0])
    # the Philox stream (counter (offset + device offset + row, high word, 0, 0), key (seed lo, seed hi)): a launch whose
    # rows cross the carry into the counter's high word draws exactly what the host restatement's uniforms draw
    seed, first = 0x0123456789ABCDEF, 2 ** 32 - M // 2
    u_host = torch.from_numpy(philox_uniform(philox_rows(seed, first, M)[:, 0])).float().to(DEV)
    draws = []
    for kw in (dict(seed=seed, offset=first - 12345, offset_dev=ctr), dict(u=u_host)):
        a_, l_ = torch.empty(M, dtype=torch.int64, device=DEV), torch.empty(M, device=DEV)
        ops.policy_infer_fused(s, x, M, A, actions_i64_out=a_, logp_out=l_, **kw)
        draws.append((a_, l_))
    torch.cuda.synchronize()
    assert torch.equal(draws[0][0], draws[1][0]) and torch.equal(bits(draws[0][1]), bits(draws[1][1]))


VINFER_CASES = [((256, 256, 256), 89, M) for M in (1, 129, 3000)] + [((128,), 20, 3000), ((64, 64), 89, 3000),
                                                                     ((256, 192, 128, 64), 200, 1100)]


@pytest.mark.parametrize("hidden,obs,M", VINFER_CASES, ids=[_iid(h, o, 1, M) for h, o, M in VINFER_CASES])
def test_value_infer_fused(ops, hidden, obs, M):
    """rlppo_value_infer_fused: values_out within [v_lo - acc, v_hi + acc], v_lo / v_hi from interval_chain's last
    activation and the signs of w_head, acc as value_tail's accumulation term.  Control: b_head + 3e-4 fails it
    (for M > 1, as the logp control of test_policy_infer_fused).
    Where the training launch runs the same (single-tile) form, value_train_fused's values_out equals it bit for bit.
    Measured on a B200: interval half-widths from 4e-4 ((128,), M = 3000) to 0.083 ((256, 192, 128, 64), M = 1100)."""
    net = Net(obs, hidden, 1, False, 1300 + M)
    x = make_x(M, obs, 1400 + M)
    lo, hi = interval_chain(net, x, M)
    w, b = net.w_head.double(), net.b(net.L)
    wp, wn = w.clamp_min(0), w.clamp_max(0)
    acc = (hidden[-1] / 8 + 5) * U * (hi @ w.abs() + b.abs())
    v_lo, v_hi = lo @ wp + hi @ wn + b - acc, hi @ wp + lo @ wn + b + acc
    vals = f32_sentinel(M + 1)
    ops.value_infer_fused(net.struct(x.stride(0)), x, M, net.w_head, vals)
    torch.cuda.synchronize()
    got = vals[:M].double()
    assert int(bits(vals)[M]) == F32_SENTINEL
    assert bool(((got >= v_lo) & (got <= v_hi)).all())
    if M > 1:
        assert not bool(((got >= v_lo + STALE) & (got <= v_hi + STALE)).all()), "values control passed"
    print(f"value infer {_iid(hidden, obs, 1, M)}: max interval half-width {float(((v_hi - v_lo) / 2).max()):.3g}")
    if form(hidden) == "single":
        d = Rows(M, 1, 1500 + M)
        launch_train(ops, [(net, Outs(net, M))], x, M, d)
        torch.cuda.synchronize()
        assert torch.equal(bits(d.values), bits(vals))
