"""GPU tests, kernel level: the "fp32" precision mode's split-operand kernels and the autograd head backward kernels,
called directly through rlgym_ppo_b200.ops and compared with fp64 references on the CPU.

Split layout (rlppo_split in include/rlppo.h): an f32 matrix is stored as `parts` bf16 matrices side by side, part q in
columns [q * pstride, q * pstride + cols), value = part0 + part1 + part2.  The references are computed in fp64 from the
f32 master values, never from the bf16 parts, so a kernel that splits, schedules or reassembles parts wrongly shows up as
a precision loss.

Error measure of the GEMMs: e = max_ij |y_ij - y64_ij| / (sum_k |x_ik w_jk| + |b_j|), the error of an inner product in
units of its own magnitude; it scales with the accumulation and survives cancellation.  u = 2^-24 (fp32 unit roundoff).

Test operands for the GEMMs ("tailed" values): every element is s * 2^e * (1 + a/128) + 2^e * (127 * 2^-15 + 63 * 2^-23)
with a in [1, 4).  Its parts are exactly the bf16 head, then +0.99 * 2^-8 and +0.49 * 2^-16 relative to 2^e: both tails
are positive whatever the sign s.  One operand of every GEMM has random signs (the sums cancel, so fp32 accumulation error
stays small) and the other is positive.  Of the products a GEMM must not drop (part_i x part_j, i + j = order - 1), those
whose random-signed factor is a tail all have one sign: part1 x part1 and (positive operand's part 0) x part2 in the
forward (the third, part2 of the positive operand x part 0 of the random one, takes that operand's random sign and
cancels), part1 x part0 in the backward.  A kernel that drops them is then off by a deterministic ~1.4 * 2^-16
(forward) or ~2^-8 (backward) in e, not by a random walk that could hide below the tolerance.  Each GEMM test runs the
same data with one order less and asserts that this run fails the bound.

Run with `pytest -m gpu` on a B200."""
import itertools
import math

import numpy as np
import pytest
import torch

from oracle import ref_oracle as O
from parity_helpers import DEV, SENTINEL, bits, philox_rows, philox_uniform, recon, sentinel, split_rows

pytestmark = pytest.mark.gpu

U = 2.0 ** -24


@pytest.fixture(scope="module")
def ops():
    from rlgym_ppo_b200 import _lib, ops as _ops
    _lib.require_device()
    return _ops


# ------------------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------------------
TAIL = 127 * 2.0 ** -15 + 63 * 2.0 ** -23


def tailed(shape, seed, positive, device="cpu"):
    """The GEMM test operands described in the module docstring, generated in f32 (every step is exact)."""
    g = torch.Generator(device=device).manual_seed(seed)
    e = torch.randint(-2, 1, shape, generator=g, device=device).float()
    a = torch.randint(1, 4, shape, generator=g, device=device).float()
    s = 1.0 if positive else torch.randint(0, 2, shape, generator=g, device=device).float() * 2 - 1
    return (s * (1 + a / 128) + TAIL) * torch.exp2(e)


def gemm_err(y, ref, absum):
    return float(((y - ref).abs() / absum).max())


def split_weight(ops, w, q_parts, q_pstride, out_rows, t_parts=0, t_pstride=0, in_rows=0):
    wq = torch.zeros((out_rows, q_parts * q_pstride), dtype=torch.bfloat16, device=DEV)
    wt = torch.zeros((in_rows, t_parts * t_pstride), dtype=torch.bfloat16, device=DEV) if t_parts else None
    ops.weight_split(w.to(DEV).contiguous(), wq, q_parts, q_pstride, wt, t_parts, t_pstride)
    return wq, wt


def sample_rows(M):
    """All rows of small GEMMs; for large ones ~300 rows spread over every 128-row tile region plus the last tile."""
    if M <= 1024:
        return torch.arange(M)
    return torch.tensor(sorted(set(range(0, M, M // 300)) | set(range(M - 130, M))))


def rel_l2(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float((a - b).norm() / max(float(b.norm()), 1e-300))


# ------------------------------------------------------------------------------------------------------------
# 1. operand preparation
# ------------------------------------------------------------------------------------------------------------
def _special_values():
    """f32 values over exponents 2^-100 .. 2^100, +-0, and values whose splits hit round-to-nearest-even ties:
    low 16 bits 0x8000 (part 0 is a tie), 0x0101 (part 1 is a tie), and a few other low patterns."""
    g = torch.Generator().manual_seed(0)
    n = 1 << 16
    e = torch.randint(-100, 101, (n,), generator=g)
    m = torch.randint(0, 1 << 23, (n,), generator=g)
    s = torch.randint(0, 2, (n,), generator=g)
    spread = ((s << 31) | ((e + 127) << 23) | m).to(torch.int32)
    hi = torch.randint(0, 1 << 16, (7, 2048), generator=g).to(torch.int32)   # random sign and top significand bits,
    hi = (hi & 0xC03F) | 0x1F00                                               # exponent 2^-65 or 2^63
    lows = torch.tensor([0x8000, 0x0101, 0x8080, 0x7F80, 0xFFFF, 0x0001, 0x0080], dtype=torch.int32)[:, None]
    ties = ((hi << 16) | lows).flatten()
    zeros = torch.tensor([0x00000000, -0x80000000], dtype=torch.int64).to(torch.int32)
    return torch.cat([spread, ties, zeros]).view(torch.float32)


def test_rows_split_reconstruction_exact(ops):
    """Three parts carry 3 x 8 = 24 significand bits: part0 + part1 + part2 (fp64) equals the f32 input exactly.

    Limits, found by sweeping the exponent (and reproduced below):
      - exact for 2^-110 <= |x|; below that the last part would need bits under bf16's smallest subnormal step
        (2^-133), and the reconstruction error is at most 2^-134 (half that step) -- absolute, not relative;
      - the sign of zero is carried by part 0 only: for x = -0.0, part 0 is bf16 -0.0 and x - part0 = +0.0, so the parts
        sum to +0.0.  The only consumer that looks at a zero's sign, the dgrad ReLU mask, reads part 0;
      - |x| >= 2^128 * (1 - 2^-9) would round to a bf16 infinity in part 0 (values of that size are not tested)."""
    x = _special_values()
    width = 1000
    n = (x.numel() + width - 1) // width
    xp = torch.zeros(n * width)
    xp[:x.numel()] = x
    src = xp.view(n, width)
    ps = ops.pad64(width)
    buf = sentinel(n + 2, 3 * ps + 64)
    ops.rows_split(src.to(DEV), buf, 3, ps)
    torch.cuda.synchronize()
    r = recon(buf, 3, ps, width, rows=slice(0, n))
    want = src.double()
    nz = want != 0
    assert torch.equal(r[nz], want[nz])
    assert bool((r[~nz] == 0).all())
    p0 = buf[:n, :width].cpu()
    assert torch.equal(torch.signbit(p0.float())[~nz], torch.signbit(src)[~nz])     # -0.0 keeps its sign in part 0
    # nothing written past the parts or below the rows
    assert bool((bits(buf[:n, 3 * ps:]) == SENTINEL).all()) and bool((bits(buf[n:]) == SENTINEL).all())
    # padding columns of every part are zero
    for q in range(3):
        assert bool((bits(buf[:n, q * ps + width:(q + 1) * ps]) == 0).all())

    # the subnormal end: exact from 2^-110 up, within 2^-134 below
    g = torch.Generator().manual_seed(1)
    rows = []
    for ex in range(-135, -100):
        m = torch.randint(0, 1 << 23, (512,), generator=g).to(torch.int32)
        rows.append(((m | ((ex + 127) << 23)) if ex >= -126 else (m >> (-126 - ex))).view(torch.float32))
    sub = torch.stack(rows)
    buf = torch.zeros((sub.shape[0], 3 * 512), dtype=torch.bfloat16, device=DEV)
    ops.rows_split(sub.to(DEV), buf, 3, 512)
    r = recon(buf, 3, 512, 512)
    err = (r - sub.double()).abs()
    assert float(err.max()) <= 2.0 ** -134
    exact_from = 135 - 110
    assert float(err[exact_from:].max()) == 0.0
    assert float(err[exact_from - 1].max()) > 0.0        # the limit is where it is claimed to be


def test_rows_split_two_parts_error(ops):
    """Two parts: |part0 + part1 - x| <= 2^-16 |x| (each bf16 rounding leaves at most 2^-8 of what it rounds)."""
    x = _special_values()
    x = x[x != 0]
    width = 512
    n = x.numel() // width
    src = x[:n * width].view(n, width)
    buf = sentinel(n, 2 * width)
    ops.rows_split(src.to(DEV), buf, 2, width)
    r = recon(buf, 2, width, width)
    rel = ((r - src.double()).abs() / src.double().abs()).max()
    assert float(rel) <= 2.0 ** -16, float(rel)


@pytest.mark.parametrize("out_f,in_f", [(90, 89), (256, 256), (21, 256), (1024, 2048)])
def test_weight_split_parts_padding_transpose(ops, out_f, in_f):
    """W -> 3-part W [out_rows, 3 * pad64(in)] and 2-part W^T [in_rows, 2 * pad64(out)]: the parts reconstruct W exactly,
    padding rows and columns of every part are zero (the next GEMM's k loop and TMA boxes read them), and W^T's parts
    are the transposes of W's."""
    w = tailed((out_f, in_f), 7, positive=False) * torch.randn(out_f, in_f, generator=torch.Generator().manual_seed(8))
    qs, ts = ops.pad64(in_f), ops.pad64(out_f)
    out_rows, in_rows = ops.pad8(out_f), ops.pad8(in_f)
    wq = sentinel(out_rows + 8, 3 * qs + 64)
    wt = sentinel(in_rows + 8, 2 * ts + 64)
    ops.weight_split(w.to(DEV), wq[:out_rows], 3, qs, wt[:in_rows], 2, ts)
    torch.cuda.synchronize()
    wq_c, wt_c = wq.cpu(), wt.cpu()
    assert torch.equal(recon(wq_c[:out_f], 3, qs, in_f), w.double())
    assert float((recon(wt_c[:in_f], 2, ts, out_f) - w.t().double()).abs().max()) <= 2.0 ** -16 * float(w.abs().max())
    for q in range(3):
        part = bits(wq_c[:out_rows, q * qs:(q + 1) * qs])
        assert bool((part[:, in_f:] == 0).all()) and bool((part[out_f:] == 0).all())
    for q in range(2):
        part = bits(wt_c[:in_rows, q * ts:(q + 1) * ts])
        assert bool((part[:, out_f:] == 0).all()) and bool((part[in_f:] == 0).all())
        # W^T part q == (W part q)^T over the common padded extent
        wq_q = bits(wq_c[:out_rows, q * qs:(q + 1) * qs])
        n_o, n_i = min(out_rows, ts), min(in_rows, qs)
        assert torch.equal(part[:n_i, :n_o], wq_q[:n_o, :n_i].t())
    # beyond the declared extents nothing was written
    assert bool((bits(wq_c[out_rows:]) == SENTINEL).all()) and bool((bits(wq_c[:, 3 * qs:]) == SENTINEL).all())
    assert bool((bits(wt_c[in_rows:]) == SENTINEL).all()) and bool((bits(wt_c[:, 2 * ts:]) == SENTINEL).all())


def test_rows_split_standardized_matches_f32_rows(ops):
    """With mean/std/clip the split parts reconstruct exactly the f32 standardised rows that rows_to_bf16 writes to
    dst_f32 for the same input (clip((x - mean) / std, -5, 5), batched_agent_manager.py:303-315)."""
    g = torch.Generator().manual_seed(3)
    n, width = 1001, 89
    x = torch.randn(n, width, generator=g) * 3
    x[::7, ::5] *= 40                                   # some values clip
    mean = torch.randn(width, generator=g)
    std = torch.rand(width, generator=g) + 0.05
    ps = ops.pad64(width)
    parts = sentinel(n, 3 * ps)
    ops.rows_split(x.to(DEV), parts, 3, ps, mean.to(DEV), std.to(DEV), 5.0)
    f32 = torch.full((n, width), float("nan"), device=DEV)
    bf = torch.zeros((n, ops.pad8(width)), dtype=torch.bfloat16, device=DEV)
    ops.rows_to_bf16(x.to(DEV), bf, mean.to(DEV), std.to(DEV), 5.0, dst_f32=f32)
    torch.cuda.synchronize()
    want = f32.cpu()
    assert float(want.abs().max()) == 5.0
    assert torch.equal(recon(parts, 3, ps, width), want.double())
    assert torch.equal(parts[:, :width].cpu(), bf[:, :width].cpu())      # part 0 is the bf16 mode's operand


# ------------------------------------------------------------------------------------------------------------
# 2. split GEMMs against fp64
# ------------------------------------------------------------------------------------------------------------
def fwd_bound(n_products, K, order, out_parts):
    """Bound on e for the forward over 3-part operands.
      dropped products: |part_i| <= 2^-8i |x| per operand, so the products with i + j >= order add at most
        sum_{i+j>=order, i,j<3} 2^-8(i+j): 2 * 2^-24 + 2^-32 for order 3;
      fp32 accumulation of T = n_products * K exact products (bf16 x bf16 fits fp32): the worst case T * u (7e-4 at
        K = 2048) could not tell a dropped 2^-16 product from rounding.  With one operand of random sign the partial
        sums random-walk far below sum |x w|, and rounding errors add like a random walk too: sqrt(T) * u bounds it here
        (the measured errors below are ~50x under it);
      output: out_parts bf16 parts keep 8 * out_parts bits, |y - parts| <= 2^(-8 out_parts) |y| (3 parts: exact).
    Measured on a B200: order 3, out_parts 3: e <= 2.7e-7 at every shape (bound >= 1.5e-6); order 2: e >= 2.3e-5."""
    dropped = sum(2.0 ** (-8 * (i + j)) for i in range(3) for j in range(3) if i + j >= order)
    out = 0.0 if out_parts == 3 else 2.0 ** (-8 * out_parts)
    return dropped + math.sqrt(n_products * K) * U + out


FWD_SHAPES = [(256, 89, 0), (256, 256, 0), (1024, 2048, 0), (2048, 1024, 0), (24, 256, 21), (16, 256, 16)]


@pytest.mark.parametrize("M", [1, 127, 129, 50000])
@pytest.mark.parametrize("N,K,bias_n", FWD_SHAPES, ids=[f"{n}x{k}" for n, k, _ in FWD_SHAPES])
def test_linear_fwd_split(ops, M, N, K, bias_n):
    """rlppo_linear_fwd with make_split(3,3,3,out_parts) (forward_hidden / logits in "fp32" mode) for relu 0/1 and
    out_parts 1..3; make_split(3,3,2,3) must fail the bound; make_split(1,1,1,3) (the bf16 mode's logits: single-part
    operands, output as 3 parts) against fp64 of the bf16 operands, bound sqrt(K) * u.  The output starts as a sentinel:
    rows >= M and the columns between N and the part stride stay untouched; with relu every part of a negative
    pre-activation is zero."""
    n_real = bias_n or N
    x = tailed((M, K), 11 + M, positive=True, device=DEV)
    w = torch.zeros(N, K)
    w[:n_real] = tailed((n_real, K), 12, positive=False)
    b = torch.zeros(N)
    b[:n_real] = torch.randn(n_real, generator=torch.Generator().manual_seed(13)) * 0.25
    kp, op = ops.pad64(K), ops.pad64(N)
    xs = split_rows(ops, x, 3, kp)
    wq, _ = split_weight(ops, w[:n_real], 3, kp, N)
    bias = b[:n_real].to(DEV)
    rows = sample_rows(M)
    xr, t = x[rows.to(DEV)].cpu().double(), w.double()
    ref = xr @ t.t() + b.double()
    absum = xr.abs() @ t.abs().t() + b.double().abs() + 1e-300
    pad_rows = 3
    errs = {}
    for relu, out_parts in itertools.product((0, 1), (1, 2, 3)):
        y = sentinel(M + pad_rows, 3 * op)
        sp = ops.make_split(3, 3, 3, out_parts, kp, kp, op)
        ops.linear_fwd(xs, wq, bias, y, N, K, relu, M=M, split=sp, bias_n=bias_n)
        torch.cuda.synchronize()
        got = recon(y, out_parts, op, N, rows=rows)
        want = torch.relu(ref) if relu else ref
        e = gemm_err(got, want, absum)
        errs[(relu, out_parts)] = e
        assert e <= fwd_bound(6, K, 3, out_parts), (relu, out_parts, e)
        yb = bits(y)
        assert bool((yb[M:] == SENTINEL).all())
        for q in range(3):
            blk = yb[:M, q * op:(q + 1) * op]
            assert bool((blk[:, N:] == SENTINEL).all()), ("padding columns written", q)
            if q >= out_parts:
                assert bool((blk == SENTINEL).all())
        if relu:
            # clearly negative pre-activations only: one within the kernel's error of zero may round either way
            neg = ref < -fwd_bound(6, K, 3, 3) * absum
            assert bool(neg.any())
            for q in range(out_parts):
                assert bool((y[rows, q * op:q * op + N].cpu().float()[neg] == 0).all())
    # the degraded schedule: one order less drops part_i x part_j with i + j = 2 -- it must fail the bound
    y = sentinel(M, 3 * op)
    ops.linear_fwd(xs, wq, bias, y, N, K, 0, M=M, split=ops.make_split(3, 3, 2, 3, kp, kp, op), bias_n=bias_n)
    e_deg = gemm_err(recon(y, 3, op, N, rows=rows), ref, absum)
    e_ok = errs[(0, 3)]
    print(f"fwd M={M} N={N} K={K}: e(order 3) = {e_ok:.2e}  e(order 2) = {e_deg:.2e}  bound {fwd_bound(6, K, 3, 3):.2e}")
    assert e_deg > fwd_bound(6, K, 3, 3) and e_deg >= 30 * e_ok, (e_deg, e_ok)

    # bf16-mode logits: one-part operands (part 0 of the same buffers), f32-exact output in three parts
    y = sentinel(M + pad_rows, 3 * op)
    ops.linear_fwd(xs, wq, bias, y, N, K, 0, M=M, split=ops.make_split(1, 1, 1, 3, 0, 0, op), bias_n=bias_n)
    torch.cuda.synchronize()
    xb, wb = x[rows.to(DEV)].cpu().bfloat16().double(), w.bfloat16().double()
    ref1 = xb @ wb.t() + b.double()
    e1 = gemm_err(recon(y, 3, op, N, rows=rows), ref1, xb.abs() @ wb.abs().t() + b.double().abs() + 1e-300)
    assert e1 <= (math.sqrt(K) + 1) * U, e1          # accumulation, and the bias added in fp32
    assert bool((bits(y)[M:] == SENTINEL).all()) and bool((bits(y)[:M, N:op] == SENTINEL).all())


def bwd_bound(n_products, T, out_parts):
    """Bound on e for dgrad / wgrad over 2-part operands (make_split(2,2,2,.)), reference from the f32 masters:
      x = part0 + part1 + r with |r| <= 2^-16 |x| for each operand, and the dropped product part1 x part1 is
      <= 2^-16 |x w|: 3 * 2^-16 in all;
      accumulation of T terms: sqrt(T) * u, as for the forward;
      output written as out_parts parts: + 2^(-8 out_parts) (out_parts 1: the wgrad's fp32 dW is exact, pass 3).
    Measured on a B200: e <= 2.9e-5 against bounds >= 4.7e-5 (the tails of the test operands all have one sign, so r
    and the dropped product add up rather than cancel); the order-1 run, which also drops part1 x part0, gives
    e >= 4.0e-3."""
    out = 0.0 if out_parts == 3 else 2.0 ** (-8 * out_parts)
    return 3 * 2.0 ** -16 + math.sqrt(n_products * T) * U + out


def _hprev(M, K, seed):
    """A ReLU output with tiny positives (normal and subnormal) and -0.0 among ordinary values."""
    g = torch.Generator().manual_seed(seed)
    h = torch.relu(torch.randn(M, K, generator=g))
    pick = torch.randint(0, 6, (M, K), generator=g)
    h[pick == 0] = 1e-30
    h[pick == 1] = -0.0
    h[(pick == 2) & (torch.rand(M, K, generator=g) < 0.1)] = 1e-40
    h[(pick == 3) & (torch.rand(M, K, generator=g) < 0.1)] = 2.0 ** -126
    return h


@pytest.mark.parametrize("M", [129, 5000])
@pytest.mark.parametrize("N,K", [(96, 256), (89, 256), (256, 1024), (1024, 256)])
def test_linear_dgrad_split(ops, M, N, K):
    """rlppo_linear_dgrad, make_split(2,2,2,2, d_ps, pad64(N), d_ps) as backward_hidden / head_backward pass it:
    dX = (dY W) (.) (hprev > 0), hprev a 3-part ReLU output whose mask is read from part 0; db_below += fp64 column sums of
    the reconstructed f32 dX.  N = 96 is the head's out_pad; N = 89 a contraction that is not a multiple of 8 (its
    padding columns in dY and W^T must be zero).  Masked entries are +0 in both parts."""
    d_ps, n_ps, k_ps = ops.pad64(max(N, K)), ops.pad64(N), ops.pad64(K)
    dy = tailed((M, N), 21, positive=False)
    w = tailed((N, K), 22, positive=True)
    h = _hprev(M, K, 23)
    dys = split_rows(ops, dy, 2, d_ps)
    _, wt = split_weight(ops, w, 1, k_ps, ops.pad8(N), 2, n_ps, K)
    hs = split_rows(ops, h, 3, k_ps)
    hr = recon(hs, 3, k_ps, K)
    mask = (hr > 0).double()
    assert bool((mask[h == 1e-30] == 1).all()) and bool((mask[torch.signbit(h) & (h == 0)] == 0).all())
    ref = (dy.double() @ w.double()) * mask
    absum = (dy.double().abs() @ w.double().abs()) * mask + 1e-300
    db0 = torch.randn(K, generator=torch.Generator().manual_seed(24))

    def run(order):
        dx = sentinel(M + 2, 2 * d_ps)
        db = db0.clone().to(DEV)
        ops.linear_dgrad(dys, wt, hs, dx, N, K, M=M, db_below=db, split=ops.make_split(2, 2, order, 2, d_ps, n_ps, d_ps))
        torch.cuda.synchronize()
        return dx, db

    dx, db = run(2)
    got = recon(dx, 2, d_ps, K, rows=slice(0, M))
    e = gemm_err(got, ref, absum)
    bound = bwd_bound(3, N, 2)
    dx_d, _ = run(1)
    e_deg = gemm_err(recon(dx_d, 2, d_ps, K, rows=slice(0, M)), ref, absum)
    print(f"dgrad M={M} N={N} K={K}: e(order 2) = {e:.2e}  e(order 1) = {e_deg:.2e}  bound {bound:.2e}")
    assert e <= bound, e
    assert e_deg > bound and e_deg >= 30 * e, (e_deg, e)
    xb = bits(dx.cpu())
    for q in range(2):
        blk = xb[:M, q * d_ps:q * d_ps + K]
        assert bool((blk[mask == 0] == 0).all()), "masked entries must be +0 in every part"
        assert bool((xb[:M, q * d_ps + K:(q + 1) * d_ps] == SENTINEL).all())
    assert bool((xb[M:] == SENTINEL).all())
    # db_below: the column sums of the f32 dX (summed before the split).  The parts reconstruct it to 2^-16 per
    # element; the fp32 sums add at most M u: |db - (db0 + colsum)| <= (2^-16 + M u)(sum|dX| + |db0|)
    want = db0.double() + got.sum(0)
    scale = got.abs().sum(0) + db0.double().abs()
    err = float(((db.cpu().double() - want).abs() / scale).max())
    assert err <= 2.0 ** -16 + M * U, err


@pytest.mark.parametrize("M", [129, 5000])
@pytest.mark.parametrize("N,K,a_ps", [(1024, 89, 1024), (256, 89, 1024), (90, 256, 128)])
def test_linear_wgrad_split(ops, M, N, K, a_ps):
    """rlppo_linear_wgrad, make_split(2,2,2,1, a_pstride, b_pstride) with a_pstride != b_pstride, as
    backward_hidden passes it for hidden widths (1024, 256) and K = 89 (d_ps = pad64(max(hidden)) = 1024 against
    pad64(K)), and as head_backward passes it for 90 logits (pad64(90) against pad64(256)).  dW and db start nonzero and
    are accumulated into; db is the column sum of ALL parts of dY."""
    b_ps = ops.pad64(K)
    dy = tailed((M, N), 31, positive=False)
    x = tailed((M, K), 32, positive=True)
    dys = split_rows(ops, dy, 2, a_ps)
    xs = split_rows(ops, x, 2, b_ps)
    dw0 = torch.randn(N, K, generator=torch.Generator().manual_seed(33))
    db0 = torch.randn(N, generator=torch.Generator().manual_seed(34))
    ref = dy.double().t() @ x.double() + dw0.double()
    absum = dy.double().abs().t() @ x.double().abs() + dw0.double().abs()

    def run(order):
        dw, db = dw0.clone().to(DEV), db0.clone().to(DEV)
        ops.linear_wgrad(dys, xs, dw, db, N, K, M=M, split=ops.make_split(2, 2, order, 1, a_ps, b_ps))
        torch.cuda.synchronize()
        return dw.cpu().double(), db.cpu().double()

    dw, db = run(2)
    e = gemm_err(dw, ref, absum)
    bound = bwd_bound(3, M, 3)
    dw_d, _ = run(1)
    e_deg = gemm_err(dw_d, ref, absum)
    print(f"wgrad M={M} N={N} K={K}: e(order 2) = {e:.2e}  e(order 1) = {e_deg:.2e}  bound {bound:.2e}")
    assert e <= bound, e
    assert e_deg > bound and e_deg >= 30 * e, (e_deg, e)
    # db: sum over rows of part0 + part1 (2^-16 from the f32 master) in fp32: (2^-16 + 2M u) of sum|dy| + |db0|;
    # summing part 0 alone would be off by the tails' 2^-8
    want = dy.double().sum(0) + db0.double()
    err = float(((db - want).abs() / (dy.double().abs().sum(0) + db0.double().abs())).max())
    assert err <= 2.0 ** -16 + 2 * M * U, err


# ------------------------------------------------------------------------------------------------------------
# 3. split heads against fp64
# ------------------------------------------------------------------------------------------------------------
def _head_operands(ops, M, K, A, seed, scale=1.0):
    """f32 masters h (ReLU output) [M, K], w [A, K], b [A] and their 3-part device operands."""
    g = torch.Generator().manual_seed(seed)
    h = torch.relu(torch.randn(M, K, generator=g))
    w = torch.randn(A, K, generator=g) * scale * math.sqrt(2.0 / K)      # logits ~ N(0, scale^2)
    b = torch.randn(A, generator=g) * 0.1
    kp = ops.pad64(K)
    hs = split_rows(ops, h, 3, kp)
    wq, _ = split_weight(ops, w, 3, kp, ops.pad8(A))
    z64 = h.double() @ w.double().t() + b.double()
    zabs = h.double() @ w.double().abs().t() + b.double().abs()
    return h, w, b, hs, wq, z64, zabs


def _prob_bound(z64, zabs, A):
    """|s - p64| <= p64 * eps per entry, eps from: logits fp32-exact (2^-22 * sum|h w|, doubled for the difference
    z - max z); __expf(x) within (2 + 1.173 |x|) ulp of e^x (CUDA Math API, x = z - max z <= 0) on the numerator and on
    every term of the sum; the fp32 sum of A terms (A u) and the reciprocal / product (2 u)."""
    dz = 2 * 2.0 ** -22 * zabs.max(-1, keepdim=True).values
    xmax = (z64.max(-1, keepdim=True).values - z64.min(-1, keepdim=True).values)
    ulp_exp = 2 * (2 + 1.173 * xmax) * 2.0 ** -23
    return 2 * dz + ulp_exp + (A + 2) * U


@pytest.mark.parametrize("A", [1, 2, 21, 90, 128, 256])
def test_policy_head_sample_split(ops, A):
    """rlppo_policy_head_sample, schedule (3,3,3,1) (Stack.policy_head_sample in "fp32" mode): probs against the
    fp64 softmax of the fp64 logits within _prob_bound (measured on a B200: at most 0.15 of it), log-prob of the drawn
    action against log(clamp(p64[a])), actions against O.sample_inverse_cdf on the fp64 probabilities -- a differing row
    must have u * P within the fp32 CDF's error of a CDF boundary -- and the deterministic per-row argmax."""
    M, K = 3000, 256
    h, w, b, hs, wq, z64, zabs = _head_operands(ops, M, K, A, 40 + A)
    kp = ops.pad64(K)
    sp = ops.make_split(3, 3, 3, 1, kp, kp)
    u = torch.rand(M, generator=torch.Generator().manual_seed(41), dtype=torch.float64).float()
    acts = torch.empty(M, dtype=torch.int64, device=DEV)
    logp = torch.empty(M, device=DEV)
    probs = torch.empty(M, A, device=DEV)
    ops.policy_head_sample(hs, wq, b.to(DEV), A, K, u=u.to(DEV), actions_i64_out=acts, logp_out=logp, probs_out=probs,
                           split=sp)
    torch.cuda.synchronize()
    p64 = torch.softmax(z64, -1)
    eps = _prob_bound(z64, zabs, A)
    err = (probs.cpu().double() - p64).abs()
    print(f"sample A={A}: max |s-p|/(p eps) = {float((err / (p64 * eps)).max()):.3f}")
    assert bool((err <= p64 * eps + 1e-30).all())
    a = acts.cpu()
    a_ref = O.sample_inverse_cdf(p64, u.double())
    pc = p64.clamp(1e-11, 1.0)
    cdf = pc.cumsum(-1)
    thr = u.double() * cdf[:, -1]
    diff = (a != a_ref).nonzero().flatten()
    slack = (A + 2) * 2.0 ** -23 + eps.max()                # fp32 running sum of A clamped probabilities
    for r in diff.tolist():
        j = min(int(a[r]), int(a_ref[r]))
        assert abs(float(cdf[r, j] - thr[r])) <= float(slack) * float(cdf[r, -1]), (r, int(a[r]), int(a_ref[r]))
    assert diff.numel() <= max(2, M // 500)
    lp_ref = torch.log(pc.gather(-1, a.view(-1, 1))).flatten()
    lp_tol = float(eps.max()) + 2 * 2.0 ** -23 * max(1.0, float(lp_ref.abs().max()))     # + logf's rounding
    assert float((logp.cpu().double() - lp_ref).abs().max()) <= lp_tol
    # the Philox stream (counter (offset + row, high word, 0, 0), key (seed lo, seed hi)): a launch whose rows cross the
    # carry into the counter's high word draws exactly what the host restatement's uniforms draw when injected
    seed, off = 0x0123456789ABCDEF, 2 ** 32 - M // 2
    u_host = torch.from_numpy(philox_uniform(philox_rows(seed, off, M)[:, 0])).float().to(DEV)
    draws = []
    for kw in (dict(seed=seed, offset=off), dict(u=u_host)):
        a_, l_ = torch.empty(M, dtype=torch.int64, device=DEV), torch.empty(M, device=DEV)
        ops.policy_head_sample(hs, wq, b.to(DEV), A, K, actions_i64_out=a_, logp_out=l_, split=sp, **kw)
        draws.append((a_, l_))
    torch.cuda.synchronize()
    assert torch.equal(draws[0][0], draws[1][0]) and torch.equal(draws[0][1].view(torch.int32), draws[1][1].view(torch.int32))
    ops.policy_head_sample(hs, wq, b.to(DEV), A, K, deterministic=True, actions_i64_out=acts, logp_out=logp, split=sp)
    torch.cuda.synchronize()
    top2 = z64.topk(min(2, A), -1).values
    clear = (top2[:, 0] - top2[:, -1] > 4 * 2.0 ** -22 * zabs.max(-1).values) if A > 1 else torch.ones(M, dtype=torch.bool)
    assert torch.equal(acts.cpu()[clear], z64.argmax(-1)[clear])
    lp_det = torch.log(p64.max(-1).values.clamp(1e-11, 1.0))
    assert float((logp.cpu().double() - lp_det).abs().max()) <= float(eps.max()) + 2 * 2.0 ** -23 * max(1.0, float(lp_det.abs().max()))


def _ppo_reference(z64, acts, old, adv, B_total, clip=0.2, ent_coef=0.01):
    """The loss block of test_kernels_gpu.test_policy_head_train in fp64 with autograd; torch.clamp then log."""
    zt = z64.clone().requires_grad_(True)
    p = torch.softmax(zt, -1).clamp(1e-11, 1.0)
    lpa = torch.log(p)
    lp = lpa.gather(-1, acts.long().view(-1, 1)).flatten()
    ent = -(lpa * p).sum(-1)
    ratio = torch.exp(lp - old.double())
    surr = torch.min(ratio * adv.double(), ratio.clamp(1 - clip, 1 + clip) * adv.double())
    loss = (-surr.sum() - ent_coef * ent.sum()) / B_total
    loss.backward()
    kl = (ratio - 1) - (lp - old.double())
    clipped = ((ratio - 1).abs() > clip).double()
    return zt.grad, lp.detach(), ent.detach(), kl.detach(), clipped, surr.detach()


def _check_train(ops, M, K, A, scale, split):
    h, w, b, hs, wq, z64, zabs = _head_operands(ops, M, K, A, 50, scale=scale)
    kp, zp = ops.pad64(K), ops.pad64(A)
    g = torch.Generator().manual_seed(51)
    acts = torch.randint(0, A, (M,), generator=g).float()
    lp64 = torch.log(torch.softmax(z64, -1).clamp(1e-11, 1.0)).gather(-1, acts.long().view(-1, 1)).flatten()
    old = (lp64 + torch.randn(M, generator=g, dtype=torch.float64) * 0.3).float()
    adv = (torch.randn(M, generator=g) * 0.5).float()
    B_total = 2 * M
    metrics = torch.zeros(8, device=DEV)
    logp = torch.empty(M, device=DEV)
    if split:
        dz = sentinel(M, 2 * zp)
        ops.policy_head_train(hs, wq, b.to(DEV), A, K, acts.to(DEV), old.to(DEV), adv.to(DEV), 1.0 / B_total, 0.2, 0.01,
                              dz, metrics, logp_out=logp, split=ops.make_split(3, 3, 3, 2, kp, kp, zp))
    else:   # bf16 mode: bf16 operands, reference on the bf16-rounded h, w
        hb, wb = h.bfloat16(), torch.zeros(ops.pad8(A), K, dtype=torch.bfloat16)
        wb[:A] = w.bfloat16()
        z64 = hb.double() @ wb[:A].double().t() + b.double()
        dz = sentinel(M, ops.pad8(A))
        ops.policy_head_train(hb.to(DEV), wb.to(DEV), b.to(DEV), A, K, acts.to(DEV), old.to(DEV), adv.to(DEV),
                              1.0 / B_total, 0.2, 0.01, dz, metrics, logp_out=logp)
    torch.cuda.synchronize()
    dz_ref, lp, ent, kl, clipped, surr = _ppo_reference(z64, acts, old, adv, B_total)
    if split:
        got = recon(dz, 2, zp, A)
        pad = bits(dz.cpu())
        for q in range(2):
            assert bool((pad[:, q * zp + A:(q + 1) * zp] == 0).all())
    else:
        got = dz.cpu()[:, :A].double()
        assert bool((bits(dz.cpu())[:, A:] == 0).all())
    lp_tol = float(_prob_bound(z64, zabs, A).max()) + 2 * 2.0 ** -23 * max(1.0, float(lp.abs().max()))
    return got, dz_ref, logp.cpu().double(), lp, metrics.cpu().double(), ent, kl, clipped, surr, z64, lp_tol


@pytest.mark.parametrize("A", [21, 90, 256])
def test_policy_head_train_split(ops, A):
    """rlppo_policy_head_train, schedule (3,3,3,2): dz (2 parts) against fp64 autograd of the PPO loss block.
    Bound rel-L2 <= 3e-5: the 2-part output keeps 16 bits (2^-16 per element), and __expf / __logf (a few ulp, 2^-21.4
    absolute for __logf near 1) move s and log p by ~1e-6 relative.  Measured on a B200: 2.5e-6.  logp_out within
    _prob_bound's eps plus logf's rounding; metrics [0..4] against the fp64 means."""
    M, K = 2000, 256
    got, ref, logp, lp, m, ent, kl, clipped, surr, _, lp_tol = _check_train(ops, M, K, A, 1.0, True)
    err = rel_l2(got, ref)
    print(f"train_split A={A}: dz rel-L2 {err:.2e}")
    assert err <= 3e-5, err
    assert float((logp - lp).abs().max()) <= lp_tol
    assert m[4] == M
    assert abs(m[0] / M - float(ent.mean())) <= 1e-5 * max(1.0, abs(float(ent.mean())))
    assert abs(m[1] / M - float(kl.mean())) <= 1e-5
    assert abs(m[2] - float(clipped.sum())) <= 2          # a ratio within rounding of 1 +- clip may count either way
    assert abs(m[3] / M - float(surr.mean())) <= 1e-5


@pytest.mark.parametrize("split", [False, True], ids=["bf16", "split"])
def test_policy_head_train_saturated_logits(ops, split):
    """Logit scale ~30: softmax entries below 1e-11 (the clamp passes no gradient there) and entries equal to 1.0 in
    f32.  The reference is torch's clamp-then-log expression in fp64.  Bounds as test_policy_head_train_split (split)
    and the bf16 test's 6e-3 (bf16 operands and a bf16 dz, 2^-9 per element); at logit scale 30 the logits' own fp32
    error (u sum|h w| ~ 1e-5) dominates the log-prob error, which _prob_bound accounts for.  Measured on a B200: dz
    rel-L2 7.6e-6 (split), 1.6e-3 (bf16)."""
    M, K, A = 1000, 256, 90
    got, ref, logp, lp, m, ent, kl, clipped, surr, z64, lp_tol = _check_train(ops, M, K, A, 30.0, split)
    p64 = torch.softmax(z64, -1)
    assert bool((p64 < 1e-11).any()) and float(p64.max()) > 1 - 2.0 ** -25    # both clamp edges are exercised
    err = rel_l2(got, ref)
    print(f"train saturated {'split' if split else 'bf16'}: dz rel-L2 {err:.2e}")
    assert err <= (3e-5 if split else 6e-3), err
    assert float((logp - lp).abs().max()) <= lp_tol
    assert m[4] == M
    assert abs(m[0] / M - float(ent.mean())) <= (1e-5 if split else 1e-2) * max(1.0, abs(float(ent.mean())))


@pytest.mark.parametrize("M,K", [(129, 256), (1000, 1024)])
def test_value_head_split(ops, M, K):
    """rlppo_value_head: H in 3 parts (fp32-exact), dH written as 2 parts, targets given.  Bounds (rigorous, from
    the kernel's summation order: K/256 chunks of 8 fused multiply-adds per lane, a 5-level warp tree, + b):
      |v - v64| <= (8 K/256 + 6) u (sum_k |h w| + |b|);
      dv = 2 inv (v - t): |dv - dv64| <= 2 inv (|v - v64| + u |v - t|) + 2 u |dv| (inv is passed as f32);
      dH = dv w masked: |dH - dH64| <= |w| |dv - dv64| + (2^-16 + u) |dv64 w|;
      dw, db, metrics[5]: the row sums of those, plus M u of fp32 accumulation."""
    g = torch.Generator().manual_seed(60)
    h = _hprev(M, K, 61)
    w = torch.randn(K, generator=g) * 0.1
    b = torch.tensor([0.3])
    tgt = torch.randn(M, generator=g)
    kp, d_ps = ops.pad64(K), ops.pad64(K) + 64
    hs = split_rows(ops, h, 3, kp)
    v = torch.empty(M, device=DEV)
    dh = sentinel(M, 2 * d_ps)
    dw0 = torch.randn(K, generator=g)
    dw, db = dw0.clone().to(DEV), torch.full((1,), 0.5, device=DEV)
    metrics = torch.zeros(8, device=DEV)
    inv_b = 1.0 / (3 * M)
    ops.value_head(hs, w.to(DEV), b.to(DEV), K, values_out=v, targets=tgt.to(DEV), inv_batch=inv_b, dh=dh, dw=dw, db=db,
                   metrics=metrics, h_parts=3, h_pstride=kp, dh_parts=2, dh_pstride=d_ps)
    torch.cuda.synchronize()
    hd, wd = h.double(), w.double()
    v64 = hd @ wd + 0.3
    dv_err = (8 * ((K + 255) // 256) + 6) * U * (hd.abs() @ wd.abs() + 0.3)
    assert bool(((v.cpu().double() - v64).abs() <= dv_err).all())
    d64 = 2 * inv_b * (v64 - tgt.double())
    ddv = 2 * inv_b * (dv_err + U * (v64 - tgt.double()).abs()) + 2 * U * d64.abs()     # + inv_batch rounded to f32
    mask = (hd > 0).double()
    dh_ref = d64[:, None] * wd[None, :] * mask
    dh_bound = (wd.abs()[None, :] * ddv[:, None] + (2.0 ** -16 + U) * dh_ref.abs()) * mask
    got = recon(dh, 2, d_ps, K)
    assert bool(((got - dh_ref).abs() <= dh_bound + 1e-300).all())
    assert bool((bits(dh.cpu())[:, :K][mask == 0] == 0).all())
    for q in range(2):
        assert bool((bits(dh.cpu())[:, q * d_ps + K:(q + 1) * d_ps] == SENTINEL).all())
    dw_ref = (d64[:, None] * hd).sum(0) + dw0.double()
    dw_bound = (hd.abs() * ddv[:, None]).sum(0) + M * U * ((d64.abs()[:, None] * hd).sum(0) + dw0.double().abs())
    assert bool(((dw.cpu().double() - dw_ref).abs() <= dw_bound).all())
    db_ref = float(d64.sum()) + 0.5
    assert abs(float(db.cpu()) - db_ref) <= float(ddv.sum()) + M * U * (float(d64.abs().sum()) + 0.5)
    m = metrics.cpu().double()
    sq = float(((v64 - tgt.double()) ** 2).sum())
    assert m[6] == M
    assert abs(m[5] - sq) <= 1e-5 * sq


# ------------------------------------------------------------------------------------------------------------
# 4. head backward kernels, every subset of upstream gradients
# ------------------------------------------------------------------------------------------------------------
def _subsets(names):
    return [tuple(c) for r in range(len(names) + 1) for c in itertools.combinations(names, r)]


def _sid(s):
    return "+".join(s) if s else "none"


DISC = _subsets(("d_logp", "d_ent", "d_probs"))


@pytest.mark.parametrize("saturated", [False, True], ids=["normal", "saturated"])
@pytest.mark.parametrize("M", [1, 129])
@pytest.mark.parametrize("split", [False, True], ids=["bf16", "split"])
@pytest.mark.parametrize("given", DISC, ids=[_sid(s) for s in DISC])
def test_policy_head_backward_subsets(ops, given, split, M, saturated):
    """rlppo_policy_head_backward with every subset of (d_logp, d_ent, d_probs), the rest NULL (actions NULL too
    when d_logp is): dz against fp64 autograd of [log p[a], mean entropy, softmax] (clamp then log) with zeros for the
    missing gradients.  dz is written over more columns than the head has (128 for 90 logits); those come out zero.

    Bound, per element: dz_j = s_j (g_j - G) with g = d(outputs)/d(softmax) and G = sum_k g_k s_k.  With s good to eps
    relative (_prob_bound), __logf to 2^-21 absolute and the fp32 sum G to (A + 2) u,
      |dz_j - dz64_j| <= (eps + 2^-21 + (A + 2) u) s_j (max_k |g_k| + sum_k |g_k| s_k) + 2^(-8 parts) |dz64_j|
                         + 2^-125 (max_k |g_k| + sum_k |g_k| s_k) + 2^-134.
    Both absolute terms are range limits, not kernel faults, and at logit scale 30 both are reached:
      - __expf flushes results below 2^-126 to zero, so a tiny s_j is 0 in the kernel and so is its dz_j (measured on a
        B200 without this term: 240x-3600x over a bound relative to s_j alone);
      - dz is stored as bf16, whose subnormals are 2^-133 apart, so a dz_j below 2^-126 is stored to within 2^-134
        whatever the number of parts (the limit test_rows_split_reconstruction_exact finds for the split).  With an
        entropy gradient only, the row scale is |d_ent| / M, and at M = 129 some dz_j land there (measured without
        this term: 3.7x (bf16) and 4.2x (split) over the bound, in entries of ~1e-40).
    An fp32 emulation of the epilogue with that flush and that output rounding reproduces both excesses.
    A relative measure would not do: in a saturated row s_max is exactly 1.0 in f32 and dz_max is a difference of
    near-equal fp32 numbers, good to u |g| but not to its own (tiny) size.  The bound still catches a wrong clamp mask:
    an entry below 1e-11 that kept its gradient would be off by ~25 |d_ent / M| s_j."""
    K, A = 256, 90
    scale = 30.0 if saturated else 1.0
    h, w, b, hs, wq, z64, zabs = _head_operands(ops, M, K, A, 70 + M, scale=scale)
    kp, zp = ops.pad64(K), 128
    g = torch.Generator().manual_seed(71)
    acts = torch.randint(0, A, (M,), generator=g).float()
    up = {"d_logp": torch.randn(M, generator=g), "d_ent": torch.randn(1, generator=g),
          "d_probs": torch.randn(M, A, generator=g)}
    dv = {k: (up[k].to(DEV) if k in given else None) for k in up}
    a_dev = acts.to(DEV) if "d_logp" in given else None
    if split:
        dz = sentinel(M, 2 * zp)
        ops.policy_head_backward(hs, wq, b.to(DEV), A, K, a_dev, dv["d_logp"], dv["d_ent"], dv["d_probs"], dz,
                                 split=ops.make_split(3, 3, 3, 2, kp, kp, zp))
    else:
        hb, wb = h.bfloat16(), torch.zeros(ops.pad8(A), K, dtype=torch.bfloat16)
        wb[:A] = w.bfloat16()
        z64 = hb.double() @ wb[:A].double().t() + b.double()
        dz = sentinel(M, zp)
        ops.policy_head_backward(hb.to(DEV), wb.to(DEV), b.to(DEV), A, K, a_dev, dv["d_logp"], dv["d_ent"],
                                 dv["d_probs"], dz)
    torch.cuda.synchronize()
    zt = z64.clone().requires_grad_(True)
    s = torch.softmax(zt, -1)
    p = s.clamp(1e-11, 1.0)
    lp = torch.log(p)
    outs = [lp.gather(-1, acts.long().view(-1, 1)).flatten(), -(lp * p).sum(-1).mean(), s]
    grads = [(up[k] if k in given else torch.zeros_like(up[k])).double().view_as(o) for k, o in zip(up, outs)]
    ref, g_s = torch.autograd.grad(outs, [zt, s], grads)
    s64 = s.detach()
    eps = _prob_bound(z64, zabs, A) + 2.0 ** -21 + (A + 2) * U
    scale = g_s.abs().max(-1, keepdim=True).values + (g_s.abs() * s64).sum(-1, keepdim=True)
    bound = eps * s64 * scale + 2.0 ** -125 * scale + (2.0 ** -16 if split else 2.0 ** -8) * ref.abs() + 2.0 ** -134
    dzc = dz.cpu()
    parts = 2 if split else 1
    got = recon(dzc, parts, zp, A)
    for q in range(parts):
        assert bool((bits(dzc)[:, q * zp + A:(q + 1) * zp] == 0).all())
    if not given:
        assert float(got.abs().max()) == 0.0
        return
    ratio = float(((got - ref).abs() / bound).max())
    assert ratio <= 1.0, ratio


MD = _subsets(("d_logp", "d_ent"))


@pytest.mark.parametrize("saturated", [False, True], ids=["normal", "saturated"])
@pytest.mark.parametrize("M", [1, 129])
@pytest.mark.parametrize("dz_parts", [1, 2])
@pytest.mark.parametrize("given", MD, ids=[_sid(s) for s in MD])
def test_head_multi_discrete_backward_subsets(ops, given, dz_parts, M, saturated):
    """rlppo_head_multi_discrete_backward with every subset of (d_logp, d_ent) (actions NULL when d_logp is): dz against
    fp64 autograd through O.head_multi_discrete on the f32 logits (3 parts, fp32-exact).  dz_cols = 32 > 24: the
    columns past the 21 logits are zero.  Bounds: the per-row tail uses expf / logf (<= 2 ulp) on exact logits, so
    dz carries ~1e-6 plus its output rounding: rel-L2 <= 2^-16 + 1e-5 for 2 parts, 2^-8 for 1 part (bf16)."""
    g = torch.Generator().manual_seed(80 + M)
    z = torch.randn(M, 21, generator=g) * (30.0 if saturated else 1.0)
    acts = torch.stack([torch.randint(0, nb, (M,), generator=g) for nb in O.ROLV_BINS], -1).float()
    up = {"d_logp": torch.randn(M, generator=g), "d_ent": torch.randn(1, generator=g)}
    zs = split_rows(ops, z, 3, 64)
    dz_cols, dps = 32, 64
    dz = sentinel(M, dz_parts * dps)
    ops.head_multi_discrete_backward(zs, 3, 64, M, acts.to(DEV) if "d_logp" in given else None,
                                     up["d_logp"].to(DEV) if "d_logp" in given else None,
                                     up["d_ent"].to(DEV) if "d_ent" in given else None, dz, dz_parts, dps, dz_cols)
    torch.cuda.synchronize()
    zt = z.double().requires_grad_(True)
    logp, ent, _ = O.head_multi_discrete(zt, acts)
    grads = [(up[k] if k in given else torch.zeros_like(up[k])).double().view_as(o) for k, o in zip(up, (logp, ent))]
    (ref,) = torch.autograd.grad([logp, ent], [zt], grads)
    dzc = dz.cpu()
    got = recon(dzc, dz_parts, dps, 21)
    for q in range(dz_parts):
        assert bool((bits(dzc)[:, q * dps + 21:q * dps + dz_cols] == 0).all())
        assert bool((bits(dzc)[:, q * dps + dz_cols:(q + 1) * dps] == SENTINEL).all())
    if not given:
        assert float(got.abs().max()) == 0.0
        return
    err = rel_l2(got, ref)
    assert err <= (2.0 ** -16 + 1e-5 if dz_parts == 2 else 2.0 ** -8), err


CT = _subsets(("d_logp", "d_ent", "d_mean", "d_std"))


@pytest.mark.parametrize("saturated", [False, True], ids=["normal", "saturated"])
@pytest.mark.parametrize("M", [1, 129])
@pytest.mark.parametrize("dz_parts", [1, 2])
@pytest.mark.parametrize("given", CT, ids=[_sid(s) for s in CT])
def test_head_continuous_backward_subsets(ops, given, dz_parts, M, saturated):
    """rlppo_head_continuous_backward with every subset of (d_logp, d_ent, d_mean, d_std): dz against fp64 autograd of
    O.head_continuous (log-pdf, mean entropy) and get_output's (mean, std) = (tanh(z1), tanh(z2) m + b).  "saturated"
    puts half the pre-activations at |z| > 10: the Tanh is flat (f32 tanh is exactly +-1, fp64 leaves ~1e-8 of slope)
    and the std sits at var_min or var_max.  dz_cols = 16 > 2n = 8.  Bounds as the multi-discrete head (tanhf, logf,
    divisions: a few ulp)."""
    n, var_min, var_max = 4, 0.1, 1.0
    g = torch.Generator().manual_seed(90 + M)
    z = torch.randn(M, 2 * n, generator=g)
    if saturated:
        big = torch.rand(M, 2 * n, generator=g) < 0.5
        z[big] = torch.sign(z[big]) * (10.5 + 5 * torch.rand(int(big.sum()), generator=g))
    acts = (torch.rand(M, n, generator=g) * 2 - 1).float()
    up = {"d_logp": torch.randn(M, generator=g), "d_ent": torch.randn(1, generator=g),
          "d_mean": torch.randn(M, n, generator=g), "d_std": torch.randn(M, n, generator=g)}
    zs = split_rows(ops, z, 3, 64)
    dz_cols, dps = 16, 64
    dz = sentinel(M, dz_parts * dps)
    d = {k: (up[k].to(DEV) if k in given else None) for k in up}
    ops.head_continuous_backward(zs, 3, 64, M, n, var_min, var_max, acts.to(DEV) if "d_logp" in given else None,
                                 d["d_logp"], d["d_ent"], d["d_mean"], d["d_std"], dz, dz_parts, dps, dz_cols)
    torch.cuda.synchronize()
    zt = z.double().requires_grad_(True)
    logp, ent, _ = O.head_continuous(zt, acts.double(), var_min, var_max)
    t = torch.tanh(zt)
    m = (var_max - var_min) / 2.0
    outs = (logp, ent, t[:, :n], t[:, n:] * m + (var_min + m))
    grads = [(up[k] if k in given else torch.zeros_like(up[k])).double().view_as(o) for k, o in zip(up, outs)]
    (ref,) = torch.autograd.grad(outs, [zt], grads)
    dzc = dz.cpu()
    got = recon(dzc, dz_parts, dps, 2 * n)
    for q in range(dz_parts):
        assert bool((bits(dzc)[:, q * dps + 2 * n:q * dps + dz_cols] == 0).all())
    if not given:
        assert float(got.abs().max()) == 0.0
        return
    err = rel_l2(got, ref)
    assert err <= (2.0 ** -16 + 1e-5 if dz_parts == 2 else 2.0 ** -8), err


@pytest.mark.parametrize("with_db", [True, False])
@pytest.mark.parametrize("M", [1, 129])
@pytest.mark.parametrize("split", [False, True], ids=["bf16", "split"])
def test_value_head_backward(ops, split, M, with_db):
    """rlppo_value_head_backward: dH = dv w (.) (H > 0), dw += sum dv H, db += sum dv (db optional).  d_values
    is the head's only upstream gradient and is required (NULL is an argument error).  Bounds: dH is one f32 product
    rounded to the output's parts (2^-9 bf16 / 2^-16 + u for 2 parts); dw and db are sums of M exact-input terms:
    M u (rigorous).  H carries tiny positives and -0.0; the split dH's columns between K and its part stride stay
    untouched."""
    K = 256
    g = torch.Generator().manual_seed(100 + M)
    h = _hprev(M, K, 101)
    w = torch.randn(K, generator=g) * 0.1
    d_v = torch.randn(M, generator=g)
    dw0 = torch.randn(K, generator=g)
    dw = dw0.clone().to(DEV)
    db = torch.full((1,), 0.25, device=DEV) if with_db else None
    if split:
        kp, d_ps = ops.pad64(K), 1024
        hs = split_rows(ops, h, 3, kp)
        dh = sentinel(M, 2 * d_ps)
        ops.value_head_backward(hs, w.to(DEV), K, d_v.to(DEV), dh, dw, db, h_parts=3, h_pstride=kp, dh_parts=2,
                                dh_pstride=d_ps)
        hd = recon(hs, 3, kp, K)
    else:
        hb = h.bfloat16()
        dh = sentinel(M, K)
        ops.value_head_backward(hb.to(DEV), w.to(DEV), K, d_v.to(DEV), dh, dw, db)
        hd = hb.double()
    torch.cuda.synchronize()
    if split:
        assert torch.equal(hd > 0, h > 0)
    wd, dvd = w.double(), d_v.double()
    mask = (hd > 0).double()
    ref = dvd[:, None] * wd[None, :] * mask
    got = recon(dh, 2, d_ps, K) if split else dh.cpu().double()
    rnd = 2.0 ** -16 + U if split else 2.0 ** -8 + U
    assert bool(((got - ref).abs() <= rnd * ref.abs()).all())
    assert bool((bits(dh.cpu())[:, :K][mask == 0] == 0).all())
    if split:
        for q in range(2):
            assert bool((bits(dh.cpu())[:, q * d_ps + K:(q + 1) * d_ps] == SENTINEL).all())
    dw_ref = (dvd[:, None] * hd).sum(0) + dw0.double()
    bound = (M + 1) * U * ((dvd.abs()[:, None] * hd.abs()).sum(0) + dw0.double().abs())
    assert bool(((dw.cpu().double() - dw_ref).abs() <= bound).all())
    if with_db:
        assert abs(float(db.cpu()) - (float(dvd.sum()) + 0.25)) <= (M + 1) * U * (float(dvd.abs().sum()) + 0.25)
    from rlgym_ppo_b200._lib import RlppoError
    with pytest.raises(RlppoError, match="bad argument"):
        ops.value_head_backward(hs if split else hb.to(DEV), w.to(DEV), K, None, dh, dw, db,
                                **(dict(h_parts=3, h_pstride=kp, dh_parts=2, dh_pstride=d_ps) if split else {}))


# ------------------------------------------------------------------------------------------------------------
# module level: one upstream output at a time, so the NULL pointers reach the kernels through StackFunction
# ------------------------------------------------------------------------------------------------------------
N_ACT, N_CONT = 7, 4


def _policy(kind, precision):
    from rlgym_ppo_b200.ppo import ContinuousPolicy, DiscreteFF, MultiDiscreteFF
    if kind == "discrete":
        m = DiscreteFF(20, N_ACT, (64, 64), DEV, precision=precision)
    elif kind == "multi_discrete":
        m = MultiDiscreteFF(20, (64, 64), DEV, precision=precision)
    else:
        m = ContinuousPolicy(20, 2 * N_CONT, (64, 64), DEV, precision=precision)
    m.autograd = True
    return m


def _policy_actions(kind, rng, n):
    if kind == "discrete":
        return torch.from_numpy(rng.randint(0, N_ACT, (n, 1)).astype(np.float32))
    if kind == "multi_discrete":
        return torch.from_numpy(np.stack([rng.randint(0, b, n) for b in O.ROLV_BINS], -1).astype(np.float32))
    return torch.from_numpy(np.clip(rng.randn(n, N_CONT) * 0.5, -1, 1).astype(np.float32))


def _backprop_expr(kind, z, acts):
    """get_backprop_data's (log-prob, mean entropy) as torch expressions of the last Linear's output (the oracle's)."""
    if kind == "discrete":
        p = torch.clamp(torch.softmax(z, -1), 1e-11, 1.0)
        lp = torch.log(p)
        return lp.gather(-1, acts.view(-1, 1).long()), -(lp * p).sum(-1).mean()
    logp, ent, _ = O.head_multi_discrete(z, acts) if kind == "multi_discrete" else O.head_continuous(z, acts)
    return logp, ent


def _policy_reference_grads(m, kind, obs, acts, grads, precision):
    """Parameter gradients of get_backprop_data for the upstream `grads` on the CPU.  fp32 mode: fp64 autograd through a
    stock build_sequential module with the policy's weights.  bf16 mode: the oracle with the kernels' bf16 rounding
    points (operands of every GEMM rounded to bf16, hidden activations stored as bf16)."""
    from rlgym_ppo_b200.ppo._mlp import build_sequential
    sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    if precision == "fp32":
        st = m._stack
        seq = build_sequential(st.in_dim, st.hidden, st.out_dim, softmax=False).double()
        seq.load_state_dict({k[len("model."):]: v.double() for k, v in sd.items()})
        torch.autograd.backward(_backprop_expr(kind, seq(obs.double()), acts), [g.double() for g in grads])
        return [p.grad for p in seq.parameters()]
    params = [v.float() for v in sd.values()]
    z, layer_in = O.mlp_forward(params, obs.float(), O.quant_bf16)
    zl = z.detach().requires_grad_(True)
    (dz,) = torch.autograd.grad(_backprop_expr(kind, zl, acts), [zl], [g.float() for g in grads])
    return O.mlp_backward(params, layer_in, dz, O.quant_bf16)


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("which", ["log_probs", "entropy"])
@pytest.mark.parametrize("kind", ["discrete", "multi_discrete", "continuous"])
def test_module_single_output_backward(kind, which, precision):
    """get_backprop_data with autograd = True, then `log_probs.sum().backward()` alone or `entropy.backward()` alone:
    torch hands StackFunction a None gradient for the other output (set_materialize_grads(False)), which reaches the
    head backward kernel as a NULL pointer.  Parameter gradients against CPU autograd with a zero gradient in its place,
    tolerances as test_autograd_gpu.test_gradients_vs_cpu_autograd (1e-3 fp32, 2e-3 bf16 rel-L2 per tensor)."""
    torch.manual_seed(3)
    rng = np.random.RandomState(4)
    n, obs_dim = 129, 20
    m = _policy(kind, precision)
    obs = torch.from_numpy(rng.randn(n, obs_dim).astype(np.float32))
    acts = _policy_actions(kind, rng, n)
    logp, ent = m.get_backprop_data(obs.to(DEV), acts)
    for p in m.parameters():
        if p.grad is not None:
            p.grad.zero_()
    if which == "log_probs":
        logp.sum().backward()
        grads = [torch.ones(logp.shape), torch.zeros(())]
    else:
        ent.backward()
        grads = [torch.zeros(logp.shape), torch.ones(())]
    got = [p.grad.detach().cpu() for p in m.parameters()]
    want = _policy_reference_grads(m, kind, obs, acts, grads, precision)
    errs = [rel_l2(a, b) for a, b in zip(got, want)]
    print(f"{kind} {which} {precision}: grad rel-L2 per tensor", [float(f"{e:.2e}") for e in errs])
    assert max(errs) <= (1e-3 if precision == "fp32" else 2e-3), errs
