"""GPU tests, kernel level: the plain bf16 layer GEMMs (rlppo_linear_fwd, rlppo_linear_dgrad, rlppo_linear_wgrad with
sp == NULL, and the column-sum pass that forms linear_wgrad's db) and the one-launch weight gradient rlppo_wgrad_multi,
called through rlgym_ppo_b200.ops and checked element by element against fp64 references computed on the device.

1. Exact-integer operands.  Every operand entry is a small integer (|v| <= amp, a quarter of them zero; biases and the
   starting values of dW / db are integers too).  Every product is then exact, and so is every partial sum in any order
   while sum |a b| stays below 2^24 (each case asserts that it does).  So dW, db and db_below must equal the fp64
   reference bit for bit, whatever the row splits, atomicAdd order or TMEM accumulation order; the forward output and
   dgrad's dX must equal the round-to-nearest-even bf16 of the exact integer.  amp is sized so that those outputs
   often exceed 256 in magnitude, where bf16 rounds (and half the odd values are ties).  Zeros compare by value: the
   sign of an exact zero sum is the tensor core's choice, except in dX's padding columns, which must be +0.
2. Random operands (bf16 of N(0, 1)), per element.  e = |y - y64| / (sum_t |a_t b_t| + |bias|) <= (sqrt(T) + 2) u,
   u = 2^-24, T the contraction length (M for the weight gradients): the random-walk estimate of
   test_fused_kernels_gpu.py, whose gemm_e / excess (the distance from y64 to the reals that round to the stored bf16
   value, over e) measure the bf16 outputs.  Each check has a negative control on the same data that must fail it.
3. Layout.  Every operand sits in a NaN-filled buffer: rows past M, columns between the logical width and ld (inside
   the tensor maps for the weight gradients: dY columns N..pad8(N), X columns K..pad8(K); and past them), rows past N
   of w and past K of wt.  bias, db and db_below have 8 NaN guard floats after their last entry; y, dX and dW are
   sentinel-filled past their written extent, and each dW has one guard float after its last row (lddw == K cases put
   a write one column too far into the next row, or into that guard).  The kernels read only the logical extents
   promised in include/rlppo.h: none of this padding needs to be zero.
4. The row-split arithmetic of rlppo_linear_wgrad and rlppo_wgrad_multi is restated here (wgrad_rows, wgrad_multi_rows)
   to pick an M whose last row split is short: rounding the split size down would leave its rows uncovered.
5. wgrad_multi -> norm_clip_adam on one stream with no synchronisation (the PDL hand-off of the training step) gives
   the optimiser state bit-identical to norm_clip_adam on the exact gradients.

Measured on an NVIDIA B200 (1000 W power limit): every integer-operand case bit-exact, so tcgen05 does sum integer-valued
bf16 products below 2^24 exactly, whatever the split and order.  Largest random-operand errors as fractions of their
bounds: forward 0.126 (M = 50000, 1024 x 1024), dgrad dX 0.115 (M = 50000, 2048 x 2048), db_below 0.00061,
linear_wgrad dW / db 0.158 at M = 50000 and 0.148 at M = 200000, wgrad_multi 0.0085 at M = 200000.  Every control
fails its bound by a factor of 70 or more.  The file runs in 8 s there.

Run with `pytest -m gpu` on a B200."""
import ctypes
import math

import pytest
import torch

from test_fused_kernels_gpu import F32_SENTINEL, SENTINEL, U, bits, excess, f32_sentinel, gemm_e, pad8, sentinel
from test_split_kernels_gpu import gemm_err

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
EXACT = 2.0 ** 24          # integer sums below this are exact in fp32


@pytest.fixture(scope="module")
def ops():
    from rlgym_ppo_b200 import _lib, ops as _ops
    _lib.require_device()
    return _ops


def n_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def cdiv(a, b):
    return -(-a // b)


# ------------------------------------------------------------------------------------------------------------
# operands
# ------------------------------------------------------------------------------------------------------------
def ints(shape, seed, amp):
    """fp64 integers in [-amp, amp] on the device, a quarter of them zero."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    v = torch.randint(-amp, amp + 1, shape, generator=g, device=DEV).double()
    return v.masked_fill(torch.rand(shape, generator=g, device=DEV) < 0.25, 0.0)


def randn_bf16(shape, seed, scale=1.0):
    """fp64 copies of bf16(N(0, scale^2)) values on the device."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randn(shape, generator=g, device=DEV) * scale).bfloat16().double()


def amp_for(T, target=400.0):
    """Integer amplitude whose T-term dot products have an RMS near `target` (E a^2 ~ amp (amp + 1) / 4)."""
    a = 1
    while a < 127 and math.sqrt(T) * (a + 1) * (a + 2) / 4 <= target:
        a += 1
    return a


def operand(vals, ld, extra_rows=2):
    """fp64 values [R, C] (exact in bf16) -> bf16 [R + extra_rows, ld] with NaN everywhere else."""
    R, C = vals.shape
    buf = sentinel(R + extra_rows, ld)
    buf[:R, :C] = vals.bfloat16()
    return buf


def vec(vals, guard=8):
    """fp64 [n] -> f32 [n + guard], NaN guard floats after it."""
    buf = f32_sentinel(vals.numel() + guard)
    buf[:vals.numel()] = vals.float()
    return buf


def untouched_bf16(buf, M, cols):
    b = bits(buf)
    assert bool((b[M:] == SENTINEL).all()), "write past row M"
    assert bool((b[:M, cols:] == SENTINEL).all()), "write past the written columns"


def guard_intact(buf, n):
    assert bool((bits(buf)[n:] == F32_SENTINEL).all()), "write past the last entry"


def assert_exact(got, want, what):
    """Value equality (zeros of either sign equal) of a stored result with the exact fp64 one."""
    bad = (got.double() != want)
    assert not bool(bad.any()), (what, int(bad.sum()), bad.nonzero()[:4].tolist())


def colsum_rows_per_block(M):
    """rows_per_block of linear_wgrad's column-sum pass: NaN rows past M must cover it (a pass that read past M would
    then fail)."""
    r = cdiv(M, n_sms() * 8)
    return max(32, cdiv(r, 8) * 8)


# ------------------------------------------------------------------------------------------------------------
# row splits, restated from the host code of rlppo_linear_wgrad and rlppo_wgrad_multi
# ------------------------------------------------------------------------------------------------------------
def wgrad_rows(M, N, K, sms):
    """(m_per_split, splits) of rlppo_linear_wgrad."""
    bn = 64 if N <= 64 else (128 if N <= 128 else 256)
    tiles = cdiv(N, bn) * cdiv(K, 128)
    kblocks = cdiv(M, 64)
    splits = min(max(sms // tiles, 1), kblocks)
    return cdiv(kblocks, splits) * 64, splits


def wgrad_multi_rows(items, sms):
    """(m_per_split, splits as allocated) per item (M, N, K) of one rlppo_wgrad_multi launch."""
    tiles, kblocks, ideal, splits, nbytes = [], [], [], [], []
    for M, N, K in items:
        ntn, nkp = cdiv(N, 256), cdiv(K, 256)
        tiles.append(ntn * nkp)
        kblocks.append(cdiv(M, 64))
        nbytes.append(float(M) * 2.0 * (float(ntn) * min(K, 256 * nkp) + float(nkp) * min(N, 256 * ntn)))
    total = sum(nbytes)
    used = 0
    for i in range(len(items)):
        ideal.append(sms * (nbytes[i] / total) / tiles[i])
        splits.append(min(max(int(ideal[i]), 1), kblocks[i]))
        used += tiles[i] * splits[i]
    while True:
        best, gap = -1, 0.0
        for i in range(len(items)):
            g = ideal[i] - splits[i]
            if splits[i] < kblocks[i] and used + tiles[i] <= sms and g > gap:
                best, gap = i, g
        if best < 0:
            break
        splits[best] += 1
        used += tiles[best]
    return [(cdiv(kb, s) * 64, s) for kb, s in zip(kblocks, splits)]


def short_split(M, m_per_split, splits):
    """The last split is short, and a split size rounded down would leave rows of M uncovered."""
    kblocks = cdiv(M, 64)
    return M % m_per_split != 0 and kblocks % splits != 0 and splits * (kblocks // splits) * 64 < M


def split_edge_M(shapes_at, lo):
    """The least M >= lo, not a multiple of 64, at which every item of shapes_at(M) ((M, N, K) list) has a short last
    split under rlppo_wgrad_multi's allocation, and so does the first item under rlppo_linear_wgrad's."""
    sms = n_sms()
    M = lo
    while True:
        items = shapes_at(M)
        rows = wgrad_multi_rows(items, sms)
        if (M % 64 and all(short_split(m, *r) for (m, _, _), r in zip(items, rows))
                and short_split(M, *wgrad_rows(*items[0], sms))):
            return M
        M += 1


# ------------------------------------------------------------------------------------------------------------
# forward: Y = act(X W^T + bias) -> bf16
# ------------------------------------------------------------------------------------------------------------
FWD_NK = [(8, 1, 8), (8, 8, 8), (72, 63, 64), (136, 64, 64), (72, 65, 72), (136, 89, 96), (264, 127, 128),
          (264, 129, 136), (3000, 255, 256), (264, 256, 256), (136, 257, 264), (72, 1024, 1024), (264, 2048, 2048),
          (8, 3000, 3000)]
FWD_CASES = ([(M, 72, 65, 72) for M in (1, 63, 64, 65, 127, 128, 129)] + [(M, 264, 89, 96) for M in (1, 64, 129)]
             + [(129,) + c for c in FWD_NK]
             + [(50000, 2048, 89, 96), (50000, 2048, 2048, 2048), (50000, 1024, 2048, 2048), (50000, 1024, 1024, 1024)])


def _fid(M, N, K, ldx):
    return f"M{M}-N{N}-K{K}" + (f"-ld{ldx}" if ldx != pad8(K) else "")


def run_fwd(ops, x64, ldx, w64, b64, bias_n, relu, M, N, K):
    """One rlppo_linear_fwd on guarded operands; returns (y buffer, fp64 pre-rounding reference, bias used)."""
    x = operand(x64, ldx)
    w = operand(w64, pad8(K) + 8, extra_rows=8)                 # NaN rows past N, NaN columns past K
    bias = None if b64 is None else vec(b64[:bias_n])
    y = sentinel(M + 2, N + 8)
    ops.linear_fwd(x, w, bias, y, N, K, relu, M=M, bias_n=bias_n if bias_n != N else 0)
    torch.cuda.synchronize()
    bfull = torch.zeros(N, dtype=torch.float64, device=DEV)
    if b64 is not None:
        bfull[:bias_n] = b64[:bias_n]
    z = x64 @ w64.t() + bfull
    if bias is not None:
        guard_intact(bias, bias_n)
    untouched_bf16(y, M, N)
    return y, (z.clamp_min(0) if relu else z), bfull


@pytest.mark.parametrize("M,N,K,ldx", FWD_CASES, ids=[_fid(*c) for c in FWD_CASES])
def test_linear_fwd_exact(ops, M, N, K, ldx):
    """Integer operands: Y equals RN-even bf16 of the exact integer.  Two launches: ReLU with a bias (bias_n = N - 5
    on every other case: the columns past bias_n take no bias and the 8 NaN floats after bias_n are never read), and
    no ReLU with bias NULL."""
    amp = amp_for(K)
    x64, w64 = ints((M, K), M + K, amp), ints((N, K), N + K + 1, amp)
    b64 = ints((N,), N + 2, 600)
    bias_n = N - 5 if (M + N + K) % 2 and N > 8 else N
    absum = x64.abs() @ w64.abs().t() + b64.abs()
    assert float(absum.max()) < EXACT
    for relu, b in ((True, b64), (False, None)):
        y, ref, _ = run_fwd(ops, x64, ldx, w64, b, bias_n, relu, M, N, K)
        assert_exact(y[:M, :N].float(), ref.float().bfloat16().double(), ("fwd", relu, b is not None))
    big = float((ref.abs() > 256).double().mean())
    print(f"fwd exact {_fid(M, N, K, ldx)}: amp {amp}, {big:.0%} of |y| > 256")


FWD_RANDOM = [(129, 264, 257, 264), (4096, 136, 89, 96), (50000, 2048, 2048, 2048), (50000, 1024, 1024, 1024)]


@pytest.mark.parametrize("M,N,K,ldx", FWD_RANDOM, ids=[_fid(*c) for c in FWD_RANDOM])
def test_linear_fwd_random(ops, M, N, K, ldx):
    """bf16 N(0, 1) operands: excess over the bf16 rounding interval <= (sqrt(K) + 2) u (sum |x w| + |b|).  Control:
    the reference without the k = K - 1 term (a kernel that dropped the last contraction column) fails it."""
    x64, w64 = randn_bf16((M, K), M + K), randn_bf16((N, K), N + K + 1, 1.0 / math.sqrt(K))
    b64 = randn_bf16((N,), N + 2)
    y, z, bfull = run_fwd(ops, x64, ldx, w64, b64, N, False, M, N, K)
    e = gemm_e(x64, w64, bfull)
    r = excess(y[:M, :N], z, e)
    ctl = excess(y[:M, :N], z - x64[:, K - 1:] * w64[:, K - 1], e)
    print(f"fwd random {_fid(M, N, K, ldx)}: excess / bound {r:.3g}, control {ctl:.3g}")
    assert r <= 1.0, r
    assert ctl > 1.0, "fwd control passed"


# ------------------------------------------------------------------------------------------------------------
# dgrad: dX = (dY W) (.) (Hprev > 0) -> bf16, db_below += column sums of the stored dX
# ------------------------------------------------------------------------------------------------------------
def hprev_values(M, K, seed):
    """A ReLU input with -0.0, +0, tiny positive values (the least bf16 subnormal, 1e-30), negatives and positives."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    kind = torch.randint(0, 6, (M, K), generator=g, device=DEV)
    pool = torch.tensor([-0.0, 0.0, 2.0 ** -133, 1e-30, -3.0, 5.0], dtype=torch.float64, device=DEV)
    return pool[kind]


def run_dgrad(ops, dy64, w64, h64, M, N, K, db0=None, times=1):
    dy = operand(dy64, pad8(N) + 8)
    wt = operand(w64.t(), pad8(N) + 8, extra_rows=8)           # W^T [K, N]: NaN rows past K, NaN columns past N
    h = None if h64 is None else operand(h64, pad8(K) + 8)     # NaN in columns K..pad8(K) too
    dx = sentinel(M + 2, pad8(K) + 8)
    db = None if db0 is None else vec(db0)
    for _ in range(times):
        ops.linear_dgrad(dy, wt, h, dx, N, K, M=M, db_below=db)
    torch.cuda.synchronize()
    untouched_bf16(dx, M, pad8(K))
    assert bool((bits(dx)[:M, K:pad8(K)] == 0).all()), "dX padding columns must be +0"
    if db is not None:
        guard_intact(db, K)
    z = dy64 @ w64
    return dx, (z if h64 is None else z * (h64 > 0)), db


DGRAD_CASES = ([(M, 72, 65) for M in (1, 63, 64, 65, 127, 128, 129)] + [(M, 256, 89) for M in (1, 129)]
               + [(129, N, K) for N, K in ((8, 1), (17, 8), (90, 63), (256, 64), (40, 89), (96, 127), (300, 129),
                                           (256, 255), (64, 256), (17, 257), (1024, 1024), (256, 2048), (90, 3000))]
               + [(50000, 2048, 2048), (50000, 1024, 2048), (50000, 1024, 1024), (50000, 90, 1024)])


@pytest.mark.parametrize("M,N,K", DGRAD_CASES, ids=[f"M{M}-N{N}-K{K}" for M, N, K in DGRAD_CASES])
def test_linear_dgrad_exact(ops, M, N, K):
    """Integer operands: dX equals RN-even bf16 of the exact masked integer (mask Hprev > 0: -0.0 and +0 mask, the
    least bf16 subnormal does not), its padding columns K..pad8(K) are +0, and db_below, accumulated by two launches,
    equals its integer start plus twice the exact column sums of the stored dX.  Masked with db_below NULL (the epilogue
    branch without column sums, which the bf16 policy head's backward takes): the same dX, bit for bit.  Unmasked with
    db_below NULL: bit-exact too."""
    amp = amp_for(N, 250.0 if M > 10000 else 400.0)
    dy64, w64 = ints((M, N), M + N + 3, amp), ints((N, K), N + K + 4, amp)
    h64 = hprev_values(M, K, M + K + 5)
    db0 = ints((K,), K + 6, 1000)
    assert float((dy64.abs() @ w64.abs()).max()) < EXACT
    dx, ref, db = run_dgrad(ops, dy64, w64, h64, M, N, K, db0, times=2)
    want = ref.float().bfloat16().double()
    assert_exact(dx[:M, :K].float(), want, "dgrad dX")
    stored = dx[:M, :K].double()
    assert float((stored.abs().sum(0) * 2 + db0.abs()).max()) < EXACT
    assert_exact(db[:K], db0 + 2 * stored.sum(0), "db_below")
    dx1, _, _ = run_dgrad(ops, dy64, w64, h64, M, N, K)          # masked, db_below NULL (the bf16 head backward)
    assert_exact(dx1[:M, :K].float(), want, "dgrad dX, no db_below")
    assert torch.equal(bits(dx1), bits(dx)), "dX differs with and without db_below"
    dx2, ref2, _ = run_dgrad(ops, dy64, w64, None, M, N, K)
    assert_exact(dx2[:M, :K].float(), ref2.float().bfloat16().double(), "dgrad dX, no mask")
    print(f"dgrad exact M{M}-N{N}-K{K}: amp {amp}, {float((ref.abs() > 256).double().mean()):.0%} of |dX| > 256")


DGRAD_RANDOM = [(129, 300, 129), (50000, 2048, 2048), (50000, 1024, 1024)]


@pytest.mark.parametrize("M,N,K", DGRAD_RANDOM, ids=[f"M{M}-N{N}-K{K}" for M, N, K in DGRAD_RANDOM])
def test_linear_dgrad_random(ops, M, N, K):
    """bf16 N(0, 1) operands: dX excess <= (sqrt(N) + 2) u sum |dy w| per element; db_below (one launch) within
    (sqrt(M) + 2) u (sum |dX| + |db0|) of the fp64 column sums of the stored dX.  Controls: the reference without the
    n = N - 1 term, and db_below's reference without the first 64 rows."""
    dy64, w64 = randn_bf16((M, N), M + N), randn_bf16((N, K), N + K, 1.0 / math.sqrt(N))
    h64 = hprev_values(M, K, M + K)
    db0 = randn_bf16((K,), K)
    dx, z, db = run_dgrad(ops, dy64, w64, h64, M, N, K, db0)
    mask = h64 > 0
    e = gemm_e(dy64, w64.t()) * mask
    r = excess(dx[:M, :K], z, e)
    ctl = excess(dx[:M, :K], z - dy64[:, N - 1:] * w64[N - 1] * mask, e)
    stored = dx[:M, :K].double()
    scale = stored.abs().sum(0) + db0.abs()
    rb = gemm_err(db[:K].double(), db0 + stored.sum(0), scale) / ((math.sqrt(M) + 2) * U)
    cb = gemm_err(db[:K].double(), db0 + stored[64:].sum(0), scale) / ((math.sqrt(M) + 2) * U)
    print(f"dgrad random M{M}-N{N}-K{K}: excess / bound {r:.3g} (control {ctl:.3g}), db_below {rb:.3g} (control {cb:.3g})")
    assert r <= 1.0 and rb <= 1.0, (r, rb)
    assert ctl > 1.0 and cb > 1.0, "dgrad control passed"


# ------------------------------------------------------------------------------------------------------------
# weight gradients: dW[N, K] += dY^T X, db[N] += colsum(dY)
# ------------------------------------------------------------------------------------------------------------
class WG:
    """One weight-gradient operand set.  dY [M, N] and X [M, K] in NaN-filled buffers (ld pad8 + 8 unless given,
    colsum_rows_per_block(M) NaN rows past M); dW [N, lddw] in a sentinel buffer with one guard float after its last
    row, start values in its first K columns; db (optional) [N] + 8 guard floats."""

    def __init__(self, M, N, K, seed, ldx=None, lddw=None, with_db=True, exact=True):
        self.M, self.N, self.K = M, N, K
        if exact:
            self.dy64, self.x64 = ints((M, N), seed, 4), ints((M, K), seed + 1, 4)
            self.dw0, self.db0 = ints((N, K), seed + 2, 1000), ints((N,), seed + 3, 1000)
        else:
            self.dy64, self.x64 = randn_bf16((M, N), seed), randn_bf16((M, K), seed + 1)
            self.dw0, self.db0 = randn_bf16((N, K), seed + 2), randn_bf16((N,), seed + 3)
        rows = colsum_rows_per_block(M)
        self.dy = operand(self.dy64, pad8(N) + 8, rows)
        self.x = operand(self.x64, ldx or pad8(K) + 8, rows)
        self.lddw = lddw or K + 3
        self.dwbuf = f32_sentinel(N * self.lddw + 1)
        self.dw = self.dwbuf[:N * self.lddw].view(N, self.lddw)
        self.dw[:, :K] = self.dw0.float()
        self.db = vec(self.db0) if with_db else None
        self.frame = bits(self.dwbuf).clone()

    def item(self):
        return (self.dy, self.x, self.dw, self.N, self.K, self.db)

    def raw(self):
        """(item tuple, M) for wgrad_multi_raw."""
        return self.item(), self.M

    def ref(self, times=1):
        dy, x = self.dy64, self.x64
        return self.dw0 + times * (dy.t() @ x), self.db0 + times * dy.sum(0)

    def check_exact(self, times=1, what=""):
        ref_w, ref_b = self.ref(times)
        assert float((self.dw0.abs() + times * (self.dy64.abs().t() @ self.x64.abs())).max()) < EXACT
        assert_exact(self.dw[:, :self.K], ref_w, ("dW", what, self.M, self.N, self.K))
        frame = bits(self.dwbuf).view(-1)
        keep = torch.ones_like(frame, dtype=torch.bool)
        keep[:self.N * self.lddw].view(self.N, self.lddw)[:, :self.K] = False
        assert torch.equal(frame[keep], self.frame[keep]), ("write outside dW[:N, :K]", what)
        if self.db is not None:
            assert_exact(self.db[:self.N], ref_b, ("db", what, self.M, self.N, self.K))
            guard_intact(self.db, self.N)

    def errors(self, drop):
        """Largest per-element errors of dW and db as fractions of (sqrt(M) + 2) u, against the reference and against
        the reference without the rows `drop` (a row slice: the negative control).  Returns (ew, eb, control ew,
        control eb)."""
        dy, x = self.dy64, self.x64
        bound = (math.sqrt(self.M) + 2) * U
        dw, db = self.dw[:, :self.K].double(), None if self.db is None else self.db[:self.N].double()
        ref_w, ref_b = self.ref()
        absum = self.dw0.abs()
        for r in range(0, self.M, 16384):                # |dy|^T |x| by row chunks: no [M, K] temporaries
            absum += dy[r:r + 16384].abs().t() @ x[r:r + 16384].abs()
        out = [gemm_err(dw, ref_w, absum), gemm_err(dw, ref_w - dy[drop].t() @ x[drop], absum)]
        if db is not None:
            bsum = torch.linalg.vector_norm(dy, 1, dim=0) + self.db0.abs()
            out += [gemm_err(db, ref_b, bsum), gemm_err(db, ref_b - dy[drop].sum(0), bsum)]
        else:
            out += [0.0, math.inf]
        ew, cw, eb, cb = (e / bound for e in out)
        return ew, eb, cw, cb


def wgrad_multi_raw(items):
    """rlppo_wgrad_multi through the C ABI with a row count per item: items = [((dy, x, dW, N, K, db), M)]."""
    from rlgym_ppo_b200 import _lib
    arr = (_lib.WgradItem * len(items))()
    for a, ((dy, x, dw, N, K, db), M) in zip(arr, items):
        a.dy, a.lddy, a.x, a.ldx = dy.data_ptr(), dy.stride(0), x.data_ptr(), x.stride(0)
        a.dw, a.lddw, a.M, a.N, a.K = dw.data_ptr(), dw.stride(0), int(M), int(N), int(K)
        a.db = db.data_ptr() if db is not None else None
    _lib.call("rlppo_wgrad_multi", ctypes.cast(arr, ctypes.c_void_p), len(items), _lib.stream_ptr())


def c2_shapes(M):
    """The seven weight gradients of the bench's C2 step: policy head (90, 256), 256x256 hidden layers, 89 inputs."""
    return [(M, 90, 256), (M, 256, 256), (M, 256, 256), (M, 256, 89), (M, 256, 256), (M, 256, 256), (M, 256, 89)]


SPLIT_EDGE_M = None


def split_edge():
    global SPLIT_EDGE_M
    if SPLIT_EDGE_M is None:
        SPLIT_EDGE_M = split_edge_M(c2_shapes, 20000)
    return SPLIT_EDGE_M


WGRAD_CASES = ([(M, 17, 89, 96, None) for M in (1, 63, 64, 65, 127, 128, 129)] + [(M, 90, 257, None, 257) for M in
                                                                                  (1, 65, 129)]
               + [(129, N, K, None, lddw) for N, K, lddw in ((1, 1, 1), (17, 8, None), (90, 63, 63), (255, 64, None),
                                                             (256, 65, 65), (33, 127, None), (1, 129, 129),
                                                             (255, 255, None), (90, 256, 256), (200, 1024, None),
                                                             (17, 2048, 2048), (300, 3000, None))]
               + [("edge", 90, 256, None, None), (50000, 256, 89, 96, 89), (50000, 2048, 89, 96, None),
                  (50000, 2048, 2048, None, 2048), (50000, 1024, 2048, None, None), (50000, 1024, 1024, None, 1024),
                  (50000, 90, 1024, None, None)])


def _wid(M, N, K, ldx, lddw):
    return f"M{M}-N{N}-K{K}" + (f"-ld{ldx}" if ldx else "") + ("-lddwK" if lddw == K else "")


@pytest.mark.parametrize("M,N,K,ldx,lddw", WGRAD_CASES, ids=[_wid(*c) for c in WGRAD_CASES])
def test_linear_wgrad_exact(ops, M, N, K, ldx, lddw):
    """rlppo_linear_wgrad, integer operands: dW and db (the column-sum pass) bit-exact, twice accumulated; nothing
    written outside dW[:N, :K] and db[:N].  M = "edge": an M whose last row split is short (split_edge_M)."""
    if M == "edge":
        M = split_edge()
        assert short_split(M, *wgrad_rows(M, N, K, n_sms()))
    c = WG(M, N, K, M + N + K, ldx=ldx, lddw=lddw)
    for _ in range(2):
        ops.linear_wgrad(c.dy, c.x, c.dw, c.db, N, K, M=M)
    torch.cuda.synchronize()
    c.check_exact(times=2)


WMULTI_M = [1, 63, 64, 65, 127, 128, 129, "edge", 50000]


@pytest.mark.parametrize("M", WMULTI_M)
def test_wgrad_multi_c2_exact(ops, M):
    """rlppo_wgrad_multi on the C2 step's seven items (x ld 96 for the 89-input layers; the last item with lddw == K
    and no db), integer operands: bit-exact dW and db.  M = "edge": every item's last row split is short."""
    if M == "edge":
        M = split_edge()
    cs = [WG(M, N, K, 7 * i + M, ldx=96 if K == 89 else None, lddw=K if i >= 5 else None, with_db=i != 6)
          for i, (_, N, K) in enumerate(c2_shapes(M))]
    ops.wgrad_multi([c.item() for c in cs], M)
    torch.cuda.synchronize()
    for i, c in enumerate(cs):
        c.check_exact(what=f"item {i}")


def four_layer_nets(M):
    """The nine items of a policy (256, 192, 128, 64) with 128 actions and a value net of the same widths, obs 200."""
    widths = [200, 256, 192, 128, 64]
    hidden = [(M, widths[l + 1], widths[l]) for l in range(3, -1, -1)]
    return [(M, 128, 64)] + hidden + hidden


EDGE_ITEMS = [
    (150, 40, True),       # K - k0 = 150: the second 128-wide k tile spans a chunk the stage did not load; N = 40:
    (400, 296, True),      #   nch * 32 = 64 > bn = 48.  K = 400: k0 = 256 with 144 left, and db from the k0 == 0 pair
    (89, 17, False),       #   only.  Items without db.
    (129, 255, True),
    (513, 90, True),
    (64, 1, False),
    (1, 8, True),
    (300, 100, True),
]


@pytest.mark.parametrize("n_items", [1, 2, 3, 5, 8])
def test_wgrad_multi_items_exact(ops, n_items):
    """1 to 8 items of the tile-edge shapes, each with its own M (through the C ABI), integer operands: bit-exact."""
    Ms = [129, 63, 3001, 1, 640, 65, 2000, 127]
    cs = [WG(Ms[i], N, K, 31 * i + n_items, lddw=K if i % 2 else None, with_db=db)
          for i, (K, N, db) in enumerate(EDGE_ITEMS[:n_items])]
    wgrad_multi_raw([c.raw() for c in cs])
    torch.cuda.synchronize()
    for i, c in enumerate(cs):
        c.check_exact(what=f"item {i}")


def test_wgrad_multi_many_items_exact(ops):
    """The nine items of two 4-layer nets through ops.wgrad_multi (launches of 8 and 1); then those nine followed by the
    first four again (launches of 8 and 5), so the first four accumulate three products and the rest two.  Integer
    operands: bit-exact."""
    M = 1100
    cs = [WG(M, N, K, 13 * i, with_db=i % 4 != 3) for i, (_, N, K) in enumerate(four_layer_nets(M))]
    ops.wgrad_multi([c.item() for c in cs], M)
    torch.cuda.synchronize()
    for i, c in enumerate(cs):
        c.check_exact(what=f"item {i}")
    ops.wgrad_multi([c.item() for c in cs] + [c.item() for c in cs[:4]], M)
    torch.cuda.synchronize()
    for i, c in enumerate(cs):
        c.check_exact(times=3 if i < 4 else 2, what=f"item {i}, accumulated")


def test_wgrad_multi_more_tiles_than_sms_exact(ops):
    """One item of 12 x 13 = 156 (n, k-pair) tiles, more than the 148 SMs: CTAs loop over items and reuse TMEM after
    the drain warps release it (tempty).  A second item after it.  Integer operands: bit-exact."""
    M = 700
    a = WG(M, 3000, 3300, 1)
    b = WG(M, 90, 257, 2)
    rows = wgrad_multi_rows([(M, 3000, 3300), (M, 90, 257)], n_sms())
    assert 156 * rows[0][1] + cdiv(90, 256) * cdiv(257, 256) * rows[1][1] > n_sms()
    wgrad_multi_raw([a.raw(), b.raw()])
    torch.cuda.synchronize()
    a.check_exact(what="156 tiles")
    b.check_exact(what="after it")


WGRAD_RANDOM = [50000, 200000]


@pytest.mark.parametrize("M", WGRAD_RANDOM)
def test_wgrad_random(ops, M):
    """bf16 N(0, 1) operands, contraction over M rows: dW and db within (sqrt(M) + 2) u (sum_m |dy x| + |dW0|) per
    element, for rlppo_linear_wgrad ((2048, 2048) and (90, 1024)) and rlppo_wgrad_multi (the C2 items).  Control: the
    reference without rows 64..127 (one dropped 64-row block) fails it."""
    worst = {}

    def check(name, c):
        ew, eb, cw, cb = c.errors(drop=slice(64, 128))
        assert ew <= 1.0 and eb <= 1.0, (name, c.N, c.K, ew, eb)
        assert cw > 1.0 and cb > 1.0, ("wgrad control passed", name, c.N, c.K)
        worst[name] = max(worst.get(name, 0.0), ew, eb)

    for i, (N, K) in enumerate(((2048, 2048), (90, 1024))):     # one at a time: [M, 2048] fp64 operands are large
        c = WG(M, N, K, 1 + i, exact=False)
        ops.linear_wgrad(c.dy, c.x, c.dw, c.db, N, K, M=M)
        torch.cuda.synchronize()
        check("linear_wgrad", c)
        del c
    multi = [WG(M, N, K, 10 + i, ldx=96 if K == 89 else None, exact=False) for i, (_, N, K) in enumerate(c2_shapes(M))]
    ops.wgrad_multi([c.item() for c in multi], M)
    torch.cuda.synchronize()
    for c in multi:
        check("wgrad_multi", c)
    print(f"wgrad random M{M}: error / bound " + ", ".join(f"{k} {v:.3g}" for k, v in worst.items()))


# ------------------------------------------------------------------------------------------------------------
# the end of the training step: wgrad_multi -> norm_clip_adam, no synchronisation in between
# ------------------------------------------------------------------------------------------------------------
def test_wgrad_multi_then_norm_clip_adam(ops):
    """Integer gradients formed by rlppo_wgrad_multi in views of one gradient arena, then rlppo_norm_clip_adam enqueued
    right behind it on the same stream (the optimiser's prologue runs ahead of its griddepcontrol.wait), three steps
    with the arena zeroed before each: p, m, v, the squared norms and the step counts are bit-identical to three
    norm_clip_adam steps on an arena holding the exact gradients."""
    M = 3001
    shapes = c2_shapes(M)
    sizes = [N * K + N for _, N, K in shapes]
    total = sum(sizes)
    arena = f32_sentinel(total + 8)
    cs, off = [], 0
    for i, (_, N, K) in enumerate(shapes):
        c = WG(M, N, K, 50 + i, ldx=96 if K == 89 else None)
        c.dw = arena[off:off + N * K].view(N, K)
        c.db = arena[off + N * K:off + N * K + N]
        cs.append(c)
        off += N * K + N
    exact = torch.cat([torch.cat([(c.dy64.t() @ c.x64).flatten(), c.dy64.sum(0)]) for c in cs]).float()
    seg = [0, sum(sizes[:4]), total]
    g = torch.Generator(device=DEV).manual_seed(5)
    p0 = torch.randn(total, generator=g, device=DEV) * 0.05
    lr = torch.tensor([3e-4, 1e-4], device=DEV)
    runs = []
    for use_wgrad in (True, False):
        p, m, v = p0.clone(), torch.zeros_like(p0), torch.zeros_like(p0)
        sq, steps = torch.zeros(2, device=DEV), torch.zeros(2, dtype=torch.int64, device=DEV)
        grads = arena if use_wgrad else exact
        torch.cuda.synchronize()
        for _ in range(3):
            if use_wgrad:
                arena[:total].zero_()
                ops.wgrad_multi([c.item() for c in cs], M)
            ops.norm_clip_adam(p, grads, m, v, seg, sq, lr, steps)
        torch.cuda.synchronize()
        runs.append((p, m, v, sq, steps))
    assert torch.equal(bits(arena[:total]), bits(exact)), "wgrad_multi gradients are not exact"
    guard_intact(arena, total)
    for name, a, b in zip(("p", "m", "v", "sqnorm", "steps"), runs[0], runs[1]):
        assert torch.equal(a, b), name
    assert runs[0][4].tolist() == [3, 3]
