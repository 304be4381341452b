"""Helpers shared by the parity tests: tolerances, gradient capture, split-buffer views, and a host restatement of the
Philox4x32-10 stream every sampling kernel draws from."""
import numpy as np
import torch

DEV = "cuda:0"
SENTINEL = 0x7FC1          # a bf16 NaN: a stray write, or a read of unwritten padding, cannot go unnoticed


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64).ravel(), np.asarray(b, np.float64).ravel()
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def close(a, b, tol):
    """scale-aware tolerance of SURVEY.md 8(c): |a - b| <= tol * max(|b|, 1)."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return bool(np.all(np.abs(a - b) <= tol * np.maximum(np.abs(b), 1.0)))


def capture_steps(lr):
    """Post-clip gradients seen by Adam at every optimiser step (the golden scripts wrap optimizer.step the same way)."""
    from rlgym_ppo_b200 import ops
    captured = []
    orig = lr._optimizer_step

    def step():
        ops.grad_sqnorm(lr._grads, lr._seg, lr._sqnorm)
        gn = lr._sqnorm.sqrt().cpu().numpy()
        coef = np.minimum(1.0, 0.5 / (gn + 1e-6))
        gr = lr._grads.cpu().numpy().copy()
        n_p = int(lr._seg[1])
        gr[:n_p] *= coef[0]
        gr[n_p:] *= coef[1]
        captured.append(gr)
        orig()

    lr._optimizer_step = step
    lr.use_cuda_graph = False        # the hook reads tensors back, which a graph capture forbids
    return captured


def unflatten(lr, flat):
    shapes = [tuple(p.shape) for p in lr.policy.parameters()] + [tuple(p.shape) for p in lr.value_net.parameters()]
    out, off = [], 0
    for shp in shapes:
        n = int(np.prod(shp))
        out.append(flat[off:off + n].reshape(shp))
        off += n
    return out


# ---- split ("fp32" precision mode) buffers: value = part0 + part1 + part2, parts `pstride` columns apart -------------
def sentinel(rows, cols):
    return torch.full((rows, cols), SENTINEL, dtype=torch.int16, device=DEV).view(torch.bfloat16)


def bits(t):
    return t.view(torch.int16)


def recon(buf, parts, pstride, cols, rows=None):
    """fp64 sum of the parts of a split buffer (CPU), columns [0, cols)."""
    b = buf if rows is None else buf[rows]
    b = b.cpu()
    return sum(b[:, q * pstride:q * pstride + cols].double() for q in range(parts))


def split_rows(ops, x, parts, pstride, ld=None, rows=None):
    """f32 CPU rows -> split bf16 device buffer [rows, ld]."""
    n, w = x.shape
    rows = n if rows is None else rows
    buf = torch.zeros((rows, ld or parts * pstride), dtype=torch.bfloat16, device=DEV)
    ops.rows_split(x.to(DEV).contiguous(), buf, parts, pstride)
    return buf


# ---- Philox4x32-10 (Salmon et al., SC'11), as the kernels run it ---------------------------------------------------
M32 = 0xFFFFFFFF


def philox4x32_10(counter, key):
    """counter uint32 [..., 4], key uint32 [..., 2] (broadcast against each other) -> uint32 [..., 4].  The round
    function and Weyl constants of philox4x32_10 in csrc/heads.cu (mlp_tcgen05.cu and mlp_fused.cu carry copies)."""
    c = np.asarray(counter, dtype=np.uint32).astype(np.uint64)
    k = np.asarray(key, dtype=np.uint32).astype(np.uint64)
    c0, c1, c2, c3 = c[..., 0], c[..., 1], c[..., 2], c[..., 3]
    k0, k1 = k[..., 0], k[..., 1]
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c0, np.uint64(0xCD9E8D57) * c2        # 32 x 32 -> 64 bits, exact in uint64
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & np.uint64(M32),
                          (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & np.uint64(M32))
        k0 = (k0 + np.uint64(0x9E3779B9)) & np.uint64(M32)
        k1 = (k1 + np.uint64(0xBB67AE85)) & np.uint64(M32)
    return np.stack(np.broadcast_arrays(c0, c1, c2, c3), -1).astype(np.uint32)


def philox_uniform(r):
    """The kernels' uniform in [0, 1): the top 24 bits of a Philox word, (r >> 8) * 2^-24 (exact in f32)."""
    return (np.asarray(r, dtype=np.uint32) >> np.uint32(8)).astype(np.float64) * 2.0 ** -24


def philox_rows(seed, offset, rows, word2=0):
    """Philox words of rows 0..rows-1 of one launch: counter (ctr lo, ctr hi, word2, 0) with ctr = offset + row mod 2^64,
    key (seed lo, seed hi).  Returns uint32 [rows, 4]."""
    ctr = (int(offset) + np.arange(rows, dtype=object)) % (1 << 64)
    counter = np.zeros((rows, 4), dtype=np.uint32)
    counter[:, 0] = [int(x) & M32 for x in ctr]
    counter[:, 1] = [int(x) >> 32 for x in ctr]
    counter[:, 2] = word2
    key = np.array([int(seed) & M32, (int(seed) >> 32) & M32], dtype=np.uint32)
    return philox4x32_10(counter, key)
