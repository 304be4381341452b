"""Tensor-level wrappers over the C-ABI (one function per entry point of include/rlppo.h).

torch is used for device memory and streams only; every function enqueues hand-written kernels from
librlppo_b200.so on the current torch CUDA stream and returns without synchronising.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from ._lib import call, ptr, stream_ptr

BF16 = torch.bfloat16


def _cuda(t, dtype=None):
    assert t.is_cuda, "device tensor expected (no CPU fallback)"
    if dtype is not None:
        assert t.dtype == dtype, f"expected {dtype}, got {t.dtype}"
    return t


def pad8(n):
    return (int(n) + 7) // 8 * 8


# ---- GAE ------------------------------------------------------------------------------------------------
_gae_ws = {}


def _workspace(n, device):
    need = _lib.gae_workspace_bytes(n)
    key = (device.index if device.index is not None else torch.cuda.current_device())
    ws = _gae_ws.get(key)
    if ws is None or ws.numel() < need:
        ws = torch.empty(max(need, 1 << 16), dtype=torch.uint8, device=device)
        _gae_ws[key] = ws
    return ws


def gae_workspace(n, device):
    """A private scan workspace for n steps (callers that capture CUDA graphs must own theirs: the shared one is
    re-allocated when a longer rollout arrives)."""
    return torch.empty(max(_lib.gae_workspace_bytes(n), 1 << 12), dtype=torch.uint8, device=device)


def gae(rew, done, trunc, values, gamma, lmbda, ret_std=None, out=None, ret_head64=None, carry_in=None, ws=None):
    """compute_gae on device.  rew/done f32[n], trunc f32|f64[n], values f32[n+1], ret_std f32[1] tensor or
    None.  Returns (value_targets, advantages, returns) f32[n]."""
    n = rew.numel()
    _cuda(rew, torch.float32), _cuda(done, torch.float32), _cuda(values, torch.float32)
    assert values.numel() == n + 1 and done.numel() == n and trunc.numel() == n
    assert trunc.dtype in (torch.float32, torch.float64)
    for t in (rew, done, trunc, values):
        assert t.is_contiguous()
    if out is None:
        adv = torch.empty(n, dtype=torch.float32, device=rew.device)
        vt = torch.empty_like(adv)
        ret = torch.empty_like(adv)
    else:
        vt, adv, ret = out
    if n == 0:
        return vt, adv, ret
    if ws is None:
        ws = _workspace(n, rew.device)
    n_head = 0 if ret_head64 is None else min(ret_head64.numel(), n)
    call("rlppo_gae_f32", ptr(rew), ptr(done), ptr(trunc), int(trunc.dtype == torch.float64), ptr(values), n,
         float(gamma), float(lmbda), ptr(ret_std), ptr(adv), ptr(vt), ptr(ret), ptr(ret_head64), n_head,
         ptr(carry_in), ptr(ws), ws.numel(), stream_ptr(), work=("byte", 28 * n))
    return vt, adv, ret


def gae_chunk_summary(rew, done, trunc, values, gamma, lmbda, ret_std=None, out=None):
    n = rew.numel()
    if out is None:
        out = torch.empty(4, dtype=torch.float64, device=rew.device)
    ws = _workspace(n, rew.device)
    call("rlppo_gae_chunk_summary", ptr(rew), ptr(done), ptr(trunc), int(trunc.dtype == torch.float64), ptr(values),
         n, float(gamma), float(lmbda), ptr(ret_std), ptr(out), ptr(ws), ws.numel(), stream_ptr())
    return out


def gae_compose_carry(summaries, rank, world, out=None):
    """summaries f64 [world, 4] (all ranks' gae_chunk_summary) -> carry f64[2] for chunk `rank`."""
    assert summaries.dtype == torch.float64 and summaries.numel() == 4 * world and summaries.is_contiguous()
    if out is None:
        out = torch.empty(2, dtype=torch.float64, device=summaries.device)
    call("rlppo_gae_compose_carry", ptr(summaries), int(rank), int(world), ptr(out), stream_ptr())
    return out


# ---- Welford --------------------------------------------------------------------------------------------
def welford_update(mean, m2, count, samples, n, std_out=None, mean_out=None):
    dim = mean.numel()
    assert samples.dtype in (torch.float32, torch.float64) and count.dtype == torch.int64
    call("rlppo_welford_update", ptr(mean), ptr(m2), ptr(count), ptr(samples), int(samples.dtype == torch.float64),
         int(n), dim, ptr(std_out), ptr(mean_out), stream_ptr())


def welford_merge(mean, m2, count, others, n_others, stride_bytes, std_out=None, mean_out=None):
    """Fold n_others Welford states (blocks [count i64 | mean f32[dim] | m2 f32[dim] | ...], stride_bytes apart, starting
    at the device tensor `others`) into (mean, m2, count), in order (rlppo_welford_merge)."""
    assert count.dtype == torch.int64 and others.is_cuda and others.is_contiguous()
    assert others.numel() * others.element_size() >= int(n_others) * int(stride_bytes), "others too small"
    call("rlppo_welford_merge", ptr(mean), ptr(m2), ptr(count), ptr(others), int(stride_bytes), int(n_others),
         mean.numel(), ptr(std_out), ptr(mean_out), stream_ptr())


# ---- ring / gather --------------------------------------------------------------------------------------
def ring_append(ring, phys_first, src, n_rows, ring_bf16=None):
    cap = ring.shape[0]
    width = 1 if ring.dim() == 1 else ring.shape[1]
    ring_ld = 1 if ring.dim() == 1 else ring.stride(0)
    src_ld = 1 if src.dim() == 1 else src.stride(0)
    assert src.dtype in (torch.float32, torch.float64)
    call("rlppo_ring_append", ptr(ring), ring_ld, ptr(ring_bf16), 0 if ring_bf16 is None else ring_bf16.stride(0),
         cap, int(phys_first), ptr(src), int(src.dtype == torch.float64), src_ld, int(n_rows), width, stream_ptr(),
         work=("byte", int(n_rows) * width * (src.element_size() + 4 + (2 if ring_bf16 is not None else 0))))


def ring_append_fields(fields, capacity, phys_first, n_rows, state_dev=None):
    """fields: list of (ring, src, ring_bf16|None).  One launch for all of them.  With `state_dev` (int64[2] device
    tensor {start, size}) the position is read -- and advanced -- on the device and `phys_first` is ignored."""
    arr = (_lib.AppendField * len(fields))()
    nbytes = 0
    for a, (ring, src, rb) in zip(arr, fields):
        assert src.dtype in (torch.float32, torch.float64) and src.is_cuda
        a.ring, a.ring_ld = ring.data_ptr(), (1 if ring.dim() == 1 else ring.stride(0))
        a.ring_bf16, a.bf16_ld = (None, 0) if rb is None else (rb.data_ptr(), rb.stride(0))
        a.src, a.src_ld = src.data_ptr(), (1 if src.dim() == 1 else src.stride(0))
        a.src_is_f64 = int(src.dtype == torch.float64)
        a.width = 1 if ring.dim() == 1 else ring.shape[1]
        nbytes += int(n_rows) * (a.width * (src.element_size() + 4) + (0 if rb is None else 2 * rb.stride(0)))
    if state_dev is not None:
        assert state_dev.dtype == torch.int64 and state_dev.numel() == 2 and state_dev.is_cuda
        call("rlppo_ring_append_fields_dev", ctypes.cast(arr, ctypes.c_void_p), len(fields), int(capacity),
             ptr(state_dev), int(n_rows), stream_ptr(), work=("byte", nbytes))
        return
    call("rlppo_ring_append_fields", ctypes.cast(arr, ctypes.c_void_p), len(fields), int(capacity), int(phys_first),
         int(n_rows), stream_ptr(), work=("byte", nbytes))


def gather_batch(buf, idx, out_actions=None, out_logp=None, out_values=None, out_adv=None, out_states=None,
                 out_states_bf16=None):
    """buf: object with ring tensors (actions, log_probs, values, advantages, states[, states_bf16]),
    capacity and start.  idx int64 device tensor of LOGICAL indices."""
    B = idx.numel()
    sb = getattr(buf, "states_bf16", None)
    call("rlppo_gather_batch", ptr(buf.actions), ptr(buf.log_probs), ptr(buf.values), ptr(buf.advantages),
         ptr(buf.states), buf.states.stride(0) if buf.states is not None and buf.states.dim() == 2 else 1, ptr(sb),
         0 if sb is None else sb.stride(0), int(buf.obs_dim), int(buf.capacity), int(buf.start),
         ptr(getattr(buf, "start_dev", None)), ptr(idx), B,
         ptr(out_actions), ptr(out_logp), ptr(out_values), ptr(out_adv), ptr(out_states), ptr(out_states_bf16),
         stream_ptr(),
         work=("byte", 8 * B + 2 * B * (4 * sum(o is not None for o in (out_actions, out_logp, out_values, out_adv))
                                        + (4 * buf.obs_dim if out_states is not None else 0)
                                        + (2 * sb.stride(0) if out_states_bf16 is not None else 0))))


# ---- operand preparation ---------------------------------------------------------------------------------
def rows_to_bf16(src, dst, mean=None, std=None, clip=5.0, dst_f32=None):
    n_rows, width = src.shape
    assert dst.dtype == BF16 and dst.shape[0] >= n_rows
    call("rlppo_rows_to_bf16", ptr(src), src.stride(0), n_rows, width, ptr(mean), ptr(std), float(clip), ptr(dst),
         dst.stride(0), ptr(dst_f32), 0 if dst_f32 is None else dst_f32.stride(0), stream_ptr(),
         work=("byte", n_rows * (4 * width + 2 * dst.stride(0))))


def weight_to_bf16(w, wq, wt=None):
    out_f, in_f = w.shape
    assert w.is_contiguous() and wq.dtype == BF16
    call("rlppo_weight_to_bf16", ptr(w), out_f, in_f, ptr(wq), wq.stride(0), wq.shape[0], ptr(wt),
         0 if wt is None else wt.stride(0), 0 if wt is None else wt.shape[0], stream_ptr(),
         work=("byte", out_f * in_f * (4 + 2 + (2 if wt is not None else 0))))


# ---- split ("fp32" precision mode) operands: value = part0 + part1 + part2, parts `pstride` columns apart ---------
def pad64(n):
    return (int(n) + 63) // 64 * 64


def make_split(a_parts, b_parts, order, out_parts, a_pstride, b_pstride, out_pstride=0):
    """struct rlppo_split; kept alive by the caller for the duration of the call (ctypes.byref)."""
    sp = _lib.Split()
    sp.a_parts, sp.b_parts, sp.order, sp.out_parts = int(a_parts), int(b_parts), int(order), int(out_parts)
    sp.a_pstride, sp.b_pstride, sp.out_pstride = int(a_pstride), int(b_pstride), int(out_pstride)
    return sp


def _n_products(sp):
    return sum(1 for i in range(sp.a_parts) for j in range(sp.b_parts) if i + j < sp.order)


def _sp(sp):
    return None if sp is None else ctypes.byref(sp)


def rows_split(src, dst, parts, pstride, mean=None, std=None, clip=5.0):
    """f32 [n, width] -> `parts` bf16 parts side by side in dst [>= n, >= parts * pstride] (optionally standardised)."""
    n_rows, width = src.shape
    assert dst.dtype == BF16 and dst.shape[0] >= n_rows and src.dtype == torch.float32
    call("rlppo_rows_split_bf16", ptr(src), src.stride(0), n_rows, width, ptr(mean), ptr(std), float(clip), ptr(dst),
         dst.stride(0), int(parts), int(pstride), stream_ptr(), work=("byte", n_rows * (4 * width + 2 * parts * pstride)))


def weight_split(w, wq, q_parts, q_pstride, wt=None, t_parts=0, t_pstride=0):
    out_f, in_f = w.shape
    assert w.is_contiguous()
    call("rlppo_weight_split_bf16", ptr(w), out_f, in_f, ptr(wq), 0 if wq is None else wq.stride(0), int(q_parts),
         int(q_pstride), 0 if wq is None else wq.shape[0], ptr(wt), 0 if wt is None else wt.stride(0), int(t_parts),
         int(t_pstride), 0 if wt is None else wt.shape[0], stream_ptr(),
         work=("byte", out_f * in_f * (4 + 2 * q_parts + 2 * t_parts)))


# ---- tensor-core layers -------------------------------------------------------------------------------------
def linear_fwd(x, wq, bias, y, N, K, relu, M=None, split=None, bias_n=0):
    M = x.shape[0] if M is None else M
    if split is not None:
        work = ("flop", 2.0 * M * N * K, "mma_flop", 2.0 * M * N * K * _n_products(split),
                "byte", 2.0 * (M * K * split.a_parts + N * K * split.b_parts + M * N * split.out_parts))
    else:
        work = ("flop", 2.0 * M * N * K, "byte", 2.0 * (M * K + N * K + M * N))
    call("rlppo_linear_fwd", ptr(x), x.stride(0), ptr(wq), wq.stride(0), ptr(bias), int(bias_n), ptr(y), y.stride(0),
         int(M), int(N), int(K), int(bool(relu)), _sp(split), stream_ptr(), work=work)


def linear_dgrad(dy, wt, hprev, dx, N, K, M=None, db_below=None, split=None):
    """db_below (optional f32[K]): += column sums of dx, the bias gradient of the layer below (fused into the epilogue)."""
    M = dy.shape[0] if M is None else M
    call("rlppo_linear_dgrad", ptr(dy), dy.stride(0), ptr(wt), wt.stride(0), ptr(hprev),
         0 if hprev is None else hprev.stride(0), ptr(dx), dx.stride(0), ptr(db_below), int(M), int(N), int(K),
         _sp(split), stream_ptr(),
         work=("flop", 2.0 * M * N * K, "byte", 2.0 * (M * N + N * K + M * K * (2 if hprev is not None else 1))))


def linear_wgrad(dy, x, dw, db, N, K, M=None, split=None):
    M = dy.shape[0] if M is None else M
    a_parts, b_parts = (1, 1) if split is None else (split.a_parts, split.b_parts)
    call("rlppo_linear_wgrad", ptr(dy), dy.stride(0), ptr(x), x.stride(0), ptr(dw), dw.stride(0), ptr(db), int(M),
         int(N), int(K), _sp(split), stream_ptr(),
         work=("flop", 2.0 * M * N * K, "byte", 2.0 * M * (N * a_parts + K * b_parts) + 4.0 * N * K))


def wgrad_multi(items, M):
    """items: list of (dy, x, dw, N, K[, db]) -- all weight gradients of a step in one launch (<= 8 per call); db (optional)
    receives the column sums of dy, i.e. the Linear's bias gradient."""
    for i0 in range(0, len(items), 8):
        part = items[i0:i0 + 8]
        arr = (_lib.WgradItem * len(part))()
        flop = nbytes = 0.0
        for a, item in zip(arr, part):
            dy, x, dw, N, K = item[:5]
            db = item[5] if len(item) > 5 else None
            a.dy, a.lddy, a.x, a.ldx = dy.data_ptr(), dy.stride(0), x.data_ptr(), x.stride(0)
            a.dw, a.lddw, a.M, a.N, a.K = dw.data_ptr(), dw.stride(0), int(M), int(N), int(K)
            a.db = db.data_ptr() if db is not None else None
            flop += 2.0 * M * N * K
            nbytes += 2.0 * M * (dy.stride(0) + x.stride(0)) + 4.0 * N * K     # both bf16 operands read once, dW written
        call("rlppo_wgrad_multi", ctypes.cast(arr, ctypes.c_void_p), len(part), stream_ptr(),
             work=("flop", flop, "byte", nbytes))


def policy_head_sample(h, wq, bias, n_actions, K, M=None, u=None, seed=0, offset=0, deterministic=False,
                       actions_out=None, actions_i64_out=None, logp_out=None, probs_out=None, split=None):
    M = h.shape[0] if M is None else M
    call("rlppo_policy_head_sample", ptr(h), h.stride(0), ptr(wq), wq.stride(0), ptr(bias), int(M), int(n_actions),
         int(K), ptr(u), int(seed) & (2 ** 64 - 1), int(offset) & (2 ** 64 - 1), int(bool(deterministic)),
         ptr(actions_out), ptr(actions_i64_out), ptr(logp_out), ptr(probs_out), _sp(split), stream_ptr(),
         work=("flop", 2.0 * M * n_actions * K))


def policy_head_train(h, wq, bias, n_actions, K, actions, old_logp, adv, inv_batch, clip, ent_coef, dz, metrics,
                      logp_out=None, M=None, split=None):
    M = h.shape[0] if M is None else M
    call("rlppo_policy_head_train", ptr(h), h.stride(0), ptr(wq), wq.stride(0), ptr(bias), int(M), int(n_actions),
         int(K), ptr(actions), ptr(old_logp), ptr(adv), float(inv_batch), float(clip), float(ent_coef), ptr(dz),
         dz.stride(0), ptr(logp_out), ptr(metrics), _sp(split), stream_ptr(), work=("flop", 2.0 * M * n_actions * K))


def value_head(h, w, bias, K, values_out=None, targets=None, inv_batch=0.0, dh=None, dw=None, db=None, metrics=None,
               M=None, h_parts=1, h_pstride=0, dh_parts=1, dh_pstride=0):
    M = h.shape[0] if M is None else M
    if h_parts > 1 or dh_parts > 1:
        nbytes = M * K * 2 * (h_parts + (dh_parts if targets is not None else 0)) + 8 * M
    else:
        nbytes = M * K * 2 * (2 if targets is not None else 1) + 4 * M * (2 if targets is not None else 1)
    call("rlppo_value_head", ptr(h), h.stride(0), ptr(w), ptr(bias), int(M), int(K), ptr(values_out), ptr(targets),
         float(inv_batch), ptr(dh), 0 if dh is None else dh.stride(0), ptr(dw), ptr(db), ptr(metrics), int(h_parts),
         int(h_pstride), int(dh_parts), int(dh_pstride), stream_ptr(), work=("byte", nbytes))


# ---- the other two action heads (rlppo_head_*: per-row tails over the split logits of the last Linear) ----------------
def head_multi_discrete_train(z, z_parts, z_pstride, M, actions, old_logp, adv, inv_batch, clip, ent_coef, dz, dz_parts,
                              dz_pstride, dz_cols, metrics, logp_out=None):
    call("rlppo_head_multi_discrete_train", ptr(z), z.stride(0), int(z_parts), int(z_pstride), int(M), ptr(actions),
         actions.stride(0), ptr(old_logp), ptr(adv), float(inv_batch), float(clip), float(ent_coef), ptr(dz), dz.stride(0),
         int(dz_parts), int(dz_pstride), int(dz_cols), ptr(logp_out), ptr(metrics), stream_ptr(),
         work=("byte", M * (2 * 21 * z_parts + 2 * dz_cols * dz_parts + 4 * 11)))


def head_multi_discrete_sample(z, z_parts, z_pstride, M, actions_out, logp_out, u=None, seed=0, offset=0,
                               deterministic=False):
    call("rlppo_head_multi_discrete_sample", ptr(z), z.stride(0), int(z_parts), int(z_pstride), int(M), ptr(u),
         int(seed) & (2 ** 64 - 1), int(offset) & (2 ** 64 - 1), int(bool(deterministic)), ptr(actions_out),
         actions_out.stride(0), ptr(logp_out), stream_ptr(), work=("byte", M * (2 * 21 * z_parts + 4 * 9)))


def head_continuous_train(z, z_parts, z_pstride, M, n_act, var_min, var_max, actions, old_logp, adv, inv_batch, clip,
                          ent_coef, dz, dz_parts, dz_pstride, dz_cols, metrics, logp_out=None):
    call("rlppo_head_continuous_train", ptr(z), z.stride(0), int(z_parts), int(z_pstride), int(M), int(n_act),
         float(var_min), float(var_max), ptr(actions), actions.stride(0), ptr(old_logp), ptr(adv), float(inv_batch),
         float(clip), float(ent_coef), ptr(dz), dz.stride(0), int(dz_parts), int(dz_pstride), int(dz_cols), ptr(logp_out),
         ptr(metrics), stream_ptr(), work=("byte", M * (4 * n_act * z_parts + 2 * dz_cols * dz_parts + 4 * (n_act + 3))))


def head_continuous_sample(z, z_parts, z_pstride, M, n_act, var_min, var_max, actions_out, logp_out, normals=None, seed=0,
                           offset=0, deterministic=False):
    call("rlppo_head_continuous_sample", ptr(z), z.stride(0), int(z_parts), int(z_pstride), int(M), int(n_act),
         float(var_min), float(var_max), ptr(normals), int(seed) & (2 ** 64 - 1), int(offset) & (2 ** 64 - 1),
         int(bool(deterministic)), ptr(actions_out), actions_out.stride(0), ptr(logp_out), stream_ptr(),
         work=("byte", M * (4 * n_act * z_parts + 4 * (n_act + 1))))


# ---- wide discrete head (257..4096 actions): per-row kernels over the split logits of the last Linear ----------------
def _discrete_bytes(M, n_actions, z_parts, dz_cols=0, dz_parts=0):
    """HBM bytes of one pass: the logits once, d(logits) once, the per-row scalars."""
    return M * (2 * n_actions * z_parts + 2 * dz_cols * dz_parts + 12)


def head_discrete_sample(z, z_parts, z_pstride, M, n_actions, u=None, seed=0, offset=0, deterministic=False,
                         actions_out=None, actions_i64_out=None, logp_out=None, probs_out=None):
    nbytes = _discrete_bytes(M, n_actions, z_parts) + (4 * M * n_actions if probs_out is not None else 0)
    call("rlppo_head_discrete_sample", ptr(z), z.stride(0), int(z_parts), int(z_pstride), int(M), int(n_actions), ptr(u),
         int(seed) & (2 ** 64 - 1), int(offset) & (2 ** 64 - 1), int(bool(deterministic)), ptr(actions_out),
         ptr(actions_i64_out), ptr(logp_out), ptr(probs_out), stream_ptr(), work=("byte", nbytes))


def head_discrete_train(z, z_parts, z_pstride, M, n_actions, actions, old_logp, adv, inv_batch, clip, ent_coef, dz,
                        dz_parts, dz_pstride, dz_cols, metrics, logp_out=None):
    call("rlppo_head_discrete_train", ptr(z), z.stride(0), int(z_parts), int(z_pstride), int(M), int(n_actions),
         ptr(actions), ptr(old_logp), ptr(adv), float(inv_batch), float(clip), float(ent_coef), ptr(dz), dz.stride(0),
         int(dz_parts), int(dz_pstride), int(dz_cols), ptr(logp_out), ptr(metrics), stream_ptr(),
         work=("byte", _discrete_bytes(M, n_actions, z_parts, dz_cols, dz_parts)))


def head_discrete_backward(z, z_parts, z_pstride, M, n_actions, actions, d_logp, d_ent, d_probs, dz, dz_parts, dz_pstride,
                           dz_cols):
    """d_logp f32[M], d_ent f32[1], d_probs f32[M, n_actions]: device tensors or None."""
    nbytes = _discrete_bytes(M, n_actions, z_parts, dz_cols, dz_parts) + (4 * M * n_actions if d_probs is not None else 0)
    call("rlppo_head_discrete_backward", ptr(z), z.stride(0), int(z_parts), int(z_pstride), int(M), int(n_actions),
         ptr(actions), ptr(d_logp), ptr(d_ent), ptr(d_probs), ptr(dz), dz.stride(0), int(dz_parts), int(dz_pstride),
         int(dz_cols), stream_ptr(), work=("byte", nbytes))


# ---- backward of the heads for arbitrary upstream gradients (torch autograd through the modules) ---------------------
def policy_head_backward(h, wq, bias, n_actions, K, actions, d_logp, d_ent, d_probs, dz, M=None, split=None):
    """d_logp f32[M], d_ent f32[1], d_probs f32[M, n_actions]: device tensors or None."""
    M = h.shape[0] if M is None else M
    call("rlppo_policy_head_backward", ptr(h), h.stride(0), ptr(wq), wq.stride(0), ptr(bias), int(M), int(n_actions),
         int(K), ptr(actions), ptr(d_logp), ptr(d_ent), ptr(d_probs), ptr(dz), dz.stride(0), _sp(split), stream_ptr(),
         work=("flop", 2.0 * M * n_actions * K))


def head_multi_discrete_backward(z, z_parts, z_pstride, M, actions, d_logp, d_ent, dz, dz_parts, dz_pstride, dz_cols):
    call("rlppo_head_multi_discrete_backward", ptr(z), z.stride(0), int(z_parts), int(z_pstride), int(M), ptr(actions),
         0 if actions is None else actions.stride(0), ptr(d_logp), ptr(d_ent), ptr(dz), dz.stride(0), int(dz_parts),
         int(dz_pstride), int(dz_cols), stream_ptr(), work=("byte", M * (2 * 21 * z_parts + 2 * dz_cols * dz_parts + 4 * 9)))


def head_continuous_backward(z, z_parts, z_pstride, M, n_act, var_min, var_max, actions, d_logp, d_ent, d_mean, d_std,
                             dz, dz_parts, dz_pstride, dz_cols):
    call("rlppo_head_continuous_backward", ptr(z), z.stride(0), int(z_parts), int(z_pstride), int(M), int(n_act),
         float(var_min), float(var_max), ptr(actions), 0 if actions is None else actions.stride(0), ptr(d_logp),
         ptr(d_ent), ptr(d_mean), ptr(d_std), ptr(dz), dz.stride(0), int(dz_parts), int(dz_pstride), int(dz_cols),
         stream_ptr(), work=("byte", M * (4 * n_act * z_parts + 2 * dz_cols * dz_parts + 4 * (3 * n_act + 1))))


def value_head_backward(h, w, K, d_values, dh, dw, db, M=None, h_parts=1, h_pstride=0, dh_parts=1, dh_pstride=0):
    M = h.shape[0] if M is None else M
    call("rlppo_value_head_backward", ptr(h), h.stride(0), ptr(w), int(M), int(K), ptr(d_values), ptr(dh), dh.stride(0),
         ptr(dw), ptr(db), int(h_parts), int(h_pstride), int(dh_parts), int(dh_pstride), stream_ptr(),
         work=("byte", M * K * 2 * (h_parts + dh_parts) + 4 * M))


# ---- whole-network fused kernels --------------------------------------------------------------------------------
def _net_flops(net, M, n_out, train):
    dims = [net.in_dim] + [net.hidden[i] for i in range(net.n_hidden)]
    f = sum(2.0 * M * dims[i] * dims[i + 1] for i in range(len(dims) - 1)) + 2.0 * M * dims[-1] * n_out
    if train:   # + backward data path (all layers but the first)
        f += sum(2.0 * M * dims[i] * dims[i + 1] for i in range(1, len(dims) - 1)) + 2.0 * M * dims[-1] * n_out
    return f


def _net_bytes(net, M, n_out_pad, train, policy):
    """HBM bytes a fused launch has to move: x read once; training also writes every hidden activation, the head's
    d(logits) (policy) and every dL/dH as bf16 -- the operands of the weight-gradient GEMMs, which contract over ALL
    rows and therefore run as a second launch (DESIGN.md section 3)."""
    hid = [net.hidden[i] for i in range(net.n_hidden)]
    b = 2.0 * M * ((net.in_dim + 7) // 8 * 8)
    if train:
        b += 2.0 * M * (2 * sum(hid) - (0 if policy else hid[-1])) + (2.0 * M * n_out_pad if policy else 0.0) + 16.0 * M
    else:
        b += 8.0 * M
    return b


def policy_train_fused(net, x, M, n_actions, actions, old_logp, adv, inv_batch, clip, ent_coef, metrics, logp_out=None):
    call("rlppo_policy_train_fused", ctypes.byref(net), ptr(x), int(M), int(n_actions), ptr(actions), ptr(old_logp),
         ptr(adv), float(inv_batch), float(clip), float(ent_coef), ptr(logp_out), ptr(metrics), stream_ptr(),
         work=("flop", _net_flops(net, M, n_actions, True), "byte", _net_bytes(net, M, (n_actions + 7) // 8 * 8, True, True)))


def policy_value_train_fused(pnet, vnet, x, M, n_actions, actions, old_logp, adv, inv_batch, clip, ent_coef, w_head, targets,
                             gw_head, metrics, logp_out=None, values_out=None):
    """Both nets of a batch in one persistent launch (work items = (net, tile), policy tiles first)."""
    call("rlppo_policy_value_train_fused", ctypes.byref(pnet), ctypes.byref(vnet), ptr(x), int(M), int(n_actions),
         ptr(actions), ptr(old_logp), ptr(adv), float(inv_batch), float(clip), float(ent_coef), ptr(logp_out), ptr(w_head),
         ptr(targets), ptr(gw_head), ptr(values_out), ptr(metrics), stream_ptr(),
         work=("flop", _net_flops(pnet, M, n_actions, True) + _net_flops(vnet, M, 1, True),
               "byte", _net_bytes(pnet, M, (n_actions + 7) // 8 * 8, True, True) + _net_bytes(vnet, M, 0, True, False)))


def u64_add(counter, inc):
    """*counter += inc on the device (counter: int64[1] tensor); graph-capturable."""
    call("rlppo_u64_add", ptr(counter), int(inc), stream_ptr())


def policy_infer_fused(net, x, M, n_actions, u=None, seed=0, offset=0, deterministic=False, actions_out=None,
                       actions_i64_out=None, logp_out=None, offset_dev=None):
    call("rlppo_policy_infer_fused", ctypes.byref(net), ptr(x), int(M), int(n_actions), ptr(u), int(seed) & (2 ** 64 - 1),
         int(offset) & (2 ** 64 - 1), ptr(offset_dev), int(bool(deterministic)), ptr(actions_out), ptr(actions_i64_out),
         ptr(logp_out),
         stream_ptr(), work=("flop", _net_flops(net, M, n_actions, False), "byte", _net_bytes(net, M, 0, False, True)))


def value_train_fused(net, x, M, w_head, targets, inv_batch, gw_head, metrics, values_out=None):
    call("rlppo_value_train_fused", ctypes.byref(net), ptr(x), int(M), ptr(w_head), ptr(targets), float(inv_batch),
         ptr(gw_head), ptr(values_out), ptr(metrics), stream_ptr(),
         work=("flop", _net_flops(net, M, 1, True), "byte", _net_bytes(net, M, 0, True, False)))


def value_infer_fused(net, x, M, w_head, values_out):
    call("rlppo_value_infer_fused", ctypes.byref(net), ptr(x), int(M), ptr(w_head), ptr(values_out), stream_ptr(),
         work=("flop", _net_flops(net, M, 1, False), "byte", _net_bytes(net, M, 0, False, False)))


# ---- optimiser ------------------------------------------------------------------------------------------------
def _seg(seg_off):
    return np.ascontiguousarray(seg_off, dtype=np.int64)


def grad_sqnorm(grads, seg_off, sqnorm):
    so = _seg(seg_off)
    call("rlppo_grad_sqnorm", ptr(grads), so.ctypes.data, len(so) - 1, ptr(sqnorm), stream_ptr(),
         work=("byte", 4 * int(so[-1])))


def clip_adam(params, grads, m, v, seg_off, sqnorm, lr, step_count, max_norm=0.5, beta1=0.9, beta2=0.999, eps=1e-8,
              views=None):
    """views: optional ctypes array of _lib.Bf16View -- bf16 operands refreshed by the same launch."""
    so = _seg(seg_off)
    call("rlppo_clip_adam", ptr(params), ptr(grads), ptr(m), ptr(v), so.ctypes.data, len(so) - 1, ptr(sqnorm), ptr(lr),
         ptr(step_count), float(max_norm), float(beta1), float(beta2), float(eps),
         None if views is None else ctypes.cast(views, ctypes.c_void_p), 0 if views is None else len(views),
         stream_ptr(), work=("byte", 28 * int(so[-1])))


_nca_ws = {}


def norm_clip_adam(params, grads, m, v, seg_off, sqnorm_out, lr, step_count, max_norm=0.5, beta1=0.9, beta2=0.999,
                   eps=1e-8, views=None):
    """grad_sqnorm + clip_adam as one launch with a fixed-order (deterministic) norm; see rlppo_norm_clip_adam."""
    so = _seg(seg_off)
    ws = _nca_ws.get(params.device)
    if ws is None:
        ws = torch.zeros(int(_lib._lib.rlppo_norm_clip_adam_workspace_bytes()), dtype=torch.uint8, device=params.device)
        _nca_ws[params.device] = ws
    call("rlppo_norm_clip_adam", ptr(params), ptr(grads), ptr(m), ptr(v), so.ctypes.data, len(so) - 1, ptr(sqnorm_out),
         ptr(lr), ptr(step_count), float(max_norm), float(beta1), float(beta2), float(eps),
         None if views is None else ctypes.cast(views, ctypes.c_void_p), 0 if views is None else len(views),
         ptr(ws), ws.numel(), stream_ptr(), work=("byte", 32 * int(so[-1])))


def norm_clip_adam_peers(params, peer_grad_ptrs, peer_flag_ptrs, rank, gsum, m, v, seg_off, sqnorm_out, lr, step_count,
                         max_norm=0.5, beta1=0.9, beta2=0.999, eps=1e-8, views=None):
    """norm_clip_adam with the gradient all-reduce inside the launch (NVLink peer loads); see rlppo_norm_clip_adam_peers.
    peer_grad_ptrs / peer_flag_ptrs: device addresses (ints) of every rank's gradient arena / flag block as mapped here."""
    so = _seg(seg_off)
    ws = _nca_ws.get(params.device)
    if ws is None:
        ws = torch.zeros(int(_lib._lib.rlppo_norm_clip_adam_workspace_bytes()), dtype=torch.uint8, device=params.device)
        _nca_ws[params.device] = ws
    world = len(peer_grad_ptrs)
    gp = (ctypes.c_void_p * world)(*[int(x) for x in peer_grad_ptrs])
    fp = (ctypes.c_void_p * world)(*[int(x) for x in peer_flag_ptrs])
    call("rlppo_norm_clip_adam_peers", ptr(params), ctypes.cast(gp, ctypes.c_void_p), ctypes.cast(fp, ctypes.c_void_p),
         int(rank), world, ptr(gsum), ptr(m), ptr(v), so.ctypes.data, len(so) - 1, ptr(sqnorm_out), ptr(lr),
         ptr(step_count), float(max_norm), float(beta1), float(beta2), float(eps),
         None if views is None else ctypes.cast(views, ctypes.c_void_p), 0 if views is None else len(views),
         ptr(ws), ws.numel(), stream_ptr(), work=("byte", (32 + 4 * world) * int(so[-1])))


def norm_clip_adam_peers2(params, peer_grad_ptrs, peer_flag_ptrs, peer_red_ptrs, rank, m, v, seg_off, sqnorm_out, lr,
                          step_count, max_norm=0.5, beta1=0.9, beta2=0.999, eps=1e-8, views=None):
    """Two-shot form of norm_clip_adam_peers (rlppo_norm_clip_adam_peers2); the summed gradient ends up in
    this rank's reduced buffer (peer_red_ptrs[rank])."""
    so = _seg(seg_off)
    ws = _nca_ws.get(params.device)
    if ws is None:
        ws = torch.zeros(int(_lib._lib.rlppo_norm_clip_adam_workspace_bytes()), dtype=torch.uint8, device=params.device)
        _nca_ws[params.device] = ws
    world = len(peer_grad_ptrs)
    gp = (ctypes.c_void_p * world)(*[int(x) for x in peer_grad_ptrs])
    fp = (ctypes.c_void_p * world)(*[int(x) for x in peer_flag_ptrs])
    rp = (ctypes.c_void_p * world)(*[int(x) for x in peer_red_ptrs])
    call("rlppo_norm_clip_adam_peers2", ptr(params), ctypes.cast(gp, ctypes.c_void_p), ctypes.cast(fp, ctypes.c_void_p),
         ctypes.cast(rp, ctypes.c_void_p), int(rank), world, ptr(m), ptr(v), so.ctypes.data, len(so) - 1, ptr(sqnorm_out),
         ptr(lr), ptr(step_count), float(max_norm), float(beta1), float(beta2), float(eps),
         None if views is None else ctypes.cast(views, ctypes.c_void_p), 0 if views is None else len(views),
         ptr(ws), ws.numel(), stream_ptr(), work=("byte", 48 * int(so[-1])))


def sqdiff(a, b, seg_off, out):
    so = _seg(seg_off)
    call("rlppo_sqdiff", ptr(a), ptr(b), so.ctypes.data, len(so) - 1, ptr(out), stream_ptr(),
         work=("byte", 8 * int(so[-1])))
