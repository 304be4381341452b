"""ctypes binding of librlppo_b200.so (include/rlppo.h).

There is no CPU fallback: importing this module without the built library raises, and every compute entry
point returns RLPPO_ERR_DEVICE (raised here as RuntimeError) when no sm_100 device is current.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# RLPPO_LIB_PATH: another build of the same library (kernel A/B runs inside one GPU session); never a fallback
LIB_PATH = os.environ.get("RLPPO_LIB_PATH") or os.path.join(_HERE, "librlppo_b200.so")

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python -m rlgym_ppo_b200.build` (nvcc, sm_100a). "
        "rlgym_ppo_b200 has no CPU or PyTorch fallback for its kernels."
    )

_lib = ctypes.CDLL(LIB_PATH)

_P = ctypes.c_void_p
_I = ctypes.c_int
_L = ctypes.c_int64
_D = ctypes.c_double
_F = ctypes.c_float
_U64 = ctypes.c_uint64
_SZ = ctypes.c_size_t

_SIGS = {
    "rlppo_version": ([], _I),
    "rlppo_last_error": ([], ctypes.c_char_p),
    "rlppo_device_check": ([], _I),
    "rlppo_gae_workspace_bytes": ([_L], _SZ),
    "rlppo_gae_f32": ([_P, _P, _P, _I, _P, _L, _D, _D, _P, _P, _P, _P, _P, _L, _P, _P, _SZ, _P], _I),
    "rlppo_gae_chunk_summary": ([_P, _P, _P, _I, _P, _L, _D, _D, _P, _P, _P, _SZ, _P], _I),
    "rlppo_gae_compose_carry": ([_P, _I, _I, _P, _P], _I),
    "rlppo_welford_update": ([_P, _P, _P, _P, _I, _L, _I, _P, _P, _P], _I),
    "rlppo_welford_merge": ([_P, _P, _P, _P, _L, _I, _I, _P, _P, _P], _I),
    "rlppo_ring_append": ([_P, _L, _P, _L, _L, _L, _P, _I, _L, _L, _I, _P], _I),
    "rlppo_ring_append_fields": ([_P, _I, _L, _L, _L, _P], _I),
    "rlppo_ring_append_fields_dev": ([_P, _I, _L, _P, _L, _P], _I),
    "rlppo_gather_batch": ([_P, _P, _P, _P, _P, _L, _P, _L, _I, _L, _L, _P, _P, _L, _P, _P, _P, _P, _P, _P, _P], _I),
    "rlppo_host_permutation": ([_P, _P, _L, _P], _I),
    "rlppo_rows_to_bf16": ([_P, _L, _L, _I, _P, _P, _F, _P, _L, _P, _L, _P], _I),
    "rlppo_weight_to_bf16": ([_P, _I, _I, _P, _L, _I, _P, _L, _I, _P], _I),
    "rlppo_linear_fwd": ([_P, _L, _P, _L, _P, _I, _P, _L, _L, _I, _I, _I, _P, _P], _I),
    "rlppo_linear_dgrad": ([_P, _L, _P, _L, _P, _L, _P, _L, _P, _L, _I, _I, _P, _P], _I),
    "rlppo_linear_wgrad": ([_P, _L, _P, _L, _P, _L, _P, _L, _I, _I, _P, _P], _I),
    "rlppo_wgrad_multi": ([_P, _I, _P], _I),
    "rlppo_policy_head_sample": ([_P, _L, _P, _L, _P, _L, _I, _I, _P, _U64, _U64, _I, _P, _P, _P, _P, _P, _P], _I),
    "rlppo_policy_head_train": ([_P, _L, _P, _L, _P, _L, _I, _I, _P, _P, _P, _F, _F, _F, _P, _L, _P, _P, _P, _P], _I),
    "rlppo_value_head": ([_P, _L, _P, _P, _L, _I, _P, _P, _F, _P, _L, _P, _P, _P, _I, _L, _I, _L, _P], _I),
    "rlppo_rows_split_bf16": ([_P, _L, _L, _I, _P, _P, _F, _P, _L, _I, _L, _P], _I),
    "rlppo_weight_split_bf16": ([_P, _I, _I, _P, _L, _I, _L, _I, _P, _L, _I, _L, _I, _P], _I),
    "rlppo_head_multi_discrete_train": ([_P, _L, _I, _L, _L, _P, _L, _P, _P, _F, _F, _F, _P, _L, _I, _L, _I, _P, _P, _P], _I),
    "rlppo_head_multi_discrete_sample": ([_P, _L, _I, _L, _L, _P, _U64, _U64, _I, _P, _L, _P, _P], _I),
    "rlppo_head_continuous_train": ([_P, _L, _I, _L, _L, _I, _F, _F, _P, _L, _P, _P, _F, _F, _F, _P, _L, _I, _L, _I, _P,
                                     _P, _P], _I),
    "rlppo_head_continuous_sample": ([_P, _L, _I, _L, _L, _I, _F, _F, _P, _U64, _U64, _I, _P, _L, _P, _P], _I),
    "rlppo_policy_head_backward": ([_P, _L, _P, _L, _P, _L, _I, _I, _P, _P, _P, _P, _P, _L, _P, _P], _I),
    "rlppo_head_multi_discrete_backward": ([_P, _L, _I, _L, _L, _P, _L, _P, _P, _P, _L, _I, _L, _I, _P], _I),
    "rlppo_head_continuous_backward": ([_P, _L, _I, _L, _L, _I, _F, _F, _P, _L, _P, _P, _P, _P, _P, _L, _I, _L, _I, _P],
                                       _I),
    "rlppo_value_head_backward": ([_P, _L, _P, _L, _I, _P, _P, _L, _P, _P, _I, _L, _I, _L, _P], _I),
    "rlppo_policy_train_fused": ([_P, _P, _L, _I, _P, _P, _P, _F, _F, _F, _P, _P, _P], _I),
    "rlppo_policy_infer_fused": ([_P, _P, _L, _I, _P, _U64, _U64, _P, _I, _P, _P, _P, _P], _I),
    "rlppo_u64_add": ([_P, _U64, _P], _I),
    "rlppo_value_train_fused": ([_P, _P, _L, _P, _P, _F, _P, _P, _P, _P], _I),
    "rlppo_policy_value_train_fused": ([_P, _P, _P, _L, _I, _P, _P, _P, _F, _F, _F, _P, _P, _P, _P, _P, _P, _P], _I),
    "rlppo_value_infer_fused": ([_P, _P, _L, _P, _P, _P], _I),
    "rlppo_grad_sqnorm": ([_P, _P, _I, _P, _P], _I),
    "rlppo_clip_adam": ([_P, _P, _P, _P, _P, _I, _P, _P, _P, _D, _D, _D, _D, _P, _I, _P], _I),
    "rlppo_norm_clip_adam_workspace_bytes": ([], ctypes.c_size_t),
    "rlppo_norm_clip_adam": ([_P, _P, _P, _P, _P, _I, _P, _P, _P, _D, _D, _D, _D, _P, _I, _P, ctypes.c_size_t, _P], _I),
    "rlppo_peer_flag_bytes": ([], ctypes.c_size_t),
    "rlppo_norm_clip_adam_peers": ([_P, _P, _P, _I, _I, _P, _P, _P, _P, _I, _P, _P, _P, _D, _D, _D, _D, _P, _I, _P,
                                    ctypes.c_size_t, _P], _I),
    "rlppo_norm_clip_adam_peers2": ([_P, _P, _P, _P, _I, _I, _P, _P, _P, _I, _P, _P, _P, _D, _D, _D, _D, _P, _I, _P,
                                     ctypes.c_size_t, _P], _I),
    "rlppo_sqdiff": ([_P, _P, _P, _I, _P, _P], _I),
    "rlppo_head_discrete_sample": ([_P, _L, _I, _L, _L, _I, _P, _U64, _U64, _I, _P, _P, _P, _P, _P], _I),
    "rlppo_head_discrete_train": ([_P, _L, _I, _L, _L, _I, _P, _P, _P, _F, _F, _F, _P, _L, _I, _L, _I, _P, _P, _P], _I),
    "rlppo_head_discrete_backward": ([_P, _L, _I, _L, _L, _I, _P, _P, _P, _P, _P, _L, _I, _L, _I, _P], _I),
}

EXPORTED = tuple(_SIGS)


class AppendField(ctypes.Structure):
    """struct rlppo_append_field."""
    _fields_ = [("ring", _P), ("ring_ld", _L), ("ring_bf16", _P), ("bf16_ld", _L), ("src", _P), ("src_ld", _L),
                ("src_is_f64", ctypes.c_int32), ("width", ctypes.c_int32)]


class Split(ctypes.Structure):
    """struct rlppo_split: split bf16 operands of the "fp32" precision mode."""
    _fields_ = [("a_parts", ctypes.c_int32), ("b_parts", ctypes.c_int32), ("order", ctypes.c_int32),
                ("out_parts", ctypes.c_int32), ("a_pstride", _L), ("b_pstride", _L), ("out_pstride", _L)]


class WgradItem(ctypes.Structure):
    """struct rlppo_wgrad_item."""
    _fields_ = [("dy", _P), ("lddy", _L), ("x", _P), ("ldx", _L), ("dw", _P), ("lddw", _L), ("M", _L),
                ("N", ctypes.c_int32), ("K", ctypes.c_int32), ("db", _P)]


class Bf16View(ctypes.Structure):
    """struct rlppo_bf16_view."""
    _fields_ = [("offset", _L), ("out_f", ctypes.c_int32), ("in_f", ctypes.c_int32), ("wq", _P), ("wq_ld", _L),
                ("wt", _P), ("wt_ld", _L)]


class FusedNet(ctypes.Structure):
    """struct rlppo_fused_net (include/rlppo.h)."""
    _fields_ = [("n_hidden", _I), ("in_dim", _I), ("in_ld", _L), ("hidden", _I * 4),
                ("wq", _P * 5), ("wq_ld", _L * 5), ("wt", _P * 5), ("wt_ld", _L * 5),
                ("bias", _P * 5), ("gbias", _P * 5), ("h", _P * 4), ("h_ld", _L * 4),
                ("dh", _P * 4), ("dh_ld", _L * 4), ("dz", _P), ("dz_ld", _L)]

for _name, (_args, _res) in _SIGS.items():
    _fn = getattr(_lib, _name)  # AttributeError here = header and library disagree
    _fn.argtypes = _args
    _fn.restype = _res


class RlppoError(RuntimeError):
    pass


def last_error():
    return _lib.rlppo_last_error().decode("utf-8", "replace")


def _check(rc, name):
    if rc != 0:
        raise RlppoError(f"{name} failed ({rc}): {last_error()}")


def ptr(t):
    """Device (or host) pointer of a tensor, None -> NULL."""
    if t is None:
        return None
    return ctypes.c_void_p(t.data_ptr())


def stream_ptr():
    """The torch current stream as a cudaStream_t (so kernels order with torch ops and graph capture)."""
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


CALLS = 0          # C-ABI compute calls made so far (each enqueues at least one kernel)
_TIMING = None     # None, or a list of (name, work, start_event, end_event) while per-call timing is on


def call(name, *args, work=None):
    """Invoke a C-ABI entry point.  `work` = (kind, amount[, kind, amount]): the call's algorithmic flops ("flop") and /
    or HBM bytes ("byte"), recorded only while timing_begin() is active (bench.py's roofline pass)."""
    global CALLS
    CALLS += 1
    if _TIMING is None:
        _check(getattr(_lib, name)(*args), name)
        return
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # The stream is kept busy (a ~150 us device-side spin) while the host prepares the launch (tensor-map encoding, argument
    # checks: 20-30 us for the fused kernels): the start event then fires with the kernel already queued behind it, and the
    # interval is the kernel's duration instead of host preparation + kernel.
    torch.cuda._sleep(300_000)
    e0.record()
    rc = getattr(_lib, name)(*args)
    e1.record()
    _check(rc, name)
    _TIMING.append((name, work, e0, e1))


def timing_begin():
    global _TIMING
    _TIMING = []


def timing_end():
    """Stops per-call timing; returns {name: {"calls", "ms", "flop", "byte"}} measured with CUDA events on the
    launching stream."""
    global _TIMING
    rec, _TIMING = _TIMING, None
    torch.cuda.synchronize()
    out = {}
    for name, work, e0, e1 in rec:
        d = out.setdefault(name, {"calls": 0, "ms": 0.0, "flop": 0.0, "byte": 0.0})
        d["calls"] += 1
        d["ms"] += e0.elapsed_time(e1)
        if work is not None:
            for i in range(0, len(work), 2):
                d[work[i]] = d.get(work[i], 0.0) + float(work[i + 1])
    return out


def require_device():
    """Raise unless the current CUDA device can run the sm_100a kernels."""
    if not torch.cuda.is_available():
        raise RlppoError("rlgym_ppo_b200 needs a CUDA device (B200, sm_100); there is no CPU fallback")
    _check(_lib.rlppo_device_check(), "rlppo_device_check")


def version():
    return _lib.rlppo_version()


def gae_workspace_bytes(n):
    return int(_lib.rlppo_gae_workspace_bytes(int(n)))


def host_permutation_raw(key, pos, n, out=None):
    """The same draw on raw MT19937 state (uint32[624] array, int position): returns (perm, key_after, pos_after).
    Touches no Python-level RandomState, releases the GIL: safe to run on a worker thread."""
    import numpy as np

    key = np.ascontiguousarray(key, dtype=np.uint32).copy()
    p = np.asarray([pos], dtype=np.int32)
    if out is None:
        out = np.empty(int(n), dtype=np.int64)
    rc = _lib.rlppo_host_permutation(key.ctypes.data_as(_P), p.ctypes.data_as(_P), int(n), out.ctypes.data_as(_P))
    _check(rc, "rlppo_host_permutation")
    return out, key, int(p[0])


def host_permutation(rng, n):
    """np.random.RandomState.permutation(n), bit-exact, through the C implementation; advances `rng`."""
    import numpy as np

    st = rng.get_state()
    key = np.ascontiguousarray(st[1], dtype=np.uint32).copy()
    pos = np.asarray([st[2]], dtype=np.int32)
    out = np.empty(int(n), dtype=np.int64)
    rc = _lib.rlppo_host_permutation(key.ctypes.data_as(_P), pos.ctypes.data_as(_P), int(n), out.ctypes.data_as(_P))
    _check(rc, "rlppo_host_permutation")
    rng.set_state((st[0], key, int(pos[0]), st[3], st[4]))
    return out
