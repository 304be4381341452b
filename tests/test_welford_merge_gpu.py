"""rlppo_welford_merge against the host merge it replaces: WelfordRunningStat.increment_from_serialized_other (the
reference's Chan formula, running_stats.py:71-98) applied to the other states one after another must give the same bits
for mean, m2 and count, and std / mean the same bits as the host properties."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _state(dim, count, rng):
    """(count, mean f32[dim], m2 f32[dim]) of a state that has seen `count` samples."""
    mean = np.zeros(dim, np.float32)
    m2 = np.zeros(dim, np.float32)
    if count:
        mean = (rng.randn(dim) * 3 + rng.randn()).astype(np.float32)
        # zero variance in some dimensions: std must come out 1 there
        m2 = (rng.rand(dim) * count * (rng.rand(dim) > 0.1)).astype(np.float32)
    return count, mean, m2


def _blocks(others, dim, pad):
    """The others as device blocks [count i64 | mean f32[dim] | m2 f32[dim] | pad bytes], side by side (the layout of
    WelfordRunningStat's device state, followed by the data-parallel exchange's tail)."""
    stride = 8 + 8 * dim + pad
    raw = np.zeros(len(others) * stride + 8, np.uint8)
    for i, (count, mean, m2) in enumerate(others):
        b = raw[i * stride:(i + 1) * stride]
        b[0:8].view(np.int64)[0] = count
        b[8:8 + 8 * dim].view(np.float32)[:] = np.concatenate([mean, m2])
    return torch.from_numpy(raw).to(DEV), stride


def _device(state):
    count, mean, m2 = state
    dim = len(mean)
    return {"count": torch.tensor([count], dtype=torch.int64, device=DEV), "mean": torch.from_numpy(mean.copy()).to(DEV),
            "m2": torch.from_numpy(m2.copy()).to(DEV), "std": torch.full((dim,), -1.0, device=DEV),
            "mean_out": torch.full((dim,), -1.0, device=DEV)}


def _merge(d, blocks, n, stride):
    from rlgym_ppo_b200 import ops
    ops.welford_merge(d["mean"], d["m2"], d["count"], blocks, n, stride, d["std"], d["mean_out"])


def _host_replay(base, others):
    from rlgym_ppo_b200.util import WelfordRunningStat
    ref = WelfordRunningStat(len(base[1]))
    ref.count, ref.running_mean, ref.running_variance = base[0], base[1].copy(), base[2].copy()
    for count, mean, m2 in others:
        ref.increment_from_serialized_other(mean.tolist() + m2.tolist() + [count])
    return ref


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _check(d, ref):
    torch.cuda.synchronize()
    assert int(d["count"].item()) == ref.count
    assert np.array_equal(_bits(d["mean"].cpu().numpy()), _bits(ref.running_mean))
    assert np.array_equal(_bits(d["m2"].cpu().numpy()), _bits(ref.running_variance))
    assert np.array_equal(_bits(d["std"].cpu().numpy()), _bits(ref.std))
    assert np.array_equal(_bits(d["mean_out"].cpu().numpy()), _bits(ref.mean))


# (base count, other counts): small counts, an empty base, empty others, counts above 2^24 (not exact in f32)
SCENARIOS = {
    "one": (37, [5]),
    "eight": (1000, [3, 1, 50, 7, 2, 900, 11, 4]),
    "empty_base": (0, [6, 9, 2]),
    "empty_others": (12, [0, 4, 0, 0, 8]),
    "all_empty": (0, [0, 0]),
    "single_sample": (0, [1, 1]),
    "big_counts": ((1 << 24) + 3, [(1 << 25) + 1, 7, (1 << 24) + 5, 123_456_789_012]),
}


@pytest.mark.parametrize("dim", [1, 12, 89, 2000])
@pytest.mark.parametrize("scenario", sorted(SCENARIOS))
def test_merge_matches_host_replay(dim, scenario):
    base_count, counts = SCENARIOS[scenario]
    rng = np.random.RandomState(dim * 31 + len(counts))
    base = _state(dim, base_count, rng)
    others = [_state(dim, c, rng) for c in counts]
    blocks, stride = _blocks(others, dim, pad=40)
    d = _device(base)
    _merge(d, blocks, len(others), stride)
    _check(d, _host_replay(base, others))


def test_merge_device_on_running_stat():
    """WelfordRunningStat.merge_device folds device_block() layouts of other statistics in place."""
    from rlgym_ppo_b200.util import WelfordRunningStat
    rng = np.random.RandomState(3)
    stats = []
    for count in (20, 0, 7, 300):
        st = WelfordRunningStat(12, device=DEV)
        if count:
            st.increment(rng.randn(count, 12) * 2 + 1, count)
        stats.append(st)
    base, others = stats[0], stats[1:]
    host = [(o.count, o.running_mean.copy(), o.running_variance.copy()) for o in others]
    ref = _host_replay((base.count, base.running_mean.copy(), base.running_variance.copy()), host)
    stride = others[0].device_block().numel()
    blocks = torch.cat([o.device_block() for o in others])
    base.merge_device(blocks, len(others), stride)
    assert base.count == ref.count and np.array_equal(_bits(base.running_mean), _bits(ref.running_mean))
    assert np.array_equal(_bits(base.running_variance), _bits(ref.running_variance))
    assert np.array_equal(_bits(base.device_std().cpu().numpy()), _bits(ref.std))


def test_merge_under_graph_capture():
    """The call enqueues device work only: captured into a CUDA graph and replayed, it merges like an eager call."""
    dim, rng = 89, np.random.RandomState(5)
    base = _state(dim, 40, rng)
    others = [_state(dim, c, rng) for c in (3, 0, 17)]
    blocks, stride = _blocks(others, dim, pad=0)
    d = _device(base)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            _merge(d, blocks, len(others), stride)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    assert int(d["count"].item()) == 40          # capturing does not run the kernel
    graph.replay()
    _check(d, _host_replay(base, others))
    empty = _device(_state(dim, 0, rng))
    _merge(empty, blocks, 0, stride)              # no others: the state stays empty, std ones, mean zeros
    _check(empty, _host_replay(_state(dim, 0, rng), []))
