"""WelfordRunningStat with its state in HBM (replaces rlgym_ppo/util/running_stats.py).

The sequential Welford update (running_stats.py:37-46) runs in rlppo_welford_update, bit-faithful to the
reference's rounding (f32 state, f64 intermediates for f64 samples), so the return-normalisation scale that the
GAE kernel reads (`device_std()`, learner.py:356) never leaves the device.  The public attributes
(`running_mean`, `running_variance`, `count`, `mean`, `std`) and the serialisers keep the reference's types and
JSON layout (running_stats.py:100-137, BOOK_KEEPING_VARS.json); they read the device state back on demand.
"""
import json
import os

import numpy as np
import torch

from .. import _lib, ops


class WelfordRunningStat(object):
    def __init__(self, shape, device=None):
        self.ones = np.ones(shape=shape, dtype=np.float32)
        self.zeros = np.zeros(shape=shape, dtype=np.float32)
        self.shape = shape
        self._dim = int(np.prod(shape))
        self._h_mean = np.zeros(shape=shape, dtype=np.float32)
        self._h_m2 = np.zeros(shape=shape, dtype=np.float32)
        self._h_count = 0
        self._device = device
        self._d = None             # device state (lazy)
        self._host_is_newer = True
        self._dev_is_newer = False

    # ---- device state ---------------------------------------------------------------------------------------
    def _dev(self):
        if self._d is None:
            _lib.require_device()
            dev = torch.device(self._device if self._device is not None else "cuda:%d" % torch.cuda.current_device())
            # one contiguous allocation [count i64 | mean | m2 | std | mean_out] so the whole state is ONE broadcast
            n = self._dim
            raw = torch.zeros(8 + 16 * n, dtype=torch.uint8, device=dev)
            f = raw[8:].view(torch.float32)
            self._d = {"raw": raw, "count": raw[0:8].view(torch.int64), "mean": f[0:n], "m2": f[n:2 * n],
                       "std": f[2 * n:3 * n], "mean_out": f[3 * n:4 * n]}
            self._d["std"].fill_(1.0)
        return self._d

    def _push(self):
        d = self._dev()
        if self._host_is_newer:
            d["mean"].copy_(torch.from_numpy(np.ascontiguousarray(self._h_mean, dtype=np.float32).reshape(-1)))
            d["m2"].copy_(torch.from_numpy(np.ascontiguousarray(self._h_m2, dtype=np.float32).reshape(-1)))
            d["count"].fill_(int(self._h_count))
            ops.welford_update(d["mean"], d["m2"], d["count"], d["mean"], 0, d["std"], d["mean_out"])  # n=0: std only
            self._host_is_newer = False
        return d

    def _pull(self):
        if self._dev_is_newer:
            d = self._d
            self._h_mean = d["mean"].cpu().numpy().reshape(self.shape).copy()
            self._h_m2 = d["m2"].cpu().numpy().reshape(self.shape).copy()
            self._h_count = int(d["count"].item())
            self._dev_is_newer = False

    def broadcast_(self, src=0, group=None):
        """Make every rank's statistics those of rank `src` (device to device over NCCL, no host round trip).  Used by
        the sharded data-parallel learner: the reference updates its return statistics from the first 150 returns of
        ONE rollout (learner.py:368-372); with one rollout per rank that is rank 0's, and every rank must normalise
        rewards with the same scale."""
        import torch.distributed as dist
        d = self._push()
        dist.broadcast(d["raw"], src=src, group=group)
        self._dev_is_newer = True

    def device_block(self):
        """The device state as one uint8 block [count i64 | mean f32[dim] | m2 f32[dim] | std | mean_out], the layout
        merge_device reads."""
        return self._push()["raw"]

    def merge_device(self, blocks, n, stride_bytes):
        """Fold n device blocks (device_block layouts, stride_bytes apart in the tensor `blocks`) into these statistics in
        order: increment_from_serialized_other applied to each, bit for bit, without leaving the device."""
        d = self._push()
        ops.welford_merge(d["mean"], d["m2"], d["count"], blocks, n, stride_bytes, d["std"], d["mean_out"])
        self._dev_is_newer = True

    def copy_device_(self, other):
        """Make these statistics a copy of `other`'s (same dim), device to device."""
        self._push()["raw"].copy_(other.device_block())
        self._dev_is_newer = True

    def device_std(self):
        """f32[dim] device tensor holding `std` (running_stats.py:60-69); no host synchronisation."""
        return self._push()["std"]

    def device_mean(self):
        return self._push()["mean_out"]

    # ---- reference attributes ---------------------------------------------------------------------------------
    @property
    def running_mean(self):
        self._pull()
        return self._h_mean

    @running_mean.setter
    def running_mean(self, v):
        self._pull()
        self._h_mean = v
        self._host_is_newer = True

    @property
    def running_variance(self):
        self._pull()
        return self._h_m2

    @running_variance.setter
    def running_variance(self, v):
        self._pull()
        self._h_m2 = v
        self._host_is_newer = True

    @property
    def count(self):
        self._pull()
        return self._h_count

    @count.setter
    def count(self, v):
        self._pull()
        self._h_count = v
        self._host_is_newer = True

    # ---- updates (running_stats.py:30-46) -----------------------------------------------------------------------
    def increment(self, samples, num):
        if num > 1:
            self.increment_device(samples, num)
        else:
            self.update(samples)

    def update(self, sample):
        if type(sample) == dict:
            sample = sample["frame"]
        self.increment_device(np.asarray(sample).reshape(1, -1) if not isinstance(sample, torch.Tensor)
                              else sample.reshape(1, -1), 1)

    def increment_device(self, samples, num):
        """`num` sequential updates from samples[0:num] (numpy / list / device tensor, f32 or f64)."""
        d = self._push()
        if isinstance(samples, torch.Tensor) and samples.is_cuda:
            s = samples
            if s.dtype not in (torch.float32, torch.float64):
                s = s.to(torch.float32)
        else:
            a = np.asarray(samples[:num] if not isinstance(samples, np.ndarray) else samples[:num])
            if a.dtype not in (np.float32, np.float64):
                a = a.astype(np.float64)     # python floats / ints promote like `sample - running_mean` would
            s = torch.from_numpy(np.ascontiguousarray(a)).to(d["mean"].device)
        s = s.contiguous()
        assert s.numel() >= num * self._dim, "not enough samples"
        ops.welford_update(d["mean"], d["m2"], d["count"], s, num, d["std"], d["mean_out"])
        self._dev_is_newer = True

    def reset(self):
        self.__init__(self.shape, self._device)

    @property
    def mean(self):
        if self.count < 2:
            return self.zeros
        return self.running_mean

    @property
    def std(self):
        if self.count < 2:
            return self.ones
        var = self.running_variance / (self.count - 1)
        var = np.where(var == 0, 1.0, var)
        return np.sqrt(var)

    # ---- merge / (de)serialisation: host-side bookkeeping, the reference's formulas and layouts (:71-137) ----------
    def increment_from_serialized_other(self, serialized_other):
        n = int(np.prod(self.shape))
        other_mean = np.asarray(serialized_other[:n], dtype=np.float32).reshape(self.running_mean.shape)
        other_var = np.asarray(serialized_other[n:-1], dtype=np.float32).reshape(self.running_variance.shape)
        other_count = serialized_other[-1]
        if other_count == 0:
            return
        count = self.count + other_count
        mean_delta = other_mean - self.running_mean
        mean_delta_squared = mean_delta * mean_delta
        combined_mean = (self.count * self.running_mean + other_count * other_mean) / count
        combined_variance = self.running_variance + other_var + mean_delta_squared * self.count * other_count / count
        self.running_mean = combined_mean
        self.running_variance = combined_variance
        self.count = count

    def serialize(self):
        return self.running_mean.ravel().tolist() + self.running_variance.ravel().tolist() + [self.count]

    def deserialize(self, other):
        self.reset()
        n = int(np.prod(self.shape))
        self.running_mean = np.reshape(other[:n], self.shape)
        self.running_variance = np.reshape(other[n:-1], self.shape)
        self.count = other[-1]

    def to_json(self):
        return {"mean": self.running_mean.ravel().tolist(),
                "var": self.running_variance.ravel().tolist(),
                "shape": np.shape(self.running_mean),
                "count": self.count}

    def from_json(self, other_json):
        shape = other_json["shape"]
        # the reference's loader builds WelfordRunningStat(1) and lets from_json reshape it (learner.py:536-537)
        new_shape = tuple(shape) if len(shape) != 1 else int(shape[0])
        if int(np.prod(shape)) != self._dim:
            self.__init__(new_shape, self._device)
        self.count = other_json["count"]
        self.running_mean = np.asarray(other_json["mean"]).reshape(shape)
        self.running_variance = np.asarray(other_json["var"]).reshape(shape)
        print(F"LOADED RUNNING STATS FROM JSON | Mean: {self.running_mean} | Variance: {self.running_variance} | Count: {self.count}")

    def save(self, directory):
        full_path = os.path.join(directory, "RUNNING_STATS.json")
        with open(full_path, 'w') as f:
            json.dump(obj=self.to_json(), fp=f, indent=4)

    def load(self, directory):
        full_path = os.path.join(directory, "RUNNING_STATS.json")
        with open(full_path, 'r') as f:
            self.from_json(dict(json.load(f)))
