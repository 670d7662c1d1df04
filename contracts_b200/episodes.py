"""Per-episode metrics of a vectorised sampler, logged by the device (ssd_set_episode_log, include/ssd_b200.h).

What the reference's MetricsCallback (utils/logger_utils.py:126-151) copies from `env.metrics` at the end of every episode
(apples eaten, dirt cleaned, transfers and, for episodes that reach the horizon, equality / sustainability /
transfer_equality / transfer_sustainability: cleanup_new.py:422-445, two_stage_train.py:92-99) exists only on the device
and is zeroed by the reset that starts the next episode.  While an `EpisodeLog` is set on a batch, every kernel that
resets an env appends that env's finished episode to a ring buffer on the device — resets, auto-resets inside or behind a
step, inside a CUDA graph too — and the host drains it whenever it likes:

    log = EpisodeLog(batch)                        # capacity 2 E records by default (480 bytes each)
    batch.set_episode_log(log)
    ... steps with auto_reset=True, graph replays ...
    rec = log.drain()                              # numpy arrays of the new records, sorted by (env_id, episode)
    for m in log.metrics(rec): callback(m)         # the drop-in class's `metrics` dict at each episode's last step

Records carry the global env id (first_env_id + i), so the logs of several ranks combine by concatenation.
"""
import ctypes

import numpy as np
import torch

from . import _lib

RECORD_BYTES = 480
RECORD_DTYPE = np.dtype({"names": ["env_id", "episode", "t", "ended", "theta", "pad", "metrics"],
                         "formats": [np.uint32, np.uint32, np.int32, np.uint32, np.float64, np.float64,
                                     (np.float64, _lib.METRIC_STRIDE)],
                         "offsets": [0, 4, 8, 12, 16, 24, 32], "itemsize": RECORD_BYTES})
_FEATURE_KINDS = ("cleanup", "harvest")


class EpisodeLog:
    """The record buffer (uint8 [capacity, 480], device) and the append counter (int64 [1], device) of one batch's episode
    log.  `batch` is any of the batched envs (grid, feature, selfdrive); set the log with `batch.set_episode_log(log)`."""

    def __init__(self, batch, capacity=None):
        capacity = 2 * batch.E if capacity is None else int(capacity)
        if not 1 <= capacity < 2 ** 31:
            raise ValueError("capacity must be in [1, 2^31), got %d" % capacity)
        self.batch, self.capacity = batch, capacity
        self.records = torch.zeros((capacity, RECORD_BYTES), dtype=torch.uint8, device=batch.device)
        self.count = torch.zeros((1,), dtype=torch.int64, device=batch.device)
        self._host = None               # pinned [8 + capacity * 480] bytes: the counter, then the ring
        self._drained = 0               # counter value at the last drain

    def _struct(self):
        return _lib.ssd_episode_log(struct_size=ctypes.sizeof(_lib.ssd_episode_log), capacity=self.capacity,
                                    records_dev=self.records.data_ptr(), count_dev=self.count.data_ptr())

    def drain(self):
        """The records appended since the last drain, as numpy arrays sorted by (env_id, episode): env_id uint32,
        episode uint32, t int32, ended bool, theta float64, metrics float64 [R, 56]; plus `lost`, the number of records
        that were overwritten before they could be drained (more than `capacity` appended since the last drain).
        Enqueues the copies on the batch's current stream and synchronises it once."""
        if self._host is None:
            self._host = torch.empty((8 + self.capacity * RECORD_BYTES,), dtype=torch.uint8).pin_memory()
        host = self._host
        host[:8].copy_(self.count.view(torch.uint8), non_blocking=True)
        host[8:].copy_(self.records.view(-1), non_blocking=True)
        torch.cuda.current_stream(self.batch.device).synchronize()
        buf = host.numpy()
        count = int(buf[:8].view(np.int64)[0])
        first = max(self._drained, count - self.capacity)
        lost = first - self._drained
        self._drained = count
        ring = buf[8:].view(RECORD_DTYPE)
        recs = ring[np.arange(first, count, dtype=np.int64) % self.capacity]
        recs = recs[np.lexsort((recs["episode"], recs["env_id"]))]
        return {"env_id": recs["env_id"].copy(), "episode": recs["episode"].copy(), "t": recs["t"].copy(),
                "ended": recs["ended"] != 0, "theta": recs["theta"].copy(), "metrics": recs["metrics"].copy(), "lost": lost}

    def metrics(self, records):
        """Per record of `records` (what drain() returned), the dict the single-env drop-in class's `metrics` property
        returns at that episode's last step — equality / sustainability (and transfer_* with a contract) for the episodes
        that reached the horizon."""
        from .environments.feature_envs import feature_metrics
        from .environments.gridworld import grid_metrics
        b = self.batch
        out = []
        for raw, ended in zip(records["metrics"], records["ended"]):
            if b.kind in ("cleanup_new", "harvest_new"):
                out.append(grid_metrics(b.kind, raw, b.n, bool(ended), contract=b.contract is not None,
                                        float_rewards=b.inequity_averse_reward))
            elif b.kind in _FEATURE_KINDS:
                out.append(feature_metrics(b.kind, raw, b.n, bool(ended), contract=b.contract is not None))
            else:
                out.append({"transfers": float(raw[0])})
        return out


class EpisodeLogMixin:
    """set_episode_log shared by the batched envs (ssd_set_episode_log serves every env kind)."""

    def set_episode_log(self, log):
        """log: an EpisodeLog of this batch, or None to switch logging off.  While set, every reset of an env whose
        episode it replaces appends one record (see EpisodeLog)."""
        if log is not None and log.batch is not self:
            raise ValueError("the EpisodeLog belongs to another batch")
        self._episode_log = log                          # keep its buffers alive while the library holds their addresses
        s = log._struct() if log is not None else None
        _lib.check(self._h, self.lib.ssd_set_episode_log(self._h, ctypes.byref(s) if s is not None else None))
