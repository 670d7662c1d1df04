"""Checkpoint, restore and copy the complete state of batched envs (ssd_checkpoint_*, include/ssd_b200.h).

Every env's mutable state is one row of bytes.  Rows carry the global env ids they were taken from; since the random
stream of an env is keyed by (seed, global id), a row restored into the env with the same global id continues bit for
bit as if the run had never stopped, on any handle of the same configuration (resume, re-sharding), and a row restored
into another env continues there on THAT env's stream (branching).

    ck = env.checkpoint()                                  # EnvCheckpoint of every env (device tensors)
    torch.save(ck.state_dict(), path)
    ck = EnvCheckpoint.from_state_dict(torch.load(path))
    env.restore(ck)                                        # rows -> the envs with the same global ids
    env.restore(ck, envs=idx)                              # rows -> local envs idx
    env.copy_envs(src, dst)                                # branch envs src into envs dst
    EnvCheckpoint.cat([ck0, ck1]).select(first_env_id, num_envs)   # re-sharding
"""
import ctypes

import numpy as np
import torch

from . import _lib

_FIELDS = ("kind", "config_tag", "row_bytes", "seed", "env_ids", "rows", "obs")
_VERSION = 1


class EnvCheckpoint:
    """Rows of env state with their global ids.  kind: the env kind string; config_tag / row_bytes: the layout the rows
    were saved under (ssd_checkpoint_layout); seed: the handle's seed; env_ids int64 [count]; rows uint8 [count,
    row_bytes]; obs: the observation rows of those envs or None (uint8 [count, n, 15, 15, 3] for the grid worlds, T
    [count, n, 3, 15, 15] for a grid world with policy_dtype T, float64 [count, n, F | D] for the feature envs,
    selfdrive and a grid world with image_obs=False, T [count, n, policy_width] for those with policy_dtype T; uint8
    [count, H, W, 3] for a grid world with global_obs=True, T [count, 3, H, W] with policy_dtype T too).  The rows
    themselves do not depend on the observation form."""

    def __init__(self, kind, config_tag, row_bytes, seed, env_ids, rows, obs=None):
        self.kind, self.config_tag, self.row_bytes, self.seed = str(kind), int(config_tag), int(row_bytes), int(seed)
        self.env_ids = torch.as_tensor(env_ids, dtype=torch.int64)
        self.rows, self.obs = rows, obs
        if rows.dtype != torch.uint8 or rows.dim() != 2 or rows.shape[1] != self.row_bytes:
            raise ValueError("rows must be uint8 [count, %d], got %s %s" % (self.row_bytes, rows.dtype, tuple(rows.shape)))
        if self.env_ids.shape != (rows.shape[0],):
            raise ValueError("env_ids must be [count] = [%d], got %s" % (rows.shape[0], tuple(self.env_ids.shape)))
        if obs is not None and obs.shape[0] != rows.shape[0]:
            raise ValueError("obs must have one row per env (%d), got %s" % (rows.shape[0], tuple(obs.shape)))

    def __len__(self):
        return int(self.rows.shape[0])

    def __repr__(self):
        return "EnvCheckpoint(kind=%r, envs=%d, row_bytes=%d, config_tag=%016x, obs=%s)" % (
            self.kind, len(self), self.row_bytes, self.config_tag, self.obs is not None)

    def _like(self, env_ids, rows, obs):
        return EnvCheckpoint(self.kind, self.config_tag, self.row_bytes, self.seed, env_ids, rows, obs)

    def state_dict(self):
        """Plain types and CPU tensors only: loadable with torch.load's default weights_only=True."""
        return {"version": _VERSION, "kind": self.kind, "config_tag": self.config_tag, "row_bytes": self.row_bytes,
                "seed": self.seed, "env_ids": self.env_ids.cpu(), "rows": self.rows.cpu(),
                "obs": None if self.obs is None else self.obs.cpu()}

    @classmethod
    def from_state_dict(cls, d):
        if d.get("version") != _VERSION:
            raise ValueError("unknown EnvCheckpoint state_dict version %r" % (d.get("version"),))
        return cls(*(d[f] for f in _FIELDS))

    @classmethod
    def cat(cls, cks):
        """One checkpoint of the rows of several (e.g. one per rank of a sharded run); global ids must be distinct."""
        cks = list(cks)
        if not cks:
            raise ValueError("EnvCheckpoint.cat needs at least one checkpoint")
        c0 = cks[0]
        for c in cks[1:]:
            if (c.kind, c.config_tag, c.row_bytes, c.seed) != (c0.kind, c0.config_tag, c0.row_bytes, c0.seed):
                raise ValueError("EnvCheckpoint.cat: checkpoints of different configurations or seeds")
            if (c.obs is None) != (c0.obs is None):
                raise ValueError("EnvCheckpoint.cat: some checkpoints hold observations and some do not")
        dev = c0.rows.device
        ids = torch.cat([c.env_ids.to(dev) for c in cks])
        if torch.unique(ids).numel() != ids.numel():
            raise ValueError("EnvCheckpoint.cat: duplicate global env ids")
        obs = None if c0.obs is None else torch.cat([c.obs.to(dev) for c in cks])
        return c0._like(ids, torch.cat([c.rows.to(dev) for c in cks]), obs)

    def select(self, first_env_id, num_envs):
        """The rows of global ids first_env_id .. first_env_id + num_envs - 1 (the range of one handle), in id order."""
        ids = self.env_ids
        keep = torch.nonzero((ids >= int(first_env_id)) & (ids < int(first_env_id) + int(num_envs))).reshape(-1)
        keep = keep[torch.argsort(ids[keep])]
        k = keep.to(self.rows.device)
        return self._like(ids[keep], self.rows.index_select(0, k), None if self.obs is None else self.obs.index_select(0, k))


def _index_tensor(envs, E, device, what):
    """int32 CUDA tensor of local env indices, checked to lie in [0, E) and (dst) to be distinct."""
    idx = torch.as_tensor(np.asarray(envs) if not torch.is_tensor(envs) else envs).reshape(-1).to(device=device, dtype=torch.int64)
    if idx.numel() and (int(idx.min()) < 0 or int(idx.max()) >= E):
        raise ValueError("%s: env indices must lie in [0, %d)" % (what, E))
    return idx


class CheckpointMixin:
    """checkpoint / restore / copy_envs for BatchedGridEnv, BatchedFeatureEnv and BatchedCarEnv.  The host classes
    provide _h, lib, E, device, kind, seed, first_env_id and obs (or _obs_rows())."""

    def _obs_rows(self):
        return self.obs

    def checkpoint_layout(self):
        lay = _lib.ssd_checkpoint_layout()
        _lib.check(self._h, self.lib.ssd_checkpoint_get_layout(self._h, ctypes.byref(lay)))
        return lay

    def checkpoint(self, envs=None, with_obs=True):
        """EnvCheckpoint of the envs `envs` (local indices; None: every env) on this device, taken on the current stream
        without a host synchronisation when envs is None."""
        lay = self.checkpoint_layout()
        if envs is None:
            idx, count = None, self.E
            local = torch.arange(self.E, device=self.device, dtype=torch.int64)
        else:
            local = _index_tensor(envs, self.E, self.device, "checkpoint")
            idx, count = local.to(torch.int32), int(local.numel())
        rows = torch.empty((count, int(lay.row_bytes)), dtype=torch.uint8, device=self.device)
        _lib.check(self._h, self.lib.ssd_checkpoint_save(self._h, None if idx is None else ctypes.c_void_p(idx.data_ptr()),
                                                         count, ctypes.c_void_p(rows.data_ptr()), self._stream()))
        obs = None
        if with_obs:
            rows_obs = self._obs_rows()
            obs = rows_obs.clone() if envs is None else rows_obs.index_select(0, local)
        return EnvCheckpoint(self.kind, lay.config_tag, lay.row_bytes, self.seed, local + self.first_env_id, rows, obs)

    def restore(self, ck, envs=None):
        """Load the rows of `ck`: into the local envs with the same global ids (envs None: same seed required), or into
        the local envs `envs` (one per row, distinct), which continue on their own random streams.  The observation
        rows, when the checkpoint holds them, are written to self.obs (a grid world's policy_image in policy mode; its
        policy_contract rows follow the loaded theta).  Raises SsdError on a configuration mismatch and naming the rows
        that failed validation (they are not written; the others are); ValueError when the checkpoint's observation rows
        are of another form than the env's (with_obs=False checkpoints restore across forms)."""
        lay = self.checkpoint_layout()
        if ck.config_tag != lay.config_tag or ck.row_bytes != lay.row_bytes:
            raise _lib.SsdError("restore: checkpoint of another configuration (kind %r, config_tag %016x, row_bytes %d; this "
                                "%s handle has config_tag %016x, row_bytes %d)" % (ck.kind, ck.config_tag, ck.row_bytes,
                                                                                 self.kind, lay.config_tag, lay.row_bytes))
        own = self._obs_rows()
        if ck.obs is not None and (ck.obs.dtype != own.dtype or tuple(ck.obs.shape[1:]) != tuple(own.shape[1:])):
            raise ValueError("restore: the checkpoint's observation rows are %s %s, this env's are %s %s (another observation "
                             "form; restore a checkpoint taken with with_obs=False)" % (ck.obs.dtype, tuple(ck.obs.shape[1:]),
                                                                                      own.dtype, tuple(own.shape[1:])))
        if envs is None:
            if ck.seed != self.seed:
                raise _lib.SsdError("restore: checkpoint seed %d != handle seed %d (pass envs= to branch across seeds)"
                                    % (ck.seed, self.seed))
            dst = ck.env_ids.to(self.device) - self.first_env_id
            if dst.numel() and (int(dst.min()) < 0 or int(dst.max()) >= self.E):
                raise ValueError("restore: global env ids outside this handle's range [%d, %d)" % (self.first_env_id,
                                                                                                  self.first_env_id + self.E))
        else:
            dst = _index_tensor(envs, self.E, self.device, "restore")
            if dst.numel() != len(ck):
                raise ValueError("restore: %d destination envs for %d rows" % (dst.numel(), len(ck)))
        if torch.unique(dst).numel() != dst.numel():
            raise ValueError("restore: duplicate destination envs")
        count = int(dst.numel())
        if count == 0:
            return
        rows = ck.rows.to(self.device).contiguous()
        idx = dst.to(torch.int32)
        ok = torch.empty((count,), dtype=torch.uint8, device=self.device)
        _lib.check(self._h, self.lib.ssd_checkpoint_load(self._h, ctypes.c_uint64(lay.config_tag), ctypes.c_void_p(idx.data_ptr()),
                                                         count, ctypes.c_void_p(rows.data_ptr()), ctypes.c_void_p(ok.data_ptr()),
                                                         self._stream()))
        good = ok.bool()
        all_ok = bool(good.all())                    # the one synchronisation of a restore
        if ck.obs is not None:
            obs = ck.obs.to(self.device)
            if all_ok:
                own[dst] = obs
            else:
                own[dst[good]] = obs[good]
        if not all_ok:
            bad = torch.nonzero(~good).reshape(-1).cpu().tolist()
            raise _lib.SsdError("restore: rows %s failed validation (corrupt or not saved from this configuration); they were "
                                "not loaded" % bad)

    def copy_envs(self, src, dst):
        """Branch: envs `src` are copied into envs `dst` (local indices, same length; the two may overlap), which continue
        on their own random streams.  Observations are copied too."""
        self.restore(self.checkpoint(envs=src), envs=dst)
