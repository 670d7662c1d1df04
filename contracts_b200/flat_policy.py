"""The policy's flat input rows written by the feature-env and selfdrive steps (ssd_set_flat_policy_output).

A policy on these envs reads, per agent, the vector SeparateContractEnv builds (two_stage_train.py:113-121): the
features followed by [theta, 0] under a contract, the features alone without one, in float32 or a half type.  With
`policy_dtype=T` the env writes exactly those rows, `policy_obs` T [E*n, policy_width] (row e*n + a = agent a of env e),
with the values `torch.cat((obs, theta, 0), -1).to(torch.float32).to(T)` of the float64 rows, instead of float64 `obs`
— no second pass over the rows, and theta stays current through every call that changes it.
"""
import ctypes

import torch

from . import _lib


class FlatPolicyMixin:
    """policy_dtype for BatchedFeatureEnv and BatchedCarEnv.  The host classes provide _h, lib, E, n, device, contract
    and close()."""

    def _init_policy_output(self, policy_dtype, F):
        """Set the handle's observation form; returns True when the env writes the policy's rows (and keeps no `obs`)."""
        self.policy_dtype, self.policy_obs = policy_dtype, None
        self.policy_width = F + (2 if self.contract is not None else 0)
        if policy_dtype is None:
            return False
        try:
            code = _lib.policy_dtype_code(policy_dtype)
        except ValueError:
            self.close()
            raise
        self.policy_obs = torch.zeros((self.E * self.n, self.policy_width), dtype=policy_dtype, device=self.device)
        out = _lib.ssd_flat_policy_out(struct_size=ctypes.sizeof(_lib.ssd_flat_policy_out),
                                       dtype=code, obs_dev=self.policy_obs.data_ptr())
        _lib.check(self._h, self.lib.ssd_set_flat_policy_output(self._h, ctypes.byref(out)))
        return True

    @property
    def observation(self):
        """what reset / step return: `obs`, or `policy_obs` when the env writes the policy's rows"""
        return self.obs if self.policy_dtype is None else self.policy_obs

    def _obs_rows(self):
        """the observation rows checkpoint / restore carry: float64 [E, n, F], or T [E, n, policy_width] in policy mode"""
        return self.obs if self.policy_dtype is None else self.policy_obs.view(self.E, self.n, self.policy_width)
