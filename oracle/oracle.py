"""ctypes front-end of the C oracle (`oracle/ssd_oracle.c`).

TEST INFRASTRUCTURE (oracle/): used by tests/, bench.py's cpu_baseline / `--impl reference`
leg and `__graft_entry__.smoke()` only — never by the product path.
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libssd_oracle.so")
_LIB = None

KIND = {"cleanup": 0, "harvest": 1}
CONTRACT = {None: 0, "none": 0, "CleanupContract": 1, "HarvestFeaturemodLocalContract": 2}
METRIC_STRIDE = 8 + 6 * 8
SOURCES = ("ssd_oracle.c", "selfdrive_oracle.c", "features_oracle.c")


def build(force=False):
    """Compile the oracle with the system gcc (the image's $CC has no OpenMP runtime)."""
    srcs = [os.path.join(_HERE, f) for f in SOURCES]
    if not force and os.path.exists(_SO) and all(os.path.getmtime(_SO) >= os.path.getmtime(s) for s in srcs):
        return _SO
    os.makedirs(os.path.dirname(_SO), exist_ok=True)
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    base = [cc, "-O2", "-std=c11", "-ffp-contract=off", "-fPIC", "-shared", "-o", _SO] + srcs + ["-lm"]
    try:
        subprocess.run(base[:4] + ["-fopenmp"] + base[4:], check=True, capture_output=True)
    except (subprocess.CalledProcessError, FileNotFoundError):
        subprocess.run(base, check=True)
    return _SO


def lib():
    global _LIB
    if _LIB is None:
        build()
        L = ctypes.CDLL(_SO)
        vp, i32, u32, f64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint32, ctypes.c_double
        L.oracle_create.restype = vp
        L.oracle_create.argtypes = [i32, i32, i32, i32, i32, ctypes.c_char_p, i32, i32, f64, f64, f64, u32, u32]
        L.oracle_destroy.argtypes = [vp]
        L.oracle_reset.argtypes = [vp, vp, vp, vp]
        L.oracle_step.argtypes = [vp] * 9
        L.oracle_get_state.argtypes = [vp] * 6
        L.oracle_set_state.argtypes = [vp] * 6
        L.oracle_get_metrics.argtypes = [vp, vp]
        L.oracle_feature_dim.argtypes = [vp]
        L.oracle_negotiate.argtypes = [vp, vp, vp, vp]
        L.oracle_set_reward_shaping.argtypes = [vp, i32, f64, f64]
        L.oracle_global_view.argtypes = [vp, vp]
        L.oracle_render.argtypes = [vp, vp]
        L.oracle_set_num_threads.argtypes = [i32]
        L.feat_oracle_create.restype = vp
        L.feat_oracle_create.argtypes = [i32, i32, i32, i32, i32, ctypes.c_char_p, i32, i32, f64, f64, f64, u32, u32]
        L.feat_oracle_destroy.argtypes = [vp]
        L.feat_oracle_dim.argtypes = [vp]
        L.feat_oracle_reset.argtypes = [vp] * 4
        L.feat_oracle_step.argtypes = [vp] * 8
        L.feat_oracle_step_skip.argtypes = [vp] * 9
        L.feat_oracle_get_metrics.argtypes = [vp, vp]
        L.feat_oracle_get_state.argtypes = [vp] * 6
        L.car_oracle_create.restype = vp
        L.car_oracle_create.argtypes = [i32, i32, i32, f64, f64, f64, f64, f64, f64, f64, u32, u32]
        L.car_oracle_destroy.argtypes = [vp]
        L.car_oracle_obs_dim.argtypes = [vp]
        L.car_oracle_reset.argtypes = [vp] * 4
        L.car_oracle_step.argtypes = [vp] * 8
        L.car_oracle_step_skip.argtypes = [vp] * 9
        L.car_oracle_get_state.argtypes = [vp] * 6
        L.car_oracle_set_theta.argtypes = [vp, vp]
        L.oracle_philox4x32_10.argtypes = [vp, vp, vp]
        _LIB = L
    return _LIB


def set_num_threads(n):
    """Threads of the oracle's OpenMP loops over envs; returns the count in effect (1 without OpenMP)."""
    return int(lib().oracle_set_num_threads(int(n)))


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _skip_bytes(skip, E):
    s = np.ascontiguousarray(skip, dtype=np.uint8).reshape(-1)
    if s.shape[0] != E:
        raise ValueError(f"skip has {s.shape[0]} entries for {E} envs")
    return s


def philox4x32_10(ctr, key):
    c = np.asarray(ctr, dtype=np.uint32).copy()
    k = np.asarray(key, dtype=np.uint32).copy()
    out = np.zeros(4, dtype=np.uint32)
    lib().oracle_philox4x32_10(_p(c), _p(k), _p(out))
    return out


class GridOracle:
    """E independent cleanup_new / harvest_new envs (+ optional subgame contract wrapper)."""

    def __init__(self, kind, num_envs, num_agents, ascii_map, horizon=1000, contract=None,
                 theta_low=0.0, theta_high=None, null_prob=0.0, seed=73907, first_env_id=0,
                 use_collective_reward=False, inequity_averse_reward=False, alpha=0.0, beta=0.0):
        self.kind = kind
        self.E, self.n = int(num_envs), int(num_agents)
        self.H, self.W = len(ascii_map), len(ascii_map[0])
        if theta_high is None:      # gym Box stores float32 bounds (contract_list.py:20,43)
            theta_high = float(np.float32(0.2)) if kind == "cleanup" else float(np.float32(10.0))
        flat = "".join(ascii_map).encode("ascii")
        self._h = lib().oracle_create(KIND[kind], self.E, self.n, self.H, self.W, flat, int(horizon),
                                      CONTRACT[contract], float(theta_low), float(theta_high),
                                      float(null_prob), int(seed) & 0xFFFFFFFF, int(first_env_id))
        if not self._h:
            raise ValueError("oracle_create failed (bad sizes / map)")
        self.F = lib().oracle_feature_dim(self._h)
        self.episode = np.full(self.E, -1, dtype=np.int64)
        mode = (1 if use_collective_reward else 0) | (2 if inequity_averse_reward else 0)
        if mode and lib().oracle_set_reward_shaping(self._h, mode, float(alpha), float(beta)) != 0:
            raise ValueError("inequity_averse_reward needs more than one agent (map_env.py:294)")

    def __del__(self):
        if getattr(self, "_h", None) and lib is not None:        # (module globals are gone at interpreter shutdown)
            try:
                lib().oracle_destroy(self._h)
            except Exception:
                pass
            self._h = None

    def reset(self, mask=None):
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        sel = np.ones(self.E, bool) if m is None else m.astype(bool)
        self.episode[sel] += 1
        ep = self.episode.astype(np.uint32)
        obs = np.zeros((self.E, self.n, 15, 15, 3), dtype=np.uint8)
        lib().oracle_reset(self._h, _p(m), _p(ep), _p(obs))
        return obs

    def step(self, actions, want_features=True):
        a = np.ascontiguousarray(actions, dtype=np.int32).reshape(self.E, self.n)
        E, n = self.E, self.n
        out = {
            "obs": np.zeros((E, n, 15, 15, 3), np.uint8), "rew": np.zeros((E, n)),
            "base_rew": np.zeros((E, n)), "transfers": np.zeros((E, n)),
            "info": np.zeros((E, n, 4), np.int32), "done": np.zeros(E, np.uint8),
            "feature_obs": np.zeros((E, n, self.F)) if want_features else None,
        }
        lib().oracle_step(self._h, _p(a), _p(out["obs"]), _p(out["rew"]), _p(out["base_rew"]),
                          _p(out["transfers"]), _p(out["info"]), _p(out["feature_obs"]), _p(out["done"]))
        return out

    def get_state(self):
        E, n = self.E, self.n
        st = {"map": np.zeros((E, self.H, self.W), np.uint8), "pos": np.zeros((E, n, 2), np.int32),
              "ori": np.zeros((E, n), np.int32), "t": np.zeros(E, np.int32), "theta": np.zeros(E)}
        lib().oracle_get_state(self._h, _p(st["map"]), _p(st["pos"]), _p(st["ori"]), _p(st["t"]), _p(st["theta"]))
        return st

    def set_state(self, map=None, pos=None, ori=None, t=None, theta=None):
        def prep(x, dt, shape):
            return None if x is None else np.ascontiguousarray(np.broadcast_to(np.asarray(x, dtype=dt), shape))
        E, n = self.E, self.n
        m, p, o = prep(map, np.uint8, (E, self.H, self.W)), prep(pos, np.int32, (E, n, 2)), prep(ori, np.int32, (E, n))
        tt, th = prep(t, np.int32, (E,)), prep(theta, np.float64, (E,))
        lib().oracle_set_state(self._h, _p(m), _p(p), _p(o), _p(tt), _p(th))

    def negotiate(self, proposals, accept):
        """Agreement stage (two_stage_train.py:266-281): returns the uint8 [E] accept decisions; sets theta."""
        p = np.ascontiguousarray(np.broadcast_to(np.asarray(proposals, dtype=np.float64), (self.E,)))
        a = np.ascontiguousarray(np.broadcast_to(np.asarray(accept, dtype=np.float64), (self.E, self.n)))
        dec = np.zeros(self.E, np.uint8)
        lib().oracle_negotiate(self._h, _p(p), _p(a), _p(dec))
        return dec

    def metrics_raw(self):
        out = np.zeros((self.E, METRIC_STRIDE))
        lib().oracle_get_metrics(self._h, _p(out))
        return out

    def global_view(self):
        """MapEnv.global_view() (map_env.py:394-395) of every env: uint8 [E, H, W, 3]."""
        out = np.zeros((self.E, self.H, self.W, 3), np.uint8)
        lib().oracle_global_view(self._h, _p(out))
        return out

    def render(self):
        """MapEnv.full_map_to_colors() (map_env.py:389-392) of every env, beams of the last step included: uint8 [E, H, W, 3]."""
        out = np.zeros((self.E, self.H, self.W, 3), np.uint8)
        lib().oracle_render(self._h, _p(out))
        return out

    def set_theta(self, theta):
        self.set_state(theta=theta)


def concatenated_obs(obs):
    """JointEnv `concatenated_obs` (two_stage_train.py:527-533,604-609): np.concatenate of the agents' windows
    along the channel axis.  obs [E, n, 15, 15, 3] -> [E, 15, 15, 3 n]."""
    return np.concatenate([obs[:, a] for a in range(obs.shape[1])], axis=-1)


def solver_candidates(seed, env_id, episode, low, high, num_samples):
    """NegotiationSolver.negotiate (two_stage_train.py:705-746), the candidate contracts of one env: the null contract
    `contract_space.low` followed by `contract_param_space.sample()` x num_samples.  gym (pinned 0.21.0, not vendored by
    the reference) implements Box.sample for a bounded box as `np_random.uniform(low, high).astype(float32)`, the uniform
    evaluated in float64 as low + (high - low) * u; u is the env's Philox draw (site SOLVER, index i) at t = 0."""
    from . import philox as px
    out = [np.float64(low)]
    for i in range(num_samples):
        u = px.draws_f64(seed, env_id, episode, 0, px.SITE_SOLVER, 0, i)[0]
        out.append(np.float64(np.float32(np.float64(low) + (np.float64(high) - np.float64(low)) * u)))
    return np.array(out)


def solver_choose(params, vals, rule):
    """NegotiationSolver.compute_best_param (two_stage_train.py:748-776) for one env, restated with the reference's own
    list operations.  params [1 + S], vals [1 + S, n] (row 0 = the null contract).  Returns (parameter, index)."""
    all_vals = [tuple(np.float64(x) for x in row) for row in vals]
    all_params = list(range(len(params)))

    def best_max(vs, ps):
        welfares = []
        for k in vs:
            w = 0
            for x in k:                    # sum(k.values()): left to right from 0
                w = w + x
            welfares.append(w)
        return ps[int(np.argmax(welfares))]

    if rule == "max":
        idx = best_max(all_vals, all_params)
    elif rule == "majority":
        default = all_vals[0]
        acc_vals, acc_params = [default], [all_params[0]]
        for k1 in all_vals[1:]:
            accepted = sum(1 for a in range(len(k1)) if k1[a] > default[a])
            rejected = len(k1) - accepted
            if accepted >= rejected:
                acc_vals.append(k1)
                acc_params.append(all_params[all_vals.index(k1)])
        idx = best_max(acc_vals, acc_params)
    else:
        raise ValueError(rule)
    return np.float64(params[idx]), idx


class CarOracle:
    """E independent SelfAcceleratingCarEnv (+ optional SelfdriveContractDistprop subgame wrapper)."""

    def __init__(self, num_envs, num_agents, contract=False, low_bound=-10.0, high_bound=10.0, start_vel=0.2,
                 start_vel_ambulance=0.8, theta_low=0.0, theta_high=100.0, null_prob=0.0, seed=73907, first_env_id=0):
        self.E, self.n = int(num_envs), int(num_agents)
        self._h = lib().car_oracle_create(self.E, self.n, 1 if contract else 0, float(low_bound), float(high_bound),
                                          float(start_vel), float(start_vel_ambulance), float(theta_low),
                                          float(theta_high), float(null_prob), int(seed) & 0xFFFFFFFF, int(first_env_id))
        if not self._h:
            raise ValueError("car_oracle_create failed")
        self.D = lib().car_oracle_obs_dim(self._h)
        self.episode = np.full(self.E, -1, dtype=np.int64)

    def __del__(self):
        if getattr(self, "_h", None) and lib is not None:        # (module globals are gone at interpreter shutdown)
            try:
                lib().car_oracle_destroy(self._h)
            except Exception:
                pass
            self._h = None

    def reset(self, mask=None):
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        sel = np.ones(self.E, bool) if m is None else m.astype(bool)
        self.episode[sel] += 1
        ep = self.episode.astype(np.uint32)
        obs = np.zeros((self.E, self.n, self.D))
        lib().car_oracle_reset(self._h, _p(m), _p(ep), _p(obs))
        return obs

    def step(self, actions, skip=None):
        """Steps every env whose `skip` byte is zero (all of them without `skip`).  A skipped env keeps its state and its
        output rows stay zero, so `reset(mask)` followed by `step(a, skip=mask)` is a batch's next-step auto-reset."""
        a = np.ascontiguousarray(actions, dtype=np.float32).reshape(self.E, self.n)
        E, n = self.E, self.n
        out = {"obs": np.zeros((E, n, self.D)), "rew": np.zeros((E, n)), "base_rew": np.zeros((E, n)),
               "transfers": np.zeros((E, n)), "info": np.zeros((E, n, 4)), "done": np.zeros((E, n + 1), np.uint8)}
        args = (self._h, _p(a), _p(out["obs"]), _p(out["rew"]), _p(out["base_rew"]), _p(out["transfers"]),
                _p(out["info"]), _p(out["done"]))
        if skip is None:
            lib().car_oracle_step(*args)
        else:
            sk = _skip_bytes(skip, E)
            lib().car_oracle_step_skip(*args, _p(sk))
        return out

    def get_state(self):
        E, n = self.E, self.n
        st = {"pos": np.zeros((E, n)), "vel": np.zeros((E, n)), "theta": np.zeros(E), "transfers": np.zeros(E),
              "t": np.zeros(E, np.int32)}
        lib().car_oracle_get_state(self._h, _p(st["pos"]), _p(st["vel"]), _p(st["theta"]), _p(st["transfers"]), _p(st["t"]))
        return st

    def set_theta(self, theta):
        th = np.ascontiguousarray(np.broadcast_to(np.asarray(theta, dtype=np.float64), (self.E,)))
        lib().car_oracle_set_theta(self._h, _p(th))


class FeatOracle:
    """E independent CleanupFeatures / HarvestFeatures envs (+ optional subgame contract wrapper)."""

    def __init__(self, kind, num_envs, num_agents, ascii_map, horizon=1000, contract=None, theta_low=0.0,
                 theta_high=None, null_prob=0.0, seed=73907, first_env_id=0):
        self.kind = kind
        self.E, self.n = int(num_envs), int(num_agents)
        self.H, self.W = len(ascii_map), len(ascii_map[0])
        if theta_high is None:
            theta_high = float(np.float32(0.2)) if kind == "cleanup" else float(np.float32(10.0))
        flat = "".join(ascii_map).encode("ascii")
        self._h = lib().feat_oracle_create(KIND[kind], self.E, self.n, self.H, self.W, flat, int(horizon),
                                           CONTRACT[contract], float(theta_low), float(theta_high), float(null_prob),
                                           int(seed) & 0xFFFFFFFF, int(first_env_id))
        if not self._h:
            raise ValueError("feat_oracle_create failed (bad sizes / map)")
        self.F = lib().feat_oracle_dim(self._h)
        self.episode = np.full(self.E, -1, dtype=np.int64)

    def __del__(self):
        if getattr(self, "_h", None) and lib is not None:        # (module globals are gone at interpreter shutdown)
            try:
                lib().feat_oracle_destroy(self._h)
            except Exception:
                pass
            self._h = None

    def reset(self, mask=None):
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        sel = np.ones(self.E, bool) if m is None else m.astype(bool)
        self.episode[sel] += 1
        ep = self.episode.astype(np.uint32)
        obs = np.zeros((self.E, self.n, self.F))
        lib().feat_oracle_reset(self._h, _p(m), _p(ep), _p(obs))
        return obs

    def step(self, actions, skip=None):
        """Steps every env whose `skip` byte is zero (all of them without `skip`).  A skipped env keeps its state and its
        output rows stay zero, so `reset(mask)` followed by `step(a, skip=mask)` is a batch's next-step auto-reset."""
        a = np.ascontiguousarray(actions, dtype=np.int32).reshape(self.E, self.n)
        E, n = self.E, self.n
        out = {"obs": np.zeros((E, n, self.F)), "rew": np.zeros((E, n)), "base_rew": np.zeros((E, n)),
               "transfers": np.zeros((E, n)), "info": np.zeros((E, n, 4), np.int32), "done": np.zeros(E, np.uint8)}
        args = (self._h, _p(a), _p(out["obs"]), _p(out["rew"]), _p(out["base_rew"]), _p(out["transfers"]),
                _p(out["info"]), _p(out["done"]))
        if skip is None:
            lib().feat_oracle_step(*args)
        else:
            sk = _skip_bytes(skip, E)
            lib().feat_oracle_step_skip(*args, _p(sk))
        return out

    def metrics_raw(self):
        out = np.zeros((self.E, 40))
        lib().feat_oracle_get_metrics(self._h, _p(out))
        return out

    def get_state(self):
        E, n = self.E, self.n
        st = {"pos": np.zeros((E, n, 2), np.int32), "ori": np.zeros((E, n), np.int32),
              "cells": np.zeros((E, self.H, self.W), np.uint8), "theta": np.zeros(E), "t": np.zeros(E, np.int32)}
        lib().feat_oracle_get_state(self._h, _p(st["pos"]), _p(st["ori"]), _p(st["cells"]), _p(st["theta"]), _p(st["t"]))
        return st
