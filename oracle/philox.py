"""Philox4x32-10 and the draw-addressing scheme shared by every implementation.

TEST INFRASTRUCTURE (oracle/): imported only by tests/, bench.py's cpu_baseline /
`--impl reference` leg, `__graft_entry__.smoke()` and the golden-vector generator.

The reference (the original project) draws from NumPy's / stdlib's global MT19937 at the
call sites of SURVEY.md §8a table R.  For parity every one of those sites is replaced
by a *counter-based* draw, so that the reference, the C oracle and the CUDA kernels
all see identical randomness regardless of evaluation order:

    u32 = philox4x32_10(ctr=(idx >> 2, site | call << 8, t, episode),
                        key=(seed, env_id))[idx & 3]

* ``site``    – which reference call site (constants below, cite file:line)
* ``call``    – n-th call of that site inside one (episode, t)  (e.g. agent index)
* ``idx``     – element index inside the call
* ``t``       – ``MapEnv.timesteps`` *after* the increment at map_env.py:230; 0 in reset
* ``episode`` – number of resets done before this one (0 for the first reset)

A "uniform double" is ``u32 * 2**-32`` (exact in float64).  A "shuffle" is stateless:
bring the list into canonical order, draw one key per element, stable-sort by key.

Constants match /usr/local/cuda/include/curand_philox4x32_x.h:88-91.
"""
import numpy as np

PHILOX_M0 = 0xD2511F53
PHILOX_M1 = 0xCD9E8D57
PHILOX_W0 = 0x9E3779B9
PHILOX_W1 = 0xBB67AE85

# --- site ids (SURVEY.md §8a table R) -------------------------------------------------
SITE_MOVE_ORDER = 1      # R1  map_env.py:546   np.random.shuffle(shuffle_list)
SITE_BEAM_ORDER = 2      # R2  map_env.py:685   np.random.shuffle(agent_ids)
SITE_SPAWN_DRAWS = 3     # R3/R5 cleanup_new.py:326, harvest_new.py:294  rand(k)
SITE_WASTE_ORDER = 4     # R4  cleanup_new.py:339  np.random.shuffle(self.waste_points)
SITE_SPAWN_ROT = 5       # R6  map_env.py:831   np.random.randint(4)
SITE_SPAWN_POINT = 6     # R7  map_env.py:821   np.random.shuffle(self.spawn_points)
SITE_CONTRACT = 7        # R8  two_stage_train.py:163-164  rand(), uniform(low, high)
SITE_NEGOTIATE = 8       # R9  two_stage_train.py:271,276  random.sample, random.random
SITE_SELFDRIVE_RESET = 9 # R10 self_driving_car_accelerate.py:53,57  random.random()
SITE_FEAT_ORDER = 10     # R11 cleanup_features.py:107 / harvest_features.py:118 random.shuffle(idx)
SITE_FEAT_ROT = 11       # R11 cleanup_features.py:109 / harvest_features.py:122 np.random.randint(0,4)
SITE_FEAT_SPAWN = 12     # R11 cleanup_features.py:115,122 / harvest_features.py:148 random.random()
SITE_ACTIONS = 13        # synthetic random actions for benchmarks (not a reference site)
SITE_SOLVER = 14         # two_stage_train.py:725  contract_param_space.sample() (gym Box.sample -> uniform)

EPISODE_CONSTRUCT = 0xFFFFFFFF  # draws consumed by MapEnv.__init__ -> setup_agents (map_env.py:131)

_U32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """Vectorised Philox4x32-10.  ctr: (..., 4) uint32-like, key: (..., 2) -> (..., 4) uint32."""
    ctr = np.asarray(ctr, dtype=np.uint64)
    key = np.asarray(key, dtype=np.uint64)
    c0, c1, c2, c3 = (ctr[..., i] & _U32 for i in range(4))
    k0, k1 = (key[..., i] & _U32 for i in range(2))
    m0 = np.uint64(PHILOX_M0)
    m1 = np.uint64(PHILOX_M1)
    for _ in range(10):
        p0 = m0 * c0
        p1 = m1 * c2
        hi0, lo0 = p0 >> np.uint64(32), p0 & _U32
        hi1, lo1 = p1 >> np.uint64(32), p1 & _U32
        c0, c1, c2, c3 = (hi1 ^ c1 ^ k0) & _U32, lo1, (hi0 ^ c3 ^ k1) & _U32, lo0
        k0 = (k0 + np.uint64(PHILOX_W0)) & _U32
        k1 = (k1 + np.uint64(PHILOX_W1)) & _U32
    return np.stack([c0, c1, c2, c3], axis=-1).astype(np.uint32)


def draws_u32(seed, env_id, episode, t, site, call, idx):
    """u32 draws for element indices ``idx`` (scalar or array) of one call."""
    idx = np.atleast_1d(np.asarray(idx, dtype=np.uint64))
    ctr = np.empty(idx.shape + (4,), dtype=np.uint64)
    ctr[..., 0] = idx >> np.uint64(2)
    ctr[..., 1] = np.uint64((site & 0xFF) | ((call & 0xFFFFFF) << 8))
    ctr[..., 2] = np.uint64(t & 0xFFFFFFFF)
    ctr[..., 3] = np.uint64(episode & 0xFFFFFFFF)
    key = np.array([seed & 0xFFFFFFFF, env_id & 0xFFFFFFFF], dtype=np.uint64)
    out = philox4x32_10(ctr, np.broadcast_to(key, idx.shape + (2,)))
    return np.take_along_axis(out, (idx & np.uint64(3)).astype(np.int64)[..., None], axis=-1)[..., 0]


def draws_f64(seed, env_id, episode, t, site, call, idx):
    """Uniform doubles in [0,1) on the 2^-32 lattice."""
    return draws_u32(seed, env_id, episode, t, site, call, idx).astype(np.float64) * 2.0 ** -32


def shuffle_order(seed, env_id, episode, t, site, call, n):
    """Stateless shuffle: position j of the shuffled list holds canonical element order[j]."""
    keys = draws_u32(seed, env_id, episode, t, site, call, np.arange(n))
    return np.argsort(keys, kind="stable")


def prob_threshold_u32(p):
    """Smallest integer T with (u32 * 2^-32 < p) <=> (u32 < T), for a float64 probability p.

    p * 2^32 is exact in float64 (power-of-two scaling), so T = ceil(p * 2^32), clamped to
    [0, 2^32].  Returned as a Python int (fits uint64; 2^32 means 'always').
    """
    import math
    p = float(p)
    if not (p > 0.0):
        return 0
    if p >= 1.0:
        return 1 << 32
    return int(math.ceil(p * 4294967296.0))
