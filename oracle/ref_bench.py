"""Time the UNMODIFIED reference env loop on host cores (bench.py's cpu_baseline / `--impl reference` arm).

TEST / MEASUREMENT INFRASTRUCTURE (oracle/).  SURVEY.md §8(d): the reference (stubbed imports, its own MT19937 RNG — no
injection) stepping the env + SeparateContractSubgameStage wrapper with iid random actions, one env per process,
P processes via multiprocessing (mirrors RLlib's one env per rollout worker, utils/ray_config_utils.py:140); the rate is
P envs x n agents x steps over the SLOWEST worker's loop time.  Uses $SSD_REFERENCE_ROOT when set, else the staged copy
oracle/_ref/ (oracle/stage_reference.py).
"""
import multiprocessing as mp
import os
import time

CONFIGS = {
    # name: (base tag, num_agents, contract class, action count / None for selfdrive, base kwargs)
    "cleanup8": ("CleanupNew", 8, "CleanupContract", 8, {"image_obs": True}),
    "cleanup2": ("CleanupNew", 2, "CleanupContract", 8, {"image_obs": True}),
    "harvest16k": ("HarvestNew", 4, "HarvestFeaturemodLocalContract", 7, {"image_obs": True}),
    "features1m": ("Cleanup", 8, "CleanupContract", 8, {}),
    "harvestfeat1m": ("Harvest", 8, "HarvestFeaturemodLocalContract", 7, {}),
    "selfdrive8": ("SelfDrive", 8, "SelfdriveContractDistprop", None, {}),
}


def available():
    from . import ref_stubs
    return ref_stubs.reference_root()


def _worker(args):
    config, steps, warmup, seed = args
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    import numpy as np
    import random
    from . import ref_stubs
    ref_stubs.install(ref_stubs.reference_root())
    from utils.env_creator_functions import env_creator          # the reference's own factory
    import contract.contract_list as contract_list
    tag, n, cname, nact, kw = CONFIGS[config]
    np.random.seed(seed)
    random.seed(seed)
    base = env_creator(tag, dict(num_agents=n, env_params={}, **kw))
    contract = getattr(contract_list, cname)(n)
    env = env_creator("ContractWrapperSubgame", {"num_agents": n, "base_env": base, "contract": contract,
                                                 "convolutional": bool(kw.get("image_obs"))})
    rng = np.random.RandomState(seed + 1)
    ids = ["a%d" % i for i in range(n)]

    def actions(live):
        if nact is None:
            return {a: np.array([rng.uniform(-0.1, 0.1)], dtype=np.float32) for a in live}
        return {a: int(rng.randint(nact)) for a in live}

    obs = env.reset()
    done_steps = 0
    t0 = None
    for k in range(warmup + steps):
        if k == warmup:
            t0 = time.perf_counter()
        obs, rew, done, info = env.step(actions(list(obs.keys()) if nact is None else ids))
        done_steps += 1
        if done["__all__"]:
            obs = env.reset()
    return time.perf_counter() - t0


def run(config="cleanup8", steps=200, warmup=5, procs=None):
    """-> (agent-steps/s, procs, ms per env step of the slowest worker, sample description)"""
    root = available()
    if root is None:
        raise RuntimeError("no reference tree (neither $SSD_REFERENCE_ROOT nor oracle/_ref)")
    procs = procs or (os.cpu_count() or 1)
    n = CONFIGS[config][1]
    ctx = mp.get_context("spawn")                                  # no forked CUDA / OpenMP state in the workers
    with ctx.Pool(procs) as pool:
        times = pool.map(_worker, [(config, steps, warmup, 1000 + i) for i in range(procs)])
    slowest = max(times)
    rate = procs * n * steps / slowest
    sample = ("unmodified reference (%s), %s + SeparateContractSubgameStage, %d processes x 1 env x %d steps, native MT19937 "
              "RNG, iid random actions; rate over the slowest worker" % (os.path.basename(root.rstrip("/")) or root, CONFIGS[config][0], procs, steps))
    return rate, procs, slowest / steps * 1e3, sample


if __name__ == "__main__":
    import sys
    print(run(sys.argv[1] if len(sys.argv) > 1 else "cleanup8", int(sys.argv[2]) if len(sys.argv) > 2 else 100))
