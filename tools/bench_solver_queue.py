"""The NegotiationSolver prologue inside the vectorised sampler (contracts_b200/solver.py) against the route that existed
before it, on bench.py's steady-state workload (bench.Runner: staggered episodes, auto-reset inside the step, random
actions, CUDA graphs of 50 steps), S = 50 candidates.

For each config it times, with CUDA events over graph replays, alternating the arms for --rounds rounds:
  step        the step alone (bench.py's step, in the config's observation form below)
  queue       step + SolverQueue.rows + a trivial value function (zeros [C, 1 + S, n]) + SolverQueue.resolve
  all_envs    step + the all-E route with the same value function: ssd_solver_sample for every env, the value-query rows
              of every env built in torch, ssd_solver_choose, then theta (and its policy rows) restored for the envs that
              did not restart (t != 0)
and reports value-query rows per step of the two solver arms (C (1 + S) n against E (1 + S) n), the median and the range.
No profiler is involved.

    python tools/bench_solver_queue.py --out profiles/solver_queue_bench.json
"""
import argparse
import ctypes
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402  (bench.Runner: the workload of bench.py, reused as is)
from bench_policy_step import G, capture, gpu_info, time_graph  # noqa: E402

S = 50
# config, envs, policy dtype (None: the float64 / uint8 form), window capacity C (>= the envs that restart in a step:
# E / horizon = 131 for the horizon-1000 configs; selfdrive episodes end by themselves)
CONFIGS = [("cleanup8", 131072, "bfloat16", 256), ("features1m", 131072, "bfloat16", 256), ("selfdrive8", 131072, None, 2048)]


def stage(msg):
    import torch
    torch.cuda.synchronize()
    print("[bench_solver_queue] %s" % msg, file=sys.stderr, flush=True)


def make_runner(name, E, dtype, dev):
    """bench.Runner of config `name`, its env replaced by the same configuration in policy dtype `dtype` when given"""
    cfg = bench.CONFIGS[name]
    run = bench.Runner(name, cfg, E, 0, dev)
    if dtype is not None:
        run.env.close()
        kw = dict(contract=cfg["contract"], seed=bench.SEED, first_env_id=0, device=dev, policy_dtype=dtype)
        if cfg["family"] == "grid":
            from contracts_b200.batched import BatchedGridEnv
            run.env = BatchedGridEnv(cfg["env"], E, cfg["n"], horizon=bench.HORIZON, **kw)
            run.env.set_episode_stats(run.stats)
        elif cfg["family"] == "feat":
            from contracts_b200.features import BatchedFeatureEnv
            run.env = BatchedFeatureEnv(cfg["env"], E, cfg["n"], horizon=bench.HORIZON, **kw)
        else:
            from contracts_b200.selfdrive import BatchedCarEnv
            run.env = BatchedCarEnv(E, cfg["n"], **kw)
    run.burn_in()
    return run


def queue_arm(run, C):
    import torch
    from contracts_b200.solver import SolverQueue
    q = SolverQueue(run.env, num_samples=S, capacity=C)
    vals = torch.zeros((C, S + 1, run.n), dtype=torch.float64, device=run.dev)

    def extra():
        q.rows()
        q.resolve(vals)
    return q, extra


def all_envs_arm(run):
    """today's route for every env, restoring the envs that did not restart"""
    import torch
    from contracts_b200.batched import solver_choose, solver_sample
    env, E, n = run.env, run.E, run.n
    vals = torch.zeros((E, S + 1, n), dtype=torch.float64, device=run.dev)
    theta0 = torch.empty((E,), dtype=torch.float64, device=run.dev)
    t = torch.empty((E,), dtype=torch.int32, device=run.dev)
    th, tp = ctypes.c_void_p(theta0.data_ptr()), ctypes.c_void_p(t.data_ptr())

    def state():
        s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        if env.kind == "selfdrive":
            env.lib.ssd_selfdrive_get_state(env._h, None, None, th, None, tp, s)
        elif env.kind in ("cleanup", "harvest"):
            env.lib.ssd_feat_get_state(env._h, None, None, None, th, tp, s)
        else:
            env.lib.ssd_get_state(env._h, None, None, None, tp, th, s)

    def rows(params):
        p = params[:, :, None, None].expand(E, S + 1, n, 1)
        if getattr(env, "image_obs", False):                   # grid world, policy image: the contract part
            pt = p.float().to(env.policy_dtype) if env.policy_dtype is not None else p
            return torch.cat((pt, torch.zeros_like(pt)), -1).repeat(1, 1, 1, 5 if env.policy_dtype is not None else 1)
        if env.policy_dtype is None:
            obs = env.obs[:, None].expand(E, S + 1, n, env.obs.shape[-1])
            return torch.cat((obs, p, torch.zeros_like(p)), -1)
        W = env.policy_width
        feat = env.policy_obs.view(E, n, W)[:, None, :, :W - 2].expand(E, S + 1, n, W - 2)
        pt = p.float().to(env.policy_dtype)
        return torch.cat((feat, pt, torch.zeros_like(pt)), -1)

    def extra():
        state()
        params = solver_sample(env, S)
        rows(params)                                            # the value function's input (unused by the trivial one)
        best, _ = solver_choose(env, params, vals, "majority")
        env.set_contract_params(torch.where(t == 0, best, theta0))
    return extra


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSON file to write (default: print only)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--replays", type=int, default=10, help="graph replays of %d steps per timing" % G)
    ap.add_argument("--configs", default=",".join(c[0] for c in CONFIGS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_solver_queue needs a CUDA device")
    dev = torch.device("cuda", 0)
    result = dict(gpu_info(), graph_steps=G, replays=args.replays, rounds=args.rounds, num_samples=S, configs=[])
    for name, E, dname, C in CONFIGS:
        if name not in args.configs.split(","):
            continue
        dtype = getattr(torch, dname) if dname else None
        n = bench.CONFIGS[name]["n"]
        runs, graphs = {}, {}
        for arm in ("step", "queue", "all_envs"):
            runs[arm] = make_runner(name, E, dtype, dev)
        q, qx = queue_arm(runs["queue"], C)
        graphs["step"] = capture(runs["step"])
        graphs["queue"] = capture(runs["queue"], qx)
        graphs["all_envs"] = capture(runs["all_envs"], all_envs_arm(runs["all_envs"]))
        stage("%s captured" % name)
        ms = {k: [] for k in graphs}
        for _ in range(args.rounds):                            # alternate the arms
            for k in graphs:
                ms[k].append(time_graph(runs[k], graphs[k], args.replays))
            stage("%s round timed" % name)
        cnt = [int(x) for x in q.count.tolist()]
        row = dict(config=name, envs=E, agents=n, policy_dtype=dname or "native", capacity=C,
                   queries_per_step=dict(queue=C * (S + 1) * n, all_envs=E * (S + 1) * n),
                   last_window=dict(in_window=cnt[0], pending=cnt[1]))
        for k, v in ms.items():
            row[k] = dict(ms_per_step=float(np.median(v)), ms_min=float(min(v)), ms_max=float(max(v)))
        result["configs"].append(row)
        print(json.dumps(row), flush=True)
        del graphs, runs, q, qx
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps({k: result[k] for k in ("gpu", "power_limit")}))


if __name__ == "__main__":
    main()
