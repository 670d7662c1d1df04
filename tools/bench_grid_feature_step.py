"""Grid-world step in the feature-observation form (BatchedGridEnv(image_obs=False), ssd_set_feature_output) against the
uint8-window step that also writes the features, on bench.py's steady-state workload (bench.Runner: staggered episodes,
auto-reset with negotiation inside the step, random actions, CUDA graphs of 50 steps).

For each config it times, with CUDA events over graph replays, alternating the arms for --rounds rounds:
  u8_step          the uint8 step alone (bench.py's step)
  u8_features      the uint8 step with feature_obs_dev: the only route to the feature rows before this form.  A cost
                   comparison only: it cannot produce reset rows (an auto-reset env holds its final step's features)
  u8_features_T    u8_features, then theta from the state, features ++ [theta, 0], float32, T (float32 / float16 / bfloat16)
  feature_f64      the feature form, float64 rows
  feature_T        the feature form, the policy's rows in T
The median and the range are reported.  No profiler is involved.

    python tools/bench_grid_feature_step.py --out profiles/grid_feature_step_bench.json
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

CONFIGS = [("cleanup8", 131072), ("harvest16k", 16384)]


def stage(msg):
    """progress on stderr, synchronised: a failure is attributed to the stage it happened in"""
    import torch
    torch.cuda.synchronize()
    print("[bench_grid_feature_step] %s" % msg, file=sys.stderr, flush=True)


def make_runner(name, E, dev, image_obs=True, dtype=None, want_features=False):
    """bench.Runner of config `name`; image_obs=False swaps in the feature-form env of the same configuration,
    want_features makes its step write feature_obs beside the windows"""
    from contracts_b200.batched import BatchedGridEnv
    cfg = bench.CONFIGS[name]
    run = bench.Runner(name, cfg, E, 0, dev)
    if not image_obs:
        run.env.close()
        run.env = BatchedGridEnv(cfg["env"], E, cfg["n"], horizon=bench.HORIZON, contract=cfg["contract"], seed=bench.SEED,
                                 first_env_id=0, device=dev, image_obs=False, policy_dtype=dtype)
        run.env.set_episode_stats(run.stats)
    if want_features:
        def substep(step_index=None):
            run.gen_actions(step_index)
            run.env.step(run.actions, want_features=True, extras=False, auto_reset=True, negotiation=run.neg())
        run.substep = substep
    run.burn_in()
    stage("%s %s%s burned in" % (name, "windows" if image_obs else "features", "" if dtype is None else " " + str(dtype)))
    return run


def cat_cast(env, theta, rows32, rows):
    """after a uint8 step with features: theta from the state, features ++ [theta, 0], float32, T"""
    import torch
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    env.lib.ssd_get_state(env._h, None, None, None, None, ctypes.c_void_p(theta.data_ptr()), stream)
    F = env.F
    rows32[:, :, :F].copy_(env.feature_obs)
    rows32[:, :, F].copy_(theta.unsqueeze(1).expand(-1, env.n))      # column F + 1 stays 0
    if rows is not rows32:
        rows.copy_(rows32)


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSON file to write (default: print only)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--replays", type=int, default=20, help="graph replays of %d steps per timing" % G)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_grid_feature_step needs a CUDA device")
    dev = torch.device("cuda", 0)
    result = dict(gpu_info(), graph_steps=G, replays=args.replays, rounds=args.rounds, configs=[])
    dtypes = [("float32", torch.float32), ("float16", torch.float16), ("bfloat16", torch.bfloat16)]
    for name, E in CONFIGS:
        n = bench.CONFIGS[name]["n"]
        runs, graphs, keep = {}, {}, []          # keep: tensors the captured graphs write, alive until they are destroyed
        runs["u8_step"] = make_runner(name, E, dev)
        runs["u8_features"] = make_runner(name, E, dev, want_features=True)
        runs["feature_f64"] = make_runner(name, E, dev, image_obs=False)
        F = runs["feature_f64"].env.F
        W = F + 2
        for k in ("u8_step", "u8_features", "feature_f64"):
            graphs[k] = capture(runs[k])
            stage("%s %s captured" % (name, k))
        theta = torch.empty((E,), dtype=torch.float64, device=dev)
        rows32 = torch.zeros((E, n, W), dtype=torch.float32, device=dev)
        for dname, dt in dtypes:
            rows = rows32 if dt == torch.float32 else torch.zeros((E, n, W), dtype=dt, device=dev)
            keep.append(rows)
            u = runs["u8_features"]
            runs["u8_features_" + dname] = u
            graphs["u8_features_" + dname] = capture(u, lambda rows=rows: cat_cast(u.env, theta, rows32, rows))
            runs["feature_" + dname] = make_runner(name, E, dev, image_obs=False, dtype=dt)
            assert runs["feature_" + dname].env.policy_width == W
            graphs["feature_" + dname] = capture(runs["feature_" + dname])
            stage("%s %s arms captured" % (name, dname))
        ms = {k: [] for k in graphs}
        for _ in range(args.rounds):                            # alternate the arms
            for k in graphs:
                ms[k].append(time_graph(runs[k], graphs[k], args.replays))
            stage("%s round timed" % name)
        row = dict(config=name, envs=E, agents=n, features=F, policy_width=W)
        for k, v in ms.items():
            med = float(np.median(v))
            row[k] = dict(ms_per_step=med, ms_min=float(min(v)), ms_max=float(max(v)), agent_steps_per_s=E * n / (med * 1e-3))
        result["configs"].append(row)
        print(json.dumps({"config": name} | {k: [round(row[k]["ms_per_step"], 4), round(row[k]["ms_min"], 4),
                                                 round(row[k]["ms_max"], 4)] for k in ms}), flush=True)
        del graphs
        del runs, keep
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps({k: result[k] for k in ("gpu", "power_limit")}))


if __name__ == "__main__":
    main()
