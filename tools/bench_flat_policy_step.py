"""Feature-env and selfdrive step that writes the policy's flat input rows directly (BatchedFeatureEnv /
BatchedCarEnv(policy_dtype=T)) against the float64 step followed by the public-API route to the same rows, on bench.py's
steady-state workload (bench.Runner: staggered episodes, next-step auto-reset, random actions, CUDA graphs of 50 steps).

For each config and T in (float32, float16, bfloat16) it times, with CUDA events over graph replays:
  (a) the float64 step, then theta from the state (ssd_*_get_state with only the theta output), concatenate and cast
      into preallocated tensors: features ++ [theta, 0] to float32, then to T                       ("two_pass")
  (b) the policy-mode step                                                                           ("fused")
  (c) the float64 step alone                                                                         ("f64_step")
The arms alternate for --rounds rounds; the median and the range are reported.  Bytes are the observation bytes the arm
moves per step, from the shapes: (a) writes the float64 rows, reads them back, writes the float32 rows (and, for a
half type, reads them and writes the T rows); (b) writes the T rows; (c) writes the float64 rows.  `hbm_fraction`
divides that traffic by the time and by the HBM peak bench.py uses.  No profiler is involved: any bound stated from
these numbers is unprofiled.

    python tools/bench_flat_policy_step.py --out profiles/flat_policy_step_bench.json
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

CONFIGS = [("features1m", 131072), ("harvestfeat1m", 131072), ("selfdrive8", 131072)]


def make_runner(name, E, dtype, dev):
    """bench.Runner of config `name`; with dtype, its env is replaced by the policy-mode env of the same configuration"""
    cfg = bench.CONFIGS[name]
    run = bench.Runner(name, cfg, E, 0, dev)
    if dtype is not None:
        run.env.close()
        kw = dict(contract=cfg["contract"], seed=bench.SEED, first_env_id=0, device=dev, policy_dtype=dtype)
        if cfg["family"] == "car":
            from contracts_b200.selfdrive import BatchedCarEnv
            run.env = BatchedCarEnv(E, cfg["n"], **kw)
        else:
            from contracts_b200.features import BatchedFeatureEnv
            run.env = BatchedFeatureEnv(cfg["env"], E, cfg["n"], horizon=bench.HORIZON, **kw)
    run.burn_in()
    return run


def two_pass(env, theta, rows32, rows):
    """what a caller does today after the float64 step: theta from the state, features ++ [theta, 0], float32, T"""
    import torch
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    th = ctypes.c_void_p(theta.data_ptr())
    if env.kind == "selfdrive":
        env.lib.ssd_selfdrive_get_state(env._h, None, None, th, None, None, stream)
    else:
        env.lib.ssd_feat_get_state(env._h, None, None, None, th, None, stream)
    F = env.obs.shape[2]
    rows32[:, :, :F].copy_(env.obs)
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
        raise SystemExit("bench_flat_policy_step needs a CUDA device")
    dev = torch.device("cuda", 0)
    peak_gbs, peak_src = bench.measured_peak()
    result = dict(gpu_info(), hbm_peak_gbs=peak_gbs, hbm_peak_source=peak_src, graph_steps=G, replays=args.replays,
                  rounds=args.rounds, configs=[])
    dtypes = [("float32", torch.float32), ("float16", torch.float16), ("bfloat16", torch.bfloat16)]
    for name, E in CONFIGS:
        n = bench.CONFIGS[name]["n"]
        B = E * n
        base = make_runner(name, E, None, dev)
        F = base.env.obs.shape[2]
        W = F + 2
        g_c = capture(base)
        theta = torch.empty((E,), dtype=torch.float64, device=dev)
        rows32 = torch.zeros((E, n, W), dtype=torch.float32, device=dev)
        per_dtype = {}
        for dname, dt in dtypes:
            rows = rows32 if dt == torch.float32 else torch.zeros((E, n, W), dtype=dt, device=dev)
            g_a = capture(base, lambda rows=rows: two_pass(base.env, theta, rows32, rows))
            fused = make_runner(name, E, dt, dev)
            assert fused.env.policy_width == W
            g_b = capture(fused)
            per_dtype[dname] = dict(dt=dt, rows=rows, g_a=g_a, fused=fused, g_b=g_b, a=[], b=[])
        c_ms = []
        for _ in range(args.rounds):                            # alternate the arms
            c_ms.append(time_graph(base, g_c, args.replays))
            for d in per_dtype.values():
                d["a"].append(time_graph(base, d["g_a"], args.replays))
                d["b"].append(time_graph(d["fused"], d["g_b"], args.replays))
        f64 = B * F * 8                                         # the float64 rows
        for dname, d in per_dtype.items():
            s = torch.tensor([], dtype=d["dt"]).element_size()
            half = 0 if s == 4 else B * W * 4 + B * W * s       # float32 rows read back, T rows written
            arms = {
                "two_pass": (d["a"], f64 + f64 + B * W * 4 + half, f64 + B * W * 4 + (B * W * s if s != 4 else 0)),
                "fused": (d["b"], B * W * s, B * W * s),
                "f64_step": (c_ms, f64, f64),
            }
            row = dict(config=name, envs=E, agents=n, features=F, policy_width=W, dtype=dname)
            for arm, (ms, moved, written) in arms.items():
                med = float(np.median(ms))
                row[arm] = dict(ms_per_step=med, ms_min=float(min(ms)), ms_max=float(max(ms)),
                                agent_steps_per_s=B / (med * 1e-3), obs_bytes_written_per_step=int(written),
                                obs_bytes_moved_per_step=int(moved),
                                hbm_fraction=moved / (med * 1e-3) / (peak_gbs * 1e9))
            row["fused_speedup_vs_two_pass"] = row["two_pass"]["ms_per_step"] / row["fused"]["ms_per_step"]
            result["configs"].append(row)
            print(json.dumps({k: row[k] for k in ("config", "dtype")} |
                             {arm: [round(row[arm]["ms_per_step"], 4), round(row[arm]["ms_min"], 4), round(row[arm]["ms_max"], 4)]
                              for arm in arms} |
                             {"speedup": round(row["fused_speedup_vs_two_pass"], 3)}), flush=True)
        del base, per_dtype
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps({k: result[k] for k in ("gpu", "power_limit")}))


if __name__ == "__main__":
    main()
