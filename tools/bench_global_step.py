"""Grid-world step in JointEnv's global-observation form (BatchedGridEnv(global_obs=True), ssd_set_global_output) against
the uint8-window step followed by global_view(), on bench.py's steady-state workload (bench.Runner: staggered episodes,
auto-reset inside the step, random actions, CUDA graphs of 50 steps) without a contract, as JointEnv wraps the bare env.

For each config it times, with CUDA events over graph replays, alternating the arms for --rounds rounds:
  global_u8         the global form, uint8 [E, H, W, 3] rows
  global_bf16       the global form, bfloat16 [E, 3, H, W] rows (VisionNetwork.forward's input)
  window_view       the uint8-window step, then global_view() into a preallocated tensor: the route before this form
  window_view_bf16  window_view, then (view.double() / 255).float().permute(0, 3, 1, 2) cast to bfloat16 in torch
The median and the range are reported.  No profiler is involved.

    python tools/bench_global_step.py --out profiles/global_step_bench.json
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402  (bench.Runner: the workload of bench.py, reused as is)
from bench_policy_step import G, capture, gpu_info, time_graph  # noqa: E402

# (label, bench config whose env / map / action count is used, agents, envs): cleanup n = 2 is the shipped joint config's
# agent count, n = 8 and harvest n = 4 are bench.py's grid configs
CONFIGS = [("cleanup2", "cleanup8", 2, 131072), ("cleanup8", "cleanup8", 8, 131072), ("harvest16k", "harvest16k", 4, 16384)]


def stage(msg):
    """progress on stderr, synchronised: a failure is attributed to the stage it happened in"""
    import torch
    torch.cuda.synchronize()
    print("[bench_global_step] %s" % msg, file=sys.stderr, flush=True)


def make_runner(base, n, E, dev, global_obs, dtype=None):
    """bench.Runner of config `base` with n agents and no contract (no negotiation); global_obs swaps in the global-form env"""
    from contracts_b200.batched import BatchedGridEnv
    cfg = dict(bench.CONFIGS[base], n=n, contract=None, negotiate=False)
    run = bench.Runner(base, cfg, E, 0, dev)
    if global_obs:
        run.env.close()
        run.env = BatchedGridEnv(cfg["env"], E, n, horizon=bench.HORIZON, seed=bench.SEED, first_env_id=0, device=dev,
                                 global_obs=True, policy_dtype=dtype)
        run.env.set_episode_stats(run.stats)
    run.burn_in()
    stage("%s n=%d %s%s burned in" % (base, n, "global" if global_obs else "windows", "" if dtype is None else " " + str(dtype)))
    return run


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSON file to write (default: print only)")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--replays", type=int, default=20, help="graph replays of %d steps per timing" % G)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_global_step needs a CUDA device")
    dev = torch.device("cuda", 0)
    result = dict(gpu_info(), graph_steps=G, replays=args.replays, rounds=args.rounds, configs=[])
    for label, base, n, E in CONFIGS:
        runs, graphs = {}, {}
        runs["global_u8"] = make_runner(base, n, E, dev, True)
        runs["global_bf16"] = make_runner(base, n, E, dev, True, torch.bfloat16)
        w = runs["window_view"] = runs["window_view_bf16"] = make_runner(base, n, E, dev, False)
        H, W = w.env.H, w.env.W
        view = torch.empty((E, H, W, 3), dtype=torch.uint8, device=dev)
        img = torch.empty((E, 3, H, W), dtype=torch.bfloat16, device=dev)
        graphs["global_u8"] = capture(runs["global_u8"])
        graphs["global_bf16"] = capture(runs["global_bf16"])
        graphs["window_view"] = capture(w, lambda: w.env.global_view(out=view))
        graphs["window_view_bf16"] = capture(w, lambda: (w.env.global_view(out=view),
                                                         img.copy_((view.double() / 255).float().permute(0, 3, 1, 2))))
        stage("%s captured" % label)
        ms = {k: [] for k in graphs}
        for _ in range(args.rounds):                            # alternate the arms
            for k in graphs:
                ms[k].append(time_graph(runs[k], graphs[k], args.replays))
            stage("%s round timed" % label)
        row = dict(config=label, env=bench.CONFIGS[base]["env"], envs=E, agents=n, map=[H, W],
                   view_bytes_per_env=dict(uint8=3 * H * W, bfloat16=6 * H * W), window_bytes_per_env=675 * n)
        for k, v in ms.items():
            med = float(np.median(v))
            row[k] = dict(ms_per_step=med, ms_min=float(min(v)), ms_max=float(max(v)), env_steps_per_s=E / (med * 1e-3))
        result["configs"].append(row)
        print(json.dumps({"config": label} | {k: [round(row[k]["ms_per_step"], 4), round(row[k]["ms_min"], 4),
                                                  round(row[k]["ms_max"], 4)] for k in ms}), flush=True)
        del graphs, runs, view, img
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps({k: result[k] for k in ("gpu", "power_limit")}))


if __name__ == "__main__":
    main()
