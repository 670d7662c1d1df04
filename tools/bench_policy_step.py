"""Grid-world step that writes the policy's input tensors directly (BatchedGridEnv(policy_dtype=T)) against the uint8 step
followed by policy_inputs(T), on bench.py's steady-state workload (bench.Runner: staggered episodes, auto-reset and
negotiation in every step, random actions, CUDA graphs of 50 steps).

For each config and T in (float32, float16, bfloat16) it times, with CUDA events over graph replays:
  (a) the uint8 step, then policy_inputs(T) into preallocated tensors   ("two_pass")
  (b) the policy-mode step                                              ("fused")
  (c) the uint8 step alone                                              ("uint8_step")
The arms alternate for --rounds rounds; the median and the range are reported.  Bytes are the observation bytes the arm
moves per step, from the shapes: (a) writes the windows, reads them back and writes T image + contract rows; (b) writes
the T image; (c) writes the windows.  `hbm_fraction` divides that traffic by the time and by the HBM peak bench.py uses.

    python tools/bench_policy_step.py --out profiles/policy_step_bench.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (bench.Runner: the workload of bench.py, reused as is)

CONFIGS = [("cleanup8", 131072), ("harvest16k", 16384)]
G = 50                                                          # env steps per captured graph (bench.py's default)


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in q.split(",")]
    except Exception as exc:                                    # the figure stays absent rather than guessed
        info["power_limit"] = "unavailable (%s)" % exc
    return info


def make_runner(name, E, dtype, dev):
    """bench.Runner of config `name`; with dtype, its env is replaced by the policy-mode env of the same configuration"""
    cfg = bench.CONFIGS[name]
    run = bench.Runner(name, cfg, E, 0, dev)
    if dtype is not None:
        from contracts_b200.batched import BatchedGridEnv
        run.env.close()
        run.env = BatchedGridEnv(cfg["env"], E, cfg["n"], horizon=bench.HORIZON, contract=cfg["contract"], seed=bench.SEED,
                                 first_env_id=0, device=dev, policy_dtype=dtype)
        run.env.set_episode_stats(run.stats)
    run.burn_in()
    return run


def capture(run, extra=None):
    """a CUDA graph of G substeps (+ `extra` after each)"""
    import torch
    main = torch.cuda.current_stream()
    cap = torch.cuda.Stream()
    cap.wait_stream(main)
    with torch.cuda.stream(cap):
        for _ in range(3):
            run.substep()
            if extra:
                extra()
    main.wait_stream(cap)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=cap):
        for _ in range(G):
            run.substep()
            if extra:
                extra()
    torch.cuda.synchronize()
    return g


def time_graph(run, g, replays):
    """ms per env step over `replays` graph replays (the negotiation inputs are refreshed between replays, as in bench.py)"""
    import torch
    for _ in range(2):
        run.policy()
        g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(replays):
        run.policy()
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (replays * G)


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSON file to write (default: print only)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--replays", type=int, default=20, help="graph replays of %d steps per timing" % G)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_policy_step needs a CUDA device")
    dev = torch.device("cuda", 0)
    peak_gbs, peak_src = bench.measured_peak()
    result = dict(gpu_info(), hbm_peak_gbs=peak_gbs, hbm_peak_source=peak_src, graph_steps=G, replays=args.replays,
                  rounds=args.rounds, configs=[])
    dtypes = [("float32", torch.float32), ("float16", torch.float16), ("bfloat16", torch.bfloat16)]
    for name, E in CONFIGS:
        n = bench.CONFIGS[name]["n"]
        B = E * n
        base = make_runner(name, E, None, dev)
        g_c = capture(base)
        per_dtype = {}
        for dname, dt in dtypes:
            img = torch.empty((B, 3, 15, 15), dtype=dt, device=dev)
            con = torch.empty((B, 10), dtype=dt, device=dev)
            g_a = capture(base, lambda img=img, con=con, dt=dt: base.env.policy_inputs(dt, image=img, contract=con))
            fused = make_runner(name, E, dt, dev)
            g_b = capture(fused)
            # img / con live as long as the graph that writes them (a capture empties torch's cache of freed blocks)
            per_dtype[dname] = dict(dt=dt, img=img, con=con, g_a=g_a, fused=fused, g_b=g_b, a=[], b=[])
        c_ms = []
        for _ in range(args.rounds):                            # alternate the arms
            c_ms.append(time_graph(base, g_c, args.replays))
            for d in per_dtype.values():
                d["a"].append(time_graph(base, d["g_a"], args.replays))
                d["b"].append(time_graph(d["fused"], d["g_b"], args.replays))
        win = B * 675                                           # the uint8 windows
        for dname, d in per_dtype.items():
            s = torch.tensor([], dtype=d["dt"]).element_size()
            arms = {
                "two_pass": (d["a"], win + win + B * 675 * s + B * 10 * s, B * 675 * s + B * 10 * s + win),
                "fused": (d["b"], B * 675 * s, B * 675 * s),
                "uint8_step": (c_ms, win, win),
            }
            row = dict(config=name, envs=E, agents=n, dtype=dname)
            for arm, (ms, moved, written) in arms.items():
                med = float(np.median(ms))
                row[arm] = dict(ms_per_step=med, ms_min=float(min(ms)), ms_max=float(max(ms)),
                                agent_steps_per_s=B / (med * 1e-3), obs_bytes_written_per_step=int(written),
                                obs_bytes_moved_per_step=int(moved),
                                hbm_fraction=moved / (med * 1e-3) / (peak_gbs * 1e9))
            row["fused_speedup_vs_two_pass"] = row["two_pass"]["ms_per_step"] / row["fused"]["ms_per_step"]
            result["configs"].append(row)
            print(json.dumps({k: row[k] for k in ("config", "dtype")} |
                             {arm: round(row[arm]["ms_per_step"], 4) for arm in arms} |
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
