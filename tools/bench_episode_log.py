"""Cost of the episode log (ssd_set_episode_log, contracts_b200/episodes.py) on bench.py's steady-state workload
(bench.Runner: staggered episodes, auto-reset in every step, random actions, CUDA graphs of 50 steps).

For each config it times, with CUDA events over graph replays, the same workload with the log off (no log set, the
bench.py path) and on (an EpisodeLog of E records set on the batch; it wraps, nothing is drained while timing).  The arms
alternate for --rounds rounds; the median and the range are reported, with the records appended per step by the timed
replays of the "on" arm.

    python tools/bench_episode_log.py --out profiles/episode_log_bench.json
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
from bench_policy_step import G, capture, gpu_info  # noqa: E402

CONFIGS = ["cleanup8", "harvest16k", "features1m", "harvestfeat1m", "selfdrive8"]


def time_graph(run, g, replays):
    """ms per env step over `replays` graph replays (negotiation inputs refreshed between replays, as in bench.py)"""
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
    from contracts_b200.episodes import RECORD_BYTES, EpisodeLog
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSON file to write (default: print only)")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--replays", type=int, default=20, help="graph replays of %d steps per timing" % G)
    ap.add_argument("--configs", default=",".join(CONFIGS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_episode_log needs a CUDA device")
    dev = torch.device("cuda", 0)
    result = dict(gpu_info(), graph_steps=G, replays=args.replays, rounds=args.rounds, configs=[])
    for name in args.configs.split(","):
        cfg = bench.CONFIGS[name]
        E = cfg["envs"]
        off = bench.Runner(name, cfg, E, 0, dev)
        off.burn_in()
        g_off = capture(off)
        on = bench.Runner(name, cfg, E, 0, dev)
        log = EpisodeLog(on.env, capacity=E)
        on.env.set_episode_log(log)
        on.burn_in()
        g_on = capture(on)
        t_off, t_on, recs = [], [], []
        for _ in range(args.rounds):                            # alternate the arms
            t_off.append(time_graph(off, g_off, args.replays))
            c0 = int(log.count.item())
            t_on.append(time_graph(on, g_on, args.replays))
            recs.append((int(log.count.item()) - c0) / ((args.replays + 2) * G))
        m_off, m_on = float(np.median(t_off)), float(np.median(t_on))
        row = dict(config=name, envs=E, agents=cfg["n"],
                   log_off=dict(ms_per_step=m_off, ms_min=float(min(t_off)), ms_max=float(max(t_off))),
                   log_on=dict(ms_per_step=m_on, ms_min=float(min(t_on)), ms_max=float(max(t_on))),
                   records_per_step=float(np.median(recs)), record_bytes_per_step=float(np.median(recs)) * RECORD_BYTES,
                   overhead_ms_per_step=m_on - m_off, overhead_fraction=m_on / m_off - 1.0)
        result["configs"].append(row)
        print(json.dumps(dict(config=name, off=round(m_off, 4), on=round(m_on, 4), records_per_step=round(row["records_per_step"], 1),
                              overhead=round(row["overhead_fraction"], 4))), flush=True)
        del off, on, g_off, g_on, log
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps({k: result[k] for k in ("gpu", "power_limit")}))


if __name__ == "__main__":
    main()
