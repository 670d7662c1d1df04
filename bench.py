#!/usr/bin/env python
"""bench.py — throughput of the hot path on B200 (and the CPU reference arm).

Metric (BASELINE.json): agent-steps/s, observations included, at 1/2/4/8 GPUs; % of the HBM roofline.
`--config` picks the workload (default: the headline, BASELINE configs[2]):
  cleanup8      CleanupEnv n=8 + CleanupContract with the two-stage negotiation prologue, horizon 1000, 131072 envs / GPU
  harvest16k    HarvestEnv n=4 + HarvestFeaturemodLocalContract, horizon 1000, 16384 envs / GPU           (configs[1])
  features1m    CleanupFeatures n=8 + CleanupContract, 131072 envs / GPU = 1M envs on 8 GPUs               (configs[3])
  harvestfeat1m HarvestFeatures n=8 + HarvestFeaturemodLocalContract, 131072 envs / GPU                    (configs[3])
  selfdrive8    SelfAcceleratingCarEnv n=8 + SelfdriveContractDistprop, 131072 envs / GPU                  (configs[4])

Workload = the STEADY STATE of a vectorised sampler (RLlib resets each env when it is done, so the envs of a batch are
not in lockstep): env i's episodes start at steps = i mod horizon, every step about E / horizon envs finish, are
reset (masked `ssd_reset`) and negotiate their next contract (masked `ssd_negotiate`), and hand their episode statistics
to a device accumulator.  Every step therefore costs the same (a 20-step window equals a 1000-step window), and the
episode boundary — reset + negotiation prologue + statistics — is inside every timed step pro rata.  The steady state is
reached by an untimed burn-in of one horizon with staggered resets.  Weak scaling: every rank owns E envs with global
ids rank*E ..; no collective on the step path; the statistics vector is all-gathered (NCCL) on a side stream.

A "step" = random actions + `ssd_step` with auto_reset (the finished envs are reset and negotiate inside the step; the
feature / selfdrive envs: + a masked reset launch) over the rank's E envs.
  value   : device-resident (actions generated on device, outputs stay in HBM), CUDA-event timed, max over ranks
  e2e     : the same step through the host-buffer API: pinned host actions -> device, step, result block (rewards +
            dones) -> pinned host memory, every step; pipelined two deep (`ssd_step_host_async` / `_wait`)
  roofline: algorithmic bytes (SURVEY.md §8d) / measured duration of the step kernels (CUDA events on their stream)
  cpu_baseline / --impl reference: the UNMODIFIED reference's Python env loop on the host cores (oracle/_ref, staged by
            __graft_entry__.build()), one env per process; the C restatement (oracle/) is reported beside it.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HORIZON = 1000
SEED = 73907                       # reference seed multiplier (runner.py:130)

# alg: algorithmic bytes per agent-step (SURVEY.md §8d; DESIGN.md §4): observation + state read/write + rewards /
# actions / infos.  harvest record = 640 B map + 368 B header; feature envs: F float64 features + masks / stamps.
CONFIGS = {
    "cleanup8": dict(family="grid", env="cleanup_new", n=8, contract="CleanupContract", nact=8, envs=131072, negotiate=True,
                     alg=840.0, oracle_kind="cleanup",
                     workload="cleanup_new n=8 CleanupContract + negotiation prologue, horizon 1000, random actions"),
    "harvest16k": dict(family="grid", env="harvest_new", n=4, contract="HarvestFeaturemodLocalContract", nact=7, envs=16384,
                       negotiate=False, alg=(2700 + 2 * 1008 + 4 * (1 + 8 + 4) + 1) / 4, oracle_kind="harvest",
                       workload="harvest_new n=4 HarvestFeaturemodLocalContract, horizon 1000, random actions, 16384 envs per GPU"),
    "features1m": dict(family="feat", env="cleanup", n=8, contract="CleanupContract", nact=8, envs=131072, negotiate=False,
                       alg=(8 * 20 * 8 + 2 * (64 + 32 + 16 + 8 * 36) + 8 * 13 + 1) / 8,
                       workload="CleanupFeatures n=8 CleanupContract, horizon 1000, random actions, 131072 envs per GPU (1M on 8)"),
    "harvestfeat1m": dict(family="feat", env="harvest", n=8, contract="HarvestFeaturemodLocalContract", nact=7, envs=131072,
                          negotiate=False, alg=(8 * 26 * 8 + 2 * (64 + 32 + 16 + 8 * 36) + 8 * 13 + 1) / 8,
                          workload="HarvestFeatures n=8 HarvestFeaturemodLocalContract, horizon 1000, random actions, 131072 envs per GPU"),
    "selfdrive8": dict(family="car", n=8, contract="SelfdriveContractDistprop", envs=131072, negotiate=False,
                       alg=(8 * 21 * 8 + 2 * (16 * 8 + 44) + 8 * (4 + 8) + 9) / 8,
                       workload="SelfAcceleratingCarEnv n=8 SelfdriveContractDistprop, random accelerations in [-0.1, 0.1], 131072 envs per GPU"),
}


def config_dict(name, cfg, E, world):
    """the keys both arms print identically (the reference arm times a bounded sample of this workload)"""
    return {"workload": cfg["workload"], "name": name, "envs_per_gpu": E, "agents": cfg["n"], "horizon": HORIZON,
            "parallelism": "env batch sharded over %d GPU(s), no collective on the step path; statistics all-gather on a "
                           "side stream" % world}


def ncu_traffic(config, envs, agents):
    """DRAM bytes per step of the step kernels from the committed ncu capture (same workload and size), else None."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        t = t.get(config, t)
        if t["envs"] == envs and t["agents"] == agents:
            return t["dram_bytes_read"] + t["dram_bytes_write"]
    except Exception:
        pass
    return None


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def _nvml_sample(self):
        nv, h = self.nv, self.nvml_handle
        sm = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
        r = int(self.get_reasons(h))
        self.rows.append([str(sm), str(self.mx), "0"] + ["Active" if r & b else "Not Active" for _, b in self.bits])

    def _nvml_loop(self):
        while not self.stop_flag.wait(0.005):
            self._nvml_sample()

    def start(self):
        """NVML polled every 5 ms from a thread (the timed region can be shorter than one nvidia-smi period), first
        sample taken synchronously, last one at stop(); nvidia-smi -lms as the fallback."""
        try:
            import pynvml as nv
            nv.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(visible.split(",")[self.index]) if visible and visible.split(",")[self.index].isdigit() else self.index
            self.nv, self.nvml_handle = nv, nv.nvmlDeviceGetHandleByIndex(idx)
            names = (("hw_slowdown", "nvmlClocksEventReasonHwSlowdown", "nvmlClocksThrottleReasonHwSlowdown"),
                     ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown", "nvmlClocksThrottleReasonHwThermalSlowdown"),
                     ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown", "nvmlClocksThrottleReasonSwThermalSlowdown"),
                     ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap", "nvmlClocksThrottleReasonSwPowerCap"))
            self.bits = [(n, getattr(nv, a, None) or getattr(nv, b, 0)) for n, a, b in names]
            self.get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
            self.mx = float(nv.nvmlDeviceGetMaxClockInfo(self.nvml_handle, nv.NVML_CLOCK_SM))
            self._nvml_sample()
            self.stop_flag = threading.Event()
            self.thread = threading.Thread(target=self._nvml_loop, daemon=True)
            self.thread.start()
            self.proc = "nvml"
            return
        except Exception:
            self.proc = None
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        if self.proc == "nvml":
            self.stop_flag.set()
            self.thread.join(timeout=1.0)
            try:
                if len(self.rows) < 3:               # a region shorter than two polling periods
                    self._nvml_sample()
            except Exception:
                pass
        else:
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}



# ----------------------------------------------------------------------------------------------
def run_port(cfg, envs_per_thread, steps, warmup):
    """The C restatement (oracle/) on all host cores (OpenMP), grid configs only -> cpu_baseline-style dict or None."""
    if cfg["family"] != "grid":
        return None
    from oracle import oracle
    from contracts_b200.maps import CLEANUP_MAP, HARVEST_MAP
    cores = oracle.set_num_threads(os.cpu_count() or 1)      # torchrun exports OMP_NUM_THREADS=1: ask for every core
    E, n = envs_per_thread * cores, cfg["n"]
    o = oracle.GridOracle(cfg["oracle_kind"], E, n, CLEANUP_MAP if cfg["oracle_kind"] == "cleanup" else HARVEST_MAP,
                          horizon=HORIZON, contract=cfg["contract"], seed=SEED)
    o.reset()
    if cfg["negotiate"]:                                     # the prologue of the headline workload, like the GPU arm
        rng0 = np.random.RandomState(1)
        o.negotiate(rng0.uniform(0, 0.2, size=E), rng0.uniform(size=(E, n)))
    rng = np.random.RandomState(0)
    acts = rng.randint(0, cfg["nact"], size=(16, E, n)).astype(np.int32)
    for t in range(warmup):
        o.step(acts[t % 16], want_features=False)
    t0 = time.perf_counter()
    for t in range(steps):
        o.step(acts[t % 16], want_features=False)
    dt = time.perf_counter() - t0
    return {"value": E * n * steps / dt, "unit": "agent-steps/s", "cores": cores, "kind": "port", "ms_per_step": dt / steps * 1e3,
            "sample": "C restatement (oracle/ssd_oracle.c), OpenMP x%d, %d envs x %d steps of the same workload "
                      "(negotiated contracts, observations written, no feature_obs)" % (cores, E, steps)}


def run_reference(config, steps, warmup):
    """The UNMODIFIED reference on all host cores, one env per process -> cpu_baseline dict, or None if not staged."""
    from oracle import ref_bench
    if ref_bench.available() is None:
        print("cpu_baseline: no reference tree (build() stages oracle/_ref only when SSD_REFERENCE_ROOT names a checkout "
              "of the original project); the C restatement (kind 'port') stands in for it", file=sys.stderr)
        return None
    rate, procs, ms, sample = ref_bench.run(config, steps=steps, warmup=warmup)
    out = {"value": rate, "unit": "agent-steps/s", "cores": procs, "kind": "reference", "ms_per_env_step": ms, "sample": sample}
    if procs > 1:                                            # SURVEY.md §8(d): the one-process figure beside the P-process one
        r1, _, ms1, _ = ref_bench.run(config, steps=min(steps, 100), warmup=min(warmup, 5), procs=1)
        out["one_process"] = {"value": r1, "unit": "agent-steps/s", "ms_per_env_step": ms1, "steps": min(steps, 100)}
    return out


def cpu_arms(config, cfg, ref_steps=150, port_steps=150, ref_warmup=5):
    ref = run_reference(config, ref_steps, ref_warmup)
    port = run_port(cfg, 64, port_steps, 20)
    return ref, port


REF_ENV_STEPS_PER_STEP = 8


def reference_arm(args):
    """`--impl reference`: EXACTLY --steps K timed steps after --warmup W untimed ones.  One step of this arm is a bounded
    sample of the workload: every one of the P one-env processes advances its env by R env steps (R = 8; fewer for a very
    large K so that the run stays within minutes at ~1-2 ms per reference env step)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cfg = CONFIGS[args.config]
    steps, warm = max(args.steps, 1), max(args.warmup, 0)
    R = max(1, min(REF_ENV_STEPS_PER_STEP, 40000 // steps))
    ref = run_reference(args.config, steps * R, warm * R)
    # the C restatement: reported beside the reference on a bounded sample; the timed arm itself (exactly K steps) only
    # where no reference tree was staged
    port = run_port(cfg, 64, min(max(steps, 20), 300), 20) if ref is not None else run_port(cfg, 64, steps, warm)
    main_arm = ref or port
    if main_arm is None:
        print(json.dumps({"impl": "reference", "unavailable": "neither oracle/_ref (staged reference) nor a C port for this config"}))
        return
    line = {
        "impl": "reference", "metric": "agent-steps/sec", "value": main_arm["value"], "unit": "agent-steps/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm,
        "ms_per_step": main_arm["ms_per_env_step"] * R if main_arm is ref else main_arm["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8" if cfg["family"] == "grid" else "f64",
        "data": "synthetic",
        "config": config_dict(args.config, cfg, args.envs or cfg["envs"], int(os.environ.get("WORLD_SIZE", "1"))),
        "cpu_baseline": main_arm,
        "step_definition": "%d env steps in each of the %d one-env processes" % (R, main_arm["cores"]) if main_arm is ref
                           else "one step of the C restatement's env batch",
        "e2e": {"value": main_arm["value"], "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "kind=reference: the unmodified Python reference (staged into oracle/_ref by __graft_entry__.build()), one "
                "env per process on every host core; the C restatement of the same algorithm is reported in cpu_baseline_port",
    }
    if port is not None and main_arm is not port:
        line["cpu_baseline_port"] = port
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------
class Runner:
    """One rank's env batch, driven as a vectorised sampler in steady state."""

    def __init__(self, name, cfg, E, rank, dev):
        import torch
        self.torch, self.cfg, self.E, self.n, self.dev, self.name = torch, cfg, E, cfg["n"], dev, name
        fam = cfg["family"]
        kw = dict(contract=cfg["contract"], seed=SEED, first_env_id=rank * E, device=dev)
        if fam == "grid":
            from contracts_b200.batched import BatchedGridEnv
            self.env = BatchedGridEnv(cfg["env"], E, self.n, horizon=HORIZON, **kw)
            self.actions = torch.empty((E, self.n), dtype=torch.uint8, device=dev)
        elif fam == "feat":
            from contracts_b200.features import BatchedFeatureEnv
            self.env = BatchedFeatureEnv(cfg["env"], E, self.n, horizon=HORIZON, **kw)
            self.actions = torch.empty((E, self.n), dtype=torch.uint8, device=dev)
        else:
            from contracts_b200.selfdrive import BatchedCarEnv
            self.env = BatchedCarEnv(E, self.n, **kw)
            self.actions = torch.empty((E, self.n), dtype=torch.float32, device=dev)
            self.mask = torch.zeros((E,), dtype=torch.uint8, device=dev)
        self.fam = fam
        self.gen = torch.Generator(device=dev)
        self.gen.manual_seed(SEED + rank)
        self.stats = None
        if cfg["negotiate"]:
            self.prop = torch.zeros((E,), dtype=torch.float64, device=dev)
            self.acc = torch.zeros((E, self.n), dtype=torch.float64, device=dev)
            self.dec = torch.zeros((E,), dtype=torch.uint8, device=dev)
        if fam == "grid":
            self.stats = torch.zeros(8, dtype=torch.float64, device=dev)
            self.env.set_episode_stats(self.stats)

    # the policy's negotiation outputs (two_stage_train.py:257-281): a0 proposes theta ~ U[0, 0.2], the others'
    # acceptance probabilities ~ U[0, 1]; refreshed outside the captured graph
    def policy(self):
        if self.cfg["negotiate"]:
            self.prop.uniform_(0.0, 0.2, generator=self.gen)
            self.acc.uniform_(0.0, 1.0, generator=self.gen)

    def gen_actions(self, step_index=None):
        if self.fam == "car":
            self.env.random_actions(step_index, -0.1, 0.1, out=self.actions)
        else:
            self.env.random_actions(step_index, self.cfg["nact"], out=self.actions)

    def done_mask(self):
        if self.fam == "car":
            self.mask.copy_(self.env.done[:, self.n])
            return self.mask
        return self.env.done

    def after_step(self, mask=None):
        """finished envs restart: masked reset (+ masked negotiation prologue)"""
        m = self.done_mask() if mask is None else mask
        self.env.reset(m)
        if self.cfg["negotiate"]:
            self.env.negotiate(self.prop, self.acc, mask=m, out=self.dec)

    def neg(self):
        return (self.prop, self.acc, self.dec) if self.cfg["negotiate"] else None

    def substep(self, step_index=None):
        """everything one env step enqueues on the device (capturable in a CUDA graph)"""
        self.gen_actions(step_index)
        if self.fam == "grid":       # finished envs restart (and negotiate) inside the step: ssd_step_io.auto_reset
            self.env.step(self.actions, extras=False, auto_reset=True, negotiation=self.neg())
        else:                        # feature / selfdrive envs: next-step auto-reset inside the step kernel
            self.env.step(self.actions, extras=False, auto_reset=True)

    def burn_in(self):
        """reach the steady state: one horizon with env i (re)started at step i mod horizon"""
        torch = self.torch
        self.env.reset()
        self.policy()
        if self.cfg["negotiate"]:
            self.env.negotiate(self.prop, self.acc, out=self.dec)
        if self.fam == "car":                                  # episodes end by themselves (~130 steps): just run
            for s in range(400):
                self.substep(s)
            return
        phase = torch.arange(self.E, device=self.dev, dtype=torch.int32) % HORIZON
        for s in range(HORIZON):
            if s % 50 == 0:
                self.policy()
            self.gen_actions(s)
            self.env.step(self.actions, extras=False)
            self.after_step((phase == s).to(torch.uint8))
        if self.stats is not None:
            self.stats.zero_()

    def outputs(self):
        """what a caller of `substep` receives from the last step: the env's output tensors (rewritten in place every
        step) and, with the negotiation prologue, the decisions of the envs that negotiated in it"""
        env = self.env
        out = {"obs": env.obs, "rew": env.rew, "done": env.done}
        if self.fam != "car":                      # selfdrive writes info only with extras=True
            out["info"] = env.info
        if self.cfg["negotiate"]:
            out["negotiation_decision"] = self.dec
        return out


DUMP_BYTES = 64 * 10 ** 6                      # npy headers fit in the 4 KB kept aside


def dump_outputs(run, stats_total, out_dir):
    """Write the last timed step's outputs as DIR/<name>.npy (float64 stays float64, everything else becomes float32).
    Arrays are sampled along the env axis to keep the dump under DUMP_BYTES: the same seeded sample of env indices
    (written as env_index.npy) for every array, so that two builds run with the same arguments can be compared."""
    import torch
    outs = run.outputs()
    per_env = 8 + sum(t[0].numel() * (8 if t.dtype == torch.float64 else 4) for t in outs.values())
    S = min(run.E, (DUMP_BYTES - 4096) // per_env)
    if S < run.E:
        idx = np.sort(np.random.RandomState(SEED).choice(run.E, S, replace=False))
    else:
        idx = np.arange(run.E)
    sel = torch.as_tensor(idx, device=run.dev)
    arrays = {"env_index": idx.astype(np.float64)}
    for name, t in outs.items():
        a = t.index_select(0, sel).cpu().numpy()
        arrays[name] = a if a.dtype == np.float64 else a.astype(np.float32)
    if stats_total is not None:
        arrays["episode_stats"] = np.asarray(stats_total, dtype=np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def pin_to_cores(local, world):
    """each rank's host threads on their own block of cores (the ranks share one NUMA node on these boxes)"""
    try:
        cpus = sorted(os.sched_getaffinity(0))
        per = len(cpus) // world
        if per >= 1:
            os.sched_setaffinity(0, cpus[local * per:(local + 1) * per])
            return cpus[local * per:(local + 1) * per]
    except Exception:
        pass
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cleanup8", choices=sorted(CONFIGS))
    ap.add_argument("--envs", type=int, default=0, help="envs per GPU (0 = the config's)")
    ap.add_argument("--e2e-steps", type=int, default=300)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--graph-steps", type=int, default=50, help="env steps per captured CUDA graph (1 = no graphs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last one as DIR/<name>.npy (rank 0's envs, a "
                         "fixed sample of them when they exceed 64 MB)")
    args = ap.parse_args()
    if args.impl == "reference":
        reference_arm(args)
        return

    import torch
    import torch.distributed as dist
    from contracts_b200 import sharding

    cfg = CONFIGS[args.config]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    cores = pin_to_cores(local, int(os.environ.get("LOCAL_WORLD_SIZE", world))) if world > 1 else None
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"          # keep NCCL's version banner off stdout (one JSON line only)
        dist.init_process_group("nccl", device_id=dev)
    E, n = (args.envs or cfg["envs"]), cfg["n"]
    K, W = max(args.steps, 1), max(args.warmup, 3)

    run = Runner(args.config, cfg, E, rank, dev)
    env = run.env
    main_stream = torch.cuda.current_stream(dev)
    side = torch.cuda.Stream(dev)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- episode statistics: device accumulator -> snapshot -> all-gather, all on a side stream (no rank blocks) ----
    gathered = {"out": None, "work": None}
    snap = torch.zeros(8, dtype=torch.float64, device=dev)
    gout = torch.zeros((world * 8,), dtype=torch.float64, device=dev)

    def gather_stats():
        if run.stats is None:
            return
        side.wait_stream(main_stream)
        with torch.cuda.stream(side):
            snap.copy_(run.stats)
            if world > 1:
                gathered["work"] = dist.all_gather_into_tensor(gout, snap, async_op=True)
            else:
                gout.copy_(snap)
        gathered["out"] = gout

    run.burn_in()
    barrier()

    # ---- CUDA graph of G consecutive steps (the inner loop is launch-bound from Python) --------------------
    G = max(1, min(args.graph_steps, K))
    while K % G:
        G -= 1
    graph, per_graph = None, 0
    if G > 1:
        cap = torch.cuda.Stream(dev)
        cap.wait_stream(main_stream)
        with torch.cuda.stream(cap):
            for _ in range(3):                                   # warm the capture stream
                run.substep()
        main_stream.wait_stream(cap)
        torch.cuda.synchronize(dev)
        graph = torch.cuda.CUDAGraph()
        lcap = env.kernel_launches
        with torch.cuda.graph(graph, stream=cap):
            for _ in range(G):
                run.substep()
        torch.cuda.synchronize(dev)
        per_graph = env.kernel_launches - lcap                   # kernels captured in one graph (counted by the C ABI)
    gstep = {"i": 0}

    def run_steps(k):
        """k env steps (a multiple of G); returns the number of graph-launched kernels"""
        launched = 0
        for _ in range(k // G):
            run.policy()
            if graph is not None:
                graph.replay()
                launched += per_graph
            else:
                run.substep(gstep["i"])
            gstep["i"] += G
        return launched

    gather_stats()                                               # NCCL's lazy communicator set-up happens here, untimed
    if gathered["work"] is not None:
        gathered["work"].wait()
    run_steps(max(G, (W + G - 1) // G * G))
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = env.kernel_launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    graph_launches = 0
    done_steps = 0
    while done_steps < K:                                        # one statistics all-gather per horizon (at least one)
        chunk = min(K - done_steps, HORIZON // G * G if HORIZON >= G else G)
        graph_launches += run_steps(chunk)
        done_steps += chunk
        gather_stats()
    main_stream.wait_stream(side)                                # the collective is inside the timed region
    ev1.record()
    barrier()
    launches = (env.kernel_launches - l0) + graph_launches       # eager launches are counted by the C ABI itself
    ms_total = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if rank == 0 else None
    tmax = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_total = float(tmax.item())
    value = world * E * n * K / (ms_total * 1e-3)
    stats_total = None
    if gathered["out"] is not None:
        if gathered["work"] is not None:
            gathered["work"].wait()
        g = gathered["out"].view(world, 8)
        stats_total = g.sum(0)
        stats_total[7] = g[:, 7].max()
        stats_total = stats_total.tolist()
    if args.dump_outputs and rank == 0:
        dump_outputs(run, stats_total, args.dump_outputs)

    # ---- the step kernels alone (roofline): CUDA events around each step call of an un-graphed stretch -------
    Kk = 200
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(Kk)]
    run.policy()
    # (the event pair brackets the step kernels only: the finished envs are reset by a separate call here)
    grid = cfg["family"] == "grid"
    for k in range(Kk):
        run.gen_actions()
        kev[k][0].record()
        if grid:
            env.step(run.actions, extras=False)
        else:
            env.step(run.actions, extras=False, auto_reset=True)
        kev[k][1].record()
        if grid:
            run.after_step()
    barrier()
    step_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))
    kern_ms = None
    if cfg["family"] == "grid":
        # per-kernel split of the step (library-side CUDA events around each kernel)
        try:
            env.enable_timing(True)
            acc = []
            for k in range(100):
                run.gen_actions()
                env.step(run.actions, extras=False)
                acc.append(env.step_times_ms())
                run.after_step()
            kern_ms = (float(np.mean([a for a, _ in acc])), float(np.mean([b for _, b in acc])))
        except Exception as exc:
            print("per-kernel timing unavailable: %s" % exc, file=sys.stderr)
        finally:
            env.enable_timing(False)
        barrier()

    # ---- e2e: host actions in, host results out, every step ------------------------------------------------
    Ke = max(2, min(args.e2e_steps, max(K, 50)))
    nact = cfg.get("nact", 0)
    if cfg["family"] == "car":
        host_actions = [(torch.rand((E, n), dtype=torch.float32) * 0.2 - 0.1).pin_memory() for _ in range(4)]
    else:
        host_actions = [torch.randint(0, nact, (E, n), dtype=torch.uint8).pin_memory() for _ in range(4)]
    consumed = 0
    res = [env.new_host_result(), env.new_host_result()]
    lay = res[0].lay
    if True:
        def e2e_run(steps):
            """pipelined two deep: submit step i + 1, then wait for (and read) the result block of step i"""
            nonlocal consumed
            prev = None
            for i in range(steps):
                if i % 50 == 0:
                    run.policy()
                if cfg["family"] == "grid":
                    tk = env.step_host_async(host_actions[i % 4], res[i & 1], auto_reset=True, negotiation=run.neg())
                else:
                    tk = env.step_host_async(host_actions[i % 4], res[i & 1], auto_reset=True)
                if prev is not None:
                    env.step_host_wait(prev[0])
                    consumed += prev[1].count + int(prev[1].done.flat[0])
                prev = (tk, res[i & 1])
            env.step_host_wait(prev[0])
            consumed += prev[1].count
        e2e_note = ("ssd_step_host_async/_wait, two steps in flight: pinned %s actions up on a copy-in stream, ONE lossless "
                    "result block down per step (int8 rewards + exact float64 records of the envs that paid a transfer + dones) "
                    "while the %s runs; observations stay in the device batch tensor"
                    % ("float32" if cfg["family"] == "car" else "uint8", "observe kernel" if cfg["family"] == "grid" else "next step"))
    e2e_run(5)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    e2e_run(Ke)
    e1.record()
    barrier()
    e2e_ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_value = world * E * n * Ke / (float(e2e_ms.item()) * 1e-3)
    rec_mean = float(np.mean([r.count for r in res]))
    d2h = int(lay.records_offset + min(lay.record_capacity, 1.25 * rec_mean + 1024) * lay.record_bytes)      # the prefix ssd_step_host_async sends
    h2d = E * n * host_actions[0].element_size()
    # informational: also ship the observations to the host (PCIe-bound by construction)
    obs_to_host = None
    if rank == 0 and cfg["family"] == "grid":
        host_obs = torch.empty(env._obs_buf.shape, dtype=torch.uint8).pin_memory()
        Ko = 10
        torch.cuda.synchronize(dev)
        o0, o1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        o0.record()
        for i in range(Ko):
            tk = env.step_host_async(host_actions[i % 4], res[i & 1], auto_reset=True, negotiation=run.neg())
            host_obs.copy_(env._obs_buf, non_blocking=True)
            env.step_host_wait(tk)
            main_stream.synchronize()
        o1.record()
        torch.cuda.synchronize(dev)
        obs_to_host = {"value": E * n * Ko / (o0.elapsed_time(o1) * 1e-3), "unit": "agent-steps/s",
                       "d2h_bytes_per_step": E * n * 675 + d2h}
    barrier()

    if rank == 0:
        peak, peak_src = measured_peak()
        achieved = cfg["alg"] * E * n / (step_ms * 1e-3) / 1e9
        step_kernels = {"grid": "grid_logic_kernel + grid_obs_kernel" + (" + grid_reward_kernel" if cfg.get("env") == "harvest_new" else ""),
                        "feat": "feat_step_kernel", "car": "car_step_kernel"}[cfg["family"]]
        state_b = getattr(env, "state_bytes_per_env", 0)
        obs_b = E * n * 675 if cfg["family"] == "grid" else env.obs.numel() * 8
        line = {
            "metric": "agent-steps/sec", "value": value, "unit": "agent-steps/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8" if cfg["family"] == "grid" else "f64", "data": "synthetic",
            "config": dict(config_dict(args.config, cfg, E, world), **{
                       "phase": "steady state of a vectorised sampler: env i's episodes start at steps = i mod horizon "
                                "(untimed burn-in of one horizon); ~E/horizon envs finish, reset and negotiate in EVERY "
                                "timed step, so any window carries the episode boundary pro rata",
                       "l2": "working set %.0f MB/step (outputs %.0f MB + state) exceeds the 126 MB L2" % (
                           (obs_b + 2.0 * E * state_b) / 1e6, obs_b / 1e6),
                       "cuda_graph_steps": G, "host_cores_per_rank": len(cores) if cores else None}),
            "e2e": {"value": e2e_value, "unit": "agent-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": Ke, "note": e2e_note, "consumed": consumed},
            "e2e_obs_to_host": obs_to_host,
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": ncu_traffic(args.config, E, n), "alg_bytes_per_launch": cfg["alg"] * E * n,
                         "peak_source": peak_src,
                         "kernel": "one env step (CUDA events around the step call on its stream): " + step_kernels,
                         "kernel_ms": step_ms, "alg_bytes_per_agent_step": cfg["alg"],
                         "share_of_timed_step": step_ms / (ms_total / K)},
        }
        if kern_ms is not None:
            # the dominant kernel on its own: the observation stream + the env's 128-byte hot line (read; its mask words
            # written back when the spawn changed them)
            obs_alg = (n * 675 + 128 + 32) * E
            line["roofline"]["kernels"] = [
                {"name": "grid_logic_kernel", "ms": kern_ms[0]},
                {"name": "grid_obs_kernel" + (" + grid_reward_kernel" if cfg.get("env") == "harvest_new" else ""), "ms": kern_ms[1],
                 "alg_bytes_per_launch": obs_alg, "achieved": obs_alg / (kern_ms[1] * 1e-3) / 1e9,
                 "frac": obs_alg / (kern_ms[1] * 1e-3) / 1e9 / peak}]
        if stats_total is not None:
            s = stats_total
            line["episode_stats"] = {"apples_eaten": s[0], "raw_env_rewards": s[1], "transfers": s[2], "dirt_cleaned": s[3],
                                     "episodes": s[6], "err_flags": s[7]}
        if world == 1 and not args.no_cpu:
            ref, port = cpu_arms(args.config, cfg)
            if ref is not None:
                line["cpu_baseline"] = ref
                if port is not None:
                    line["cpu_baseline_port"] = port
            elif port is not None:
                line["cpu_baseline"] = port
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
