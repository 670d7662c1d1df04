"""Rate of ssd_checkpoint_save / ssd_checkpoint_load (full batch) against a device-to-device copy of the same bytes.

    python tools/bench_checkpoint.py [--envs 131072] [--iters 100] [--out profiles/checkpoint_bench.json]

Per config (cleanup_new n=8, cleanup features n=8, selfdrive n=8): the C entry points on every env (kernel only, CUDA
events over --iters launches after a warm-up), the Python API with and without observations (env.checkpoint() /
env.restore(), which add the allocation, the observation gather / scatter and restore's one synchronisation), and a
torch device-to-device copy of the row bytes as the yardstick.  A rate counts the bytes read plus the bytes written:
2 x E x row_bytes for the state (+ 2 x the observation bytes for the with-obs API numbers).  State + rows of a config are
67-122 MB at E = 131072, comparable to the 126 MB L2: the copy yardstick has the same footprint, so the ratio compares
like with like.  Prints one JSON object with the GPU's name and power limit.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    import torch
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q}


def timed_ms(fn, iters, warmup=5):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def make(name, E):
    if name == "cleanup_new_n8":
        from contracts_b200.batched import BatchedGridEnv
        return BatchedGridEnv("cleanup_new", E, 8, contract="CleanupContract")
    if name == "cleanup_features_n8":
        from contracts_b200.features import BatchedFeatureEnv
        return BatchedFeatureEnv("cleanup", E, 8, contract="CleanupContract")
    from contracts_b200.selfdrive import BatchedCarEnv
    return BatchedCarEnv(E, 8, contract="SelfdriveContractDistprop")


def bench(name, E, iters):
    import torch
    from contracts_b200 import _lib
    env = make(name, E)
    env.reset()
    for t in range(20):                                   # some state worth moving
        act = env.random_actions(t) if name == "selfdrive_n8" else env.random_actions(t, 9)
        env.step(act, auto_reset=True)
    lay = env.checkpoint_layout()
    rb = int(lay.row_bytes)
    rows = torch.empty((E, rb), dtype=torch.uint8, device=env.device)
    ok = torch.empty((E,), dtype=torch.uint8, device=env.device)
    stream = env._stream()
    rp, okp = ctypes.c_void_p(rows.data_ptr()), ctypes.c_void_p(ok.data_ptr())
    save = lambda: _lib.check(env._h, env.lib.ssd_checkpoint_save(env._h, None, E, rp, stream))
    load = lambda: _lib.check(env._h, env.lib.ssd_checkpoint_load(env._h, ctypes.c_uint64(lay.config_tag), None, E, rp, okp, stream))
    save()
    state_bytes = 2 * E * rb
    src = torch.empty((E * rb,), dtype=torch.uint8, device=env.device).random_(0, 255)
    dst = torch.empty_like(src)
    t_copy = timed_ms(lambda: dst.copy_(src), iters)
    t_save, t_load = timed_ms(save, iters), timed_ms(load, iters)
    assert bool(ok.all()), "a full-batch load rejected rows of the handle's own state"
    obs_bytes = 2 * env.obs.numel() * env.obs.element_size()
    ck = env.checkpoint()
    api = {}
    for with_obs in (False, True):
        ck_i = env.checkpoint(with_obs=with_obs)
        t_ck = timed_ms(lambda: env.checkpoint(with_obs=with_obs), max(iters // 5, 10))
        t_rs = timed_ms(lambda: env.restore(ck_i), max(iters // 5, 10))
        moved = state_bytes + (obs_bytes if with_obs else 0)
        api["with_obs" if with_obs else "no_obs"] = {
            "checkpoint_ms": round(t_ck, 4), "restore_ms": round(t_rs, 4),
            "checkpoint_GBps": round(moved / t_ck / 1e6, 1), "restore_GBps": round(moved / t_rs / 1e6, 1)}
    del ck
    copy_rate = state_bytes / t_copy / 1e6
    return {"config": name, "envs": E, "row_bytes": rb, "state_MB": round(E * rb / 1e6, 2),
            "copy_ms": round(t_copy, 4), "copy_GBps": round(copy_rate, 1),
            "save_ms": round(t_save, 4), "save_GBps": round(state_bytes / t_save / 1e6, 1),
            "save_vs_copy": round(t_copy / t_save, 3),
            "load_ms": round(t_load, 4), "load_GBps": round(state_bytes / t_load / 1e6, 1),
            "load_vs_copy": round(t_copy / t_load, 3), "api": api}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--envs", type=int, default=131072)
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_checkpoint needs a CUDA device")
    res = {"host": gpu_info(), "results": [bench(n, args.envs, args.iters)
                                           for n in ("cleanup_new_n8", "cleanup_features_n8", "selfdrive_n8")]}
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
