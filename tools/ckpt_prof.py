"""Checkpoints (DESIGN.md §3.14): what a save and a restore cost.

  table     ppx_count_table_load at 2^20 and 2^24 random keys: keys/s from CUDA events around the load (the table, at
            capacity 2^21 / 2^25 with 12 bytes a slot, and the 12 bytes a key of input exceed the 126 MB L2 at 2^24 only;
            at 2^20 the 24 MB table fits it).  The create / empty check / readback around the kernel are not in the window;
            `load_ms` is the whole synchronous call, host clock.
  learner   save() and load() wall time, and file size, for C2's learner (PPO+SimHash k = 64, 2048 envs, h = 64, 256 steps,
            swimmer_ppo hparams) after 20 iterations on MountainCarContinuous-v0 under make_env's VecNormalize.

    python tools/ckpt_prof.py [--out profiles/ckpt_r05.json]
"""
import argparse
import json
import os
import statistics
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
import ppo_exploration_b200 as ppx  # noqa: E402
from ppo_exploration_b200 import _lib as L  # noqa: E402
from collect_prof import gpu_meta  # noqa: E402
import ctypes as C  # noqa: E402


def table_arm(reps):
    out = {}
    rs = np.random.RandomState(0)
    for lg in (20, 24):
        n = 1 << lg
        keys = torch.from_numpy(rs.randint(-(1 << 62), 1 << 62, size=n, dtype=np.int64)).unique().cuda()
        counts = torch.from_numpy(rs.randint(1, 1000, size=keys.numel()).astype(np.int32)).cuda()
        n = keys.numel()
        cap = 1 << (lg + 1)
        ev_ms, call_ms = [], []
        for r in range(reps + 1):
            h = C.c_void_p()
            L.call("ppx_count_table_create", cap, C.byref(h))
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            L.call("ppx_count_table_load", h, keys.data_ptr(), counts.data_ptr(), n, L.stream())
            e1.record()
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            got = C.c_uint64()
            L.call("ppx_count_table_size", h, C.byref(got))
            assert got.value == n
            L.call("ppx_count_table_destroy", h)
            if r:                                               # the first call warms the module
                ev_ms.append(e0.elapsed_time(e1))
                call_ms.append((t1 - t0) * 1e3)
        med = statistics.median(ev_ms)
        out[f"2^{lg}"] = dict(keys=n, capacity=cap, event_ms_median=round(med, 3), event_ms=[round(x, 3) for x in ev_ms],
                              keys_per_s=round(n / (med * 1e-3), 0), load_ms_median=round(statistics.median(call_ms), 3))
    return out


def learner_arm(reps, iters=20):
    cfg = bench.CONFIGS["C2"]
    T, N, h = cfg["T"], cfg["N"], cfg["hidden"]
    np.random.seed(0)
    torch.manual_seed(0)

    def mk():
        return ppx.make_env("MountainCarContinuous-v0", N, seed=0)
    m = ppx.PPO(env=mk(), nstep=T, batch_size=cfg["batch"], hidden_size=h, sim_hash=True, hash_bits=cfg["hash_bits"], **cfg["hp"])
    for _ in range(iters):
        m.collect_samples()
        m.train()
    torch.cuda.synchronize()
    save_ms, load_ms = [], []
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "c2.pt")
        for r in range(reps + 1):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            m.save(p)
            t1 = time.perf_counter()
            b = ppx.PPO.load(p, env=mk())
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            assert b.resumed_env_state and torch.equal(b.policy.bank.flat, m.policy.bank.flat)
            del b
            if r:
                save_ms.append((t1 - t0) * 1e3)
                load_ms.append((t2 - t1) * 1e3)
        size = os.path.getsize(p)
        n_keys = len(m.rollout.count_table)
    return dict(workload=f"C2 learner (PPO+SimHash k={cfg['hash_bits']}, {N} envs x {T} steps, h {h}) after {iters} iterations "
                         "on MountainCarContinuous-v0 + VecNormalize",
                count_table_keys=n_keys, policy_params=int(m.policy.bank.size), file_bytes=size,
                save_ms_median=round(statistics.median(save_ms), 2), save_ms=[round(x, 2) for x in save_ms],
                load_ms_median=round(statistics.median(load_ms), 2), load_ms=[round(x, 2) for x in load_ms])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "ckpt_r05.json"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ckpt_prof.py measures on the GPU; no CUDA device found")
    torch.cuda.set_device(0)
    out = dict(gpu_meta(), tool="tools/ckpt_prof.py")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    out["table"] = table_arm(args.reps)
    print(json.dumps(out["table"]), flush=True)
    out["learner"] = learner_arm(args.reps)
    print(json.dumps(out["learner"]), flush=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
