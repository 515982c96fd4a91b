"""collect_samples() at C2's shape on its two paths: an env that lives on the GPU (device path: three libppx launches per
step, no host sync, SimHash once per rollout) against the same env returning numpy (the reference's host loop: per-step
D2H of the actions, uploads and per-step SimHash).

The env is a table lookup (observations / rewards / dones precomputed for every step, on the device for one arm and on
the host for the other), so what is timed is the learner's side of the loop.  It returns no infos; a third arm, the device
env returning the VecEnv convention's list of N (empty) info dicts, shows what update_info_buffer's Python loop over them
costs per step.  The arms alternate within one run.
Per arm: ms per collect_samples(), us per env step, libppx launches per step, ms per collect_samples() + train() (one
learn() iteration).  The GPU's name and power limit are recorded with the numbers.

    python tools/collect_prof.py [--reps 7] [--out profiles/collect_r03.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
import ppo_exploration_b200 as ppx  # noqa: E402
from ppo_exploration_b200 import _lib as L  # noqa: E402


class TableEnv:
    """Observations, rewards and dones read from [L, N, ...] tables: torch CUDA (device arm) or numpy (host arm)."""

    def __init__(self, n, d, length, device, infos, seed=0):
        rs = np.random.RandomState(seed)
        tabs = (rs.randn(length, n, d).astype(np.float32), rs.randn(length, n).astype(np.float32), rs.rand(length, n) < 0.01)
        self.tabs = [torch.as_tensor(a).to(device) for a in tabs] if device is not None else tabs
        self.num_envs, self.length = n, length
        self.observation_space, self.action_space = ppx.Box((d,)), ppx.Box((2,))
        self.infos = [{} for _ in range(n)] if infos else []

    def reset(self):
        self.t = 0
        return self.tabs[0][0]

    def step(self, actions):
        self.t += 1
        k = self.t % self.length
        rew = self.tabs[1][k]
        if isinstance(rew, np.ndarray):
            rew = rew.copy()                                    # the host loop's SimHash adds its bonus into the array it gets
        return self.tabs[0][k], rew, self.tabs[2][k], self.infos

    def unnormalize_obs(self, obs):
        return obs


def gpu_meta():
    meta = {"gpu": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                              "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        meta.update(gpu_smi=out[0].strip(), power_limit_w=float(out[1]), sm_max_mhz=float(out[2]))
    except Exception as e:                                      # the numbers stay usable; say what is missing
        meta["power_limit_w"] = f"unavailable ({e})"
    return meta


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=os.path.join("profiles", "collect_r03.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("collect_prof.py measures on the GPU; no CUDA device found")
    cfg = bench.CONFIGS["C2"]
    T, N, D, h = cfg["T"], cfg["N"], cfg["D"], cfg["hidden"]
    dev = torch.device("cuda", 0)
    arms = {}
    for name, env_dev, infos in (("device", dev, False), ("host", None, False), ("device_n_infos", dev, True)):
        np.random.seed(0)
        torch.manual_seed(0)
        env = TableEnv(N, D, T + 1, env_dev, infos)
        m = ppx.PPO(env=env, nstep=T, batch_size=cfg["batch"], hidden_size=h, sim_hash=True, hash_bits=cfg["hash_bits"],
                    device=dev, **cfg["hp"])
        assert m.device_env == (env_dev is not None)
        for _ in range(3):                                      # eager, graph capture, replay
            m.collect_samples()
            m.train()
        arms[name] = dict(m=m, collect_ms=[], learn_ms=[], launches=[])
    for _ in range(args.reps):
        for name, a in arms.items():
            m = a["m"]
            torch.cuda.synchronize()
            n0, t0 = L.launch_count(), time.perf_counter()
            m.collect_samples()
            torch.cuda.synchronize()
            a["collect_ms"].append((time.perf_counter() - t0) * 1e3)
            a["launches"].append(L.launch_count() - n0)
            m.train()                                           # keeps the two calls of the next row in step
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            m.collect_samples()
            m.train()                                           # ends in its one loss read-back (a device synchronise)
            torch.cuda.synchronize()
            a["learn_ms"].append((time.perf_counter() - t0) * 1e3)
    out = dict(gpu_meta(), tool="tools/collect_prof.py", reps=args.reps, workload=(
        f"C2 shape: PPO+SimHash k={cfg['hash_bits']}, obs {D}, Box(2), h {h}, {N} envs x {T} steps, swimmer_ppo hparams; "
        "table-lookup env (no per-step env work, no infos; device_n_infos: N empty info dicts per step); arms alternate"), arms={})
    for name, a in arms.items():
        med = statistics.median(a["collect_ms"])
        out["arms"][name] = dict(collect_ms_median=round(med, 3), collect_ms=[round(x, 3) for x in a["collect_ms"]],
                                 us_per_env_step=round(med * 1e3 / T, 2), launches_per_step=a["launches"][-1] / T,
                                 learn_iteration_ms_median=round(statistics.median(a["learn_ms"]), 3),
                                 learn_iteration_ms=[round(x, 3) for x in a["learn_ms"]])
    out["collect_speedup"] = round(out["arms"]["host"]["collect_ms_median"] / out["arms"]["device"]["collect_ms_median"], 2)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: v for k, v in out.items() if k != "arms"}))
    for name, a in out["arms"].items():
        print(name, {k: v for k, v in a.items() if not isinstance(v, list)})


if __name__ == "__main__":
    main()
