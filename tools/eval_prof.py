"""Policy evaluation on envs on the GPU (evaluate.cu, DESIGN.md §3.17): what a step of `evaluate_policy` costs.

  loop      per-step wall time of `ppx.evaluate_policy` (deterministic; forward + ppx_policy_act_eval + env.step +
            ppx_eval_episode_step, no sync) against the host loop over `ppx.ToNumpy` of the same env (`predict` on numpy
            observations, one sync per step), at C2's policy shape (2048 envs, h 64) on MountainCarContinuous-v0 and
            CartPole-v1.  Both arms run a fixed number of steps (the episode target is never reached); arms alternate.
  kernels   CUDA-event time of ppx_policy_act_eval (Box / Discrete, deterministic / stochastic) and ppx_eval_episode_step
            at N = 2048 and N = 2^20, over 1000 back-to-back launches.
  meta      the card's name and power limit, read in the same run.

    python tools/eval_prof.py [--out profiles/eval_r08.json] [--steps 400] [--reps 5]
"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import ppo_exploration_b200 as ppx  # noqa: E402
from ppo_exploration_b200 import _lib as L  # noqa: E402
from collect_prof import gpu_meta  # noqa: E402

N, H = 2048, 64


class Counting:
    """Counts env.step calls (the device loop's step count) and forwards the env surface."""

    def __init__(self, env):
        self.env, self.steps = env, 0
        self.num_envs, self.observation_space, self.action_space = env.num_envs, env.observation_space, env.action_space
        self.episode_stats = env.episode_stats

    def reset(self):
        return self.env.reset()

    def step(self, a):
        self.steps += 1
        return self.env.step(a)


def loop_arm(steps, reps):
    res = {}
    for env_id in ("MountainCarContinuous-v0", "CartPole-v1"):
        np.random.seed(0)
        torch.manual_seed(0)
        m = ppx.PPO(env=ppx.ClassicControlVecEnv(env_id, N, seed=0), nstep=16, batch_size=4096, n_epochs=1, hidden_size=H)
        assert m.policy.mlp._fused_args()["tc"]
        n_eval = N * 128                                       # not reached within `steps` steps: both arms run them all

        def device():
            env = Counting(ppx.ClassicControlVecEnv(env_id, N, seed=1))
            torch.cuda.synchronize()
            n0, t0 = L.launch_count(), time.perf_counter()
            ppx.evaluate_policy(m, env, n_eval, max_steps=steps)      # ends in a read of the tables: synchronised
            return (time.perf_counter() - t0) * 1e6 / env.steps, (L.launch_count() - n0 - 1) / env.steps

        def host():
            env = ppx.ToNumpy(ppx.ClassicControlVecEnv(env_id, N, seed=1))
            torch.cuda.synchronize()
            n0, t0 = L.launch_count(), time.perf_counter()
            obs = env.reset()
            for _ in range(steps):
                obs, _, _, _ = env.step(m.predict(obs))
            torch.cuda.synchronize()
            return (time.perf_counter() - t0) * 1e6 / steps, (L.launch_count() - n0 - 1) / steps

        arms = {"evaluate_policy": device, "host_loop_to_numpy": host}
        for f in arms.values():                                 # warm-up
            f()
        us = {k: [] for k in arms}
        launches = {}
        for _ in range(reps):
            for k, f in arms.items():
                t, n = f()
                us[k].append(t)
                launches[k] = n
        res[env_id] = {k: dict(us_per_step_median=round(statistics.median(v), 2), us_per_step=[round(x, 2) for x in v],
                               libppx_launches_per_step=round(launches[k], 3)) for k, v in us.items()}
        res[env_id]["speedup_median"] = round(res[env_id]["host_loop_to_numpy"]["us_per_step_median"]
                                              / res[env_id]["evaluate_policy"]["us_per_step_median"], 2)
    return res


def _events(fn, reps=1000):
    for _ in range(20):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return round(e0.elapsed_time(e1) * 1e3 / reps, 3)


def kernel_arm():
    out = {}
    st = L.stream()
    draw = (1 << 63) | (1 << 32)
    for n in (N, 1 << 20):
        for name, A, discrete in (("box_A1", 1, 0), ("discrete_A2", 2, 1)):
            x = torch.randn(n, A, device="cuda")
            ls = torch.zeros(A, device="cuda")
            act = torch.empty((n,) if discrete else (n, A), dtype=torch.int64 if discrete else torch.float64, device="cuda")
            for det in (1, 0):
                out[f"policy_act_eval/{name}/{'det' if det else 'stoch'}/N={n}"] = _events(
                    lambda: L.call("ppx_policy_act_eval", x.data_ptr(), ls.data_ptr(), n, A, discrete, det, 7, draw, 0,
                                   act.data_ptr(), st))
        kmax = 4
        dones = (torch.rand(n, device="cuda") < 0.05).to(torch.uint8)
        ret, lens = torch.randn(n, dtype=torch.float64, device="cuda"), torch.ones(n, dtype=torch.int64, device="cuda")
        counts, state = torch.zeros(n, dtype=torch.int64, device="cuda"), torch.zeros(3, dtype=torch.int64, device="cuda")
        tr, tl, te = (torch.zeros(n, kmax, dtype=d, device="cuda") for d in (torch.float64, torch.int64, torch.int64))
        # the tables fill during the warm-up, so the timed launches are the common step: read the done flags and counts,
        # count the missing episodes, publish the count
        out[f"eval_episode_step/N={n}"] = _events(
            lambda: L.call("ppx_eval_episode_step", dones.data_ptr(), ret.data_ptr(), lens.data_ptr(), n, n * kmax, 0, n, 0,
                           counts.data_ptr(), tr.data_ptr(), tl.data_ptr(), te.data_ptr(), kmax, state.data_ptr(), st))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "eval_r08.json"))
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    res = {"meta": gpu_meta(), "shape": dict(n_envs=N, hidden_size=H, steps=args.steps, reps=args.reps),
           "loop": loop_arm(args.steps, args.reps), "kernels_us": kernel_arm()}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
