"""Classic-control envs on the GPU (classic_control.cu, DESIGN.md §3.13): what they cost and what they buy.

  kernel    ppx_classic_step per env and N (2048, 2^20): us per step from CUDA events over 200 launches, and the model GB/s
            of the byte model below over that time.  At 2^20 envs the working set exceeds the 126 MB L2 for CartPole only.
  collect   collect_samples() at C2's learner shape (PPO+SimHash k=64, h 64, 2048 envs x 256 steps, swimmer_ppo hparams) on
            MountainCarContinuous-v0, bare and under make_env's VecNormalize, against the table env of tools/collect_prof.py
            (obs 8); arms alternate; libppx launches per step.
  target    wall clock of learn(reward_target=...) from a fixed seed on the device path and on the host loop over
            ToNumpy of the same env (bit-identical runs, so both stop at the same iteration or neither does): PPO on
            CartPole-v1 (target 475) and PPO+SimHash on MountainCar-v0 (target -110), each within a stated timestep budget.
  es        EvolutionStrategy.run_generation on MountainCarContinuous-v0 at C5's population (P = 10 000, MLP 2-64-64-1).

    python tools/envs_prof.py [--out profiles/envs_r04.json] [--skip-target]
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
import bench  # noqa: E402
import ppo_exploration_b200 as ppx  # noqa: E402
from ppo_exploration_b200 import _lib as L  # noqa: E402
from ppo_exploration_b200.classic_control import ENVS  # noqa: E402
from collect_prof import TableEnv, gpu_meta  # noqa: E402


def step_bytes(S, D):
    """Bytes one env moves per step: state S*8 read + written, elapsed / monitor return / monitor length 8 each read +
    written, the action 8 read, obs 4*D, reward 4, done 1 and the behaviour row S*8 written (the episode counter and the
    episode statistics are touched only by finished envs and not counted)."""
    return 2 * 8 * S + 3 * 16 + 8 + 4 * D + 4 + 1 + 8 * S


def kernel_arm():
    out = {}
    for env_id, (_, S, D, _, space) in ENVS.items():
        for N in (2048, 1 << 20):
            env = ppx.ClassicControlVecEnv(env_id, N, seed=0)
            env.reset()
            discrete = isinstance(env.action_space, ppx.Discrete)
            a = (torch.randint(0, env.action_space.n, (N,), device="cuda") if discrete
                 else torch.randn(N, 1, dtype=torch.float64, device="cuda"))
            for _ in range(20):
                env.step(a)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 200
            e0.record()
            for _ in range(reps):
                env.step(a)
            e1.record()
            torch.cuda.synchronize()
            us = e0.elapsed_time(e1) * 1e3 / reps
            b = step_bytes(S, D) * N
            out[f"{env_id}/N={N}"] = dict(us_per_step=round(us, 3), ns_per_env_step=round(us * 1e3 / N, 4),
                                          model_bytes=b, model_gb_s=round(b / (us * 1e-6) / 1e9, 1))
    return out


def collect_arm(reps):
    cfg = bench.CONFIGS["C2"]
    T, N, h = cfg["T"], cfg["N"], cfg["hidden"]
    envs = {"table_env_obs8": lambda: TableEnv(N, cfg["D"], T + 1, torch.device("cuda"), False),
            "mcc_bare": lambda: ppx.ClassicControlVecEnv("MountainCarContinuous-v0", N, seed=0),
            "mcc_vecnormalize": lambda: ppx.make_env("MountainCarContinuous-v0", N, seed=0)}
    arms = {}
    for name, mk in envs.items():
        np.random.seed(0)
        torch.manual_seed(0)
        m = ppx.PPO(env=mk(), nstep=T, batch_size=cfg["batch"], hidden_size=h, sim_hash=True, hash_bits=cfg["hash_bits"], **cfg["hp"])
        assert m.device_env
        for _ in range(3):
            m.collect_samples()
            m.train()
        arms[name] = dict(m=m, ms=[], launches=0)
    for _ in range(reps):
        for name, a in arms.items():
            m = a["m"]
            torch.cuda.synchronize()
            n0, t0 = L.launch_count(), time.perf_counter()
            m.collect_samples()
            torch.cuda.synchronize()
            a["ms"].append((time.perf_counter() - t0) * 1e3)
            a["launches"] = L.launch_count() - n0
            m.train()
    res = {}
    for name, a in arms.items():
        med = statistics.median(a["ms"])
        res[name] = dict(collect_ms_median=round(med, 3), collect_ms=[round(x, 3) for x in a["ms"]],
                         us_per_env_step=round(med * 1e3 / T, 2), libppx_launches_per_collect=a["launches"],
                         libppx_launches_per_step=round(a["launches"] / T, 3))
    return res


TARGETS = {
    "CartPole-v1": dict(target=475.0, budget=300_000, n_envs=8, sim_hash=False,
                        kw=dict(nstep=32, batch_size=256, n_epochs=20, gamma=0.98, gae_lam=0.8, lr=1e-3, ent_coef=0.0,
                                hidden_size=64)),
    "MountainCar-v0": dict(target=-110.0, budget=300_000, n_envs=16, sim_hash=True,
                           kw=dict(nstep=16, batch_size=256, n_epochs=4, gamma=0.99, gae_lam=0.98, ent_coef=0.0,
                                   hidden_size=64)),
}


def target_arm():
    res = {}
    for env_id, c in TARGETS.items():
        for path in ("device", "host_loop"):
            env = ppx.ClassicControlVecEnv(env_id, c["n_envs"], seed=0)
            if path == "host_loop":
                env = ppx.ToNumpy(env)
            np.random.seed(0)
            torch.manual_seed(0)
            m = ppx.PPO(env=env, sim_hash=c["sim_hash"], **c["kw"])
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            m.learn(total_timesteps=c["budget"], log_interval=None, reward_target=c["target"])
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            buf = [e["r"] for e in m.ep_info_buffer]
            mean = float(np.mean(buf)) if buf else None
            res[f"{env_id}/{path}"] = dict(
                target=c["target"], timestep_budget=c["budget"], n_envs=c["n_envs"], sim_hash=c["sim_hash"], hparams=c["kw"],
                reached=bool(mean is not None and mean > c["target"]), timesteps=int(m.num_timesteps), episodes=int(m.num_episodes),
                final_ep_rew_mean=None if mean is None else round(mean, 3), wall_s=round(wall, 3))
    return res


def es_arm(gens):
    P = 10_000
    np.random.seed(0)
    es = ppx.EvolutionStrategy(hidden_sizes=(64, 64), obs_dim=2, n_actions=1, population_size=P, sigma=0.1)
    env = ppx.ClassicControlVecEnv("MountainCarContinuous-v0", P, seed=0, reward_dtype=torch.float64)
    es.run_generation(env, max_steps=999)
    times, steps, lens = [], [], []
    for _ in range(gens):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fit, ln, _ = es.run_generation(env, max_steps=999)
        torch.cuda.synchronize()
        times.append((time.perf_counter() - t0) * 1e3)
        steps.append(int(es.last_eval_steps))
        lens.append(float(ln.double().mean()))
    return dict(population=P, network="2-64-64-1 tanh", max_steps=999, generation_ms_median=round(statistics.median(times), 3),
                generation_ms=[round(x, 3) for x in times], loop_steps=steps, mean_episode_length=[round(x, 1) for x in lens])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "envs_r04.json"))
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--skip-target", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("envs_prof.py measures on the GPU; no CUDA device found")
    torch.cuda.set_device(0)
    out = dict(gpu_meta(), tool="tools/envs_prof.py")
    out["kernel"] = dict(byte_model="per env and step: 2*8*S state + 3*16 counters + 8 action + 4*D obs + 4 reward + 1 done + "
                         "8*S behaviour bytes", arms=kernel_arm())
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)

    def save():                                                 # after every arm: a later failure keeps the earlier numbers
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(out["kernel"]["arms"]), flush=True)
    save()
    out["collect"] = collect_arm(args.reps)
    print(json.dumps({k: {kk: vv for kk, vv in v.items() if kk != "collect_ms"} for k, v in out["collect"].items()}), flush=True)
    save()
    out["es"] = es_arm(5)
    print(json.dumps(out["es"]), flush=True)
    save()
    if not args.skip_target:
        out["target"] = target_arm()
        print(json.dumps(out["target"]), flush=True)
        save()


if __name__ == "__main__":
    main()
