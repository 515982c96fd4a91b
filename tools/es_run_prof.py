"""EvolutionStrategy.run (ES-NSRA over a meta-population of M = 2 brains, DESIGN.md §3.15) on envs that live on the GPU.

Two shapes, P = 10 000 members each:
  * C5: MLP 8-64-64-2 (D = 4736) on es_eval_prof.py's table env (episodes of 250..1000 steps, behavior() of 2 columns),
    noise table 2^28 f32, the brain env the same table env with M rows;
  * MountainCarContinuous-v0 (ClassicControlVecEnv, f64 rewards), MLP 2-64-64-1, max_steps 999, brain env M envs.
Per generation: host wall time (run() reads the device once per generation, so the sum over generations is the run's wall
time), split by host clocks around the population loop (ask + evaluate + tell), the brain loop, the novelty read (the
knn launch's wait plus the blocking read) and the rest, with the steps each loop issued; and `ppx_es_act_rows` per step
(CUDA events over many launches) against its byte model M x (8 D + 4 D + 4 D0 + 8 A).  Then ES on CartPole-v1
(P = 1024, MLP 4-64-64-2, seed 0) run to reward_target 475 on f_b within a generation budget: wall clock and generations,
or "not reached".  The GPU's name and power limit are recorded with the numbers.

    python tools/es_run_prof.py [--out profiles/es_run_r06.json]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ppo_exploration_b200 as ppx  # noqa: E402
from ppo_exploration_b200 import _lib as L  # noqa: E402
from es_eval_prof import TableEnv, gpu_meta, time_events  # noqa: E402

P, M = 10_000, 2


def instrument(es):
    """Host clocks around the parts of a generation; returns the dict the wrappers fill."""
    acc = dict(population=[], brains=[], read=[], pop_steps=[], brain_steps=[])
    ask, evaluate, tell, brains, read = es.ask, es.evaluate, es.tell, es._brains, es._run_read
    cur = {}

    def t_ask(*a, **k):
        cur["t0"] = time.perf_counter()
        return ask(*a, **k)

    def t_evaluate(*a, **k):
        out = evaluate(*a, **k)
        acc["pop_steps"].append(es.last_eval_steps)
        return out

    def t_tell(*a, **k):
        out = tell(*a, **k)
        acc["population"].append(time.perf_counter() - cur.pop("t0"))
        return out

    def t_brains(*a, **k):
        t0 = time.perf_counter()
        out = brains(*a, **k)
        acc["brains"].append(time.perf_counter() - t0)
        acc["brain_steps"].append(es.last_eval_steps)
        return out

    def t_read():
        t0 = time.perf_counter()
        out = read()
        acc["read"].append(time.perf_counter() - t0)
        return out
    es.ask, es.evaluate, es.tell, es._brains, es._run_read = t_ask, t_evaluate, t_tell, t_brains, t_read
    return acc


def timed_run(es, env, benv, gens, max_steps):
    es.run(env, benv, 3, max_steps=max_steps, meta_population_size=M)    # warm-up: buffers, ask / tell graph capture
    acc = instrument(es)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    es.run(env, benv, gens, max_steps=max_steps, meta_population_size=M)
    wall = time.perf_counter() - t0
    ms = lambda xs: round(sum(xs) * 1e3 / gens, 2)
    pop, br, rd = ms(acc["population"]), ms(acc["brains"]), ms(acc["read"][:gens])
    gen = round(wall * 1e3 / gens, 2)
    return dict(generations=gens, generation_ms=gen, population_loop_ms=pop, brain_loop_ms=br, novelty_read_ms=rd,
                rest_ms=round(gen - pop - br - rd, 2), final_read_ms=round(acc["read"][-1] * 1e3, 2),
                population_steps=acc["pop_steps"], brain_steps=acc["brain_steps"],
                population_us_per_step=round(sum(acc["population"]) * 1e6 / sum(acc["pop_steps"]), 1),
                brain_us_per_step=round(sum(acc["brains"]) * 1e6 / sum(acc["brain_steps"]), 1))


def act_rows_us(es, discrete, A):
    D0 = es.shapes[0][0]
    sizes = [D0] + [s[1] for s in es.shapes]
    sizes_c = (C.c_int * len(sizes))(*sizes)
    obs = torch.randn(M, D0, device="cuda")
    alive = torch.ones(M, dtype=torch.uint8, device="cuda")
    acts = torch.empty(M, dtype=torch.int64, device="cuda") if discrete else torch.empty(M, A, dtype=torch.float64, device="cuda")
    noise = es.noise_table()
    us = time_events(lambda: L.call("ppx_es_act_rows", es.thetas.data_ptr(), noise.data_ptr(), M, sizes_c, len(sizes) - 1,
                                    obs.data_ptr(), alive.data_ptr(), int(discrete), 5, es._draw.data_ptr(), 0, acts.data_ptr(),
                                    L.stream()), 500)
    byts = M * (8 * es.D + 4 * es.D + 4 * D0 + 8 * A)
    return dict(us=round(us, 2), model_bytes=byts, model_gb_s=round(byts / us * 1e-3, 2))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "es_run_r06.json"))
    ap.add_argument("--gens", type=int, default=10)
    ap.add_argument("--cartpole-budget", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("es_run_prof.py measures on the GPU; no CUDA device found")
    torch.cuda.set_device(0)
    args.out = os.path.abspath(args.out)
    out = dict(gpu_meta(), tool="tools/es_run_prof.py", meta_population=M, arms={})
    os.chdir(tempfile.mkdtemp())                               # run() configures the logger; nothing is written to file
    # C5 on the table env
    np.random.seed(0)
    es = ppx.EvolutionStrategy(obs_dim=8, n_actions=2, hidden_sizes=(64, 64), population_size=P, sigma=0.02,
                               learning_rate=0.01, noise_table_size=1 << 28, noise_seed=1)
    r = timed_run(es, TableEnv(P, "cuda", False), TableEnv(M, "cuda", False, seed=1), args.gens, 1000)
    r["act_rows_per_step"] = act_rows_us(es, False, 2)
    out["arms"]["c5_table"] = dict(workload="P=10000, MLP 8-64-64-2, table env (episodes 250..1000 steps), max_steps 1000", **r)
    # MountainCarContinuous-v0
    np.random.seed(0)
    es = ppx.EvolutionStrategy(env_id="MountainCarContinuous-v0", obs_dim=2, n_actions=1, hidden_sizes=(64, 64),
                               population_size=P, sigma=0.1, learning_rate=0.01, noise_table_size=1 << 26, noise_seed=1)
    env = ppx.ClassicControlVecEnv("MountainCarContinuous-v0", P, seed=0, reward_dtype=torch.float64)
    benv = ppx.ClassicControlVecEnv("MountainCarContinuous-v0", M, seed=1, reward_dtype=torch.float64)
    r = timed_run(es, env, benv, args.gens, 999)
    r["act_rows_per_step"] = act_rows_us(es, False, 1)
    out["arms"]["mountaincar_continuous"] = dict(workload="P=10000, MLP 2-64-64-1, max_steps 999", **r)
    # CartPole-v1 to reward_target 475 (the configuration of tests/test_gpu_es_run.py::test_run_learns_cartpole)
    np.random.seed(0)
    es = ppx.EvolutionStrategy(env_id="CartPole-v1", hidden_sizes=(64, 64), obs_dim=4, n_actions=2, population_size=1024,
                               sigma=0.1, learning_rate=0.05, noise_seed=1, noise_table_size=1 << 22)
    env = ppx.ClassicControlVecEnv("CartPole-v1", 1024, seed=0, reward_dtype=torch.float64)
    benv = ppx.ClassicControlVecEnv("CartPole-v1", M, seed=1, reward_dtype=torch.float64)
    fb = []
    finish = es._finish_generation

    def rec(pending, vals, *a):
        fb.append(float(vals[M]))
        return finish(pending, vals, *a)
    es._finish_generation = rec
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    es.run(env, benv, args.cartpole_budget, max_steps=500, meta_population_size=M, reward_target=475)
    wall = time.perf_counter() - t0
    reached = bool(fb) and fb[-1] > 475
    out["arms"]["cartpole_to_475"] = dict(
        workload="P=1024, MLP 4-64-64-2, sigma 0.1, lr 0.05, numpy seed 0, noise seed 1, env seeds 0 / 1, max_steps 500",
        reached=reached, generations=len(fb), wall_s=round(wall, 2), budget=args.cartpole_budget,
        best_fb=max(fb), best_fb_first_60=max(fb[:60]), fb=[round(x, 1) for x in fb],
        result=(f"f_b {fb[-1]:.0f} > 475 after {len(fb)} generations, {wall:.2f} s" if reached else
                f"not reached within {len(fb)} generations ({wall:.2f} s); best f_b {max(fb):.0f}"))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: v for k, v in out.items() if k != "arms"}))
    for name, a in out["arms"].items():
        print(name, json.dumps({k: v for k, v in a.items() if k not in ("fb", "population_steps", "brain_steps")}))


if __name__ == "__main__":
    main()
