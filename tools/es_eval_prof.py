"""ES episode evaluation at C5's shape on its two paths: EvolutionStrategy.evaluate on an env that lives on the GPU (two
libppx launches per step, no host sync) against the host loop over the same env returning numpy (predict_population on the
f64 observations, a device->host copy of the actions per step, numpy accumulation; Discrete: discrete_action's one
np.random.choice per running member).

C5: P = 10 000 members, MLP 8-64-64-2 (D = 4736), noise table 2^28 f32 (1 GiB: member rows come from HBM, not L2).  The env
is a table lookup (observations / rewards from a 64-step cycle, episode lengths drawn uniformly over 250..1000 steps, a
behavior() of two columns), so what is timed is the evaluation's side of the loop.  Reported:
  * ms per generation (ask -> evaluate -> tell) on the device path, Box and Discrete, and the device evaluate alone;
  * the host loop's ms per step over its first steps (every member running) and that rate times the 1000 steps of the
    generation -- the host arm is too slow to run whole generations (Discrete: 10 000 host draws per step);
  * ppx_es_act per step at 100 / 50 / 10 % of the members running (CUDA events over many launches), against the byte
    model alive x (4 D + 4 D0) + N (A 8 + 1) bytes, next to ppx_es_forward over every member.
The GPU's name and power limit are recorded with the numbers.

    python tools/es_eval_prof.py [--out profiles/es_eval_r03.json]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ppo_exploration_b200 as ppx  # noqa: E402
from ppo_exploration_b200 import _lib as L  # noqa: E402

P, D0, HID, A_BOX, A_DISC, CYCLE, MAX_STEPS = 10_000, 8, (64, 64), 2, 2, 64, 1000


class TableEnv:
    """Observations / rewards from [CYCLE, N, ...] tables (torch CUDA or numpy), done at step len[i] (and every 250 steps
    after it, as an auto-resetting env would report), behavior() = the first two observation columns in f64."""

    def __init__(self, n, device, discrete, seed=0):
        rs = np.random.RandomState(seed)
        tabs = dict(obs=rs.randn(CYCLE, n, D0).astype(np.float32), rew=rs.randn(CYCLE, n).astype(np.float32),
                    len=rs.randint(250, MAX_STEPS + 1, n).astype(np.int64))
        self.host = device is None
        self.tabs = tabs if self.host else {k: torch.as_tensor(v).to(device) for k, v in tabs.items()}
        self.num_envs = n
        self.observation_space = ppx.Box((D0,))
        self.action_space = ppx.Discrete(A_DISC) if discrete else ppx.Box((A_BOX,))

    def reset(self):
        self.t = 0
        return self.tabs["obs"][0]

    def step(self, actions):
        self.t += 1
        k = self.t % CYCLE
        self.o = self.tabs["obs"][k]
        done = (self.t >= self.tabs["len"]) & ((self.t - self.tabs["len"]) % 250 == 0)
        return self.o, self.tabs["rew"][k], done, []

    def behavior(self):
        b = self.o[:, :2]
        return b.astype(np.float64) if self.host else b.double()


def gpu_meta():
    meta = {"gpu": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                              "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        meta.update(gpu_smi=out[0].strip(), power_limit_w=float(out[1]), sm_max_mhz=float(out[2]))
    except Exception as e:                                      # the numbers stay usable; say what is missing
        meta["power_limit_w"] = f"unavailable ({e})"
    return meta


def make_es(discrete, dev):
    np.random.seed(0)
    return ppx.EvolutionStrategy(obs_dim=D0, n_actions=A_DISC if discrete else A_BOX, hidden_sizes=HID, population_size=P,
                                 sigma=0.02, learning_rate=0.01, device=dev, noise_table_size=1 << 28, noise_seed=1)


def host_steps(es, env, pop, discrete, steps):
    """The host loop over `steps` steps (every member runs: episodes last >= 250 steps); returns ms per step."""
    np.random.seed(1)
    obs = env.reset()
    fit = np.zeros(P)
    alive = np.ones(P, bool)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        out = es.predict_population(pop, torch.as_tensor(obs).to(es.theta.device).double(), discrete=discrete)
        if discrete:
            a = np.zeros(P, np.int64)
            a[alive] = ppx.EvolutionStrategy.discrete_action(out[torch.as_tensor(alive).to(out.device)])
        else:
            a = np.where(alive[:, None], out.cpu().numpy(), 0.0)
        obs, rew, done, _ = env.step(a)
        env.behavior()
        fit[alive] += rew[alive].astype(np.float64)
        alive &= ~done
    return (time.perf_counter() - t0) * 1e3 / steps


def time_act(es, pop, obs, alive, discrete, reps):
    sizes = [D0, *HID, A_DISC if discrete else A_BOX]
    sizes_c = (C.c_int * len(sizes))(*sizes)
    acts = torch.empty(P, dtype=torch.int64, device=obs.device) if discrete else \
        torch.empty(P, A_BOX, dtype=torch.float64, device=obs.device)
    noise = es.noise_table()

    def launch():
        L.call("ppx_es_act", es.theta.data_ptr(), noise.data_ptr(), pop.data_ptr(), float(es.SIGMA), P, sizes_c, len(sizes) - 1,
               obs.data_ptr(), alive.data_ptr(), int(discrete), 3, es._draw.data_ptr(), 0, 0, None, acts.data_ptr(), L.stream())
    return time_events(launch, reps)


def time_events(fn, reps):
    for _ in range(10):
        fn()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = []
    for _ in range(5):
        s.record()
        for _ in range(reps):
            fn()
        e.record()
        e.synchronize()
        out.append(s.elapsed_time(e) * 1e3 / reps)
    return statistics.median(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "es_eval_r03.json"))
    ap.add_argument("--gens", type=int, default=3)
    ap.add_argument("--host-steps", type=int, default=30)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("es_eval_prof.py measures on the GPU; no CUDA device found")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    out = dict(gpu_meta(), tool="tools/es_eval_prof.py", workload=(
        f"C5 shape: P={P}, MLP {D0}-{HID[0]}-{HID[1]}-A (D=4736 for A=2), noise table 2^28 f32, sigma 0.02; table env, episode "
        f"lengths uniform over 250..{MAX_STEPS} steps, behavior() of 2 columns, max_steps {MAX_STEPS}"), arms={})
    for discrete in (False, True):
        name = "discrete" if discrete else "box"
        es = make_es(discrete, dev)
        env = TableEnv(P, dev, discrete)
        gen_ms, eval_ms, steps = [], [], []
        for g in range(args.gens + 2):                       # two warm-up generations: buffers, ask / tell graph capture
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fit, lens, bc = es.run_generation(env, max_steps=MAX_STEPS)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            es.evaluate(env, max_steps=MAX_STEPS)            # the evaluation alone, same population
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            if g >= 2:
                gen_ms.append((t1 - t0) * 1e3)
                eval_ms.append((t2 - t1) * 1e3)
                steps.append(es.last_eval_steps)
        lens = lens.cpu().numpy()
        n0 = L.launch_count()
        es.evaluate(env, max_steps=MAX_STEPS)
        launches = (L.launch_count() - n0) / es.last_eval_steps
        pop = es._ask_off
        host_env = TableEnv(P, None, discrete)
        host_ms = [host_steps(es, host_env, pop, discrete, args.host_steps) for _ in range(2)]
        hstep = statistics.median(host_ms)
        dgen = statistics.median(gen_ms)
        out["arms"][name] = dict(
            device_generation_ms_median=round(dgen, 2), device_generation_ms=[round(x, 2) for x in gen_ms],
            device_evaluate_ms_median=round(statistics.median(eval_ms), 2), steps_issued=steps,
            longest_episode=int(lens.max()), mean_episode=float(lens.mean()), libppx_launches_per_step=launches,
            device_us_per_step=round(statistics.median(eval_ms) * 1e3 / statistics.median(steps), 1),
            host_ms_per_step_all_running=round(hstep, 3), host_ms_per_step=[round(x, 3) for x in host_ms],
            host_steps_timed=args.host_steps,
            host_generation_ms_projected=round(hstep * int(lens.max()), 1),
            speedup_vs_projected_host=round(hstep * int(lens.max()) / dgen, 1))
        # ppx_es_act per step at 100 / 50 / 10 % running, byte model, and ppx_es_forward over every member
        obs = torch.as_tensor(np.random.RandomState(2).randn(P, D0).astype(np.float32)).to(dev)
        A = A_DISC if discrete else A_BOX
        D = es.D
        act = {}
        for frac in (1.0, 0.5, 0.1):
            alive = torch.as_tensor(np.random.RandomState(3).rand(P) < frac).to(dev).to(torch.uint8)
            n_alive = int(alive.sum())
            us = time_act(es, pop, obs, alive, discrete, 200)
            byts = n_alive * (4 * D + 4 * D0) + P * (8 * A + 1)
            act[f"{int(frac * 100)}%"] = dict(running=n_alive, us=round(us, 2), model_bytes=byts, model_gb_s=round(byts / us * 1e-3, 1))
        obs64 = obs.double()
        fwd_out = torch.empty(P, A, dtype=torch.float64, device=dev)
        sizes = [D0, *HID, A]
        sizes_c = (C.c_int * len(sizes))(*sizes)
        noise = es.noise_table()
        fwd_us = time_events(lambda: L.call("ppx_es_forward", es.theta.data_ptr(), noise.data_ptr(), pop.data_ptr(), float(es.SIGMA), P,
                                            sizes_c, len(sizes) - 1, obs64.data_ptr(), int(not discrete), fwd_out.data_ptr(),
                                            L.stream()), 200)
        out["arms"][name]["es_act_per_step"] = act
        out["arms"][name]["es_forward_all_members_us"] = round(fwd_us, 2)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: v for k, v in out.items() if k != "arms"}))
    for name, a in out["arms"].items():
        print(name, json.dumps(a))


if __name__ == "__main__":
    main()
