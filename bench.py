"""Benchmark of the learner hot path on B200 (contract: see the task statement / DESIGN.md §6).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config C1|C2|C3|C4]     ppx arm (this repo's CUDA path)
  python bench.py --impl reference ...                                           CPU arm: the reference itself
  python bench.py ... --dump-outputs DIR          also write what the last timed step computed to DIR/<name>.npy

Workloads = BASELINE.json `configs` (SURVEY §8d pins their sizes); the headline line is C2, the configuration the
metric is quoted on.  A default run also measures C1 / C3 / C4 (sub-records under `configs`, N = 1 only) and one
ES-NSRA step at C5 (`es`).

  C1  PPO, CartPole-shaped: 8 envs x 128 steps, obs 4, Discrete(2), reference defaults (h 128, B 128, 10 epochs)
  C2  PPO + SimHash, Swimmer-shaped: 2048 envs x 256 steps per GPU, obs 8, Box(2), k = 64, `swimmer_ppo` hparams
      (hyperparameters.py:7-8), 4 minibatches per epoch x 10 epochs
  C3  PPO_RND, Atari-shaped flat frames: 128 envs x 128 steps, obs 28224, dual-head GAE (gamma .999 / .99), h 128
  C4  PPO_ICM, Atari-shaped features: 32 envs x 128 steps per GPU (256 over 8), obs 3136, h = f = 512, Discrete(18)

One "step" = one learner pass over a rollout: bonus over all T*N transitions -> GAE -> train() (all epochs x
minibatches: shuffle-gather, MLP forward, fused loss fwd+bwd, MLP backward, clip+Adam).  value = transitions
(T*N per GPU x N GPUs) per second, rollout resident in HBM; e2e = the same with the rollout copied from pinned host
memory every step and the loss log read back.

CPU arm: the UNMODIFIED reference (vendored into oracle/_ref by __graft_entry__.build(), kind "reference"; the
oracle port only if that copy is absent) on the host's cores, on a bounded sample scaled linearly (stated in `sample`).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "transitions/s through GAE+bonus+PPO update"
SWIMMER_PPO = dict(lr=3e-4, gamma=0.999, gae_lam=0.95, vf_coef=1, max_grad_norm=5, n_epochs=10, clip_range=0.2, ent_coef=0.0)
REF_DEFAULTS = dict(lr=3e-4, gamma=0.99, gae_lam=0.95, vf_coef=1, max_grad_norm=0.2, n_epochs=10, clip_range=0.2, ent_coef=0.01)
CONFIGS = {
    "C1": dict(alg="ppo", T=128, N=8, D=4, space=("Discrete", 2), hidden=128, batch=128, hp=REF_DEFAULTS, sim_hash=False,
               obs="normal", ref_sample=dict(N=8, n_epochs=10),
               workload="C1: PPO, obs 4, Discrete(2), 8 envs x 128 steps, reference defaults (h 128, B 128, 10 epochs)"),
    "C2": dict(alg="ppo", T=256, N=2048, D=8, space=("Box", 2), hidden=64, batch=131072, hp=SWIMMER_PPO, sim_hash=True,
               hash_bits=64, obs="normal", ref_sample=dict(N=2048, n_epochs=2, hash_envs=512, hash_steps=64),
               workload="C2: PPO+SimHash, obs 8, Box(2), k=64, 2048 envs x 256 steps per GPU, swimmer_ppo hparams, "
                        "4 minibatches/epoch x 10 epochs"),
    "C3": dict(alg="rnd", T=128, N=128, D=28224, space=("Discrete", 18), hidden=128, int_hidden=128, batch=4096,
               hp=dict(lr=3e-4, gamma=0.999, int_gamma=0.99, gae_lam=0.95, n_epochs=4, clip_range=0.2, ent_coef=0.01, vf_coef=0.5,
                       int_vf_coef=0.5, max_grad_norm=0.2),
               sim_hash=False, obs="frames", ref_sample=dict(N=64, n_epochs=1, bonus_steps=8),
               workload="C3: PPO_RND, flat 84x84x4 frames (obs 28224), Discrete(18), 128 envs x 128 steps, dual-head GAE "
                        "(gamma .999 / .99), h 128, 4 epochs x 4 minibatches of 4096"),
    "C4": dict(alg="icm", T=128, N=32, D=3136, space=("Discrete", 18), hidden=128, int_hidden=512, batch=1024,
               hp=dict(lr=3e-4, int_lr=3e-4, gae_lam=0.95, n_epochs=4, clip_range=0.2, ent_coef=0.01, vf_coef=0.5, max_grad_norm=0.2),
               sim_hash=False, obs="frames", ref_sample=dict(N=16, n_epochs=1, bonus_steps=16),
               workload="C4: PPO_ICM, obs 3136 (7x7x64 features), Discrete(18), 32 envs x 128 steps per GPU (256 over 8), "
                        "h = f = 512, 4 epochs x 4 minibatches of 1024"),
}
# DRAM bytes per launch of the fused MLP kernels at the C2 minibatch, from the committed ncu captures
NCU_TRAFFIC = {"ppx_mlp3_bwd": 144.0e6, "ppx_mlp3_fwd": 81.9e6, "ppx_mlp3_tc_bwd": 145.1e6, "ppx_mlp3_tc_fwd": 82.0e6}
NCU_TRAFFIC_SRC = ("ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch (profiles/ncu_top5_r02.md: the kernel inside a pass; "
                   "SIMT pair: profiles/ncu_mlp3_r01b.md)")


def action_dims(cfg):
    kind, n = cfg["space"]
    return (1, n) if kind == "Discrete" else (n, n)            # (stored action width, actor outputs)


def synth_rollout(cfg, seed, n_envs=None):
    """Seeded synthetic rollout in the reference's [T,N,...] layout (SURVEY §8d)."""
    T, N, D = cfg["T"], n_envs or cfg["N"], cfg["D"]
    kind, n = cfg["space"]
    A = action_dims(cfg)[0]
    rs = np.random.RandomState(seed)
    if cfg["obs"] == "frames":                                   # uniform{0..255}/255, like stacked frames
        obs = rs.randint(0, 256, size=(T, N, D), dtype=np.uint8).astype(np.float32) / np.float32(255.0)
        final_obs = rs.randint(0, 256, size=(N, D), dtype=np.uint8).astype(np.float32) / np.float32(255.0)
    else:
        obs = rs.randn(T, N, D).astype(np.float32)
        final_obs = rs.randn(N, D).astype(np.float32)
    out = dict(observations=obs,
               actions=(rs.randn(T, N, A) if kind == "Box" else rs.randint(0, n, size=(T, N, 1)).astype(np.float64)),
               rewards=rs.randn(T, N).astype(np.float32), values=rs.randn(T, N).astype(np.float32),
               masks=(rs.rand(T, N) < 0.02).astype(np.uint8),
               action_log_probs=((-1.4 if kind == "Box" else -np.log(n)) + 0.3 * rs.randn(T, N, A)).astype(np.float32),
               last_value=rs.randn(N).astype(np.float32), final_obs=final_obs)
    if cfg["alg"] == "rnd":
        out["int_values"] = rs.randn(T, N).astype(np.float32)
        out["last_int_value"] = rs.randn(N).astype(np.float32)
    return out


ROLLOUT_FIELDS = ("observations", "actions", "rewards", "values", "masks", "action_log_probs", "int_values")
# --dump-outputs: at most 4 MB per array and at most 9 arrays (PPO_RND) -> well under 64 MB per dump
DUMP_MAX_BYTES = 4 << 20
DUMP_TOTAL_BYTES = 64 << 20


def dump_array(x):
    """Tensor / ndarray -> host ndarray, f64 kept, everything else as f32.  An array over DUMP_MAX_BYTES is reduced to a
    fixed sample of its flattened elements (sorted indices from a private seeded stream): the same elements in every run
    of the same configuration, and the global numpy stream the learner's shuffles draw from is not touched."""
    import torch
    t = torch.as_tensor(x).detach()
    dt = np.float64 if t.dtype == torch.float64 else np.float32
    cap = DUMP_MAX_BYTES // np.dtype(dt).itemsize
    if t.numel() > cap:
        idx = np.sort(np.random.RandomState(0).choice(t.numel(), cap, replace=False))
        t = t.reshape(-1)[torch.as_tensor(idx, device=t.device)]
    return t.cpu().numpy().astype(dt)


def write_outputs(out_dir, arrays):
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_TOTAL_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------
# CPU arm
# ---------------------------------------------------------------------------------------------
def host_threads():
    import torch
    return dict(cpu_count=os.cpu_count(), affinity=len(os.sched_getaffinity(0)), torch_threads=torch.get_num_threads())


def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm must use the same cores at every N."""
    import torch
    n = len(os.sched_getaffinity(0))
    torch.set_num_threads(n)
    return n


def cpu_pass_reference(name, seed=0, shrink=1):
    """One learner pass of the UNMODIFIED reference (oracle/_ref) on a bounded sample, scaled linearly to the full
    pass.  Returns (transitions_per_s, detail)."""
    import torch
    from oracle import ref_runtime as RT
    cfg = CONFIGS[name]
    algorithms = RT.install()
    RT.silence_logger()
    T, D, B = cfg["T"], cfg["D"], cfg["batch"]
    kind, n = cfg["space"]
    smp = dict(cfg["ref_sample"])
    Ns = max(1, smp["N"] // shrink)
    n_ep = smp["n_epochs"]
    space = RT.Box((n,)) if kind == "Box" else RT.Discrete(n)
    RT.set_env_factory(lambda: RT.FakeVecEnv(Ns, D, space, seed=seed))
    np.random.seed(seed); torch.manual_seed(seed)
    hp = dict(cfg["hp"], n_epochs=n_ep)
    kw = dict(env_id="synthetic", nstep=T, batch_size=min(B, T * Ns), hidden_size=cfg["hidden"], **hp)
    if cfg["alg"] == "ppo":
        m = algorithms.PPO(sim_hash=cfg["sim_hash"], **kw)
    elif cfg["alg"] == "rnd":
        m = algorithms.PPO_RND(int_hidden_size=cfg["int_hidden"], rnd_start=0, **kw)
    else:
        m = algorithms.PPO_ICM(int_hidden_size=cfg["int_hidden"], **kw)
    ro = m.rollout
    host = synth_rollout(cfg, seed, n_envs=Ns)
    ro.reset()
    for k in ROLLOUT_FIELDS:
        if k in host:
            getattr(ro, k)[...] = host[k].reshape(getattr(ro, k).shape)
    ro.pos, ro.full = T, True
    split, scale_note = {}, []
    # ---- bonus over the rollout (scaled from a sample of env steps)
    t_bonus = 0.0
    if cfg["sim_hash"]:                                          # buffer.py:188-200: a python loop over every observation
        ro.A = np.random.randn(cfg["hash_bits"], D)               # k is hard-wired to 16 upstream (buffer.py:137); A is a plain attribute
        he, hs = max(1, smp["hash_envs"] // shrink), smp["hash_steps"]
        t0 = time.perf_counter()
        for t in range(hs):
            ro.sim_hash(host["observations"][t, :he], ro.rewards[t, :he])
        t_bonus = (time.perf_counter() - t0) * (T * cfg["N"]) / (hs * he)
        scale_note.append(f"sim_hash on {he} envs x {hs} steps")
    elif cfg["alg"] == "rnd":                                     # algorithms.py:394-398 per env step
        bs = smp["bonus_steps"]
        nxt = np.concatenate([host["observations"][1:], host["final_obs"][None]], 0)
        t0 = time.perf_counter()
        for t in range(bs):
            nobs = m.normalize_obs(nxt[t])
            ri = m.rnd.int_reward(nobs).detach().numpy()
            m.int_rew_rms.update(ri)
            ri /= (np.sqrt(m.int_rew_rms.var) + 1e-08)
            ro.int_rewards[t] = ri
        t_bonus = (time.perf_counter() - t0) * (T * cfg["N"]) / (bs * Ns)
        scale_note.append(f"RND bonus on {Ns} envs x {bs} steps")
    elif cfg["alg"] == "icm":                                     # algorithms.py:629-630 per env step
        bs = smp["bonus_steps"]
        nxt = np.concatenate([host["observations"][1:], host["final_obs"][None]], 0)
        t0 = time.perf_counter()
        for t in range(bs):
            act = torch.tensor(host["actions"][t])                    # Discrete: ids [N] (policy.act's sample shape); Box: [N,A]
            ri = m.intrinsic_module.int_reward(torch.Tensor(host["observations"][t]), torch.Tensor(nxt[t]),
                                               act.squeeze(-1) if kind == "Discrete" else act)
            ro.rewards[t] = (1 - m.int_rew_integration) * ro.rewards[t] + m.int_rew_integration * ri.detach().numpy()
        t_bonus = (time.perf_counter() - t0) * (T * cfg["N"]) / (bs * Ns)
        scale_note.append(f"ICM bonus on {Ns} envs x {bs} steps")
    split["bonus_s"] = t_bonus
    # ---- GAE
    lv = torch.tensor(host["last_value"])
    dones = host["masks"][-1].astype(bool)
    t0 = time.perf_counter()
    if cfg["alg"] == "rnd":
        ro.compute_returns_and_advantages(lv, torch.tensor(host["last_int_value"]), dones)
    else:
        ro.compute_returns_and_advantages(lv, dones)
    split["gae_s"] = (time.perf_counter() - t0) * cfg["N"] / Ns
    # ---- train(): n_ep epochs over Ns envs, scaled to the configured epochs over N envs (same minibatch size)
    steps_done = n_ep * -(-T * Ns // kw["batch_size"])
    steps_full = cfg["hp"]["n_epochs"] * -(-T * cfg["N"] // B)
    t0 = time.perf_counter()
    m.train()
    split["train_s"] = (time.perf_counter() - t0) * steps_full / steps_done
    scale_note.append(f"GAE on {Ns} of {cfg['N']} envs" if Ns != cfg["N"] else "GAE full size")
    scale_note.append(f"{steps_done} of {steps_full} optimiser steps at B={kw['batch_size']}")
    total = sum(split.values())
    return (T * cfg["N"]) / total, dict(split_s_per_pass=split, kind="reference",
                                        sample="; ".join(scale_note) + "; each scaled linearly to one pass")


def cpu_pass_port(name, seed=0, shrink=1):
    """Fallback when oracle/_ref is absent: the oracle port (numpy SimHash loop, numpy GAE, torch-CPU train); PPO only."""
    import torch
    from oracle import rollout as OR
    from oracle import learner as OL
    cfg = CONFIGS[name]
    if cfg["alg"] != "ppo" or cfg["space"][0] != "Box":
        return None, dict(kind="port", sample="not available for this config without oracle/_ref")
    T, N, D, B = cfg["T"], cfg["N"], cfg["D"], cfg["batch"]
    A = cfg["space"][1]
    np.random.seed(seed); torch.manual_seed(seed)
    ro = synth_rollout(cfg, seed)
    smp = cfg["ref_sample"]
    split = {}
    if cfg["sim_hash"]:
        A_mat = np.random.randn(cfg["hash_bits"], D)
        tab = OR.CountTable(0.1)
        he, hs = max(1, smp["hash_envs"] // shrink), smp["hash_steps"]
        t0 = time.perf_counter()
        for t in range(hs):
            tab.update(A_mat, ro["observations"][t, :he], ro["rewards"][t, :he])
        split["bonus_s"] = (time.perf_counter() - t0) * (T * N) / (hs * he)
    t0 = time.perf_counter()
    adv, ret = OR.gae(ro["rewards"], ro["values"], ro["masks"].astype(np.int64), ro["last_value"], ro["masks"][-1],
                      cfg["hp"]["gamma"], cfg["hp"]["gae_lam"])
    split["gae_s"] = time.perf_counter() - t0
    p = OL.make_policy_params(D, A, cfg["hidden"])
    opt = torch.optim.Adam(OL._policy_param_list(p), lr=cfg["hp"]["lr"])
    buf = dict(ro, advantages=adv, returns=ret)
    steps_full = cfg["hp"]["n_epochs"] * -(-T * N // B)
    k = min(8, steps_full)
    t0 = time.perf_counter()
    OL.ppo_train(p, opt, buf, dict(cfg["hp"], batch_size=B), discrete=False, max_steps=k)
    split["train_s"] = (time.perf_counter() - t0) * steps_full / k
    return (T * N) / sum(split.values()), dict(split_s_per_pass=split, kind="port",
                                               sample=f"oracle port; {k} of {steps_full} optimiser steps; scaled linearly")


def cpu_pass(name, seed=0, shrink=1):
    import warnings
    from oracle import ref_runtime as RT
    with warnings.catch_warnings():
        # the reference's own numpy reductions overflow f32 on the synthetic C3-scale returns (RuntimeWarning from inside
        # its code); irrelevant to what is timed
        warnings.simplefilter("ignore", RuntimeWarning)
        if RT.available():
            return cpu_pass_reference(name, seed, shrink)
        return cpu_pass_port(name, seed, shrink)


def cpu_es_step(P_sample=1000, P=10000):
    """ES-NSRA step of the reference (evolution_strategies.py:137-145, 172-182, 217-239, 264-281) on P_sample members,
    scaled to P."""
    from oracle import ref_runtime as RT
    if not RT.available():
        return None
    RT.install()
    import evolution_strategies as refes

    class E:
        pass
    es = E.__new__(E)
    ES = refes.EvolutionStrategy
    np.random.seed(0)
    es.weights = [np.random.randn(*s) for s in [(8, 64), (64, 64), (64, 2)]]
    es.POPULATION_SIZE, es.SIGMA, es.learning_rate, es.decay, es.novelty_param, es.K = P_sample, 0.1, 0.01, 0.9995, 0.5, 10
    archive = [np.random.randn(1, 2) for _ in range(10000)]
    t0 = time.perf_counter()
    pop = ES._get_population(es)
    for member in pop:
        ES._get_weights_try(es, es.weights, member)
    nov = ES.get_kNN(es, archive, np.random.randn(1, 2), es.K)
    ES._update_weights(es, np.random.randn(P_sample), pop, nov)
    dt = time.perf_counter() - t0
    return dict(value=P_sample / dt, unit="perturbations/s", kind="reference",
                sample=f"{P_sample} of {P} members (population draw + perturb + kNN over 10000 + update), scaled linearly",
                cores=host_threads()["torch_threads"])


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = use_all_host_threads()
    cfg = CONFIGS[args.config]
    shrink = 4 if args.config == "C2" else 1                     # K steps + warm-up must end within minutes
    cpu_pass(args.config, seed=99, shrink=8)                     # always one untimed pass: torch's CPU thread pool / MKL start-up
    vals, det = [], None
    t_all = time.perf_counter()
    for s in range(args.steps):
        v, det = cpu_pass(args.config, seed=s, shrink=shrink)
        vals.append(v)
    wall = time.perf_counter() - t_all
    v = float(np.mean(vals))
    th = host_threads()
    trans = cfg["T"] * cfg["N"]
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "transitions/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * trans / v, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": cfg["workload"], "name": args.config},
            "cpu_baseline": {"value": v, "unit": "transitions/s", "cores": cores, "kind": det["kind"], "sample": det["sample"],
                             "host": th, "measured_wall_s": wall, "split_s_per_pass": det.get("split_s_per_pass")},
            "e2e": {"value": v, "unit": "transitions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------
# ppx arm
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc, self.index = None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out = self.proc.communicate(timeout=5)[0]
        except Exception:
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in out.strip().splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, val in zip(names, f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


class OpTimer:
    """CUDA-event brackets around selected C-ABI calls on the launching stream (roofline measurement)."""
    # name -> indices of (M, K, N, batch) among the call's arguments (None = 1)
    SHAPE_ARGS = {"ppx_linear_fwd": (4, 5, 6, 10), "ppx_linear_bwd_data": (3, 4, 5, 11), "ppx_linear_bwd_weight": (4, 5, 6, 10),
                  "ppx_mlp3_fwd": (2, 3, 4, 5), "ppx_mlp3_bwd": (2, 3, 4, 5), "ppx_mlp3_tc_fwd": (2, 3, 4, 5),
                  "ppx_mlp3_tc_bwd": (2, 3, 4, 5), "ppx_tc_linear": (5, 6, 7, None), "ppx_tc_linear_ws": (5, 6, 7, None), "ppx_tc_wgrad": (4, 5, 6, None)}

    def __init__(self, L, torch):
        self.L, self.torch, self.rec, self.orig = L, torch, [], L.call
        self.last_bwd = self.last_fwd = None

    def __enter__(self):
        def timed(name, *args):
            if name in self.SHAPE_ARGS:
                s, e = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
                s.record()
                rc = self.orig(name, *args)
                e.record()
                if name == "ppx_mlp3_tc_bwd":
                    self.last_bwd = args                        # (pointers into persistent scratch: valid after the pass)
                if name == "ppx_mlp3_tc_fwd":
                    self.last_fwd = args
                self.rec.append((name, tuple(1 if i is None else args[i] for i in self.SHAPE_ARGS[name]), s, e))
                return rc
            return self.orig(name, *args)
        self.L.call = timed
        for mod in self._mods():
            mod.L.call = timed
        return self

    def _mods(self):
        import ppo_exploration_b200 as ppx
        return [ppx.models, ppx.algorithms, ppx.buffer, ppx.util]

    def __exit__(self, *a):
        self.L.call = self.orig

    def bwd_kernel_ms(self, reps=24):
        """Device time of the backward KERNEL alone and of the reduce kernel behind it: the last forward + backward calls
        of the pass are re-issued `reps` times back to back (optimiser tail off; activations and gradients are simply
        rewritten with the same values) so the GPU never waits for the host and the backward finds the caches as it does
        in a pass (the forward has just written the activations it reads); the library records an event between the two
        kernels of every backward call (ppx_mlp3_tc_bwd_probe)."""
        if self.last_bwd is None:
            return None, None
        torch, args = self.torch, list(self.last_bwd)
        args[23], args[24] = None, None                         # step_dev, adam: leave the optimiser state alone
        ev = []
        for i in range(reps + 4):
            a, b, c = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            if self.last_fwd is not None:
                self.orig("ppx_mlp3_tc_fwd", *self.last_fwd)
            a.record()
            b.record()                                          # creates the CUDA event; re-recorded by the library
            self.orig("ppx_mlp3_tc_bwd_probe", b.cuda_event)
            self.orig("ppx_mlp3_tc_bwd", *args)
            c.record()
            ev.append((a, b, c))
        torch.cuda.synchronize()
        ev = ev[4:]
        return (sum(a.elapsed_time(b) for a, b, _ in ev) / len(ev), sum(b.elapsed_time(c) for _, b, c in ev) / len(ev))

    def summary(self):
        self.torch.cuda.synchronize()
        agg = {}
        for name, shape, s, e in self.rec:
            a = agg.setdefault((name, shape), [0.0, 0])
            a[0] += s.elapsed_time(e); a[1] += 1
        return agg


def roofline_of(agg, cfg, peaks):
    """Roofline record of the op that took the most device time in one pass."""
    A_out = action_dims(cfg)[1]
    tf_peak = peaks.get("bf16_tflops_sustained", 1400.0)
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    (op, (M_, K_, N_, b_)), (tot_ms, cnt) = max(agg.items(), key=lambda kv: kv[1][0])
    ms_launch = tot_ms / cnt
    so = A_out + b_ - 1                                           # head outputs over the G nets (actor + G-1 value heads)
    if op in ("ppx_mlp3_fwd", "ppx_mlp3_tc_fwd"):                 # shape = (M, D, H, G)
        flops = 2.0 * M_ * (b_ * (K_ * N_ + N_ * N_) + N_ * so)
    elif op in ("ppx_mlp3_bwd", "ppx_mlp3_tc_bwd"):               # dgrad (layers 3,2) + wgrad (layers 3,2,1)
        flops = 2.0 * M_ * (b_ * (K_ * N_ + 2 * N_ * N_) + 2 * N_ * so)
    else:
        flops = 2.0 * M_ * K_ * N_ * b_
    achieved = flops / (ms_launch / 1e3) / 1e12
    ops = sorted(((f"{k[0]}{list(k[1])}", round(v[0], 3), v[1]) for k, v in agg.items()), key=lambda x: -x[1])[:8]
    common = {"ms_per_launch": ms_launch, "launches_per_step": cnt, "top_ops_ms_per_step": ops,
              "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"}
    if op.startswith("ppx_mlp3_tc"):
        # fused policy-MLP kernel, GEMMs on tcgen05: what bounds it is the HBM stream of the saved activations plus the
        # elementwise work -> HBM roofline with the algorithmic bytes 4 M (D + 2 G H + sum o); tensor figures beside it
        mlp_bytes = 4.0 * M_ * (K_ + 2 * b_ * N_ + so)
        gbs = mlp_bytes / (ms_launch / 1e3) / 1e9
        return dict(common, bound="hbm", kernel=f"{op} M={M_} D={K_} H={N_} G={b_}", achieved=gbs, peak=hbm_peak, unit="GB/s",
                    frac=gbs / hbm_peak, traffic=NCU_TRAFFIC.get(op) if M_ == 131072 else None,
                    traffic_source=NCU_TRAFFIC_SRC if (op in NCU_TRAFFIC and M_ == 131072) else None,
                    alg_bytes_per_launch=mlp_bytes, fp32_equiv_tflops=achieved, tf32_mma_tflops=3.0 * achieved,
                    tf32_frac_of_bf16_peak=3.0 * achieved / tf_peak,
                    note="fused policy-MLP kernel with its 64x64 GEMMs on tcgen05 (3xTF32, fp32-equivalent); algorithmic bytes = "
                         "4 M (D + 2 G H + sum o); tf32_mma_tflops counts the three tensor passes")
    if op in ("ppx_tc_linear", "ppx_tc_linear_ws", "ppx_tc_wgrad"):
        return dict(common, bound="tensor", kernel=f"{op} M={M_} K={K_} N={N_}", achieved=achieved, peak=tf_peak, unit="TFLOP/s",
                    frac=achieved / tf_peak, traffic=None, tf32_mma_tflops=3.0 * achieved, tf32_frac_of_bf16_peak=3.0 * achieved / tf_peak,
                    note="wide dense layer on tcgen05 (3xTF32: fp32-equivalent result from three tf32 passes); achieved = "
                         "algorithmic 2 M K N flops / time, against the measured bf16 peak; tf32_mma_tflops = the executed passes")
    return dict(common, bound="tensor", kernel=f"{op} M={M_} K/D={K_} N/H={N_} batch/G={b_}", achieved=achieved, peak=tf_peak,
                unit="TFLOP/s", frac=achieved / tf_peak, traffic=NCU_TRAFFIC.get(op) if M_ == 131072 else None,
                fp32_frac=achieved / 74.4,
                note="exact-fp32 SIMT kernel (FFMA-bound; 1e-5 parity path), fraction quoted against the bf16 tensor peak; "
                     "fp32_frac = achieved / 74.4 TFLOP/s (148 SMs x 128 FMA/clk x 1.965 GHz)")


def es_step_bench(torch, ppx, dev, world, rank, steps=20, warmup=5):
    """ES-NSRA step at C5 (P=10 000 members, MLP 8-64-64-2 -> D=4736, noise table 2^28 f32, K=10, archive 10 000):
    sample offsets -> theta + sigma*eps for this rank's P/W members -> fitness exchange -> novelty k-NN -> update.
    Strong scaling (the population is fixed).  Returns perturbations/s and ms/step."""
    import torch.distributed as dist
    P, M = 10000 - 10000 % world, 10000
    np.random.seed(0)
    es = ppx.EvolutionStrategy(obs_dim=8, n_actions=2, hidden_sizes=(64, 64), population_size=P, sigma=0.1,
                               learning_rate=0.01, decay=0.9995, novelty_param=0.5, device=dev,
                               noise_table_size=1 << 28, noise_seed=0)
    es.noise_table()
    g = torch.Generator(device=dev).manual_seed(1)
    archive = torch.randn(M, 2, dtype=torch.float64, device=dev, generator=g)
    queries = torch.randn(2, 2, dtype=torch.float64, device=dev, generator=g)
    fit_local = torch.randn(P // world, dtype=torch.float64, device=dev, generator=g)
    def step():
        pop, w, nov = es.ask(archive, queries)                  # population drawn on the device, [P/W, D] f32 for the evaluators, k-NN novelty
        es.tell(fit_local)                                      # fitness exchange, (sharded) update
        return w
    for _ in range(warmup):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item()) / steps
    hbm = 6553.0
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        hbm = json.load(open(pk)).get("hbm_gbs", hbm)
    gbs = 56832.0 * (P / world) / (ms / 1e3) / 1e9
    return {"metric": "ES perturbations/s", "value": P / (ms / 1e3), "unit": "perturbations/s", "ms_per_step": ms,
            "scaling": "strong", "hbm_frac_per_gpu": gbs / hbm,
            "config": {"workload": "C5: ES-NSRA, P=%d, MLP 8-64-64-2 (D=4736), noise table 2^28 f32, "
                                   "K=10, archive 10000, z-score shaping" % P,
                       "alg_bytes_per_perturbation": 56832, "update": getattr(es, "update_mode", "replicated")}}


class PpxPass:
    """One config on this rank's GPU: learner, pinned synthetic rollout, the resident and end-to-end step functions."""

    def __init__(self, name, torch, ppx, dev, rank, world):
        from ppo_exploration_b200 import _lib as L
        self.name, self.cfg, self.torch, self.ppx, self.dev, self.rank, self.world, self.L = name, CONFIGS[name], torch, ppx, dev, rank, world, L
        cfg = self.cfg
        T, N, D = cfg["T"], cfg["N"], cfg["D"]
        kind, n = cfg["space"]
        space = ppx.Box((n,)) if kind == "Box" else ppx.Discrete(n)
        np.random.seed(0); torch.manual_seed(0)                 # one shuffle stream ("global": identical on every rank), replicated weights
        env = ppx.SyntheticVecEnv(N, D, space, seed=rank)
        kw = dict(env=env, nstep=T, batch_size=cfg["batch"], hidden_size=cfg["hidden"], device=dev, **cfg["hp"])
        if cfg["alg"] == "ppo":
            m = ppx.PPO(sim_hash=cfg["sim_hash"], hash_bits=cfg.get("hash_bits", 16), **kw)
        elif cfg["alg"] == "rnd":
            m = ppx.PPO_RND(int_hidden_size=cfg["int_hidden"], **kw)
        else:
            m = ppx.PPO_ICM(int_hidden_size=cfg["int_hidden"], **kw)
        self.m, self.ro = m, m.rollout
        host = synth_rollout(cfg, 100 + rank)
        self.pinned = {k: torch.as_tensor(v).pin_memory() for k, v in host.items()}
        self.dones = self.pinned["masks"][-1].clone().pin_memory()
        self.h2d = sum(v.numel() * v.element_size() for v in self.pinned.values()) + self.dones.numel()
        self.last_value_dev = self.pinned["last_value"].to(dev)
        self.dones_dev = self.dones.to(dev)
        self.final_obs_dev = self.pinned["final_obs"].to(dev)
        if cfg["alg"] == "rnd":
            self.last_int_dev = self.pinned["last_int_value"].to(dev)
        if cfg["alg"] in ("rnd", "icm"):
            self.next_obs = torch.empty(T, N, D, dtype=torch.float32, device=dev)
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        self.load()
        self.raw_rewards = self.ro.rewards.clone()

    def load(self):
        # overlap: the fields the bonus does not read go up on a side stream under the bonus kernels (the learner's own
        # methods wait for them); the ICM / RND bonus legs read ro.actions / int fields directly, so they load in order
        self.ro.load_rollout(overlap=self.cfg["alg"] == "ppo", **{k: v for k, v in self.pinned.items() if k in ROLLOUT_FIELDS})

    def bonus_and_gae(self):
        cfg, m, ro = self.cfg, self.m, self.ro
        if cfg["sim_hash"]:
            ro.sim_hash_sharded(ro.observations, ro.rewards)     # W = 1: the plain whole-rollout sim_hash
        if cfg["alg"] in ("rnd", "icm"):
            self.next_obs[:-1].copy_(ro.observations[1:])
            self.next_obs[-1].copy_(self.final_obs_dev)
        if cfg["alg"] == "rnd":
            ro.int_rewards.copy_(m.rnd_bonus_rollout(self.next_obs))
            ro.compute_returns_and_advantages(self.last_value_dev, self.last_int_dev, self.dones_dev)
        elif cfg["alg"] == "icm":
            T, N, D = cfg["T"], cfg["N"], cfg["D"]
            m.intrinsic_module.int_reward(ro.observations.view(T * N, D), self.next_obs.view(T * N, D), ro.actions.view(T * N, 1),
                                          rewards=ro.rewards.view(T * N), eta=m.int_rew_integration)
            ro.compute_returns_and_advantages(self.last_value_dev, self.dones_dev)
        else:
            ro.compute_returns_and_advantages(self.last_value_dev, self.dones_dev)

    def step_resident(self):
        self.flush.zero_()                                      # L2 flush (256 MiB > 126 MB L2), inside the timed region
        self.ro.rewards.copy_(self.raw_rewards)                 # the bonus is applied in place; restore the raw rewards
        self.bonus_and_gae()
        self.m.train()                                          # ends with the D2H read of the loss log

    def step_e2e(self):
        self.flush.zero_()
        self.load()                                             # H2D of the whole rollout from pinned host memory
        self.last_value_dev.copy_(self.pinned["last_value"], non_blocking=True)
        self.dones_dev.copy_(self.dones, non_blocking=True)
        self.final_obs_dev.copy_(self.pinned["final_obs"], non_blocking=True)
        self.bonus_and_gae()
        self.m.train()

    def outputs(self):
        """What one learner pass hands its caller: the loss log of train(), the updated weights of every network it trains,
        and the rollout's rewards (bonus applied), advantages and returns."""
        m, ro, alg = self.m, self.ro, self.cfg["alg"]
        out = {"losses": m.last_losses, "policy_params": m.policy.bank.flat}
        if alg == "rnd":
            out["rnd_params"] = m.rnd.bank.flat
        if alg == "icm":
            out["icm_params"] = m.intrinsic_module.bank.flat
        names = ["rewards", "advantages", "returns"] + (["int_rewards", "int_advantages", "int_returns"] if alg == "rnd" else [])
        out.update((k, getattr(ro, k)) for k in names)
        return {k: dump_array(v) for k, v in out.items()}

    def timed(self, fn, steps):
        import torch.distributed as dist
        torch = self.torch
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=self.dev)
        if self.world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.barrier()
        return float(ms.item())

    def measure(self, steps, warmup, peaks, clocks=None, dump_dir=None):
        """warm-up, K resident steps, K end-to-end steps, one per-op timed pass.  Returns the record (dict).
        dump_dir: write the outputs of the last resident step there (before the end-to-end steps change them)."""
        cfg, m, L, torch = self.cfg, self.m, self.L, self.torch
        for _ in range(warmup):
            self.step_resident()
        torch.cuda.synchronize()
        l0, w0 = L.launch_count(), m.rng_wait_s
        ms = self.timed(self.step_resident, steps)
        launches, rng_wait = L.launch_count() - l0, m.rng_wait_s - w0
        clk = clocks.stop() if clocks is not None else None
        if dump_dir is not None:
            write_outputs(dump_dir, self.outputs())
        self.step_e2e()
        ms_e2e = self.timed(self.step_e2e, steps)
        m.use_cuda_graph = False                                # per-op events need the individual launches, not a graph replay
        self.step_resident()
        with OpTimer(L, torch) as ot:
            self.step_resident()
        agg = ot.summary()
        m.use_cuda_graph = True
        trans = cfg["T"] * cfg["N"] * self.world
        n_mb = cfg["hp"]["n_epochs"] * -(-cfg["T"] * cfg["N"] // cfg["batch"])
        perm_bytes = cfg["hp"]["n_epochs"] * cfg["T"] * cfg["N"] * (4 if m._device_apply() else 8)
        rec = {"value": trans * steps / (ms / 1e3), "unit": "transitions/s", "ms_per_step": ms / steps,
               "e2e": {"value": trans * steps / (ms_e2e / 1e3), "unit": "transitions/s",
                       "h2d_bytes_per_step": int(self.h2d + perm_bytes), "d2h_bytes_per_step": int(n_mb * 64),
                       "ms_per_step": ms_e2e / steps},
               "gpu_launches": int(launches), "launches_per_step": launches / steps,
               "host_rng_wait_ms_per_step": 1e3 * rng_wait / steps,
               "roofline": roofline_of(agg, cfg, peaks) if agg else None}
        if rec["roofline"] and rec["roofline"]["kernel"].startswith("ppx_mlp3_tc_bwd"):
            k_ms, r_ms = ot.bwd_kernel_ms()
            if k_ms:
                rf = rec["roofline"]
                scale = rf["ms_per_launch"] / k_ms               # the entry point = backward kernel + reduce kernel (+ host gaps when eager)
                rf["entry_point_ms_per_call_eager"] = rf["ms_per_launch"]
                rf["ms_per_launch"] = k_ms
                for key in ("achieved", "frac", "fp32_equiv_tflops", "tf32_mma_tflops", "tf32_frac_of_bf16_peak"):
                    if key in rf:
                        rf[key] *= scale
                rf["reduce_kernel_ms_per_launch"] = r_ms
                rf["timing"] = ("CUDA events on the launching stream around the backward kernel ALONE: the last forward + backward "
                                "calls are re-issued 24x back to back after the timed region and the library records the second event "
                                "between the backward kernel and its reduce kernel (ppx_mlp3_tc_bwd_probe); the timed region itself "
                                "replays CUDA graphs, which take no events inside")
        if clk is not None:
            rec["clocks"] = clk
        return rec


def run_ppx(args):
    import torch
    import torch.distributed as dist
    import ppo_exploration_b200 as ppx
    from ppo_exploration_b200 import _lib as L

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    peaks = {}
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        peaks = json.load(open(pk))

    cfg = CONFIGS[args.config]
    bp = PpxPass(args.config, torch, ppx, dev, rank, world)
    m = bp.m
    dump_dir = args.dump_outputs if rank == 0 else None        # sharded: rank 0's envs
    if args.profile:
        for _ in range(args.warmup):
            bp.step_resident()
        ms = bp.timed(bp.step_resident, args.steps)
        if dump_dir is not None:
            write_outputs(dump_dir, bp.outputs())
        if rank == 0:
            print(json.dumps({"profile_run": True, "ms_per_step": ms / args.steps, "launches": L.launch_count()}))
        return
    clocks = ClockSampler(local_rank)                           # sampled over warm-up + timed region (same load; nvidia-smi
    clocks.start()                                              # needs a few hundred ms to produce its first line)
    warm = max(args.warmup, 5)                                  # two staging sets x (eager, capture) before the graphs replay
    sharded = world > 1
    # N > 1: the headline shards the reference's unit of work the data-parallel way -- every rank is the reference's learner
    # on its own envs (its own np.random.permutation over its T x N rollout, buffer.py:239), gradients / loss sums /
    # advantage moments exchanged ("local").  The exact emulation of ONE reference learner over all W x N envs ("global":
    # one permutation of W x T x N indices, identical on every rank) is timed right after as a labelled secondary number:
    # its draws are a single sequential MT19937 stream, W x longer per pass, which no GPU work can hide beyond W = 2
    # (DESIGN.md §5).  PPO_ICM pairs consecutive rows across the shuffle and only has the global mode.
    headline_mode = ("local" if cfg["alg"] != "icm" else "global") if sharded else None
    if sharded:
        m.shard_shuffle = headline_mode
        np.random.seed(1000 + rank if headline_mode == "local" else 0)
    rec = bp.measure(args.steps, warm, peaks, clocks, dump_dir=dump_dir)
    line = {"metric": METRIC, "value": rec["value"], "unit": "transitions/s", "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": rec["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": {"workload": cfg["workload"], "name": args.config},
            "run_config": {"l2": "flushed every step (256 MiB memset inside the timed region)",
                           "shuffle": ("np.random.permutation each epoch inside the timed region (bit-exact reference stream): draws on "
                                       "the host, " + ("swaps on the GPU (copy stream)" if m._device_apply() else "swaps on host worker threads")),
                           "global_minibatch": cfg["batch"] * world,
                           "cuda_graph": "per-minibatch launch sequence replayed as a CUDA graph",
                           "shard_shuffle": (m.shard_shuffle if sharded else "n/a (1 GPU)")},
            "e2e": rec["e2e"], "gpu_launches": rec["gpu_launches"], "clocks": rec["clocks"], "roofline": rec["roofline"],
            "host_rng_wait_ms_per_step": rec["host_rng_wait_ms_per_step"]}
    if sharded and headline_mode == "local":
        m.shard_shuffle = "global"
        np.random.seed(0)                                       # one stream, identical on every rank (checked by the learner)
        w0 = m.rng_wait_s
        for _ in range(5):
            bp.step_resident()
        w0 = m.rng_wait_s
        ms_g = bp.timed(bp.step_resident, args.steps)
        line["global_shuffle"] = {"value": cfg["T"] * cfg["N"] * world * args.steps / (ms_g / 1e3), "unit": "transitions/s",
                                  "ms_per_step": ms_g / args.steps,
                                  "host_rng_wait_ms_per_step": 1e3 * (m.rng_wait_s - w0) / args.steps,
                                  "draws_per_step": cfg["hp"]["n_epochs"] * cfg["T"] * cfg["N"] * world,
                                  "note": "shard_shuffle='global': ONE np.random.permutation(W*T*N) per epoch, drawn identically on every "
                                          "rank (the reference's single learner over all envs, bit-exact index stream); rank r takes "
                                          "its slice of every global minibatch from the all-gathered rollout"}
    del bp, m
    torch.cuda.empty_cache()
    if args.config == "C2":
        line["es"] = es_step_bench(torch, ppx, dev, world, rank)
    if world == 1 and rank == 0:
        use_all_host_threads()
        # the other named shapes (driver-visible numbers for every config of BASELINE.json)
        if args.config == "C2" and not args.no_subconfigs:
            subs = {}
            for name in ("C1", "C3", "C4"):
                try:
                    sp = PpxPass(name, torch, ppx, dev, rank, world)
                    r = sp.measure(3, 5, peaks)
                    r["workload"] = CONFIGS[name]["workload"]
                    del sp
                    torch.cuda.empty_cache()
                    v, det = cpu_pass(name, shrink=1)
                    r["cpu_baseline"] = {"value": v, "unit": "transitions/s", "cores": host_threads()["torch_threads"],
                                         "kind": det["kind"], "sample": det["sample"], "split_s_per_pass": det.get("split_s_per_pass")}
                    subs[name] = r
                except Exception as e:                          # a sub-record must never take the headline down
                    subs[name] = {"error": f"{type(e).__name__}: {e}"}
            line["configs"] = subs
            ces = cpu_es_step()
            if ces is not None and "es" in line:
                line["es"]["cpu_baseline"] = ces
        v, det = cpu_pass(args.config, shrink=1)
        th = host_threads()
        line["cpu_baseline"] = {"value": v, "unit": "transitions/s", "cores": th["torch_threads"], "kind": det["kind"],
                                "sample": det["sample"], "host": th, "split_s_per_pass": det.get("split_s_per_pass")}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        # NCCL communicators referenced by captured CUDA graphs do not tear down cleanly (destroy_process_group
        # blocks); everything is flushed and synchronised here, so leave without the destructor chain.
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush(); sys.stderr.flush()
        os._exit(0)


def main():
    # watchdog: a wedged collective must not burn the box -- dump every thread's stack and exit
    import faulthandler
    faulthandler.dump_traceback_later(int(os.environ.get("PPX_BENCH_WATCHDOG_S", "900")), exit=True)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ppx", choices=["ppx", "reference"])
    ap.add_argument("--config", default="C2", choices=sorted(CONFIGS))
    ap.add_argument("--no-subconfigs", action="store_true", help="C2 headline only (skip the C1/C3/C4 sub-records)")
    ap.add_argument("--profile", action="store_true", help="short run for ncu: W warm-up + K steps only, no e2e/CPU legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (losses, trained weights, rewards, advantages, "
                         "returns) as DIR/<name>.npy; arrays over 4 MB as a fixed seeded sample (ppx arm only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ppx":
        ap.error("--dump-outputs needs --impl ppx")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ppx(args)


if __name__ == "__main__":
    main()
