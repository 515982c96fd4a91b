"""ES-NSRA with a novelty per member (novelty_mode="member", DESIGN.md §3.16) on the GPU.

  * k-NN: ppx_knn_novelty (one warp per query and archive slice, a square root per pair, a merge launch) against
    ppx_knn_novelty_many (one thread per query, squared distances, square roots of the K winners only) at Q = 2 and
    Q = 10 000 queries, M in {1e2, 1e3, 1e4, 1e5} archive rows, dim 2, K 10: CUDA events over many launches, pairs/s,
    and the model Q*M*3*dim f64 flops, M*dim*8 bytes per CTA pass of the archive.  The archive (<= 1.6 MB) stays in L2.
  * update: ppx_es_update_member against ppx_es_update at C5 (P = 10 000, D = 4736, table offsets, z-score) against the
    4*D bytes per perturbation of the noise read.
  * run(): per generation in both modes on the C5 table env and MountainCarContinuous-v0 (tools/es_run_prof.py's
    instrumentation).
  * MountainCar-v0 (P = 1024, M = 2, MLP 2-64-64-3): the first generation whose f_b > -200, both modes, several seeds.
The GPU's name and power limit are recorded with the numbers.

    python tools/es_member_prof.py [--out profiles/es_member_r07.json]
"""
import argparse
import json
import os
import sys
import tempfile

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ppo_exploration_b200 as ppx  # noqa: E402
from ppo_exploration_b200 import _lib as L  # noqa: E402
from es_eval_prof import TableEnv, gpu_meta, time_events  # noqa: E402
import es_run_prof  # noqa: E402


def knn_arm(Q, M, dim=2, K=10):
    rs = np.random.RandomState(Q + M)
    a = torch.as_tensor(rs.randn(M, dim)).cuda()
    q = torch.as_tensor(rs.randn(Q, dim)).cuda()
    s = torch.empty(Q, dtype=torch.float64, device="cuda")
    n = torch.empty_like(s)
    reps = int(max(3, min(500, 2e9 / (Q * M))))
    out = dict(Q=Q, M=M, dim=dim, K=K, model_flop=3 * Q * M * dim, model_bytes_per_cta_pass=M * dim * 8)
    res = {}
    for name in ("ppx_knn_novelty", "ppx_knn_novelty_many"):
        us = time_events(lambda: L.call(name, a.data_ptr(), M, q.data_ptr(), Q, dim, K, s.data_ptr(), n.data_ptr(), L.stream()),
                         reps)
        res[name] = n.clone()
        out[name] = dict(us=round(us, 2), pairs_per_s=float(f"{Q * M / (us * 1e-6):.4g}"),
                         gflop_s=round(3 * Q * M * dim / (us * 1e3), 1))
    out["bit_identical"] = bool(torch.equal(res["ppx_knn_novelty"], res["ppx_knn_novelty_many"]))
    return out


def update_arm():
    P, D = 10_000, 4736
    np.random.seed(0)
    es = ppx.EvolutionStrategy(obs_dim=8, n_actions=2, hidden_sizes=(64, 64), population_size=P, sigma=0.02,
                               learning_rate=0.01, noise_table_size=1 << 28, noise_seed=1)
    assert es.D == D
    off = es._get_population()
    r = torch.randn(P, dtype=torch.float64, device="cuda")
    nov = torch.rand(P, dtype=torch.float64, device="cuda")
    noise = es.noise_table()
    ws = torch.zeros(max(L.call("ppx_es_update_workspace", P, D), L.call("ppx_es_update_member_workspace", P, D)) // 8 + 1,
                     dtype=torch.float64, device="cuda")
    lr = torch.full((1,), 0.01, dtype=torch.float64, device="cuda")
    st = torch.zeros(1, dtype=torch.int32, device="cuda")
    th = es.theta

    def brain():
        L.call("ppx_es_update", th.data_ptr(), noise.data_ptr(), off.data_ptr(), r.data_ptr(), P, D, 0.02, 0.5, 0.3, None, 1, 0,
               1.0, lr.data_ptr(), st.data_ptr(), ws.data_ptr(), L.stream())

    def member():
        L.call("ppx_es_update_member", th.data_ptr(), noise.data_ptr(), off.data_ptr(), r.data_ptr(), nov.data_ptr(), P, 0, P, D,
               0.02, 0.5, 0, 1.0, lr.data_ptr(), st.data_ptr(), ws.data_ptr(), None, None, None, 1, 0, None, None, L.stream())
    out = dict(P=P, D=D, model_bytes=4 * D * P)
    for name, fn in (("ppx_es_update", brain), ("ppx_es_update_member", member)):
        us = time_events(fn, 200)
        out[name] = dict(us=round(us, 2), model_gb_s=round(4 * D * P / (us * 1e3), 1))
    return out


def run_arms(gens):
    out = {}
    for mode in ("brain", "member"):
        np.random.seed(0)
        es = ppx.EvolutionStrategy(obs_dim=8, n_actions=2, hidden_sizes=(64, 64), population_size=es_run_prof.P, sigma=0.02,
                                   learning_rate=0.01, noise_table_size=1 << 28, noise_seed=1, novelty_mode=mode)
        r = es_run_prof.timed_run(es, TableEnv(es_run_prof.P, "cuda", False), TableEnv(es_run_prof.M, "cuda", False, seed=1),
                                  gens, 1000)
        out[f"c5_table_{mode}"] = dict(workload="P=10000, MLP 8-64-64-2, table env, max_steps 1000", **r)
        np.random.seed(0)
        es = ppx.EvolutionStrategy(env_id="MountainCarContinuous-v0", obs_dim=2, n_actions=1, hidden_sizes=(64, 64),
                                   population_size=es_run_prof.P, sigma=0.1, learning_rate=0.01, noise_table_size=1 << 26,
                                   noise_seed=1, novelty_mode=mode)
        env = ppx.ClassicControlVecEnv("MountainCarContinuous-v0", es_run_prof.P, seed=0, reward_dtype=torch.float64)
        benv = ppx.ClassicControlVecEnv("MountainCarContinuous-v0", es_run_prof.M, seed=1, reward_dtype=torch.float64)
        r = es_run_prof.timed_run(es, env, benv, gens, 999)
        out[f"mountaincar_continuous_{mode}"] = dict(workload="P=10000, MLP 2-64-64-1, max_steps 999", **r)
    return out


def mountaincar(mode, seed, budget, P=1024, M=2):
    """tests/test_gpu_es_member_novelty.py::mountaincar_run's configuration: the f_b of every generation."""
    np.random.seed(seed)
    es = ppx.EvolutionStrategy(env_id="MountainCar-v0", hidden_sizes=(64, 64), obs_dim=2, n_actions=3, population_size=P,
                               sigma=0.1, learning_rate=0.05, noise_seed=seed + 1, noise_table_size=1 << 22, novelty_mode=mode)
    env = ppx.ClassicControlVecEnv("MountainCar-v0", P, seed=seed, reward_dtype=torch.float64)
    benv = ppx.ClassicControlVecEnv("MountainCar-v0", M, seed=seed + 1, env_offset=0, reward_dtype=torch.float64)
    fb = []
    finish = es._finish_generation

    def rec(pending, vals, *a):
        fb.append(float(vals[M]))
        return finish(pending, vals, *a)
    es._finish_generation = rec
    es.run(env, benv, budget, max_steps=200, meta_population_size=M, reward_target=-200)
    reached = bool(fb) and fb[-1] > -200
    return dict(mode=mode, seed=seed, budget=budget, reached=reached, generations=len(fb),
                first_generation_above_minus_200=len(fb) if reached else None, last_fb=fb[-1] if fb else None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "es_member_r07.json"))
    ap.add_argument("--gens", type=int, default=10)
    ap.add_argument("--mc-budget", type=int, default=150)
    ap.add_argument("--mc-seeds", type=int, default=6)
    ap.add_argument("--skip-run", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("es_member_prof.py measures on the GPU; no CUDA device found")
    torch.cuda.set_device(0)
    args.out = os.path.abspath(args.out)
    out = dict(gpu_meta(), tool="tools/es_member_prof.py")
    os.chdir(tempfile.mkdtemp())                               # run() configures the logger; nothing is written to file
    out["knn"] = [knn_arm(Q, M) for Q in (2, 10_000) for M in (100, 1000, 10_000, 100_000)]
    for k in out["knn"]:
        print("knn", json.dumps(k))
    out["update_c5"] = update_arm()
    print("update", json.dumps(out["update_c5"]))
    out["mountaincar_v0"] = [mountaincar(mode, s, args.mc_budget) for s in range(args.mc_seeds) for mode in ("member", "brain")]
    for m in out["mountaincar_v0"]:
        print("mountaincar", json.dumps(m))
    if not args.skip_run:
        out["run"] = run_arms(args.gens)
        for name, a in out["run"].items():
            print(name, json.dumps({k: v for k, v in a.items() if k not in ("population_steps", "brain_steps")}))
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: v for k, v in out.items() if k not in ("knn", "run", "mountaincar_v0", "update_c5")}))


if __name__ == "__main__":
    main()
