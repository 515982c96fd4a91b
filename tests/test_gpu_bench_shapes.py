"""GPU parity at the BENCHMARKED shapes (VERDICT r1 item 2): the fixtures of test_gpu_learners.py are small
(B <= 128); the kernels take different paths at the C2 minibatch (B = 131 072: multi-CTA loss partials + last-CTA
tail, 148-CTA MLP grids), at the C3 shape (D = 28 224: tcgen05 wide-layer GEMMs) and at the C5 population.

Tolerance = north_star's: 1e-5 relative for losses; gradients are compared per tensor against the tensor's own scale.
Also the teacher-forced walk: ppx is handed the ORACLE's parameters before every minibatch, so every step of a train()
-- not only the first -- is checked at 1e-5 (no Adam amplification of summation-order noise in between)."""
import numpy as np
import pytest
import torch

import bench
from conftest import Golden
from oracle import es as OE
from oracle import learner as OL
from oracle import rollout as OR
from test_oracle_golden import PPO_CASES, RND_CASES, _params, _ro

pytestmark = pytest.mark.gpu

ROLLOUT_FIELDS = bench.ROLLOUT_FIELDS


def _grad_close(got, ref, name, tol=1e-5):
    ref = np.asarray(ref)
    scale = max(float(np.abs(ref).max()), 1e-30)
    err = float(np.abs(np.asarray(got).reshape(ref.shape) - ref).max())
    assert err <= tol * scale, f"{name}: max err {err:.3e} vs scale {scale:.3e} (rel {err / scale:.2e})"


def _loss_close(got, want, tol=1e-5):
    want = np.asarray(want, np.float64)
    got = np.asarray(got, np.float64)
    # the absolute floor covers the policy loss: a mean of O(1) normalised-advantage terms that cancels to ~1e-7 at ratio 1
    assert np.all(np.abs(got - want) <= tol * np.maximum(np.abs(want), 1e-3) + 2e-6), (got, want)


def test_c2_first_minibatch_loss_and_gradients():
    """C2: T=256, N=2048, B=131072, h=64 (tensor-core MLP pair): GAE, loss scalars and every gradient vs the oracle."""
    import ppo_exploration_b200 as ppx
    cfg = bench.CONFIGS["C2"]
    T, N, D, B = cfg["T"], cfg["N"], cfg["D"], cfg["batch"]
    host = bench.synth_rollout(cfg, 5)
    np.random.seed(0); torch.manual_seed(0)
    env = ppx.SyntheticVecEnv(N, D, ppx.Box((2,)))
    m = ppx.PPO(env=env, nstep=T, batch_size=B, hidden_size=cfg["hidden"], **cfg["hp"])
    assert m.policy.mlp._fused_args()["tc"]
    ro = m.rollout
    ro.load_rollout(**{k: v for k, v in host.items() if k in ROLLOUT_FIELDS})
    ro.compute_returns_and_advantages(torch.tensor(host["last_value"]), host["masks"][-1])
    adv, ret = OR.gae(host["rewards"], host["values"], host["masks"].astype(np.int64), host["last_value"], host["masks"][-1],
                      cfg["hp"]["gamma"], cfg["hp"]["gae_lam"])
    np.testing.assert_allclose(ro.advantages.cpu().numpy(), adv, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(ro.returns.cpu().numpy(), ret, rtol=1e-5, atol=1e-5)
    np.random.seed(3)
    idx = ro.permutation()[:B]
    bufs = ro._minibatch_buffers(B)
    ok = m._gather_with_stats(ro, idx, bufs)
    losses = torch.zeros(8, dtype=torch.float64, device="cuda")
    m._policy_step(bufs, B, losses.data_ptr(), stats_ready=ok)
    got = m.policy.state_dict(grad=True)
    p = {k: v.clone().requires_grad_(True) for k, v in m.policy.state_dict().items()}
    buf = {k: host[k] for k in ("observations", "actions", "values", "action_log_probs")}
    buf.update(advantages=ro.advantages.cpu().numpy(), returns=ro.returns.cpu().numpy(), rewards=host["rewards"])
    batch = OL._to_torch(OR.gather_single(buf, idx.cpu().numpy()))
    total, pl, vl, el = OL.ppo_losses(p, batch, dict(cfg["hp"]), False)
    total.backward()
    _loss_close(losses.cpu().numpy()[:4], [total.item(), pl.item(), vl.item(), el.item()])
    for k, v in p.items():
        if v.grad is None:
            assert float(got[k].abs().max()) == 0.0, k
            continue
        _grad_close(got[k].numpy(), v.grad.numpy(), k)


@pytest.mark.parametrize("name", ["ppo_box_small", "ppo_c1_discrete"])
def test_ppo_teacher_forced_every_step(name):
    """Every minibatch of a whole train(): ppx gets the oracle's parameters, then both evaluate the same minibatch."""
    import ppo_exploration_b200 as ppx
    from test_gpu_learners import _env
    g, c = Golden(name), PPO_CASES[name]
    env, T, N = _env(g, c["discrete"])
    hidden = g["init/actor.0.weight"].shape[0]
    m = ppx.PPO(env=env, nstep=T, hidden_size=hidden, lr=c["lr"], **c["hp"])
    ro_host = _ro(g)
    m.rollout.load_rollout(**ro_host)
    p = _params(g, "init")
    opt = torch.optim.Adam(OL._policy_param_list(p), lr=c["lr"])
    plist = OL._policy_param_list(p)
    row = torch.zeros(8, dtype=torch.float64, device="cuda")
    np.random.seed(int(g["train_seed"]))
    steps = 0
    for _ in range(c["hp"]["n_epochs"]):
        perm = OR.epoch_permutation(T, N)
        for s, e in OR.minibatch_slices(T * N, c["hp"]["batch_size"]):
            m.policy.load_state_dict({k: v.detach().clone() for k, v in p.items()})          # teacher forcing
            idx = torch.as_tensor(perm[s:e]).cuda()
            b = idx.numel()
            bufs = m.rollout._minibatch_buffers(c["hp"]["batch_size"])
            ok = m._gather_with_stats(m.rollout, idx, bufs)
            m._policy_step(bufs, b, row.data_ptr(), stats_ready=ok)
            batch = OL._to_torch(OR.gather_single(ro_host, perm[s:e]))
            total, pl, vl, el = OL.ppo_losses(p, batch, c["hp"], c["discrete"])
            _loss_close(row.cpu().numpy()[:4], [total.item(), pl.item(), vl.item(), el.item()])
            opt.zero_grad()
            total.backward()
            if steps % 7 == 0:                                   # spot-check the gradients along the way too
                got = m.policy.state_dict(grad=True)
                for k, v in p.items():
                    if v.grad is not None:
                        _grad_close(got[k].numpy(), v.grad.numpy(), f"step {steps} {k}", tol=1e-4)
            torch.nn.utils.clip_grad_norm_(plist, c["hp"]["max_grad_norm"])
            opt.step()
            steps += 1
    assert steps >= 8


def test_rnd_teacher_forced_every_step():
    import ppo_exploration_b200 as ppx
    from test_gpu_learners import _env
    name = sorted(RND_CASES)[0]
    g, c = Golden(name), RND_CASES[name]
    env, T, N = _env(g, c["discrete"])
    hidden = g["init/actor.0.weight"].shape[0]
    ih = g["rnd_init/predictor.0.weight"].shape[0]
    m = ppx.PPO_RND(env=env, nstep=T, hidden_size=hidden, int_hidden_size=ih, **c["hp"])
    ro_host = _ro(g)
    m.rollout.load_rollout(**ro_host)
    p = _params(g, "init")
    opt = torch.optim.Adam(OL._policy_param_list(p), lr=3e-4)
    plist = OL._policy_param_list(p)
    row = torch.zeros(8, dtype=torch.float64, device="cuda")
    np.random.seed(int(g["train_seed"]))
    for _ in range(c["hp"]["n_epochs"]):
        perm = OR.epoch_permutation(T, N)
        for s, e in OR.minibatch_slices(T * N, c["hp"]["batch_size"]):
            m.policy.load_state_dict({k: v.detach().clone() for k, v in p.items()})
            idx = torch.as_tensor(perm[s:e]).cuda()
            bufs = m.rollout._minibatch_buffers(c["hp"]["batch_size"])
            ok = m._gather_with_stats(m.rollout, idx, bufs, dual=True)
            m._policy_step(bufs, idx.numel(), row.data_ptr(), dual=True, int_vf_coef=m.int_vf_coef, stats_ready=ok)
            batch = OL._to_torch(OR.gather_dual(ro_host, perm[s:e]))
            total, pl, vl, el, ivl = OL.rnd_losses(p, batch, c["hp"], c["discrete"])
            _loss_close(row.cpu().numpy()[:5], [total.item(), pl.item(), vl.item(), el.item(), ivl.item()])
            opt.zero_grad()
            total.backward()
            torch.nn.utils.clip_grad_norm_(plist, c["hp"]["max_grad_norm"])
            opt.step()


def test_c3_shaped_dual_head_step():
    """C3 shape: D = 28 224 flat frames, h = 128, dual value heads, B = 4096: losses + gradients vs the oracle
    (the first layer runs on the tcgen05 wide-layer GEMM, forward and weight gradient)."""
    import ppo_exploration_b200 as ppx
    cfg = dict(bench.CONFIGS["C3"], N=32)                        # 32 envs x 128 steps = one minibatch of 4096
    T, N, D, B = cfg["T"], cfg["N"], cfg["D"], cfg["batch"]
    host = bench.synth_rollout(cfg, 7)
    np.random.seed(0); torch.manual_seed(0)
    env = ppx.SyntheticVecEnv(N, D, ppx.Discrete(18))
    m = ppx.PPO_RND(env=env, nstep=T, batch_size=B, hidden_size=cfg["hidden"], int_hidden_size=16, **cfg["hp"])
    ro = m.rollout
    ro.load_rollout(**{k: v for k, v in host.items() if k in ROLLOUT_FIELDS})
    ro.int_rewards.copy_(torch.as_tensor(np.abs(np.random.RandomState(1).randn(T, N)).astype(np.float32)))
    ro.compute_returns_and_advantages(torch.tensor(host["last_value"]), torch.tensor(host["last_int_value"]), host["masks"][-1])
    np.random.seed(3)
    idx = ro.permutation()[:B]
    bufs = ro._minibatch_buffers(B)
    ok = m._gather_with_stats(ro, idx, bufs, dual=True)
    losses = torch.zeros(8, dtype=torch.float64, device="cuda")
    m._policy_step(bufs, B, losses.data_ptr(), dual=True, int_vf_coef=m.int_vf_coef, stats_ready=ok)
    got = m.policy.state_dict(grad=True)
    p = {k: v.clone().requires_grad_(True) for k, v in m.policy.state_dict().items()}
    buf = {k: host[k] for k in ("observations", "actions", "values", "int_values", "action_log_probs")}
    for k in ("advantages", "returns", "int_advantages", "int_returns"):
        buf[k] = getattr(ro, k).cpu().numpy()
    batch = OL._to_torch(OR.gather_dual(buf, idx.cpu().numpy()))
    total, pl, vl, el, ivl = OL.rnd_losses(p, batch, dict(cfg["hp"]), True)
    total.backward()
    _loss_close(losses.cpu().numpy()[:5], [total.item(), pl.item(), vl.item(), el.item(), ivl.item()])
    for k, v in p.items():
        if v.grad is not None:
            _grad_close(got[k].numpy(), v.grad.numpy(), k, tol=2e-5)


def test_c5_sized_es_update():
    """C5: P = 10 000 members, D = 4736 (MLP 8-64-64-2): _update_weights vs the oracle, novelty mix included."""
    import ppo_exploration_b200 as ppx
    P = 10000
    np.random.seed(11)
    es = ppx.EvolutionStrategy(obs_dim=8, n_actions=2, hidden_sizes=(64, 64), population_size=P, sigma=0.1,
                               learning_rate=0.01, decay=0.9995, novelty_param=0.5)
    w0 = es.get_weights()
    rs = np.random.RandomState(2)
    eps = rs.randn(P, es.D).astype(np.float32)
    rewards = rs.randn(P)
    es._update_weights(rewards, eps, novelty=0.37)
    got = es.get_weights()
    pop = []
    for m_ in range(P):
        o, layers = 0, []
        for sh, n in zip(es.shapes, es.layer_sizes):
            layers.append(eps[m_, o:o + n].reshape(sh).astype(np.float64))
            o += n
        pop.append(layers)
    want, lr = OE.update_weights(w0, rewards, pop, 0.01, 0.1, 0.5, 0.9995, novelty=0.37)
    for a, b in zip(got, want):
        np.testing.assert_allclose(a, b, rtol=1e-10, atol=1e-12)
    assert abs(es.learning_rate - lr) < 1e-15


def test_novelty_distribution_and_brain_pick_product():
    """calc_noveltiy_distribution (evolution_strategies.py:283-290) and the brain pick (:327-333) of the PRODUCT class
    against the oracle's restatement, same host RNG draw."""
    import ppo_exploration_b200 as ppx
    np.random.seed(0)
    es = ppx.EvolutionStrategy(obs_dim=4, n_actions=2, hidden_sizes=(8,), population_size=4)
    for nov in ([0.3, 0.7], [1.0, 1.0, 5e-3], [0.123456, 0.2, 0.31, 0.05]):
        probs = es.calc_noveltiy_distribution(nov)
        assert probs == [round(n / sum(nov), 4) for n in nov]
        want = OE.novelty_distribution(nov)
        np.random.seed(5)
        want_idx = int(np.random.choice(list(range(len(nov))), p=want))
        np.random.seed(5)
        idx, n = es.pick_brain(nov)
        assert idx == want_idx and n == nov[idx]


def test_dump_outputs_are_the_last_timed_step(tmp_path, monkeypatch):
    """bench.py --dump-outputs: measure(dump_dir=...) writes the outputs of the last timed resident step, before the
    end-to-end steps move the learner on -- a fresh pass object stepped warm-up + K times by hand computes the same arrays
    bit for bit (C2 at 64 envs x 64 steps)."""
    import os
    import ppo_exploration_b200 as ppx
    monkeypatch.setitem(bench.CONFIGS, "C2", dict(bench.CONFIGS["C2"], N=64, T=64, batch=1024))
    dev = torch.device("cuda", 0)
    bp = bench.PpxPass("C2", torch, ppx, dev, 0, 1)
    bp.measure(2, 5, {}, dump_dir=str(tmp_path))
    del bp
    got = {f[:-4]: np.load(os.path.join(tmp_path, f)) for f in os.listdir(tmp_path)}
    assert set(got) == {"losses", "policy_params", "rewards", "advantages", "returns"}
    assert got["losses"].dtype == np.float64 and got["losses"].shape == (40, 8) and got["advantages"].shape == (64, 64)
    bp = bench.PpxPass("C2", torch, ppx, dev, 0, 1)
    for _ in range(5 + 2):
        bp.step_resident()
    for k, v in bp.outputs().items():
        assert v.dtype == got[k].dtype and np.array_equal(v, got[k]), k
    bp.step_resident()
    assert not np.array_equal(bp.outputs()["policy_params"], got["policy_params"])
