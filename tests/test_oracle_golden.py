"""Pins the CPU oracle (oracle/) against fixtures produced by the unmodified reference
(tests/golden/make_golden.py).  CPU-only; runs everywhere."""
import numpy as np
import pytest
import torch

from oracle import es as OE
from oracle import learner as OL
from oracle import rollout as OR
from conftest import Golden


@pytest.fixture(autouse=True)
def _one_torch_thread():
    """torch's CPU kernels split some reductions by the intra-op thread count, so the last bit of a trained weight would
    depend on how many cores the host grants (ppo_c1_discrete differs at 3, 5, 6 or 7 threads).  One thread gives the
    fixtures' values bit for bit whatever the core count."""
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    yield
    torch.set_num_threads(n)


@pytest.mark.parametrize("tag", ["a", "b", "c", "d"])
def test_gae_single_bit_exact(tag):
    g = Golden("gae_single").group(tag)
    adv, ret = OR.gae(g["rewards"], g["values"], g["masks"].astype(np.int64), g["last_value"], g["dones"],
                      g["hp"][0], g["hp"][1])
    assert np.array_equal(adv, g["adv"]) and np.array_equal(ret, g["ret"])


@pytest.mark.parametrize("tag", ["a", "b"])
def test_gae_dual_bit_exact(tag):
    g = Golden("gae_dual").group(tag)
    adv, ret, iadv, iret = OR.gae_dual(g["rewards"], g["values"], g["masks"].astype(np.int64), g["last_value"],
                                       g["dones"], g["hp"][0], g["hp"][2], g["int_rewards"], g["int_values"],
                                       g["last_int_value"], g["hp"][1])
    for a, b in ((adv, "adv"), (ret, "ret"), (iadv, "int_adv"), (iret, "int_ret")):
        assert np.array_equal(a, g[b]), b


def test_discount_with_dones():
    g = Golden("discount")
    out = OR.discount_with_dones(g["rewards"], g["dones"], float(g["gamma"]))
    assert np.array_equal(out, g["out"])


@pytest.mark.parametrize("tag,k", [("k16", 16), ("k64", 64), ("k8dup", 8)])
def test_simhash_counts_and_bonus(tag, k):
    g = Golden("simhash").group(tag)
    tab = OR.CountTable(beta=0.1)
    int_tab = {}
    for t in range(g["obs"].shape[0]):
        r, counts = tab.update(g["A"], g["obs"][t], g["rew_in"][t].copy())
        assert np.array_equal(r, g["rew_out"][t])
        codes = OR.pack_bits(OR.simhash_bits(g["A"], g["obs"][t]))
        assert np.array_equal(OR.count_update_codes(int_tab, codes), counts)
    want = {int(OR.pack_bits(b[None].astype(int))[0]): int(c) for b, c in zip(g["table_bits"], g["table_counts"])}
    assert tab.as_code_dict(k) == want == int_tab
    assert counts.max() > 1


def test_simhash_f64_rewards():
    g = Golden("simhash").group("f64")
    r, _ = OR.CountTable().update(g["A"], g["obs"], g["rew_in"].copy())
    assert r.dtype == np.float64 and np.array_equal(r, g["rew_out"])


def test_pack_roundtrip():
    rs = np.random.RandomState(0)
    bits = rs.randint(0, 2, (50, 64))
    codes = OR.pack_bits(bits)
    for c, b in zip(codes, bits):
        assert np.array_equal(OR.unpack_code(c, 64), b)


def test_get_single_indices_and_samples():
    g = Golden("get_single")
    raw = g.group("raw")
    np.random.seed(123)
    for ep in range(2):
        perm = OR.epoch_permutation(8, 3)
        assert np.array_equal(perm, g[f"perm{ep}"])
        for bi, (s, e) in enumerate(OR.minibatch_slices(24, 5)):
            b = OR.gather_single(raw, perm[s:e])
            for f, v in b.items():
                want = g[f"ep{ep}/b{bi}/{f}"]
                assert v.shape == want.shape and v.dtype == want.dtype and np.array_equal(v, want), f
    t, n = OR.flat_to_tn(np.arange(24), 8)
    assert np.array_equal(OR.swap_and_flatten(raw["values"])[:, 0], raw["values"][t, n])


def test_get_dual_samples():
    g = Golden("get_dual")
    raw = g.group("raw")
    np.random.seed(77)
    perm = OR.epoch_permutation(8, 3)
    for bi, (s, e) in enumerate(OR.minibatch_slices(24, 7)):
        b = OR.gather_dual(raw, perm[s:e])
        for f, v in b.items():
            want = g[f"b{bi}/{f}"]
            assert v.shape == want.shape and np.array_equal(v, want), f


def test_running_mean_std():
    g = Golden("rnd_bonus")
    rms = OR.RunningMeanStd()
    for row in g["rms_seq"]:
        rms.update(row[:-3].astype(np.float32))
        assert (rms.mean, rms.var, rms.count) == tuple(row[-3:])
    rv = OR.RunningMeanStd()
    for x in g["rmsv_in"]:
        rv.update(x)
    assert np.array_equal(rv.mean, g["rmsv_mean"]) and np.array_equal(rv.var, g["rmsv_var"])


@pytest.mark.parametrize("norm_reward", [True, False])
def test_vecnormalize_restatement_flags(norm_reward):
    """VecNormalizeRef's training / norm_reward logic (stable_baselines3's step_wait / _update_reward): the statistics
    and the returns move only while training, whatever norm_reward; rewards are divided only with norm_reward; a done
    zeroes its return in every mode."""
    rs = np.random.RandomState(0)
    n, gamma = 5, 0.9
    v = OR.VecNormalizeRef(n, (2,), gamma=gamma, norm_reward=norm_reward)
    v.reset(rs.randn(n, 2))
    ret = np.zeros(n)
    for step in range(12):
        v.training = not (4 <= step < 8)
        obs, r, done = rs.randn(n, 2), rs.randn(n) * 3, rs.rand(n) < 0.3
        before = (v.obs_rms.count, v.ret_rms.count, v.ret_rms.var.copy(), v.obs_rms.mean.copy())
        _, out = v.step(obs, r, done)
        if v.training:
            ret = ret * gamma + r
            assert v.obs_rms.count == before[0] + n and v.ret_rms.count == before[1] + n
        else:
            assert (v.obs_rms.count, v.ret_rms.count) == before[:2]
            assert np.array_equal(v.ret_rms.var, before[2]) and np.array_equal(v.obs_rms.mean, before[3])
        want = np.clip(r / np.sqrt(v.ret_rms.var + 1e-8), -10, 10) if norm_reward else r
        assert np.array_equal(out, want)
        ret[done] = 0
        assert np.array_equal(v.ret, ret)


def _params(g, prefix, requires_grad=True):
    out = {}
    for k, v in g.group(prefix).items():
        t = torch.tensor(v)
        out[k] = t.requires_grad_(True) if (requires_grad and not k.startswith("target")) else t
    return out


def test_rnd_int_reward():
    g = Golden("rnd_bonus")
    for pfx, key in (("rnd", "r"), ("rnd0", "r0")):
        r = OL.rnd_int_reward(_params(g, pfx), g["obs"]).detach().numpy()
        assert np.array_equal(r, g[key])


def _ro(g):
    return g.group("ro")


def _check_params(p, g, prefix, rtol=0, atol=0):
    for k, v in g.group(prefix).items():
        got = p[k].detach().numpy()
        if rtol == 0 and atol == 0:
            assert np.array_equal(got, v), k
        else:
            np.testing.assert_allclose(got, v, rtol=rtol, atol=atol, err_msg=k)


PPO_CASES = {
    "ppo_c1_discrete": dict(discrete=True, hp=dict(n_epochs=10, batch_size=128, clip_range=0.2, ent_coef=0.01,
                                                   vf_coef=1, max_grad_norm=0.2), lr=3e-4),
    "ppo_box_small": dict(discrete=False, hp=dict(n_epochs=3, batch_size=40, clip_range=0.2, ent_coef=0.0,
                                                  vf_coef=1, max_grad_norm=5), lr=3e-4),
    "ppo_box_simhash": dict(discrete=False, hp=dict(n_epochs=2, batch_size=32, clip_range=0.2, ent_coef=0.01,
                                                    vf_coef=1, max_grad_norm=0.2), lr=3e-4),
}


@pytest.mark.parametrize("name", list(PPO_CASES))
def test_ppo_train_matches_reference(name):
    g, c = Golden(name), PPO_CASES[name]
    p = _params(g, "init")
    opt = torch.optim.Adam(OL._policy_param_list(p), lr=c["lr"])
    np.random.seed(int(g["train_seed"]))
    log = OL.ppo_train(p, opt, _ro(g), c["hp"], c["discrete"])
    _check_params(p, g, "final")
    np.testing.assert_allclose(log.mean(axis=0), g["log"], rtol=1e-12)


RND_CASES = {
    "rnd_box_small": dict(discrete=False, hp=dict(n_epochs=3, batch_size=32, clip_range=0.2, ent_coef=0.01,
                                                  vf_coef=0.5, int_vf_coef=0.5, max_grad_norm=5)),
    "rnd_discrete_small": dict(discrete=True, hp=dict(n_epochs=2, batch_size=16, clip_range=0.2, ent_coef=0.01,
                                                      vf_coef=0.5, int_vf_coef=0.5, max_grad_norm=0.2)),
}


@pytest.mark.parametrize("name", list(RND_CASES))
def test_rnd_train_matches_reference(name):
    g, c = Golden(name), RND_CASES[name]
    p, rnd = _params(g, "init"), _params(g, "rnd_init")
    opt = torch.optim.Adam(OL._policy_param_list(p), lr=3e-4)
    rnd_opt = torch.optim.Adam([v for k, v in rnd.items() if k.startswith("predictor")], lr=3e-4)
    np.random.seed(int(g["train_seed"]))
    log, rlog = OL.rnd_train(p, opt, rnd, rnd_opt, _ro(g), c["hp"], c["discrete"], g["rms0/obs_mean"], g["rms0/obs_var"])
    _check_params(p, g, "final")
    _check_params(rnd, g, "rnd_final")
    np.testing.assert_allclose(log.mean(axis=0), g["log"], rtol=1e-12)
    assert np.isfinite(rlog).any()


@pytest.mark.parametrize("name", list(RND_CASES))
def test_rnd_rollout_bonus_matches_reference(name):
    """int_rewards stored by collect_samples (algorithms.py:394-400) from next-obs, frozen obs_rms
    and the running int-reward variance."""
    g = Golden(name)
    ro = _ro(g)
    rnd = _params(g, "rnd_init", requires_grad=False)
    rms = OR.RunningMeanStd()
    # np.float64 (strong dtype), NOT python floats: f32 - python float would stay f32 under NEP 50
    rms.mean, rms.var, rms.count = np.float64(g["rms0/int_mean"]), np.float64(g["rms0/int_var"]), float(g["rms0/int_count"])
    T = ro["observations"].shape[0]
    nxt = np.concatenate([ro["observations"][1:], g["final_obs"][None]], axis=0)
    for t in range(T):
        r = OL.rnd_bonus_step(rnd, nxt[t], g["rms0/obs_mean"], g["rms0/obs_var"], rms)
        assert np.array_equal(r.astype(np.float32), ro["int_rewards"][t]), t
    assert rms.var == float(g["rms1/int_var"])


ICM_CASES = {
    "icm_box_small": dict(discrete=False, hp=dict(n_epochs=2, batch_size=32, clip_range=0.2, ent_coef=0.01,
                                                  vf_coef=0.5, max_grad_norm=0.2, policy_weight=1)),
    "icm_discrete_small": dict(discrete=True, hp=dict(n_epochs=2, batch_size=16, clip_range=0.2, ent_coef=0.01,
                                                      vf_coef=0.5, max_grad_norm=0.2, policy_weight=1)),
}


@pytest.mark.parametrize("name", list(ICM_CASES))
def test_icm_matches_reference(name):
    g, c = Golden(name), ICM_CASES[name]
    p, icm = _params(g, "init"), _params(g, "icm_init")
    a = torch.tensor(g["bonus/a"])
    r = OL.icm_int_reward(icm, torch.tensor(g["bonus/s"]), torch.tensor(g["bonus/ns"]), a, c["discrete"])
    assert np.array_equal(r.detach().numpy(), g["bonus/r"])
    opt = torch.optim.Adam(OL._policy_param_list(p), lr=3e-4)
    icm_opt = torch.optim.Adam(list(icm.values()), lr=3e-4)
    np.random.seed(int(g["train_seed"]))
    log = OL.icm_train(p, opt, icm, icm_opt, _ro(g), c["hp"], c["discrete"])
    _check_params(p, g, "final")
    _check_params(icm, g, "icm_final")
    np.testing.assert_allclose(log.mean(axis=0), g["log"], rtol=1e-12)


def test_es_update_and_knn():
    g = Golden("es")
    shapes = [(8, 16), (16, 16), (16, 2)]
    sizes = [a * b for a, b in shapes]
    offs = np.cumsum([0] + sizes)
    w = [g[f"w0/{i}"] for i in range(3)]
    pop = [[e[offs[l]:offs[l + 1]].reshape(shapes[l]) for l in range(3)] for e in g["eps"]]
    wt = OE.weights_try(w, pop[3], 0.1)
    assert np.array_equal(np.concatenate([x.ravel() for x in wt]), g["try3"])
    w1, lr1 = OE.update_weights(w, g["rewards"], pop, 0.01, 0.1, 0.5, 0.9995, novelty=0.37)
    for i in range(3):
        assert np.array_equal(w1[i], g[f"w1/{i}"])
    assert lr1 == float(g["lr1"])
    w2, lr2 = OE.update_weights(w1, g["rewards"] * 0 + 2.5, pop, lr1, 0.1, 0.5, 0.9995, novelty=0.37)
    assert lr2 == float(g["lr2"]) == lr1 and all(np.array_equal(a, b) for a, b in zip(w1, w2))
    w3, lr3 = OE.update_weights(w2, g["rewards"][::-1].copy(), pop, lr2, 0.1, 0.2, 0.9995)
    for i in range(3):
        assert np.array_equal(w3[i], g[f"w3/{i}"])
    assert lr3 == float(g["lr3"])
    for M in (1, 5, 10, 30, 500):
        s = OE.knn_sum(g[f"knn{M}/archive"], g[f"knn{M}/q"], min(10, M))
        np.testing.assert_allclose(s, float(g[f"knn{M}/sum"]), rtol=1e-13)
    assert np.array_equal(np.array([round(x / g["probs_in"].sum(), 4) for x in g["probs_in"]]), g["probs"])


def test_es_population_rng_order():
    shapes = OE.layer_shapes(8, [16, 16], 2)
    np.random.seed(9)
    pop = OE.get_population(shapes, 3)
    np.random.seed(9)
    for m in pop:
        for l, s in zip(m, shapes):
            assert np.array_equal(l, np.random.randn(*s))


def test_centered_ranks_spec():
    r = np.array([0.3, -1.0, 0.3, 2.0, -1.0])
    ranks, c = OE.centered_ranks(r)
    assert ranks.tolist() == [2, 0, 3, 4, 1]
    assert c.min() == -0.5 and c.max() == 0.5


def test_es_predict_matches_reference():
    """FeedForwardNetwork.predict (evolution_strategies.py:48-61): Box -> tanh(logits); Discrete -> the same
    np.random.choice draws as the reference under the same seed."""
    g = Golden("es_predict")
    for tag, disc in (("box", False), ("disc", True)):
        w = [g[f"{tag}/w/{i}"] for i in range(3)]
        np.random.seed(31)
        got = np.array([OE.predict(w, o, discrete=disc) for o in g[f"{tag}/obs"]]).reshape(6, -1)
        if disc:
            assert np.array_equal(got, g[f"{tag}/actions"])
        else:
            np.testing.assert_allclose(got, g[f"{tag}/actions"], rtol=1e-14, atol=0)


def test_parallel_fisher_yates_equals_sequential():
    """The dependence-free resolution of the shuffle's swaps (the algorithm of csrc/shuffle_dev.cu, restated in
    oracle/rollout.py) equals the sequential swaps on random and adversarial partner lists, and numpy's own
    permutation when fed numpy's draws."""
    rs = np.random.RandomState(0)
    cases = []
    for n in (1, 2, 3, 5, 8, 33, 257, 2000):
        for _ in range(6):
            cases.append(np.array([0] + [rs.randint(0, i + 1) for i in range(1, n)]))
        cases.append(np.zeros(n, dtype=np.int64))                      # everything swaps with position 0 (longest group)
        cases.append(np.arange(n))                                     # only self-swaps
        cases.append(np.maximum(np.arange(n) - 1, 0))                  # a chain: step i targets i-1
    for j in cases:
        assert np.array_equal(OR.fy_apply_parallel(j), OR.fy_apply_sequential(j)), j
    # numpy's own draws (restated bit-exactly in host_rng.cpp, a host function of libppx) -> numpy's permutation
    import ctypes as C
    from ppo_exploration_b200 import _lib as L
    for n in (2, 10, 1000, 4097):
        np.random.seed(n)
        st = np.random.get_state()
        want = np.random.permutation(n)
        key, pos, j = np.ascontiguousarray(st[1], dtype=np.uint32).copy(), C.c_int(int(st[2])), np.zeros(n, np.int32)
        L.call("ppx_np_shuffle_draws32", key.ctypes.data, C.byref(pos), n, j.ctypes.data)
        assert np.array_equal(OR.fy_apply_parallel(j), want), n


def test_logger_csv_schema_matches_reference(tmp_path):
    """ppo-exploration_b200/logger.py writes the reference's CSV schema (logger.py:13-52): same columns ('group/name' ->
    'name'), same cells per row, earlier rows padded when the header grows.  The fixture was written by the reference's
    own CSVOutputFormat (tests/golden/make_golden.py logger); the reference appends new columns in set order (hash
    dependent), so the comparison is by column name, which is how pandas / the notebook read the file."""
    import csv
    import importlib.util
    import os
    from conftest import GOLDEN, ROOT
    spec = importlib.util.spec_from_file_location("ppx_logger", os.path.join(ROOT, "ppo-exploration_b200", "logger.py"))
    lg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(lg)
    dumps = [{"time/total timesteps": 2048, "rollout/ep_rew_mean": 1.5},
             {"time/total timesteps": 4096, "train/value_loss": 0.25, "train/entropy_loss": -1.4, "plain": 3},
             {"rollout/ep_rew_mean": 2.5, "train/value_loss": 0.125}]
    path = str(tmp_path / "run.csv")
    log = lg.Logger([lg.CSVOutputFormat(path)])
    for d in dumps:
        for k, v in d.items():
            log.record(k, v)
        log.dump()
    log.close()

    def table(p):
        with open(p) as f:
            rows = list(csv.DictReader(f))
        return [{k: v for k, v in r.items()} for r in rows]
    got, want = table(path), table(os.path.join(GOLDEN, "logger_ref.csv"))
    assert got == want
