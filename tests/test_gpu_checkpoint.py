"""GPU tests of checkpoints (DESIGN.md §3.14): restoring a SimHash count table (ppx_count_table_load), and learners / ES that
are saved, loaded into fresh objects and continued -- bit-identical to the run that was never interrupted, and to one that
never saved.  The 2-GPU case is skipped below 2 GPUs."""
import os
import socket
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
M64 = (1 << 64) - 1


def _ppx():
    import ppo_exploration_b200 as ppx
    return ppx


# ---------------------------------------------------------------- count table
def _unxorshift(x, s):
    y = x
    for _ in range(64 // s + 1):
        y = x ^ (y >> s)
    return y


def _unmix64(h):
    """Inverse of simhash.cu's splitmix64 finaliser: the code whose home slot hash is h."""
    x = _unxorshift(h, 31)
    x = (x * pow(0x94d049bb133111eb, -1, 1 << 64)) & M64
    x = _unxorshift(x, 27)
    x = (x * pow(0xbf58476d1ce4e5b9, -1, 1 << 64)) & M64
    return _unxorshift(x, 30)


def _mix64(x):
    x ^= x >> 30
    x = (x * 0xbf58476d1ce4e5b9) & M64
    x ^= x >> 27
    x = (x * 0x94d049bb133111eb) & M64
    return x ^ (x >> 31)


def _codes(vals):
    return torch.from_numpy(np.array(vals, dtype=np.uint64).view(np.int64)).cuda()


def _table_cases():
    rs = np.random.RandomState(7)
    rand = rs.randint(0, 1 << 62, size=1 << 20, dtype=np.int64).astype(np.uint64) * np.uint64(3) + np.uint64(1)
    h0 = 0x123456789ABCDEF0 & M64
    collide = [_unmix64((h0 & ((1 << 20) - 1)) | (j << 20)) for j in range(1, 65)]   # one home slot for any capacity <= 2^20
    assert len({_mix64(c) & ((1 << 20) - 1) for c in collide}) == 1
    return {
        "empty": [],
        "one": [42, 42, 42],
        "all_ones": [M64, 5, M64],
        "random_2^20": np.concatenate([rand, rand[:1000]]),
        "collide": collide + collide[:10] + [M64],
    }


@pytest.mark.parametrize("case", list(_table_cases()))
def test_count_table_load_equals_dump(case):
    ppx = _ppx()
    codes = _table_cases()[case]
    t = ppx.CountTable()
    if len(codes):
        t.update_codes(_codes(codes))
    sd = t.state_dict()
    k = sd["keys"].numpy().view(np.uint64)
    assert np.all(k[1:] > k[:-1]), "state_dict keys are not sorted"
    r = ppx.CountTable(1024)
    r.load_state_dict(sd)
    assert r.items() == t.items()
    assert len(r) == len(t) == len(np.unique(np.array(codes, dtype=np.uint64)))
    assert r.capacity() == t.capacity()
    if case == "all_ones":
        assert r.items()[M64] == 2


@pytest.mark.parametrize("grow", [False, True])
def test_restored_table_continues_bit_identically(grow):
    """The same code stream applied to the original and to the restored table gives the same counts_out, SimHash bonuses
    and tables -- including a stream that makes both grow."""
    ppx = _ppx()
    from ppo_exploration_b200 import _lib as L
    rs = np.random.RandomState(3)
    t = ppx.CountTable(1 << 16)                                 # growth is decided per call from its length
    first = rs.randint(0, 1500, size=20000).astype(np.uint64) * np.uint64(0x9E3779B97F4A7C15)
    t.update_codes(_codes(first))
    r = ppx.CountTable()
    r.load_state_dict(t.state_dict())
    assert r.capacity() == t.capacity() == 1 << 16
    n_new = 40000 if grow else 200
    more = np.concatenate([first[:5000], rs.randint(1, 1 << 60, size=n_new).astype(np.uint64), [M64]])
    rs.shuffle(more)
    c_t, c_r = t.update_codes(_codes(more)), r.update_codes(_codes(more))
    assert torch.equal(c_t, c_r)
    # SimHash bonuses from observations (codes computed on the device), on both tables
    D, k, n = 6, 24, 30000
    A = torch.from_numpy(rs.randn(k, D)).cuda()
    obs = torch.from_numpy((rs.randn(n, D) * 0.3).astype(np.float32)).cuda()
    rew = []
    for tab in (t, r):
        out = torch.zeros(n, dtype=torch.float64, device="cuda")
        L.call("ppx_simhash_update", tab._h, A.data_ptr(), obs.data_ptr(), k, D, n, 0.1, out.data_ptr(), 1, None, None,
               L.stream())
        rew.append(out)
    assert torch.equal(rew[0], rew[1])
    assert t.items() == r.items()
    assert t.capacity() == r.capacity()
    assert (t.capacity() > 1 << 16) == grow


def test_count_table_load_rejects_bad_input():
    ppx = _ppx()
    from ppo_exploration_b200 import _lib as L

    def load(tab, keys, counts):
        k = _codes(keys)
        c = torch.tensor(counts, dtype=torch.int32, device="cuda")
        L.call("ppx_count_table_load", tab._h, k.data_ptr(), c.data_ptr(), len(keys), L.stream())

    t = ppx.CountTable()
    with pytest.raises(RuntimeError, match="duplicate"):
        load(t, [1, 2, 3, 2], [1, 1, 1, 4])
    assert len(t) == 0 and t.items() == {}, "a rejected load left a partial table"
    with pytest.raises(RuntimeError, match="duplicate"):
        load(t, [M64, 9, M64], [1, 1, 1])
    assert len(t) == 0
    with pytest.raises(RuntimeError, match="zero count"):
        load(t, [5, 6], [3, 0])
    assert len(t) == 0
    load(t, [5, 6, M64], [3, 1, 2])                             # the table is still usable
    assert t.items() == {5: 3, 6: 1, M64: 2}
    with pytest.raises(RuntimeError, match="not empty"):
        load(t, [7], [1])
    assert t.items() == {5: 3, 6: 1, M64: 2}


# ---------------------------------------------------------------- learners
FIELDS = ("observations", "actions", "rewards", "int_rewards", "values", "returns", "action_log_probs", "masks", "advantages",
          "int_values", "int_returns", "int_advantages")
BASE = dict(nstep=32, batch_size=128, n_epochs=2)


def _env(kind):
    ppx = _ppx()
    if kind == "mcc_vecnorm":
        return ppx.make_env("MountainCarContinuous-v0", 16, seed=4)
    if kind == "cartpole":
        return ppx.ClassicControlVecEnv("CartPole-v1", 16, seed=9)
    if kind == "host_cartpole":
        return ppx.ToNumpy(ppx.EpisodeMonitor(ppx.ClassicControlVecEnv("CartPole-v1", 16, seed=9)))
    raise KeyError(kind)


CASES = {   # learner, constructor arguments, env, iterations before the save, after it
    "ppo_simhash_box_vecnorm": ("PPO", dict(hidden_size=64, sim_hash=True, hash_bits=64), "mcc_vecnorm", 2, 2),
    "ppo_discrete": ("PPO", dict(hidden_size=64), "cartpole", 2, 2),
    "rnd_during_warmup": ("PPO_RND", dict(hidden_size=64, int_hidden_size=32, rnd_start=40), "cartpole", 1, 2),
    "rnd_after_warmup": ("PPO_RND", dict(hidden_size=64, int_hidden_size=32, rnd_start=40), "cartpole", 2, 2),
    "icm": ("PPO_ICM", dict(hidden_size=64, int_hidden_size=32), "cartpole", 2, 2),
    "host_ppo_simhash": ("PPO", dict(hidden_size=64, sim_hash=True, hash_bits=32), "host_cartpole", 2, 2),
    "host_rnd": ("PPO_RND", dict(hidden_size=64, int_hidden_size=32, rnd_start=40), "host_cartpole", 1, 2),
}


def _iterate(m, n):
    """n iterations; per iteration the rollout the collect produced and the loss log of the train."""
    out = []
    for _ in range(n):
        m.collect_samples()
        roll = {k: getattr(m.rollout, k).clone() for k in FIELDS if hasattr(m.rollout, k)}
        m.train()
        out.append((roll, m.last_losses.copy()))
    torch.cuda.synchronize()
    return out


def _state(m):
    """Everything a resume must reproduce, on the host."""
    s = {"banks": {k: b.state_dict() for k, b in m._ckpt_banks().items()},
         "rms": {k: r.state_dict() for k, r in m._ckpt_rms().items()},
         "table": m.rollout.count_table.items() if m.rollout.count_table is not None else None,
         "A": m.rollout.A.copy(), "episodes": m.num_episodes, "timesteps": m.num_timesteps, "n_updates": m._n_updates,
         "draws": m.policy._draws, "infos": list(m.ep_info_buffer), "np": np.random.get_state(),
         "env": m.env.state_dict() if hasattr(m.env, "state_dict") else None}
    return s


def _equal(a, b, path="state"):
    if isinstance(a, torch.Tensor):
        assert isinstance(b, torch.Tensor) and a.dtype == b.dtype and torch.equal(a, b), f"{path} differs"
    elif isinstance(a, np.ndarray):
        assert np.array_equal(a, b) and a.dtype == b.dtype, f"{path} differs"
    elif isinstance(a, dict):
        assert set(a) == set(b), f"{path}: keys {set(a) ^ set(b)}"
        for k in a:
            _equal(a[k], b[k], f"{path}.{k}")
    elif isinstance(a, (list, tuple)):
        assert len(a) == len(b), f"{path}: length"
        for i, (x, y) in enumerate(zip(a, b)):
            _equal(x, y, f"{path}[{i}]")
    else:
        assert a == b, f"{path}: {a!r} != {b!r}"


def _same_runs(x, y):
    for i, ((ra, la), (rb, lb)) in enumerate(zip(x, y)):
        _equal(ra, rb, f"iteration {i} rollout")
        assert np.array_equal(la, lb), f"iteration {i}: last_losses differ"


@pytest.mark.parametrize("case", list(CASES))
def test_resume_equals_uninterrupted(case, tmp_path):
    ppx = _ppx()
    algo, kw, env_kind, k, m_after = CASES[case]
    cls = getattr(ppx, algo)
    p = str(tmp_path / "ck.pt")
    # the run that never saved
    np.random.seed(3)
    torch.manual_seed(3)
    ref = cls(env=_env(env_kind), **dict(BASE, **kw))
    _iterate(ref, k)
    ref_tail = _iterate(ref, m_after)
    ref_state = _state(ref)
    # the run that saves after k iterations and goes on
    np.random.seed(3)
    torch.manual_seed(3)
    a = cls(env=_env(env_kind), **dict(BASE, **kw))
    _iterate(a, k)
    a.save(p)
    a_tail = _iterate(a, m_after)
    a_state = _state(a)
    _same_runs(ref_tail, a_tail)
    _equal(ref_state, a_state)
    # a fresh learner from the file, over a fresh env, continues identically
    np.random.seed(99)                                          # load() restores numpy's state
    torch.manual_seed(99)
    b = cls.load(p, env=_env(env_kind))
    assert b.resumed_env_state is True
    assert b.device_env == a.device_env == (not env_kind.startswith("host"))
    b_tail = _iterate(b, m_after)
    _same_runs(a_tail, b_tail)
    _equal(a_state, _state(b))
    if kw.get("sim_hash"):
        assert len(a_state["table"]) > 0
    if env_kind != "mcc_vecnorm":                               # MountainCarContinuous runs 999-step episodes: none end here
        assert a_state["episodes"] > 0 and len(a_state["infos"]) > 0


def test_learn_resume_stops_at_the_same_iteration(tmp_path):
    """learn(T1), save, load, learn(T2) equals learn(T2), where the reward target stops the run after the resume."""
    ppx = _ppx()
    T2, it = 16 * 32 * 40, 16 * 32
    kw = dict(BASE, hidden_size=64)

    def fresh():
        np.random.seed(0)
        torch.manual_seed(0)
        return ppx.PPO(env=ppx.ClassicControlVecEnv("CartPole-v1", 16, seed=2), **kw)

    ref = fresh().learn(total_timesteps=T2, log_interval=None, reward_target=25)
    stop = ref.num_timesteps // it
    assert 2 <= stop < 40, f"the reward target stopped the run after {stop} iterations"
    a = fresh().learn(total_timesteps=(stop - 1) * it, log_interval=None, reward_target=25)
    assert a.num_timesteps == (stop - 1) * it
    p = str(tmp_path / "ck.pt")
    a.save(p)
    b = ppx.PPO.load(p, env=ppx.ClassicControlVecEnv("CartPole-v1", 16, seed=2))
    b.learn(total_timesteps=T2, log_interval=None, reward_target=25)
    assert b.num_timesteps == ref.num_timesteps
    _equal(_state(ref), _state(b))
    assert np.array_equal(ref.last_losses, b.last_losses)
    # learn(T2) without a target runs on past the stop: equal too.  Both runs draw from numpy's global RNG, so the
    # uninterrupted one finishes before the resumed one is loaded (load() sets the global state the resume continues from)
    d = fresh().learn(total_timesteps=(stop - 1) * it, log_interval=None, reward_target=25)
    d.learn(total_timesteps=(stop + 2) * it, log_interval=None)
    d_state = _state(d)
    c = ppx.PPO.load(p, env=ppx.ClassicControlVecEnv("CartPole-v1", 16, seed=2))
    c.learn(total_timesteps=(stop + 2) * it, log_interval=None)
    _equal(d_state, _state(c))


def test_env_without_state_protocol_resets(tmp_path):
    ppx = _ppx()
    np.random.seed(1)
    torch.manual_seed(1)
    m = ppx.PPO(env=ppx.SyntheticVecEnv(16, 4, ppx.Discrete(2)), **dict(BASE, hidden_size=64))
    _iterate(m, 1)
    p = str(tmp_path / "ck.pt")
    m.save(p)
    assert torch.load(p, weights_only=True)["env"] is None
    b = ppx.PPO.load(p, env=ppx.SyntheticVecEnv(16, 4, ppx.Discrete(2)))
    assert b.resumed_env_state is False
    _equal(_state(m)["banks"], _state(b)["banks"])
    _iterate(b, 1)


# ---------------------------------------------------------------- errors and format
def _saved(tmp_path, **kw):
    ppx = _ppx()
    np.random.seed(0)
    torch.manual_seed(0)
    m = ppx.PPO(env=ppx.SyntheticVecEnv(16, 4, ppx.Discrete(2)), **dict(BASE, hidden_size=64, sim_hash=True, **kw))
    p = str(tmp_path / "ck.pt")
    m.save(p)
    return m, p


def test_mismatches_raise_value_error(tmp_path):
    ppx = _ppx()
    Syn, Dis, Box = ppx.SyntheticVecEnv, ppx.Discrete, ppx.Box
    m, p = _saved(tmp_path)
    ppx.PPO.load(p, env=Syn(16, 4, Dis(2)))                     # fits
    with pytest.raises(ValueError, match="PPO_RND"):
        ppx.PPO_RND.load(p, env=Syn(16, 4, Dis(2)))
    for env, what in ((Syn(8, 4, Dis(2)), "num_envs"), (Syn(16, 3, Dis(2)), "obs_dim"), (Syn(16, 4, Box((2,))), "action_space"),
                      (Syn(16, 4, Dis(3)), "action_n")):
        with pytest.raises(ValueError, match=what):
            ppx.PPO.load(p, env=env)
    ck = torch.load(p, weights_only=True)
    for key, val in (("hidden_size", 32), ("nstep", 64), ("hash_bits", 8), ("world_size", 2), ("rank", 1)):
        bad = dict(ck, shape=dict(ck["shape"], **{key: val}))
        q = str(tmp_path / f"bad_{key}.pt")
        torch.save(bad, q)
        with pytest.raises(ValueError, match=key):
            ppx.PPO.load(q, env=Syn(16, 4, Dis(2)))
    q = str(tmp_path / "bad_version.pt")
    torch.save(dict(ck, version=2), q)
    with pytest.raises(ValueError, match="version"):
        ppx.PPO.load(q, env=Syn(16, 4, Dis(2)))


def test_save_with_an_untrained_rollout_raises(tmp_path):
    ppx = _ppx()
    m = ppx.PPO(env=ppx.ClassicControlVecEnv("CartPole-v1", 16, seed=0), **dict(BASE, hidden_size=64))
    m.save(str(tmp_path / "before.pt"))
    m.collect_samples()
    with pytest.raises(RuntimeError, match="not been trained"):
        m.save(str(tmp_path / "mid.pt"))
    m.train()
    m.save(str(tmp_path / "after.pt"))


def test_file_is_weights_only_and_deterministic(tmp_path):
    ppx = _ppx()
    np.random.seed(2)
    torch.manual_seed(2)
    m = ppx.PPO(env=ppx.make_env("MountainCarContinuous-v0", 64, seed=1), **dict(BASE, hidden_size=64, sim_hash=True))
    _iterate(m, 2)
    st = np.random.get_state()
    m.save(str(tmp_path / "a.pt"))
    m.save(str(tmp_path / "b.pt"))
    _equal(st, np.random.get_state())                           # saving draws nothing
    a = torch.load(str(tmp_path / "a.pt"), weights_only=True)
    b = torch.load(str(tmp_path / "b.pt"), weights_only=True)
    assert a["format"] == "ppx-checkpoint" and a["version"] == 1 and a["class"] == "PPO"
    assert a["simhash"]["count_table"]["keys"].numel() > 1
    _equal(a, b, "checkpoint")


# ---------------------------------------------------------------- ES
@pytest.mark.parametrize("env_id", ["MountainCarContinuous-v0", "CartPole-v1"])
def test_es_resume_equals_uninterrupted(env_id, tmp_path):
    ppx = _ppx()
    P, steps, k, m_after = 256, 200, 2, 3
    obs_dim, n_act = (2, 1) if env_id.startswith("Mountain") else (4, 2)

    def env():
        return ppx.ClassicControlVecEnv(env_id, P, seed=11, reward_dtype=torch.float64)

    def gens(es, e, n):
        out = []
        for _ in range(n):
            f, l, _ = es.run_generation(e, max_steps=steps)
            out.append((f.clone(), l.clone(), es.theta.clone(), es._lr.clone(), es._draw.clone()))
        torch.cuda.synchronize()
        return out

    np.random.seed(4)
    es = ppx.EvolutionStrategy(hidden_sizes=(16, 16), obs_dim=obs_dim, n_actions=n_act, population_size=P, sigma=0.1,
                               learning_rate=0.05, decay=0.999, noise_table_size=1 << 20, noise_seed=5)
    e = env()
    gens(es, e, k)
    p = str(tmp_path / "es.pt")
    es.save(p)
    env_sd = e.state_dict()
    tail = gens(es, e, m_after)
    es2 = ppx.EvolutionStrategy.load(p)
    e2 = env()
    e2.load_state_dict(env_sd)
    tail2 = gens(es2, e2, m_after)
    for i, (x, y) in enumerate(zip(tail, tail2)):
        for name, u, v in zip(("fitness", "lengths", "theta", "lr", "draw"), x, y):
            assert torch.equal(u, v), f"generation {i}: {name} differs"
    assert not torch.equal(tail[0][2], tail[-1][2]), "theta did not move"
    assert int(tail[-1][4][0]) == k + m_after


# ---------------------------------------------------------------- 2 GPUs
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, d):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", rank), rank=rank, world_size=world)
    import ppo_exploration_b200 as ppx
    kw = dict(BASE, hidden_size=64, sim_hash=True, hash_bits=64)

    def env():
        return ppx.ClassicControlVecEnv("MountainCarContinuous-v0", 16, seed=4)

    np.random.seed(3)
    torch.manual_seed(3)
    a = ppx.PPO(env=env(), **kw)
    assert a.shard_shuffle == "global" and a.env.env_offset == 16 * rank
    _iterate(a, 2)
    p = os.path.join(d, f"ck_rank{rank}.pt")
    a.save(p)
    tail = _iterate(a, 2)
    sa = _state(a)
    b = ppx.PPO.load(p, env=env())
    tail_b = _iterate(b, 2)
    _same_runs(tail, tail_b)
    _equal(sa, _state(b))
    ck = torch.load(p, weights_only=True)
    assert ck["shape"]["world_size"] == world and ck["shape"]["rank"] == rank and ck["simhash"]["count_table"]["sharded"]
    dist.barrier()
    torch.cuda.synchronize()
    os._exit(0)                                                # NCCL communicators referenced by captured graphs do not tear down cleanly


def test_sharded_resume_equals_uninterrupted(tmp_path):
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    ctx = mp.spawn(_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=False)
    while not ctx.join(timeout=600):
        pass
