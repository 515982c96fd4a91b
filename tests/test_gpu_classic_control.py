"""GPU tests of the classic-control envs (classic_control.cu, `ppx.ClassicControlVecEnv`) and of the device-side episode
statistics: dynamics teacher-forced against the numpy restatement in oracle/classic_control.py, time limits, reset draws,
env offsets, the episode monitor, learner parity between the host loop (over `ToNumpy`) and the device path, VecNormalize
over an env on the GPU, launch counts without syncs, ES evaluation, and a seeded learning smoke run."""
import numpy as np
import pytest
import torch

from oracle import classic_control as OC

pytestmark = pytest.mark.gpu

ENV_IDS = list(OC.SPECS)


def _ppx():
    import ppo_exploration_b200 as ppx
    return ppx


def _random_actions(env_id, rs, N):
    kind = OC.SPECS[env_id]["action"]
    if kind[0] == "discrete":
        return rs.randint(0, kind[1], size=N).astype(np.int64)
    return (rs.randn(N, 1) * 2.0 * kind[2]).astype(np.float64)       # often outside the action bounds


def _crafted_states(env_id, rs, n):
    """States at the edges the dynamics treat specially: walls and clips, the |theta| threshold, angles far below -pi."""
    if env_id == "CartPole-v1":
        return np.stack([rs.uniform(-2.45, 2.45, n), rs.uniform(-3, 3, n), OC.THETA_THRESHOLD * rs.uniform(-1.1, 1.1, n),
                         rs.uniform(-3, 3, n)], axis=1)
    if env_id == "Pendulum-v0":
        return np.stack([rs.uniform(-30, 30, n), rs.uniform(-8, 8, n)], axis=1)
    p = np.where(rs.rand(n) < 0.3, -1.2, rs.uniform(-1.2, 0.6, n))
    p = np.where(rs.rand(n) < 0.2, rs.uniform(0.4, 0.6, n), p)
    v = np.where(rs.rand(n) < 0.3, rs.choice([-0.07, 0.07], n) * rs.uniform(0.9, 1.0, n), rs.uniform(-0.07, 0.07, n))
    return np.stack([p, v], axis=1)


def _near_threshold(env_id, s):
    """Oracle states within 1e-12 of a termination threshold (where CUDA's cos / sin may legitimately flip the done)."""
    e = 1e-12
    if env_id == "CartPole-v1":
        return (np.abs(np.abs(s[:, 0]) - 2.4) < e) | (np.abs(np.abs(s[:, 2]) - OC.THETA_THRESHOLD) < e)
    if env_id == "Pendulum-v0":
        return np.zeros(len(s), bool)
    goal = 0.5 if env_id == "MountainCar-v0" else 0.45
    return (np.abs(s[:, 0] - goal) < e) | (np.abs(s[:, 1]) < e)


@pytest.mark.parametrize("N", [1, 1000])
@pytest.mark.parametrize("env_id", ENV_IDS)
def test_dynamics_teacher_forced(env_id, N):
    """Every step: the device state is copied back, the oracle steps it with the same actions, and the pre-reset state,
    reward, done, observation and the monitor's episode returns are compared.  Every 7th step a quarter of the envs (at
    least one) is set to a crafted edge state first."""
    ppx = _ppx()
    rs = np.random.RandomState(11)
    spec = OC.SPECS[env_id]
    env = ppx.ClassicControlVecEnv(env_id, N, seed=3)
    env.reset()
    elapsed = np.zeros(N, np.int64)
    ret = np.zeros(N)
    length = np.zeros(N, np.int64)
    near, episodes = 0, 0
    for t in range(600):
        if t % 7 == 0:
            k = max(1, N // 4)
            st = env.state.cpu().numpy().T.copy()
            st[:k] = _crafted_states(env_id, rs, k)
            env.state.copy_(torch.as_tensor(st.T.copy()))
        s0 = env.state.cpu().numpy().T.copy()
        a = _random_actions(env_id, rs, N)
        obs, rew, done, infos = env.step(torch.as_tensor(a).cuda())
        assert infos == []
        want, r64, term = OC.step(env_id, s0, a)
        got = env.behavior().cpu().numpy()
        err = np.abs(got - want) / (1 + np.abs(want))
        assert err.max() <= 1e-13, f"step {t}: state differs by {err.max():.3g} (relative)"
        r32 = r64.astype(np.float32)
        rew = rew.cpu().numpy()
        assert np.all(np.abs(rew - r32) <= np.spacing(np.abs(r32))), f"step {t}: rewards differ"
        elapsed += 1
        want_done = term | (elapsed >= spec["limit"])
        done = done.cpu().numpy().astype(bool)
        bad = done != want_done
        nb = _near_threshold(env_id, want)
        assert not np.any(bad & ~nb), f"step {t}: dones differ away from a threshold"
        near += int(np.sum(bad))
        ret = ret + r64
        length += 1
        if done.any():
            ep_r, ep_l = (x.cpu().numpy()[done] for x in env.episode_stats())
            assert np.array_equal(ep_l, length[done])
            assert np.all(np.abs(ep_r - ret[done]) <= 1e-12 * (1 + np.abs(ret[done]))), "monitor returns differ"
            episodes += int(done.sum())
            ret[done], length[done], elapsed[done] = 0.0, 0, 0
        s1 = env.state.cpu().numpy().T
        assert np.array_equal(s1[~done], got[~done]), "an env that did not finish changed state after the step"
        want_obs = OC.observation(env_id, s1)
        o = obs.cpu().numpy()
        if env_id == "Pendulum-v0":
            assert np.abs(o - want_obs).max() <= 1e-6
        else:
            assert np.array_equal(o, want_obs)
    assert near <= max(1, N // 100), f"{near} dones differ next to a threshold"
    if N > 1:
        assert episodes > 0


@pytest.mark.parametrize("env_id", ENV_IDS)
def test_time_limit_resets_and_counters(env_id):
    """Held at a state that never terminates, every env reports done exactly at the time limit; the episode counter
    advances and the next episode again lasts the full limit."""
    ppx = _ppx()
    limit = OC.SPECS[env_id]["limit"]
    N = 300
    env = ppx.ClassicControlVecEnv(env_id, N, seed=1)
    env.reset()
    hold = {"CartPole-v1": [0.0, 0.0, 0.0, 0.0], "Pendulum-v0": [0.5, 0.0]}.get(env_id, [-0.5, 0.0])
    a = torch.as_tensor(_random_actions(env_id, np.random.RandomState(0), N)).cuda()
    if env_id == "MountainCarContinuous-v0":
        a.zero_()
    for t in range(1, 2 * limit + 1):
        env.state.copy_(torch.tensor(hold, dtype=torch.float64).view(-1, 1).expand(-1, N))
        _, _, done, _ = env.step(a)
        d = done.cpu().numpy()
        assert np.all(d == (1 if t % limit == 0 else 0)), f"step {t}: done flags wrong"
        if t % limit == 0:
            assert np.all(env.episode_stats()[1].cpu().numpy() == limit)
            assert np.all(env._episode.cpu().numpy() == 1 + t // limit)
            assert np.all(env._elapsed.cpu().numpy() == 0)


@pytest.mark.parametrize("env_id", ENV_IDS)
def test_reset_draws_uniform_deterministic_and_offset_exact(env_id):
    from scipy import stats
    ppx = _ppx()
    N = 20000
    env = ppx.ClassicControlVecEnv(env_id, N, seed=7)
    env.reset()
    s = env.state.cpu().numpy()
    for k, rng in enumerate(OC.RESET_RANGES[env_id]):
        if isinstance(rng, tuple):
            lo, hi = rng
            assert lo <= s[k].min() and s[k].max() < hi
            assert stats.kstest(s[k], "uniform", args=(lo, hi - lo)).pvalue > 1e-3, f"component {k} is not uniform"
        else:
            assert np.all(s[k] == rng)
    env.reset()                                                   # the second episode draws anew
    assert not np.array_equal(env.state.cpu().numpy(), s)
    again = ppx.ClassicControlVecEnv(env_id, N, seed=7)
    again.reset()
    assert np.array_equal(again.state.cpu().numpy(), s), "reset draws are not deterministic"
    other = ppx.ClassicControlVecEnv(env_id, N, seed=8)
    other.reset()
    assert not np.array_equal(other.state.cpu().numpy(), s)
    # rows [k, k + n) of a larger env, bit for bit, over several episodes
    big_n, n, k = 96, 40, 29
    big = ppx.ClassicControlVecEnv(env_id, big_n, seed=5)
    small = ppx.ClassicControlVecEnv(env_id, n, seed=5, env_offset=k)
    big.reset()
    small.reset()
    rs = np.random.RandomState(2)
    for _ in range(2 * OC.SPECS[env_id]["limit"] + 50):
        a = _random_actions(env_id, rs, big_n)
        ob, rb, db, _ = big.step(torch.as_tensor(a).cuda())
        os_, rsm, ds, _ = small.step(torch.as_tensor(a[k:k + n]).cuda())
        assert torch.equal(ob[k:k + n], os_) and torch.equal(rb[k:k + n], rsm) and torch.equal(db[k:k + n], ds)
    assert torch.equal(big.state[:, k:k + n], small.state)
    assert int(small._episode.min()) >= 3, "too few episodes"


def test_episode_monitor_over_a_table_env_is_exact():
    ppx = _ppx()
    rs = np.random.RandomState(4)
    T, N = 200, 333
    rew = rs.randn(T, N).astype(np.float32)
    done = rs.rand(T, N) < 0.05

    class Table:
        num_envs = N
        observation_space, action_space = None, None

        def __init__(self):
            self.r, self.d = torch.as_tensor(rew).cuda(), torch.as_tensor(done).cuda()

        def reset(self):
            self.t = 0
            return torch.zeros(N, 1, device="cuda")

        def step(self, a):
            self.t += 1
            return torch.zeros(N, 1, device="cuda"), self.r[self.t - 1], self.d[self.t - 1], []

    m = ppx.EpisodeMonitor(Table())
    m.reset()
    acc, ln = np.zeros(N), np.zeros(N, np.int64)
    for t in range(T):
        m.step(None)
        acc += rew[t].astype(np.float64)
        ln += 1
        r, l = (x.cpu().numpy() for x in m.episode_stats())
        assert np.array_equal(r[done[t]], acc[done[t]]) and np.array_equal(l[done[t]], ln[done[t]])
        acc[done[t]], ln[done[t]] = 0.0, 0


# ---------------------------------------------------------------- learners
FIELDS = ("observations", "actions", "rewards", "int_rewards", "values", "returns", "action_log_probs", "masks", "advantages",
          "int_values", "int_returns", "int_advantages")
LEARNERS = {
    "ppo": ("PPO", dict(hidden_size=64)),
    "ppo_simhash": ("PPO", dict(hidden_size=64, sim_hash=True, hash_bits=64)),
    "rnd": ("PPO_RND", dict(hidden_size=64, int_hidden_size=32, rnd_start=40)),
    "icm": ("PPO_ICM", dict(hidden_size=64, int_hidden_size=32)),
}
BASE = dict(nstep=32, batch_size=128, n_epochs=2)


def _run(cls, env, kw, iters=3, seed=3):
    np.random.seed(seed)
    torch.manual_seed(seed)
    m = cls(env=env, **dict(BASE, **kw))
    rolls = []
    for _ in range(iters):
        m.collect_samples()
        rolls.append({k: getattr(m.rollout, k).clone() for k in FIELDS if hasattr(m.rollout, k)})
        m.train()
    torch.cuda.synchronize()
    banks = [m.policy.bank.flat.clone()] + [getattr(m, x).bank.flat.clone() for x in ("rnd", "intrinsic_module") if hasattr(m, x)]
    return dict(m=m, rolls=rolls, banks=banks, episodes=m.num_episodes, infos=list(m.ep_info_buffer))


def _assert_same(a, b):
    for i, (ra, rb) in enumerate(zip(a["rolls"], b["rolls"])):
        for k in ra:
            assert torch.equal(ra[k], rb[k]), f"iteration {i}: rollout.{k} differs"
    for wa, wb in zip(a["banks"], b["banks"]):
        assert torch.equal(wa, wb), "weights differ"
    assert a["episodes"] == b["episodes"] > 0
    assert a["infos"] == b["infos"] and len(a["infos"]) > 0, "ep_info_buffer differs"


@pytest.mark.parametrize("case", list(LEARNERS))
def test_learner_device_path_equals_host_loop(case):
    ppx = _ppx()
    algo, kw = LEARNERS[case]
    cls = getattr(ppx, algo)
    host = _run(cls, ppx.ToNumpy(ppx.ClassicControlVecEnv("CartPole-v1", 16, seed=9)), kw)
    dev = _run(cls, ppx.ClassicControlVecEnv("CartPole-v1", 16, seed=9), kw)
    assert host["m"].device_env is False and dev["m"].device_env is True
    _assert_same(host, dev)
    assert all(set(e) == {"r", "l"} for e in dev["infos"])


@pytest.mark.parametrize("case", ["ppo", "rnd"])
def test_learn_stops_at_the_same_iteration(case):
    ppx = _ppx()
    algo, kw = LEARNERS[case]
    cls = getattr(ppx, algo)
    out = []
    for env in (ppx.ToNumpy(ppx.ClassicControlVecEnv("CartPole-v1", 16, seed=2)), ppx.ClassicControlVecEnv("CartPole-v1", 16, seed=2)):
        np.random.seed(0)
        torch.manual_seed(0)
        m = cls(env=env, **dict(BASE, **kw))
        m.learn(total_timesteps=16 * 32 * 40, log_interval=1, reward_target=25)
        out.append((m.num_timesteps, m.num_episodes, list(m.ep_info_buffer), m.policy.bank.flat.clone()))
    assert out[0][:3] == out[1][:3]
    assert out[0][0] < 16 * 32 * 40, "the reward target was not reached"
    assert torch.equal(out[0][3], out[1][3])


@pytest.mark.parametrize("norm_reward", [True, False])
def test_vecnormalize_over_a_gpu_env_equals_the_host_inner_env(norm_reward):
    ppx = _ppx()

    def dev_env():
        if norm_reward:
            return ppx.make_env("MountainCarContinuous-v0", 16, seed=4, normalize=True)
        return ppx.VecNormalize(ppx.ClassicControlVecEnv("MountainCarContinuous-v0", 16, seed=4), norm_reward=False)

    host_env = ppx.VecNormalize(ppx.ToNumpy(ppx.ClassicControlVecEnv("MountainCarContinuous-v0", 16, seed=4)),
                                norm_reward=norm_reward)
    kw = dict(hidden_size=64, sim_hash=True, hash_bits=64)
    host = _run(ppx.PPO, host_env, kw, iters=4)
    env = dev_env()
    dev = _run(ppx.PPO, env, kw, iters=4)
    for i, (ra, rb) in enumerate(zip(host["rolls"], dev["rolls"])):
        for k in ra:
            assert torch.equal(ra[k], rb[k]), f"iteration {i}: rollout.{k} differs"
    for name in ("obs_rms", "ret_rms"):
        for f in ("mean_dev", "var_dev", "count_dev"):
            assert torch.equal(getattr(getattr(host_env, name), f), getattr(getattr(env, name), f)), f"{name}.{f} differs"
    assert torch.equal(host_env.ret, env.ret)
    assert host["infos"] == dev["infos"] and host["episodes"] == dev["episodes"]


def test_device_collect_on_a_builtin_env_has_no_sync_and_five_launches_per_step():
    """2048 envs, MountainCarContinuous-v0, h = 64, SimHash k = 64: per step forward + act_record + env step +
    record_step + episode log."""
    ppx = _ppx()
    from ppo_exploration_b200 import _lib as L
    n, t = 2048, 8
    np.random.seed(0)
    torch.manual_seed(0)
    env = ppx.ClassicControlVecEnv("MountainCarContinuous-v0", n, seed=0)
    m = ppx.PPO(env=env, nstep=t, batch_size=4096, n_epochs=1, hidden_size=64, sim_hash=True, hash_bits=64)
    assert m.device_env and m.policy.mlp._fused_args()["tc"]
    m.collect_samples()
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        n0 = L.launch_count()
        m.collect_samples()
        n1 = L.launch_count()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    ro = m.rollout
    ro.sim_hash_recorded()
    ro.compute_returns_and_advantages(ro.values[-1], ro.masks[-1])
    m._episode_log_end()
    n2 = L.launch_count()
    assert (n1 - n0) - (n2 - n1) == 5 * t, (n1 - n0, n2 - n1)


class _FirstEpisode:
    """Latches each env's first finished episode: the monitor's return / length and the pre-reset state."""

    def __init__(self, env):
        self.env, self.num_envs = env, env.num_envs
        self.observation_space, self.action_space = env.observation_space, env.action_space

    def reset(self):
        N = self.num_envs
        self.seen = torch.zeros(N, dtype=torch.bool, device="cuda")
        self.ret = torch.zeros(N, dtype=torch.float64, device="cuda")
        self.len = torch.zeros(N, dtype=torch.int64, device="cuda")
        self.bc = torch.zeros(N, 2, dtype=torch.float64, device="cuda")
        return self.env.reset()

    def step(self, a):
        out = self.env.step(a)
        new = out[2].bool() & ~self.seen
        r, l = self.env.episode_stats()
        self.ret = torch.where(new, r, self.ret)
        self.len = torch.where(new, l, self.len)
        self.bc = torch.where(new[:, None], self.env.behavior(), self.bc)
        self.seen |= new
        return out

    def behavior(self):
        return self.env.behavior()


def test_es_evaluate_on_mountain_car_continuous():
    ppx = _ppx()
    P = 512
    np.random.seed(5)
    es = ppx.EvolutionStrategy(hidden_sizes=(16, 16), obs_dim=2, n_actions=1, population_size=P, sigma=0.5,
                               noise_table_size=1 << 20)
    pop = es._get_population()
    env = _FirstEpisode(ppx.ClassicControlVecEnv("MountainCarContinuous-v0", P, seed=1, reward_dtype=torch.float64))
    fit, lens, bc = (x.clone() for x in es.evaluate(env, pop, max_steps=999))
    assert bool(env.seen.all())
    assert torch.equal(fit, env.ret), "fitness differs from the monitor's first-episode return"
    assert torch.equal(lens, env.len) and int(lens.max()) <= 999
    assert torch.equal(bc, env.bc), "behaviour differs from the pre-reset state of the terminating step"
    assert int((lens < 999).sum()) > 0, "no member reached the goal: the test does not exercise termination"
    halves = []
    for lo in (0, P // 2):
        e = ppx.ClassicControlVecEnv("MountainCarContinuous-v0", P // 2, seed=1, env_offset=lo, reward_dtype=torch.float64)
        halves.append(es.evaluate(e, pop[lo:lo + P // 2], max_steps=999, member_lo=lo)[0].clone())
    assert torch.equal(torch.cat(halves), fit)


SMOKE_BOUND = 300.0      # measured 493.7 on a B200 (DESIGN.md §3.13)


def test_ppo_learns_cartpole_on_the_device_path():
    ppx = _ppx()
    np.random.seed(0)
    torch.manual_seed(0)
    env = ppx.make_env("CartPole-v1", 8, seed=0)
    m = ppx.PPO(env=env, nstep=256, batch_size=64, n_epochs=10, hidden_size=64, lr=3e-4, ent_coef=0.0, max_grad_norm=0.5)
    m.learn(total_timesteps=60_000, log_interval=None)
    got = float(np.mean([e["r"] for e in m.ep_info_buffer]))
    print(f"CartPole-v1 device-path PPO: ep_rew_mean {got:.1f} after {m.num_timesteps} steps")
    assert got > SMOKE_BOUND
