"""GPU tests of EvolutionStrategy.evaluate / run_generation on envs that live on the GPU (INTEGRATION.md §4).

Twin envs with identical table-driven dynamics -- one numpy (stepped by ppx's host loop: predict_population + numpy +
f64 accumulation), one torch-CUDA (stepped by evaluate) -- with a per-member episode length, observations and rewards that
depend on the action through exact f32 (or f64) arithmetic, a behavior() method, and rewards / behaviours of 1e6 after a
member's episode has ended (the env keeps stepping, as an auto-resetting VecEnv does).  Fitness, lengths and behaviours
must be bit-identical between the two loops."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import es as OE

pytestmark = pytest.mark.gpu

F32 = np.float32
BIG = 1e5                                  # anything above this leaked from after an episode's end


def _tables(N, D0, steps, lengths, seed=0):
    rs = np.random.RandomState(seed)
    return dict(obs=rs.randn(steps + 1, N, D0).astype(F32), rew=rs.randn(steps, N).astype(F32), rew64=rs.randn(steps, N),
                len=np.asarray(lengths, np.int64))


class NumpyTwin:
    """Member i at step t (all members step together from reset): pre = obs[t+1, i] + 0.25 a0, reward = rew[t, i] + hit
    (Box: a0 > 0, Discrete: a == 1), + 1e6 once t+1 > len[i]; done at t+1 == len[i] and every third step after; behavior()
    = (pre_0, t+1 + pre_1 / 2) of the state reached, + 1e6 after the episode; a done env returns the reset obs[0, i]."""

    def __init__(self, tabs, space, f64=False):
        import ppo_exploration_b200 as ppx
        self.tabs, self.space, self.f64 = tabs, space, f64
        _, self.num_envs, D0 = tabs["obs"].shape
        self.observation_space = ppx.Box((D0,))
        self.action_space = ppx.Box((2,)) if space == "box" else ppx.Discrete(3)
        self.actions = []

    def reset(self):
        self.t = 0
        return self.tabs["obs"][0].copy()

    def dyn(self, t, a, idx):
        tb = self.tabs
        a = np.asarray(a)
        a0 = (a[:, 0] if self.space == "box" else a).astype(F32)
        hit = (a0 > 0) if self.space == "box" else (a == 1)
        ln = tb["len"][idx]
        post = t + 1 > ln
        pre = tb["obs"][t + 1, idx] + F32(0.25) * a0[:, None]
        rew = tb["rew64"][t, idx] + hit.astype(np.float64) if self.f64 else tb["rew"][t, idx] + hit.astype(F32)
        rew = np.where(post, rew + (1e6 if self.f64 else F32(1e6)), rew)
        done = (t + 1 >= ln) & ((t + 1 - ln) % 3 == 0)
        bc = np.stack([pre[:, 0].astype(np.float64), (t + 1) + 0.5 * pre[:, 1].astype(np.float64)], 1)
        bc = np.where(post[:, None], bc + 1e6, bc)
        obs = np.where(done[:, None], tb["obs"][0, idx], pre)
        return obs, rew, done, bc

    def step(self, a):
        self.actions.append(np.array(a))
        t, self.t = self.t, self.t + 1
        obs, rew, done, self._bc = self.dyn(t, a, np.arange(self.num_envs))
        return obs, rew, done, []

    def behavior(self):
        return self._bc


class DeviceTwin(NumpyTwin):
    def __init__(self, tabs, space, f64=False):
        super().__init__(tabs, space, f64)
        self.d = {k: torch.as_tensor(v).cuda() for k, v in tabs.items()}

    def reset(self):
        self.t = 0
        return self.d["obs"][0].clone()

    def step(self, a):
        assert a.is_cuda and a.dtype == (torch.float64 if self.space == "box" else torch.int64)
        self.actions.append(a.clone())
        t, self.t = self.t, self.t + 1
        d = self.d
        a0 = (a[:, 0] if self.space == "box" else a).float()
        hit = (a0 > 0) if self.space == "box" else (a == 1)
        ln = d["len"]
        post = t + 1 > ln
        pre = d["obs"][t + 1] + 0.25 * a0[:, None]
        rew = d["rew64"][t] + hit.double() if self.f64 else d["rew"][t] + hit.float()
        rew = torch.where(post, rew + 1e6, rew)
        done = (t + 1 >= ln) & ((t + 1 - ln) % 3 == 0)
        bc = torch.stack([pre[:, 0].double(), (t + 1) + 0.5 * pre[:, 1].double()], 1)
        self._bc = torch.where(post[:, None], bc + 1e6, bc)
        obs = torch.where(done[:, None], d["obs"][0], pre)
        return obs, rew, done, []


def _host_loop(es, pop, env, max_steps, sigma=None):
    """The batched host loop: predict_population on the f64 observations, numpy env, f64 accumulation while running."""
    obs = env.reset()
    N = env.num_envs
    fit, lens, alive, bc = np.zeros(N), np.zeros(N, np.int64), np.ones(N, bool), np.zeros((N, 2))
    for t in range(max_steps):
        out = es.predict_population(pop, torch.as_tensor(obs).cuda().double(), sigma=sigma).cpu().numpy()
        obs, rew, done, _ = env.step(np.where(alive[:, None], out, 0.0))
        b = env.behavior()
        fit[alive] += rew[alive].astype(np.float64)
        lens[alive] += 1
        end = alive & (done | (t == max_steps - 1))
        bc[end] = b[end]
        alive &= ~end
        if not alive.any():
            break
    return fit, lens, bc


def _member_major_discrete(es, pop, env, max_steps):
    """The reference's order for Discrete: member after member, one episode each, one np.random.choice per step
    (EvolutionStrategy.discrete_action on predict_population's logits)."""
    import ppo_exploration_b200 as ppx
    N = env.num_envs
    fit, lens, bc = np.zeros(N), np.zeros(N, np.int64), np.zeros((N, 2))
    acts = np.zeros((max_steps, N), np.int64)
    for i in range(N):
        o = env.tabs["obs"][0, i]
        for t in range(max_steps):
            logits = es.predict_population(pop[i:i + 1], torch.as_tensor(o[None]).cuda().double(), discrete=True)
            a = int(ppx.EvolutionStrategy.discrete_action(logits)[0])
            acts[t, i] = a
            obs, r, d, b = env.dyn(t, np.array([a]), np.array([i]))
            o = obs[0]
            fit[i] += float(r[0])
            lens[i] += 1
            if d[0] or t == max_steps - 1:
                bc[i] = b[0]
                break
    return fit, lens, bc, acts


def _es(hidden, P, seed=5, **kw):
    import ppo_exploration_b200 as ppx
    np.random.seed(seed)
    return ppx.EvolutionStrategy(hidden_sizes=hidden, obs_dim=8, n_actions=kw.pop("n_actions", 2), population_size=P, sigma=0.1,
                                 noise_table_size=1 << 20, **kw)


def _pop(es, table, seed=7):
    if table:
        return es._get_population()
    return np.random.RandomState(seed).randn(es.POPULATION_SIZE, es.D).astype(F32)


def _np(x):
    return x if x is None or isinstance(x, np.ndarray) else x.cpu().numpy()


def _assert_same(dev, host):
    fit, lens, bc = (_np(x) for x in dev)
    assert np.array_equal(lens, host[1]), "episode lengths differ"
    assert np.array_equal(fit, host[0]), f"fitness differs: max |diff| {np.abs(fit - host[0]).max()}"
    assert np.array_equal(bc, host[2]), "behaviour characterisations differ"
    assert fit.max() < BIG and bc.max() < BIG, "a reward or behaviour from after an episode's end leaked"


N, MAXS = 64, 40


@pytest.mark.parametrize("hidden,table,f64", [([64, 64], True, False), ([64, 64], False, True), ([40, 130, 7], True, True),
                                              ([40, 130, 7], False, False)])
def test_box_equals_host_loop(hidden, table, f64):
    lengths = np.random.RandomState(1).randint(1, 31, N)
    tabs = _tables(N, 8, MAXS, lengths, seed=2)
    es = _es(hidden, N)
    pop = _pop(es, table)
    want = _host_loop(es, pop, NumpyTwin(tabs, "box", f64), MAXS)
    got = es.evaluate(DeviceTwin(tabs, "box", f64), pop, max_steps=MAXS)
    _assert_same(got, want)
    assert np.array_equal(_np(got[1]), lengths)


class SmoothEnv:
    """Observations from a table whatever the action, reward = the first action component (f64), one episode of len[i]."""

    def __init__(self, tabs):
        import ppo_exploration_b200 as ppx
        self.d = {k: torch.as_tensor(v).cuda() for k, v in tabs.items()}
        self.num_envs = tabs["obs"].shape[1]
        self.observation_space, self.action_space = ppx.Box((8,)), ppx.Box((2,))

    def reset(self):
        self.t = 0
        return self.d["obs"][0]

    def step(self, a):
        self.t += 1
        return self.d["obs"][self.t], a[:, 0].clone(), self.d["len"] == self.t, []


def test_box_fitness_matches_f64_oracle():
    lengths = np.random.RandomState(3).randint(5, 31, N)
    tabs = _tables(N, 8, MAXS, lengths, seed=4)
    es = _es([64, 64], N)
    pop = _pop(es, True)
    fit = _np(es.evaluate(SmoothEnv(tabs), pop, max_steps=MAXS)[0])
    eps = es.noise_table()[(pop[:, None] + torch.arange(es.D, device=pop.device)[None, :])].cpu().numpy().astype(np.float64)
    theta = es.theta.cpu().numpy()
    cut = np.cumsum([0] + es.layer_sizes)
    for i in range(N):
        w = [(theta[cut[l]:cut[l + 1]] + 0.1 * eps[i, cut[l]:cut[l + 1]]).reshape(es.shapes[l]) for l in range(len(es.shapes))]
        want = sum(OE.predict(w, tabs["obs"][t, i].astype(np.float64))[0, 0] for t in range(lengths[i]))
        np.testing.assert_allclose(fit[i], want, rtol=1e-5, atol=1e-5 * lengths[i])


def _uniforms_member_major(lengths, max_steps, seed):
    """numpy's uniforms in the order the reference consumes them (member-major, one per step) laid out [step, member]."""
    steps = np.minimum(lengths, max_steps)
    np.random.seed(seed)
    u = np.random.random_sample(int(steps.sum()))
    U = np.full((max_steps, len(lengths)), 0.5)
    o = 0
    for i, s in enumerate(steps):
        U[:s, i] = u[o:o + s]
        o += s
    return U


@pytest.mark.parametrize("table", [True, False])
def test_discrete_replays_numpy_choice(table):
    n, maxs = 32, 24
    lengths = np.random.RandomState(8).randint(1, 21, n)
    tabs = _tables(n, 8, maxs, lengths, seed=9)
    es = _es([64, 64], n, n_actions=3)
    pop = _pop(es, table)
    U = _uniforms_member_major(lengths, maxs, seed=11)
    np.random.seed(11)
    want_fit, want_len, want_bc, want_acts = _member_major_discrete(es, pop, NumpyTwin(tabs, "discrete"), maxs)
    env = DeviceTwin(tabs, "discrete")
    got = es.evaluate(env, pop, max_steps=maxs, uniforms=torch.as_tensor(U).cuda())
    _assert_same(got, (want_fit, want_len, want_bc))
    acts = torch.stack(env.actions).cpu().numpy()
    for i in range(n):
        assert np.array_equal(acts[:lengths[i], i], want_acts[:lengths[i], i]), f"member {i}: actions differ"
    assert len(np.unique(acts[0])) == 3, "every action should be drawn"


def test_discrete_philox_is_deterministic_and_rank_independent():
    n, maxs = 32, 24
    lengths = np.random.RandomState(12).randint(1, 21, n)
    tabs = _tables(n, 8, maxs, lengths, seed=13)
    es = _es([64, 64], n, n_actions=3)
    pop = _pop(es, True)
    runs = []
    for _ in range(2):
        env = DeviceTwin(tabs, "discrete")
        out = es.evaluate(env, pop, max_steps=maxs)
        runs.append(([_np(x).copy() for x in out], torch.stack(env.actions).cpu().numpy()))
    for a, b in zip(runs[0][0], runs[1][0]):
        assert np.array_equal(a, b), "the Philox draw is not deterministic"
    assert np.array_equal(runs[0][1], runs[1][1])
    # the second half of the members evaluated on their own (as rank 1 of 2 would): same actions for the same global member
    half = {k: (v[:, n // 2:] if k != "len" else v[n // 2:]) for k, v in tabs.items()}
    env = DeviceTwin(half, "discrete")
    out = es.evaluate(env, pop[n // 2:], max_steps=maxs, member_lo=n // 2)
    acts = torch.stack(env.actions).cpu().numpy()
    full = runs[0][1]
    for i in range(n // 2):
        L_ = lengths[n // 2 + i]
        assert np.array_equal(acts[:L_, i], full[:L_, n // 2 + i])
    assert np.array_equal(_np(out[0]), runs[0][0][0][n // 2:])
    # a new population draw (the draw counter moves on) draws new actions
    es._get_population()
    env = DeviceTwin(tabs, "discrete")
    es.evaluate(env, pop, max_steps=maxs)
    assert not np.array_equal(torch.stack(env.actions).cpu().numpy(), runs[0][1])


class ConstEnv:
    """The same observation for every env at every step, no reward, no end: every draw sees the same logits."""

    def __init__(self, n, obs):
        import ppo_exploration_b200 as ppx
        self.num_envs = n
        self.o = torch.as_tensor(obs, dtype=torch.float32).cuda().expand(n, -1).contiguous()
        self.observation_space, self.action_space = ppx.Box((8,)), ppx.Discrete(3)
        self.actions = []

    def reset(self):
        return self.o

    def step(self, a):
        self.actions.append(a.clone())
        return self.o, torch.zeros(self.num_envs, device="cuda"), torch.zeros(self.num_envs, dtype=torch.bool, device="cuda"), []


def test_discrete_philox_draws_follow_softmax():
    from scipy.stats import chisquare
    n, steps = 4096, 16
    es = _es([16, 16], n, n_actions=3, seed=14)
    es.theta.mul_(0.3)                                         # softmax(logits) ~ (0.25, 0.53, 0.23)
    obs = np.random.RandomState(15).randn(8) * 0.3
    logits = es.predict(obs.astype(F32).astype(np.float64), discrete=True).cpu().numpy()[0]
    p = np.exp(logits) / np.exp(logits).sum()
    assert p.min() > 0.1, p
    env = ConstEnv(n, obs.astype(F32))
    es.evaluate(env, max_steps=steps, sigma=0.0)
    counts = np.bincount(torch.stack(env.actions).cpu().numpy().ravel(), minlength=3)
    assert counts.sum() == n * steps
    assert chisquare(counts, p * n * steps).pvalue > 1e-3, (counts, p * n * steps)


def test_masking_check_every_and_truncation():
    lengths = np.random.RandomState(16).randint(1, 31, N)
    tabs = _tables(N, 8, 200, lengths, seed=17)
    es = _es([64, 64], N)
    pop = _pop(es, True)
    ref = None
    for max_steps in (40, 200):
        for check_every in (1, 8, 64):
            out = [_np(x).copy() for x in es.evaluate(DeviceTwin(tabs, "box"), pop, max_steps=max_steps, check_every=check_every)]
            assert out[0].max() < BIG and out[2].max() < BIG
            if ref is None:
                ref = out
                _assert_same(out, _host_loop(es, pop, NumpyTwin(tabs, "box"), max_steps))
            for a, b in zip(out, ref):
                assert np.array_equal(a, b), (max_steps, check_every)
            assert es.last_eval_steps < max_steps or max_steps == 40
    # truncation: members still running at max_steps keep the sum so far and the behaviour of that step
    cap = 10
    out = es.evaluate(DeviceTwin(tabs, "box"), pop, max_steps=cap, check_every=4)
    _assert_same(out, _host_loop(es, pop, NumpyTwin(tabs, "box"), cap))
    assert np.array_equal(_np(out[1]), np.minimum(lengths, cap))
    assert es.last_eval_steps == cap
    assert (lengths > cap).any()


def test_numpy_env_is_rejected():
    tabs = _tables(8, 8, 4, np.full(8, 2), seed=18)
    es = _es([16, 16], 8)
    with pytest.raises(TypeError, match="CUDA tensor"):
        es.evaluate(NumpyTwin(tabs, "box"), _pop(es, True), max_steps=4)


def test_device_eval_has_no_sync_and_two_launches_per_step():
    from ppo_exploration_b200 import _lib as L
    n = 2048
    lengths = np.random.RandomState(19).randint(5, 33, n)
    tabs = _tables(n, 8, 48, lengths, seed=20)
    for space, nact in (("box", 2), ("discrete", 3)):
        es = _es([64, 64], n, n_actions=nact)
        pop = _pop(es, True)
        es.evaluate(DeviceTwin(tabs, space), pop, max_steps=48)     # warm-up: buffers, pinned memory
        torch.cuda.synchronize()
        env = DeviceTwin(tabs, space)
        torch.cuda.set_sync_debug_mode("error")
        try:
            n0 = L.launch_count()
            es.evaluate(env, pop, max_steps=48)
            n1 = L.launch_count()
        finally:
            torch.cuda.set_sync_debug_mode(0)
        assert n1 - n0 == 2 * es.last_eval_steps, (n1 - n0, es.last_eval_steps)
        assert 32 <= es.last_eval_steps <= 48


def test_run_generation_equals_ask_host_loop_tell():
    """Three generations with the novelty mix: run_generation on the device twin against ask -> the host loop -> tell."""
    import ppo_exploration_b200 as ppx
    n, maxs = 64, 32
    lengths = np.random.RandomState(21).randint(1, 31, n)
    tabs = _tables(n, 8, maxs, lengths, seed=22)
    arch = torch.as_tensor(np.random.RandomState(23).randn(40, 2)).cuda()
    qs = torch.as_tensor(np.random.RandomState(24).randn(2, 2)).cuda()

    def make():
        np.random.seed(25)
        return ppx.EvolutionStrategy(hidden_sizes=[64, 64], obs_dim=8, n_actions=2, population_size=n, sigma=0.1,
                                     noise_table_size=1 << 20, noise_seed=3)
    a, b = make(), make()
    fb = torch.zeros(n, dtype=torch.float64, device="cuda")
    for g in range(3):
        fit, lens, bc = a.run_generation(DeviceTwin(tabs, "box"), max_steps=maxs, archive=arch, queries=qs)
        pop, _, _ = b.ask(arch, qs)
        want = _host_loop(b, pop, NumpyTwin(tabs, "box"), maxs)
        fb.copy_(torch.as_tensor(want[0]))
        b.tell(fb)
        _assert_same((fit, lens, bc), want)
        assert torch.equal(a.theta, b.theta), f"generation {g}: theta differs"
        assert a.learning_rate == b.learning_rate


# ---------------------------------------------------------------- two GPUs
def _worker(rank, world, port):
    import torch.distributed as dist
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    sys.path.insert(0, os.path.join(root, "tests"))
    from test_gpu_sharded import _single
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank),
                      LOCAL_WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", device_id=dev, rank=rank, world_size=world)
    import ppo_exploration_b200 as ppx
    n, maxs = 32, 24                                           # members per rank
    P = n * world
    lengths = np.random.RandomState(31).randint(1, 21, P)
    tabs = _tables(P, 8, maxs, lengths, seed=32)
    sl = slice(rank * n, (rank + 1) * n)
    mine = {k: (v[:, sl] if k != "len" else v[sl]) for k, v in tabs.items()}

    def make():
        np.random.seed(33)
        return ppx.EvolutionStrategy(hidden_sizes=[64, 64], obs_dim=8, n_actions=3, population_size=P, sigma=0.1, device=dev,
                                     noise_table_size=1 << 20, noise_seed=4)
    sharded, union, single = make(), make(), make()
    fb = torch.zeros(n, dtype=torch.float64, device=dev)
    for g in range(3):
        fit, _, _ = sharded.run_generation(DeviceTwin(mine, "discrete"), max_steps=maxs)
        gathered = sharded.gather_fitness(fit).clone()
        union.ask()
        with _single():                                        # one GPU evaluating the union env
            fit_u = union.evaluate(DeviceTwin(tabs, "discrete"), max_steps=maxs)[0].clone()
            single.run_generation(DeviceTwin(tabs, "discrete"), max_steps=maxs)
        fb.copy_(fit_u[sl])
        union.tell(fb)
        torch.cuda.synchronize()
        assert torch.equal(gathered, fit_u), f"generation {g}: gathered fitness differs from one GPU's"
        assert torch.equal(sharded.theta, union.theta), f"generation {g}: theta differs"
        np.testing.assert_allclose(sharded.theta.cpu().numpy(), single.theta.cpu().numpy(), rtol=1e-12, atol=1e-14)
    allt = [torch.empty_like(sharded.theta) for _ in range(world)]
    dist.all_gather(allt, sharded.theta)
    assert all(torch.equal(allt[0], x) for x in allt), "ES replicas diverged"
    dist.barrier()
    torch.cuda.synchronize()
    os._exit(0)


def test_sharded_evaluation_equals_single_gpu():
    import torch.multiprocessing as mp
    from test_gpu_sharded import _free_port
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    ctx = mp.spawn(_worker, args=(2, _free_port()), nprocs=2, join=False)
    while not ctx.join(timeout=600):
        pass
