"""EvolutionStrategy.run: the ES-NSRA loop over a meta-population on envs that live on the GPU (DESIGN.md §3.15).

CPU tests pin ppx's novelty-weight adaptation rule and the f64 oracle loop (oracle/es_nsra.py).  GPU tests check the brain
forward `ppx_es_act_rows` against `ppx_es_act` row by row, run() against the same loop composed on the host from public
pieces (novelty_batch, pick_brain, ask, evaluate, tell, one evaluate(sigma=0) per brain, the oracle rule), the f64 oracle
teacher-forced with the device's fitness vectors and behaviours, the one read per generation, the graph keyed on
novelty_param, reward_target, the CSV log, resume, the sharded run and a CartPole learning run."""
import contextlib
import csv
import ctypes as C
import glob
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from oracle import es as OE                                             # noqa: E402
from oracle import es_nsra as ON                                        # noqa: E402

gpu = pytest.mark.gpu
F32 = np.float32


# ---------------------------------------------------------------- CPU: the adaptation rule and the oracle loop
def test_nsr_adapt_rule():
    rule = dict(nsr_plateu=1.5, nsr_range=(0, 1), nsr_update=0.05)
    inf = -np.inf
    # a history shorter than 5 (or between windows) changes nothing
    for fb in ([], [1.0], [1.0, 2, 3, 4], [1.0] * 6, [1.0] * 9):
        assert ON.nsr_adapt(0.5, fb, 3.0, **rule) == (0.5, 3.0)
    # first window: any reward beats B = -inf -> improvement, w decreases
    assert ON.nsr_adapt(0.5, [1.0, 2, 3, 4, 5], inf, **rule) == (0.5 - 0.05, 5.0)
    # improvement: R = 9 > B + 1.5
    assert ON.nsr_adapt(0.5, [0, 0, 0, 0, 0, 1, 9, 2, 3, 4], 7.0, **rule) == (0.5 - 0.05, 9.0)
    # plateau: R = 8 <= 7 + 1.5
    assert ON.nsr_adapt(0.5, [1.0, 8, 2, 3, 4], 7.0, **rule) == (0.5 + 0.05, 8.0)
    # margin exactly nsr_plateu: a plateau
    assert ON.nsr_adapt(0.5, [8.5, 0, 0, 0, 0], 7.0, **rule) == (0.5 + 0.05, 8.5)
    # R below B: plateau, B stays
    assert ON.nsr_adapt(0.5, [1.0] * 5, 7.0, **rule) == (0.5 + 0.05, 7.0)
    # clamping at both ends of nsr_range
    assert ON.nsr_adapt(0.02, [9.0] * 5, 0.0, **rule) == (0.0, 9.0)
    assert ON.nsr_adapt(0.98, [1.0] * 5, 7.0, **rule) == (1.0, 7.0)
    assert ON.nsr_adapt(0.3, [1.0] * 5, 7.0, nsr_plateu=1.5, nsr_range=(0.1, 0.32), nsr_update=0.05) == (0.32, 7.0)


class _NumpyTableEnv:
    """Table-driven episodes: at step t the env shows obs[t]; reward = obs[t, 0] * (2 a0 - 1) with a0 = tanh(logit 0);
    episode length len[i]; the behaviour is the (reward sum, last observation component 1)."""

    def __init__(self, obs, lengths):
        self.obs, self.len = obs, lengths

    def episode(self, weights, i):
        f = 0.0
        for t in range(self.len[i]):
            a = OE.predict(weights, self.obs[t, i])[0, 0]
            f += float(self.obs[t, i, 0]) * (2 * a - 1)
        return f, np.array([f, float(self.obs[self.len[i] - 1, i, 1])])


def test_oracle_loop_composes_the_pinned_pieces():
    rs = np.random.RandomState(0)
    shapes = OE.layer_shapes(3, [8], 1)
    D_ = sum(a * b for a, b in shapes)
    P, M, G, sigma = 16, 3, 12, 0.1
    pop_env = _NumpyTableEnv(rs.randn(12, P, 3), rs.randint(3, 12, P))
    brain_env = _NumpyTableEnv(rs.randn(12, M, 3), rs.randint(3, 12, M))
    cut = np.cumsum([0] + [a * b for a, b in shapes])
    split = lambda v: [v[cut[l]:cut[l + 1]].reshape(shapes[l]) for l in range(len(shapes))]
    eps = [rs.randn(P, D_) for _ in range(G)]

    def brains_of(g, thetas):
        out = [brain_env.episode(split(thetas[m]), m) for m in range(M)]
        return np.array([o[1] for o in out]), np.array([o[0] for o in out])

    def fitness_of(g, theta):
        return np.array([pop_env.episode(split(theta + sigma * eps[g][i]), i)[0] for i in range(P)])

    thetas0 = rs.randn(M, D_)
    kw = dict(shapes=shapes, sigma=sigma, decay=0.999, novelty_param=0.5, nsr_plateu=0.2, nsr_range=(0, 1), nsr_update=0.05,
              eps_of=lambda g: eps[g], fitness_of=fitness_of, brains_of=brains_of)
    np.random.seed(1)
    out = ON.nsra_run(thetas0, 0.05, G, **kw)
    # recompose by hand from the pinned pieces
    np.random.seed(1)
    thetas, lr, w, best, fb = thetas0.copy(), 0.05, 0.5, -np.inf, []
    bc, f = brains_of(-1, thetas)
    archive = list(bc)
    for g in range(G):
        nov = [float(OE.novelty(np.array(archive), bc[m])) for m in range(M)]
        b = int(np.random.choice(list(range(M)), p=OE.novelty_distribution(nov)))
        assert b == out["picks"][g]
        new, lr = OE.update_weights(split(thetas[b]), fitness_of(g, thetas[b]), [split(e) for e in eps[g]], lr, sigma, w,
                                    0.999, novelty=nov[b])
        thetas[b] = np.concatenate([x.ravel() for x in new])
        bc, f = brains_of(g, thetas)
        archive.append(bc[b])
        fb.append(f[b])
        w, best = ON.nsr_adapt(w, fb, best, 0.2, (0, 1), 0.05)
        assert w == out["w"][g]
    assert np.array_equal(thetas, out["thetas"]) and lr == out["lr"]
    assert np.array_equal(np.array(archive), out["archive"]) and out["archive"].shape == (M + G, 2)
    assert len(set(out["picks"])) > 1
    # reward_target stops after the first generation whose f_b exceeds it
    np.random.seed(1)
    k = int(np.argmax(out["fb"][:6]))
    tgt = np.nextafter(out["fb"][k], -np.inf)
    stop = next(j for j, v in enumerate(out["fb"]) if v > tgt)
    np.random.seed(1)
    assert len(ON.nsra_run(thetas0, 0.05, G, reward_target=tgt, **kw)["picks"]) == stop + 1


# ---------------------------------------------------------------- GPU helpers
def _ppx():
    import ppo_exploration_b200 as ppx
    return ppx


@contextlib.contextmanager
def _rng(holder):
    """Run the block on numpy's global RNG state kept in holder[0] (two loops drawing from 'the' global RNG side by side)."""
    saved = np.random.get_state()
    np.random.set_state(holder[0])
    try:
        yield
    finally:
        holder[0] = np.random.get_state()
        np.random.set_state(saved)


def _make(P, seed=25, hidden=(64, 64), n_actions=2, **kw):
    np.random.seed(seed)
    return _ppx().EvolutionStrategy(env_id="table", hidden_sizes=hidden, obs_dim=8, n_actions=n_actions, population_size=P,
                                    sigma=0.1, learning_rate=0.05, noise_table_size=1 << 20, noise_seed=3, **kw)


def _rows(tabs, sl):
    return {k: (v[:, sl] if k != "len" else v[sl]) for k, v in tabs.items()}


def _csv_rows(root, env_id="table"):
    rows = []
    for p in sorted(glob.glob(os.path.join(root, "logs", "ES", env_id, "run-*.csv"))):
        with open(p) as fh:
            rows += list(csv.DictReader(fh))
    return rows


class _Composition:
    """run() composed on the host from public pieces, one generation per step()."""

    def __init__(self, es, tabs_pop, tabs_brain, M, maxs, rule):
        from test_gpu_es_device_eval import DeviceTwin
        self.es, self.M, self.maxs, self.rule = es, M, maxs, rule
        self.pop_env = lambda: DeviceTwin(tabs_pop, "box")
        self.brain_envs = [DeviceTwin(_rows(tabs_brain, slice(m, m + 1)), "box") for m in range(M)]
        self.thetas = [es.theta.clone()] + [torch.as_tensor(np.concatenate([np.random.randn(*s).ravel() for s in es.shapes]))
                                            .cuda() for _ in range(M - 1)]
        self.bc, self.f = self.brains()
        self.archive = self.bc.clone()
        self.w, self.best, self.fb, self.picks, self.ws = es.novelty_param, -np.inf, [], [], []
        self.rec = dict(bc=[self.bc.cpu().numpy()], f=[self.f.cpu().numpy()], eps=[], fit=[], rows=[])

    def brains(self):
        es, keep = self.es, self.es.theta.clone()
        bcs, fs = [], []
        for m in range(self.M):
            es.theta.copy_(self.thetas[m])
            f, _, bc = es.evaluate(self.brain_envs[m], torch.zeros(1, dtype=torch.int64, device="cuda"), max_steps=self.maxs,
                                   sigma=0.0)
            bcs.append(bc.clone())
            fs.append(f.clone())
        es.theta.copy_(keep)
        return torch.cat(bcs), torch.cat(fs)

    def step(self):
        es = self.es
        nov = es.novelty_batch(self.archive, self.bc)[1]
        b, _ = es.pick_brain([float(x) for x in nov.cpu().numpy()])
        es.novelty_param = self.w
        es.theta.copy_(self.thetas[b])
        pop, _, _ = es.ask(self.archive, self.bc)
        fit = es.evaluate(self.pop_env(), max_steps=self.maxs)[0]
        es.tell(fit, brain=b)
        self.thetas[b] = es.theta.clone()
        self.rec["eps"].append(es.noise_table()[pop[:, None] + torch.arange(es.D, device="cuda")[None]].double().cpu().numpy())
        self.rec["fit"].append(fit.cpu().numpy().copy())
        self.bc, self.f = self.brains()
        self.rec["bc"].append(self.bc.cpu().numpy())
        self.rec["f"].append(self.f.cpu().numpy())
        self.archive = torch.cat([self.archive, self.bc[b:b + 1]])
        fb = float(self.f[b])
        self.fb.append(fb)
        self.picks.append(b)
        self.rec["rows"].append(dict(reward=fb, brain=b, novelty_param=self.w, learning_rate=es.learning_rate,
                                     fitness_mean=float(fit.mean()), fitness_max=float(fit.max()),
                                     archive_size=self.archive.shape[0]))
        self.w, self.best = ON.nsr_adapt(self.w, self.fb, self.best, **self.rule)
        self.ws.append(self.w)
        return fb


def _tables_for(P, M, maxs, seed):
    from test_gpu_es_device_eval import _tables
    rs = np.random.RandomState(seed)
    return _tables(P, 8, maxs, rs.randint(1, maxs, P), seed=seed + 1), _tables(M, 8, maxs, rs.randint(4, maxs, M), seed=seed + 2)


RULE = dict(nsr_plateu=0.3, nsr_range=(0, 1), nsr_update=0.05)


# ---------------------------------------------------------------- GPU: the brain forward
@gpu
@pytest.mark.parametrize("hidden", [[64, 64], [40, 130, 7]])
@pytest.mark.parametrize("space", ["box", "discrete"])
def test_act_rows_equals_es_act_per_row(hidden, space):
    from ppo_exploration_b200 import _lib as L
    M, A = 5, (2 if space == "box" else 3)
    es = _make(8, hidden=hidden, n_actions=A)
    rs = np.random.RandomState(3)
    thetas = torch.as_tensor(rs.randn(M, es.D) * 0.5).cuda()
    obs = torch.as_tensor(rs.randn(M, 8).astype(F32)).cuda()
    alive = torch.tensor([1, 1, 0, 1, 1], dtype=torch.uint8, device="cuda")
    draw = torch.tensor([7, 0], dtype=torch.int64, device="cuda")
    noise = es.noise_table()
    sizes = [8, *hidden, A]
    sizes_c = (C.c_int * len(sizes))(*sizes)
    disc = int(space == "discrete")
    seen = set()
    for step in range(4):
        got = torch.full((M,) if disc else (M, A), -5, dtype=torch.int64 if disc else torch.float64, device="cuda")
        L.call("ppx_es_act_rows", thetas.data_ptr(), noise.data_ptr(), M, sizes_c, len(sizes) - 1, obs.data_ptr(), alive.data_ptr(),
               disc, 99, draw.data_ptr(), step, got.data_ptr(), L.stream())
        for m in range(M):
            want = torch.full((1,) if disc else (1, A), -5, dtype=got.dtype, device="cuda")
            th = thetas[m].contiguous()
            L.call("ppx_es_act", th.data_ptr(), noise.data_ptr(), torch.zeros(1, dtype=torch.int64, device="cuda").data_ptr(), 0.0,
                   1, sizes_c, len(sizes) - 1, obs[m:m + 1].contiguous().data_ptr(), alive[m:m + 1].contiguous().data_ptr(), disc,
                   99, draw.data_ptr(), step, m, None, want.data_ptr(), L.stream())
            assert torch.equal(got[m:m + 1], want), (m, step, got[m], want)
            if disc and alive[m]:
                seen.add(int(got[m]))
    if disc:
        assert len(seen) > 1, "the Philox draw never changed the action"
    else:
        assert (got[2] == 0).all() and (got[[0, 1, 3, 4]].abs() > 0).all()


# ---------------------------------------------------------------- GPU: run() == the host composition == the f64 oracle
@gpu
@pytest.mark.parametrize("M", [2, 3])
def test_run_equals_host_composition_and_oracle(M, tmp_path, monkeypatch):
    from test_gpu_es_device_eval import DeviceTwin
    monkeypatch.chdir(tmp_path)
    P, maxs, G = 64, 32, 12
    tp, tb = _tables_for(P, M, maxs, seed=40 + M)
    a, b = _make(P, **RULE), _make(P, **RULE)
    lr0, theta0 = b.learning_rate, b.theta.clone()
    st = np.random.get_state()
    ra, rb, ro = [st], [st], [st]
    env, benv = DeviceTwin(tp, "box"), DeviceTwin(tb, "box")
    with _rng(rb):
        host = _Composition(b, tp, tb, M, maxs, RULE)
    for g in range(G):
        with _rng(ra):
            a.run(env, benv, 1, max_steps=maxs, meta_population_size=M, log_to_file=True)
        with _rng(rb):
            host.step()
        assert torch.equal(a.thetas, torch.stack(host.thetas)), f"generation {g}: thetas differ"
        assert torch.equal(a.archive, host.archive), f"generation {g}: archive differs"
        assert a.novelty_param == host.w, f"generation {g}: novelty_param"
        assert a.learning_rate == b.learning_rate
    rows = _csv_rows(str(tmp_path))
    assert len(rows) == G
    for g, (r, want) in enumerate(zip(rows, host.rec["rows"])):
        assert int(r["iteration"]) == g + 1 and float(r["total_time"]) >= 0
        for k, v in want.items():
            assert float(r[k]) == float(v), (g, k, r[k], v)
    assert [int(r["brain"]) for r in rows] == host.picks and len(set(host.picks)) > 1
    assert len(set(host.ws)) > 1, "novelty_param never moved"
    assert np.array_equal(ra[0][1], rb[0][1]) and ra[0][2] == rb[0][2], "numpy's RNG states differ after the two loops"
    # the f64 oracle, teacher-forced with the device's fitness vectors and behaviours
    rec = host.rec
    with _rng(ro):
        thetas0 = np.stack([theta0.cpu().numpy()] + [np.concatenate([np.random.randn(*s).ravel() for s in b.shapes])
                                                      for _ in range(M - 1)])
        out = ON.nsra_run(thetas0, lr0, G, shapes=b.shapes, sigma=b.SIGMA, decay=b.decay, novelty_param=0.5, **RULE,
                          eps_of=lambda g: rec["eps"][g], fitness_of=lambda g, th: rec["fit"][g],
                          brains_of=lambda g, th: (rec["bc"][g + 1], rec["f"][g + 1]))
    assert out["picks"] == host.picks
    assert out["w"] == host.ws
    np.testing.assert_allclose(a.thetas.cpu().numpy(), out["thetas"], rtol=1e-12, atol=1e-14)
    assert np.array_equal(a.archive.cpu().numpy(), out["archive"])
    np.testing.assert_allclose(a.learning_rate, out["lr"], rtol=1e-15)


@gpu
def test_changed_novelty_param_reaches_a_replayed_tell():
    P = 64
    arch = torch.as_tensor(np.random.RandomState(23).randn(40, 2)).cuda()
    qs = torch.as_tensor(np.random.RandomState(24).randn(2, 2)).cuda()
    fit = torch.as_tensor(np.random.RandomState(26).randn(P)).cuda()
    a, ref = _make(P), _make(P)
    for g, w in enumerate([0.5, 0.5, 0.5, 0.9, 0.9, 0.2]):
        a.novelty_param = ref.novelty_param = w
        a.ask(arch, qs)
        a.tell(fit)                                            # graphs: eager, captured, then replayed
        pop = ref._get_population()                            # the same step without graphs
        _, nov = ref.novelty_batch(arch, qs)
        ref._update_weights(fit, pop, novelty=nov[0:1])
        assert torch.equal(a.theta, ref.theta), f"step {g} (novelty_param {w}): theta differs"


# ---------------------------------------------------------------- GPU: one read per generation, launches per step
@gpu
def test_one_read_per_generation_and_two_launches_per_step():
    from test_gpu_es_device_eval import DeviceTwin
    from ppo_exploration_b200 import _lib as L
    P, M, maxs = 2048, 2, 48
    tp, tb = _tables_for(P, M, maxs, seed=60)
    es = _make(P, nsr_range=(0.5, 0.5))      # novelty_param stays put: a new value captures a new tell graph, which synchronises
    env, benv = DeviceTwin(tp, "box"), DeviceTwin(tb, "box")
    es.run(env, benv, 3, max_steps=maxs)                       # warm-up: buffers, the ask / tell graphs
    torch.cuda.synchronize()
    reads, steps = [], []
    read, episodes = es._run_read, es._episodes

    def counted_read():
        torch.cuda.set_sync_debug_mode(0)
        try:
            return read()
        finally:
            reads.append(1)
            torch.cuda.set_sync_debug_mode("error")

    def counted_episodes(*a, **kw):
        out = episodes(*a, **kw)
        steps.append(es.last_eval_steps)
        return out

    es._run_read, es._episodes = counted_read, counted_episodes
    per_gen = []
    for G in (1, 2):
        reads.clear()
        steps.clear()
        torch.cuda.set_sync_debug_mode("error")
        try:
            n0 = L.launch_count()
            es.run(env, benv, G, max_steps=maxs)
            n1 = L.launch_count()
        finally:
            torch.cuda.set_sync_debug_mode(0)
        assert len(reads) == G + 1, "one read per generation, plus the last generation's row at the end of run()"
        assert len(steps) == 2 * G and all(s >= 8 for s in steps)
        per_gen.append(n1 - n0 - 2 * sum(steps))
    # outside the two loops a generation adds the same few launches: novelty, ask's graph and tell's graph
    assert per_gen[1] == 2 * per_gen[0] and 0 < per_gen[0] <= 12, per_gen


# ---------------------------------------------------------------- GPU: reward_target and the CSV
@gpu
def test_reward_target_stops_at_the_host_generation(tmp_path, monkeypatch):
    from test_gpu_es_device_eval import DeviceTwin
    monkeypatch.chdir(tmp_path)
    P, M, maxs = 64, 2, 32
    tp, tb = _tables_for(P, M, maxs, seed=70)
    b = _make(P, **RULE)
    st = [np.random.get_state()]
    with _rng(st):
        host = _Composition(b, tp, tb, M, maxs, RULE)
        fb = [host.step() for _ in range(8)]
    k = int(np.argmax(fb[:6]))
    target = float(np.nextafter(fb[k], -np.inf))
    stop = next(j for j, v in enumerate(fb) if v > target)
    a = _make(P, **RULE)
    a.run(DeviceTwin(tp, "box"), DeviceTwin(tb, "box"), 20, max_steps=maxs, reward_target=target, log_to_file=True)
    assert a._generation == stop + 1
    rows = _csv_rows(str(tmp_path))
    assert len(rows) == stop + 1
    cols = {"iteration", "total_time", "reward", "brain", "novelty_param", "learning_rate", "fitness_mean", "fitness_max",
            "archive_size"}
    assert cols <= set(rows[0])
    assert float(rows[-1]["reward"]) == fb[stop] > target
    assert int(rows[-1]["archive_size"]) == M + stop + 1


# ---------------------------------------------------------------- GPU: save / load
def _cartpole_es(P, seed=6):
    np.random.seed(seed)
    return _ppx().EvolutionStrategy(env_id="CartPole-v1", hidden_sizes=(16, 16), obs_dim=4, n_actions=2, population_size=P,
                                    sigma=0.1, learning_rate=0.05, decay=0.999, noise_table_size=1 << 20, noise_seed=7,
                                    nsr_plateu=5.0)


def _cartpole_envs(P, M):
    ppx = _ppx()
    return (ppx.ClassicControlVecEnv("CartPole-v1", P, seed=3, reward_dtype=torch.float64),
            ppx.ClassicControlVecEnv("CartPole-v1", M, seed=5, env_offset=0, reward_dtype=torch.float64))


@gpu
def test_resume_equals_uninterrupted(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    ppx = _ppx()
    P, M, maxs = 128, 2, 200
    kw = dict(max_steps=maxs, meta_population_size=M)
    a = _cartpole_es(P)
    a.run(*_cartpole_envs(P, M), 10, **kw)
    want_rng = np.random.get_state()
    b = _cartpole_es(P)
    e, be = _cartpole_envs(P, M)
    b.run(e, be, 6, **kw)
    p = str(tmp_path / "es_run.pt")
    b.save(p)
    np.random.seed(12345)                                      # whatever happens in between
    e2, be2 = _cartpole_envs(P, M)
    c = ppx.EvolutionStrategy.load(p, env=e2, brain_env=be2)
    c.run(e2, be2, 4, **kw)
    got_rng = np.random.get_state()
    assert torch.equal(c.thetas, a.thetas)
    assert torch.equal(c.archive, a.archive)
    assert torch.equal(c.theta, a.theta) and torch.equal(c._draw, a._draw)
    assert c.novelty_param == a.novelty_param and c.learning_rate == a.learning_rate
    assert c._generation == a._generation == 10
    assert got_rng[1].tolist() == want_rng[1].tolist() and got_rng[2:] == want_rng[2:]
    # a checkpoint without a run still loads as before, with numpy's RNG left alone
    d = _cartpole_es(P)
    q = str(tmp_path / "es_plain.pt")
    d.save(q)
    st = np.random.get_state()
    d2 = ppx.EvolutionStrategy.load(q)
    assert d2.thetas is None and torch.equal(d2.theta, d.theta)
    assert np.random.get_state()[2] == st[2]


# ---------------------------------------------------------------- GPU: learning smoke
ES_SMOKE_GENERATIONS, ES_SMOKE_BOUND = 60, 400.0    # measured on a B200: f_b 500 > 475 at generation 44 (DESIGN.md §3.15)


@gpu
def test_run_learns_cartpole(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    ppx = _ppx()
    P, M = 1024, 2
    np.random.seed(0)
    es = ppx.EvolutionStrategy(env_id="CartPole-v1", hidden_sizes=(64, 64), obs_dim=4, n_actions=2, population_size=P,
                               sigma=0.1, learning_rate=0.05, noise_seed=1, noise_table_size=1 << 22)
    env = ppx.ClassicControlVecEnv("CartPole-v1", P, seed=0, reward_dtype=torch.float64)
    benv = ppx.ClassicControlVecEnv("CartPole-v1", M, seed=1, reward_dtype=torch.float64)
    es.run(env, benv, ES_SMOKE_GENERATIONS, max_steps=500, meta_population_size=M, reward_target=475, log_to_file=True)
    rows = _csv_rows(str(tmp_path), "CartPole-v1")
    best = max(float(r["reward"]) for r in rows)
    print(f"ES-NSRA CartPole-v1: best f_b {best:.1f} within {len(rows)} generations")
    assert best > ES_SMOKE_BOUND


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
    P, M, G, maxs = 64 * world, 2, 6, 200
    os.chdir(os.path.join(os.environ.get("PPX_ES_RUN_TMP", "."), f"rank{rank}"))

    def make():
        np.random.seed(33)
        return ppx.EvolutionStrategy(env_id="CartPole-v1", hidden_sizes=(16, 16), obs_dim=4, n_actions=2, population_size=P,
                                     sigma=0.1, learning_rate=0.05, device=dev, noise_table_size=1 << 20, noise_seed=4)

    def benv():
        return ppx.ClassicControlVecEnv("CartPole-v1", M, seed=9, env_offset=0, device=dev, reward_dtype=torch.float64)
    sharded = make()                                           # make() seeds numpy: both runs draw from the same state
    sharded.run(ppx.ClassicControlVecEnv("CartPole-v1", P // world, seed=8, device=dev, reward_dtype=torch.float64),
                benv(), G, max_steps=maxs, meta_population_size=M)
    with _single():                                            # one GPU over the union env
        union = make()
        union.run(ppx.ClassicControlVecEnv("CartPole-v1", P, seed=8, env_offset=0, device=dev, reward_dtype=torch.float64),
                  benv(), G, max_steps=maxs, meta_population_size=M)
    torch.cuda.synchronize()
    assert torch.equal(sharded.archive, union.archive), "the archive (and so the picks) differs from one GPU's"
    assert sharded.novelty_param == union.novelty_param
    np.testing.assert_allclose(sharded.thetas.cpu().numpy(), union.thetas.cpu().numpy(), rtol=1e-12, atol=1e-14)
    for t in (sharded.thetas, sharded.archive, torch.tensor([sharded.novelty_param], device=dev, dtype=torch.float64)):
        allt = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(allt, t.contiguous())
        assert all(torch.equal(allt[0], x) for x in allt), "ES run replicas diverged"
    dist.barrier()
    torch.cuda.synchronize()
    os._exit(0)


@gpu
def test_sharded_run_equals_single_gpu(tmp_path):
    import torch.multiprocessing as mp
    from test_gpu_sharded import _free_port
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    for r in range(2):
        os.makedirs(tmp_path / f"rank{r}")
    os.environ["PPX_ES_RUN_TMP"] = str(tmp_path)
    ctx = mp.spawn(_worker, args=(2, _free_port()), nprocs=2, join=False)
    while not ctx.join(timeout=600):
        pass
