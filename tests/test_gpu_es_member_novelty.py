"""ES-NSRA with a novelty per member (NSRA-ES, Conti et al. 2018, Alg. 3; DESIGN.md §3.16): novelty_mode="member".

CPU tests pin the f64 oracle update (oracle/es_member.py `update_weights_member`) and the squared-distance selection of the k-NN.
GPU tests check `ppx_knn_novelty_many` bit for bit against `ppx_knn_novelty` and the oracle, `ppx_es_update_member` against
the oracle, tell() through its CUDA graph, run() against a host composition of public pieces and against the teacher-forced
oracle loop, flat fitness, launches and reads per generation, save / load, two GPUs and a MountainCar-v0 learning run."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from oracle import es as OE                                             # noqa: E402
from oracle import es_member as OM                                      # noqa: E402
from oracle import es_nsra as ON                                        # noqa: E402

gpu = pytest.mark.gpu
F32 = np.float32


# ---------------------------------------------------------------- CPU: the oracle update
def _split(v, shapes):
    cut = np.cumsum([0] + [a * b for a, b in shapes])
    return [v[cut[l]:cut[l + 1]].reshape(shapes[l]) for l in range(len(shapes))]


def _pop(rs, P, shapes):
    return [[rs.randn(*s) for s in shapes] for _ in range(P)]


def test_member_update_with_zero_weight_is_the_reference_update():
    rs = np.random.RandomState(0)
    shapes = OE.layer_shapes(3, [5], 2)
    w = [rs.randn(*s) for s in shapes]
    pop = _pop(rs, 9, shapes)
    r = rs.randn(9)
    for nov_scalar in (0.0, 0.37, 12.5):
        want, lr_w = OE.update_weights(w, r, pop, 0.02, 0.1, 0.0, 0.999, novelty=nov_scalar)
        got, lr_g = OM.update_weights_member(w, r, rs.randn(9), pop, 0.02, 0.1, 0.0, 0.999)
        assert lr_w == lr_g
        assert all(np.array_equal(a, b) for a, b in zip(want, got))


def test_member_update_zero_std_cases():
    rs = np.random.RandomState(1)
    shapes = OE.layer_shapes(2, [4], 1)
    w = [rs.randn(*s) for s in shapes]
    pop = _pop(rs, 6, shapes)
    # both stds 0: untouched weights and lr
    out, lr = OM.update_weights_member(w, np.full(6, -200.0), np.full(6, 0.3), pop, 0.05, 0.1, 0.5, 0.99)
    assert out is w and lr == 0.05
    # flat fitness, varying novelty: the novelty-only update, lr decays
    nov = rs.rand(6)
    out, lr = OM.update_weights_member(w, np.full(6, -200.0), nov, pop, 0.05, 0.1, 0.5, 0.99)
    assert lr == 0.05 * 0.99
    N = (nov - nov.mean()) / nov.std()
    for l in range(len(w)):
        E = np.array([m[l] for m in pop])
        want = w[l] + 0.05 / (6 * 0.1) * (0.5 * np.dot(E.T, np.zeros(6)).T + 0.5 * np.dot(E.T, N).T) / 2
        assert np.array_equal(out[l], want)
        assert not np.array_equal(out[l], w[l])
    # centred ranks never skip
    out, lr = OM.update_weights_member(w, np.full(6, 1.0), np.full(6, 1.0), pop, 0.05, 0.1, 0.5, 0.99, shaping="centered_rank")
    assert lr == 0.05 * 0.99


def test_member_update_hand_computed():
    # P = 3, one 1x1 layer: eps = 1, 2, 3; r = 0, 1, 2 -> F~ = (-1, 0, 1) * sqrt(3/2); nov = 1, 1, 4 -> N~ = (-1, -1, 2) / sqrt(2)
    pop = [[np.array([[1.0]])], [np.array([[2.0]])], [np.array([[3.0]])]]
    w = [np.array([[0.5]])]
    lr, sigma, nw = 0.3, 0.1, 0.25
    out, lr2 = OM.update_weights_member(w, [0.0, 1.0, 2.0], [1.0, 1.0, 4.0], pop, lr, sigma, nw, 0.9)
    F = np.array([-1.0, 0.0, 1.0]) * np.sqrt(1.5)
    N = np.array([-1.0, -1.0, 2.0]) / np.sqrt(2.0)
    e = np.array([1.0, 2.0, 3.0])
    want = 0.5 + lr / (3 * sigma) * ((1 - nw) * (e @ F) + nw * (e @ N)) / 2
    assert abs(out[0][0, 0] - want) < 1e-14 and lr2 == lr * 0.9
    # centred ranks: r ranks (0, 1, 2) -> (-0.5, 0, 0.5); nov ranks with the index tie rule (0, 1, 2) -> same
    out, _ = OM.update_weights_member(w, [0.0, 1.0, 2.0], [1.0, 1.0, 4.0], pop, lr, sigma, nw, 0.9, shaping="centered_rank")
    c = np.array([-0.5, 0.0, 0.5])
    assert abs(out[0][0, 0] - (0.5 + lr / (3 * sigma) * ((1 - nw) * (e @ c) + nw * (e @ c)) / 2)) < 1e-14


# ---------------------------------------------------------------- CPU: selection on squared distances
def test_squared_selection_equals_knn_sum():
    rs = np.random.RandomState(2)
    for trial in range(200):
        M, dim, k = rs.randint(1, 60), rs.randint(1, 5), rs.randint(1, 33)
        if trial % 2:
            a = rs.randn(M, dim) * 10.0 ** rs.randint(-4, 4)
            q = rs.randn(dim) * 10.0 ** rs.randint(-4, 4)
        else:                                                    # integer grid: equal distances and duplicate points
            a = rs.randint(-3, 4, (M, dim)).astype(np.float64)
            q = a[rs.randint(M)] if trial % 4 == 0 else rs.randint(-3, 4, dim).astype(np.float64)
        S = min(k, M)
        assert OM.knn_sum_sq(a, q, S) == OE.knn_sum(a, q, S), (trial, M, dim, k)


# ---------------------------------------------------------------- GPU helpers
def _ppx():
    import ppo_exploration_b200 as ppx
    return ppx


def _L():
    from ppo_exploration_b200 import _lib as L
    return L


def _knn(name, archive, queries, K):
    L = _L()
    a, q = archive.contiguous(), queries.contiguous()
    s = torch.full((q.shape[0],), -1.0, dtype=torch.float64, device="cuda")
    n = torch.full_like(s, -1.0)
    L.call(name, a.data_ptr(), a.shape[0], q.data_ptr(), q.shape[0], a.shape[1], K, s.data_ptr(), n.data_ptr(), L.stream())
    return s, n


def _check_rows(archive, queries, K, s, n, rows):
    a, q = archive.cpu().numpy(), queries.cpu().numpy()
    S = min(K, a.shape[0])
    for i in rows:
        assert s[i] == OE.knn_sum(a, q[i], S), (i, s[i])
        assert n[i] == OE.novelty(a, q[i], K), (i, n[i])


KNN_MAX_DIM = 8


# ---------------------------------------------------------------- GPU: ppx_knn_novelty_many
@gpu
@pytest.mark.parametrize("K", [1, 10, 16, 32])
@pytest.mark.parametrize("dim", [1, 2, KNN_MAX_DIM])
def test_knn_many_equals_knn_novelty_and_oracle(K, dim):
    rs = np.random.RandomState(K * 10 + dim)
    for Q in (1, 7, 10_000):
        for M in sorted({max(1, K - 1), K, K + 1, 255, 257, 50_000}):
            if Q == 10_000 and M == 50_000 and K != 10:
                continue                                         # the largest case once per dim (K = 10) keeps the file short
            archive = torch.as_tensor(rs.randn(M, dim)).cuda()
            queries = torch.as_tensor(rs.randn(Q, dim)).cuda()
            s0, n0 = _knn("ppx_knn_novelty", archive, queries, K)
            s1, n1 = _knn("ppx_knn_novelty_many", archive, queries, K)
            assert torch.equal(s0, s1) and torch.equal(n0, n1), (Q, M)
            rows = range(Q) if Q * M <= 200_000 else rs.choice(Q, 5, replace=False)
            _check_rows(archive, queries, K, s1.cpu().numpy(), n1.cpu().numpy(), rows)


@gpu
@pytest.mark.parametrize("K", [1, 10, 32])
def test_knn_many_ties_duplicates_and_the_floor(K):
    rs = np.random.RandomState(5)
    for dim in (1, 2, 4):
        grid = rs.randint(-2, 3, (3000, dim)).astype(np.float64)        # every point many times over, distances tie
        archive = torch.as_tensor(grid).cuda()
        q = np.concatenate([grid[rs.choice(3000, 40)], rs.randint(-3, 4, (40, dim)).astype(np.float64)])
        queries = torch.as_tensor(q).cuda()
        s0, n0 = _knn("ppx_knn_novelty", archive, queries, K)
        s1, n1 = _knn("ppx_knn_novelty_many", archive, queries, K)
        assert torch.equal(s0, s1) and torch.equal(n0, n1)
        n = n1.cpu().numpy()
        if dim < 4:                                              # 5 or 25 grid points: each is in the archive >= 32 times
            assert (n[:40] == 5e-3).all(), "a query on a point present >= K times has novelty 0, floored to 5e-3"
        _check_rows(archive, queries, K, s1.cpu().numpy(), n, range(80))


@gpu
def test_knn_many_beyond_the_old_grid_limit():
    rs = np.random.RandomState(6)
    archive = torch.as_tensor(rs.randn(2000, 3)).cuda()
    queries = torch.as_tensor(rs.randn(70_000, 3)).cuda()
    s, n = _knn("ppx_knn_novelty_many", archive, queries, 10)
    rows = list(rs.choice(70_000, 40, replace=False)) + [0, 65_535, 65_536, 69_999]
    _check_rows(archive, queries, 10, s.cpu().numpy(), n.cpu().numpy(), rows)


@gpu
def test_knn_many_rejects_bad_shapes():
    a = torch.zeros(4, KNN_MAX_DIM + 1, dtype=torch.float64, device="cuda")
    with pytest.raises(RuntimeError, match="dim"):
        _knn("ppx_knn_novelty_many", a, a, 2)
    a = torch.zeros(4, 2, dtype=torch.float64, device="cuda")
    with pytest.raises(RuntimeError, match="K"):
        _knn("ppx_knn_novelty_many", a, a, 33)


# ---------------------------------------------------------------- GPU: ppx_es_update_member
def _make(P, seed=25, hidden=(64, 64), n_actions=2, obs_dim=8, **kw):
    np.random.seed(seed)
    return _ppx().EvolutionStrategy(env_id="table", hidden_sizes=hidden, obs_dim=obs_dim, n_actions=n_actions,
                                    population_size=P, sigma=0.1, learning_rate=0.05, noise_table_size=1 << 20, noise_seed=3,
                                    **kw)


def _eps_rows(es, off):
    return es.noise_table()[off[:, None] + torch.arange(es.D, device="cuda")[None]].double().cpu().numpy()


@gpu
@pytest.mark.parametrize("shaping", ["zscore", "centered_rank"])
@pytest.mark.parametrize("table", [False, True])
@pytest.mark.parametrize("w", [0.0, 0.5, 1.0])
def test_update_member_equals_oracle(shaping, table, w):
    P = 300
    es = _make(P, hidden=(16,), fitness_shaping=shaping, novelty_mode="member")
    es.novelty_param = w
    rs = np.random.RandomState(7)
    for step in range(3):
        r, nov = rs.randn(P), rs.rand(P) * 3
        if step == 2:
            r[::3] = r[0]                                        # ties for the ranks
            nov[::2] = nov[1]
        if table:
            pop = es._get_population()
            eps = _eps_rows(es, pop)
        else:
            eps = rs.randn(P, es.D).astype(F32).astype(np.float64)
            pop = eps
        theta0, lr0 = es.theta.cpu().numpy(), es.learning_rate
        es._update_weights(r, pop, novelty=torch.as_tensor(nov).cuda())
        want, lr = OM.update_weights_member(_split(theta0, es.shapes), r, nov, [_split(e, es.shapes) for e in eps], lr0,
                                            es.SIGMA, w, es.decay, shaping=shaping)
        np.testing.assert_allclose(es.theta.cpu().numpy(), np.concatenate([x.ravel() for x in want]), rtol=1e-12, atol=1e-14)
        assert es.learning_rate == lr and not es.update_skipped


@gpu
def test_update_member_zero_std_cases():
    P = 64
    es = _make(P, hidden=(16,), novelty_mode="member")
    rs = np.random.RandomState(8)
    eps = rs.randn(P, es.D).astype(F32)
    theta0, lr0 = es.theta.clone(), es.learning_rate
    es._update_weights(np.full(P, -200.0), eps, novelty=torch.full((P,), 0.25, dtype=torch.float64, device="cuda"))
    assert es.update_skipped and torch.equal(es.theta, theta0) and es.learning_rate == lr0
    nov = rs.rand(P)
    es._update_weights(np.full(P, -200.0), eps, novelty=torch.as_tensor(nov).cuda())
    assert not es.update_skipped and es.learning_rate == lr0 * es.decay
    want, _ = OM.update_weights_member(_split(theta0.cpu().numpy(), es.shapes), np.full(P, -200.0), nov,
                                       [_split(e.astype(np.float64), es.shapes) for e in eps], lr0, es.SIGMA, es.novelty_param,
                                       es.decay)
    np.testing.assert_allclose(es.theta.cpu().numpy(), np.concatenate([x.ravel() for x in want]), rtol=1e-12, atol=1e-14)
    assert not torch.equal(es.theta, theta0)


@gpu
@pytest.mark.parametrize("table", [False, True])
def test_update_member_zero_weight_is_bit_identical_to_es_update(table):
    P = 2000
    a = _make(P, novelty_mode="member")
    b = _make(P)
    a.novelty_param = b.novelty_param = 0.0
    rs = np.random.RandomState(9)
    for _ in range(3):
        r = torch.as_tensor(rs.randn(P)).cuda()
        pop = a._get_population() if table else rs.randn(P, a.D).astype(F32)
        if table:
            b._get_population()
        a._update_weights(r, pop, novelty=torch.as_tensor(rs.rand(P)).cuda())
        b._update_weights(r, pop, novelty=float(rs.rand()))
        assert torch.equal(a.theta, b.theta) and a.learning_rate == b.learning_rate


@gpu
def test_member_mode_arguments():
    es = _make(16, hidden=(8,), novelty_mode="member")
    with pytest.raises(ValueError, match="novelty"):
        es._update_weights(np.random.randn(16), np.random.randn(16, es.D).astype(F32))
    with pytest.raises(ValueError):
        _make(16, novelty_mode="members")
    brain = _make(16, hidden=(8,))
    brain.ask()
    fit = torch.zeros(16, dtype=torch.float64, device="cuda")
    with pytest.raises(ValueError, match="local_novelty"):
        brain.tell(fit, local_novelty=fit)
    es.ask()
    with pytest.raises(ValueError, match="local_novelty"):
        es.tell(fit)


# ---------------------------------------------------------------- GPU: tell() through its graph
@gpu
@pytest.mark.parametrize("shaping", ["zscore", "centered_rank"])
def test_member_tell_graph_equals_eager_update(shaping):
    P = 256
    a, ref = _make(P, fitness_shaping=shaping, novelty_mode="member"), _make(P, fitness_shaping=shaping, novelty_mode="member")
    fit = torch.zeros(P, dtype=torch.float64, device="cuda")
    nov = torch.zeros(P, dtype=torch.float64, device="cuda")
    rs = np.random.RandomState(10)
    for g, w in enumerate([0.5, 0.5, 0.5, 0.9, 0.9, 0.2, 0.2]):
        fit.copy_(torch.as_tensor(rs.randn(P)))
        nov.copy_(torch.as_tensor(rs.rand(P)))
        a.novelty_param = ref.novelty_param = w
        a.ask()
        a.tell(fit, local_novelty=nov)                           # eager, captured, replayed; recaptured for a new w
        pop = ref._get_population()
        ref._update_weights(fit, pop, novelty=nov)
        assert torch.equal(a.theta, ref.theta), f"step {g} (novelty_param {w}): theta differs"
        assert a.learning_rate == ref.learning_rate


# ---------------------------------------------------------------- GPU: run() == host composition == oracle
from test_gpu_es_run import RULE, _Composition, _csv_rows, _rng, _tables_for  # noqa: E402


class _MemberComposition(_Composition):
    """run(novelty_mode="member") composed on the host from public pieces: ask -> evaluate -> member_novelty -> tell."""

    def __init__(self, *a):
        super().__init__(*a)
        self.rec["bcp"] = []
        self.nov = None

    def step(self):
        es = self.es
        nov = es.novelty_batch(self.archive, self.bc)[1]
        b, _ = es.pick_brain([float(x) for x in nov.cpu().numpy()])
        es.novelty_param = self.w
        es.theta.copy_(self.thetas[b])
        pop, _, _ = es.ask()
        fit, _, bcp = es.evaluate(self.pop_env(), max_steps=self.maxs)
        if self.nov is None:
            self.nov = torch.zeros(bcp.shape[0], dtype=torch.float64, device="cuda")
        es.member_novelty(self.archive, bcp, out=self.nov)
        es.tell(fit, local_novelty=self.nov)
        self.thetas[b] = es.theta.clone()
        self.rec["eps"].append(_eps_rows(es, pop))
        self.rec["fit"].append(fit.cpu().numpy().copy())
        self.rec["bcp"].append(bcp.cpu().numpy().copy())
        self.bc, self.f = self.brains()
        self.rec["bc"].append(self.bc.cpu().numpy())
        self.rec["f"].append(self.f.cpu().numpy())
        self.archive = torch.cat([self.archive, self.bc[b:b + 1]])
        fb = float(self.f[b])
        self.fb.append(fb)
        self.picks.append(b)
        self.rec["rows"].append(dict(reward=fb, brain=b, novelty_param=self.w, learning_rate=es.learning_rate,
                                     fitness_mean=float(fit.mean()), fitness_max=float(fit.max()),
                                     archive_size=self.archive.shape[0], novelty_mean=float(self.nov.mean())))
        self.w, self.best = ON.nsr_adapt(self.w, self.fb, self.best, **self.rule)
        self.ws.append(self.w)
        return fb


@gpu
@pytest.mark.parametrize("M", [2, 3])
def test_member_run_equals_host_composition_and_oracle(M, tmp_path, monkeypatch):
    from test_gpu_es_device_eval import DeviceTwin
    monkeypatch.chdir(tmp_path)
    P, maxs, G = 64, 32, 12
    tp, tb = _tables_for(P, M, maxs, seed=40 + M)
    a, b = _make(P, novelty_mode="member", **RULE), _make(P, novelty_mode="member", **RULE)
    lr0, theta0 = b.learning_rate, b.theta.clone()
    st = np.random.get_state()
    ra, rb, ro = [st], [st], [st]
    env, benv = DeviceTwin(tp, "box"), DeviceTwin(tb, "box")
    with _rng(rb):
        host = _MemberComposition(b, tp, tb, M, maxs, RULE)
    for g in range(G):
        with _rng(ra):
            a.run(env, benv, 1, max_steps=maxs, meta_population_size=M, log_to_file=True)
        with _rng(rb):
            host.step()
        assert torch.equal(a.thetas, torch.stack(host.thetas)), f"generation {g}: thetas differ"
        assert torch.equal(a.archive, host.archive), f"generation {g}: archive differs"
        assert a.novelty_param == host.w and a.learning_rate == b.learning_rate
    rows = _csv_rows(str(tmp_path))
    assert len(rows) == G
    for g, (r, want) in enumerate(zip(rows, host.rec["rows"])):
        for k, v in want.items():
            assert float(r[k]) == float(v), (g, k, r[k], v)
    assert [int(r["brain"]) for r in rows] == host.picks and len(set(host.picks)) > 1
    rec = host.rec
    with _rng(ro):
        thetas0 = np.stack([theta0.cpu().numpy()] + [np.concatenate([np.random.randn(*s).ravel() for s in b.shapes])
                                                      for _ in range(M - 1)])
        out = OM.nsra_run_member(thetas0, lr0, G, shapes=b.shapes, sigma=b.SIGMA, decay=b.decay, novelty_param=0.5, **RULE,
                                 eps_of=lambda g: rec["eps"][g], fitness_of=lambda g, th: rec["fit"][g],
                                 brains_of=lambda g, th: (rec["bc"][g + 1], rec["f"][g + 1]),
                                 member_bcs_of=lambda g: rec["bcp"][g])
    assert out["picks"] == host.picks and out["w"] == host.ws
    np.testing.assert_allclose(a.thetas.cpu().numpy(), out["thetas"], rtol=1e-12, atol=1e-14)
    assert np.array_equal(a.archive.cpu().numpy(), out["archive"])
    np.testing.assert_allclose(a.learning_rate, out["lr"], rtol=1e-15)


class _FlatEnv:
    """Every member earns reward 0 at every step of a 6-step episode; the behaviour is the running sum of its actions."""

    def __init__(self, N):
        ppx = _ppx()
        self.num_envs = N
        self.observation_space, self.action_space = ppx.Box((8,)), ppx.Box((2,))
        self.obs = torch.as_tensor(np.random.RandomState(N).randn(7, N, 8).astype(F32)).cuda()

    def reset(self):
        self.t = 0
        self.acc = torch.zeros(self.num_envs, 2, dtype=torch.float64, device="cuda")
        return self.obs[0].clone()

    def step(self, a):
        self.t += 1
        self.acc = self.acc + a
        done = torch.full((self.num_envs,), self.t >= 6, dtype=torch.uint8, device="cuda")
        return self.obs[self.t].clone(), torch.zeros(self.num_envs, dtype=torch.float64, device="cuda"), done, []

    def behavior(self):
        return self.acc


@gpu
def test_flat_fitness_moves_only_member_mode():
    P, M = 128, 2
    for mode in ("brain", "member"):
        es = _make(P, hidden=(16,), novelty_mode=mode)
        env, benv = _FlatEnv(P), _FlatEnv(M)
        es.run(env, benv, 0, max_steps=6, meta_population_size=M)
        thetas0, archive0 = es.thetas.clone(), es.archive.clone()
        es.run(env, benv, 1, max_steps=6, meta_population_size=M)
        if mode == "brain":
            assert torch.equal(es.thetas, thetas0), "brain mode: std(r) == 0 skips the update"
            continue
        moved = [m for m in range(M) if not torch.equal(es.thetas[m], thetas0[m])]
        assert len(moved) == 1
        b = moved[0]
        bcp = es._eval[("bc", "population", P, 2)].cpu().numpy()
        nov = [OE.novelty(archive0.cpu().numpy(), x) for x in bcp]
        eps = _eps_rows(es, es._ask_off)
        want, lr = OM.update_weights_member(_split(thetas0[b].cpu().numpy(), es.shapes), np.zeros(P), nov,
                                            [_split(e, es.shapes) for e in eps], 0.05, es.SIGMA, 0.5, es.decay)
        np.testing.assert_allclose(es.thetas[b].cpu().numpy(), np.concatenate([x.ravel() for x in want]), rtol=1e-12,
                                   atol=1e-14)
        assert es.learning_rate == lr


# ---------------------------------------------------------------- GPU: reads and launches per generation
MEMBER_EXTRA_LAUNCHES = 1       # the ppx_knn_novelty_many of the members; tell's graph has 3 launches in both modes


@gpu
def test_one_read_and_one_extra_launch_per_generation():
    from test_gpu_es_device_eval import DeviceTwin
    L = _L()
    P, M, maxs = 2048, 2, 48
    tp, tb = _tables_for(P, M, maxs, seed=60)
    per_mode = {}
    for mode in ("brain", "member"):
        es = _make(P, nsr_range=(0.5, 0.5), novelty_mode=mode)
        env, benv = DeviceTwin(tp, "box"), DeviceTwin(tb, "box")
        es.run(env, benv, 3, max_steps=maxs)
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
        G = 2
        torch.cuda.set_sync_debug_mode("error")
        try:
            n0 = L.launch_count()
            es.run(env, benv, G, max_steps=maxs)
            n1 = L.launch_count()
        finally:
            torch.cuda.set_sync_debug_mode(0)
        assert len(reads) == G + 1
        per_mode[mode] = (n1 - n0 - 2 * sum(steps)) / G
    assert per_mode["member"] == per_mode["brain"] + MEMBER_EXTRA_LAUNCHES, per_mode


# ---------------------------------------------------------------- GPU: save / load
@gpu
@pytest.mark.parametrize("env_id", ["CartPole-v1", "MountainCarContinuous-v0"])
def test_member_resume_equals_uninterrupted(env_id, tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    ppx = _ppx()
    P, M, maxs = 128, 2, 120
    spec = {"CartPole-v1": (4, 2), "MountainCarContinuous-v0": (2, 1)}[env_id]

    def make():
        np.random.seed(6)
        return ppx.EvolutionStrategy(env_id=env_id, hidden_sizes=(16, 16), obs_dim=spec[0], n_actions=spec[1],
                                     population_size=P, sigma=0.1, learning_rate=0.05, decay=0.999, noise_table_size=1 << 20,
                                     noise_seed=7, nsr_plateu=5.0, novelty_mode="member")

    def envs():
        return (ppx.ClassicControlVecEnv(env_id, P, seed=3, reward_dtype=torch.float64),
                ppx.ClassicControlVecEnv(env_id, M, seed=5, env_offset=0, reward_dtype=torch.float64))
    kw = dict(max_steps=maxs, meta_population_size=M)
    a = make()
    a.run(*envs(), 8, **kw)
    b = make()
    e, be = envs()
    b.run(e, be, 5, **kw)
    p = str(tmp_path / "es_member.pt")
    b.save(p)
    np.random.seed(12345)
    e2, be2 = envs()
    c = ppx.EvolutionStrategy.load(p, env=e2, brain_env=be2)
    assert c.novelty_mode == "member"
    c.run(e2, be2, 3, **kw)
    assert torch.equal(c.thetas, a.thetas) and torch.equal(c.archive, a.archive)
    assert torch.equal(c.theta, a.theta) and c.learning_rate == a.learning_rate and c.novelty_param == a.novelty_param
    # a checkpoint written before novelty_mode existed loads as "brain"
    ck = torch.load(p, weights_only=True)
    del ck["config"]["novelty_mode"]
    q = str(tmp_path / "es_old.pt")
    torch.save(ck, q)
    assert ppx.EvolutionStrategy.load(q).novelty_mode == "brain"


# ---------------------------------------------------------------- GPU: MountainCar-v0 learning
# measured on a B200 (DESIGN.md §3.16): from seed 0 member mode first reached f_b > -200 at generation 32; brain mode stayed
# at -200 for 150 generations (not asserted).  The budget leaves margin over the measured count.
MC_SEED, MC_GENERATIONS = 0, 60


def mountaincar_run(mode, generations, seed=MC_SEED, P=1024, M=2):
    """ES-NSRA on MountainCar-v0 (-1 per step until the flag; 200-step episodes): the f_b of every generation."""
    ppx = _ppx()
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
    es.run(env, benv, generations, max_steps=200, meta_population_size=M, reward_target=-200)
    return fb


@gpu
def test_member_mode_leaves_the_mountaincar_plateau(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    fb = mountaincar_run("member", MC_GENERATIONS)
    print(f"MountainCar-v0 member mode: f_b {fb[-1]:.0f} after {len(fb)} generations")
    assert fb[-1] > -200, f"f_b stayed at -200 for {len(fb)} generations"


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
    os.chdir(os.path.join(os.environ.get("PPX_ES_MEMBER_TMP", "."), f"rank{rank}"))

    def make():
        np.random.seed(33)
        return ppx.EvolutionStrategy(env_id="CartPole-v1", hidden_sizes=(16, 16), obs_dim=4, n_actions=2, population_size=P,
                                     sigma=0.1, learning_rate=0.05, device=dev, noise_table_size=1 << 20, noise_seed=4,
                                     novelty_mode="member")

    def benv():
        return ppx.ClassicControlVecEnv("CartPole-v1", M, seed=9, env_offset=0, device=dev, reward_dtype=torch.float64)
    sharded = make()
    sharded.run(ppx.ClassicControlVecEnv("CartPole-v1", P // world, seed=8, device=dev, reward_dtype=torch.float64),
                benv(), G, max_steps=maxs, meta_population_size=M)
    assert sharded.update_mode.startswith("sharded")
    with _single():
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
def test_sharded_member_run_equals_single_gpu(tmp_path):
    import torch.multiprocessing as mp
    from test_gpu_sharded import _free_port
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    for r in range(2):
        os.makedirs(tmp_path / f"rank{r}")
    os.environ["PPX_ES_MEMBER_TMP"] = str(tmp_path)
    ctx = mp.spawn(_worker, args=(2, _free_port()), nprocs=2, join=False)
    while not ctx.join(timeout=600):
        pass
