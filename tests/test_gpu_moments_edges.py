"""The running-moment, normalisation and advantage-statistics kernels (bonus.cu, gather.cu) against float64 NumPy
references, at the tile, grid, alignment and ticket edges the small goldens never reach; and the scratch lifetime of the
entry points whose buffers a captured CUDA graph holds.

Every reference gets the float64 cast of the f32 inputs the kernel reads, so NumPy accumulates in f64 like the kernels.

Tolerances.  u = 2^-53 is the unit roundoff of f64.
- Summation.  A recursive f64 sum of k terms has an error that behaves like a random walk of k roundings, each at most
  u times the running magnitude: about sqrt(k) u sum|x|.  The worst case (k u sum|x|) is never approached by random data;
  the bounds below take ten standard deviations, S(k) = 10 sqrt(k + 8) u, where k is the longest chain of additions in the
  kernel (the per-thread loop plus the shuffle and shared-memory trees, + 8 for the tree depths and the final divide).
  For 65537 rows in 8 row phases that is S = 1e-13, the "about 1e-13" of the running moments.
- Running moments (ppx_rms_update, rnd_normalize_rollout, vecnorm_reward).  The batch moments are two-pass, so the batch
  variance is a sum of positive squares with no cancellation: relative error S(k).  The merge (util.py:30-44) adds only
  positive terms to the variance and rounds a handful of times (bonus.cu is built with FMA contraction, so it may round
  once where NumPy rounds twice): a few u more.  The mean is checked against S(k) (|mean_prev| + mean|x|), the variance
  against S(k) (var + 2 |delta| (|mean_prev| + mean|x|) count n / tot^2), the second term being the error of delta^2.
  The count is an f64 sum of the same operands in the same order: exact.
- One-pass statistics (ppx_mean_std, the gather's advantage moments): var = (sum x^2 - sum x * mean) / (n - 1) cancels a
  factor (mean^2 + var) / var.  The bound is S(k) sum x^2 / ((n - 1) var) on the variance, half of it on the std.  At
  |mean| = 1e3 std that is ~1e6 S(k) (the std is off by ~3e-10 at n = 2^22 + 3; 1e-12 holds to |mean| ~ 1e2 std, as
  gather.cu states).  Centred data is held to ~1e-14.
- ppx_moments_pack / _merge: Chan's merge of W records, every M2 term positive: 1e-13 relative.
- Elementwise f64 -> f32 results.  ppx_obs_istd, ppx_vecnorm_obs and ppx_rnd_sqerr perform the reference's IEEE
  operations one for one (no multiply-add to contract): bit-exact.  ppx_normalize_obs multiplies by the f64 reciprocal
  where the reference divides (bonus.cu:88-90): the two f64 values are within 1.5 f64 ulps, so their f32 roundings differ
  only where the reference lies within 2 f64 ulps of an f32 rounding boundary (a midpoint between two f32 values), and
  then by one f32 ulp.  The test finds every differing element and asserts exactly that of each one.  The reward
  divisions of rnd_normalize_rollout / vecnorm_reward use a divisor within ~1e-13 of the reference's: 1 f32 ulp.
- Gathered fields are copies: bit-exact.
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from oracle import rollout as OR

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
F32, F64 = np.float32, np.float64


def _L():
    from ppo_exploration_b200 import _lib as L
    return L


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def S(k):
    return 10.0 * math.sqrt(k + 8) * U


def _dev(a):
    return torch.as_tensor(np.ascontiguousarray(a)).cuda()


def _host(t):
    torch.cuda.synchronize()
    return t.cpu().numpy()


def _ulp_ok(got, want, ulps=1):
    """|got - want| <= ulps f32 ulps of want, elementwise (f32 arrays)"""
    want = np.asarray(want, F32)
    return np.abs(got.astype(F64) - want.astype(F64)) <= ulps * np.spacing(np.abs(want)).astype(F64)


def _near_f32_boundary(y, ulps=2):
    """True where the f64 value y lies within `ulps` f64 ulps of a midpoint between two adjacent f32 values"""
    f = y.astype(F32)
    toward = np.where(y > f.astype(F64), np.inf, -np.inf).astype(F32)
    mid = (f.astype(F64) + np.nextafter(f, toward).astype(F64)) / 2
    return np.abs(y - mid) <= ulps * np.spacing(np.abs(y))


# ----------------------------------------------------------------------------------------------------------------------
# running moments
# ----------------------------------------------------------------------------------------------------------------------
def _rms_state(dim, mean=0.0, var=1.0, count=1e-4):
    return (torch.full((dim,), mean, dtype=torch.float64, device="cuda"), torch.full((dim,), var, dtype=torch.float64, device="cuda"),
            torch.full((1,), count, dtype=torch.float64, device="cuda"))


def _rms_check(st, ref, x64, prev_mean, k, what):
    """st: the device state, ref: oracle RunningMeanStd after the same update, x64: the batch, prev_mean: before it"""
    m, v, c = (_host(t) for t in st)
    n = x64.shape[0]
    tot = ref.count
    sm = np.abs(prev_mean) + np.abs(x64).mean(0)
    delta = np.abs(x64.mean(0) - prev_mean)
    cnt = tot - n
    assert c[0] == ref.count, f"{what}: count {c[0]!r} != {ref.count!r}"
    err_m = np.abs(m - ref.mean)
    assert np.all(err_m <= S(k) * sm), f"{what}: mean off by {np.max(err_m / sm):.3g} of its scale (bound {S(k):.3g})"
    tol_v = S(k) * (ref.var + 2 * delta * sm * cnt * n / tot ** 2)
    err_v = np.abs(v - ref.var)
    assert np.all(err_v <= tol_v), f"{what}: var off by {np.max(err_v / ref.var):.3g} relative"


def _rms_k(n, dim):
    return -(-n // 8) + 8 if dim > 1 else -(-n // 1024) + 10


@pytest.mark.parametrize("dim", [1, 31, 32, 33, 257, 28224])
@pytest.mark.parametrize("f64", [False, True])
def test_rms_update_against_f64(dim, f64):
    """Column tiles of 32 (rms_cols_kernel), the one-CTA scalar kernel beyond 1024 rows, f32 and f64 inputs (f64 values
    no f32 holds, so an f32 load is caught), several updates in a row.  28224 x 65537 (7.4 GB) is left out: its column
    tiles are those of 28224 x 1025 and its row phases those of 257 x 65537."""
    L = _L()
    rs = np.random.RandomState(dim + 7 * f64)
    st = _rms_state(dim)
    ref = OR.RunningMeanStd(shape=(dim,))
    ref.mean, ref.var = np.zeros(dim), np.ones(dim)
    for n in (1, 2, 7, 8, 9, 1025, 65537):
        if dim * n > 40_000_000:
            continue
        x64 = rs.randn(n, dim) * 3.0 + rs.randn(dim)
        if not f64:
            x64 = x64.astype(F32).astype(F64)
        x = _dev(x64 if f64 else x64.astype(F32))
        prev = ref.mean.copy()
        L.call("ppx_rms_update", x.data_ptr(), int(f64), n, dim, st[0].data_ptr(), st[1].data_ptr(), st[2].data_ptr(), None,
               L.stream())
        ref.update(x64)
        _rms_check(st, ref, x64, prev, _rms_k(n, dim), f"dim={dim} n={n} f64={f64}")
        # continue from the device state exactly (the next update's reference starts where the kernel is)
        ref.mean, ref.var = _host(st[0]).copy(), _host(st[1]).copy()


@pytest.mark.parametrize("dim", [1, 33])
@pytest.mark.parametrize("n", [1025, 65537])
def test_rms_update_offset_batch_and_large_prior_count(dim, n):
    """A batch whose mean is 1e4 x its std (two-pass: no cancellation allowance), then one row merged into a prior count
    of 1e9."""
    L = _L()
    rs = np.random.RandomState(n + dim)
    st = _rms_state(dim)
    ref = OR.RunningMeanStd(shape=(dim,))
    ref.mean, ref.var = np.zeros(dim), np.ones(dim)
    x64 = (1e4 + rs.randn(n, dim)).astype(F32).astype(F64)
    x = _dev(x64.astype(F32))
    L.call("ppx_rms_update", x.data_ptr(), 0, n, dim, st[0].data_ptr(), st[1].data_ptr(), st[2].data_ptr(), None, L.stream())
    ref.update(x64)
    _rms_check(st, ref, x64, np.zeros(dim), _rms_k(n, dim), "mean = 1e4 std")
    # prior count 1e9 + a 1-row batch
    st = _rms_state(dim, mean=0.5, var=2.0, count=1e9)
    ref.mean, ref.var, ref.count = np.full(dim, 0.5), np.full(dim, 2.0), 1e9
    one = rs.randn(1, dim) * 1e3
    xo = _dev(one)
    L.call("ppx_rms_update", xo.data_ptr(), 1, 1, dim, st[0].data_ptr(), st[1].data_ptr(), st[2].data_ptr(), None, L.stream())
    ref.update(one)
    _rms_check(st, ref, one, np.full(dim, 0.5), 9, "count 1e9 + 1 row")


def test_obs_istd_bit_exact():
    L = _L()
    rs = np.random.RandomState(1)
    for dim in (1, 255, 256, 257, 28224):
        var = np.exp(rs.uniform(-40, 40, dim))
        var[::7] = 0.0
        var[1::11] = 1e-10
        var[2::13] = 2.0 ** 40
        v = _dev(var)
        out = torch.empty(dim, dtype=torch.float64, device="cuda")
        L.call("ppx_obs_istd", v.data_ptr(), dim, out.data_ptr(), L.stream())
        assert np.array_equal(_host(out), 1.0 / np.sqrt(var + 1e-10)), f"dim={dim}"


def _normalize_case(rs, n, dim):
    """observations spread to +-7 standard deviations, var = 0 columns, and exact +-5 edges: a column with var = 2^40
    (var + 1e-10 rounds to 2^40, istd = 2^-20 exactly) and mean 0 holding +-5 * 2^20 and one more / less"""
    mean = rs.randn(dim) * 2
    var = np.exp(rs.uniform(-6, 6, dim))
    var[rs.rand(dim) < 0.1] = 0.0
    obs = (mean + np.sqrt(var + 1e-10) * rs.uniform(-7, 7, (n, dim))).astype(F32)
    obs[rs.rand(n, dim) < 0.05] = F32(0)
    c = dim // 2
    mean[c], var[c] = 0.0, 2.0 ** 40
    edge = np.array([5, -5, 5 + 2.0 ** -20, -5 - 2.0 ** -20, 5 - 2.0 ** -20, 0], F64) * 2 ** 20
    obs[:, c] = edge[np.arange(n) % len(edge)]
    return obs, mean, var


def _normalize_check(got, obs, mean, var, what):
    y = np.clip((obs.astype(F64) - mean) / np.sqrt(var + 1e-10), -5, 5)
    want = y.astype(F32)
    diff = got != want
    near = _near_f32_boundary(y)
    bad = diff & ~near
    assert not bad.any(), f"{what}: {bad.sum()} elements differ off an f32 rounding boundary, first at {np.argwhere(bad)[0]}"
    assert np.all(_ulp_ok(got[diff], want[diff])), f"{what}: a boundary element differs by more than 1 f32 ulp"
    # an exception needs y within 2 f64 ulps of a midpoint: ~2^-27 of the f32 ulp interval, so they are rare
    assert diff.sum() <= 8 + got.size * 2.0 ** -20, f"{what}: {diff.sum()} double-rounding exceptions of {got.size}"


@pytest.mark.parametrize("dim", [1, 3, 4, 5, 1023, 1024, 1025, 28224])
def test_normalize_obs_contract(dim):
    """bonus.cu:88-90.  More rows than the grid's row slices, scalar and float4 paths (dim % 4, and pointers one float off
    16-byte alignment with dim % 4 == 0)."""
    L = _L()
    rs = np.random.RandomState(dim)
    gx = -(-dim // 1024)
    gy = -(-16 * _sms() // gx)
    n = 2 * gy + 3
    obs, mean, var = _normalize_case(rs, n, dim)
    m, v = _dev(mean), _dev(var)
    offsets = [(0, 0)] + ([(1, 1), (1, 0), (0, 1)] if dim % 4 == 0 else [])
    for oi, oo in offsets:
        src = torch.zeros(n * dim + 4, dtype=torch.float32, device="cuda")
        dst = torch.full((n * dim + 4,), float("nan"), dtype=torch.float32, device="cuda")
        src[oi:oi + n * dim] = _dev(obs.reshape(-1))
        L.call("ppx_normalize_obs", src.data_ptr() + 4 * oi, n, dim, m.data_ptr(), v.data_ptr(), dst.data_ptr() + 4 * oo, L.stream())
        full = _host(dst)
        got = full[oo:oo + n * dim].reshape(n, dim)
        assert np.isnan(full[:oo]).all() and np.isnan(full[oo + n * dim:]).all(), "normalize_obs wrote outside its rows"
        _normalize_check(got, obs, mean, var, f"dim={dim} n={n} offsets={oi, oo}")


def test_rnd_sqerr_bit_exact():
    L = _L()
    rs = np.random.RandomState(2)
    for n in (1, 255, 256, 257, 100003):
        p, t = rs.randn(n).astype(F32) * 3, rs.randn(n).astype(F32)
        pd, td = _dev(p), _dev(t)
        r = torch.empty(n, dtype=torch.float32, device="cuda")
        L.call("ppx_rnd_sqerr", pd.data_ptr(), td.data_ptr(), n, r.data_ptr(), L.stream())
        d = p - t
        assert np.array_equal(_host(r), d * d), f"n={n}"


def _rnd_rollout(L, r32, st):
    T, N = r32.shape
    r = _dev(r32)
    L.call("ppx_rnd_normalize_rollout", r.data_ptr(), T, N, st[0].data_ptr(), st[1].data_ptr(), st[2].data_ptr(), L.stream())
    return _host(r)


@pytest.mark.parametrize("T", [1, 2, 128])
def test_rnd_normalize_rollout_step_by_step(T):
    """rnd_bonus_step's update-and-divide (oracle/learner.py:123-129) in t order; two calls continue one state."""
    L = _L()
    rs = np.random.RandomState(T)
    for N in (1, 2, 255, 256, 257, 4096):
        st = _rms_state(1)
        ref = OR.RunningMeanStd()
        for call in range(2):
            r32 = (rs.exponential(size=(T, N)) * (1 + call)).astype(F32)
            got = _rnd_rollout(L, r32, st)
            for t in range(T):
                row = r32[t].astype(F64)
                ref.update(row)
                want = (row / (np.sqrt(ref.var) + 1e-08)).astype(F32)
                assert np.all(_ulp_ok(got[t], want)), f"T={T} N={N} call {call} step {t}: reward off by more than 1 ulp"
            m, v, c = (_host(x)[0] for x in st)
            k = -(-N // 256) + 10 + 2 * T
            assert c == ref.count
            assert abs(m - ref.mean) <= S(k) * (abs(ref.mean) + np.sqrt(ref.var)), f"T={T} N={N}: mean"
            assert abs(v - ref.var) <= S(k) * ref.var, f"T={T} N={N}: var"


def test_rnd_normalize_rollout_grows_its_scratch():
    """A call with more steps than any other in this file (the scratch grows; the old block is kept)."""
    L = _L()
    rs = np.random.RandomState(9)
    T, N = 3000, 3
    st = _rms_state(1)
    ref = OR.RunningMeanStd()
    r32 = rs.exponential(size=(T, N)).astype(F32)
    got = _rnd_rollout(L, r32, st)
    for t in range(T):
        ref.update(r32[t].astype(F64))
        assert np.all(_ulp_ok(got[t], (r32[t].astype(F64) / (np.sqrt(ref.var) + 1e-08)).astype(F32))), f"step {t}"
    assert _host(st[2])[0] == ref.count
    assert abs(_host(st[1])[0] - ref.var) <= S(2 * T) * ref.var


# ----------------------------------------------------------------------------------------------------------------------
# VecNormalize
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,dim", [(1, 1), (7, 6), (1000, 1000), (3, 250000)])
def test_vecnorm_obs_bit_exact(n, dim):
    """Clip edges (10, and 0.3 which no f32 holds) and n * dim beyond the grid cap (the grid-stride loop)."""
    L = _L()
    rs = np.random.RandomState(n * dim)
    mean, var = rs.randn(dim), np.exp(rs.uniform(-4, 4, dim))
    var[::5] = 0.0
    obs = (mean + np.sqrt(var + 1e-8) * rs.uniform(-15, 15, (n, dim))).astype(F32)
    o, m, v = _dev(obs), _dev(mean), _dev(var)
    out = torch.empty_like(o)
    for eps, clip in ((1e-8, 10.0), (1e-8, 0.3), (0.5, 1.0)):
        L.call("ppx_vecnorm_obs", o.data_ptr(), n, dim, m.data_ptr(), v.data_ptr(), eps, clip, out.data_ptr(), L.stream())
        want = np.clip((obs.astype(F64) - mean) / np.sqrt(var + eps), -clip, clip).astype(F32)
        assert np.array_equal(_host(out), want), f"eps={eps} clip={clip}"


def _vn_reward_step(L, r32, done, ret, st, gamma, eps, clip, update):
    out = torch.empty(len(r32), dtype=torch.float32, device="cuda")
    r, d = _dev(r32), _dev(done.astype(np.uint8))
    L.call("ppx_vecnorm_reward", r.data_ptr(), d.data_ptr(), ret.data_ptr(), len(r32), gamma,
           st[0].data_ptr(), st[1].data_ptr(), st[2].data_ptr(), eps, clip, int(update), out.data_ptr(), L.stream())
    return _host(out)


@pytest.mark.parametrize("n", [1, 2, 1023, 1024, 1025, 4097])
def test_vecnorm_reward_step_by_step(n):
    """Each step is checked from the device state before it (ret, ret_rms) against the restatement's arithmetic: ret =
    ret * gamma + r rounds once on the device (FMA) and twice in NumPy, within u (|gamma ret| + 2 |ret|); training is
    switched off for a stretch (update_stats = 0: returns frozen, ret_rms bit-identical), a done zeroes ret exactly."""
    L = _L()
    rs = np.random.RandomState(n)
    gamma, eps, clip = 0.99, 1e-8, 10.0
    ret = torch.zeros(n, dtype=torch.float64, device="cuda")
    st = _rms_state(1)
    for step in range(40):
        update = not (15 <= step < 25)
        r32 = (rs.randn(n) * 5).astype(F32)
        done = rs.rand(n) < 0.1
        ret0, (m0, v0, c0) = _host(ret).copy(), (_host(x)[0] for x in st)
        out = _vn_reward_step(L, r32, done, ret, st, gamma, eps, clip, update)
        ret1, (m1, v1, c1) = _host(ret), (_host(x)[0] for x in st)
        ref = OR.RunningMeanStd()
        ref.mean, ref.var, ref.count = m0, v0, c0
        what = f"n={n} step {step} update={update}"
        if update:
            acc = ret0 * gamma + r32.astype(F64)
            err = np.abs(np.where(done, acc, ret1) - acc)
            assert np.all(err <= 2 * U * (np.abs(gamma * ret0) + np.abs(acc))), f"{what}: ret"
            ref.update(acc)
            k = -(-n // 1024) + 10
            assert c1 == ref.count, f"{what}: count"
            assert abs(m1 - ref.mean) <= S(k) * (abs(m0) + np.abs(acc).mean()), f"{what}: ret_rms mean"
            assert abs(v1 - ref.var) <= S(k) * (ref.var + 2 * abs(acc.mean() - m0) * (abs(m0) + np.abs(acc).mean())), \
                f"{what}: ret_rms var"
        else:
            assert (m1, v1, c1) == (m0, v0, c0), f"{what}: ret_rms changed while not training"
            assert np.array_equal(np.where(done, ret0, ret1), ret0), f"{what}: returns accumulated while not training"
        assert np.all(ret1[done] == 0.0), f"{what}: a done did not zero its return"
        want = np.clip(r32.astype(F64) / np.sqrt(ref.var + eps), -clip, clip).astype(F32)
        assert np.all(_ulp_ok(out, want)), f"{what}: normalised rewards"


class _HostEnv:
    def __init__(self, n, d, seed, cuda=False):
        import ppo_exploration_b200 as ppx
        self.num_envs, self.rs, self.cuda, self.d = n, np.random.RandomState(seed), cuda, d
        self.observation_space, self.action_space = ppx.Box((d,)), ppx.Box((2,))

    def _out(self, x):
        return torch.as_tensor(x).cuda() if self.cuda else x

    def reset(self):
        return self._out((self.rs.randn(self.num_envs, self.d) * 3 + 1).astype(F32))

    def step(self, a):
        o = (self.rs.randn(self.num_envs, self.d) * 3 + 1).astype(F32)
        r = (self.rs.randn(self.num_envs) * 5).astype(F32)
        d = self.rs.rand(self.num_envs) < 0.2
        return self._out(o), self._out(r), self._out(d), [{} for _ in range(self.num_envs)]


@pytest.mark.parametrize("cuda", [False, True])
@pytest.mark.parametrize("norm_reward", [True, False])
def test_vecnormalize_training_and_norm_reward_flags(norm_reward, cuda):
    """Every combination of `training` and `norm_reward` over many steps, training switched off and on again, against
    the restatement: statistics and returns move only while training, rewards are divided only with norm_reward."""
    import ppo_exploration_b200 as ppx
    n = 16
    vn = ppx.VecNormalize(_HostEnv(n, 6, 3, cuda), norm_reward=norm_reward)
    src, ref = _HostEnv(n, 6, 3), OR.VecNormalizeRef(n, (6,), norm_reward=norm_reward)
    vn.reset()
    ref.reset(src.reset().astype(F64))
    for step in range(36):
        vn.training = ref.training = not (12 <= step < 24)
        before = [getattr(vn.ret_rms, k).clone() for k in ("mean_dev", "var_dev", "count_dev")] + [vn.obs_rms.count_dev.clone()]
        ret0 = vn.ret.clone()
        o, r, d, _ = vn.step(np.zeros((n, 2)))
        ro, rr, rd, _ = src.step(None)
        wo, wr = ref.step(ro.astype(F64), rr.astype(F64), rd)
        d = d.cpu().numpy().astype(bool) if isinstance(d, torch.Tensor) else d
        assert np.array_equal(d, rd)
        what = f"step {step} training={vn.training}"
        if not norm_reward:
            assert np.array_equal(r.cpu().numpy(), rr), f"{what}: rewards changed without norm_reward"
        else:
            np.testing.assert_allclose(r.cpu().numpy(), wr, rtol=1e-5, atol=1e-6, err_msg=what)
        np.testing.assert_allclose(o.cpu().numpy(), wo, rtol=1e-5, atol=1e-6, err_msg=what)
        np.testing.assert_allclose(vn.ret.cpu().numpy(), ref.ret, rtol=1e-12, atol=1e-12, err_msg=what)
        assert vn.ret_rms.count == ref.ret_rms.count and vn.obs_rms.count == ref.obs_rms.count, what
        np.testing.assert_allclose(vn.ret_rms.var, ref.ret_rms.var, rtol=1e-12, err_msg=what)
        if not vn.training:
            after = [getattr(vn.ret_rms, k) for k in ("mean_dev", "var_dev", "count_dev")] + [vn.obs_rms.count_dev]
            assert all(torch.equal(a, b) for a, b in zip(before, after)), f"{what}: statistics moved"
            assert torch.equal(torch.where(torch.as_tensor(rd).cuda(), ret0, vn.ret), ret0), f"{what}: returns moved"
        assert np.all(vn.ret.cpu().numpy()[rd] == 0.0), what


# ----------------------------------------------------------------------------------------------------------------------
# advantage statistics
# ----------------------------------------------------------------------------------------------------------------------
def _onepass_check(mean, std, x64, k, what):
    n = len(x64)
    rm, rv = x64.mean(), x64.var(ddof=1)
    assert abs(mean - rm) <= S(k) * np.abs(x64).mean(), f"{what}: mean {mean!r} vs {rm!r}"
    tol = 0.5 * S(k) * np.sum(x64 * x64) / ((n - 1) * rv) + 2 * U
    assert abs(std - np.sqrt(rv)) <= tol * np.sqrt(rv), f"{what}: std off by {abs(std / np.sqrt(rv) - 1):.3g} (bound {tol:.3g})"


@pytest.mark.parametrize("n", [2, 3, 2047, 2048, 2049, 256 * 2048, 256 * 2048 + 1, 2 ** 22 + 3])
def test_mean_std(n):
    """One or many blocks, the 256-block cap; two calls back to back (the last-block ticket is re-armed); centred data
    and |mean| = 1e3 std; a constant input gives exactly that mean."""
    L = _L()
    rs = np.random.RandomState(n % 1000)
    nb = max(1, min(256, -(-n // 2048)))
    k = -(-n // (nb * 256)) + 18
    out = torch.empty(2, dtype=torch.float64, device="cuda")
    for offset in (0.0, 1e3):
        # n <= 3: fixed values, so that a near-zero sample variance cannot loosen the bound
        z = np.array([-1.0, 0.5, 1.0])[:n] if n <= 3 else rs.randn(n)
        x64 = (offset + z).astype(F32).astype(F64)
        x = _dev(x64.astype(F32))
        L.call("ppx_mean_std", x.data_ptr(), n, out.data_ptr(), L.stream())
        m, s = _host(out)
        _onepass_check(m, s, x64, k, f"n={n} mean offset {offset}")
    # a constant c: every partial sum of c is exact (24-bit c, n < 2^29), so the mean is c exactly.  With c = 0.75 the
    # squares are exact too and the std is exactly 0; a 24-bit c such as f32(0.3) leaves q rounded, and the std is only
    # bounded by the cancellation: sqrt(S(k) q / (n - 1)) ~ sqrt(S(k)) c
    for c, exact in ((0.75, True), (float(F32(0.3)), False)):
        x = torch.full((n,), c, dtype=torch.float32, device="cuda")
        L.call("ppx_mean_std", x.data_ptr(), n, out.data_ptr(), L.stream())
        m, s = _host(out)
        assert m == c, (c, m)
        assert (s == 0.0) if exact else (s <= math.sqrt(S(k) * n / max(n - 1, 1)) * c), (c, s)


@pytest.mark.parametrize("W", [1, 2, 3, 8])
def test_moments_pack_merge(W):
    L = _L()
    rs = np.random.RandomState(W)
    sizes = rs.randint(2, 90, W)
    sizes[1::3] = 2                                         # some records of two rows
    parts = [rs.randn(k) * 2 + 0.7 + r for r, k in enumerate(sizes)]
    x = np.concatenate(parts)
    recs = torch.empty(W, 3, dtype=torch.float64, device="cuda")
    for r, p in enumerate(parts):
        st = _dev(np.array([p.mean(), p.std(ddof=1)]))
        L.call("ppx_moments_pack", st.data_ptr(), len(p), recs[r].data_ptr(), L.stream())
    out = torch.empty(2, dtype=torch.float64, device="cuda")
    L.call("ppx_moments_merge", recs.data_ptr(), W, out.data_ptr(), L.stream())
    m, s = _host(out)
    assert abs(m - x.mean()) <= 1e-13 * (abs(x.mean()) + x.std(ddof=1))
    assert abs(s - x.std(ddof=1)) <= 1e-13 * x.std(ddof=1)


def _row_of(i, T, N, n_shard):
    n, t = i // T, i % T
    if n_shard <= 0:
        return t * N + n
    r = n // n_shard
    return (r * T + t) * n_shard + (n - r * n_shard)


class _Rollout:
    """Source fields [T, N, ...] (sharded: [N / n_shard, T, n_shard, ...]) and their flat host copies by storage row."""

    def __init__(self, rs, T, N, fields, n_shard=0):
        self.T, self.N, self.n_shard = T, N, n_shard
        self.host, self.dev = [], []
        for cols in fields:
            a = (rs.randn(T * N, cols) * 2 + 0.5).astype(F32)
            self.host.append(a)
            self.dev.append(_dev(a))

    def run(self, L, idx_dev, B, stats, opts=None, idx_off=0):
        n = len(self.host)
        srcs, dsts, rb = (C.c_void_p * n)(), (C.c_void_p * n)(), (C.c_int * n)()
        outs = []
        for i, a in enumerate(self.dev):
            o = torch.full((B, a.shape[1]), float("nan"), dtype=torch.float32, device="cuda")
            outs.append(o)
            srcs[i], dsts[i], rb[i] = a.data_ptr(), o.data_ptr(), 4 * a.shape[1]
        so = torch.full((len(stats), 2), float("nan"), dtype=torch.float64, device="cuda")
        sf = (C.c_int * len(stats))(*stats)
        sp = (C.c_void_p * len(stats))(*[so[k].data_ptr() for k in range(len(stats))])
        L.call("ppx_gather_minibatch_stats", srcs, dsts, rb, n, idx_dev.data_ptr() + 8 * idx_off, B, self.T, self.N, sf, sp,
               len(stats), C.byref(opts) if opts is not None else None, L.stream())
        return [_host(o) for o in outs], _host(so)

    def check(self, got, st, idx, base, B, stats, stat_range, what):
        """the launch's index slice starts at idx[base]; its statistics cover idx[base + lo : base + hi]"""
        rows = _row_of(idx[base:base + B], self.T, self.N, self.n_shard)
        for f, (a, g) in enumerate(zip(self.host, got)):
            assert np.array_equal(g.view(np.uint32), a[rows].view(np.uint32)), f"{what}: field {f} gathered wrong"
        lo, hi = stat_range
        srows = _row_of(idx[base + lo:base + hi], self.T, self.N, self.n_shard)
        for slot, f in enumerate(stats):
            x64 = self.host[f][srows, 0].astype(F64)
            _onepass_check(st[slot, 0], st[slot, 1], x64, -(-len(x64) // 256) + 24, f"{what}: slot {slot}")


@pytest.mark.parametrize("B", [2, 3, 257, 300000])
def test_gather_stats_row_per_thread(B):
    """Narrow fields on the row-per-thread slice: one slot, then two (dual); a 48-byte field on its own slice; a B whose
    grid reaches the 16 x SMs cap (300000 rows: 3 x 16-byte words each of the wide field); two launches in a row."""
    L = _L()
    rs = np.random.RandomState(B)
    T, N = 512, 1024
    ro = _Rollout(rs, T, N, [1, 1, 12, 2])
    for stats in ([0], [0, 1], [1, 0]):
        for rep in range(2):
            idx = rs.permutation(T * N)[:max(B, 2)].astype(np.int64)
            got, st = ro.run(L, _dev(idx), B, stats)
            ro.check(got, st, idx, 0, B, stats, (0, B), f"B={B} stats={stats} launch {rep}")


@pytest.mark.parametrize("B", [2, 257, 300000])
def test_gather_stats_per_field_slices(B):
    """Fewer than two narrow fields: every field on its own slice, the statistics field finishing on its own."""
    L = _L()
    rs = np.random.RandomState(B + 1)
    T, N = 512, 1024
    ro = _Rollout(rs, T, N, [12, 1])
    for rep in range(2):
        idx = rs.permutation(T * N)[:B].astype(np.int64)
        got, st = ro.run(L, _dev(idx), B, [1])
        ro.check(got, st, idx, 0, B, [1], (0, B), f"B={B} launch {rep}")


@pytest.mark.parametrize("B", [3, 257, 4099])
def test_gather_stats_global_range_and_cursor(B):
    """The sharded "global" range (algorithms.py:640): the local rows [lo, lo + B) of a minibatch of bg rows, statistics
    over all bg (stat_lo = -lo < 0, wider than the slice on both sides), sources in the all-gathered env-shard layout;
    then the device step cursor picks the minibatch (row_dev, n_mb, epoch_stride, mb_stride), with and without a range."""
    L = _L()
    rs = np.random.RandomState(B + 2)
    T, N, W = 64, 1024, 4
    n_shard = N // W
    ro = _Rollout(rs, T, N, [1, 1, 12, 2], n_shard=n_shard)
    total = T * N
    bg = 4 * B + 5
    lo = B + 1
    idx = rs.permutation(total).astype(np.int64)
    for stats in ([0], [0, 1]):
        opts = L.GatherOpts(n_shard, -lo, bg, None, 1, 0, 0)
        got, st = ro.run(L, _dev(idx), B, stats, opts, idx_off=lo)
        ro.check(got, st, idx, lo, B, stats, (-lo, bg - lo), f"global B={B} stats={stats}")
    # device step cursor: epoch e, minibatch j -> idx + e * total + j * Bg
    n_mb, E = -(-total // bg), 2
    perms = np.concatenate([rs.permutation(total) for _ in range(E)]).astype(np.int64)
    pd = _dev(perms)
    cur = torch.zeros(1, dtype=torch.int64, device="cuda")
    assert n_mb >= 4
    for step in (0, 1, n_mb - 2, n_mb, n_mb + 1):                # full minibatches of both epochs
        cur.fill_(step)
        base = (step // n_mb) * total + (step % n_mb) * bg
        opts = L.GatherOpts(0, 0, 0, cur.data_ptr(), n_mb, total, bg)
        plain = _Rollout(np.random.RandomState(step), T, N, [1, 1, 12])
        got, st = plain.run(L, pd, B, [0, 1], opts)
        plain.check(got, st, perms, base, B, [0, 1], (0, B), f"cursor step {step}")
        opts = L.GatherOpts(n_shard, -lo, bg, cur.data_ptr(), n_mb, total, bg)
        got, st = ro.run(L, pd, B, [1], opts, idx_off=lo)
        ro.check(got, st, perms, base + lo, B, [1], (-lo, bg - lo), f"cursor step {step}, global range")


# ----------------------------------------------------------------------------------------------------------------------
# scratch that a captured graph holds
# ----------------------------------------------------------------------------------------------------------------------
def _rnd_learner(D, N, T, seed):
    import ppo_exploration_b200 as ppx
    from test_gpu_device_collect import DeviceTwin, _tables
    np.random.seed(seed)
    torch.manual_seed(seed)
    return ppx.PPO_RND(env=DeviceTwin(_tables(N, D, 4 * T + 1, seed=seed), "box"), nstep=T, batch_size=128, n_epochs=4,
                       hidden_size=64, int_hidden_size=32, rnd_start=8)


def _rnd_phase(m, seed):
    np.random.seed(seed)
    torch.manual_seed(seed)
    m.collect_samples()
    m.train()


def _in_fresh_process(scenario):
    """Runs `scenario` (a function of this module) in a new Python process.  The scratch of ppx_normalize_obs,
    ppx_rnd_normalize_rollout and ppx_knn_novelty is process-wide: in a pytest session the tests before it have already
    grown it past what the scenario's second caller asks for, and nothing would be re-allocated under the graph."""
    import os
    import subprocess
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    root = os.path.dirname(here)
    code = f"import sys; sys.path[:0] = [{root!r}, {here!r}]; import test_gpu_moments_edges as t; t.{scenario.__name__}()"
    args = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", code]
    p = subprocess.run(args, cwd=root, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, f"{scenario.__name__} failed:\n{p.stdout[-3000:]}\n{p.stderr[-6000:]}"


def _assert_first_caller():
    assert _L().launch_count() == 0, "the scenario must start in a process that has launched nothing: its scratch is unsized"


def _rnd_scenario():
    """The first learner (8-wide observations, one env step per bonus call) sizes the istd and moment scratch and
    captures its graphs; the second learner's 200-wide observations and 512-step rollout need more of both."""
    from ppo_exploration_b200.models import _Scratch
    _assert_first_caller()
    runs = []
    for wide in (False, True):
        m = _rnd_learner(8, 64, 16, seed=3)
        _rnd_phase(m, 11)
        _rnd_phase(m, 12)
        assert any(k[0] == "rnd_pred" and isinstance(e, tuple) for k, e in m._graphs.items()), "no rnd_pred graph captured"
        if wide:
            gen = _Scratch.generation
            w = _rnd_learner(200, 16, 8, seed=5)
            obs = torch.randn(512, 16, 200, device="cuda") * 3
            w.rnd_bonus_rollout(obs)
            w.rnd_bonus(obs[0])
            from ppo_exploration_b200 import normalize_obs
            normalize_obs(obs.reshape(-1, 200), w.obs_rms)
            torch.cuda.synchronize()
            assert _Scratch.generation == gen and m._graph_state == m._hp_state(), "the graphs would be re-captured"
        _rnd_phase(m, 13)
        torch.cuda.synchronize()
        runs.append((m.policy.bank.flat.clone(), m.rnd.bank.flat.clone(), m.last_losses.copy(), m.rollout.int_rewards.clone()))
    for a, b in zip(*runs):
        assert (torch.equal(a, b) if isinstance(a, torch.Tensor) else np.array_equal(a, b))


def test_rnd_graph_survives_a_wider_learner():
    """PPO_RND's captured ("rnd_pred", ...) graph normalises through ppx_normalize_obs' scratch.  A second learner with
    25x wider observations (and a longer rollout through ppx_rnd_normalize_rollout) needs more scratch; the first
    learner's next train() replays its graph and must equal, bit for bit, a twin that never saw the second learner.
    Runs in a fresh process, where the first learner is the first caller."""
    _in_fresh_process(_rnd_scenario)


def _es_scenario():
    """2 queries size the candidate scratch (2 x 3 archive slices x K = 10) before the ask graph captures it; 8000
    queries then need 8000 x 1 x 10."""
    import ppo_exploration_b200 as ppx
    _assert_first_caller()
    es = ppx.EvolutionStrategy(hidden_sizes=[16], obs_dim=4, n_actions=2, population_size=8, noise_table_size=1 << 16)
    rs = np.random.RandomState(0)
    archive, queries = _dev(rs.randn(600, 3)), _dev(rs.randn(2, 3))
    want = es.novelty_batch(archive, queries)[1].clone()
    for _ in range(3):
        es.ask(archive, queries)
    assert any(isinstance(e, tuple) for e in es._graphs.values()), "no ask graph captured"
    big_a, big_q = _dev(rs.randn(5000, 3)), _dev(rs.randn(8000, 3))
    big = es.novelty_batch(big_a, big_q)[1]
    nov = es.ask(archive, queries)[2]
    torch.cuda.synchronize()
    assert torch.equal(nov, want)
    assert torch.equal(big, es.novelty_batch(big_a, big_q)[1])


def test_es_ask_graph_survives_a_larger_novelty_batch():
    """The ES ask graph holds ppx_knn_novelty's candidate scratch; a larger novelty_batch grows it, and the next replay
    must still give the eager novelties bit for bit.  Runs in a fresh process, where the ES object is the first caller."""
    _in_fresh_process(_es_scenario)
