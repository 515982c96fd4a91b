"""clip_grad_norm_ + Adam on every path ppx runs it on, checked one step at a time against oracle/optim.py (f64).

ppx restates the reference's optimiser (torch.nn.utils.clip_grad_norm_ + torch.optim.Adam) in four places:
  * ppx_clip_adam (optim.cu: sumsq_kernel + adam_kernel) -- ParamBank.adam_step: the RND predictor (clipped), ICM
    (unclipped) and every policy the fused MLP declines;
  * the cooperative optimiser tail of the fused MLP reduce kernel (mlp_fused.cu) -- _policy_step(fuse_adam=True), on the
    SIMT and on the tcgen05 pair;
  * the fallback of that tail when the reduce grid cannot all be resident: plain reduce, then ppx_clip_adam with the
    reduce's sum-of-squares buffer as its workspace;
  * ppx_clip_adam_pre -- ParamBank.adam_step_pre: the producer of the gradients already left the sum-of-squares partials.

Method, everywhere: teacher-forced per step.  Before a step the device's f32 p, m, v, gradient and step counter are read;
the oracle takes exactly those values, and the device's result is compared after the step.  Rounding noise cannot pile
up, so the bounds are tight:
  exp_avg     |d| <= 1e-6 (|m_ref| + |g_clipped|)
  exp_avg_sq  |d| <= 1e-6 v_ref
  param       |d| <= ulp(p_ref) + 1e-5 * the step's size before exp_avg cancels (oracle.optim.step_scale)
  norm_dev    1e-10 relative;  step_dev exact.
With lr = 1e-2 and |p| <= 0.05 one ulp of p is ~1e-7 of a step, so an error of 1e-4 of one Adam step fails.  The first
test (no GPU) pins the oracle itself to torch's optimiser.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import optim as OO

BETAS, EPS = (0.9, 0.999), 1e-8
LR = 1e-2
SENT = -12345.0                     # guard-band / bank-padding sentinel
GUARD = 1024


# ----------------------------------------------------------------------------------------------------------------------
# shared pieces
# ----------------------------------------------------------------------------------------------------------------------
def _signed_logu(rs, n, lo, hi):
    return np.exp(rs.uniform(np.log(lo), np.log(hi), n)) * rs.choice(np.array([-1.0, 1.0]), n)


def _grads(rs, n, zero_frac=0.05):
    """magnitudes 1e-9 ... 10, mixed signs, some exact zeros"""
    g = _signed_logu(rs, n, 1e-9, 10.0)
    g[rs.rand(n) < zero_frac] = 0.0
    return g.astype(np.float32)


def _moments(rs, n):
    """nonzero exp_avg over 1e-9 ... 1 (so a zero gradient still moves p) and exp_avg_sq >= exp_avg^2"""
    m = _signed_logu(rs, n, 1e-9, 1.0)
    v = (np.abs(m) * np.exp(rs.uniform(0.0, np.log(30.0), n))) ** 2
    return m.astype(np.float32), v.astype(np.float32)


def _within(what, got, ref, tol):
    got = np.asarray(got, np.float64)
    err = np.abs(got - ref)
    bad = ~(err <= tol)
    if bad.any():
        i = int(np.argmax(np.where(bad, err - tol, -np.inf)))
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.size} elements out of bound; worst [{i}]: got {got[i]!r} "
                             f"ref {ref[i]!r} |d| {err[i]:.3e} > tol {tol[i]:.3e}")


def _check_step(what, got, before, t, lr, max_norm=0.0, n_clip=None, extra=None):
    """got = (p, m, v) after the step, before = (p, g, m, v) as the step read them.  Returns (norm, coef) of the oracle."""
    p0, g, m0, v0 = before
    p_ref, m_ref, v_ref, norm, coef = OO.clip_adam(p0, g, m0, v0, t, lr, BETAS, EPS, max_norm, n_clip, extra)
    gc = np.asarray(g, np.float64).copy()
    if norm is not None:
        gc[:(gc.size if n_clip is None else n_clip)] *= coef
    _within(f"{what} exp_avg (t={t})", got[1], m_ref, 1e-6 * (np.abs(m_ref) + np.abs(gc)))
    _within(f"{what} exp_avg_sq (t={t})", got[2], v_ref, 1e-6 * v_ref)
    ulp = np.spacing(np.abs(p_ref).astype(np.float32)).astype(np.float64)
    _within(f"{what} param (t={t})", got[0], p_ref, ulp + 1e-5 * OO.step_scale(gc, m_ref, v_ref, t, lr, BETAS, EPS))
    return norm, coef


def _norm_close(got, want):
    assert abs(float(got) - want) <= 1e-10 * want, (float(got), want)


# ----------------------------------------------------------------------------------------------------------------------
# the oracle against torch (CPU)
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("max_norm", [0.5, 1e6, 0.0], ids=["clip-active", "clip-inactive", "no-clip"])
def test_oracle_matches_torch_adam(max_norm):
    """20 steps of torch.optim.Adam(foreach=False) (+ clip_grad_norm_ unless max_norm = 0) on f32 tensors; before every
    step the oracle is handed torch's own state and must land on torch's result to f32 rounding."""
    rs = np.random.RandomState(7)
    shapes = [(37, 5), (11,), (3, 1)]
    params = [torch.nn.Parameter(torch.from_numpy(rs.uniform(-0.05, 0.05, s).astype(np.float32))) for s in shapes]
    opt = torch.optim.Adam(params, lr=LR, betas=BETAS, eps=EPS, foreach=False)
    flat = lambda ts: np.concatenate([t.detach().reshape(-1).numpy().astype(np.float64) for t in ts])
    coefs = []
    for step in range(1, 21):
        for prm in params:
            prm.grad = torch.from_numpy(_grads(rs, prm.numel()).reshape(prm.shape))
        if step == 5:
            params[1].grad.zero_()                                      # exact zeros with nonzero exp_avg
        st = [opt.state.get(prm, {}) for prm in params]
        p0, g0 = flat(params), flat([prm.grad for prm in params])
        m0 = flat([s["exp_avg"] if s else torch.zeros_like(prm) for s, prm in zip(st, params)])
        v0 = flat([s["exp_avg_sq"] if s else torch.zeros_like(prm) for s, prm in zip(st, params)])
        total = torch.nn.utils.clip_grad_norm_(params, max_norm) if max_norm > 0 else None
        opt.step()
        assert all(float(opt.state[prm]["step"]) == step for prm in params)
        got = (flat(params), flat([opt.state[prm]["exp_avg"] for prm in params]),
               flat([opt.state[prm]["exp_avg_sq"] for prm in params]))
        norm, coef = _check_step(f"torch step {step}", got, (p0, g0, m0, v0), step, LR, max_norm)
        if max_norm > 0:
            assert abs(float(total) - norm) <= 1e-6 * norm
        coefs.append(coef)
    if max_norm == 0.5:
        assert max(coefs) < 1.0
    else:
        assert min(coefs) == 1.0


# ----------------------------------------------------------------------------------------------------------------------
# A. ppx_clip_adam
# ----------------------------------------------------------------------------------------------------------------------
def _c3_bank_size():
    """the C3 policy bank: D = 28 224, h = 128, actor | critic | int_critic, Discrete(18) (about 10.9 M parameters)"""
    from ppo_exploration_b200.models import ParallelMLP
    specs = ParallelMLP.specs(["actor", "critic", "int_critic"], 28224, 128, [18, 1, 1]) + [("action_log_std", (18,))]
    return sum((int(np.prod(s)) + 3) // 4 * 4 for _, s in specs)


def _guarded(a, off, dtype=torch.float32):
    """device copy of `a` at element offset `off` inside a sentinel-filled buffer with a guard band behind it"""
    buf = torch.full((off + a.size + GUARD,), SENT, dtype=dtype, device="cuda")
    buf[off:off + a.size].copy_(torch.from_numpy(a))
    return buf, buf[off:off + a.size]


def _bands_intact(name, buf, off, n):
    assert bool((buf[:off] == SENT).all()) and bool((buf[off + n:] == SENT).all()), f"{name}: wrote outside its {n} elements"


def _ragged(n):
    """an n_clip that ends inside a float4 group of the vector body (n_clip % 4 == 2)"""
    return max(1, min(n - 1, (n // 2) // 4 * 4 + 2))


# (n_clip, max_norm, t, device step counter, all-zero gradient)
CLIP_ADAM_CASES = [
    ("all", "active", 1, True, False),
    ("all", "inactive", 2, False, False),
    ("ragged", "active", 10, True, False),
    ("ragged", "active", 1000, False, False),
    ("none", "active", 1000, True, False),               # n_clip = 0: nothing is clipped even with max_norm > 0
    ("all", "zero", 2, True, False),                     # max_norm = 0
    ("all", "zero", 10, False, False),
    ("all", "active", 1, True, True),
]


@pytest.mark.gpu
@pytest.mark.parametrize("off", [0, 1], ids=["aligned", "offset1"])
@pytest.mark.parametrize("n", [1, 3, 4, 7, 4099, 2 ** 21 + 5, "c3"])
def test_clip_adam(n, off):
    """ppx_clip_adam over n parameters starting `off` floats into their allocations (offset 1: the scalar path only),
    both step forms, every clip branch; the 512-block sum-of-squares cap and the grid-stride loop at the large sizes.
    Guard bands behind p / g / m / v and the workspace stay untouched, the gradient is read-only."""
    from ppo_exploration_b200 import _lib as L
    n = _c3_bank_size() if n == "c3" else n
    rs = np.random.RandomState(n % 1000 + off)
    ws = torch.full((512 + GUARD,), SENT, dtype=torch.float64, device="cuda")
    norm_dev = torch.zeros(1, dtype=torch.float64, device="cuda")
    step_dev = torch.zeros(1, dtype=torch.int64, device="cuda")
    for kind, mode, t, on_dev, zero_grad in CLIP_ADAM_CASES:
        n_clip = {"all": n, "ragged": _ragged(n), "none": 0}[kind]
        p = rs.uniform(-0.05, 0.05, n).astype(np.float32)
        g = np.zeros(n, np.float32) if zero_grad else _grads(rs, n)
        m, v = _moments(rs, n)
        norm_g = float(np.sqrt(np.sum(g[:n_clip].astype(np.float64) ** 2)))
        max_norm = {"active": 0.3 * norm_g if norm_g > 0 else 0.5, "inactive": 10.0 * norm_g + 1.0, "zero": 0.0}[mode]
        bufs = [_guarded(a, off) for a in (p, g, m, v)]
        (pb, pd), (gb, gd), (mb, md), (vb, vd) = bufs
        step_dev.fill_(t - 1)
        norm_dev.fill_(-1.0)
        L.call("ppx_clip_adam", pd.data_ptr(), gd.data_ptr(), md.data_ptr(), vd.data_ptr(), n, float(max_norm), n_clip, LR,
               BETAS[0], BETAS[1], EPS, 0 if on_dev else t, step_dev.data_ptr() if on_dev else None, norm_dev.data_ptr(),
               ws.data_ptr(), L.stream())
        torch.cuda.synchronize()
        what = f"n={n} off={off} n_clip={n_clip} max_norm={max_norm:.3g} t={t} dev={on_dev}"
        norm, coef = _check_step(what, (pd.cpu().numpy(), md.cpu().numpy(), vd.cpu().numpy()), (p, g, m, v), t, LR,
                                 max_norm, n_clip)
        if mode == "active" and kind != "none" and norm_g > 0:
            assert coef < 1.0, what
        if mode == "inactive":
            assert coef == 1.0, what
        if norm is not None:
            _norm_close(norm_dev.item(), norm)
        if on_dev:
            assert int(step_dev.item()) == t, f"{what}: step_dev {int(step_dev.item())}, want {t}"
        assert np.array_equal(gd.cpu().numpy(), g), f"{what}: the gradient was modified"
        for name, (b, _) in zip("pgmv", bufs):
            _bands_intact(f"{what} {name}", b, off, n)
        assert bool((ws[512:] == SENT).all()), f"{what}: workspace guard"


# ----------------------------------------------------------------------------------------------------------------------
# B. ppx_clip_adam_pre
# ----------------------------------------------------------------------------------------------------------------------
# (partials, extra gradients, max_norm, t): "extras" puts max_norm between the norm of g and the norm of g + extras,
# so the coefficient is 1 unless the extras enter the norm
PRE_CASES = [(1, 0, "active", 1), (37, 5, "extras", 2), (1, 3, "extras", 10), (37, 0, "inactive", 1000), (512, 2, "active", 3)]


@pytest.mark.gpu
@pytest.mark.parametrize("off", [0, 1], ids=["aligned", "offset1"])
@pytest.mark.parametrize("n", [7, 4099, 2 ** 21 + 5])
def test_clip_adam_pre(n, off):
    """ppx_clip_adam_pre: the norm comes from caller-supplied f64 sum-of-squares partials plus the extra gradients (which
    the kernel reads, never writes), the coefficient scales all n gradients, and step_dev -- already bumped by the
    producer of the partials -- is used as it is."""
    from ppo_exploration_b200 import _lib as L
    rs = np.random.RandomState(n + off)
    norm_dev = torch.zeros(1, dtype=torch.float64, device="cuda")
    step_dev = torch.zeros(1, dtype=torch.int64, device="cuda")
    for n_part, n_extra, mode, t in PRE_CASES:
        p = rs.uniform(-0.05, 0.05, n).astype(np.float32)
        g = _grads(rs, n)
        m, v = _moments(rs, n)
        g64 = g.astype(np.float64)
        norm_g = float(np.sqrt(np.sum(g64 ** 2)))
        extra = None
        if n_extra:
            e = rs.randn(n_extra)
            extra = (e * np.sqrt(8.0) * norm_g / np.linalg.norm(e)).astype(np.float32)     # |g, extras| = 3 |g|
        max_norm = {"active": 0.3 * norm_g, "extras": 2.0 * norm_g, "inactive": 10.0 * norm_g}[mode]
        partials = np.array([np.sum(c ** 2) for c in np.array_split(g64, n_part)])
        bufs = [_guarded(a, off) for a in (p, g, m, v)]
        (pb, pd), (gb, gd), (mb, md), (vb, vd) = bufs
        pa_b, pa = _guarded(partials, 0, torch.float64)
        ex_b, ex = _guarded(extra, 0) if extra is not None else (None, None)
        step_dev.fill_(t)
        L.call("ppx_clip_adam_pre", pd.data_ptr(), gd.data_ptr(), md.data_ptr(), vd.data_ptr(), n, float(max_norm), LR,
               BETAS[0], BETAS[1], EPS, step_dev.data_ptr(), norm_dev.data_ptr(), pa.data_ptr(), n_part,
               ex.data_ptr() if ex is not None else None, n_extra, L.stream())
        torch.cuda.synchronize()
        what = f"n={n} off={off} partials={n_part} extras={n_extra} {mode} t={t}"
        norm, coef = _check_step(what, (pd.cpu().numpy(), md.cpu().numpy(), vd.cpu().numpy()), (p, g, m, v), t, LR,
                                 max_norm, None, extra)
        assert coef < 1.0 if mode != "inactive" else coef == 1.0, what
        _norm_close(norm_dev.item(), norm)
        assert int(step_dev.item()) == t, what
        assert np.array_equal(gd.cpu().numpy(), g), what
        for name, (b, _) in zip("pgmv", bufs):
            _bands_intact(f"{what} {name}", b, off, n)
        _bands_intact(f"{what} partials", pa_b, 0, n_part)
        if ex is not None:
            assert np.array_equal(ex.cpu().numpy(), extra)
            _bands_intact(f"{what} extras", ex_b, 0, n_extra)


# ----------------------------------------------------------------------------------------------------------------------
# C. the optimiser tail of the fused MLP backward
# ----------------------------------------------------------------------------------------------------------------------
def _space(spec):
    import ppo_exploration_b200 as ppx
    kind, k = spec
    return ppx.Box((k,)) if kind == "Box" else ppx.Discrete(k)


def _policy(D, h, space, intrinsic, seed=0):
    import ppo_exploration_b200 as ppx
    env = ppx.SyntheticVecEnv(4, D, _space(space), seed=0)
    torch.manual_seed(seed)
    return ppx.models.Policy(env, h, intrinsic_model=intrinsic, device="cuda")


def _fused_blocks(pol):
    """ppx_mlp3_fused_adam_blocks: > 0 = the cooperative tail runs, 0 = plain reduce + ppx_clip_adam"""
    from ppo_exploration_b200 import _lib as L
    mlp = pol.mlp
    return int(L.call("ppx_mlp3_fused_adam_blocks", mlp.D, mlp.h, mlp.G, (C.c_int * mlp.G)(*mlp.outs)))


def _real_mask(bank):
    """True on the elements that belong to a named tensor, False on the bank's alignment padding"""
    mask = np.zeros(bank.size, bool)
    for name, o in bank.offsets.items():
        mask[o:o + int(np.prod(bank.shapes[name]))] = True
    return mask


# (id, D, h, action space, three nets, tcgen05 pair)
TAIL_CFGS = [
    ("tc-h64-G2-box", 8, 64, ("Box", 2), False, True),
    ("tc-h64-G3-discrete", 8, 64, ("Discrete", 3), True, True),
    ("simt-h64-G2-box", 8, 64, ("Box", 2), False, False),
    ("h128-G2-D4-discrete2", 4, 128, ("Discrete", 2), False, False),     # C1
    ("h128-G2-D8-discrete3", 8, 128, ("Discrete", 3), False, False),    # the widest h = 128 input the fused pair takes
    ("h128-G3-box", 8, 128, ("Box", 2), True, False),                    # PPO_RND's default policy
]


def _tail_policy(cfg):
    name, D, h, space, intrinsic, tc = cfg
    pol = _policy(D, h, space, intrinsic)
    fa = pol.mlp._fused_args()
    assert fa["ok"], name
    if tc:
        assert fa["tc"], f"{name}: the tensor-core pair must be the one under test"
    fa["tc"] = tc
    return pol


@pytest.mark.gpu
def test_tail_configs_cover_both_paths():
    """Which shapes get the cooperative tail depends on how many reduce blocks the device keeps resident; the h = 64
    shapes always do, and the set under test must contain at least one fallback."""
    blocks = {cfg[0]: _fused_blocks(_tail_policy(cfg)) for cfg in TAIL_CFGS}
    print("fused optimiser tail: " + ", ".join(f"{k}: {'cooperative' if b else 'fallback'} ({b})" for k, b in blocks.items()))
    assert all(blocks[c[0]] > 0 for c in TAIL_CFGS if c[2] == 64), blocks
    assert any(b > 0 for b in blocks.values()) and any(b == 0 for b in blocks.values()), blocks


def _bank_state(bank):
    torch.cuda.synchronize()
    return (bank.flat.cpu().numpy(), bank.grad.cpu().numpy(), bank.exp_avg.cpu().numpy(), bank.exp_avg_sq.cpu().numpy(),
            int(bank.step_dev.item()))


def _check_bank(what, bank, before, lr, max_norm, real=None):
    """the step the bank just took, against the oracle applied to `before` and the gradient the bank holds now"""
    p0, _, m0, v0, t0 = before
    p, g, m, v, t = _bank_state(bank)
    assert t == t0 + 1, f"{what}: step_dev {t0} -> {t}"
    norm, coef = _check_step(what, (p, m, v), (p0, g, m0, v0), t, lr, max_norm)
    if norm is not None:
        _norm_close(bank.norm_dev.item(), norm)
    if real is not None:                                         # padding: never part of the update
        pad = ~real
        assert np.array_equal(p[pad], p0[pad]) and not m[pad].any() and not v[pad].any() and not g[pad].any(), what
    return coef


@pytest.mark.gpu
@pytest.mark.parametrize("max_norm", [0.2, 1e6, 0.0], ids=["clip-active", "clip-inactive", "no-clip"])
@pytest.mark.parametrize("cfg", TAIL_CFGS, ids=[c[0] for c in TAIL_CFGS])
def test_fused_tail(cfg, max_norm):
    """ParallelMLP.backward(with_sumsq=True, adam=bank.fused_adam(...)): three eager calls, then a captured CUDA graph
    replayed twice.  Every step: the gradient equals the same backward without the tail bit for bit, the step counter
    advances once, the rendezvous counters are re-armed, the update matches the oracle (norm over the MLP gradients plus
    action_log_std's), and the bank padding is left alone."""
    name, D, h, space, intrinsic, tc = cfg
    pol = _tail_policy(cfg)
    bank, mlp = pol.bank, pol.mlp
    coop = _fused_blocks(pol) > 0
    if h == 64:
        assert coop, name
    rs = np.random.RandomState(D * h + int(max_norm))
    real = _real_mask(bank)
    k = int(real.sum())
    p = np.full(bank.size, SENT, np.float32)
    p[real] = rs.uniform(-0.05, 0.05, k)
    m, v = np.zeros(bank.size, np.float32), np.zeros(bank.size, np.float32)
    m[real], v[real] = _moments(rs, k)
    for dst, a in ((bank.flat, p), (bank.exp_avg, m), (bank.exp_avg_sq, v)):
        dst.copy_(torch.from_numpy(a))
    bank.grad.zero_()
    t_first = {0.2: 1, 1e6: 10, 0.0: 1000}[max_norm]
    bank.step_dev.fill_(t_first - 1)
    gen = torch.Generator().manual_seed(5)
    M = 300
    x = torch.randn(M, D, generator=gen).cuda()
    d_outs = [torch.randn(M, o, generator=gen).cuda() for o in pol.outs]
    A, o_als = pol.action_dim, bank.offsets["action_log_std"]
    als_grad = torch.tensor([3.0, -40.0] if space[0] == "Box" else [0.0] * A, dtype=torch.float32, device="cuda")
    rec = bank.fused_adam(LR, max_norm, extra_name="action_log_std")

    def step(run, label):
        bank.grad[o_als:o_als + A].copy_(als_grad)                 # written by the loss head in the learners
        mlp.backward(d_outs, with_sumsq=False)
        g_plain = bank.grad.clone()
        before = _bank_state(bank)
        run()
        torch.cuda.synchronize()
        what = f"{name} {'cooperative' if coop else 'fallback'} max_norm={max_norm} {label}"
        assert torch.equal(bank.grad, g_plain), f"{what}: the tail changed the gradient"
        assert bank._ticket.tolist() == [0, 0], what
        coef = _check_bank(what, bank, before, LR, max_norm, real)
        assert coef < 1.0 if max_norm == 0.2 else coef == 1.0, what

    tail = lambda: mlp.backward(d_outs, with_sumsq=True, adam=rec)
    for call in range(3):
        pol.forward_raw(x)
        step(tail, f"eager call {call}")
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        tail()
    for r in range(2):
        step(graph.replay, f"graph replay {r}")
    assert int(bank.step_dev.item()) == t_first + 4


# ----------------------------------------------------------------------------------------------------------------------
# D. the learners, end to end
# ----------------------------------------------------------------------------------------------------------------------
T_LRN, N_LRN = 16, 8
# (id, learner, D, action space, constructor arguments, policy on the fused MLP pair)
LEARNERS = [
    ("ppo-h64-box", "PPO", 8, ("Box", 2), dict(hidden_size=64), True),
    ("ppo-h128-discrete", "PPO", 4, ("Discrete", 2), dict(hidden_size=128), True),
    # h = 128 with D = 32 and 18 actions needs more shared memory than the fused pair has: layer by layer + adam_step
    ("ppo-h128-D32-discrete18", "PPO", 32, ("Discrete", 18), dict(hidden_size=128), False),
    ("rnd-defaults", "PPO_RND", 8, ("Box", 2), dict(), True),                          # h = 128, three nets: the fallback
    ("icm-defaults", "PPO_ICM", 8, ("Discrete", 3), dict(), True),
    ("rnd-wide", "PPO_RND", 1024, ("Discrete", 4), dict(int_hidden_size=16), False),   # tensor-core weight shadows
]


def _rnd_decisions(seed, calls, total):
    """PPO_RND.train's host draws with one minibatch per call: np.random.permutation(T*N), then one randn() < 0.25"""
    st = np.random.get_state()
    np.random.seed(seed)
    out = []
    for _ in range(calls):
        np.random.permutation(total)
        out.append(bool(np.random.randn() < 0.25))
    np.random.set_state(st)
    return out


def _learner(kind, D, space, kw, seed):
    import ppo_exploration_b200 as ppx
    np.random.seed(seed)
    torch.manual_seed(seed)
    env = ppx.SyntheticVecEnv(N_LRN, D, _space(space), seed=1)
    extra = dict(int_lr=LR) if kind != "PPO" else {}
    m = getattr(ppx, kind)(env=env, nstep=T_LRN, batch_size=T_LRN * N_LRN, n_epochs=1, lr=LR, **extra, **kw)
    ro = m.rollout
    rs = np.random.RandomState(seed)
    T, N = T_LRN, N_LRN
    if space[0] == "Box":
        actions = rs.randn(*ro.actions.shape)
    else:
        actions = rs.randint(0, space[1], size=tuple(ro.actions.shape)).astype(np.float64)
    arrs = dict(observations=rs.randn(T, N, D).astype(np.float32), actions=actions, rewards=rs.randn(T, N).astype(np.float32),
                values=rs.randn(T, N).astype(np.float32), masks=(rs.rand(T, N) < 0.05).astype(np.uint8),
                action_log_probs=(-1.0 + 0.3 * rs.randn(*ro.action_log_probs.shape)).astype(np.float32))
    lv = rs.randn(N).astype(np.float32)
    if kind == "PPO_RND":
        arrs.update(int_values=rs.randn(T, N).astype(np.float32), int_rewards=np.abs(rs.randn(T, N)).astype(np.float32))
        ro.load_rollout(**arrs)
        ro.compute_returns_and_advantages(torch.tensor(lv), torch.tensor(rs.randn(N).astype(np.float32)), arrs["masks"][-1])
    else:
        ro.load_rollout(**arrs)
        ro.compute_returns_and_advantages(torch.tensor(lv), arrs["masks"][-1])
    return m


def _shadows_exact(what, bank):
    for tw in bank.tc_weights:
        o = (tw.w_ptr - bank.flat.data_ptr()) // 4
        W = bank.flat[o:o + tw.K * tw.N].view(tw.K, tw.N)
        assert torch.equal(tw.hiT + tw.loT, W.t()), f"{what}: tensor-core shadow of a {tw.K}x{tw.N} weight is stale"
        if tw.hi is not None:
            assert torch.equal(tw.hi + tw.lo, W), f"{what}: tensor-core shadow of a {tw.K}x{tw.N} weight is stale"


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", LEARNERS, ids=[c[0] for c in LEARNERS])
def test_learner_optimiser_steps(cfg):
    """One minibatch per train() (batch_size = T*N, one epoch), train() called six times on the same loaded rollout:
    eager, then captured, then replayed, for each of the two permutation staging sets.  Each call, every bank against the
    oracle applied to its snapshot and to the gradient left in bank.grad: the policy clipped with max_grad_norm (its norm
    includes action_log_std), the RND predictor clipped with max_grad_norm and untouched -- step counter included -- when
    the call drew no RND update (torch skips rnd_opt.step()), the ICM bank unclipped.  Tensor-core weight shadows equal
    the new weights after every step."""
    name, kind, D, space, kw, fused = cfg
    calls = 6
    seed = 0
    if kind == "PPO_RND":                                        # a seed whose calls include RND updates and skips
        seed = next(s for s in range(100) if len(set(_rnd_decisions(s, calls, T_LRN * N_LRN))) == 2)
    m = _learner(kind, D, space, kw, seed)
    assert m.policy.mlp.fused() == fused, name
    pol_bank = m.policy.bank
    banks = [("policy", pol_bank, m.lr, m.max_grad_norm)]
    if kind == "PPO_RND":
        banks.append(("rnd", m.rnd.bank, m.int_lr, m.max_grad_norm))
    if kind == "PPO_ICM":
        banks.append(("icm", m.intrinsic_module.bank, m.int_lr, 0.0))
    if D >= 256:
        assert pol_bank.tc_weights and m.rnd.bank.tc_weights, "the wide case must carry tensor-core shadows"
    real = {b[0]: _real_mask(b[1]) for b in banks}
    rnd_pattern = []
    np.random.seed(seed)
    for call in range(calls):
        before = {b[0]: _bank_state(b[1]) for b in banks}
        m.train()
        for label, bank, lr, max_norm in banks:
            what = f"{name} {label} train() call {call}"
            if label == "rnd" and m.rnd_trained_steps == 0:
                p, g, mm, v, t = _bank_state(bank)
                p0, g0, m0, v0, t0 = before[label]
                assert t == t0 and np.array_equal(p, p0) and np.array_equal(mm, m0) and np.array_equal(v, v0), \
                    f"{what}: no RND update was drawn, yet the bank moved"
                continue
            coef = _check_bank(what, bank, before[label], lr, max_norm, real[label])
            if max_norm > 0:
                assert coef < 1.0, f"{what}: the clip must be active for this check to mean anything"
            _shadows_exact(what, bank)
        if kind == "PPO_RND":
            rnd_pattern.append(m.rnd_trained_steps > 0)
    if kind == "PPO_RND":
        assert len(set(rnd_pattern)) == 2, rnd_pattern
    policy_keys = [k for k in m._graphs if k[0] in ("ppo", "rnd_policy", "icm")]
    assert policy_keys and all(isinstance(m._graphs[k], tuple) for k in policy_keys), "train() never reached graph replay"
