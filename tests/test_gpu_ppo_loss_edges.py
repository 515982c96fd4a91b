"""The fused PPO loss kernels (ppo_loss.cu) and the ICM / RND loss pieces (ppo_loss.cu, bonus.cu) against float64
references, at the clip, branch and sharding edges the train-parity tests almost never reach.

The head reference restates oracle/learner.py (_surrogate, _clipped_value_loss and the Categorical / Normal parts of
evaluate) with torch autograd in float64 on the same f32-valued inputs the kernel sees; actor_out is the leaf.  Two pieces
of the reference's own f32 arithmetic are kept as they are in float32: the advantage normalisation (algorithms.py:219 runs
on f32 tensors; the kernel gets {mean, unbiased std} computed here in f64 and normalises in f32 exactly like torch), and
torch.distributions' probability clamp, which uses finfo(float32).eps because the reference's probabilities are f32.

Decisions.  Random inputs keep every f32 decision of the kernel clear of its boundary, and the tests assert it: each
surrogate ratio at least 1e-3 (relative) away from 1 +- clip, each |v - v_old| at least 1e-3 clip away from clip, the two
value means at least 1e-4 (relative) apart.  The only inputs on a boundary are built to be exact: values == old_values
(an exact tie of the value means, split 0.5 / 0.5), old_values = 0 with values = +-f32(clip) (the inclusive value-clip
edge), and ratios of exactly 1 at clip_range = 0 (the inclusive surrogate-clip edge): Box inputs whose log-prob is
IEEE-exact to replay on the host (_exact_ratio_one), Discrete old log-probs that the head itself reads back as a ratio of
exactly 1 (_head_ratio_probe).

Tolerances.  The kernel is f64 on the Box surrogate path and f32 elsewhere: softmax, log, the value errors and every
per-row gradient are single f32 operations or short f32 chains (relative error a few 1e-7), the per-row terms are summed in
f64.  So each gradient array is checked to 1e-5 * max|ref| + 1e-7 (about 30x the f32 chain error), the loss scalars to
1e-6 relative with an absolute floor of 1e-9 * the largest loss.  The policy loss (and the total) also gets a floor of
3e-7 * mean|adv * ratio|: it is a mean of terms of both signs that can cancel (to ~1e-8 in the first epoch, where it is
-mean(adv)), and no mean can be closer than the f32 log-probs of its terms, each within ~2e-7 of the f64 one.
A gradient routed through the wrong branch of a clip or a max is off by O(1) of its own size and fails these bounds by
four orders of magnitude.
"""
import ctypes as C
import warnings

import numpy as np
import pytest
import torch

from conftest import Golden
from oracle import learner as OL
from oracle import rollout as OR

pytestmark = pytest.mark.gpu

EPS32 = float(np.finfo(np.float32).eps)           # torch.distributions.utils.clamp_probs on f32 probabilities
CLIP = float(np.float32(0.2))                     # the kernel receives the f32 clip_range
HALF_LOG_2PI = 0.91893853320467274178
IN_KEYS = ("actor_out", "log_std", "actions", "old_lp", "adv", "adv_stats", "values", "old_values", "returns",
           "int_adv", "int_adv_stats", "int_values", "old_int_values", "int_returns")


def _L():
    from ppo_exploration_b200 import _lib as L
    return L


def _grid_cap():
    return min(1024, 2 * torch.cuda.get_device_properties(0).multi_processor_count)


# ----------------------------------------------------------------------------------------------------------------------
# cases: f32 / f64 host arrays with every decision clear of its boundary, or exactly on it
# ----------------------------------------------------------------------------------------------------------------------
def _stats(a):
    a = np.asarray(a, np.float64)
    return (float(a.mean()), float(a.std(ddof=1))) if a.size >= 2 else (0.25, 1.5)


def _norm_adv(a, st):
    """algorithms.py:219 in f32 with the statistics handed in (the kernel casts them to f32 the same way)"""
    return (a - np.float32(st[0])) / (np.float32(st[1]) + np.float32(1e-8))


def _logprob(c, actor_out=None):
    """the head's own log-probability, numpy f64 from the f32 inputs: [B] (Discrete) or [B, A] (Box)"""
    x = np.asarray(c["actor_out"] if actor_out is None else actor_out, np.float64)
    if c["discrete"]:
        e = np.exp(x - x.max(1, keepdims=True))
        q = e / e.sum(1, keepdims=True)
        q = q / q.sum(1, keepdims=True)
        lq = np.log(np.clip(q, EPS32, 1 - EPS32))
        return lq[np.arange(len(x)), c["actions"].astype(np.int64)]
    mu, sd = np.tanh(x), np.exp(np.asarray(c["log_std"], np.float64))
    return -(c["actions"] - mu) ** 2 / (2 * sd * sd) - np.log(sd) - HALF_LOG_2PI


def _ratios(rs, shape, clip):
    """target ratios: 0 inside the window, 1 above 1 + clip, 2 below 1 - clip, drawn well clear of both edges"""
    side = rs.randint(0, 3, shape)
    r = np.where(side == 0, rs.uniform(1 - 0.7 * clip, 1 + 0.7 * clip, shape),
                 np.where(side == 1, rs.uniform(1 + 1.5 * clip, 1 + 4 * clip, shape),
                          rs.uniform(max(0.05, 1 - 4 * clip), 1 - 1.5 * clip, shape)))
    return r


def _value_arrays(rs, B, clip, mode, v=None):
    """(values, old_values, returns) f32 [B] and the row kinds: 0 inside the value-clip window, 1 above it, 2 below it,
    3 exactly on its edge (old_values = 0, values = +-f32(clip)).  mode: 'w1' the unclipped mean is the larger (returns
    beyond the clipped value), 'w0' the clipped one (returns beyond the value), 'tie' values == old_values off the edge
    rows (an exact tie of the means), 'mixed' returns anywhere.  `v` (optional) fixes the values; the edge rows are then
    those where old_values = v -+ clip makes v - old_values exactly +-clip.  clip = 0 has no inside: v == v_old is the
    edge."""
    clip32 = np.float32(clip)
    kind = (np.arange(B) + 1) % 4 if B <= 4 else rs.randint(0, 4, B)
    if v is not None:                                   # about half the edge candidates can be made exact
        kind = rs.choice(4, B, p=[0.2, 0.2, 0.2, 0.4])
    if clip == 0:
        kind[kind == 0] = 3
    w = clip if clip > 0 else 0.2
    d = np.where(kind == 0, rs.uniform(-0.7, 0.7, B) * clip,
                 np.where(kind == 1, rs.uniform(1.5, 4, B) * w, -rs.uniform(1.5, 4, B) * w))
    sgn = np.where(rs.rand(B) < 0.5, np.float32(-1), np.float32(1))
    edge = kind == 3
    if v is None:
        v = rs.randn(B).astype(np.float32)
        v[edge] = sgn[edge] * clip32
        ov = (v - d).astype(np.float32)
        ov[edge] = 0.0
    else:
        v = np.asarray(v, np.float32)
        ov = (v - d).astype(np.float32)                 # an edge row that cannot be made exact stays below the window
        e = (v - sgn * clip32).astype(np.float32)
        exact = np.asarray(v, np.float64) - np.asarray(e, np.float64) == np.asarray(sgn, np.float64) * np.float64(clip32)
        ov[edge & exact] = e[edge & exact]
        kind[edge & ~exact] = 2
    if mode == "tie":
        ov[kind != 3] = v[kind != 3]
        kind[kind != 3] = 0
    vc = np.asarray(ov, np.float64) + np.clip(np.asarray(v, np.float64) - np.asarray(ov, np.float64), -clip, clip)
    u = rs.uniform(0.2, 1.0, B)
    R = np.asarray(v, np.float64) + 0.8 * rs.randn(B)
    out = (kind == 1) | (kind == 2)
    away = np.sign(np.asarray(v, np.float64) - vc)
    if mode == "w1":
        R[out] = (vc - away * u)[out]
    elif mode == "w0":
        R[out] = (np.asarray(v, np.float64) + away * u)[out]
    return v, ov, R.astype(np.float32), kind


def _case(B, A, discrete, dual=False, *, seed=0, clip=CLIP, pw=1.0, ent_coef=0.01, vf_coef=0.5, int_vf_coef=0.7,
          value_mode="mixed", actor_scale=None):
    rs = np.random.RandomState(seed)
    c = dict(B=B, A=A, discrete=bool(discrete), dual=bool(dual), clip=float(np.float32(clip)), pw=pw, ent_coef=ent_coef,
             vf_coef=vf_coef, int_vf_coef=int_vf_coef)
    if discrete:
        c["actor_out"] = ((1.5 if actor_scale is None else actor_scale) * rs.randn(B, A)).astype(np.float32)
        c["log_std"] = None
        c["actions"] = rs.randint(0, A, B).astype(np.float64)
    else:
        c["actor_out"] = ((0.8 if actor_scale is None else actor_scale) * rs.randn(B, A)).astype(np.float32)
        c["log_std"] = rs.uniform(-0.5, 0.3, A).astype(np.float32)
        mu, sd = np.tanh(c["actor_out"].astype(np.float64)), np.exp(c["log_std"].astype(np.float64))
        c["actions"] = mu + sd * rs.randn(B, A)
    c["adv"] = (2.0 * rs.randn(B) + 0.3).astype(np.float32)
    c["adv_stats"] = _stats(c["adv"])
    c["values"], c["old_values"], c["returns"], c["vkind"] = _value_arrays(rs, B, c["clip"], value_mode)
    if dual:
        c["int_adv"] = (0.7 * rs.randn(B) - 0.2).astype(np.float32)
        c["int_adv_stats"] = _stats(c["int_adv"])
        c["int_values"], c["old_int_values"], c["int_returns"], c["ivkind"] = _value_arrays(rs, B, c["clip"], value_mode)
    else:
        for k in ("int_adv", "int_adv_stats", "int_values", "old_int_values", "int_returns"):
            c[k] = None
    lp = _logprob(c)
    c["old_lp"] = (lp - np.log(_ratios(rs, lp.shape, c["clip"]))).astype(np.float32)
    return c


def _adv_n(c):
    a = _norm_adv(c["adv"], c["adv_stats"])
    if c["dual"]:
        a = a + _norm_adv(c["int_adv"], c["int_adv_stats"])                 # algorithms.py:431-434, in f32
    return a


# ----------------------------------------------------------------------------------------------------------------------
# the float64 reference
# ----------------------------------------------------------------------------------------------------------------------
def _ref_losses(c, actor_out, log_std, values, int_values):
    """(total, policy, value, entropy, int_value) as f64 tensors, plus the ratio and the value means (detached)"""
    f64 = lambda a: torch.as_tensor(np.asarray(a, np.float64))
    clip = c["clip"]
    adv = f64(_adv_n(c))[:, None]
    if c["discrete"]:
        # Categorical(probs=softmax(x)): probs renormalised, logits = log(clamp_probs(probs))   models.py:58-64
        q = torch.softmax(actor_out, dim=-1)
        q = q / q.sum(-1, keepdim=True)
        lq = torch.log(q.clamp(EPS32, 1 - EPS32))
        lp = lq.gather(1, f64(c["actions"]).long()[:, None])
        ent = -(lq * q).sum(-1)
        old_lp = f64(c["old_lp"])[:, None]
    else:
        # Normal(tanh(x), exp(log_std)).log_prob / .entropy, models.py:66-71, written out: torch's log(sqrt(2 pi)) is one
        # ulp below the correctly rounded constant the kernel uses, and an exact ratio of 1 must stay exact here too
        mu, scale = torch.tanh(actor_out), torch.exp(log_std).expand_as(actor_out)
        lp = -((f64(c["actions"]) - mu) ** 2) / (2 * scale ** 2) - torch.log(scale) - HALF_LOG_2PI
        ent = 0.5 + HALF_LOG_2PI + torch.log(scale)
        old_lp = f64(c["old_lp"])
    pl = OL._surrogate(adv, lp, old_lp, clip)
    vl = OL._clipped_value_loss(f64(c["returns"]), values, f64(c["old_values"]), clip)
    el = -torch.mean(ent)
    total = c["pw"] * (pl + c["ent_coef"] * el + c["vf_coef"] * vl)
    ivl = torch.zeros((), dtype=torch.float64)
    if c["dual"]:
        ivl = OL._clipped_value_loss(f64(c["int_returns"]), int_values, f64(c["old_int_values"]), clip)
        total = total + c["int_vf_coef"] * ivl

    def means(R, v, ov):
        v, R, ov = v.detach(), f64(R), f64(ov)
        vc = ov + (v - ov).clamp(-clip, clip)
        return float(((R - v) ** 2).mean()), float(((R - vc) ** 2).mean())
    ratio = torch.exp(lp - old_lp).detach()
    aux = dict(ratio=ratio.numpy(), pl_scale=float((adv * ratio).abs().mean()), m=means(c["returns"], values, c["old_values"]),
               im=means(c["int_returns"], int_values, c["old_int_values"]) if c["dual"] else None)
    return (total, pl, vl, el, ivl), aux


def _reference(c):
    f64 = lambda a: torch.tensor(np.asarray(a, np.float64), requires_grad=True)
    ao, v = f64(c["actor_out"]), f64(c["values"])
    ls = None if c["discrete"] else f64(c["log_std"])
    iv = f64(c["int_values"]) if c["dual"] else None
    losses, aux = _ref_losses(c, ao, ls, v, iv)
    losses[0].backward()
    ref = dict(losses=np.array([float(x) for x in losses]), d_actor=ao.grad.numpy(), d_values=v.grad.numpy(),
               d_log_std=None if ls is None else ls.grad.numpy(), d_int_values=iv.grad.numpy() if c["dual"] else None)
    w = lambda m: 1.0 if m[0] > m[1] else (0.0 if m[0] < m[1] else 0.5)
    ref["branch"] = np.array([w(aux["m"]), 1 - w(aux["m"])] + ([w(aux["im"]), 1 - w(aux["im"])] if c["dual"] else [0.0, 1.0]))
    ref.update(aux)
    return ref


def _assert_margins(c, ref, exact_ratio=None, value_tie=False):
    """every f32 decision of the kernel is clear of its boundary (or on it by construction)"""
    clip, r = c["clip"], ref["ratio"].reshape(c["B"], -1)
    if clip > 0:
        for edge in (1 - clip, 1 + clip):
            assert np.all(np.abs(r - edge) >= 1e-3 * edge), f"ratio within 1e-3 of {edge}"
    else:
        assert exact_ratio is not None
        assert np.all((np.abs(r - 1) >= 1e-3) | exact_ratio), "clip_range = 0: a ratio near 1 that is not exactly 1"
    for pre, m in (("", ref["m"]), ("int_", ref["im"])):
        if m is None:
            continue
        if value_tie:
            assert m[0] == m[1], "the value means are not an exact tie"
        else:
            assert abs(m[0] - m[1]) >= 1e-4 * max(m[0], m[1]), f"{pre}value means {m} within 1e-4"
        kind = c["vkind" if pre == "" else "ivkind"]
        d = np.abs(np.asarray(c[pre + "values"], np.float64) - np.asarray(c["old_" + pre + "values"], np.float64))
        off = kind != 3
        if clip > 0:
            assert np.all(np.abs(d[off] - clip) >= 1e-3 * clip), "|v - v_old| near the value-clip edge"
        else:
            assert np.all(d[off] >= 1e-3), "clip_range = 0: |v - v_old| near 0 off the edge rows"
        assert np.all(d[~off] == clip), "edge rows are not exactly on the edge"


# ----------------------------------------------------------------------------------------------------------------------
# device calls
# ----------------------------------------------------------------------------------------------------------------------
def _upload(c):
    def t(k):
        a = c[k]
        if a is None:
            return None
        dt = torch.float64 if k in ("actions", "adv_stats", "int_adv_stats") else torch.float32
        return torch.as_tensor(np.ascontiguousarray(np.asarray(a, np.float64 if dt == torch.float64 else np.float32))).to("cuda", dt)
    return {k: t(k) for k in IN_KEYS}


def _ptrs(d, lo=0, hi=None):
    """input pointers, rows [lo, hi) of the per-row arrays"""
    out = []
    for k in IN_KEYS:
        a = d[k]
        if a is None:
            out.append(None)
        elif k in ("log_std", "adv_stats", "int_adv_stats"):
            out.append(a.data_ptr())
        else:
            out.append(a[lo:hi].data_ptr())
    return out


def _cfg(c, B=None, B_total=0, row_dev=None, row_hold=0):
    L = _L()
    return L.PpoCfg(c["B"] if B is None else B, B_total, c["A"], int(c["discrete"]), int(c["dual"]), c["clip"],
                    c["ent_coef"], c["vf_coef"], c["int_vf_coef"], c["pw"], row_dev, row_hold)


def _outs(c, B=None):
    B = c["B"] if B is None else B
    nan = lambda n, dt=torch.float32: torch.full((n,), float("nan"), dtype=dt, device="cuda")
    ws = _L().call("ppx_ppo_loss_workspace", B, c["A"])
    return dict(d_actor=nan(B * c["A"]), d_log_std=None if c["discrete"] else nan(c["A"]), d_values=nan(B),
                d_int_values=nan(B) if c["dual"] else None, losses=nan(8, torch.float64), branch=nan(4, torch.float64),
                sums=nan(32, torch.float64), ws=torch.zeros(ws // 8, dtype=torch.float64, device="cuda"))


def _p(t):
    return None if t is None else t.data_ptr()


def _run(entry, c, d, cfg=None):
    """one entry point on the case; the outputs it does not write stay NaN"""
    L = _L()
    o = _outs(c)
    cfg = _cfg(c) if cfg is None else cfg
    ins, st = _ptrs(d), L.stream()
    if entry == "fwd_bwd":
        L.call("ppx_ppo_loss_fwd_bwd", C.byref(cfg), *ins, _p(o["d_actor"]), _p(o["d_log_std"]), _p(o["d_values"]),
               _p(o["d_int_values"]), _p(o["losses"]), _p(o["ws"]), st)
    elif entry == "head+finish":
        L.call("ppx_ppo_loss_head", C.byref(cfg), *ins, _p(o["d_actor"]), _p(o["sums"]), _p(o["ws"]), st)
        L.call("ppx_ppo_loss_finish", C.byref(cfg), _p(o["sums"]), _p(d["log_std"]), _p(d["values"]), _p(d["old_values"]),
               _p(d["returns"]), _p(d["int_values"]), _p(d["old_int_values"]), _p(d["int_returns"]), _p(o["d_log_std"]),
               _p(o["d_values"]), _p(o["d_int_values"]), _p(o["losses"]), _p(o["ws"]), st)
    elif entry == "head+finalize":
        L.call("ppx_ppo_loss_head", C.byref(cfg), *ins, _p(o["d_actor"]), _p(o["sums"]), _p(o["ws"]), st)
        L.call("ppx_ppo_loss_finalize", C.byref(cfg), _p(o["sums"]), _p(d["log_std"]), _p(o["d_log_std"]), _p(o["losses"]),
               _p(o["branch"]), st)
    elif entry == "head_final":
        L.call("ppx_ppo_loss_head_final", C.byref(cfg), *ins, _p(o["d_actor"]), _p(o["d_log_std"]), _p(o["losses"]),
               _p(o["branch"]), _p(o["ws"]), st)
    else:
        raise ValueError(entry)
    torch.cuda.synchronize()
    return {k: (None if v is None else v.cpu().numpy()) for k, v in o.items() if k not in ("ws",)}


ENTRIES = ("fwd_bwd", "head+finish", "head+finalize", "head_final")


def _run_all(c, d=None):
    """the four entry points on the same inputs: every output two of them share is bitwise identical.  Returns the
    fwd_bwd outputs with the branch weights of head_final."""
    d = _upload(c) if d is None else d
    r = {e: _run(e, c, d) for e in ENTRIES}
    same = lambda a, b: np.array_equal(a, b, equal_nan=False)
    for e in ENTRIES[1:]:
        for k in ("losses", "d_actor") + (() if c["discrete"] else ("d_log_std",)):
            assert same(r[e][k], r["fwd_bwd"][k]), f"{e} vs fwd_bwd: {k} differs"
    assert same(r["head+finish"]["d_values"], r["fwd_bwd"]["d_values"])
    if c["dual"]:
        assert same(r["head+finish"]["d_int_values"], r["fwd_bwd"]["d_int_values"])
    assert same(r["head+finalize"]["branch"], r["head_final"]["branch"]), "branch weights differ"
    out = dict(r["fwd_bwd"])
    out["branch"] = r["head_final"]["branch"]
    return out


# ----------------------------------------------------------------------------------------------------------------------
# checks
# ----------------------------------------------------------------------------------------------------------------------
def _check_losses(got, ref, pl_scale, pw, what=""):
    got = np.asarray(got[:5], np.float64)
    tol = 1e-6 * np.abs(ref) + 1e-9 * np.abs(ref).max() + 3e-7 * pl_scale * np.array([abs(pw), 1, 0, 0, 0])
    bad = ~(np.abs(got - ref) <= tol)
    names = ("total", "policy", "value", "entropy", "int_value")
    assert not bad.any(), f"{what} losses {[names[i] for i in np.flatnonzero(bad)]}: got {got} ref {ref}"


def _check_grad(name, got, ref, masks=None, floor=1e-7):
    """|got - ref| <= 1e-5 * max|ref| + floor over the whole array; with masks {label: bool array} the rows are checked
    label by label so that a failure names them"""
    ref = np.asarray(ref, np.float64)
    got = np.asarray(got, np.float64).reshape(ref.shape)
    tol = 1e-5 * np.abs(ref).max() + floor
    for label, m in (masks or {"all": np.ones(ref.shape, bool)}).items():
        m = np.broadcast_to(m.reshape(m.shape + (1,) * (ref.ndim - m.ndim)), ref.shape)
        err = np.where(m, np.abs(got - ref), 0.0)
        if not np.all(err <= tol):
            i = np.unravel_index(int(np.argmax(err)), ref.shape)
            raise AssertionError(f"{name} [{label}]: {int((err > tol).sum())} of {int(m.sum())} out of bound; worst {i}: "
                                 f"got {got[i]!r} ref {ref[i]!r} tol {tol:.3e}")


def _quadrants(c, ref):
    """d actor_out masks per surrogate quadrant: sign of the normalised advantage x side of the clip window"""
    a = _adv_n(c).astype(np.float64)[:, None]
    r = ref["ratio"].reshape(c["B"], -1)
    lo, hi = 1 - c["clip"], 1 + c["clip"]
    m = {"adv>0, ratio>1+clip": (a > 0) & (r > hi), "adv>0, ratio<1-clip": (a > 0) & (r < lo),
         "adv<0, ratio>1+clip": (a < 0) & (r > hi), "adv<0, ratio<1-clip": (a < 0) & (r < lo),
         "inside the window": (r >= lo) & (r <= hi)}
    if c["discrete"]:                                      # the row's ratio decides all A logits of the row
        m = {k: v[:, 0] for k, v in m.items()}
    return m


def _value_masks(kind):
    return {"inside the value-clip window": kind == 0, "above the window": kind == 1, "below the window": kind == 2,
            "on the value-clip edge": kind == 3}


def _check_case(c, got, ref, quadrants_required=False):
    _check_losses(got["losses"], ref["losses"], ref["pl_scale"], c["pw"])
    q = _quadrants(c, ref)
    if quadrants_required:
        for k, m in q.items():
            assert m.any(), f"case has no row in quadrant {k}"
    _check_grad("d actor_out", got["d_actor"], ref["d_actor"], q)
    if not c["discrete"]:
        _check_grad("d log_std", got["d_log_std"], ref["d_log_std"])
    _check_grad("d values", got["d_values"], ref["d_values"], _value_masks(c["vkind"]))
    if c["dual"]:
        _check_grad("d int_values", got["d_int_values"], ref["d_int_values"], _value_masks(c["ivkind"]))
    assert np.array_equal(got["branch"], ref["branch"]), f"branch weights {got['branch']} != {ref['branch']}"


# ----------------------------------------------------------------------------------------------------------------------
# the head and its entry points
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("value_mode", ["w1", "w0", "tie", "mixed"])
@pytest.mark.parametrize("dual", [False, True], ids=["single", "dual"])
@pytest.mark.parametrize("discrete", [True, False], ids=["discrete", "box"])
def test_head_quadrants_and_value_branch(discrete, dual, value_mode):
    """all four surrogate quadrants plus rows inside the window; a value branch that is one-sided (w1 = 1 or 0), an exact
    tie or whatever the data gives, with rows outside the value-clip window and exactly on its edge; the four entry
    points bitwise identical"""
    seed = 11 + 2 * int(discrete) + int(dual) + 10 * ["w1", "w0", "tie", "mixed"].index(value_mode)
    c = _case(600, 5 if discrete else 3, discrete, dual, seed=seed, pw=0.8 if dual else 1.0, value_mode=value_mode)
    ref = _reference(c)
    _assert_margins(c, ref, value_tie=value_mode == "tie")
    want = {"w1": 1.0, "w0": 0.0, "tie": 0.5}.get(value_mode)
    if want is not None:
        assert ref["branch"][0] == want and (not dual or ref["branch"][2] == want)
    _check_case(c, _run_all(c), ref, quadrants_required=True)


def test_categorical_saturated_probability_clamp():
    """logits at +-40: the probabilities clamp at eps and 1 - eps, so the drawn action's log-prob has no gradient
    (torch's clamp passes none outside its range) and only the entropy term reaches the logits.  The ratios are put
    inside the clip window, so a ratio gradient that leaked through the clamp would be O(1 / B)."""
    B, A = 96, 6
    c = _case(B, A, True, seed=5)
    rs = np.random.RandomState(6)
    big = rs.randint(0, A, B)
    x = np.full((B, A), -40.0, np.float32)
    x[np.arange(B), big] = 40.0
    c["actor_out"] = x
    act = big.copy()
    act[::3] = (big[::3] + 1 + rs.randint(0, A - 1, len(act[::3]))) % A   # every third row drew a clamped-low action
    c["actions"] = act.astype(np.float64)
    lp = _logprob(c)
    c["old_lp"] = (lp - np.log(rs.uniform(0.9, 1.1, B))).astype(np.float32)
    ref = _reference(c)
    _assert_margins(c, ref)
    got = _run_all(c)
    _check_case(c, got, ref)
    # the ratio gradient vanishes: what is left is the entropy term, tiny at saturation
    assert np.abs(ref["d_actor"]).max() < 1e-6
    assert np.abs(got["d_actor"]).max() < 1e-6


def test_categorical_one_action_head_has_zero_gradient():
    """A = 1: softmax is identically 1, so d actor_out is exactly 0 (the clamp at 1 - eps and the renormalised softmax
    both cancel); the losses still follow the reference"""
    c = _case(300, 1, True, seed=7)
    ref = _reference(c)
    _assert_margins(c, ref)
    got = _run_all(c)
    assert np.all(got["d_actor"] == 0.0)
    _check_case(c, got, ref)


def test_categorical_18_actions():
    c = _case(700, 18, True, True, seed=9, pw=1.3, actor_scale=2.5)
    ref = _reference(c)
    _assert_margins(c, ref)
    _check_case(c, _run_all(c), ref, quadrants_required=True)


@pytest.mark.parametrize("A", [1, 3, 16])
def test_box_widths(A):
    c = _case(400, A, False, seed=20 + A, ent_coef=0.03)
    ref = _reference(c)
    _assert_margins(c, ref)
    _check_case(c, _run_all(c), ref, quadrants_required=True)


def test_box_head_wider_than_16_is_refused():
    L = _L()
    c = _case(8, 17, False, seed=1)
    d = _upload(c)
    o = _outs(c)
    with pytest.raises(RuntimeError, match="Box head supports A <= 16"):
        L.call("ppx_ppo_loss_head_final", C.byref(_cfg(c)), *_ptrs(d), _p(o["d_actor"]), _p(o["d_log_std"]),
               _p(o["losses"]), _p(o["branch"]), _p(o["ws"]), L.stream())


@pytest.mark.parametrize("B", ["1", "255", "257", "grid+1"])
def test_batch_sizes(B):
    """B = 1, one CTA short of 256, one row past it, and one row past 256 rows x the grid cap (the grid-stride loop takes
    a second row in CTA 0 and the tail reduction reads every partial of a full grid); the largest case runs twice and
    must be bitwise identical"""
    n = {"1": 1, "255": 255, "257": 257, "grid+1": 256 * _grid_cap() + 1}[B]
    kw = {"1": dict(discrete=True, A=4), "255": dict(discrete=False, A=2, pw=0.6),
          "257": dict(discrete=True, A=3, dual=True, pw=1.3), "grid+1": dict(discrete=False, A=3, dual=True, pw=0.8)}[B]
    c = _case(n, kw.pop("A"), kw.pop("discrete"), kw.pop("dual", False), seed=30 + n % 97, **kw)
    ref = _reference(c)
    _assert_margins(c, ref)
    d = _upload(c)
    got = _run_all(c, d)
    _check_case(c, got, ref)
    if B == "grid+1":
        again = _run_all(c, d)
        for k in ("losses", "d_actor", "d_log_std", "d_values", "d_int_values", "branch"):
            assert np.array_equal(again[k], got[k]), f"two runs differ in {k}"


def _exact_ratio_one(rs, n):
    """(actions, log-prob) pairs for actor_out = 0, log_std = 0 whose f64 log-prob is an f32 number, so that an f32
    old_log_prob equal to it gives the Box head lp - old_lp == 0 and a ratio of exactly 1.  With mu = tanh(0) = 0 and
    sigma = exp(0) = 1 the head's log-prob is fl(fl(-fl(a * a) * 0.5) - log(sqrt(2 pi))), IEEE-exact to replay here."""
    acts, lps = [], []
    while len(acts) < n:
        target = np.float32(-HALF_LOG_2PI - 0.5 * rs.uniform(0.05, 1.5))
        a0 = np.sqrt(2.0 * (-np.float64(target) - HALF_LOG_2PI))
        for k in range(-64, 65):
            a = a0 + k * np.spacing(a0)
            lp = -(a * a) * 0.5 - HALF_LOG_2PI
            if np.float64(np.float32(lp)) == lp:
                acts.append(a if rs.rand() < 0.5 else -a)
                lps.append(np.float32(lp))
                break
    return np.array(acts), np.array(lps, np.float32)


def test_box_ratio_exactly_on_the_clip_edge():
    """clip_range = 0: the window is the single point 1, so a ratio of exactly 1 lies on both of its edges.  torch's
    clamp passes the gradient there (inclusive bounds), min(x, y) ties, and d actor_out is adv * d lp.  Every other
    element is at least 1e-3 away from 1.  The value errors tie on v == v_old rows, which are on the value-clip edge."""
    B, A = 256, 2
    c = _case(B, A, False, seed=41, clip=0.0, ent_coef=0.02, value_mode="w0")
    rs = np.random.RandomState(42)
    c["log_std"] = np.zeros(A, np.float32)
    exact = rs.rand(B, A) < 0.5
    acts, lps = _exact_ratio_one(rs, int(exact.sum()))
    c["actor_out"][exact] = 0.0
    c["actions"][exact] = acts
    lp = _logprob(c)
    assert np.array_equal(lp[exact], np.asarray(lps, np.float64))
    r = np.where(rs.rand(B, A) < 0.5, rs.uniform(1.05, 1.6, (B, A)), rs.uniform(0.4, 0.95, (B, A)))
    c["old_lp"] = (lp - np.log(r)).astype(np.float32)
    c["old_lp"][exact] = lps
    ref = _reference(c)
    assert np.all(ref["ratio"][exact] == 1.0)
    _assert_margins(c, ref, exact_ratio=exact)
    got = _run_all(c)
    _check_case(c, got, ref)
    _check_grad("d actor_out on the clip edge", got["d_actor"].reshape(B, A)[exact], ref["d_actor"][exact])


def test_discrete_first_epoch_ratio():
    """old_log_probs from ppx_policy_sample on the same logits: the first epoch.  Sampler and head evaluate the same
    clamped-softmax formula (sample_math.cuh), so the ratios are 1 up to the rounding of two separately compiled
    kernels; they must lie inside the clip window and the gradient is the unclipped one.  Whether they are exactly 1 is
    reported, not asserted: at clip_range = 0 (the window is the point 1) the head gives the same d actor_out only if
    every ratio is exactly 1, and that depends on how both kernels are compiled, not on the loss."""
    L = _L()
    B, A = 512, 7
    c = _case(B, A, True, seed=50, value_mode="tie")
    ao = torch.as_tensor(c["actor_out"]).cuda()
    acts = torch.empty(B, dtype=torch.float64, device="cuda")
    lp = torch.empty(B, dtype=torch.float32, device="cuda")
    L.call("ppx_policy_sample", ao.data_ptr(), None, B, A, 1, 1234, 0, acts.data_ptr(), lp.data_ptr(), L.stream())
    c["actions"], c["old_lp"] = acts.cpu().numpy(), lp.cpu().numpy()
    ref = _reference(c)
    _assert_margins(c, ref, value_tie=True)
    assert np.all(np.abs(ref["ratio"] - 1) < 1e-5)
    got = _run_all(c)
    _check_case(c, got, ref)
    got0 = _run_all(dict(c, clip=0.0))
    if not np.array_equal(got0["d_actor"], got["d_actor"]):
        warnings.warn("first-epoch ratios are not all exactly 1: ppx_policy_sample's log-prob differs in its last bits "
                      "from the loss head's", RuntimeWarning)


def _head_ratio_probe(logits, actions, old_lp):
    """the Discrete head's own f32 ratio exp(lq - old_lp) of each row, read back bitwise: one single-row launch per row
    with a normalised advantage of exactly 1 ((1 - 0) / (1 + 1e-8) rounds to 1 in f32) and the ratio inside the window,
    so the policy loss is -(double)ratio"""
    L = _L()
    n, A = logits.shape
    d = dict(actor_out=torch.as_tensor(np.ascontiguousarray(logits, np.float32)).cuda(), log_std=None,
             actions=torch.as_tensor(np.asarray(actions, np.float64)).cuda(),
             old_lp=torch.as_tensor(np.asarray(old_lp, np.float32)).cuda(), adv=torch.ones(n, device="cuda"),
             adv_stats=torch.tensor([0.0, 1.0], dtype=torch.float64, device="cuda"), values=torch.zeros(n, device="cuda"),
             old_values=torch.zeros(n, device="cuda"), returns=torch.zeros(n, device="cuda"))
    d.update({k: None for k in ("int_adv", "int_adv_stats", "int_values", "old_int_values", "int_returns")})
    cfg = L.PpoCfg(1, 0, A, 1, 0, float(np.float32(0.5)), 0.0, 0.0, 0.0, 1.0, None, 0)
    losses = torch.full((n, 8), float("nan"), dtype=torch.float64, device="cuda")
    branch = torch.empty(4, dtype=torch.float64, device="cuda")
    ws = torch.zeros(L.call("ppx_ppo_loss_workspace", 1, A) // 8, dtype=torch.float64, device="cuda")
    da = torch.empty(A, device="cuda")
    for i in range(n):
        L.call("ppx_ppo_loss_head_final", C.byref(cfg), *_ptrs(d, i, i + 1), da.data_ptr(), None, losses[i].data_ptr(),
               branch.data_ptr(), ws.data_ptr(), L.stream())
    return -losses[:, 1].cpu().numpy()


def test_discrete_ratio_exactly_on_the_clip_edge():
    """clip_range = 0, Discrete: rows whose ratio is exactly 1 lie on both edges of the window, where torch's clamp passes
    the gradient, so their d actor_out is the unclipped one -- bitwise what the head gives the same rows at clip 0.2,
    where they are well inside.  The exact rows are found with the head itself: for each row, old_log_prob candidates
    within a few ulps of the f64 log-prob go through _head_ratio_probe, and one whose ratio reads back as exactly 1.0 is
    kept.  Every other row's ratio is at least 0.05 from 1, and those rows follow the f64 reference at clip 0."""
    B, A = 256, 5
    c = _case(B, A, True, seed=55, value_mode="w1")
    rs = np.random.RandomState(56)
    exact = rs.rand(B) < 0.5
    r = _ratios(rs, B, CLIP)
    r[np.abs(r - 1) < 0.05] = 1.1
    lp = _logprob(c)
    old_lp = (lp - np.log(r)).astype(np.float32)
    idx = np.flatnonzero(exact)
    steps = np.arange(-8, 9)
    cand = np.empty((len(idx), len(steps)), np.float32)
    for j, k in enumerate(steps):
        x = lp[idx].astype(np.float32)
        for _ in range(abs(k)):
            x = np.nextafter(x, np.float32(np.copysign(np.inf, k)))
        cand[:, j] = x
    ratio = _head_ratio_probe(np.repeat(c["actor_out"][idx], len(steps), 0), np.repeat(c["actions"][idx], len(steps)),
                              cand.reshape(-1)).reshape(len(idx), len(steps))
    hit = ratio == 1.0
    assert hit.any(1).all(), "no old_log_prob within 8 ulps of the f64 log-prob gives the head a ratio of exactly 1"
    old_lp[idx] = cand[np.arange(len(idx)), hit.argmax(1)]
    c["old_lp"] = old_lp
    ref = _reference(c)
    _assert_margins(c, ref)
    got = _run_all(c)
    _check_case(c, got, ref)
    c0 = dict(c, clip=0.0)
    ref0 = _reference(c0)
    assert np.all(np.abs(ref0["ratio"][~exact] - 1) >= 0.04)
    got0 = _run_all(c0)
    rows = lambda a: a.reshape(B, A)
    assert np.array_equal(rows(got0["d_actor"])[exact], rows(got["d_actor"])[exact]), \
        "a ratio of exactly 1 at clip_range = 0 did not get the unclipped gradient (the clamp edge is inclusive)"
    _check_grad("d actor_out off the edge (clip_range = 0)", got0["d_actor"], ref0["d_actor"], {"off the edge": ~exact})


@pytest.mark.parametrize("discrete", [True, False], ids=["discrete", "box"])
def test_sharded_halves_match_one_call(discrete):
    """two row halves through ppx_ppo_loss_head with B_total = B, their 32 sums added on the device in rank order (the
    NCCL all-reduce path), ppx_ppo_loss_finalize: each half's d actor_out is the single call's rows bitwise, the losses
    and d_log_std agree to 1e-12"""
    L = _L()
    B = 1001
    c = _case(B, 4 if discrete else 3, discrete, True, seed=60 + int(discrete), pw=0.7)
    ref = _reference(c)
    _assert_margins(c, ref)
    d = _upload(c)
    one = _run("head_final", c, d)
    h0 = B // 2
    sums, d_actor = [], []
    ws = _outs(c)["ws"]
    for lo, hi in ((0, h0), (h0, B)):
        s = torch.full((32,), float("nan"), dtype=torch.float64, device="cuda")
        da = torch.full(((hi - lo) * c["A"],), float("nan"), device="cuda")
        L.call("ppx_ppo_loss_head", C.byref(_cfg(c, B=hi - lo, B_total=B)), *_ptrs(d, lo, hi), da.data_ptr(), s.data_ptr(),
               ws.data_ptr(), L.stream())
        sums.append(s)
        d_actor.append(da)
    total = sums[0] + sums[1]
    o = _outs(c)
    L.call("ppx_ppo_loss_finalize", C.byref(_cfg(c, B=h0, B_total=B)), total.data_ptr(), _p(d["log_std"]),
           _p(o["d_log_std"]), _p(o["losses"]), _p(o["branch"]), L.stream())
    torch.cuda.synchronize()
    A = c["A"]
    assert np.array_equal(d_actor[0].cpu().numpy(), one["d_actor"][:h0 * A]), "first half's d actor_out"
    assert np.array_equal(d_actor[1].cpu().numpy(), one["d_actor"][h0 * A:]), "second half's d actor_out"
    losses = o["losses"].cpu().numpy()
    np.testing.assert_allclose(losses, one["losses"], rtol=1e-12, atol=0)
    if not discrete:
        np.testing.assert_allclose(o["d_log_std"].cpu().numpy(), one["d_log_std"], rtol=1e-12, atol=0)
    assert np.array_equal(o["branch"].cpu().numpy(), one["branch"])
    _check_losses(losses, ref["losses"], ref["pl_scale"], c["pw"])


def test_loss_row_cursor():
    """with row_dev the losses land in row *row_dev, which then advances; with row_hold it stays; other rows are kept"""
    L = _L()
    c = _case(200, 3, False, True, seed=70)
    d = _upload(c)
    plain = _run("head_final", c, d)
    for entry in ("head_final", "fwd_bwd"):
        log = torch.full((4 * 8,), -7.0, dtype=torch.float64, device="cuda")
        row = torch.tensor([1], dtype=torch.int64, device="cuda")
        for hold, want_row in ((0, 2), (1, 2), (0, 3)):
            cfg = _cfg(c, row_dev=row.data_ptr(), row_hold=hold)
            o = _outs(c)
            written = int(row.item())
            if entry == "head_final":
                L.call("ppx_ppo_loss_head_final", C.byref(cfg), *_ptrs(d), _p(o["d_actor"]), _p(o["d_log_std"]),
                       log.data_ptr(), _p(o["branch"]), _p(o["ws"]), L.stream())
            else:
                L.call("ppx_ppo_loss_fwd_bwd", C.byref(cfg), *_ptrs(d), _p(o["d_actor"]), _p(o["d_log_std"]),
                       _p(o["d_values"]), _p(o["d_int_values"]), log.data_ptr(), _p(o["ws"]), L.stream())
            assert int(row.item()) == want_row, (entry, hold)
            rows = log.view(4, 8).cpu().numpy()
            assert np.array_equal(rows[written], plain["losses"]), (entry, written)
        assert np.all(rows[0] == -7.0) and np.all(rows[3] == -7.0)


# ----------------------------------------------------------------------------------------------------------------------
# the value gradient inside the fused MLP backward (PPO._policy_step)
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("branch", ["unclipped", "clipped"])
@pytest.mark.parametrize("name", ["ppo_box_small", "ppo_c1_discrete"])
def test_policy_step_gradients_away_from_the_tie(name, branch):
    """One minibatch of PPO._policy_step on a golden policy whose rollout was edited so that the ratios fall in every
    surrogate quadrant, the value branch is one-sided (unclipped: w1 = 1, clipped: w1 = 0) and rows lie outside the
    value-clip window and exactly on its edge.  With the fused policy MLP the value gradient exists only inside
    ppx_mlp3_bwd / ppx_mlp3_tc_bwd, evaluated from the branch weights; every parameter gradient is compared with float64
    autograd of the reference loss on a float64 copy of the parameters.

    The reference evaluates its f64 networks, then takes the kernel's own f32 forward outputs as the values of actor_out
    and the critic (x32 + (x64 - x64.detach())): an exact value-clip edge does not survive a re-evaluation in f64, and
    the gradient still flows through the f64 networks.  The forward outputs are checked against the f64 networks first
    (1e-4 of their largest value; the forward kernels have tests of their own).
    Bounds: 1e-4 relative + 1e-5 * max|ref| per array, the f32 backward's summation noise (the whole value-branch term of
    the critic is O(max|ref|))."""
    import ppo_exploration_b200 as ppx
    from test_gpu_learners import _env, _sd
    from test_oracle_golden import PPO_CASES, _ro
    g, cs = Golden(name), PPO_CASES[name]
    discrete = cs["discrete"]
    hp = dict(cs["hp"], ent_coef=0.01)
    env, T, N = _env(g, discrete)
    hidden = g["init/actor.0.weight"].shape[0]
    m = ppx.PPO(env=env, nstep=T, hidden_size=hidden, lr=cs["lr"], **hp)
    m.policy.load_state_dict(_sd(g, "init"))
    assert m.policy.mlp.fused(), "the value gradient under test is the one inside the fused MLP backward"
    ro = {k: np.array(v) for k, v in _ro(g).items()}
    m.rollout.load_rollout(**ro)
    np.random.seed(3)
    idx = m.rollout.permutation()[:hp["batch_size"]]
    B, ii = idx.numel(), idx.cpu().numpy()
    bufs = m.rollout._minibatch_buffers(B)
    m.rollout.gather_into(idx, bufs)
    fwd = m.policy.forward_raw(bufs["observations"][:B])
    a32, v32 = fwd[0].cpu().numpy().astype(np.float32), fwd[1].reshape(-1).cpu().numpy().astype(np.float32)

    p = {k: torch.tensor(np.asarray(v, np.float64), requires_grad=True) for k, v in g.group("init").items()}
    obs = torch.tensor(OR.gather_single(ro, ii)["observations"], dtype=torch.float64)
    a64, v64 = OL._mlp3(p, "actor", obs), OL._mlp3(p, "critic", obs).reshape(-1)
    for what, x32, x64 in (("actor_out", a32, a64), ("values", v32, v64)):
        x64 = x64.detach().numpy()
        assert np.abs(x32 - x64).max() <= 1e-4 * np.abs(x64).max(), f"forward {what} is not the f64 network's"

    # edit the rollout at the minibatch's rows (flat index = env * T + t, buffer.py:40-52)
    rs = np.random.RandomState(17)
    A = a32.shape[1]
    c = dict(B=B, A=A, discrete=discrete, dual=False, clip=float(np.float32(hp["clip_range"])), pw=1.0,
             ent_coef=hp["ent_coef"], vf_coef=float(hp["vf_coef"]), int_vf_coef=0.0, actor_out=a32,
             log_std=None if discrete else g["init/action_log_std"].reshape(-1))
    batch0 = OR.gather_single(ro, ii)
    c["actions"] = batch0["actions"].reshape(B) if discrete else batch0["actions"]
    lp = _logprob(c)
    c["old_lp"] = (lp - np.log(_ratios(rs, lp.shape, c["clip"]))).astype(np.float32)
    c["values"], c["old_values"], c["returns"], c["vkind"] = _value_arrays(
        rs, B, c["clip"], "w1" if branch == "unclipped" else "w0", v=v32)
    assert (c["vkind"] == 3).sum() >= max(2, B // 16), "too few exact value-clip edge rows"
    t_, n_ = ii % T, ii // T
    ro["action_log_probs"][t_, n_] = c["old_lp"].reshape(B, -1)
    ro["values"][t_, n_] = c["old_values"]
    ro["returns"][t_, n_] = c["returns"]
    m.rollout.load_rollout(**ro)
    m.rollout.gather_into(idx, bufs)
    c["adv"] = bufs["advantages"][:B].cpu().numpy()
    c["adv_stats"] = _stats(c["adv"])
    losses = torch.zeros(8, dtype=torch.float64, device="cuda")
    m._policy_step(bufs, B, losses.data_ptr())
    got = m.policy.state_dict(grad=True)

    ls = p["action_log_std"]
    # x32 + (x64 - x64.detach()): exactly the f32 value (x64 + x32 - x64 would round), the f64 network's gradient
    losses_ref, aux = _ref_losses(c, torch.as_tensor(a32, dtype=torch.float64) + (a64 - a64.detach()), ls,
                                  torch.as_tensor(v32, dtype=torch.float64) + (v64 - v64.detach()), None)
    _assert_margins(c, dict(ratio=aux["ratio"], m=aux["m"], im=None))
    assert (aux["m"][0] > aux["m"][1]) == (branch == "unclipped")
    for k, want in _quadrants(c, dict(ratio=aux["ratio"])).items():
        assert want.any(), f"no row in quadrant {k}"
    losses_ref[0].backward()
    _check_losses(losses.cpu().numpy(), np.array([float(x) for x in losses_ref]), aux["pl_scale"], 1.0, name)
    for k, v in p.items():
        if v.grad is None:
            assert float(got[k].abs().max()) == 0.0, k
            continue
        ref = v.grad.numpy()
        gk = got[k].numpy().reshape(ref.shape).astype(np.float64)
        err, tol = np.abs(gk - ref), 1e-4 * np.abs(ref) + 1e-5 * np.abs(ref).max()
        assert np.all(err <= tol), f"{name} {branch}: d {k} off by {err.max():.3e} (max|ref| {np.abs(ref).max():.3e})"


# ----------------------------------------------------------------------------------------------------------------------
# ICM / RND loss pieces
# ----------------------------------------------------------------------------------------------------------------------
def test_mse_fwd_bwd():
    """loss = scale * mean((a - b)^2) is ADDED to loss_accum; d_a = -d_b = 2 scale (a - b) / n; either may be NULL.
    n spans more rows than 256 x the grid cap, so each CTA strides."""
    L = _L()
    n, scale = 256 * _grid_cap() * 2 + 123, 0.37
    rs = np.random.RandomState(80)
    a, b = rs.randn(n).astype(np.float32), (0.5 * rs.randn(n)).astype(np.float32)
    diff = np.asarray(a, np.float64) - np.asarray(b, np.float64)
    loss = scale * np.mean(diff * diff)
    grad = 2 * scale * diff / n
    ad, bd = torch.as_tensor(a).cuda(), torch.as_tensor(b).cuda()
    for with_a, with_b in ((True, True), (True, False), (False, True), (False, False)):
        acc = torch.tensor([0.75], dtype=torch.float64, device="cuda")
        da = torch.full((n,), float("nan"), device="cuda") if with_a else None
        db = torch.full((n,), float("nan"), device="cuda") if with_b else None
        for _ in range(2):
            L.call("ppx_mse_fwd_bwd", ad.data_ptr(), bd.data_ptr(), n, scale, _p(da), _p(db), acc.data_ptr(), L.stream())
        got = float(acc.item())
        assert abs(got - (0.75 + 2 * loss)) <= 1e-6 * 2 * loss, (got, 0.75 + 2 * loss)
        # f32: gs = 2 scale / n and a - b are rounded once each, their product once: 3 roundings
        if with_a:
            assert np.all(np.abs(da.cpu().numpy() - grad) <= 2e-7 * np.abs(grad)), "d_a"
        if with_b:
            assert np.all(np.abs(db.cpu().numpy() + grad) <= 2e-7 * np.abs(grad)), "d_b"


@pytest.mark.parametrize("C_,stride", [(5, 1), (5, 3), (1, 2), (9, 1)])
def test_xent_fwd_bwd(C_, stride):
    """scale * mean(-log softmax(logits)[target]) added to loss_accum, d_logits = scale (softmax - onehot) / B; f64 targets
    read at target_stride; logits of +-80 in some rows (no overflow)"""
    L = _L()
    B, scale = 777, 0.8
    rs = np.random.RandomState(90 + C_ + stride)
    x = (3 * rs.randn(B, C_)).astype(np.float32)
    x[::7] = np.where(rs.rand(len(x[::7]), C_) < 0.5, np.float32(80), np.float32(-80))
    t = rs.randint(0, C_, B)
    tgt = rs.randint(0, C_, (B, stride)).astype(np.float64)          # the entries between targets are valid ids too
    tgt[:, 0] = t
    x64 = torch.tensor(x, dtype=torch.float64, requires_grad=True)
    ref_loss = scale * torch.nn.functional.cross_entropy(x64, torch.as_tensor(t))
    ref_loss.backward()
    xd, td = torch.as_tensor(x).cuda(), torch.as_tensor(tgt.reshape(-1)).cuda()
    dl = torch.full((B * C_,), float("nan"), device="cuda")
    acc = torch.tensor([-0.5], dtype=torch.float64, device="cuda")
    L.call("ppx_xent_fwd_bwd", xd.data_ptr(), td.data_ptr(), stride, B, C_, scale, dl.data_ptr(), acc.data_ptr(), L.stream())
    got = float(acc.item()) + 0.5
    want = float(ref_loss)
    assert np.isfinite(got) and abs(got - want) <= 1e-6 * abs(want) + 1e-12, (got, want)
    _check_grad("d_logits", dl.cpu().numpy().reshape(B, C_), x64.grad.numpy(), floor=0.0)
    if C_ == 1:
        assert got == 0.0 and np.all(dl.cpu().numpy() == 0.0)


@pytest.mark.parametrize("ids_f64", [False, True], ids=["int64", "f64"])
def test_embedding_fwd_bwd(ids_f64):
    """out[b, :C] = table[id[b]] with leading dimension ldo > C (the other columns untouched), ids read at id_stride;
    bwd sums the rows of repeated ids (float64 index_add reference); B = 0 writes a zero gradient"""
    L = _L()
    Cn, B, ldo, stride = 5, 300, 8, 2
    rs = np.random.RandomState(100 + int(ids_f64))
    table = rs.randn(Cn, Cn).astype(np.float32)
    ids = rs.randint(0, Cn, (B, stride))
    dt = torch.float64 if ids_f64 else torch.int64
    idd = torch.as_tensor(ids.reshape(-1)).to("cuda", dt)
    td = torch.as_tensor(table).cuda()
    out = torch.full((B, ldo), -3.25, device="cuda")
    L.call("ppx_embedding_fwd", td.data_ptr(), Cn, idd.data_ptr(), int(ids_f64), stride, B, out.data_ptr(), ldo, L.stream())
    o = out.cpu().numpy()
    assert np.array_equal(o[:, :Cn], table[ids[:, 0]])
    assert np.all(o[:, Cn:] == -3.25)
    dout = rs.randn(B, ldo).astype(np.float32)
    dd = torch.as_tensor(dout).cuda()
    dtab = torch.full((Cn * Cn,), float("nan"), device="cuda")
    L.call("ppx_embedding_bwd", dd.data_ptr(), ldo, idd.data_ptr(), int(ids_f64), stride, B, Cn, dtab.data_ptr(), L.stream())
    want = torch.zeros(Cn, Cn, dtype=torch.float64).index_add_(0, torch.as_tensor(ids[:, 0]),
                                                              torch.as_tensor(np.asarray(dout[:, :Cn], np.float64))).numpy()
    mag = torch.zeros(Cn, Cn, dtype=torch.float64).index_add_(0, torch.as_tensor(ids[:, 0]),
                                                             torch.as_tensor(np.abs(np.asarray(dout[:, :Cn], np.float64)))).numpy()
    k = np.bincount(ids[:, 0], minlength=Cn)[:, None]
    # an f32 running sum of k terms is within k * 2^-24 * sum|terms| of the exact sum
    assert np.all(np.abs(dtab.cpu().numpy().reshape(Cn, Cn) - want) <= k * 2.0 ** -24 * mag)
    dtab.fill_(float("nan"))
    L.call("ppx_embedding_bwd", dd.data_ptr(), ldo, idd.data_ptr(), int(ids_f64), stride, 0, Cn, dtab.data_ptr(), L.stream())
    assert np.all(dtab.cpu().numpy() == 0.0)
    out.fill_(-3.25)
    L.call("ppx_embedding_fwd", td.data_ptr(), Cn, idd.data_ptr(), int(ids_f64), stride, 0, out.data_ptr(), ldo, L.stream())
    assert np.all(out.cpu().numpy() == -3.25)


@pytest.mark.parametrize("F", [1, 31, 33, 288])
def test_icm_bonus_tail(F):
    """ri = clamp(mean_f((pred - feat)^2), -5, 5); rewards = (1 - eta) rewards + eta ri; rows above 5 clip to exactly 5;
    rewards_inout and ri_out may each be NULL"""
    L = _L()
    n, eta = 37, 0.3
    rs = np.random.RandomState(110 + F)
    pred = rs.randn(n, F).astype(np.float32)
    feat = (pred + rs.randn(n, F) * rs.uniform(0.1, 1.5, (n, 1))).astype(np.float32)
    feat[::4] = pred[::4] + np.float32(3.0)                            # mean square 9: clipped
    r0 = rs.randn(n).astype(np.float32)
    dsq = (np.asarray(pred, np.float64) - np.asarray(feat, np.float64)) ** 2
    ri = np.minimum(dsq.mean(1), 5.0)
    pd, fd = torch.as_tensor(pred).cuda(), torch.as_tensor(feat).cuda()
    for with_r, with_ri in ((True, True), (False, True), (True, False)):
        rw = torch.as_tensor(r0).cuda() if with_r else None
        rio = torch.full((n,), float("nan"), device="cuda") if with_ri else None
        L.call("ppx_icm_bonus_tail", pd.data_ptr(), fd.data_ptr(), n, F, eta, _p(rw), _p(rio), L.stream())
        # a lane sums F / 32 squares, five shuffles combine the lanes, one division: <= 15 f32 roundings of positive terms
        if with_ri:
            g = rio.cpu().numpy()
            assert np.all(np.abs(g - ri) <= 2e-6 * ri + 1e-12)
            assert np.all(g[::4] == 5.0)
        if with_r:
            want = (1 - eta) * np.asarray(r0, np.float64) + eta * ri
            assert np.all(np.abs(rw.cpu().numpy() - want) <= 2e-6 * (np.abs(r0) + ri) + 1e-12)


@pytest.mark.parametrize("add_to_total", [0, 1])
def test_loss_row_commit(add_to_total):
    L = _L()
    log = torch.arange(32, dtype=torch.float64, device="cuda") * 0.5
    row = torch.tensor([2], dtype=torch.int64, device="cuda")
    val = torch.tensor([3.75], dtype=torch.float64, device="cuda")
    want = log.cpu().numpy().copy()
    L.call("ppx_loss_row_commit", log.data_ptr(), row.data_ptr(), val.data_ptr(), 5, add_to_total, L.stream())
    want[8 * 2 + 5] = 3.75
    if add_to_total:
        want[8 * 2] += 3.75
    assert np.array_equal(log.cpu().numpy(), want)
    assert int(row.item()) == 3
