"""GPU numerics at the edges of both fused policy-MLP pairs: the tensor-core pair (mlp_tc.cu, tcgen05 3xTF32, h = 64) and
the SIMT pair (mlp_fused.cu, fp32, h = 64 / 128), called through their C entry points and checked stage by stage against
float64 references.

Network (ParallelMLP's bank layout, in-major): G groups of  D -> h -> h -> o_g  tanh MLPs sharing X,
  Z1 = X W1 + b1,  H1 = tanh Z1,  Z2_g = H1_g W2_g + b2_g,  H2_g = tanh Z2_g,  out_g = H2_g W3_g + b3_g,
  dP2 = (dOut W3^T)(1 - H2^2),  dP1 = (dP2 W2^T)(1 - H1^2),
  dW3 = H2^T dOut, db3 = 1^T dOut, dW2 = H1^T dP2, db2 = 1^T dP2, dW1 = X^T dP1, db1 = 1^T dP1.

Checks
------
* Teacher-forced stages.  Every stage is recomputed in float64 from the kernel's OWN inputs to that stage: H1 from X, H2 from
  the decoded H1, the outputs from the decoded H2, dW3 / db3 from dOut and H2, dW2 / db2 from H1 and dP2, dW1 / db1 from X and
  dP1 (dP2, dP1 are not saved: they are recomputed in float64 from the decoded activations, and the kernel's rounding of them
  is carried as a propagated bound, below).  The saved activations are decoded from the tensor-core tile layout
  Ht[G][tile][16 column quads][128 samples][4] (header of mlp_tc.cu) or read as [M, G*h] (SIMT).
* End to end.  float64 autograd of the same network on the same f32 parameters, with a bound propagated through the three
  layers and back, checked element by element in every parameter block.
* Every case launches forward + backward twice and must be bitwise identical; with the sum-of-squares partials, their f64 sum
  must equal the f64 sum of squares of the f32 gradients the reduce wrote (1e-12 relative: two orderings of one f64 sum).
* Inputs sit in guard bands: X rows past M (and pad columns with ldx > D) hold poison (NaN or 1e30), as do the rows past M of
  every dOut and of the value-head inputs; a kernel that reads a dead row or column gives a wrong or non-finite number.  Output
  rows past M must keep their sentinel; every gradient element (pre-filled with NaN) must be written.

Error model and tolerances
--------------------------
u = 2^-24 is the fp32 unit roundoff; one fp32 ulp is 2u relative.  An element that is a sum of products gets the bound
    |got - ref| <= (1 + gamma) (|A| + eA)(|B| + eB) - |A||B|                                                        (1)
(matrix products of absolute values, biases as a ones column): gamma * sum|terms| for the arithmetic of this stage, plus the
first-order effect of the propagated input errors eA, eB (zero for exact inputs).  Any summation order of n fp32 terms is
within (n - 1) u sum|terms| of the exact sum, so gamma only needs an operation COUNT n along the longest chain; we charge every
operation a full ulp, 2u, which also covers round-toward-zero steps:
  * 3xTF32 products (tensor core): a = hi + lo with hi = a truncated to tf32 (11 significant bits), so |lo| < 2^-10 |a|; the
    MMA truncates lo to tf32 again (error < 2^-21 |a|) and drops lo_a lo_b (< 2^-20 |a b|).  Per product: EPS_3X = 2^-19.
  * TMEM accumulation: an MMA aligns and adds 8 products into the fp32 accumulator; both steps truncate (< 1 ulp each), so
    every MMA instruction counts 2 operations: a 64-deep reduction as 3 x 8 MMAs = 48, the 128-sample weight-gradient GEMMs
    as 3 x 16 = 96, the layer-1 GEMM of fwd2 as 3 x (DP + 8) / 8 (x2).
  * fp32 register sums over a CTA's tiles: one operation per tile (kt = max tiles of one CTA, from the launch grid).
  * the fixed-order reduce over the n_cta partials: 8 slices x 2 chains of ceil(n_cta / 16), then 1 + 7 adds: ceil(n/16) + 9.
  * SIMT stages are plain fp32 FMA chains: layer 1 Dp + 1, layer 2 h + 1, heads h + 6, the thin column sums (dW3, db2, db3,
    dW1, db1) at most 32 in-tile + 9 cross-warp + kt, dW2 kt * 128 / NG (its per-thread register chain runs over all tiles).
The activations: tanh is 1-Lipschitz, so |H - tanh z| <= |z~ - z| + TANH_ABS, TANH_ABS the error of tanh_fast at an exact
argument (test_tanh_fast_abs_error measures it on exact pre-activations).  The derivative factor s = 1 - h^2 is computed as
fl(1 - fl(h h)) (error < 2 ulp absolute), the product with the upstream term rounds once more:
    e_dP <= e_a (|s| + e_s) + |a| e_s + 2u (|a| + e_a)(|s| + e_s),   e_s = 2 |h| e_h + e_h^2 + 4u.                     (2)
The upstream term of dP2, a = dOut W3^T, is an o-term fp32 sum (o + 1 operations); that of dP1 is the 3xTF32 GEMM 2 (tensor
core) or an h-deep FMA chain (SIMT).  The value head's in-kernel output gradient takes ~8 fp32 operations on values of
magnitude at most scale (|w1| 2 (|R| + |v|) + |w2| 2 (|R| + |v_old| + clip)) / B_total; it is charged 20 ulp of that.

Sensitivity.  Worst-case bounds allow errors n times larger than random rounding produces; an accuracy regression well inside
(1) (say lo operands dropped in one GEMM) would pass them.  So every stage also reports rho = RMS over its elements of
err / (u ||t||_2 + ||p||_2 + TANH_ABS [activations only]), t the terms of the element and p its propagated input-error terms
(eA B + A eB).  Model: the error is a sum of independent events -- each of the K 3xTF32 products errs by at most
EPS_3X |t_k| (RMS <= EPS_3X ||t||_2 / sqrt 3), each of the n accumulation steps by at most one ulp of a partial sum, and a
partial sum of random-sign terms is of the size of ||t||_2 (RMS <= 2 u ||t||_2 sqrt(n / 3)), every propagated input error by
at most its bound (RMS <= ||p||_2), tanh_fast by at most TANH_ABS.  Hence the ceiling
    RHO_MAX = 2 sqrt(n / 3) + [3xTF32] (EPS_3X / u) / sqrt 3 + 2,
asserted per stage.  A dropped hi.lo product or a one-bit-short lo operand errs by ~2^-11 of every term, the same sign as the
term: rho ~ 2^-11 / (u sqrt 3) ~ 4700, far above any ceiling here (< 60).
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

U = 2.0 ** -24                 # fp32 unit roundoff
ULP = 2.0 ** -23               # one fp32 ulp (relative), charged per operation
EPS_3X = 2.0 ** -19            # 3xTF32 product error (see the module docstring)
TANH_ABS = 3e-7                # absolute error of tanh_fast at an exact argument (mlp_tc.cu / mlp_fused.cu)
TM = 128
SENT = -12345.0
D_LIST = (1, 2, 3, 4, 6, 7, 8, 9, 12, 15, 16, 17, 20, 24, 31, 32)


def _L():
    from ppo_exploration_b200 import _lib as L
    L.load()
    return L


_SM = []


def sm_count():
    if not _SM:
        n = C.c_int(0)
        _L().call("ppx_device_info", C.addressof(n), None, None)
        assert n.value > 0
        _SM.append(n.value)
    return _SM[0]


def dp_of(D):
    return 8 if D <= 8 else (16 if D <= 16 else 32)


def n_tiles(M):
    return (M + TM - 1) // TM


def grid_of(pair, M, G, h):
    """CTAs per group of the backward kernel (mlp_tc.cu bwd_grid, mlp_fused.cu grid_x)."""
    per_sm = 1 if pair == "tc" else (2 if h == 64 else 1)
    return max(1, min(n_tiles(M), max(1, sm_count() * per_sm // G)))


def variant_of(pair, D, h):
    if pair == "simt":
        return f"mlp3_fwd/bwd<{h}>"
    return {8: "fwd2<8>+bwd2<8,32>", 16: "fwd2<16>+bwd2<16,32>", 32: "fwd<32>+bwd<32,32,false>"}[dp_of(D)]


# ------------------------------------------------------------------------------------------------ operation counts
def gammas(pair, D, h, M, G, omax):
    """gamma per stage (module docstring): EPS_3X per product where the tensor core multiplies, ULP per operation."""
    n = grid_of(pair, M, G, h)
    kt = -(-n_tiles(M) // n)
    red = -(-n // 16) + 9
    if pair == "tc":
        n1 = 2 * 3 * ((dp_of(D) + 8) // 8)              # fwd2 layer 1: 3 x (DP + 8) / 8 MMAs
        g = dict(h1=(EPS_3X + ULP * n1) if D <= 16 else ULP * (D + 1),
                 h2=EPS_3X + ULP * (48 + 1), out=ULP * (h + 6), a2=ULP * (omax + 1), a1=EPS_3X + ULP * 48,
                 thin=ULP * (32 + 6 + kt + red), w2=EPS_3X + ULP * (96 + kt + red))
        g["w1"] = g["b1"] = g["w2"] if D <= 16 else ULP * (32 + 1 + 4 + kt + red)
        n_ops = dict(h1=n1 if D <= 16 else D + 1, h2=49, out=h + 6, thin=38 + kt + red,
                     w2=96 + kt + red, w1=(96 + kt + red) if D <= 16 else 37 + kt + red)
        k3x = dict(h1=D + 1 if D <= 16 else 0, h2=h + 1, out=0, thin=0, w2=TM, w1=TM if D <= 16 else 0)
    else:
        NG = 256 // (2 * h)
        g = dict(h1=ULP * (D + 4), h2=ULP * (h + 1), out=ULP * (h + 6), a2=ULP * (omax + 1), a1=ULP * (h + 1),
                 thin=ULP * (32 + 10 + kt + red), w2=ULP * (kt * TM // NG + 2 + red), w1=ULP * (32 + 10 + kt + red))
        g["b1"] = g["w1"]
        n_ops = dict(h1=D + 4, h2=h + 1, out=h + 6, thin=42 + kt + red, w2=kt * TM // NG + 2 + red, w1=42 + kt + red)
        k3x = dict(h1=0, h2=0, out=0, thin=0, w2=0, w1=0)
    g["rho"] = {k: 2.0 * math.sqrt(n_ops[k] / 3.0) + (EPS_3X / U / math.sqrt(3.0) if k3x[k] else 0.0) + 2.0 for k in n_ops}
    return g


def generic_gammas(M, D, h):
    """Plain fp32 code of unknown summation order (the layer-by-layer path): n-term sums, n - 1 operations (+ margin)."""
    g = dict(h1=ULP * (D + 8), h2=ULP * (h + 8), out=ULP * (h + 8), a2=ULP * 40, a1=ULP * (h + 8),
             thin=ULP * (M + 16), w2=ULP * (M + 16), w1=ULP * (M + 16), b1=ULP * (M + 16))
    g["rho"] = None
    return g


# ------------------------------------------------------------------------------------------------ bounds
def mm_bound(A, eA, B, eB, gamma):
    """(1): bound on |fl(A~ B~) - A B| for |A~ - A| <= eA, |B~ - B| <= eB; A, B are absolute values.  Also returns the
    random-walk normaliser of the sensitivity statistic, u ||terms||_2 + ||propagated terms||_2."""
    S = (A + eA) @ (B + eB)
    if not torch.is_tensor(eA):
        eA = torch.zeros_like(A)
    if not torch.is_tensor(eB):
        eB = torch.zeros_like(B)
    T2 = ((A * A) @ (B * B)).sqrt()
    P2 = ((eA * eA) @ ((B + eB) ** 2) + (A * A) @ (eB * eB)).sqrt()
    return gamma * S + (S - A @ B), U * T2 + P2


def deriv_bound(a, e_a, h, e_h):
    """(2): bound on the kernel's a~ (1 - h~^2) against a (1 - h^2)."""
    s = (1.0 - h * h).abs()
    e_s = 2.0 * h.abs() * e_h + e_h * e_h + 4.0 * U
    aa = a.abs()
    return e_a * (s + e_s) + aa * e_s + ULP * (aa + e_a) * (s + e_s)


def ones_col(X):
    return torch.cat([X, torch.ones(X.shape[0], 1, dtype=X.dtype, device=X.device)], 1)


class Report:
    """Collects per-stage violations and the sensitivity statistic; one assert at the end lists every failure."""

    def __init__(self, tag):
        self.tag, self.fail, self.rho = tag, [], {}

    def check(self, name, got, ref, bound, S=None, rho_key=None, rho_max=None):
        got, ref = got.double(), ref.double()
        err = (got - ref).abs()
        bad = ~(err <= bound)
        if bool(bad.any()):
            i = int(torch.nonzero(bad.reshape(-1))[0])
            self.fail.append(f"{name}: {int(bad.sum())}/{bad.numel()} outside; first flat {i}: got {got.reshape(-1)[i].item():.9g} "
                             f"ref {ref.reshape(-1)[i].item():.9g} bound {bound.reshape(-1)[i].item():.3g}")
        if S is not None and rho_max is not None:
            r = float(((err / S.clamp_min(1e-300)) ** 2).mean().sqrt()) if err.numel() else 0.0
            self.rho[name] = r
            if not r <= rho_max[rho_key]:
                self.fail.append(f"{name}: rho {r:.3g} above the random-walk ceiling {rho_max[rho_key]:.3g}")

    def done(self):
        print(self.tag, " ".join(f"{k}={v:.2g}" for k, v in self.rho.items()))
        assert not self.fail, self.tag + "\n  " + "\n  ".join(self.fail)


def forward_checks(rep, net, X, H1k, H2k, outk, gam):
    """Teacher-forced forward stages (H1 from X, H2 from H1k, out from H2k) and the end-to-end forward.  Returns the f64
    reference activations and their propagated bounds for the end-to-end backward."""
    D, G, h = net["D"], net["G"], net["h"]
    Xa = ones_col(X.double())
    W1a = torch.cat([net["W1"].double(), net["b1"].double()[None]], 0)
    b, S = mm_bound(Xa.abs(), 0.0, W1a.abs(), 0.0, gam["h1"])
    z1 = Xa @ W1a
    H1r = torch.tanh(z1)
    if H1k is not None:
        rep.check("H1", H1k, H1r, b + TANH_ABS, S + TANH_ABS, "h1", gam["rho"])
    eH1 = (b + TANH_ABS).clamp(max=2.0)
    H2r, eH2 = [], []
    for g in range(G):
        sl = slice(g * h, (g + 1) * h)
        W2a = torch.cat([net["W2"][g].double(), net["b2"][g].double()[None]], 0)
        W3a = torch.cat([net["W3"][g].double(), net["b3"][g].double()[None]], 0)
        if H1k is not None:
            A = ones_col(H1k[:, sl].double())
            b, S = mm_bound(A.abs(), 0.0, W2a.abs(), 0.0, gam["h2"])
            rep.check(f"H2[{g}]", H2k[:, sl], torch.tanh(A @ W2a), b + TANH_ABS, S + TANH_ABS, "h2", gam["rho"])
            A = ones_col(H2k[:, sl].double())
            b, S = mm_bound(A.abs(), 0.0, W3a.abs(), 0.0, gam["out"])
            rep.check(f"out[{g}]", outk[g], A @ W3a, b, S, "out", gam["rho"])
        # end to end: propagate the activation errors through the layers
        A = ones_col(H1r[:, sl])
        eA = torch.cat([eH1[:, sl], torch.zeros_like(eH1[:, :1])], 1)
        b, _ = mm_bound(A.abs(), eA, W2a.abs(), 0.0, gam["h2"])
        h2 = torch.tanh(A @ W2a)
        e2 = (b + TANH_ABS).clamp(max=2.0)
        A = ones_col(h2)
        eA = torch.cat([e2, torch.zeros_like(e2[:, :1])], 1)
        b, _ = mm_bound(A.abs(), eA, W3a.abs(), 0.0, gam["out"])
        y = A @ W3a
        rep.check(f"e2e out[{g}]", outk[g], y, b)
        H2r.append(h2), eH2.append(e2)
    return H1r, eH1, H2r, eH2


def backward_checks(rep, net, X, H1, eH1, H2s, eH2s, dOut, e_dOut, grads, gam, prefix, rho=True):
    """Weight-gradient stages from the given activations (teacher forced: the kernel's own, zero error; end to end: the f64
    reference with propagated bounds) and the given output gradients."""
    D, G, h = net["D"], net["G"], net["h"]
    Xd = X.double()
    rk = gam["rho"] if rho else None
    ones = torch.ones(1, X.shape[0], dtype=torch.float64, device=X.device)
    dP1_all, e_dP1_all = [], []
    for g in range(G):
        sl = slice(g * h, (g + 1) * h)
        H1g, eH1g = H1[:, sl].double(), eH1[:, sl] if torch.is_tensor(eH1) else 0.0
        H2g, eH2g = H2s[g].double(), eH2s[g]
        W2, W3 = net["W2"][g].double(), net["W3"][g].double()
        d, ed = dOut[g].double(), e_dOut[g]
        b, S = mm_bound(H2g.abs().t(), eH2g.t() if torch.is_tensor(eH2g) else 0.0, d.abs(), ed, gam["thin"])
        rep.check(f"{prefix}dW3[{g}]", grads["dW3"][g], H2g.t() @ d, b, S, "thin", rk)
        b, S = mm_bound(ones, 0.0, d.abs(), ed, gam["thin"])
        rep.check(f"{prefix}db3[{g}]", grads["db3"][g], (ones @ d)[0], b[0], S[0], "thin", rk)
        a2 = d @ W3.t()
        e_a2, _ = mm_bound(d.abs(), ed, W3.abs().t(), 0.0, gam["a2"])
        dP2 = a2 * (1.0 - H2g * H2g)
        e_dP2 = deriv_bound(a2, e_a2, H2g, eH2g)
        b, S = mm_bound(H1g.abs().t(), eH1g.t() if torch.is_tensor(eH1g) else 0.0, dP2.abs(), e_dP2, gam["w2"])
        rep.check(f"{prefix}dW2[{g}]", grads["dW2"][g], H1g.t() @ dP2, b, S, "w2", rk)
        b, S = mm_bound(ones, 0.0, dP2.abs(), e_dP2, gam["thin"])
        rep.check(f"{prefix}db2[{g}]", grads["db2"][g], (ones @ dP2)[0], b[0], S[0], "thin", rk)
        a1 = dP2 @ W2.t()
        e_a1, _ = mm_bound(dP2.abs(), e_dP2, W2.abs().t(), 0.0, gam["a1"])
        dP1_all.append(a1 * (1.0 - H1g * H1g))
        e_dP1_all.append(deriv_bound(a1, e_a1, H1g, eH1g))
    dP1, e_dP1 = torch.cat(dP1_all, 1), torch.cat(e_dP1_all, 1)
    b, S = mm_bound(Xd.abs().t(), 0.0, dP1.abs(), e_dP1, gam["w1"])
    rep.check(f"{prefix}dW1", grads["dW1"], Xd.t() @ dP1, b, S, "w1", rk)
    b, S = mm_bound(ones, 0.0, dP1.abs(), e_dP1, gam["b1"])
    rep.check(f"{prefix}db1", grads["db1"], (ones @ dP1)[0], b[0], S[0], "w1", rk)


def autograd_grads(net, X, dOut):
    """float64 autograd of the network on the f32 parameters (the end-to-end reference)."""
    G, h = net["G"], net["h"]
    P = {k: (net[k].double().clone().requires_grad_(True)) for k in ("W1", "b1", "W2", "b2")}
    W3 = [w.double().clone().requires_grad_(True) for w in net["W3"]]
    b3 = [w.double().clone().requires_grad_(True) for w in net["b3"]]
    H1 = torch.tanh(X.double() @ P["W1"] + P["b1"])
    loss = 0.0
    for g in range(G):
        H2 = torch.tanh(H1[:, g * h:(g + 1) * h] @ P["W2"][g] + P["b2"][g])
        loss = loss + ((H2 @ W3[g] + b3[g]) * dOut[g].double()).sum()
    loss.backward()
    return dict(dW1=P["W1"].grad, db1=P["b1"].grad, dW2=P["W2"].grad, db2=P["b2"].grad,
                dW3=[w.grad for w in W3], db3=[w.grad for w in b3])


def end_to_end_checks(rep, net, X, H1r, eH1, H2r, eH2, dOut, e_dOut, grads, gam):
    ref = autograd_grads(net, X, dOut)
    # the bound of every block is the propagated per-element bound of backward_checks at the reference activations;
    # the autograd values replace the reference values of that computation
    sub = Report(rep.tag)
    backward_checks(sub, net, X, H1r, eH1, H2r, eH2, dOut, e_dOut, grads, gam, "e2e ", rho=False)
    rep.fail += sub.fail
    # the hand-written f64 backward used for the bounds is float64 autograd, to f64 rounding
    chk = Report("autograd")
    tight = {k: 1e-12 for k in ("a1", "a2", "thin", "w2", "w1", "b1")}
    backward_checks(chk, net, X, H1r, 0.0, H2r, [0.0] * net["G"], dOut, [0.0] * net["G"], ref, tight, "", rho=False)
    assert not chk.fail, chk.fail


# ------------------------------------------------------------------------------------------------ network and inputs
def make_net(D, h, outs, regime, seed):
    gen = torch.Generator().manual_seed(seed)
    G = len(outs)

    def orth(rows, cols):          # torch.nn.Linear weight [out, in] -> orthogonal(sqrt 2) -> in-major [in, out]
        w = torch.empty(rows, cols)
        torch.nn.init.orthogonal_(w, math.sqrt(2), generator=gen)
        return w.t().contiguous()

    W1 = torch.cat([orth(h, D) for _ in range(G)], 1)
    W2 = torch.stack([orth(h, h) for _ in range(G)])
    W3 = [orth(o, h) for o in outs]
    b1, b2, b3 = torch.zeros(G * h), torch.zeros(G, h), [torch.zeros(o) for o in outs]
    if regime == "sat":
        b1 = 3.0 * torch.randn(G * h, generator=gen)
        b2 = 3.0 * torch.randn(G, h, generator=gen)
        b3 = [torch.randn(o, generator=gen) for o in outs]
    elif regime == "mixed":
        def scales(n):
            s = 10.0 ** (torch.rand(n, generator=gen) * 9.0 - 6.0)
            s[torch.rand(n, generator=gen) < 0.15] = 0.0
            return s
        W1 = W1 * scales(D)[:, None]
        W2 = W2 * torch.stack([scales(h) for _ in range(G)])[:, :, None]
        W3 = [w * scales(h)[:, None] for w in W3]
        b1 = torch.randn(G * h, generator=gen) * (torch.rand(G * h, generator=gen) < 0.5)
        b2 = torch.randn(G, h, generator=gen)
        b3 = [torch.randn(o, generator=gen) for o in outs]
    net = dict(D=D, h=h, G=G, outs=list(outs), W1=W1, b1=b1, W2=W2, b2=b2, W3=W3, b3=b3)
    for k in ("W1", "b1", "W2", "b2"):
        net[k] = net[k].float().contiguous().cuda()
    net["W3"] = [w.float().contiguous().cuda() for w in net["W3"]]
    net["b3"] = [w.float().contiguous().cuda() for w in net["b3"]]
    return net


def make_x(M, D, regime, gen):
    if regime == "init":
        return torch.randn(M, D, generator=gen)
    if regime == "sat":                       # raw classic-control magnitudes: |x| up to 30, pre-activations up to ~40
        X = 30.0 * (2.0 * torch.rand(M, D, generator=gen) - 1.0)
        X[:, 0] = torch.where(torch.rand(M, generator=gen) < 0.5, -30.0, 30.0)
        return X
    s = 10.0 ** (torch.rand(D, generator=gen) * 9.0 - 6.0)      # mixed: columns spanning 1e-6 .. 1e3, exact zeros
    X = torch.randn(M, D, generator=gen) * s
    X[torch.rand(M, D, generator=gen) < 0.1] = 0.0
    if D >= 2:
        X[:, D // 2] = 0.0
    return X


def guarded_x(X, pad, off, poison):
    """X [M, D] inside a buffer of rows ldx = D + pad, 4 poison rows after M, poison pad columns, base `off` floats in."""
    M, D = X.shape
    ldx = D + pad
    buf = torch.full((off + (M + 4) * ldx,), poison)
    buf[off:off + M * ldx].view(M, ldx)[:, :D] = X
    return buf.cuda(), ldx


def guarded(t, poison):
    """[M, ...] -> device buffer with 4 poison rows after M."""
    pad = torch.full((4,) + tuple(t.shape[1:]), poison, dtype=t.dtype)
    return torch.cat([t, pad]).contiguous().cuda()


# ------------------------------------------------------------------------------------------------ the pair under test
def _ptrs(ts):
    return (C.c_void_p * len(ts))(*[t.data_ptr() if t is not None else None for t in ts])


def decode(pair, Hbuf, M, G, h):
    """saved activations -> [M, G*h]"""
    if pair == "tc":
        nT = n_tiles(M)
        return Hbuf.view(G, nT, h // 4, TM, 4).permute(1, 3, 0, 2, 4).reshape(nT * TM, G * h)[:M]
    return Hbuf.view(M, G * h)


def run_pair(pair, net, M, xbuf, off, ldx, dbufs, vh=None, clip=0.0, B_total=0):
    """forward + backward through the C entry points; returns outputs, decoded activations, gradients, sumsq partials."""
    L = _L()
    D, G, h, outs = net["D"], net["G"], net["h"], net["outs"]
    oi = (C.c_int * G)(*outs)
    sfx = "_tc" if pair == "tc" else ""
    st = L.stream()
    n_act = L.call("ppx_mlp3_tc_act_elems", M, h, G) if pair == "tc" else M * G * h
    H1 = torch.full((n_act,), float("nan"), device="cuda")
    H2 = torch.full((n_act,), float("nan"), device="cuda")
    out = [torch.full(((M + 4) * o,), SENT, device="cuda") for o in outs]
    xp = xbuf.data_ptr() + 4 * off
    n0 = L.launch_count()
    L.call(f"ppx_mlp3{sfx}_fwd", xp, ldx, M, D, h, G, oi, net["W1"].data_ptr(), net["b1"].data_ptr(), net["W2"].data_ptr(),
           net["b2"].data_ptr(), _ptrs(net["W3"]), _ptrs(net["b3"]), H1.data_ptr(), H2.data_ptr(), _ptrs(out), st)
    assert L.launch_count() - n0 == 1
    ws = torch.full((L.call(f"ppx_mlp3{sfx}_bwd_workspace", M, D, h, G, oi),), float("nan"), device="cuda")
    nan = lambda *s: torch.full(s, float("nan"), device="cuda")
    gr = dict(dW1=nan(D, G * h), db1=nan(G * h), dW2=nan(G, h, h), db2=nan(G, h), dW3=[nan(h, o) for o in outs],
              db3=[nan(o) for o in outs])
    n_ss = L.call("ppx_mlp3_sumsq_partials", D, h, G, oi)
    ss = torch.full((n_ss,), float("nan"), dtype=torch.float64, device="cuda")
    vhs = None
    if vh:
        vhs = (L.ValueHead * G)()
        for g, (v, ov, R, br, scale) in vh.items():
            vhs[g] = L.ValueHead(v.data_ptr(), ov.data_ptr(), R.data_ptr(), br.data_ptr(), float(scale))
    n0 = L.launch_count()
    L.call(f"ppx_mlp3{sfx}_bwd", xp, ldx, M, D, h, G, oi, net["W2"].data_ptr(), _ptrs(net["W3"]), H1.data_ptr(), H2.data_ptr(),
           _ptrs(dbufs), vhs, float(clip), int(B_total), gr["dW1"].data_ptr(), gr["db1"].data_ptr(), gr["dW2"].data_ptr(),
           gr["db2"].data_ptr(), _ptrs(gr["dW3"]), _ptrs(gr["db3"]), ws.data_ptr(), ss.data_ptr(), None, None, st)
    assert L.launch_count() - n0 == 2                      # backward kernel + fixed-order reduce
    torch.cuda.synchronize()
    return dict(out=out, H1=H1, H2=H2, grads=gr, ss=ss)


def _flat(res):
    g = res["grads"]
    return [*res["out"], res["H1"], res["H2"], g["dW1"], g["db1"], g["dW2"], g["db2"], *g["dW3"], *g["db3"], res["ss"]]


def check_case(pair, D, h, outs, M, regime="init", pad=0, off=0, poison=float("nan"), vh_groups=(), sparse=None, seed=0,
               B_total=None):
    L = _L()
    G = len(outs)
    oi = (C.c_int * G)(*outs)
    assert L.call("ppx_mlp3_supported", D, h, G, oi) == 1
    if pair == "tc":
        assert L.call("ppx_mlp3_tc_supported", D, h, G, oi) == 1, "the tensor-core pair must take this shape"
    net = make_net(D, h, outs, regime, seed)
    gen = torch.Generator().manual_seed(1000 + seed)
    X = make_x(M, D, regime, gen)
    xbuf, ldx = guarded_x(X, pad, off, poison)
    X = X.cuda()
    nT = n_tiles(M)
    rows = torch.ones(M, 1)
    if sparse == "ragged":                    # only the last (ragged) tile carries an output gradient
        rows[:(nT - 1) * TM] = 0.0
    elif sparse == "cta0_last":               # only the last tile of CTA 0 (which has >= 2 tiles)
        n = grid_of(pair, M, G, h)
        assert nT >= 2 * n
        last = ((nT - 1) // n) * n
        rows.zero_()
        rows[last * TM:(last + 1) * TM] = 1.0
    dOut = [torch.randn(M, o, generator=gen) * rows for o in outs]
    e_dOut = [0.0] * G
    vh = {}
    Bt = B_total if B_total is not None else 0
    clip, scale = 0.2, 0.5
    for g in vh_groups:
        assert outs[g] == 1
        v = torch.randn(M, generator=gen)
        dd = 0.6 * torch.randn(M, generator=gen)
        dd = torch.where((dd.abs() - clip).abs() < 1e-3, dd + 0.01, dd)
        ov = v - dd
        R = torch.randn(M, generator=gen) * rows[:, 0]
        br = torch.tensor([0.3, 0.7], dtype=torch.float64)
        vh[g] = (guarded(v, poison), guarded(ov, poison), guarded(R, poison), br.cuda(), scale)
        Bt_eff = float(Bt if Bt > 0 else M)
        w1, w2 = float(np.float32(br[0])), float(np.float32(br[1]))
        vd, ovd, Rd = v.double(), ov.double(), R.double()
        dd32 = (v - ov).double()                   # the kernel's branch test runs on the f32 difference
        assert bool(((dd32.abs() - clip).abs() > 1e-4).all())
        vc = ovd + dd32.clamp(-clip, clip)
        pas = ((dd32 >= -clip) & (dd32 <= clip)).double()
        d = scale * (w1 * (-2.0 * (Rd - vd)) + w2 * (-2.0 * (Rd - vc)) * pas) / Bt_eff
        dOut[g] = d[:, None]                       # the f64 reference output gradient of this head
        e_dOut[g] = (20 * ULP * abs(scale) / Bt_eff * (abs(w1) * 2 * (Rd.abs() + vd.abs()) +
                                                        abs(w2) * 2 * (Rd.abs() + ovd.abs() + clip)))[:, None].cuda()
    dbufs = [None if g in vh else guarded(dOut[g].float(), poison) for g in range(G)]
    dOut = [t.cuda() for t in dOut]
    vh_args = {g: vh[g] for g in vh}
    res = run_pair(pair, net, M, xbuf, off, ldx, dbufs, vh_args, clip, Bt)
    res2 = run_pair(pair, net, M, xbuf, off, ldx, dbufs, vh_args, clip, Bt)
    for a, b in zip(_flat(res), _flat(res2)):
        assert torch.equal(a.view(torch.uint8), b.view(torch.uint8)), "two launches differ"
    tag = f"[{pair} {variant_of(pair, D, h)} D={D} h={h} outs={tuple(outs)} M={M} {regime} pad={pad} off={off}]"
    rep = Report(tag)
    # guard bands: output rows past M untouched, every gradient written
    for g, o in enumerate(outs):
        if not bool((res["out"][g][M * o:] == SENT).all()):
            rep.fail.append(f"out[{g}] written past row M")
    outk = [res["out"][g][:M * o].view(M, o) for g, o in enumerate(outs)]
    for k, t in res["grads"].items():
        for i, tt in enumerate(t if isinstance(t, list) else [t]):
            if not bool(torch.isfinite(tt).all()):
                rep.fail.append(f"{k}[{i}] not finite (unwritten or poisoned)")
    H1k, H2k = decode(pair, res["H1"], M, G, h), decode(pair, res["H2"], M, G, h)
    gam = gammas(pair, D, h, M, G, max(outs))
    H1r, eH1, H2r, eH2 = forward_checks(rep, net, X, H1k, H2k, outk, gam)
    gr = res["grads"]
    backward_checks(rep, net, X, H1k.double(), 0.0, [H2k[:, g * h:(g + 1) * h].double() for g in range(G)], [0.0] * G,
                    dOut, e_dOut, gr, gam, "")
    end_to_end_checks(rep, net, X, H1r, eH1, H2r, eH2, dOut, e_dOut, gr, gam)
    # sum of squares of the gradients the reduce wrote, f64 over f32 values
    ref_ss = sum(float((t.double() ** 2).sum()) for k, v in gr.items() for t in (v if isinstance(v, list) else [v]))
    got_ss = float(res["ss"].sum())
    if not abs(got_ss - ref_ss) <= 1e-12 * ref_ss:
        rep.fail.append(f"sumsq {got_ss!r} vs {ref_ss!r}")
    rep.done()


# ------------------------------------------------------------------------------------------------ coverage matrix
TC_WIDTHS = [(4,), (2, 1), (3, 1, 1), (4, 1, 1, 3), (1,), (3, 1), (2, 1, 1), (1, 4, 2, 1)]
SIMT_WIDTHS = [(32,), (18, 1), (3, 1, 1), (1, 7, 32, 2), (5,), (32, 1), (9, 1, 1), (4, 1, 1, 3)]


def _variant_cases():
    cases = []
    for i, D in enumerate(D_LIST):
        M = (300, 1000, 129, 4099)[i % 4]
        cases.append(("tc", D, 64, TC_WIDTHS[i % 8], M, 0, 0))
        cases.append(("simt", D, 64, SIMT_WIDTHS[i % 8], M, 0, 0))
    for D in (4, 16, 32):            # D = DP (or a float4 row) read through a strided / misaligned X: scalar loads
        cases += [("tc", D, 64, (2, 1), 515, 3, 0), ("tc", D, 64, (2, 1, 1), 515, 0, 1), ("tc", D, 64, (4, 1), 700, 4, 0),
                  ("simt", D, 64, (2, 1), 515, 4, 0), ("simt", D, 64, (6, 1, 1), 515, 0, 1)]
    for D in (3, 7, 9, 15, 17, 31):  # odd D with a padded row
        cases += [("tc", D, 64, (2, 1), 333, 1, 0), ("simt", D, 64, (2, 1), 333, 2, 0)]
    for D, outs in ((1, (2, 1)), (2, (3, 1, 1)), (4, (1,)), (6, (3, 1, 1)), (8, (2, 1)), (4, (1, 1, 1, 1))):
        cases.append(("simt", D, 128, outs, 1000, 0, 0))
    cases.append(("simt", 4, 128, (2, 1), 600, 4, 0))
    return cases


VARIANT_CASES = _variant_cases()


def test_matrix_covers_every_variant():
    """Every tensor-core instantiation (the variant follows from D) and both SIMT widths, both X loads per DP bucket,
    D = DP in every bucket, G = 1..4."""
    seen = {variant_of(p, D, h) for p, D, h, *_ in VARIANT_CASES}
    assert seen == {"fwd2<8>+bwd2<8,32>", "fwd2<16>+bwd2<16,32>", "fwd<32>+bwd<32,32,false>", "mlp3_fwd/bwd<64>",
                    "mlp3_fwd/bwd<128>"}
    for dp in (8, 16, 32):
        ds = {(D, pad, off) for p, D, h, o, M, pad, off in VARIANT_CASES if p == "tc" and dp_of(D) == dp}
        assert any(D % 4 == 0 and pad % 4 == 0 and off == 0 for D, pad, off in ds), dp      # float4 X load
        assert any(D % 4 or pad % 4 or off for D, pad, off in ds), dp                       # scalar X load
        assert any(D == dp for D, _, _ in ds), dp
    assert {len(c[3]) for c in VARIANT_CASES} == {1, 2, 3, 4}
    assert set(D_LIST) <= {c[1] for c in VARIANT_CASES if c[0] == "tc"} and set(D_LIST) <= {c[1] for c in VARIANT_CASES if c[0] == "simt"}


@pytest.mark.parametrize("pair,D,h,outs,M,pad,off", VARIANT_CASES)
def test_variant(pair, D, h, outs, M, pad, off):
    check_case(pair, D, h, outs, M, pad=pad, off=off, seed=D * 7 + M)


SCHEDULES = ("k1", "k1_2", "k2", "k2_3", "k7_8")


def _sched_tiles(name, n):
    return {"k1": n, "k1_2": n + max(1, n // 2), "k2": 2 * n, "k2_3": 2 * n + max(1, n // 3), "k7_8": 7 * n + max(1, (2 * n) // 3)}[name]


@pytest.mark.parametrize("pair", ["tc", "simt"])
@pytest.mark.parametrize("G", [1, 2, 3, 4])
@pytest.mark.parametrize("sched", SCHEDULES)
def test_tile_schedule(pair, G, sched):
    """M from the device's SM count so that the backward grid gives every CTA 1 tile, a 1/2 mix, 2, a 2/3 mix, 7/8."""
    n = grid_of(pair, 1 << 30, G, 64)
    nT = _sched_tiles(sched, n)
    rag = (0, 1, 127)[(G + SCHEDULES.index(sched)) % 3]          # M % 128
    M = nT * TM if rag == 0 else (nT - 1) * TM + rag
    assert n_tiles(M) == nT and grid_of(pair, M, G, 64) == min(n, nT)
    D = (8, 12, 24, 3)[G - 1]
    outs = ((4,), (2, 1), (3, 1, 1), (4, 1, 1, 3))[G - 1] if pair == "tc" else ((9,), (2, 1), (3, 1, 1), (1, 6, 1, 2))[G - 1]
    check_case(pair, D, 64, outs, M, seed=G * 10 + SCHEDULES.index(sched))


EDGE_CASES = [
    # pair, D, outs, M, regime, pad, off, poison, vh_groups, sparse, B_total
    *[(p, 8, (2, 1), M, "init", 0, 0, float("nan"), (), None, None) for p in ("tc", "simt") for M in (1, 127, 128, 129)],
    *[(p, D, (2, 1, 1), 131072, "init", 0, 0, float("nan"), (), None, None) for p, D in (("tc", 8), ("simt", 4))],
    *[(p, D, (3, 1), 3000, "sat", 0, 0, float("nan"), (), None, None) for p in ("tc", "simt") for D in (6, 12, 24)],
    *[(p, D, (2, 1, 1), 3000, "mixed", 0, 0, float("nan"), (), None, None) for p in ("tc", "simt") for D in (4, 9, 20)],
    *[(p, D, (2, 1), 1000, r, 5, 0, 1e30, (), None, None) for p in ("tc", "simt") for D, r in ((8, "sat"), (16, "mixed"))],
    *[(p, 8, (2, 1, 1), 5000 + 77, "init", 0, 0, float("nan"), (), "ragged", None) for p in ("tc", "simt")],
    *[(p, 12, (3, 1), 0, "init", 0, 0, float("nan"), (), "cta0_last", None) for p in ("tc", "simt")],
    *[(p, D, (2, 1, 1), 2000 + 13, "init", 0, 0, po, (1, 2), None, 3 * 2013 + 7)
      for p in ("tc", "simt") for D, po in ((8, float("nan")), (20, 1e30))],
    *[(p, 4, (1, 1), 777, "sat", 3, 0, float("nan"), (0, 1), None, None) for p in ("tc", "simt")],
    *[(p, 16, (2, 1), 20000, "init", 0, 0, float("nan"), (1,), "ragged", 12345) for p in ("tc", "simt")],
]


@pytest.mark.parametrize("pair,D,outs,M,regime,pad,off,poison,vh_groups,sparse,B_total", EDGE_CASES)
def test_edges(pair, D, outs, M, regime, pad, off, poison, vh_groups, sparse, B_total):
    if sparse == "cta0_last":                 # CTA 0 gets 3 tiles, the others 2 or 3
        M = (2 * grid_of(pair, 1 << 30, len(outs), 64) + 3) * TM - 50
    check_case(pair, D, 64, outs, M, regime=regime, pad=pad, off=off, poison=poison, vh_groups=vh_groups, sparse=sparse,
               seed=M % 97 + D, B_total=B_total)


@pytest.mark.parametrize("pair", ["tc", "simt"])
def test_forward_m0_launches_nothing(pair):
    L = _L()
    net = make_net(8, 64, (2, 1), "init", 0)
    oi = (C.c_int * 2)(2, 1)
    x = torch.zeros(8, device="cuda")
    H = torch.zeros(4, device="cuda")
    out = [torch.zeros(4, device="cuda") for _ in range(2)]
    sfx = "_tc" if pair == "tc" else ""
    n0 = L.launch_count()
    rc = L.call(f"ppx_mlp3{sfx}_fwd", x.data_ptr(), 8, 0, 8, 64, 2, oi, net["W1"].data_ptr(), net["b1"].data_ptr(),
                net["W2"].data_ptr(), net["b2"].data_ptr(), _ptrs(net["W3"]), _ptrs(net["b3"]), H.data_ptr(), H.data_ptr(),
                _ptrs(out), L.stream())
    assert rc == 0 and L.launch_count() == n0


def _simt_limit(D, h):
    L = _L()
    ok = lambda o: L.call("ppx_mlp3_supported", D, h, 2, (C.c_int * 2)(o, 1)) == 1
    assert ok(1)
    o = 1
    while ok(o + 1):
        o += 1
    return o


@pytest.mark.parametrize("h,D", [(64, 1), (64, 32), (128, 1), (128, 4), (128, 8)])
def test_simt_width_limit(h, D):
    """The largest head width the SIMT pair accepts runs correctly; one more is declined (shared-memory limit or MAXO)."""
    o = _simt_limit(D, h)
    L = _L()
    assert L.call("ppx_mlp3_supported", D, h, 2, (C.c_int * 2)(o + 1, 1)) == 0
    assert L.call("ppx_mlp3_supported", D, h, 2, (C.c_int * 2)(1, o + 1)) == 0
    print(f"SIMT h={h} D={D}: widest head {o}")
    check_case("simt", D, h, (o, 1), 515, seed=o + D)


# ------------------------------------------------------------------------------------------------ tanh_fast
@pytest.mark.parametrize("pair,D,h", [("tc", 1, 64), ("tc", 17, 64), ("simt", 1, 64), ("simt", 3, 128)])
def test_tanh_fast_abs_error(pair, D, h):
    """Exact pre-activations (tf32-exact x and w, one live input, zero bias: every product and sum is exact on both the
    tensor core and the FMA pipe), so H1 - tanh(z) is tanh_fast's own error, over z in [-32, 32].  The kernels' comments
    once claimed 2e-7; the largest error here is 2.2e-7 (at z = -2.66), inside the derived 3e-7."""
    M = 4097
    x = (torch.arange(M, dtype=torch.float64) - 2048) / 256.0                # 11 significant bits at most
    X = torch.zeros(M, D)
    X[:, 0] = x.float()
    net = make_net(D, h, (2, 1), "init", 5)
    w = (64.0 + torch.arange(2 * h) % 64) / 32.0                             # 7 significant bits, [2, 4)
    net["W1"].zero_()
    net["W1"][0] = w.float().cuda()
    net["b1"].zero_()
    xbuf, ldx = guarded_x(X, 0, 0, float("nan"))
    d = [guarded(torch.zeros(M, o), 0.0) for o in (2, 1)]
    res = run_pair(pair, net, M, xbuf, 0, ldx, d)
    H1 = decode(pair, res["H1"], M, 2, h).double().cpu()
    z = x[:, None] * w[None, :]
    assert torch.equal(z, (x.float()[:, None] * w.float()[None, :]).double()), "pre-activations must be exact in fp32"
    err = (H1 - torch.tanh(z)).abs()
    print(f"tanh_fast max abs error {float(err.max()):.3e} at z = {float(z.reshape(-1)[int(err.argmax())]):.6g}")
    assert float(err.max()) <= TANH_ABS


# ------------------------------------------------------------------------------------------------ Policy level
def _policy(D, h, space, intrinsic):
    import ppo_exploration_b200 as ppx
    env = ppx.SyntheticVecEnv(4, D, space, seed=0)
    torch.manual_seed(3 * D + h)
    return ppx.models.Policy(env, h, intrinsic_model=intrinsic, device="cuda")


def _policy_cases():
    cases = []
    for D, sp, n, h, path in ((4, "D", 2, 128, "simt"), (2, "D", 3, 64, "tc"), (6, "D", 3, 64, "tc"), (3, "B", 1, 64, "tc"),
                              (2, "B", 1, 64, "tc"), (8, "B", 2, 64, "tc"), (8, "D", 4, 64, "tc"), (24, "B", 4, 64, "tc"),
                              (17, "B", 6, 64, "simt"), (33, "B", 2, 64, "layer"), (8, "B", 2, 96, "layer"),
                              (4, "D", "simt+1", 128, "layer")):
        for intrinsic in (False, True):
            cases.append((D, sp, n, h, intrinsic, path))
    return cases


@pytest.mark.parametrize("D,space,n,h,intrinsic,path", _policy_cases())
def test_policy_paths(D, space, n, h, intrinsic, path):
    """Production shapes through Policy: the dispatch predicates pick the expected path, and it matches float64."""
    import ppo_exploration_b200 as ppx
    if n == "simt+1":
        n = _simt_limit(D, h) + 1
    pol = _policy(D, h, ppx.Discrete(n) if space == "D" else ppx.Box((n,)), intrinsic)
    fa = pol.mlp._fused_args()
    assert (fa["ok"], fa["tc"]) == {"tc": (True, True), "simt": (True, False), "layer": (False, False)}[path]
    G, outs, b = pol.mlp.G, pol.outs, pol.bank
    net = dict(D=D, h=h, G=G, outs=list(outs), W1=b.view("W1"), b1=b.view("b1"), W2=b.view("W2"), b2=b.view("b2"),
               W3=[b.view(f"W3.{g}") for g in pol.names], b3=[b.view(f"b3.{g}") for g in pol.names])
    M = 1000
    gen = torch.Generator().manual_seed(D + n)
    X = torch.randn(M, D, generator=gen).cuda()
    d = [torch.randn(M, o, generator=gen).cuda() / M for o in outs]
    outk = [o.clone() for o in pol.forward_raw(X)]
    _, H1s, H2s = pol.mlp._saved
    H1k = decode(path, H1s, M, G, h) if path == "tc" else H1s.view(M, G * h)
    H2k = decode(path, H2s, M, G, h) if path == "tc" else H2s.view(M, G * h)
    b.grad.fill_(float("nan"))
    pol.mlp.backward(d)
    torch.cuda.synchronize()
    gr = dict(dW1=b.view("W1", grad=True), db1=b.view("b1", grad=True), dW2=b.view("W2", grad=True),
              db2=b.view("b2", grad=True), dW3=[b.view(f"W3.{g}", grad=True) for g in pol.names],
              db3=[b.view(f"b3.{g}", grad=True) for g in pol.names])
    gam = gammas(path, D, h, M, G, max(outs)) if path != "layer" else generic_gammas(M, D, h)
    rep = Report(f"[policy {path} D={D} h={h} outs={tuple(outs)}]")
    H1r, eH1, H2r, eH2 = forward_checks(rep, net, X, H1k.double(), H2k.double(), outk, gam)
    backward_checks(rep, net, X, H1k.double(), 0.0, [H2k[:, g * h:(g + 1) * h].double() for g in range(G)], [0.0] * G,
                    d, [0.0] * G, gr, gam, "")
    end_to_end_checks(rep, net, X, H1r, eH1, H2r, eH2, d, [0.0] * G, gr, gam)
    rep.done()
