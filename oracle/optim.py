"""Oracle for the optimiser step of every ppx parameter bank  --  TEST INFRASTRUCTURE, see oracle/__init__.py.

The reference steps every network with ``torch.nn.utils.clip_grad_norm_(params, max_norm)`` followed by
``torch.optim.Adam.step()`` (algorithms.py:243-244, :465-466, :501-502, :697-699): amsgrad off, no weight decay.  This is
the single-tensor form of that pair (torch/optim/adam.py ``_single_tensor_adam``) restated in f64 for ONE step from a given
f32 state, so a device step can be checked against it without rounding noise piling up over many steps.
"""
import math

import numpy as np


def clip_adam(p, g, m, v, t, lr, betas=(0.9, 0.999), eps=1e-8, max_norm=0.0, n_clip=None, extra=None):
    """One clip_grad_norm_ + Adam step in f64.

    p, g, m, v: 1-D parameter, gradient, exp_avg and exp_avg_sq vectors (any float dtype; read as f64).
    t: the step number of this update (>= 1; torch's ``state['step']`` after its increment).
    max_norm > 0: clip_grad_norm_ over g[:n_clip] (default: all of g) plus `extra`, a gradient vector of parameters that
      enter the norm but are updated elsewhere (ppx: ``action_log_std`` when it is not part of the clipped range).  The
      coefficient min(max_norm / (norm + 1e-6), 1) scales g[:n_clip]; g[n_clip:] is used unscaled.
    max_norm == 0 (or n_clip == 0): no clip_grad_norm_ call at all (the reference's ICM optimiser, :699).

    Returns (p', m', v', norm, coef): f64 arrays, the total norm (None when nothing was clipped) and the coefficient."""
    p, g, m, v = (np.asarray(a, dtype=np.float64).reshape(-1) for a in (p, g, m, v))
    n_clip = g.size if n_clip is None else int(n_clip)
    norm, coef = None, 1.0
    if max_norm > 0.0 and n_clip > 0:
        ss = float(np.sum(g[:n_clip] * g[:n_clip]))
        if extra is not None:
            e = np.asarray(extra, dtype=np.float64).reshape(-1)
            ss += float(np.sum(e * e))
        norm = math.sqrt(ss)
        coef = min(max_norm / (norm + 1e-6), 1.0)                   # clip_coef_clamped = clamp(max_norm/(norm+1e-6), max=1)
        g = g.copy()
        g[:n_clip] *= coef
    beta1, beta2 = betas
    m = m + (1.0 - beta1) * (g - m)                                 # exp_avg.lerp_(grad, 1 - beta1)
    v = v * beta2 + (1.0 - beta2) * g * g                           # exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
    step_size = lr / (1.0 - beta1 ** t)
    denom = np.sqrt(v) / math.sqrt(1.0 - beta2 ** t) + eps
    p = p - step_size * (m / denom)                                 # param.addcdiv_(exp_avg, denom, value=-step_size)
    return p, m, v, norm, coef


def step_scale(g, m_new, v_new, t, lr, betas=(0.9, 0.999), eps=1e-8):
    """Per-element size of one Adam step before the first moment can cancel: step_size * (|m'| + (1-beta1)|g|) / denom.
    A tolerance stated as a fraction of it stays meaningful where exp_avg happens to cancel to ~0 (there the update
    itself is ~0, but the f32 rounding of the lerp is not)."""
    beta1, beta2 = betas
    g, m_new, v_new = (np.asarray(a, dtype=np.float64).reshape(-1) for a in (g, m_new, v_new))
    denom = np.sqrt(v_new) / math.sqrt(1.0 - beta2 ** t) + eps
    return lr / (1.0 - beta1 ** t) * (np.abs(m_new) + (1.0 - beta1) * np.abs(g)) / denom
