"""Oracle for EvolutionStrategy.run, the ES-NSRA loop over a meta-population (reference: evolution_strategies.py:293-384).

TEST INFRASTRUCTURE -- see oracle/__init__.py.  numpy float64 throughout, as the reference.  The per-generation pieces are
those of oracle/es.py, pinned to reference fixtures; the loop and the novelty-weight rule are not (see nsr_adapt).
"""
import numpy as np

from .es import novelty, novelty_distribution, update_weights


def nsr_adapt(w, fb, best, nsr_plateu, nsr_range, nsr_update, every=5):
    """The novelty weight w = novelty_param after a generation, given fb = the brain fitness f_b of every generation so far
    and best = B, the best f_b before the current window (-inf at the start).  Returns (w, B).
    PARITY UNPINNED: the reference stores nsr_plateu / nsr_range / nsr_update but its run loop is not vendored here; this
    numpy definition is the specification (NSRA-ES, Conti et al. 2018).  Every `every` generations, R = the largest f_b of
    the last `every`: R > B + nsr_plateu (reward improving) -> w = max(lo, w - nsr_update), weighting reward more;
    otherwise (a plateau) w = min(hi, w + nsr_update), exploring more; then B = max(B, R)."""
    if len(fb) < every or len(fb) % every:
        return w, best
    R = max(fb[-every:])
    if R > best + nsr_plateu:
        w = max(nsr_range[0], w - nsr_update)
    else:
        w = min(nsr_range[1], w + nsr_update)
    return w, max(best, R)


def nsra_run(thetas, lr, iterations, *, shapes, sigma, decay, novelty_param, nsr_plateu, nsr_range, nsr_update, eps_of,
             fitness_of, brains_of, K=10, reward_target=None):
    """EvolutionStrategy.run: ES-NSRA over a meta-population of M flat f64 parameter vectors `thetas` [M, D].
    PARITY UNPINNED (see nsr_adapt): the order of operations is SURVEY §3.4's; each piece it calls is pinned (novelty,
    novelty_distribution + np.random.choice = pick_brain, update_weights).
      brains_of(g, thetas) -> (bc [M, k], f [M]): one episode per brain at sigma = 0 (g = -1: before the first generation)
      eps_of(g) -> [P, D] f64 noise of generation g;  fitness_of(g, theta_b) -> [P] fitness of theta_b + sigma * eps
    A fresh run seeds the archive with every brain's behaviour; each generation picks brain b by novelty against the
    archive (numpy's global RNG), updates it with novelty nu_b and weight w, runs the brains, appends BC_b to the archive,
    adapts w (nsr_adapt) and stops once f_b > reward_target.
    Returns dict(thetas, archive, picks, w = w after every generation, lr, fb)."""
    thetas = np.array(thetas, np.float64)
    M = thetas.shape[0]
    cut = np.cumsum([0] + [a * b for a, b in shapes])
    split = lambda v: [v[cut[l]:cut[l + 1]].reshape(shapes[l]) for l in range(len(shapes))]
    bc, f = brains_of(-1, thetas)
    archive = [np.asarray(x, np.float64) for x in bc]
    w, best, fb, picks, ws = novelty_param, -np.inf, [], [], []
    for g in range(iterations):
        nov = [float(novelty(np.array(archive), bc[m], K)) for m in range(M)]
        probs = novelty_distribution(nov)
        b = int(np.random.choice(list(range(M)), p=probs))
        eps = np.asarray(eps_of(g), np.float64)
        rewards = fitness_of(g, thetas[b])
        new_w, lr = update_weights(split(thetas[b]), rewards, [split(e) for e in eps], lr, sigma, w, decay, novelty=nov[b])
        thetas[b] = np.concatenate([x.ravel() for x in new_w])
        bc, f = brains_of(g, thetas)
        archive.append(np.asarray(bc[b], np.float64))
        fb.append(float(f[b]))
        picks.append(b)
        w, best = nsr_adapt(w, fb, best, nsr_plateu, nsr_range, nsr_update)
        ws.append(w)
        if reward_target is not None and f[b] > reward_target:
            break
    return dict(thetas=thetas, archive=np.array(archive), picks=picks, w=ws, lr=lr, fb=fb)
