"""Oracle for ES-NSRA with a novelty per member (NSRA-ES, Conti et al. 2018, Alg. 3; DESIGN.md §3.16).

TEST INFRASTRUCTURE -- see oracle/__init__.py.  numpy float64 throughout.  PARITY UNPINNED: the reference broadcasts one
scalar novelty over the population (oracle/es.py `update_weights`); these numpy definitions are the specification of
`novelty_mode="member"`.  The pinned pieces they call (novelty, novelty_distribution, centered_ranks, nsr_adapt) live in
oracle/es.py and oracle/es_nsra.py.
"""
import numpy as np

from .es import centered_ranks, novelty, novelty_distribution
from .es_nsra import nsr_adapt


def _shape(v, shaping):
    """z-score (ddof 0; a vector whose std is 0 shapes to 0) or centred ranks."""
    v = np.asarray(v, np.float64)
    if shaping == "centered_rank":
        return centered_ranks(v)[1]
    std = v.std()
    return np.zeros(v.shape) if std == 0 else (v - v.mean()) / std


def update_weights_member(w, rewards, novelties, population, lr, sigma, novelty_param, decay, shaping="zscore"):
    """The update with a novelty per member.  Returns (new_w, new_lr).
    F~ = shape(rewards), N~ = shape(novelties) over all P members (z-score with ddof 0, a zero-std vector shaping to 0,
    or centred ranks); score = ((1 - w) E^T F~ + w E^T N~) / 2, keeping update_weights' /2 so that w = 0 is
    update_weights' step; theta += lr/(P sigma) * score, lr *= decay.  z-score with BOTH stds 0 returns (w, lr)
    untouched; centred ranks never skip."""
    rewards = np.asarray(rewards, np.float64)
    novelties = np.asarray(novelties, np.float64)
    if shaping != "centered_rank" and rewards.std() == 0 and novelties.std() == 0:
        return w, lr
    F, N = _shape(rewards, shaping), _shape(novelties, shaping)
    P = len(population)
    f = lr / (P * sigma)
    out = []
    for l, wl in enumerate(w):
        E = np.array([m[l] for m in population])                     # [P, in, out]
        score = ((1 - novelty_param) * np.dot(E.T, F).T + novelty_param * np.dot(E.T, N).T) / 2
        out.append(wl + f * score)
    return out, lr * decay


def knn_sum_sq(archive, query, k):
    """oracle/es.py `knn_sum` by selection on SQUARED distances, square roots of the k winners only (the order of
    ppx_knn_novelty_many).  Equal to knn_sum because a correctly rounded square root is monotone."""
    a = np.concatenate(archive) if isinstance(archive, list) else np.asarray(archive)
    q = np.asarray(query, np.float64).reshape(-1)
    d2 = np.zeros(len(a), np.float64)
    for j in range(a.shape[1]):                                       # sequential over dims, no FMA
        diff = a[:, j] - q[j]
        d2 = d2 + diff * diff
    return sum(np.sqrt(np.sort(d2)[:k]))


def nsra_run_member(thetas, lr, iterations, *, shapes, sigma, decay, novelty_param, nsr_plateu, nsr_range, nsr_update,
                    eps_of, fitness_of, brains_of, member_bcs_of, K=10, reward_target=None, shaping="zscore"):
    """EvolutionStrategy.run(novelty_mode="member"): oracle/es_nsra.py `nsra_run` with the update of every generation
    replaced by update_weights_member.  member_bcs_of(g) -> [P, k] BCs of generation g's members; every member's novelty
    is scored against the archive BEFORE BC_b is appended.  The brain pick (novelties of the brains), the archive and
    nsr_adapt are nsra_run's.  Returns dict(thetas, archive, picks, w, lr, fb) as nsra_run."""
    thetas = np.array(thetas, np.float64)
    M = thetas.shape[0]
    cut = np.cumsum([0] + [a * b for a, b in shapes])
    split = lambda v: [v[cut[l]:cut[l + 1]].reshape(shapes[l]) for l in range(len(shapes))]
    bc, f = brains_of(-1, thetas)
    archive = [np.asarray(x, np.float64) for x in bc]
    w, best, fb, picks, ws = novelty_param, -np.inf, [], [], []
    for g in range(iterations):
        arch = np.array(archive)
        nov = [float(novelty(arch, bc[m], K)) for m in range(M)]
        b = int(np.random.choice(list(range(M)), p=novelty_distribution(nov)))
        eps = np.asarray(eps_of(g), np.float64)
        rewards = fitness_of(g, thetas[b])
        nov_p = [float(novelty(arch, x, K)) for x in np.asarray(member_bcs_of(g), np.float64)]
        new_w, lr = update_weights_member(split(thetas[b]), rewards, nov_p, [split(e) for e in eps], lr, sigma, w, decay,
                                          shaping=shaping)
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
