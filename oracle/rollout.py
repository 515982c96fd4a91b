"""Oracle for the rollout-buffer half of the hot path (reference: buffer.py, sil_module.py).

TEST INFRASTRUCTURE -- see oracle/__init__.py.  Plain numpy, written as free functions over
explicit arrays instead of the reference's stateful classes.  dtype promotion follows what
numpy 2.x does for the reference's expressions; each place where that matters is commented.
"""
import numpy as np


# --------------------------------------------------------------------------------------
# GAE reverse scans                                                    buffer.py:203-230
# --------------------------------------------------------------------------------------
def gae(rewards, values, masks, last_value, dones, gamma, lam):
    """Single-head GAE + returns.  buffer.py:217-230.

    rewards/values: f32 [T,N]; masks: integer [T,N] (the `dones` stored by add(), buffer.py:180);
    last_value: f32 [N]; dones: bool/int [N].

    Precision (all forced by numpy promotion in the reference, SURVEY "Hard parts"):
      * ``gamma * next_value``      python float x f32 array -> f32 product   (buffer.py:227)
      * ``1.0 - masks[t+1]``        int64 -> f64, so delta and the carry are f64 (buffer.py:225)
      * ``advantages[t] = carry``   rounded to f32 on store                   (buffer.py:229)
      * ``returns = adv + values``  f32 + f32                                 (buffer.py:230)
    Off-by-one: step t is cut by masks[t+1]; the last step by `dones` (buffer.py:221-226).
    """
    T, N = rewards.shape
    adv = np.zeros((T, N), np.float32)
    carry = np.zeros(N, np.float64)
    g32 = np.float32(gamma)
    gl = float(gamma) * float(lam)
    for t in range(T - 1, -1, -1):
        if t == T - 1:
            nnt = 1.0 - np.asarray(dones).astype(np.float64)
            nv = np.asarray(last_value, np.float32).reshape(N)
        else:
            nnt = 1.0 - masks[t + 1].astype(np.float64)
            nv = values[t + 1]
        gv = (g32 * nv).astype(np.float32)                       # f32 product
        delta = rewards[t].astype(np.float64) + gv.astype(np.float64) * nnt - values[t].astype(np.float64)
        carry = delta + gl * nnt * carry
        adv[t] = carry.astype(np.float32)
    ret = adv + values.astype(np.float32)
    return adv, ret


def gae_dual(rewards, values, masks, last_value, dones, gamma, lam,
             int_rewards, int_values, last_int_value, int_gamma):
    """Dual-head GAE (RND).  buffer.py:337-362.

    Extrinsic head exactly as `gae`.  Intrinsic head is NON-episodic (no terminal masking,
    buffer.py:357-358) and, because no int64 array enters the expression, stays float32 end to
    end: ``int_gamma * next_int`` and ``int_gamma * gae_lam * carry`` are python-float x f32.
    """
    adv, ret = gae(rewards, values, masks, last_value, dones, gamma, lam)
    T, N = rewards.shape
    iadv = np.zeros((T, N), np.float32)
    icarry = np.zeros(N, np.float32)
    gi = np.float32(int_gamma)
    gil = np.float32(float(int_gamma) * float(lam))
    for t in range(T - 1, -1, -1):
        niv = np.asarray(last_int_value, np.float32).reshape(N) if t == T - 1 else int_values[t + 1]
        idelta = (int_rewards[t] + gi * niv) - int_values[t]     # f32 throughout
        icarry = (idelta + gil * icarry).astype(np.float32)
        iadv[t] = icarry
    iret = iadv + int_values.astype(np.float32)
    return adv, ret, iadv, iret


def discount_with_dones(rewards, dones, gamma):
    """R_t = r_t + gamma * R_{t+1} * (1 - done_t).  sil_module.py:99-105 (python-float carry = f64).

    rewards/dones: [T] or [T,N] (the reference handles one episode list at a time; the [T,N]
    form runs the same recurrence per column)."""
    r = np.asarray(rewards, np.float64)
    d = np.asarray(dones, np.float64)
    out = np.zeros_like(r)
    carry = np.zeros(r.shape[1:], np.float64)
    for t in range(r.shape[0] - 1, -1, -1):
        carry = r[t] + gamma * carry * (1.0 - d[t])
        out[t] = carry
    return out


# --------------------------------------------------------------------------------------
# SimHash                                                              buffer.py:188-200
# --------------------------------------------------------------------------------------
def simhash_bits(A, obs):
    """bits[i,b] = (A[b] . obs[i] > 0).  buffer.py:194 (f64 A times f32 obs -> f64 dot)."""
    return np.greater(np.dot(A, obs.T).T, 0).astype(int)


def pack_bits(bits):
    """bit b of the uint64 code <-> column b of the reference's bit row (k <= 64)."""
    k = bits.shape[1]
    assert k <= 64
    w = (np.uint64(1) << np.arange(k, dtype=np.uint64))
    return (bits.astype(np.uint64) * w).sum(axis=1, dtype=np.uint64)


def unpack_code(code, k):
    return np.array([(int(code) >> b) & 1 for b in range(k)], dtype=int)


def bits_key(row):
    """The dict key the reference builds (buffer.py:195).  np.array_str line-wraps rows longer
    than 75 chars (k=64 keys carry a newline) -- harmless, still injective; kept verbatim."""
    return np.array_str(row).replace('[', '').replace(']', '').replace(' ', '')


class CountTable:
    """The persistent defaultdict of buffer.py:136 plus the sequential update of :197-199."""

    def __init__(self, beta=0.1):
        self.table = {}
        self.beta = beta

    def update(self, A, obs, rewards):
        """Mutates and returns `rewards` (like the reference); also returns the per-obs count
        *after* that obs' own increment, in env order (duplicates inside one batch see c+1, c+2, ...).
        ``rewards[i] += beta/np.sqrt(count)``: the bonus is f64; the sum is rounded to the dtype
        of `rewards` when stored back (f32 array -> f32)."""
        bits = simhash_bits(A, obs)
        counts = np.zeros(len(bits), np.uint32)
        for i, row in enumerate(bits):
            key = bits_key(row)
            c = self.table.get(key, 0) + 1
            self.table[key] = c
            counts[i] = c
            rewards[i] += self.beta / np.sqrt(c)
        return rewards, counts

    def as_code_dict(self, k):
        """{uint64 code: count} view for comparison with the device table dump."""
        out = {}
        for key, c in self.table.items():
            bits = np.array([int(ch) for ch in key if ch in '01'], dtype=int)
            assert len(bits) == k
            out[int(pack_bits(bits[None, :])[0])] = c
        return out


def count_update_codes(table, codes):
    """Integer-only restatement on packed codes: table is {code:int}; returns sequential counts."""
    counts = np.zeros(len(codes), np.uint32)
    for i, c in enumerate(codes.tolist()):
        n = table.get(c, 0) + 1
        table[c] = n
        counts[i] = n
    return counts


# --------------------------------------------------------------------------------------
# flatten / shuffle / gather                                 buffer.py:40-52, 233-267
# --------------------------------------------------------------------------------------
def swap_and_flatten(arr):
    """[T,N,...] -> [N*T,...], env-major: flat[i] = arr[i % T, i // T].  buffer.py:49-52.
    2-D inputs gain a trailing singleton dim (so advantages come out [T*N,1])."""
    shape = arr.shape
    if len(shape) < 3:
        shape = shape + (1,)
    return arr.swapaxes(0, 1).reshape(shape[0] * shape[1], *shape[2:])


def flat_to_tn(idx, T):
    """Inverse of the env-major flatten: flat index i lives at (t, n) = (i % T, i // T)."""
    idx = np.asarray(idx)
    return idx % T, idx // T


def epoch_permutation(T, N):
    """One global-numpy-RNG permutation per `get()` call.  buffer.py:239."""
    return np.random.permutation(T * N)


def minibatch_slices(total, batch_size):
    """Start/stop of each minibatch; the last one may be short.  buffer.py:251-254."""
    if batch_size is None:
        batch_size = total
    return [(s, min(s + batch_size, total)) for s in range(0, total, batch_size)]


def gather_single(buf, idx):
    """RolloutSample for one minibatch.  buffer.py:261-267.  `buf` holds [T,N,...] arrays."""
    f = {k: swap_and_flatten(buf[k]) for k in
         ('observations', 'actions', 'values', 'action_log_probs', 'advantages', 'returns')}
    return dict(observations=f['observations'][idx], actions=f['actions'][idx],
                old_values=f['values'][idx].flatten(), old_log_probs=f['action_log_probs'][idx],
                advantages=f['advantages'][idx], returns=f['returns'][idx].flatten())


def gather_dual(buf, idx):
    """RND RolloutSample, field order of buffer.py:287-295 / :385-393."""
    out = gather_single(buf, idx)
    for src, dst, flat in (('int_values', 'int_values', True), ('int_advantages', 'int_advantages', False),
                           ('int_returns', 'int_returns', True)):
        a = swap_and_flatten(buf[src])[idx]
        out[dst] = a.flatten() if flat else a
    return out


# --------------------------------------------------------------------------------------
# running moments                                                         util.py:9-44
# --------------------------------------------------------------------------------------
class RunningMeanStd:
    """Parallel-variance running moments, float64.  util.py:10-44."""

    def __init__(self, epsilon=1e-4, shape=()):
        self.mean = np.zeros(shape, np.float64)
        self.var = np.ones(shape, np.float64)
        self.count = epsilon

    def update(self, arr):
        bm, bv, bc = np.mean(arr, axis=0), np.var(arr, axis=0), arr.shape[0]
        delta = bm - self.mean
        tot = self.count + bc
        new_mean = self.mean + delta * bc / tot
        m2 = self.var * self.count + bv * bc + np.square(delta) * self.count * bc / (self.count + bc)
        self.mean, self.var, self.count = new_mean, m2 / (self.count + bc), bc + self.count


def normalize_obs(obs, mean, var):
    """clip((obs-mean)/sqrt(var+1e-10), -5, 5) in f64.  algorithms.py:117."""
    return np.clip((obs - mean) / np.sqrt(var + 1e-10), -5, 5).astype(float)


def fy_apply_sequential(j):
    """The swaps of numpy's legacy shuffle given its partner list: for i = n-1 .. 1: swap(a[i], a[j[i]]) on arange(n)
    (what buffer.py:239's np.random.permutation does after drawing j_i = random_interval(i)).  j[0] is unused."""
    n = len(j)
    a = np.arange(n)
    for i in range(n - 1, 0, -1):
        a[i], a[j[i]] = a[j[i]], a[i]
    return a


def fy_apply_parallel(j):
    """The same result without the sequential dependence -- the algorithm of csrc/shuffle_dev.cu restated in numpy
    (test infrastructure: pins the algorithm on the CPU, the kernels are checked against numpy on the GPU).

    Position i is final after its own step and receives what position j[i] held just before it; a position p holds,
    before step i, what the most recent earlier step that targeted p (smallest s > i with j[s] == p) moved in -- the
    content position s had before ITS step -- or p itself.  first[p] = smallest step targeting p, nxt[s] = next larger
    step with the same target; V(s) = V(first[s]) follows a strictly increasing chain."""
    n = len(j)
    steps = [i for i in range(1, n) if j[i] != i]                      # self-swaps move nothing
    groups = {}
    for i in sorted(steps):
        groups.setdefault(int(j[i]), []).append(i)
    first = {p: g[0] for p, g in groups.items()}
    nxt = {}
    for g in groups.values():
        for a, b in zip(g, g[1:]):
            nxt[a] = b

    def chase(q):
        while q in first:
            q = first[q]
        return q

    out = np.empty(n, dtype=np.int64)
    for i in range(n):
        t = int(j[i]) if i else 0
        if t == i:
            out[i] = chase(i)
        elif i in nxt:
            out[i] = chase(nxt[i])
        else:
            out[i] = t
    return out


class VecNormalizeRef(object):
    """numpy restatement of stable_baselines3.common.vec_env.VecNormalize.step_wait with norm_obs / norm_reward (the wrapper
    the reference puts around its envs, env.py:11) -- NOT part of the reference tree and not installed here: PARITY UNPINNED
    upstream; the arithmetic below is the published one (running moments = the reference's own util.py:9-44 rule, which is
    pinned by tests/golden/rnd_bonus.npz).

    `training` and `norm_reward` follow the published step_wait / _update_reward: the observation and return statistics
    are updated, and the discounted returns accumulated, only while training (`norm_reward` does not matter for that);
    the rewards are divided only with norm_reward; a done zeroes its return in every mode.  This flag logic is equally a
    restatement of the published code, not checked against an installed stable_baselines3: parity is still unpinned."""

    def __init__(self, n_envs, obs_shape, clip_obs=10.0, clip_reward=10.0, gamma=0.99, epsilon=1e-8, training=True,
                 norm_reward=True):
        self.obs_rms, self.ret_rms = RunningMeanStd(shape=obs_shape), RunningMeanStd(shape=())
        self.ret = np.zeros(n_envs)
        self.clip_obs, self.clip_reward, self.gamma, self.epsilon = clip_obs, clip_reward, gamma, epsilon
        self.training, self.norm_reward = training, norm_reward

    def reset(self, obs):
        self.ret = np.zeros_like(self.ret)
        if self.training:
            self.obs_rms.update(obs)
        return self.normalize_obs(obs)

    def normalize_obs(self, obs):
        return np.clip((obs - self.obs_rms.mean) / np.sqrt(self.obs_rms.var + self.epsilon), -self.clip_obs, self.clip_obs)

    def step(self, obs, rews, dones):
        if self.training:
            self.obs_rms.update(obs)
        obs_n = self.normalize_obs(obs)
        if self.training:                                   # _update_reward
            self.ret = self.ret * self.gamma + rews
            self.ret_rms.update(self.ret)
        if self.norm_reward:
            rews = np.clip(rews / np.sqrt(self.ret_rms.var + self.epsilon), -self.clip_reward, self.clip_reward)
        self.ret[dones] = 0
        return obs_n, rews
