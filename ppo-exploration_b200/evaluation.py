"""Evaluation of a trained policy on an environment that lives on the GPU (DESIGN.md §3.17).

`evaluate_policy` is stable_baselines3's `evaluate_policy` as a device loop: per step the policy forward, one launch forming
the actions (`ppx_policy_act_eval`), the user's env.step and one launch recording the finished episodes
(`ppx_eval_episode_step`), with no host round trip.  The loop polls a device count of the episodes still missing through
pinned memory every `check_every` steps, as EvolutionStrategy.evaluate does.
"""
import numpy as np
import torch

from . import _lib as L
from . import dist as D
from .env import VecNormalize


def episode_targets(n_eval_episodes, total_envs):
    """Episodes that global env g contributes: SB3's (n_eval_episodes + g) // total_envs, which sum to n_eval_episodes."""
    return (int(n_eval_episodes) + np.arange(int(total_envs), dtype=np.int64)) // int(total_envs)


def merge_episode_tables(returns, lengths, ends, counts):
    """The recorded episodes of per-env tables ([G, kmax] returns / lengths / end steps, counts [G] valid columns per env,
    rows in global env order) in completion order -- by end step, then global env index, the order in which SB3's
    `evaluate_policy` lists them.  Returns (returns f64 [n], lengths int64 [n])."""
    G, kmax = returns.shape
    valid = np.arange(kmax)[None, :] < np.asarray(counts).reshape(G, 1)
    env = np.broadcast_to(np.arange(G)[:, None], (G, kmax))[valid]
    order = np.lexsort((env, ends[valid]))
    return (np.asarray(returns[valid], dtype=np.float64)[order], np.asarray(lengths[valid], dtype=np.int64)[order])


def _check_spaces(policy, env):
    sp = env.action_space
    kind = sp.__class__.__name__
    n = int(sp.n) if kind == "Discrete" else int(sp.shape[0])
    obs_dim = int(env.observation_space.shape[0])
    if kind != policy.action_type or n != policy.action_dim or obs_dim != policy.state_dim:
        raise ValueError(f"the eval env has {kind}({n}) actions and {obs_dim}-dim observations, the policy "
                         f"{policy.action_type}({policy.action_dim}) and {policy.state_dim}")


def _sync_normalization(train_env, env):
    """SB3's sync_envs_normalization for observations: the eval env normalises with the training env's statistics."""
    t = isinstance(train_env, VecNormalize) and train_env.norm_obs
    e = isinstance(env, VecNormalize) and env.norm_obs
    if t != e:
        raise ValueError("the training env and the eval env must both normalise observations (ppx.VecNormalize with "
                         f"norm_obs) or neither; training: {t}, eval: {e}")
    if t:
        for k in ("mean_dev", "var_dev", "count_dev"):
            getattr(env.obs_rms, k).copy_(getattr(train_env.obs_rms, k))


def _buffers(policy, N, kmax):
    key = (N, kmax)
    bufs = getattr(policy, "_eval_bufs", None)
    if bufs is None:
        bufs = policy._eval_bufs = {}
    if key not in bufs:
        dev, discrete = policy.device, policy.action_type == "Discrete"
        z = lambda *s, dtype: torch.zeros(*s, dtype=dtype, device=dev)
        bufs[key] = dict(
            ret=z(N, kmax, dtype=torch.float64), len=z(N, kmax, dtype=torch.int64), end=z(N, kmax, dtype=torch.int64),
            counts=z(N, dtype=torch.int64), state=z(3, dtype=torch.int64),
            actions=z(N, dtype=torch.int64) if discrete else z(N, policy.action_dim, dtype=torch.float64),
            poll=torch.zeros(1, dtype=torch.int64).pin_memory(), poll_event=torch.cuda.Event(),
            host=torch.zeros(N * (3 * kmax + 1), dtype=torch.float64).pin_memory(), host_event=torch.cuda.Event())
    return bufs[key]


def evaluate_policy(model, env, n_eval_episodes=10, *, deterministic=True, max_steps=None, check_every=8):
    """Run `model`'s policy on `env`, an env on the GPU (INTEGRATION.md §4), until n_eval_episodes episodes have finished;
    returns (returns f64 [n], lengths int64 [n]) as numpy arrays in completion order (by end step, then global env index).

    As SB3's `evaluate_policy`, env g of the W x N envs of all ranks contributes its first (n_eval_episodes + g) // (W * N)
    episodes; later episodes are ignored.  Returns and lengths come from the env's `episode_stats()` -- the raw
    (unnormalised) return and length of the episodes the last step ended -- so the env must have it (ppx.EpisodeMonitor adds
    it to any env on the GPU); `infos` are not read.  The env is reset first.  deterministic: the policy's mode
    (`Policy.eval_actions`); otherwise draws from the policy's evaluation stream, keyed by global env, which moves
    `Policy._eval_draws` by one and never the training stream.  max_steps (None: no bound) stops the loop: episodes
    unfinished then are not counted and fewer than n come back.  Steps issued after the last wanted episode ended change
    nothing, so the result does not depend on `check_every`.

    VecNormalize: when `model.env` and `env` both normalise observations, env gets a device copy of the training
    statistics and runs with training=False (restored afterwards); `model.env` is not modified.  Under torch.distributed
    every rank steps its shard (global envs rank * N ...) and all ranks return the same arrays, those of one GPU holding
    every env."""
    n_eval_episodes, check_every = int(n_eval_episodes), int(check_every)
    if n_eval_episodes < 1 or n_eval_episodes >= 1 << 31:
        raise ValueError(f"n_eval_episodes must be in [1, 2^31), got {n_eval_episodes}")
    if check_every < 1 or (max_steps is not None and int(max_steps) < 1):
        raise ValueError(f"check_every={check_every} and max_steps={max_steps} must be >= 1")
    policy = model.policy
    _check_spaces(policy, env)
    stats = getattr(env, "episode_stats", None)
    if not callable(stats):
        raise TypeError("evaluate_policy() reads finished episodes from env.episode_stats() (CUDA f64 returns, int64 lengths); "
                        "wrap the env in ppx.EpisodeMonitor to add it")
    _sync_normalization(getattr(model, "env", None), env)
    was_training = env.training if isinstance(env, VecNormalize) else None
    if was_training is not None:
        env.training = False
    try:
        return _run(policy, env, stats, n_eval_episodes, deterministic, max_steps, check_every)
    finally:
        if was_training is not None:
            env.training = was_training


def _run(policy, env, stats, n, deterministic, max_steps, check_every):
    W, N, Dn = D.world_size(), int(env.num_envs), policy.state_dim
    total, offset = W * N, D.rank() * N
    kmax = int(episode_targets(n, total).max())                # = ceil(n / total)
    obs = env.reset()
    if not (isinstance(obs, torch.Tensor) and obs.is_cuda):
        raise TypeError("evaluate_policy() steps environments that live on the GPU: env.reset() must return a CUDA tensor "
                        f"(got {type(obs).__name__}); for an env returning numpy, loop over predict() on the host")
    b = _buffers(policy, N, kmax)
    b["counts"].zero_()
    b["state"].zero_()
    draw = 0
    if not deterministic:
        policy._eval_draws += 1
        draw = policy.EVAL_DRAW | (policy._eval_draws << 32)
    st = L.stream()
    t, polled = 0, False
    while max_steps is None or t < max_steps:
        if not deterministic and t >= 1 << 32:
            raise RuntimeError("evaluate_policy(): more than 2^32 steps in one stochastic evaluation")
        x = obs.reshape(N, Dn).to(torch.float32).contiguous()
        policy.eval_actions(x, deterministic, (draw | t) if draw else 0, offset, out=b["actions"])
        obs, _, done, _ = env.step(b["actions"])
        ret, lens = stats()
        if not (ret.is_cuda and ret.dtype == torch.float64 and lens.dtype == torch.int64 and ret.is_contiguous()
                and lens.is_contiguous() and ret.numel() == lens.numel() == N):
            raise TypeError("env.episode_stats() must return contiguous CUDA (f64 [N] returns, int64 [N] lengths)")
        d = done.reshape(N).contiguous()
        d = d.view(torch.uint8) if d.dtype == torch.bool else d if d.dtype == torch.uint8 else (d != 0).to(torch.uint8)
        L.call("ppx_eval_episode_step", d.data_ptr(), ret.data_ptr(), lens.data_ptr(), N, n, offset, total, t,
               b["counts"].data_ptr(), b["ret"].data_ptr(), b["len"].data_ptr(), b["end"].data_ptr(), kmax,
               b["state"].data_ptr(), st)
        t += 1
        if t % check_every == 0:
            if polled and b["poll_event"].query() and int(b["poll"][0]) == 0:
                break
            b["poll"].copy_(b["state"][2:3], non_blocking=True)
            b["poll_event"].record()
            polled = True
    # one exchange of [ret | len | end | counts] per rank (f64: lengths and steps are exact below 2^53), one read
    packed = torch.cat([b["ret"].view(-1), b["len"].view(-1).double(), b["end"].view(-1).double(), b["counts"].double()])
    h = b["host"][:packed.numel()] if W == 1 else torch.empty(W * packed.numel(), dtype=torch.float64).pin_memory()
    h.copy_(D.all_gather_cat(packed).view(-1), non_blocking=True)
    b["host_event"].record()
    b["host_event"].synchronize()
    a = h.numpy().reshape(W, -1)
    m = N * kmax
    tab = lambda i: a[:, i * m:(i + 1) * m].reshape(total, kmax)
    return merge_episode_tables(tab(0), tab(1).astype(np.int64), tab(2).astype(np.int64), a[:, 3 * m:].reshape(total).astype(np.int64))
