"""GPU tests of collect_samples' device path (an env whose reset() returns CUDA tensors, INTEGRATION.md §4).

Twin envs with identical table-driven dynamics -- one numpy (the reference's host loop), one torch-CUDA (the device path)
-- whose observations and rewards depend on the action through exact f32 (or f64) arithmetic, so any difference in the
drawn actions shows up.  With the same seeds, every rollout array, the episode count, the count table and the numpy RNG
state after the run must be bit-identical, and so must train()'s losses and weights."""
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

F32 = np.float32


def _tables(N, D, L, seed=0):
    rs = np.random.RandomState(seed)
    return dict(obs=rs.randn(L, N, D).astype(F32), rew=rs.randn(L, N).astype(F32), rew64=rs.randn(L, N),
                done=rs.rand(L, N) < 0.1)


class NumpyTwin:
    """obs' = obs_tab[t+1] + 0.25*a0, reward = rew_tab[t] + [a0 > 0] (Box) / [a == 0] (Discrete), done = done_tab[t]."""

    def __init__(self, tabs, space, f64=False, clamp=False):
        import ppo_exploration_b200 as ppx
        self.tabs, self.space, self.f64, self.clamp = tabs, space, f64, clamp
        self.L, self.num_envs, D = tabs["obs"].shape
        self.observation_space = ppx.Box((D,))
        self.action_space = ppx.Box((2,)) if space == "box" else ppx.Discrete(3)

    def reset(self):
        self.t = 0
        return self.tabs["obs"][0].copy()

    def unnormalize_obs(self, obs):
        return obs

    def step(self, a):
        a = np.array(a)
        if self.clamp:
            lo, hi = (-0.5, 0.5) if self.space == "box" else (0, 1)
            np.clip(a, lo, hi, out=a)
        a0 = (a[:, 0] if self.space == "box" else a).astype(F32)
        hit = (a0 > 0) if self.space == "box" else (a == 0)
        t, self.t = self.t, self.t + 1
        obs = self.tabs["obs"][(t + 1) % self.L] + F32(0.25) * a0[:, None]
        if self.f64:
            rew = self.tabs["rew64"][t % self.L] + hit.astype(np.float64)
        else:
            rew = self.tabs["rew"][t % self.L] + hit.astype(F32)
        done = self.tabs["done"][t % self.L].copy()
        infos = [{"episode": {"r": float(t)}} if (i == 0 and done[0]) else {} for i in range(self.num_envs)]
        return obs, rew, done, infos


class DeviceTwin(NumpyTwin):
    """The same dynamics on the GPU.  reuse: the returned obs / reward / done tensors are overwritten in place every
    step; clamp: the action tensor received is clamped in place (the learner must not depend on either)."""

    def __init__(self, tabs, space, f64=False, clamp=False, reuse=False):
        super().__init__(tabs, space, f64, clamp)
        self.reuse = reuse
        self.d = {k: torch.as_tensor(v).cuda() for k, v in tabs.items()}
        self.bufs = None

    def reset(self):
        self.t = 0
        o = self.d["obs"][0].clone()
        if self.reuse:
            self.bufs = (o, None, None)
        return o

    def step(self, a):
        assert a.is_cuda and a.dtype == (torch.float64 if self.space == "box" else torch.int64)
        if self.clamp:
            lo, hi = (-0.5, 0.5) if self.space == "box" else (0, 1)
            a.clamp_(lo, hi)
        a0 = (a[:, 0] if self.space == "box" else a).float()
        hit = (a0 > 0) if self.space == "box" else (a == 0)
        t, self.t = self.t, self.t + 1
        obs = self.d["obs"][(t + 1) % self.L] + 0.25 * a0[:, None]
        rew = self.d["rew64"][t % self.L] + hit.double() if self.f64 else self.d["rew"][t % self.L] + hit.float()
        done = self.d["done"][t % self.L].clone()
        infos = [{"episode": {"r": float(t)}} if (i == 0 and bool(self.tabs["done"][t % self.L][0])) else {}
                 for i in range(self.num_envs)]
        if self.reuse:
            o, r, d = self.bufs
            o.copy_(obs)
            r = rew if r is None else r.copy_(rew)
            d = done if d is None else d.copy_(done)
            self.bufs = (o, r, d)
            obs, rew, done = o, r, d
        return obs, rew, done, infos


FIELDS = ("observations", "actions", "rewards", "int_rewards", "values", "returns", "action_log_probs", "masks", "advantages",
          "int_values", "int_returns", "int_advantages")


def _run(cls, env, kw, iters=2, seed=3):
    np.random.seed(seed)
    torch.manual_seed(seed)
    m = cls(env=env, **kw)
    rolls = []
    for _ in range(iters):
        m.collect_samples()
        rolls.append({k: getattr(m.rollout, k).clone() for k in FIELDS if hasattr(m.rollout, k)})
        m.train()
        rolls[-1]["losses"] = m.last_losses.copy()
    torch.cuda.synchronize()
    banks = [m.policy.bank.flat.clone()]
    for extra in ("rnd", "intrinsic_module"):
        if hasattr(m, extra):
            banks.append(getattr(m, extra).bank.flat.clone())
    table = m.rollout.count_table.items() if getattr(m.rollout, "count_table", None) is not None else None
    return dict(m=m, rolls=rolls, banks=banks, table=table, episodes=m.num_episodes, infos=len(m.ep_info_buffer),
                rng=np.random.get_state(), timesteps=m.num_timesteps)


def _assert_same(a, b):
    from ppo_exploration_b200.buffer import rng_states_equal
    assert a["m"].device_env is False and b["m"].device_env is True
    for i, (ra, rb) in enumerate(zip(a["rolls"], b["rolls"])):
        for k in ra:
            if k == "losses":
                assert np.array_equal(ra[k], rb[k]), f"iteration {i}: train() losses differ"
            else:
                assert torch.equal(ra[k], rb[k]), f"iteration {i}: rollout.{k} differs"
    for wa, wb in zip(a["banks"], b["banks"]):
        assert torch.equal(wa, wb), "weights after train() differ"
    assert a["table"] == b["table"], "SimHash count tables differ"
    assert a["episodes"] == b["episodes"] and a["infos"] == b["infos"] and a["timesteps"] == b["timesteps"]
    assert a["episodes"] > 0
    assert rng_states_equal(a["rng"], b["rng"]), "numpy RNG state differs"


N, D, T = 64, 8, 16
BASE = dict(nstep=T, batch_size=256, n_epochs=2)

CASES = {
    "ppo_box_h64": ("PPO", "box", False, dict(hidden_size=64)),
    "ppo_box_h64_hash": ("PPO", "box", False, dict(hidden_size=64, sim_hash=True, hash_bits=64)),
    "ppo_box_h64_hash_f64": ("PPO", "box", True, dict(hidden_size=64, sim_hash=True, hash_bits=64)),
    "ppo_discrete_h64_hash": ("PPO", "discrete", False, dict(hidden_size=64, sim_hash=True, hash_bits=64)),
    "ppo_discrete_h128_f64": ("PPO", "discrete", True, dict(hidden_size=128)),
    "ppo_box_h32_hash_f64": ("PPO", "box", True, dict(hidden_size=32, sim_hash=True, hash_bits=64)),
    "rnd_box_h64": ("PPO_RND", "box", False, dict(hidden_size=64, int_hidden_size=32, rnd_start=24)),
    "rnd_discrete_h64_f64": ("PPO_RND", "discrete", True, dict(hidden_size=64, int_hidden_size=32, rnd_start=24)),
    "icm_box_h64": ("PPO_ICM", "box", False, dict(hidden_size=64, int_hidden_size=32)),
    "icm_discrete_h32": ("PPO_ICM", "discrete", False, dict(hidden_size=32, int_hidden_size=32)),
}


@pytest.mark.parametrize("case", list(CASES))
def test_device_path_equals_host_path(case):
    """Whole rollouts (two iterations; PPO_RND's second rollout straddles rnd_start) and train() on both paths."""
    import ppo_exploration_b200 as ppx
    algo, space, f64, kw = CASES[case]
    cls = getattr(ppx, algo)
    tabs = _tables(N, D, 3 * T + 1)
    host = _run(cls, NumpyTwin(tabs, space, f64), dict(BASE, **kw))
    dev = _run(cls, DeviceTwin(tabs, space, f64), dict(BASE, **kw))
    _assert_same(host, dev)


@pytest.mark.parametrize("algo,space,kw", [
    ("PPO", "box", dict(hidden_size=64, sim_hash=True, hash_bits=64)),
    ("PPO_RND", "discrete", dict(hidden_size=64, int_hidden_size=32, rnd_start=24)),
    ("PPO_ICM", "box", dict(hidden_size=64, int_hidden_size=32)),
    ("PPO_ICM", "discrete", dict(hidden_size=64, int_hidden_size=32)),
])
def test_env_buffer_reuse_and_in_place_action_clamp(algo, space, kw):
    """The device env overwrites its returned tensors in place every step and clamps the actions it is given in place:
    the rollout (RND warm-up statistics and ICM bonus included) still equals the numpy twin's."""
    import ppo_exploration_b200 as ppx
    cls = getattr(ppx, algo)
    tabs = _tables(N, D, 3 * T + 1, seed=1)
    host = _run(cls, NumpyTwin(tabs, space, clamp=True), dict(BASE, **kw))
    dev = _run(cls, DeviceTwin(tabs, space, clamp=True, reuse=True), dict(BASE, **kw))
    _assert_same(host, dev)


class _NumpyFacade:
    """VecNormalize's arithmetic behind a numpy surface, so the learner runs the host loop over it."""

    def __init__(self, vn):
        self.vn, self.num_envs = vn, vn.num_envs
        self.observation_space, self.action_space = vn.observation_space, vn.action_space

    def reset(self):
        return self.vn.reset().cpu().numpy()

    def step(self, a):
        o, r, d, i = self.vn.step(a)
        return o.cpu().numpy(), r.cpu().numpy(), d, i

    def unnormalize_obs(self, obs):
        return self.vn.unnormalize_obs(obs)


@pytest.mark.parametrize("algo,kw", [("PPO", dict(hidden_size=64, sim_hash=True, hash_bits=64)),
                                     ("PPO_RND", dict(hidden_size=64, int_hidden_size=32, rnd_start=24))])
def test_vecnormalize_takes_the_device_path_unchanged(algo, kw):
    import ppo_exploration_b200 as ppx
    cls = getattr(ppx, algo)
    tabs = _tables(N, D, 3 * T + 1, seed=2)
    host = _run(cls, _NumpyFacade(ppx.VecNormalize(NumpyTwin(tabs, "box"))), dict(BASE, **kw))
    dev = _run(cls, ppx.VecNormalize(NumpyTwin(tabs, "box")), dict(BASE, **kw))
    _assert_same(host, dev)


def test_device_collect_has_no_sync_and_three_launches_per_step():
    """C2's tensor-core shape (2048 envs, D = 8, Box(2), h = 64, SimHash k = 64): collect_samples runs under
    torch.cuda.set_sync_debug_mode("error"); libppx launches per step = forward + act_record + record_step."""
    import ppo_exploration_b200 as ppx
    from ppo_exploration_b200 import _lib as L
    n, t = 2048, 8
    np.random.seed(0)
    torch.manual_seed(0)
    env = DeviceTwin(_tables(n, 8, 4 * t + 1), "box", reuse=True)
    m = ppx.PPO(env=env, nstep=t, batch_size=4096, n_epochs=1, hidden_size=64, sim_hash=True, hash_bits=64)
    assert m.device_env and m.policy.mlp._fused_args()["tc"]
    m.collect_samples()                                        # warm-up: scratch buffers, SimHash projection upload
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        n0 = L.launch_count()
        m.collect_samples()
        n1 = L.launch_count()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    ro = m.rollout
    ro.sim_hash_recorded()                                     # the per-rollout tail once more, to count its launches
    ro.compute_returns_and_advantages(ro.values[-1], ro.masks[-1])
    n2 = L.launch_count()
    assert (n1 - n0) - (n2 - n1) == 3 * t, (n1 - n0, n2 - n1)


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

    class FixedEnv:
        """Observations, rewards and dones from tables only (the two runs draw different actions per env)."""

        def __init__(self, tabs, cols, f64):
            self.o = torch.round(torch.as_tensor(tabs["obs"][:, cols]) * 0.6).to(dev)      # coarse: repeated codes
            self.r = torch.as_tensor(tabs["rew64" if f64 else "rew"][:, cols]).to(dev)
            self.d = torch.as_tensor(tabs["done"][:, cols]).to(dev)
            self.num_envs = self.o.shape[1]
            self.observation_space, self.action_space = ppx.Box((self.o.shape[2],)), ppx.Box((2,))

        def reset(self):
            self.t = 0
            return self.o[0].clone()

        def step(self, a):
            self.t += 1
            k = self.t % self.o.shape[0]
            return self.o[k].clone(), self.r[k].clone(), self.d[k].clone(), [{}] * self.num_envs

    n, t = 32, 16
    tabs = _tables(n * world, 8, 2 * t + 1, seed=4)
    sl = slice(rank * n, (rank + 1) * n)

    def run(cols, f64):
        np.random.seed(5)
        torch.manual_seed(5)
        m = ppx.PPO(env=FixedEnv(tabs, cols, f64), nstep=t, batch_size=256, n_epochs=1, hidden_size=64, sim_hash=True,
                    hash_bits=16, device=dev)
        rewards = []
        for _ in range(2):                                     # the table persists across rollouts
            m.collect_samples()
            rewards.append(m.rollout.rewards.clone())
        torch.cuda.synchronize()
        return torch.stack(rewards).cpu().numpy(), m.rollout.count_table.items()

    for f64 in (False, True):
        with _single():
            r_ref, tab_ref = run(slice(None), f64)
        r_sh, tab_sh = run(sl, f64)
        assert np.array_equal(r_sh, r_ref[:, :, sl]), f"f64={f64}: sharded device-path SimHash rewards differ from 1 GPU"
        assert tab_sh == tab_ref, f"f64={f64}: sharded count table differs from 1 GPU"
    dist.barrier()
    torch.cuda.synchronize()
    os._exit(0)


def test_sharded_device_collect_simhash_equals_single_gpu():
    import torch.multiprocessing as mp
    from test_gpu_sharded import _free_port
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    ctx = mp.spawn(_worker, args=(2, _free_port()), nprocs=2, join=False)
    while not ctx.join(timeout=600):
        pass
