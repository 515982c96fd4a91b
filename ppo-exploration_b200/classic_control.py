"""Gym classic-control environments that live on the GPU (classic_control.cu; DESIGN.md §3.13), and device-side episode
statistics for any env on the GPU.

`ClassicControlVecEnv` steps N copies of CartPole-v1, MountainCar-v0, MountainCarContinuous-v0 or Pendulum-v0 (gym 0.17.x
with its TimeLimit, the 4-tuple API) with ONE libppx launch per step: f64 state on the device, f32 observations, rewards
rounded once from f64 (DummyVecEnv's f32 buffer), uint8 dones, finished envs reset in place.  It follows the env protocol of
INTEGRATION.md §4, so `collect_samples()` and `EvolutionStrategy.evaluate` step it without a host round trip, and it
reports finished episodes through `episode_stats()` instead of `infos` dicts (the learner's `ep_info_buffer` reads them on
the device).  `make_env` is the reference's `make_env` (env.py:8-12) over it; `ToNumpy` puts a numpy surface with SB3-style
`infos` on it, so the host loop can run on identical dynamics.
"""
import numpy as np
import torch

from . import _lib as L
from . import dist as D
from .env import VecNormalize
from .spaces import Box, Discrete

# env id -> (kernel id, state dim, observation dim, time limit, action space)
ENVS = {
    "CartPole-v1": (0, 4, 4, 500, lambda: Discrete(2)),
    "MountainCar-v0": (1, 2, 2, 200, lambda: Discrete(3)),
    "MountainCarContinuous-v0": (2, 2, 2, 999, lambda: Box((1,))),
    "Pendulum-v0": (3, 2, 3, 200, lambda: Box((1,))),
}


class ClassicControlVecEnv:
    """`num_envs` copies of a gym classic-control task on the GPU.

    Reset draws come from Philox keyed by (seed, global env index, the env's episode number): an env's episodes depend on
    neither num_envs nor the rank, and `env_offset` (default under torch.distributed: rank * num_envs) makes this env the
    slice [env_offset, env_offset + num_envs) of a larger one, bit for bit.  `step()` takes CUDA actions (int64 [N] for
    Discrete, f64 [N, 1] for Box; other dtypes and numpy arrays are converted) and returns the env's persistent output
    buffers (obs f32 [N, D], reward [N], done uint8 [N]), overwritten by the next step, and `infos = []`.
    reward_dtype: torch.float32 (DummyVecEnv's buffer, what the learner sees) or torch.float64 (gym's own rewards, e.g. for
    ES fitness).  `episode_stats()` gives the raw f64 return and length of the episodes that the last step() ended;
    `behavior()` the f64 state [N, S] that step reached before any reset (the behaviour characterisation of ES-NSRA)."""

    def __init__(self, env_id, num_envs, seed=0, env_offset=None, device="cuda", reward_dtype=torch.float32):
        if env_id not in ENVS:
            raise ValueError(f"unknown env id {env_id!r}; available: {', '.join(ENVS)}")
        if int(num_envs) < 1:
            raise ValueError(f"num_envs must be >= 1, got {num_envs}")
        if reward_dtype not in (torch.float32, torch.float64):
            raise ValueError(f"reward_dtype must be torch.float32 or torch.float64, got {reward_dtype}")
        self.env_id = env_id
        self._kind, S, obs_dim, self.time_limit, space = ENVS[env_id]
        self.num_envs = N = int(num_envs)
        self.observation_space = Box((obs_dim,))
        self.action_space = space()
        self.discrete = isinstance(self.action_space, Discrete)
        self.device = torch.device(device)
        if env_offset is None:
            env_offset = D.rank() * N if D.world_size() > 1 else 0
        if int(env_offset) < 0:
            raise ValueError(f"env_offset must be >= 0, got {env_offset}")
        self.env_offset, self.seed = int(env_offset), int(seed) % (1 << 64)

        def z(*shape, dtype):
            return torch.zeros(*shape, dtype=dtype, device=self.device)
        self.state = z(S, N, dtype=torch.float64)                   # [S, N]: coalesced in the kernel
        self._elapsed, self._episode = z(N, dtype=torch.int64), z(N, dtype=torch.int64)
        self._mon_ret, self._mon_len = z(N, dtype=torch.float64), z(N, dtype=torch.int64)
        self._ep_ret, self._ep_len = z(N, dtype=torch.float64), z(N, dtype=torch.int64)
        self._obs = z(N, obs_dim, dtype=torch.float32)
        self._rew = z(N, dtype=reward_dtype)
        self._done = z(N, dtype=torch.uint8)
        self._behavior = z(N, S, dtype=torch.float64)
        self._act = z(N, dtype=torch.int64) if self.discrete else z(N, 1, dtype=torch.float64)

    def reset(self):
        """Every env starts its next episode; returns the observation buffer."""
        L.call("ppx_classic_reset", self._kind, self.num_envs, self.env_offset, self.seed, self.state.data_ptr(),
               self._elapsed.data_ptr(), self._episode.data_ptr(), self._mon_ret.data_ptr(), self._mon_len.data_ptr(),
               self._obs.data_ptr(), L.stream())
        return self._obs

    def _actions(self, actions):
        a = self._act
        if (isinstance(actions, torch.Tensor) and actions.device == a.device and actions.dtype == a.dtype
                and actions.is_contiguous() and actions.numel() == a.numel()):
            return actions
        if not isinstance(actions, torch.Tensor):
            actions = torch.as_tensor(np.asarray(actions))
        if actions.numel() != a.numel():
            raise ValueError(f"{self.env_id}: expected {a.numel()} actions, got {actions.numel()}")
        a.copy_(actions.reshape(a.shape), non_blocking=True)
        return a

    def step(self, actions):
        a = self._actions(actions)
        L.call("ppx_classic_step", self._kind, self.num_envs, self.env_offset, self.seed, a.data_ptr(), self.state.data_ptr(),
               self._elapsed.data_ptr(), self._episode.data_ptr(), self._mon_ret.data_ptr(), self._mon_len.data_ptr(),
               self._ep_ret.data_ptr(), self._ep_len.data_ptr(), self._obs.data_ptr(), self._rew.data_ptr(),
               int(self._rew.dtype == torch.float64), self._done.data_ptr(), self._behavior.data_ptr(), L.stream())
        return self._obs, self._rew, self._done, []

    def episode_stats(self):
        """(returns f64 [N], lengths int64 [N]) of the episodes that the last step() ended (other entries are stale)."""
        return self._ep_ret, self._ep_len

    def behavior(self):
        return self._behavior

    def unnormalize_obs(self, obs):
        return obs

    # the device tensors that make up the env's state, and the settings a checkpoint must agree with
    _STATE = ("state", "_elapsed", "_episode", "_mon_ret", "_mon_len", "_ep_ret", "_ep_len", "_obs", "_rew", "_done",
              "_behavior")

    def _settings(self):
        return {"env_id": self.env_id, "num_envs": self.num_envs, "seed": self.seed, "env_offset": self.env_offset,
                "reward_dtype": str(self._rew.dtype).replace("torch.", "")}

    def state_dict(self):
        """Everything the next step() depends on, as CPU tensors (INTEGRATION.md §4): the f64 state, elapsed steps, episode
        numbers (they key the reset draws), the monitor accumulators, the last episode statistics and the output buffers,
        plus env_id, num_envs, seed, env_offset and the reward dtype."""
        sd = self._settings()
        sd.update({k.lstrip("_"): getattr(self, k).cpu() for k in self._STATE})
        return sd

    def load_state_dict(self, sd):
        """Restore `state_dict()`; ValueError if the settings or shapes differ from this env's."""
        from .checkpoint import tensor_into
        for k, mine in self._settings().items():
            if sd.get(k) != mine:
                raise ValueError(f"{self.env_id}: the saved env has {k}={sd.get(k)!r}, this one {mine!r}")
        for k in self._STATE:
            tensor_into(getattr(self, k), sd[k.lstrip("_")], f"env '{k.lstrip('_')}'")


class EpisodeMonitor:
    """`episode_stats()` for any env on the GPU (INTEGRATION.md §4): one extra launch per step accumulates the f64 return
    and the length of every env's episode.  Everything else is forwarded to the wrapped env."""

    def __init__(self, venv):
        self.venv = venv
        self.num_envs = N = venv.num_envs
        self.observation_space, self.action_space = venv.observation_space, venv.action_space
        dev = getattr(venv, "device", None) or torch.device("cuda")
        self._acc_ret, self._ep_ret = (torch.zeros(N, dtype=torch.float64, device=dev) for _ in range(2))
        self._acc_len, self._ep_len = (torch.zeros(N, dtype=torch.int64, device=dev) for _ in range(2))
        if callable(getattr(venv, "state_dict", None)):        # the state protocol only if the wrapped env has it
            self.state_dict, self.load_state_dict = self._state_dict, self._load_state_dict

    def __getattr__(self, name):
        return getattr(self.__dict__["venv"], name)

    def reset(self):
        obs = self.venv.reset()
        self._acc_ret.zero_()
        self._acc_len.zero_()
        return obs

    def step(self, actions):
        obs, rew, done, infos = self.venv.step(actions)
        r = rew.reshape(-1).contiguous()
        if r.dtype not in (torch.float32, torch.float64):
            r = r.double()
        d = done.reshape(-1).contiguous()
        d = d.view(torch.uint8) if d.dtype == torch.bool else (d != 0).to(torch.uint8) if d.dtype != torch.uint8 else d
        L.call("ppx_episode_monitor_step", r.data_ptr(), int(r.dtype == torch.float64), d.data_ptr(), self.num_envs,
               self._acc_ret.data_ptr(), self._acc_len.data_ptr(), self._ep_ret.data_ptr(), self._ep_len.data_ptr(), L.stream())
        return obs, rew, done, infos

    def episode_stats(self):
        return self._ep_ret, self._ep_len

    def _state_dict(self):
        sd = {k.lstrip("_"): getattr(self, k).cpu() for k in ("_acc_ret", "_acc_len", "_ep_ret", "_ep_len")}
        sd["venv"] = self.venv.state_dict()
        return sd

    def _load_state_dict(self, sd):
        from .checkpoint import tensor_into
        for k in ("_acc_ret", "_acc_len", "_ep_ret", "_ep_len"):
            tensor_into(getattr(self, k), sd[k.lstrip("_")], f"episode monitor '{k.lstrip('_')}'")
        self.venv.load_state_dict(sd["venv"])


class ToNumpy:
    """A numpy surface over an env on the GPU: numpy obs / rewards / bool dones and SB3-style `infos` whose finished envs
    carry {"episode": {"r": round(return, 6), "l": length}} from `episode_stats()`, as SB3's Monitor writes them.  One sync
    per step.  Lets the learner's host loop run on exactly the dynamics the device path steps."""

    def __init__(self, env):
        self.env = env
        self.num_envs = env.num_envs
        self.observation_space, self.action_space = env.observation_space, env.action_space
        if callable(getattr(env, "state_dict", None)):          # the state protocol is the wrapped env's
            self.state_dict, self.load_state_dict = env.state_dict, env.load_state_dict

    def reset(self):
        return self.env.reset().cpu().numpy()

    def step(self, actions):
        obs, rew, done, _ = self.env.step(actions)
        ret, lens = self.env.episode_stats()
        o, r, d = obs.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy().astype(bool)
        infos = [{} for _ in range(self.num_envs)]
        idx = np.flatnonzero(d)
        if len(idx):
            rs, ls = ret.cpu().numpy()[idx], lens.cpu().numpy()[idx]
            for k, i in enumerate(idx):
                infos[i] = {"episode": {"r": round(float(rs[k]), 6), "l": int(ls[k])}}
        return o, r, d, infos

    def unnormalize_obs(self, obs):
        return obs


def make_env(env_id, n_envs, seed=0, normalize=True, device="cuda"):
    """The reference's make_env (env.py:8-12) on the GPU: `VecNormalize(env, norm_reward=True)` over a
    ClassicControlVecEnv of n_envs copies (normalize=False: the bare env)."""
    env = ClassicControlVecEnv(env_id, n_envs, seed=seed, device=device)
    return VecNormalize(env, norm_reward=True, device=device) if normalize else env
