"""Device-side VecNormalize (SURVEY §8f.3).

The reference builds its envs as `VecNormalize(make_vec_env(...), norm_reward=True)` (env.py:8-12): stable_baselines3's
wrapper keeps running moments of the observations and of the discounted returns, and hands the learner normalised
observations / rewards (clip 10, epsilon 1e-8, gamma 0.99).  This class does the same arithmetic on the GPU around any
host vec-env (num_envs, observation_space, action_space, reset(), step()): the raw observations and rewards are
uploaded once per step, the statistics are updated and the normalisation applied by libppx kernels, and the results
stay on the device -- `Policy.act` and `RolloutStorage.add` take CUDA tensors, so the rollout row is written without
another host round trip.  `unnormalize_obs` (used by PPO_RND's warm-up, algorithms.py:392) is provided.  An inner env
that lives on the GPU (its reset() returns a CUDA tensor) is wrapped with no upload at all: actions go to it as CUDA
tensors and its CUDA dones come back; its `episode_stats()` / `behavior()` (raw, unnormalised) are forwarded.

stable_baselines3 is not part of the reference tree nor of this image: the arithmetic follows its published
VecNormalize.step_wait / RunningMeanStd (same update rule as the reference's util.py:9-44, which IS pinned) and is
checked against the numpy restatement in oracle/rollout.py (parity unpinned upstream, stated in DESIGN.md §4).
"""
import numpy as np
import torch

from . import _lib as L
from .util import RunningMeanStd


class VecNormalize(object):
    def __init__(self, venv, training=True, norm_obs=True, norm_reward=True, clip_obs=10.0, clip_reward=10.0, gamma=0.99,
                 epsilon=1e-8, device="cuda"):
        self.venv = venv
        self.num_envs = venv.num_envs
        self.observation_space, self.action_space = venv.observation_space, venv.action_space
        self.device = torch.device(device)
        self.training, self.norm_obs, self.norm_reward = training, norm_obs, norm_reward
        self.clip_obs, self.clip_reward, self.gamma, self.epsilon = float(clip_obs), float(clip_reward), float(gamma), float(epsilon)
        self.obs_rms = RunningMeanStd(shape=tuple(self.observation_space.shape), device=self.device)
        self.ret_rms = RunningMeanStd(shape=(), device=self.device)
        self.ret = torch.zeros(self.num_envs, dtype=torch.float64, device=self.device)
        self.old_obs = None                                     # raw observations of the last step (device)
        self._cuda_inner = False                                # set by reset(): the inner env returns CUDA tensors
        for name in ("episode_stats", "behavior"):              # raw episode statistics / states pass through
            if callable(getattr(venv, name, None)):
                setattr(self, name, getattr(venv, name))

    # ---- helpers ----
    def _up(self, x, dtype):
        return torch.as_tensor(np.ascontiguousarray(x)).to(self.device, dtype, non_blocking=True)

    def normalize_obs(self, obs_dev):
        if not self.norm_obs:
            return obs_dev
        x = obs_dev.reshape(self.num_envs, -1).contiguous()
        out = torch.empty_like(x)
        L.call("ppx_vecnorm_obs", x.data_ptr(), x.shape[0], x.shape[1], self.obs_rms.mean_dev.data_ptr(), self.obs_rms.var_dev.data_ptr(),
               self.epsilon, self.clip_obs, out.data_ptr(), L.stream())
        return out.view(obs_dev.shape)

    def unnormalize_obs(self, obs):
        """obs * sqrt(var + eps) + mean (clipping is not invertible, as upstream)."""
        if not self.norm_obs:
            return obs
        o = obs if isinstance(obs, torch.Tensor) else self._up(obs, torch.float32)
        return (o.double() * torch.sqrt(self.obs_rms.var_dev + self.epsilon) + self.obs_rms.mean_dev).float()

    def get_original_obs(self):
        return self.old_obs

    # ---- VecEnv surface ----
    def reset(self):
        o = self.venv.reset()
        self._cuda_inner = isinstance(o, torch.Tensor) and o.is_cuda
        if self._cuda_inner:
            return self._reset_cuda(o)
        obs = self._up(o, torch.float32)
        self.old_obs = obs
        self.ret.zero_()
        if self.training and self.norm_obs:
            self.obs_rms.update(obs)
        return self.normalize_obs(obs)

    def step(self, actions):
        """actions: CUDA tensor or numpy.  Returns (obs, rewards) as CUDA f32 tensors, dones as the env's numpy bools, infos.
        An inner env on the GPU gets the actions as they are and its CUDA dones come back (no host round trip)."""
        if self._cuda_inner:
            return self._step_cuda(actions)
        a = actions.detach().cpu().numpy() if isinstance(actions, torch.Tensor) else actions
        obs, rews, dones, infos = self.venv.step(a)
        obs_d, r_d = self._up(obs, torch.float32), self._up(rews, torch.float32)
        d_d = self._up(np.asarray(dones), torch.uint8)
        self.old_obs = obs_d
        if self.training and self.norm_obs:
            self.obs_rms.update(obs_d)
        obs_n = self.normalize_obs(obs_d)
        if self.norm_reward:
            out = torch.empty_like(r_d)
            L.call("ppx_vecnorm_reward", r_d.data_ptr(), d_d.data_ptr(), self.ret.data_ptr(), self.num_envs, self.gamma,
                   self.ret_rms.mean_dev.data_ptr(), self.ret_rms.var_dev.data_ptr(), self.ret_rms.count_dev.data_ptr(), self.epsilon,
                   self.clip_reward, int(self.training), out.data_ptr(), L.stream())
            r_d = out
        else:
            self.ret.mul_(self.gamma).add_(r_d.double())
            self.ret[d_d.bool()] = 0.0
        return obs_n, r_d, dones, infos

    # ---- inner env on the GPU: the same arithmetic, no host upload ----
    def _reset_cuda(self, o):
        obs = o.to(torch.float32).contiguous().clone()              # the inner env may overwrite its buffer on step()
        self.old_obs = obs
        self.ret.zero_()
        if self.training and self.norm_obs:
            self.obs_rms.update(obs)
        return self.normalize_obs(obs)

    def _step_cuda(self, actions):
        obs, rews, dones, infos = self.venv.step(actions)
        obs_d = obs.to(torch.float32).contiguous().clone()
        r_d = rews.to(torch.float32).reshape(self.num_envs).contiguous()
        d = dones.reshape(self.num_envs).contiguous()
        d_d = d.view(torch.uint8) if d.dtype == torch.bool else d if d.dtype == torch.uint8 else (d != 0).to(torch.uint8)
        self.old_obs = obs_d
        if self.training and self.norm_obs:
            self.obs_rms.update(obs_d)
        obs_n = self.normalize_obs(obs_d)
        out = torch.empty_like(r_d)
        if self.norm_reward:
            L.call("ppx_vecnorm_reward", r_d.data_ptr(), d_d.data_ptr(), self.ret.data_ptr(), self.num_envs, self.gamma,
                   self.ret_rms.mean_dev.data_ptr(), self.ret_rms.var_dev.data_ptr(), self.ret_rms.count_dev.data_ptr(), self.epsilon,
                   self.clip_reward, int(self.training), out.data_ptr(), L.stream())
        else:
            out.copy_(r_d)
            self.ret.mul_(self.gamma).add_(r_d.double())
            self.ret.masked_fill_(d_d.bool(), 0.0)                  # not boolean indexing: that syncs
        return obs_n, out, d_d, infos
