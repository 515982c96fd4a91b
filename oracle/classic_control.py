"""numpy restatement of gym 0.17.x classic_control (CartPole-v1, MountainCar-v0, MountainCarContinuous-v0, Pendulum-v0)
with its TimeLimit, the 4-tuple API the reference and stable-baselines3 1.x use.

gym is not part of this image: the equations are written from the published gym 0.17 source, in its evaluation order, so
every + - * / rounds as gym's does (parity unpinned upstream, DESIGN.md §4).  Vectorised over envs: state [N, S] f64.
`step` returns the pre-reset state, the f64 reward and the termination flag; the time limit and resets are the caller's.
"""
import math

import numpy as np

SPECS = {  # state dim, obs dim, time limit, action space ("discrete", n) / ("box", low, high)
    "CartPole-v1": dict(S=4, D=4, limit=500, action=("discrete", 2)),
    "MountainCar-v0": dict(S=2, D=2, limit=200, action=("discrete", 3)),
    "MountainCarContinuous-v0": dict(S=2, D=2, limit=999, action=("box", -1.0, 1.0)),
    "Pendulum-v0": dict(S=2, D=3, limit=200, action=("box", -2.0, 2.0)),
}
RESET_RANGES = {  # per state component: uniform (low, high), or a constant
    "CartPole-v1": [(-0.05, 0.05)] * 4,
    "MountainCar-v0": [(-0.6, -0.4), 0.0],
    "MountainCarContinuous-v0": [(-0.6, -0.4), 0.0],
    "Pendulum-v0": [(-np.pi, np.pi), (-1.0, 1.0)],
}
THETA_THRESHOLD = 12 * 2 * math.pi / 360


def _cartpole(s, a):
    gravity, masscart, masspole, length, force_mag, tau = 9.8, 1.0, 0.1, 0.5, 10.0, 0.02
    total_mass = masspole + masscart
    polemass_length = masspole * length
    x, x_dot, theta, theta_dot = s[:, 0], s[:, 1], s[:, 2], s[:, 3]
    force = np.where(np.asarray(a).reshape(-1) == 1, force_mag, -force_mag)
    costheta, sintheta = np.cos(theta), np.sin(theta)
    temp = (force + polemass_length * theta_dot ** 2 * sintheta) / total_mass
    thetaacc = (gravity * sintheta - costheta * temp) / (length * (4.0 / 3.0 - masspole * costheta ** 2 / total_mass))
    xacc = temp - polemass_length * thetaacc * costheta / total_mass
    x = x + tau * x_dot
    x_dot = x_dot + tau * xacc
    theta = theta + tau * theta_dot
    theta_dot = theta_dot + tau * thetaacc
    new = np.stack([x, x_dot, theta, theta_dot], axis=1)
    term = (x < -2.4) | (x > 2.4) | (theta < -THETA_THRESHOLD) | (theta > THETA_THRESHOLD)
    return new, np.ones(len(s)), term


def _mountain_car(s, a):
    position, velocity = s[:, 0].copy(), s[:, 1].copy()
    a = np.asarray(a).reshape(-1).astype(np.int64)
    velocity += (a - 1) * 0.001 + np.cos(3 * position) * (-0.0025)
    velocity = np.clip(velocity, -0.07, 0.07)
    position += velocity
    position = np.clip(position, -1.2, 0.6)
    velocity[(position == -1.2) & (velocity < 0)] = 0
    term = (position >= 0.5) & (velocity >= 0)
    return np.stack([position, velocity], axis=1), -np.ones(len(s)), term


def _mountain_car_continuous(s, a):
    position, velocity = s[:, 0].copy(), s[:, 1].copy()
    a = np.asarray(a, dtype=np.float64).reshape(-1)
    force = np.minimum(np.maximum(a, -1.0), 1.0)
    velocity += force * 0.0015 - 0.0025 * np.cos(3 * position)
    velocity = np.where(velocity > 0.07, 0.07, velocity)
    velocity = np.where(velocity < -0.07, -0.07, velocity)
    position += velocity
    position = np.where(position > 0.6, 0.6, position)
    position = np.where(position < -1.2, -1.2, position)
    velocity[(position == -1.2) & (velocity < 0)] = 0
    term = (position >= 0.45) & (velocity >= 0)
    reward = np.where(term, 100.0, 0.0) - a * a * 0.1             # math.pow(action[0], 2) * 0.1: the unclipped action
    return np.stack([position, velocity], axis=1), reward, term


def angle_normalize(x):
    return ((x + np.pi) % (2 * np.pi)) - np.pi


def _pendulum(s, a):
    g, m, l, dt = 10.0, 1.0, 1.0, 0.05
    th, thdot = s[:, 0], s[:, 1]
    u = np.clip(np.asarray(a, dtype=np.float64).reshape(-1), -2.0, 2.0)
    costs = angle_normalize(th) ** 2 + .1 * thdot ** 2 + .001 * (u ** 2)
    newthdot = thdot + (-3 * g / (2 * l) * np.sin(th + np.pi) + 3. / (m * l ** 2) * u) * dt
    newth = th + newthdot * dt
    newthdot = np.clip(newthdot, -8.0, 8.0)
    return np.stack([newth, newthdot], axis=1), -costs, np.zeros(len(s), dtype=bool)


_STEP = {"CartPole-v1": _cartpole, "MountainCar-v0": _mountain_car, "MountainCarContinuous-v0": _mountain_car_continuous,
         "Pendulum-v0": _pendulum}


def step(env_id, state, actions):
    """One step from state [N, S] f64: (new state [N, S] f64 before any reset, reward f64 [N], terminated bool [N])."""
    return _STEP[env_id](np.asarray(state, dtype=np.float64), actions)


def observation(env_id, state):
    """The f32 observation DummyVecEnv's buffer holds for state [N, S]."""
    s = np.asarray(state, dtype=np.float64)
    if env_id == "Pendulum-v0":
        return np.stack([np.cos(s[:, 0]), np.sin(s[:, 0]), s[:, 1]], axis=1).astype(np.float32)
    return s.astype(np.float32)
