"""Raw environments available without third-party simulators (no gymnasium / ALE / SMAC in this image):
``CartPoleEnv`` - CartPole-v1 dynamics restated from the classic-control equations (BASELINE config 1 plumbing) -
and ``SyntheticAtariEnv`` - Atari-SHAPED frames (84x84x4 uint8), sign-clipped rewards, rare terminals (the
synthetic workload of BASELINE config 2; SURVEY.md section 8d) - and ``SyntheticMuJoCoEnv`` - MuJoCo-SHAPED continuous
control (17-d state, 6-d action in [-1, 1], HalfCheetah / Walker2d sizes) with a reward a policy can learn.  ``XuanCeEnvWrapper`` adds the episode_step /
episode_score bookkeeping of xuance/environment/utils/wrapper.py:76-97 (actions are NOT rescaled: appendix B #17)."""
import math

import numpy as np

from ..common.spaces import Box, Discrete


class CartPoleEnv:
    max_episode_steps = 500

    def __init__(self, seed=None):
        self.gravity, self.masscart, self.masspole = 9.8, 1.0, 0.1
        self.total_mass = self.masspole + self.masscart
        self.length = 0.5
        self.polemass_length = self.masspole * self.length
        self.force_mag, self.tau = 10.0, 0.02
        self.theta_threshold = 12 * 2 * math.pi / 360
        self.x_threshold = 2.4
        high = np.array([self.x_threshold * 2, np.finfo(np.float32).max, self.theta_threshold * 2,
                         np.finfo(np.float32).max], dtype=np.float32)
        self.observation_space = Box(-high, high, dtype=np.float32)
        self.action_space = Discrete(2)
        self.rng = np.random.default_rng(seed)
        self.state, self.steps = None, 0

    def reset(self, seed=None, **kwargs):
        if seed is not None:
            self.rng = np.random.default_rng(seed)
        self.state = self.rng.uniform(-0.05, 0.05, size=4)
        self.steps = 0
        return self.state.astype(np.float32), {}

    def step(self, action):
        x, x_dot, theta, theta_dot = self.state
        force = self.force_mag if int(action) == 1 else -self.force_mag
        costheta, sintheta = math.cos(theta), math.sin(theta)
        temp = (force + self.polemass_length * theta_dot ** 2 * sintheta) / self.total_mass
        thetaacc = (self.gravity * sintheta - costheta * temp) / (
            self.length * (4.0 / 3.0 - self.masspole * costheta ** 2 / self.total_mass))
        xacc = temp - self.polemass_length * thetaacc * costheta / self.total_mass
        x, x_dot = x + self.tau * x_dot, x_dot + self.tau * xacc
        theta, theta_dot = theta + self.tau * theta_dot, theta_dot + self.tau * thetaacc
        self.state = np.array([x, x_dot, theta, theta_dot])
        self.steps += 1
        terminated = bool(x < -self.x_threshold or x > self.x_threshold or theta < -self.theta_threshold
                          or theta > self.theta_threshold)
        truncated = self.steps >= self.max_episode_steps
        return self.state.astype(np.float32), 1.0, terminated, truncated, {}

    def close(self):
        pass

    def render(self, *a, **k):
        return None


class SyntheticAtariEnv:
    max_episode_steps = 27000

    def __init__(self, seed=None, n_actions=4, obs_shape=(84, 84, 4), p_term=0.01):
        self.observation_space = Box(0, 255, obs_shape, np.uint8)
        self.action_space = Discrete(n_actions)
        self.rng = np.random.default_rng(seed)
        self.p_term, self.steps = p_term, 0

    def _frame(self):
        return self.rng.integers(0, 256, size=self.observation_space.shape, dtype=np.uint8)

    def reset(self, seed=None, **kwargs):
        self.steps = 0
        return self._frame(), {}

    def step(self, action):
        self.steps += 1
        r = float(self.rng.choice([-1.0, 0.0, 1.0], p=[0.05, 0.9, 0.05]))
        terminated = bool(self.rng.random() < self.p_term)
        return self._frame(), r, terminated, self.steps >= self.max_episode_steps, {}

    def close(self):
        pass

    def render(self, *a, **k):
        return None


class SyntheticMuJoCoEnv:
    """Continuous-control stand-in of the MuJoCo shapes: observations are i.i.d. standard normal 17-vectors, the action is
    clipped to the Box bounds, and the reward is -||a - W o||^2 for a FIXED matrix W (the same for every env and seed), so a
    policy that learns the linear map o -> W o scores higher than the initial one.  Episodes end by truncation only."""
    max_episode_steps = 100
    obs_dim, act_dim = 17, 6

    def __init__(self, seed=None):
        self.observation_space = Box(-np.inf, np.inf, (self.obs_dim,), np.float32)
        self.action_space = Box(-1.0, 1.0, (self.act_dim,), np.float32)
        # target map: rows of norm ~0.5, so the best action 0.5 * N(0, 1) per dimension mostly lies inside the bounds
        self.W = (np.random.default_rng(12345).normal(size=(self.act_dim, self.obs_dim)) * (0.5 / math.sqrt(self.obs_dim))
                  ).astype(np.float32)
        self.rng = np.random.default_rng(seed)
        self.obs, self.steps = None, 0

    def _observe(self):
        self.obs = self.rng.normal(size=self.obs_dim).astype(np.float32)
        return self.obs.copy()

    def reset(self, seed=None, **kwargs):
        if seed is not None:
            self.rng = np.random.default_rng(seed)
        self.steps = 0
        return self._observe(), {}

    def step(self, action):
        a = np.clip(np.asarray(action, np.float32).reshape(self.act_dim), self.action_space.low, self.action_space.high)
        reward = -float(np.square(a - self.W @ self.obs).sum())
        self.steps += 1
        return self._observe(), reward, False, self.steps >= self.max_episode_steps, {}

    def close(self):
        pass

    def render(self, *a, **k):
        return None


class XuanCeEnvWrapper:
    def __init__(self, env, **kwargs):
        self.env = env
        self._episode_step, self._episode_score = 0, 0.0

    observation_space = property(lambda self: self.env.observation_space)
    action_space = property(lambda self: self.env.action_space)
    max_episode_steps = property(lambda self: self.env.max_episode_steps)

    def reset(self, **kwargs):
        out = self.env.reset(**kwargs)
        obs, info = out if isinstance(out, tuple) else (out, {})
        self._episode_step, self._episode_score = 0, 0.0
        info["episode_step"] = self._episode_step
        return obs, info

    def step(self, action):
        obs, reward, terminated, truncated, info = self.env.step(action)
        self._episode_step += 1
        self._episode_score += reward
        info["episode_step"] = self._episode_step
        info["episode_score"] = self._episode_score
        return obs, reward, terminated, truncated, info

    def render(self, *a, **k):
        return self.env.render(*a, **k)

    def close(self):
        return self.env.close()


REGISTRY_ENV = {"CartPole-v1": CartPoleEnv, "SyntheticAtari": SyntheticAtariEnv, "SyntheticMuJoCo": SyntheticMuJoCoEnv}
