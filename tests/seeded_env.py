"""A pure-NumPy environment whose observation stream follows the seed its worker passes to `action_space.seed` (manager
seed + process id), for the data-parallel Learner check (tests/dp_learner_check.py): ranks seed their workers differently,
so they really collect different data.  Two agents, 12-dim observations, episodes of 11 steps."""
import numpy as np


class _Space:
    def __init__(self, n=None, shape=()):
        if n is not None:
            self.n = n
        self.shape = shape
        self.seed_value = 0

    def seed(self, s):
        self.seed_value = int(s)


class MultiDiscrete(_Space):
    """Named like gym's space: the workers report action-space type 1 from the class name."""


class SeededEnv:
    N_AGENTS, OBS, ACT, LEN = 2, 12, 5, 11
    MD = False

    def __init__(self):
        self.action_space = MultiDiscrete(shape=(8,)) if self.MD else _Space(n=self.ACT)
        self.observation_space = _Space(shape=(self.OBS,))
        self.rng = None
        self.t = 0
        self.obs = None

    def _draw(self):
        # the first reset comes after the worker has seeded the action space
        if self.rng is None:
            self.rng = np.random.RandomState(self.action_space.seed_value)
        return (self.rng.randn(self.N_AGENTS, self.OBS) * 2.0 + 0.5).astype(np.float32)

    def reset(self):
        self.t = 0
        self.obs = self._draw()
        return self.obs

    def step(self, actions):
        a = np.asarray(actions, np.float32).reshape(self.N_AGENTS, -1)
        rew = (a[:, 0] == self.obs.argmax(-1) % (3 if self.MD else self.ACT)).astype(np.float32)
        self.t += 1
        self.obs = self._draw()
        return self.obs, list(rew), self.t >= self.LEN, {"state": None}

    def close(self):
        pass


class SeededEnvMD(SeededEnv):
    MD = True


def make_env():
    return SeededEnv()


def make_env_md():
    return SeededEnvMD()
