"""Generates the frozen oracle replays of MountainCar, MountainCarContinuous and Acrobot
(`tests/golden/orc_{mountaincar,mountaincar_continuous,acrobot}_replay.npz`), in the format of make_golden.py's
orc_cartpole_replay / orc_pendulum_replay, from its own random generator so that the other fixtures are untouched.

Run from the repo root:  python tests/golden/make_golden_envs.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from make_golden import _replay, save  # noqa: E402
from oracle import classic_envs as CE  # noqa: E402

f32 = np.float32


def orc_new_env_replay():
    rng = np.random.default_rng(1)
    n, steps = 16, 60
    a = rng.integers(1, 4, (steps, n))
    save("orc_mountaincar_replay", actions=a, seed=np.array(5), max_steps=np.array(25),
         **_replay(CE.MountainCarBatch(n, seed=5, max_steps=25), a))
    a = rng.uniform(-1.5, 1.5, (steps, n, 1)).astype(f32)
    save("orc_mountaincar_continuous_replay", actions=a, seed=np.array(5), max_steps=np.array(25),
         **_replay(CE.MountainCarContinuousBatch(n, seed=5, max_steps=25), a))
    a = rng.integers(1, 4, (steps, n))
    save("orc_acrobot_replay", actions=a, seed=np.array(5), max_steps=np.array(25),
         **_replay(CE.AcrobotBatch(n, seed=5, max_steps=25), a))


if __name__ == "__main__":
    orc_new_env_replay()
