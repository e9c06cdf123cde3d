"""Generates the frozen oracle replays of the five classic-control envs with an observation history
(`tests/golden/orc_<kind>_history_replay.npz`): k = 3 frames, randomised per-env ranges (some envs fixed, lo == hi), replayed
actions, observations of oracle/env_history.py, in the format of make_golden_env_obs_params.py's replays plus `history_len`,
`mask_velocities` and `scaling`.  CartPole and Acrobot frames are velocity-free, Pendulum runs under ScalingWrapperEnv.
Episodes end by truncation in every kind and by termination in CartPole.  Own random generator, so the other fixtures are
untouched.

Run from the repo root:  python tests/golden/make_golden_env_history.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from make_golden import save  # noqa: E402
from make_golden_env_params import MAX_STEPS, N, SEED, STEPS, actions_for, random_ranges  # noqa: E402
from oracle import envs as OE  # noqa: E402
from oracle import env_history as EH  # noqa: E402

KINDS = ("cartpole", "pendulum", "mountaincar", "mountaincar_continuous", "acrobot")
HISTORY_LEN = 3
MASKED = ("cartpole", "acrobot")
SCALED = {"pendulum": (OE.PENDULUM_OBS_LOW, OE.PENDULUM_OBS_HIGH)}


def make_env(kind, lo, hi, seed=SEED):
    return OE.ParallelEnv(EH.make(kind, N, HISTORY_LEN, kind in MASKED, seed=seed, max_steps=MAX_STEPS[kind],
                                  param_ranges=(lo, hi), scaling=SCALED.get(kind)))


def replay(kind, lo, hi, actions):
    env = make_env(kind, lo, hi)
    obs = [env.observe()]
    R, TE, TR, TO = [], [], [], []
    for a in actions:
        r, te, tr, info = env.act(a)
        R.append(r); TE.append(te); TR.append(tr)
        to = np.zeros_like(obs[0])
        for i in np.nonzero(tr)[0]:
            to[i] = info["terminal_observation"][i]
        TO.append(to); obs.append(env.observe())
    return dict(obs=np.stack(obs), rewards=np.stack(R), term=np.stack(TE), trunc=np.stack(TR), terminal_obs=np.stack(TO))


def orc_env_history_replay():
    rng = np.random.default_rng(18)
    for kind in KINDS:
        lo, hi = random_ranges(kind, N, rng)
        a = actions_for(kind, rng, STEPS, N)
        save(f"orc_{kind}_history_replay", actions=a, seed=np.array(SEED), max_steps=np.array(MAX_STEPS[kind]), lo=lo, hi=hi,
             history_len=np.array(HISTORY_LEN), mask_velocities=np.array(kind in MASKED), scaling=np.array(kind in SCALED),
             **replay(kind, lo, hi, a))


if __name__ == "__main__":
    orc_env_history_replay()
