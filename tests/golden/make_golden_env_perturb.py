"""Generates the frozen oracle replays of the five classic-control envs with observation noise and action delay
(`tests/golden/orc_<kind>_perturb_replay.npz`): mixed per-env noise deviations (some envs and components 0), per-env delays
0 to 4, randomised per-env ranges (some envs fixed, lo == hi), replayed actions, observations of oracle/env_perturb.py, in
the format of make_golden_env_history.py's replays plus `obs_noise` and `action_delay`.  Pendulum also runs under
ScalingWrapperEnv with a k = 3 history, Acrobot with a velocity-free k = 3 history.  Episodes end by truncation in every kind
and by termination in CartPole.  Own random generator, so the other fixtures are untouched.

Run from the repo root:  python tests/golden/make_golden_env_perturb.py
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
from oracle import env_perturb as PB  # noqa: E402

KINDS = ("cartpole", "pendulum", "mountaincar", "mountaincar_continuous", "acrobot")
HISTORY = {"pendulum": (3, False), "acrobot": (3, True)}
SCALED = {"pendulum": (OE.PENDULUM_OBS_LOW, OE.PENDULUM_OBS_HIGH)}
NOISE_SCALE = {"cartpole": 0.05, "pendulum": 0.1, "mountaincar": 0.01, "mountaincar_continuous": 0.01, "acrobot": 0.1}


def random_noise(kind, n, rng):
    """(F0, n) deviations in [0, scale); every third env and a quarter of the other entries 0"""
    s = rng.uniform(0.0, NOISE_SCALE[kind], (PB.BASE_OBS_DIM[kind], n)).astype(np.float32)
    s[rng.random(s.shape) < 0.25] = 0.0
    s[:, ::3] = 0.0
    return s


def make_env(kind, lo, hi, sigma, delay, seed=SEED):
    k, mask = HISTORY.get(kind, (1, False))
    return OE.ParallelEnv(PB.make(kind, N, sigma, delay, k, mask, seed=seed, max_steps=MAX_STEPS[kind], param_ranges=(lo, hi),
                                  scaling=SCALED.get(kind)))


def replay(kind, lo, hi, sigma, delay, actions):
    env = make_env(kind, lo, hi, sigma, delay)
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


def orc_env_perturb_replay():
    rng = np.random.default_rng(19)
    for kind in KINDS:
        lo, hi = random_ranges(kind, N, rng)
        sigma = random_noise(kind, N, rng)
        delay = (np.arange(N) % (PB.MAX_ACTION_DELAY + 1)).astype(np.int32)
        a = actions_for(kind, rng, STEPS, N)
        k, mask = HISTORY.get(kind, (1, False))
        save(f"orc_{kind}_perturb_replay", actions=a, seed=np.array(SEED), max_steps=np.array(MAX_STEPS[kind]), lo=lo, hi=hi,
             obs_noise=sigma, action_delay=delay, history_len=np.array(k), mask_velocities=np.array(mask),
             scaling=np.array(kind in SCALED), **replay(kind, lo, hi, sigma, delay, a))


if __name__ == "__main__":
    orc_env_perturb_replay()
