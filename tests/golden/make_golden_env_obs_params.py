"""Generates the frozen oracle replays of the five classic-control envs with parameter-augmented observations
(`tests/golden/orc_<kind>_obs_params_replay.npz`): randomised per-env ranges (some envs fixed, lo == hi), replayed actions,
observations [base | parameter values] of oracle/env_obs_params.py, in the format of make_golden_env_params.py's replays.
Episodes end by truncation in every kind and by termination in CartPole.  Own random generator, so the other fixtures are
untouched.

Run from the repo root:  python tests/golden/make_golden_env_obs_params.py
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
from oracle import env_obs_params as EOP  # noqa: E402

KINDS = ("cartpole", "pendulum", "mountaincar", "mountaincar_continuous", "acrobot")


def replay(kind, lo, hi, actions):
    env = OE.ParallelEnv(EOP.make(kind, N, seed=SEED, max_steps=MAX_STEPS[kind], param_ranges=(lo, hi)))
    obs, P = [env.observe()], [env.b.p.copy()]
    R, TE, TR, TO = [], [], [], []
    for a in actions:
        r, te, tr, info = env.act(a)
        R.append(r); TE.append(te); TR.append(tr)
        to = np.zeros_like(obs[0])
        for i in np.nonzero(tr)[0]:
            to[i] = info["terminal_observation"][i]
        TO.append(to); obs.append(env.observe()); P.append(env.b.p.copy())
    return dict(obs=np.stack(obs), rewards=np.stack(R), term=np.stack(TE), trunc=np.stack(TR), terminal_obs=np.stack(TO),
                params=np.stack(P))


def orc_env_obs_params_replay():
    rng = np.random.default_rng(16)
    for kind in KINDS:
        lo, hi = random_ranges(kind, N, rng)
        a = actions_for(kind, rng, STEPS, N)
        save(f"orc_{kind}_obs_params_replay", actions=a, seed=np.array(SEED), max_steps=np.array(MAX_STEPS[kind]), lo=lo, hi=hi,
             **replay(kind, lo, hi, a))


if __name__ == "__main__":
    orc_env_obs_params_replay()
