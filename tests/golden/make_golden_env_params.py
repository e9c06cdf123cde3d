"""Generates the frozen oracle replays of the five classic-control envs with per-env parameters
(`tests/golden/orc_<kind>_params_replay.npz`): randomised per-env ranges (some envs fixed, lo == hi), replayed actions, and
every env's parameter values after each step, in the format of make_golden.py's replays plus `lo`, `hi` (P, n) and
`params` (steps + 1, P, n).  Own random generator, so the other fixtures are untouched.

Run from the repo root:  python tests/golden/make_golden_env_params.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from make_golden import save  # noqa: E402
from oracle import envs as OE  # noqa: E402
from oracle import env_params as EP  # noqa: E402

f32 = np.float32
N, STEPS, SEED = 16, 60, 5
MAX_STEPS = {"cartpole": 25, "pendulum": 20, "mountaincar": 25, "mountaincar_continuous": 25, "acrobot": 25}


def random_ranges(kind, n, rng, spread=0.5):
    """per-env [lo, hi] inside default * [1 - spread, 1 + spread]; every fourth env fixed (lo == hi)"""
    d = np.array([v for _, v in EP.ENV_PARAMS[kind]], dtype=np.float64)[:, None]
    a = d * rng.uniform(1 - spread, 1 + spread, (len(d), n))
    b = d * rng.uniform(1 - spread, 1 + spread, (len(d), n))
    lo, hi = np.minimum(a, b).astype(f32), np.maximum(a, b).astype(f32)
    hi[:, ::4] = lo[:, ::4]
    return lo, hi


def actions_for(kind, rng, steps, n):
    if kind == "cartpole":
        return rng.integers(1, 3, (steps, n))
    if kind in ("mountaincar", "acrobot"):
        return rng.integers(1, 4, (steps, n))
    hi = 2.5 if kind == "pendulum" else 1.5
    return rng.uniform(-hi, hi, (steps, n, 1)).astype(f32)


def replay(kind, lo, hi, actions):
    env = OE.ParallelEnv(EP.PARAM_BATCHES[kind](N, seed=SEED, max_steps=MAX_STEPS[kind], param_ranges=(lo, hi)))
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


def orc_env_params_replay():
    rng = np.random.default_rng(6)
    for kind in ("cartpole", "pendulum", "mountaincar", "mountaincar_continuous", "acrobot"):
        lo, hi = random_ranges(kind, N, rng)
        a = actions_for(kind, rng, STEPS, N)
        save(f"orc_{kind}_params_replay", actions=a, seed=np.array(SEED), max_steps=np.array(MAX_STEPS[kind]), lo=lo, hi=hi,
             **replay(kind, lo, hi, a))


if __name__ == "__main__":
    orc_env_params_replay()
