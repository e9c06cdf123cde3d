"""Oracle (test infrastructure): parameter-augmented observations over the batches of oracle/env_params.py.

With observe_params on, env n's observation is [base observation (D components) | p_0 ... p_{P-1}]: the values of the running
episode's parameters in table order, raw fp32, exactly what dril_env_get_params returns.  ObsParamBatch sits above
ScalingBatch (Scaling maps the D base components only) and below ParallelEnv, MonitorWrapper and NormalizeWrapper, which
restate the rest unchanged: ParallelEnv reads the terminal observation before it resets, so a truncated step's terminal
observation carries the values of the episode that ended, and the observation after a reset the values just drawn.

A batch without ranges observes the built-in defaults (lo = hi = the defaults), as the device does.
"""
import numpy as np

from .env_params import ENV_PARAMS, PARAM_BATCHES, default_ranges

f32 = np.float32
BASE_OBS_DIM = {"cartpole": 4, "pendulum": 3, "mountaincar": 2, "mountaincar_continuous": 2, "acrobot": 6}


def obs_params_dim(kind):
    """D + P of the augmented observation"""
    return BASE_OBS_DIM[kind] + len(ENV_PARAMS[kind])


class ObsParamBatch:
    """`batch`: a *ParamBatch, optionally inside a ScalingBatch.  obs() = [batch.obs() | p.T]; everything else forwarded."""

    def __init__(self, batch):
        self.b = batch
        if batch.p is None:
            batch.set_param_ranges(*default_ranges(batch.kind, batch.n))

    def __getattr__(self, name):            # n, kind, p, set_param_ranges, steps, terminated, truncated, state, ...
        return getattr(self.b, name)

    @property
    def obs_dim(self):
        return obs_params_dim(self.b.kind)

    def obs(self):
        return np.concatenate([np.asarray(self.b.obs(), dtype=f32), self.b.p.T.astype(f32)], axis=1)

    def step(self, actions):
        return self.b.step(actions)

    def reset_idx(self, idx):
        self.b.reset_idx(idx)

    def reset_all(self):
        self.b.reset_all()


def make(kind, n, seed=0, max_steps=None, gid_offset=0, param_ranges=None, scaling=None):
    """ObsParamBatch over PARAM_BATCHES[kind]; scaling = (obs_low, obs_high) of the base observation puts a ScalingBatch
    between the two"""
    from .envs import ScalingBatch
    kw = dict(seed=seed, gid_offset=gid_offset, param_ranges=param_ranges)
    if max_steps is not None:
        kw["max_steps"] = max_steps
    b = PARAM_BATCHES[kind](n, **kw)
    if scaling is not None:
        b = ScalingBatch(b, *scaling)
    return ObsParamBatch(b)
