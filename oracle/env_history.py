"""Oracle (test infrastructure): observation history (frame stacking) and velocity-free frames over any batch.

With history_len = k, env n's observation at step t is [f_{t-k+1} | ... | f_{t-1} | f_t], oldest first; f_j is the frame at
step j: the wrapped batch's observation (raw, or mapped by ScalingBatch), restricted to its non-velocity components
(VELOCITY_FREE) when mask_velocities is set.  HistoryBatch sits above ScalingBatch and the env_params batches and below
ParallelEnv, MonitorWrapper and NormalizeWrapper, which restate the rest unchanged:
  - step() pushes the frame the action was chosen on into the history, then steps; ParallelEnv reads the terminal
    observation after the step and before the reset, so it is the stack that ends in the ended episode's final frame;
  - reset_idx() / reset_all() refill the history with the new frame (Gymnasium's padding_type="reset"), as does restart()
    (the device's reset!, set_state and rewrapping);
  - obs() only reads the history.
"""
import numpy as np

f32 = np.float32
BASE_OBS_DIM = {"cartpole": 4, "pendulum": 3, "mountaincar": 2, "mountaincar_continuous": 2, "acrobot": 6}
VELOCITY_FREE = {"cartpole": (0, 2), "pendulum": (0, 1), "mountaincar": (0,), "mountaincar_continuous": (0,),
                 "acrobot": (0, 1, 2, 3)}
MAX_HISTORY = 4


def frame_dim(kind, mask_velocities=False):
    return len(VELOCITY_FREE[kind]) if mask_velocities else BASE_OBS_DIM[kind]


def history_obs_dim(kind, history_len, mask_velocities=False):
    """F * k of the stacked observation"""
    return frame_dim(kind, mask_velocities) * history_len


class HistoryBatch:
    """`batch`: any batch of a state-based kind (plain, ScalingBatch, or an env_params batch).  obs() = the k-frame stack;
    everything else is forwarded."""

    def __init__(self, batch, history_len=1, mask_velocities=False):
        assert 1 <= history_len <= MAX_HISTORY
        self.b = batch
        self.history_len, self.mask_velocities = int(history_len), bool(mask_velocities)
        self.cols = list(VELOCITY_FREE[batch.kind]) if mask_velocities else list(range(BASE_OBS_DIM[batch.kind]))
        self.hist = np.zeros((batch.n, self.history_len - 1, len(self.cols)), dtype=f32)   # older frames, oldest first
        self.restart()

    def __getattr__(self, name):            # n, kind, p, set_param_ranges, steps, terminated, truncated, state, ...
        return getattr(self.b, name)

    @property
    def obs_dim(self):
        return history_obs_dim(self.b.kind, self.history_len, self.mask_velocities)

    def frame(self):
        return np.asarray(self.b.obs(), dtype=f32)[:, self.cols]

    def _fill(self, idx):
        self.hist[idx] = self.frame()[idx][:, None, :]

    def restart(self):
        """every env's history refilled with its current frame"""
        self._fill(np.arange(self.b.n))

    def obs(self):
        return np.concatenate([self.hist.reshape(self.b.n, -1), self.frame()], axis=1)

    def step(self, actions):
        if self.history_len > 1:
            self.hist = np.concatenate([self.hist[:, 1:], self.frame()[:, None, :]], axis=1)
        return self.b.step(actions)

    def reset_idx(self, idx):
        self.b.reset_idx(idx)
        self._fill(np.asarray(idx))

    def reset_all(self):
        self.b.reset_all()
        self.restart()


def make(kind, n, history_len=1, mask_velocities=False, seed=0, max_steps=None, gid_offset=0, param_ranges=None,
         scaling=None):
    """HistoryBatch over PARAM_BATCHES[kind] (the plain batch when param_ranges is None: it is that batch unchanged);
    scaling = (obs_low, obs_high) of the base observation puts a ScalingBatch between the two"""
    from .env_params import PARAM_BATCHES
    from .envs import ScalingBatch
    kw = dict(seed=seed, gid_offset=gid_offset, param_ranges=param_ranges)
    if max_steps is not None:
        kw["max_steps"] = max_steps
    b = PARAM_BATCHES[kind](n, **kw)
    if scaling is not None:
        b = ScalingBatch(b, *scaling)
    return HistoryBatch(b, history_len, mask_velocities)
