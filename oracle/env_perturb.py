"""Oracle (test infrastructure): observation noise (a noisy sensor) and action delay (a delayed actuator) over a plain or
env_params batch, restated in NumPy like csrc/env.cuh.

Noise: component j of env n's base observation, in its episode e (the index its reset and parameter draws used, i.e.
batch.episode - 1) after s = batch.steps steps of it, is o_j + sigma[j][n] * z_j in fp32 (sigma == 0 leaves o_j untouched);
z_j comes from Philox block (gid, e, 2 s + j // 4, TAG_OBS_NOISE = 7), word pair (j // 2) % 2 as u1 = u01_f32_open,
u2 = u01_f32, through Box-Muller in fp64 with one rounding to fp32: r cos(th) for even j, r sin(th) for odd j,
r = sqrt(-2 log u1), th = 2 pi u2.  The fp64 value lies far closer to its fp32 rounding than fp64's own last-bit differences
between libm implementations (the argument of sincos_rn), so this reproduces the device bit for bit.

Delay: env n applies the action chosen d[n] steps earlier in its episode.  Each env keeps a FIFO queue of the actions its
step() receives; the first action after a restart (a reset, restart_queue(), new delays) fills it.

PerturbBatch sits below ScalingBatch (noise in raw units; the queue holds the actions Scaling has mapped, which is the same
as mapping the action that leaves it), and below HistoryBatch, ParallelEnv, Monitor and Normalize, which restate the rest
unchanged.
"""
import numpy as np

from . import philox

f32 = np.float32
TAG_OBS_NOISE = 7
MAX_ACTION_DELAY = 4
BASE_OBS_DIM = {"cartpole": 4, "pendulum": 3, "mountaincar": 2, "mountaincar_continuous": 2, "acrobot": 6}


def noise_z(gid, episode, steps, n_comp, seed):
    """(n, n_comp) float32 standard normals z_j of envs gid (n,) in episodes `episode` after `steps` steps"""
    gid = np.asarray(gid, dtype=np.int64)
    e = np.asarray(episode, dtype=np.int64) & 0xFFFFFFFF
    s = np.asarray(steps, dtype=np.int64)
    out = np.empty((gid.shape[0], n_comp), dtype=f32)
    for b in range((n_comp + 3) // 4):
        xs = philox.philox4x32(gid, e, (2 * s + b) & 0xFFFFFFFF, TAG_OBS_NOISE, seed)
        for p in range(2):
            if 4 * b + 2 * p >= n_comp:
                break
            u1 = philox.u01_f32_open(xs[2 * p]).astype(np.float64)
            u2 = philox.u01_f32(xs[2 * p + 1]).astype(np.float64)
            r = np.sqrt(-2.0 * np.log(u1))
            th = 6.283185307179586 * u2
            out[:, 4 * b + 2 * p] = (r * np.cos(th)).astype(f32)
            if 4 * b + 2 * p + 1 < n_comp:
                out[:, 4 * b + 2 * p + 1] = (r * np.sin(th)).astype(f32)
    return out


def add_noise(o, sigma, z):
    """o + sigma * z per component in fp32, o itself where sigma == 0 (o, z (n, F0); sigma (F0, n))"""
    o = np.asarray(o, dtype=f32)
    sig = np.asarray(sigma, dtype=f32).T
    return np.where(sig != 0, o + sig * z, o).astype(f32)


def check_noise(kind, sigma, n):
    """the validation of dril_env_set_obs_noise; raises ValueError"""
    sigma = np.asarray(sigma, dtype=f32)
    if sigma.shape != (BASE_OBS_DIM[kind], n):
        raise ValueError(f"{kind}: noise of shape {sigma.shape}, need {(BASE_OBS_DIM[kind], n)}")
    if not (np.isfinite(sigma).all() and (sigma >= 0).all()):
        raise ValueError("noise std must be finite and >= 0")


def check_delay(delay, n):
    """the validation of dril_env_set_action_delay; raises ValueError"""
    d = np.asarray(delay)
    if d.shape != (n,) or (d < 0).any() or (d > MAX_ACTION_DELAY).any():
        raise ValueError(f"delays must be (n,) in [0, {MAX_ACTION_DELAY}]")


class PerturbBatch:
    """`batch`: a plain or env_params batch of a state-based kind.  obs() = the noisy observation, step() applies the
    delayed actions; everything else is forwarded.  obs_noise: (F0, n) deviations or None; action_delay: (n,) or None."""

    def __init__(self, batch, obs_noise=None, action_delay=None):
        self.b = batch
        self.sigma = self.delay = None
        self.q = None
        self.set_obs_noise(obs_noise)
        self.set_action_delay(action_delay)

    def __getattr__(self, name):            # n, kind, p, set_param_ranges, steps, episode, terminated, truncated, state, ...
        return getattr(self.b, name)

    def set_obs_noise(self, sigma):
        if sigma is not None:
            check_noise(self.b.kind, sigma, self.b.n)
            sigma = np.array(sigma, dtype=f32)
        self.sigma = sigma

    def set_action_delay(self, delay):
        if delay is not None:
            check_delay(delay, self.b.n)
            delay = np.array(delay, dtype=np.int64)
        self.delay = delay
        self.restart_queue()

    def restart_queue(self, idx=None):
        """the queues of envs idx (all by default) restart: their next action fills them"""
        if self.q is None or idx is None:
            self.fresh = np.ones(self.b.n, dtype=bool)
            self.q = None
        if idx is not None:
            self.fresh[idx] = True

    def obs(self):
        o = np.asarray(self.b.obs(), dtype=f32)
        if self.sigma is None:
            return o
        z = noise_z(self.b.gid, self.b.episode - 1, self.b.steps, o.shape[1], self.b.seed)
        return add_noise(o, self.sigma, z)

    def step(self, actions):
        if self.delay is None:
            return self.b.step(actions)
        a = np.asarray(actions)
        if self.q is None:
            self.q = np.zeros((self.b.n, MAX_ACTION_DELAY) + a.shape[1:], dtype=a.dtype)
        self.q[self.fresh] = a[self.fresh][:, None]
        self.fresh[:] = False
        d = self.delay
        rows = np.arange(self.b.n)
        out = np.where((d > 0).reshape((-1,) + (1,) * (a.ndim - 1)), self.q[:, 0], a)
        self.q = np.roll(self.q, -1, axis=1)
        has = d > 0
        self.q[rows[has], d[has] - 1] = a[has]
        return self.b.step(out)

    def reset_idx(self, idx):
        self.b.reset_idx(idx)
        self.restart_queue(np.asarray(idx))

    def reset_all(self):
        self.b.reset_all()
        self.restart_queue(np.arange(self.b.n))


def make(kind, n, obs_noise=None, action_delay=None, history_len=1, mask_velocities=False, seed=0, max_steps=None,
         gid_offset=0, param_ranges=None, scaling=None):
    """PerturbBatch over PARAM_BATCHES[kind], then ScalingBatch (scaling = (obs_low, obs_high)) and HistoryBatch as asked"""
    from .env_history import HistoryBatch
    from .env_params import PARAM_BATCHES
    from .envs import ScalingBatch
    kw = dict(seed=seed, gid_offset=gid_offset, param_ranges=param_ranges)
    if max_steps is not None:
        kw["max_steps"] = max_steps
    b = PerturbBatch(PARAM_BATCHES[kind](n, **kw), obs_noise, action_delay)
    if scaling is not None:
        b = ScalingBatch(b, *scaling)
    if history_len != 1 or mask_velocities:
        b = HistoryBatch(b, history_len, mask_velocities)
    return b
