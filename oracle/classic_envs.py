"""Oracle (test infrastructure): MountainCar, MountainCarContinuous and Acrobot batches, restated in NumPy fp32 from the
Gymnasium MountainCar-v0 / MountainCarContinuous-v0 / Acrobot-v1 equations; PARITY UNPINNED (the reference takes its
classic-control envs from the un-vendored ClassicControlEnvironments.jl).

Same conventions as the CartPole / Pendulum batches of oracle/envs.py: every fp32 operation written out one rounding at a time
(no FMA), sin/cos the correctly rounded fp32 values (fp64, rounded once), resets from the Philox RESET stream, Discrete actions
as env-space ints (index = a - act_start).  The batches have the reset_idx / obs / step interface, so ParallelEnv,
MonitorWrapper, NormalizeWrapper and ScalingBatch of oracle/envs.py wrap them unchanged.
"""
import numpy as np

from . import philox
from .envs import _sincos32

f32 = np.float32

MOUNTAINCAR_OBS_LOW = np.array([-1.2, -0.07], dtype=f32)         # MountainCar(-Continuous)-v0 (position, velocity)
MOUNTAINCAR_OBS_HIGH = np.array([0.6, 0.07], dtype=f32)
ACROBOT_OBS_HIGH = np.array([1.0, 1.0, 1.0, 1.0, 4 * np.pi, 9 * np.pi], dtype=f32)   # Acrobot-v1 (cos/sin of both angles, velocities)
ACROBOT_OBS_LOW = -ACROBOT_OBS_HIGH


class _MountainCarBase:
    """Shared state, reset and position update of Gymnasium MountainCar-v0 / MountainCarContinuous-v0, fp32.
    Reset: position U(-0.6, -0.4), velocity 0."""
    obs_dim = 2
    state_dim = 2

    MIN_POS = f32(-1.2)
    MAX_POS = f32(0.6)
    MAX_SPEED = f32(0.07)

    def __init__(self, n_envs, seed=0, max_steps=200, gid_offset=0):
        self.n = n_envs
        self.seed = seed
        self.max_steps = max_steps
        self.gid = np.arange(n_envs, dtype=np.int64) + gid_offset
        self.state = np.zeros((2, n_envs), dtype=f32)
        self.steps = np.zeros(n_envs, dtype=np.int32)
        self.episode = np.zeros(n_envs, dtype=np.int64)
        self.terminated = np.zeros(n_envs, dtype=bool)
        self.truncated = np.zeros(n_envs, dtype=bool)
        self.reset_all()

    def reset_idx(self, idx):
        xs = philox.philox4x32(self.gid[idx], self.episode[idx], 0, philox.TAG_RESET, self.seed)
        self.state[0, idx] = f32(-0.6) + f32(0.2) * philox.u01_f32(xs[0])
        self.state[1, idx] = f32(0.0)
        self.episode[idx] += 1
        self.steps[idx] = 0
        self.terminated[idx] = False
        self.truncated[idx] = False

    def reset_all(self):
        self.reset_idx(np.arange(self.n))

    def obs(self):
        return self.state.T.copy()  # (n, 2): position, velocity

    def _move(self, dv, goal):
        """velocity += dv, clip, position += velocity, clip, left wall; sets terminated."""
        pos, vel = self.state[0], self.state[1]
        vel = np.clip(vel + dv, -self.MAX_SPEED, self.MAX_SPEED).astype(f32)
        pos = np.clip(pos + vel, self.MIN_POS, self.MAX_POS).astype(f32)
        vel = np.where((pos == self.MIN_POS) & (vel < 0), f32(0.0), vel).astype(f32)
        self.state = np.stack([pos, vel]).astype(f32)
        self.steps += 1
        self.terminated = (pos >= goal) & (vel >= f32(0.0))
        self.truncated = self.steps >= self.max_steps


class MountainCarBatch(_MountainCarBase):
    """Gymnasium MountainCar-v0, Discrete(3) (push left / none / right), 200-step TimeLimit, fp32."""
    kind = "mountaincar"
    act_kind = "discrete"
    n_actions = 3

    FORCE = f32(0.001)
    GRAVITY = f32(0.0025)
    GOAL = f32(0.5)

    def __init__(self, n_envs, seed=0, max_steps=200, gid_offset=0, act_start=1):
        self.act_start = act_start
        super().__init__(n_envs, seed, max_steps, gid_offset)

    def step(self, actions):
        """actions: env-space ints (act_start based). Returns rewards (n,) f32."""
        a = (np.asarray(actions).astype(np.int64) - self.act_start - 1).astype(f32)
        _, c = _sincos32(f32(3.0) * self.state[0])
        self._move((a * self.FORCE) + (c * -self.GRAVITY), self.GOAL)
        return np.full(self.n, -1.0, dtype=f32)


class MountainCarContinuousBatch(_MountainCarBase):
    """Gymnasium MountainCarContinuous-v0, Box(1) force on [-1, 1], 999-step TimeLimit, fp32."""
    kind = "mountaincar_continuous"
    act_kind = "continuous"
    act_dim = 1
    act_low = np.array([-1.0], dtype=f32)
    act_high = np.array([1.0], dtype=f32)

    POWER = f32(0.0015)
    GRAVITY = f32(0.0025)
    GOAL = f32(0.45)

    def __init__(self, n_envs, seed=0, max_steps=999, gid_offset=0):
        super().__init__(n_envs, seed, max_steps, gid_offset)

    def step(self, actions):
        """actions: (n, 1) or (n,) fp32 forces (env-space; clipped to [-1, 1] for the dynamics, not for the reward)."""
        a = np.asarray(actions, dtype=f32).reshape(self.n)
        force = np.clip(a, f32(-1.0), f32(1.0)).astype(f32)
        _, c = _sincos32(f32(3.0) * self.state[0])
        self._move((force * self.POWER) - (self.GRAVITY * c), self.GOAL)
        bonus = np.where(self.terminated, f32(100.0), f32(0.0)).astype(f32)
        return (bonus - (a * a) * f32(0.1)).astype(f32)


class AcrobotBatch:
    """Gymnasium Acrobot-v1 ("book" dynamics, no torque noise), Discrete(3) torque -1 / 0 / +1, one RK4 step of dt = 0.2,
    500-step TimeLimit, fp32.  State (theta1, theta2, omega1, omega2); observation
    (cos theta1, sin theta1, cos theta2, sin theta2, omega1, omega2).  Constants m1 = m2 = l1 = I1 = I2 = 1, lc1 = lc2 = 0.5,
    g = 9.8 are folded into exact fp32 products (1.5 g is rounded once)."""
    kind = "acrobot"
    obs_dim = 6
    state_dim = 4
    act_kind = "discrete"
    n_actions = 3

    DT = f32(0.2)
    DT2 = f32(0.1)
    DT6 = f32(0.2) / f32(6.0)
    PI = f32(np.pi)
    TWO_PI = f32(2 * np.pi)
    HALF_PI = f32(np.pi / 2)
    MAX_VEL_1 = f32(4 * np.pi)
    MAX_VEL_2 = f32(9 * np.pi)
    G_LC2 = f32(0.5) * f32(9.8)        # m2 lc2 g
    G_12 = f32(1.5) * f32(9.8)         # (m1 lc1 + m2 l1) g

    def __init__(self, n_envs, seed=0, max_steps=500, gid_offset=0, act_start=1):
        self.n = n_envs
        self.seed = seed
        self.max_steps = max_steps
        self.act_start = act_start
        self.gid = np.arange(n_envs, dtype=np.int64) + gid_offset
        self.state = np.zeros((4, n_envs), dtype=f32)
        self.steps = np.zeros(n_envs, dtype=np.int32)
        self.episode = np.zeros(n_envs, dtype=np.int64)
        self.terminated = np.zeros(n_envs, dtype=bool)
        self.truncated = np.zeros(n_envs, dtype=bool)
        self.reset_all()

    def reset_idx(self, idx):
        xs = philox.philox4x32(self.gid[idx], self.episode[idx], 0, philox.TAG_RESET, self.seed)
        for k in range(4):
            self.state[k, idx] = f32(-0.1) + f32(0.2) * philox.u01_f32(xs[k])
        self.episode[idx] += 1
        self.steps[idx] = 0
        self.terminated[idx] = False
        self.truncated[idx] = False

    def reset_all(self):
        self.reset_idx(np.arange(self.n))

    def obs(self):
        s1, c1 = _sincos32(self.state[0])
        s2, c2 = _sincos32(self.state[1])
        return np.stack([c1, s1, c2, s2, self.state[2], self.state[3]], axis=1).astype(f32)

    @classmethod
    def dsdt(cls, s, a):
        """the book dynamics f(s) for torque a; s: (4, n) f32 -> (4, n) f32"""
        th1, th2, w1, w2 = s
        s2, c2 = _sincos32(th2)
        d1 = ((f32(0.25) + (f32(1.25) + c2)) + f32(1.0)) + f32(1.0)
        d2 = (f32(0.25) + f32(0.5) * c2) + f32(1.0)
        _, cp2 = _sincos32((th1 + th2) - cls.HALF_PI)
        phi2 = cls.G_LC2 * cp2
        _, cp1 = _sincos32(th1 - cls.HALF_PI)
        phi1 = (((f32(-0.5) * (w2 * w2)) * s2 - (w2 * w1) * s2) + cls.G_12 * cp1) + phi2
        num = ((a + (d2 / d1) * phi1) - (f32(0.5) * (w1 * w1)) * s2) - phi2
        al2 = num / (f32(1.25) - (d2 * d2) / d1)
        al1 = -((d2 * al2) + phi1) / d1
        return np.stack([w1, w2, al1, al2]).astype(f32)

    @classmethod
    def _wrap(cls, x):
        """Gymnasium's wrap(x, -pi, pi); non-finite angles are left as they are instead of looping forever"""
        x = x.copy()
        while True:
            m = (x > cls.PI) & np.isfinite(x)
            if not m.any():
                break
            x[m] = x[m] - cls.TWO_PI
        while True:
            m = (x < -cls.PI) & np.isfinite(x)
            if not m.any():
                break
            x[m] = x[m] + cls.TWO_PI
        return x

    @classmethod
    def advance(cls, s, a):
        """one RK4 step + wrap / clip; returns (new state, terminated)"""
        k1 = cls.dsdt(s, a)
        k2 = cls.dsdt(s + cls.DT2 * k1, a)
        k3 = cls.dsdt(s + cls.DT2 * k2, a)
        k4 = cls.dsdt(s + cls.DT * k3, a)
        ns = (s + cls.DT6 * (((k1 + f32(2.0) * k2) + f32(2.0) * k3) + k4)).astype(f32)
        ns[0] = cls._wrap(ns[0])
        ns[1] = cls._wrap(ns[1])
        ns[2] = np.clip(ns[2], -cls.MAX_VEL_1, cls.MAX_VEL_1)
        ns[3] = np.clip(ns[3], -cls.MAX_VEL_2, cls.MAX_VEL_2)
        _, c1 = _sincos32(ns[0])
        _, c12 = _sincos32(ns[1] + ns[0])
        return ns, (-c1 - c12) > f32(1.0)

    def step(self, actions):
        """actions: env-space ints (act_start based). Returns rewards (n,) f32."""
        a = (np.asarray(actions).astype(np.int64) - self.act_start - 1).astype(f32)
        self.state, self.terminated = self.advance(self.state, a)
        self.steps += 1
        self.truncated = self.steps >= self.max_steps
        return np.where(self.terminated, f32(0.0), f32(-1.0)).astype(f32)
