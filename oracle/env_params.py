"""Oracle (test infrastructure): per-env physical parameters and per-episode domain randomisation for the classic-control
batches of oracle/envs.py and oracle/classic_envs.py, restated in NumPy fp32 one rounding at a time like those batches.

Parameter k of env n during its episode e (the index the RESET stream used for that episode's start state) is
lo + (hi - lo) * u, three fp32 roundings, u = u01_f32 of Philox block (gid, e, k // 4, TAG_ENV_PARAMS = 6) word k % 4.
Every reset draws anew; lo == hi is a fixed value.  The derived coefficients are the fixed fp32 sequences of csrc/env.cuh
(the step functions and their *_coef); at the default values they equal the folded constants of the unparametrised batches bit for bit.

The *ParamBatch classes subclass the unparametrised batches: without param_ranges they are those batches unchanged.
"""
import numpy as np

from . import philox
from .classic_envs import AcrobotBatch, MountainCarBatch, MountainCarContinuousBatch
from .envs import CartPoleBatch, PendulumBatch, _sincos32

f32 = np.float32
TAG_ENV_PARAMS = 6

# (name, default) in the order of the parameter arrays (include/dril_b200.h); names are Gymnasium's attributes
ENV_PARAMS = {
    "cartpole": (("gravity", 9.8), ("masscart", 1.0), ("masspole", 0.1), ("length", 0.5), ("force_mag", 10.0), ("tau", 0.02)),
    "pendulum": (("g", 10.0), ("m", 1.0), ("l", 1.0), ("dt", 0.05)),
    "synthetic": (),
    "mountaincar": (("force", 0.001), ("gravity", 0.0025)),
    "mountaincar_continuous": (("power", 0.0015), ("gravity", 0.0025)),
    "acrobot": (("link_length_1", 1.0), ("link_mass_1", 1.0), ("link_mass_2", 1.0), ("link_com_pos_1", 0.5),
                ("link_com_pos_2", 0.5), ("link_moi", 1.0)),
}
# parameters that must be > 0 (the others, gravity / g / force / force_mag / power, must be >= 0)
POSITIVE = {"masscart", "masspole", "length", "tau", "m", "l", "dt", "link_length_1", "link_mass_1", "link_mass_2",
            "link_com_pos_1", "link_com_pos_2", "link_moi"}


def env_param_values(gid, episode, lo, hi, seed):
    """lo, hi (P, n) float32 ranges of the envs with global ids gid (n,) in episode `episode` (n,) -> (P, n) float32."""
    lo = np.asarray(lo, dtype=f32)
    hi = np.asarray(hi, dtype=f32)
    out = np.empty_like(lo)
    ep = np.asarray(episode, dtype=np.int64) & 0xFFFFFFFF
    for k in range(lo.shape[0]):
        if k % 4 == 0:
            xs = philox.philox4x32(gid, ep, k // 4, TAG_ENV_PARAMS, seed)
        out[k] = lo[k] + (hi[k] - lo[k]) * philox.u01_f32(xs[k % 4])
    return out


def default_ranges(kind, n):
    """(lo, hi), both (P, n) float32 at the defaults"""
    d = np.repeat(np.array([v for _, v in ENV_PARAMS[kind]], dtype=f32)[:, None], n, axis=1)
    return d, d.copy()


def check_ranges(kind, lo, hi):
    """the validation of dril_env_set_params: finite, lo <= hi, and the sign each parameter needs; raises ValueError"""
    lo, hi = np.asarray(lo, dtype=f32), np.asarray(hi, dtype=f32)
    for k, (name, _) in enumerate(ENV_PARAMS[kind]):
        if not (np.isfinite(lo[k]).all() and np.isfinite(hi[k]).all() and (lo[k] <= hi[k]).all()):
            raise ValueError(f"{name}: range not finite with lo <= hi")
        if not ((lo[k] > 0).all() if name in POSITIVE else (lo[k] >= 0).all()):
            raise ValueError(f"{name}: lo must be {'>' if name in POSITIVE else '>='} 0")


class _ParamMixin:
    """self.p: (P, n) float32 values of each env's running episode, or None for the built-in constants."""

    def _init_params(self, param_ranges):
        self.plo = self.phi = self.p = None
        if param_ranges is not None:
            npar = len(ENV_PARAMS[self.kind])
            lo, hi = param_ranges
            check_ranges(self.kind, np.reshape(lo, (npar, self.n)), np.reshape(hi, (npar, self.n)))
            self.plo = np.array(lo, dtype=f32).reshape(npar, self.n)
            self.phi = np.array(hi, dtype=f32).reshape(npar, self.n)
            self.p = self.plo.copy()

    def reset_idx(self, idx):
        if self.p is not None:   # the values of the episode that starts now (drawn before the episode counter advances)
            self.p[:, idx] = env_param_values(self.gid[idx], self.episode[idx], self.plo[:, idx], self.phi[:, idx], self.seed)
        super().reset_idx(idx)

    def set_param_ranges(self, lo, hi=None):
        """new ranges: the running episode takes the value its own (gid, episode) draws from them"""
        self._init_params((lo, lo if hi is None else hi))
        self.p = env_param_values(self.gid, self.episode - 1, self.plo, self.phi, self.seed)


class CartPoleParamBatch(_ParamMixin, CartPoleBatch):
    """(gravity, masscart, masspole, length, force_mag, tau); total_mass = masspole + masscart,
    polemass_length = masspole * length"""

    def __init__(self, n_envs, seed=0, max_steps=500, gid_offset=0, act_start=1, param_ranges=None):
        self.n = n_envs
        self._init_params(param_ranges)
        super().__init__(n_envs, seed, max_steps, gid_offset, act_start)

    def step(self, actions):
        if self.p is None:
            return super().step(actions)
        gravity, masscart, masspole, length, force_mag, tau = self.p
        total_mass, pml = masspole + masscart, masspole * length
        a = np.asarray(actions).astype(np.int64) - self.act_start
        x, x_dot, th, th_dot = (self.state[k] for k in range(4))
        force = np.where(a == 1, force_mag, -force_mag).astype(f32)
        sinth, costh = _sincos32(th)
        temp = (force + (pml * (th_dot * th_dot)) * sinth) / total_mass
        thetaacc = ((gravity * sinth) - (costh * temp)) / (length * (self.FOUR_THIRDS - ((masspole * (costh * costh)) / total_mass)))
        xacc = temp - (((pml * thetaacc) * costh) / total_mass)
        x_new = x + tau * x_dot
        x_dot_new = x_dot + tau * xacc
        th_new = th + tau * th_dot
        th_dot_new = th_dot + tau * thetaacc
        self.state = np.stack([x_new, x_dot_new, th_new, th_dot_new]).astype(f32)
        self.steps += 1
        self.terminated = ((x_new < -self.X_THR) | (x_new > self.X_THR) | (th_new < -self.THETA_THR) | (th_new > self.THETA_THR))
        self.truncated = self.steps >= self.max_steps
        return np.ones(self.n, dtype=f32)


class PendulumParamBatch(_ParamMixin, PendulumBatch):
    """(g, m, l, dt); the 15 and 3 of the default step become (3 g) / (2 l) and 3 / (m (l l))"""

    def __init__(self, n_envs, seed=0, max_steps=200, gid_offset=0, param_ranges=None):
        self.n = n_envs
        self._init_params(param_ranges)
        super().__init__(n_envs, seed, max_steps, gid_offset)

    def step(self, actions):
        if self.p is None:
            return super().step(actions)
        g, m, l, dt = self.p
        c_sin, c_u = (f32(3.0) * g) / (f32(2.0) * l), f32(3.0) / (m * (l * l))
        u = np.clip(np.asarray(actions, dtype=f32).reshape(self.n), -self.MAX_TORQUE, self.MAX_TORQUE)
        th, thdot = self.state[0], self.state[1]
        xp = th + self.PI
        an = (xp - self.TWO_PI * np.floor(xp / self.TWO_PI)) - self.PI
        cost = ((an * an) + (f32(0.1) * (thdot * thdot))) + (f32(0.001) * (u * u))
        sinth, _ = _sincos32(th)
        newthdot = thdot + (((c_sin * sinth) + (c_u * u)) * dt)
        newthdot = np.clip(newthdot, -self.MAX_SPEED, self.MAX_SPEED).astype(f32)
        newth = th + newthdot * dt
        self.state = np.stack([newth, newthdot]).astype(f32)
        self.steps += 1
        self.truncated = self.steps >= self.max_steps
        return (-cost).astype(f32)


class MountainCarParamBatch(_ParamMixin, MountainCarBatch):
    """(force, gravity)"""

    def __init__(self, n_envs, seed=0, max_steps=200, gid_offset=0, act_start=1, param_ranges=None):
        self.n = n_envs
        self._init_params(param_ranges)
        super().__init__(n_envs, seed, max_steps, gid_offset, act_start)

    def step(self, actions):
        if self.p is None:
            return super().step(actions)
        force, gravity = self.p
        a = (np.asarray(actions).astype(np.int64) - self.act_start - 1).astype(f32)
        _, c = _sincos32(f32(3.0) * self.state[0])
        self._move((a * force) + (c * -gravity), self.GOAL)
        return np.full(self.n, -1.0, dtype=f32)


class MountainCarContinuousParamBatch(_ParamMixin, MountainCarContinuousBatch):
    """(power, gravity)"""

    def __init__(self, n_envs, seed=0, max_steps=999, gid_offset=0, param_ranges=None):
        self.n = n_envs
        self._init_params(param_ranges)
        super().__init__(n_envs, seed, max_steps, gid_offset)

    def step(self, actions):
        if self.p is None:
            return super().step(actions)
        power, gravity = self.p
        a = np.asarray(actions, dtype=f32).reshape(self.n)
        force = np.clip(a, f32(-1.0), f32(1.0)).astype(f32)
        _, c = _sincos32(f32(3.0) * self.state[0])
        self._move((force * power) - (gravity * c), self.GOAL)
        bonus = np.where(self.terminated, f32(100.0), f32(0.0)).astype(f32)
        return (bonus - (a * a) * f32(0.1)).astype(f32)


class AcrobotParamBatch(_ParamMixin, AcrobotBatch):
    """(link_length_1 l1, link_mass_1 m1, link_mass_2 m2, link_com_pos_1 lc1, link_com_pos_2 lc2, link_moi I), I1 = I2 = I,
    g = 9.8, through the coefficients of `coef` (env.cuh acrobot_coef / acrobot_dsdt)"""

    def __init__(self, n_envs, seed=0, max_steps=500, gid_offset=0, act_start=1, param_ranges=None):
        self.n = n_envs
        self._init_params(param_ranges)
        super().__init__(n_envs, seed, max_steps, gid_offset, act_start)

    @staticmethod
    def coef(p):
        """each coefficient rounded once in the order written"""
        l1, m1, m2, lc1, lc2, moi = (np.asarray(v, dtype=f32) for v in p)
        q = l1 * lc2
        h = m2 * q
        l2 = lc2 * lc2
        return dict(a1=m1 * (lc1 * lc1), p=(l1 * l1) + (lc2 * lc2), k=(f32(2.0) * l1) * lc2, m2=m2, i=moi, l2=l2, q=q,
                    h=h, h2=f32(2.0) * h, g_lc2=(m2 * lc2) * f32(9.8), g_12=((m1 * lc1) + (m2 * l1)) * f32(9.8),
                    j=(m2 * l2) + moi)

    @classmethod
    def dsdt_p(cls, s, a, C):
        """d1 = ((a1 + m2 (p + k c2)) + I) + I, d2 = m2 (l2 + q c2) + I, phi2 = g_lc2 cp2,
        phi1 = (((-h) w2^2) s2 - (h2 (w2 w1)) s2 + g_12 cp1) + phi2, al2 = (((a + (d2 / d1) phi1) - (h w1^2) s2) - phi2) /
        (j - d2^2 / d1), al1 = -(d2 al2 + phi1) / d1"""
        th1, th2, w1, w2 = s
        s2, c2 = _sincos32(th2)
        d1 = ((C["a1"] + C["m2"] * (C["p"] + C["k"] * c2)) + C["i"]) + C["i"]
        d2 = C["m2"] * (C["l2"] + C["q"] * c2) + C["i"]
        _, cp2 = _sincos32((th1 + th2) - cls.HALF_PI)
        phi2 = C["g_lc2"] * cp2
        _, cp1 = _sincos32(th1 - cls.HALF_PI)
        phi1 = ((((-C["h"]) * (w2 * w2)) * s2 - (C["h2"] * (w2 * w1)) * s2) + C["g_12"] * cp1) + phi2
        num = ((a + (d2 / d1) * phi1) - (C["h"] * (w1 * w1)) * s2) - phi2
        al2 = num / (C["j"] - (d2 * d2) / d1)
        al1 = -((d2 * al2) + phi1) / d1
        return np.stack([w1, w2, al1, al2]).astype(f32)

    @classmethod
    def advance_p(cls, s, a, C):
        """one RK4 step of dsdt_p + wrap / clip (AcrobotBatch.advance with the parametrised dynamics)"""
        k1 = cls.dsdt_p(s, a, C)
        k2 = cls.dsdt_p(s + cls.DT2 * k1, a, C)
        k3 = cls.dsdt_p(s + cls.DT2 * k2, a, C)
        k4 = cls.dsdt_p(s + cls.DT * k3, a, C)
        ns = (s + cls.DT6 * (((k1 + f32(2.0) * k2) + f32(2.0) * k3) + k4)).astype(f32)
        ns[0] = cls._wrap(ns[0])
        ns[1] = cls._wrap(ns[1])
        ns[2] = np.clip(ns[2], -cls.MAX_VEL_1, cls.MAX_VEL_1)
        ns[3] = np.clip(ns[3], -cls.MAX_VEL_2, cls.MAX_VEL_2)
        _, c1 = _sincos32(ns[0])
        _, c12 = _sincos32(ns[1] + ns[0])
        return ns, (-c1 - c12) > f32(1.0)

    def step(self, actions):
        if self.p is None:
            return super().step(actions)
        a = (np.asarray(actions).astype(np.int64) - self.act_start - 1).astype(f32)
        self.state, self.terminated = self.advance_p(self.state, a, self.coef(self.p))
        self.steps += 1
        self.truncated = self.steps >= self.max_steps
        return np.where(self.terminated, f32(0.0), f32(-1.0)).astype(f32)


PARAM_BATCHES = {"cartpole": CartPoleParamBatch, "pendulum": PendulumParamBatch, "mountaincar": MountainCarParamBatch,
                 "mountaincar_continuous": MountainCarContinuousParamBatch, "acrobot": AcrobotParamBatch}
