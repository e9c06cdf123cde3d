"""Handles over the C ABI: Context, CudaBatchedEnv (the AbstractParallelEnv), layer/policy,
RolloutBuffer. Mirrors the reference's dispatch surface (src/interfaces/environments.jl:19-157,
src/interfaces/layers.jl:32-134, src/buffers/buffer_types.jl:3-15) in Python because no Julia
toolchain exists in this image; julia/DRiLB200.jl is the same mapping for Julia hosts."""
import ctypes as C

import numpy as np

from . import _lib as L
from .spaces import Box, Discrete

ENV_KINDS = {"cartpole": 0, "pendulum": 1, "synthetic": 2, "mountaincar": 3, "mountaincar_continuous": 4, "acrobot": 5}
ENV_STATE_DIMS = {"cartpole": 4, "pendulum": 2, "synthetic": 0, "mountaincar": 2, "mountaincar_continuous": 2, "acrobot": 4}
# per-env physical parameters (dril_b200.h): (name, default) in the order of the C arrays; names are Gymnasium's attributes
ENV_PARAMS = {
    "cartpole": (("gravity", 9.8), ("masscart", 1.0), ("masspole", 0.1), ("length", 0.5), ("force_mag", 10.0), ("tau", 0.02)),
    "pendulum": (("g", 10.0), ("m", 1.0), ("l", 1.0), ("dt", 0.05)),
    "synthetic": (),
    "mountaincar": (("force", 0.001), ("gravity", 0.0025)),
    "mountaincar_continuous": (("power", 0.0015), ("gravity", 0.0025)),
    "acrobot": (("link_length_1", 1.0), ("link_mass_1", 1.0), ("link_mass_2", 1.0), ("link_com_pos_1", 0.5),
                ("link_com_pos_2", 0.5), ("link_moi", 1.0)),
}


def observation_space_with_params(space, kind):
    """The observation space of an env with observe_params=True: the base space's bounds (scaled or not), then [0, inf) per
    parameter -- the components are raw values, validated >= 0, so the space does not change when the ranges do."""
    P = len(ENV_PARAMS[kind])
    low = np.concatenate([np.asarray(space.low, np.float32).ravel(), np.zeros(P, np.float32)])
    high = np.concatenate([np.asarray(space.high, np.float32).ravel(), np.full(P, np.inf, np.float32)])
    return Box(low, high)


# the non-velocity components of each kind's observation: the frame of an env with mask_velocities=True
VELOCITY_FREE = {"cartpole": (0, 2), "pendulum": (0, 1), "mountaincar": (0,), "mountaincar_continuous": (0,),
                 "acrobot": (0, 1, 2, 3)}
MAX_HISTORY = 4
MAX_ACTION_DELAY = 4
# components of each kind's base observation: the rows of an observation-noise array
BASE_OBS_DIM = {"cartpole": 4, "pendulum": 3, "mountaincar": 2, "mountaincar_continuous": 2, "acrobot": 6}


def observation_space_with_history(space, kind, history_len, mask_velocities):
    """The observation space of an env with an observation history: the bounds (scaled or not) of the frame's components
    (the kept ones with mask_velocities), tiled history_len times, oldest frame first."""
    low, high = np.asarray(space.low, np.float32).ravel(), np.asarray(space.high, np.float32).ravel()
    if mask_velocities:
        idx = list(VELOCITY_FREE[kind])
        low, high = low[idx], high[idx]
    return Box(np.tile(low, history_len), np.tile(high, history_len))


class Context:
    """One CUDA device + stream; not thread-safe (one per GPU)."""
    _default = {}

    def __init__(self, device=0, seed=0):
        self.lib = L.load()
        h = L.P()
        L.check(self.lib.dril_ctx_create(int(device), int(seed), C.byref(h)))
        self.h, self.device, self.seed = h, device, seed
        self.rank, self.nranks = 0, 1

    @classmethod
    def default(cls, device=0):
        if device not in cls._default:
            cls._default[device] = cls(device)
        return cls._default[device]

    def synchronize(self):
        L.check(self.lib.dril_ctx_synchronize(self.h))

    def launch_count(self):
        n = L.c_i64(0)
        L.check(self.lib.dril_ctx_launch_count(self.h, C.byref(n)))
        return n.value

    def sm_count(self):
        n = L.c_i32(0)
        L.check(self.lib.dril_ctx_sm_count(self.h, C.byref(n)))
        return n.value

    def event_record(self, slot):
        L.check(self.lib.dril_ctx_event_record(self.h, slot))

    def event_elapsed_ms(self, a, b):
        ms = L.c_f32(0)
        L.check(self.lib.dril_ctx_event_elapsed_ms(self.h, a, b, C.byref(ms)))
        return ms.value

    def flush_l2(self):
        L.check(self.lib.dril_ctx_flush_l2(self.h))

    def set_profiling(self, on):
        L.check(self.lib.dril_ctx_set_profiling(self.h, int(bool(on))))

    def reset_profile(self):
        L.check(self.lib.dril_ctx_reset_profile(self.h))

    def profile(self):
        out = {}
        for i, name in enumerate(L.KERNEL_KINDS):
            ms, n = L.c_f64(0), L.c_i64(0)
            L.check(self.lib.dril_ctx_get_profile(self.h, i, C.byref(ms), C.byref(n)))
            out[name] = (ms.value, n.value)
        return out

    def comm_init(self, rank, nranks, uid_bytes):
        buf = (C.c_uint8 * 128).from_buffer_copy(uid_bytes)
        L.check(self.lib.dril_comm_init(self.h, rank, nranks, buf))
        self.rank, self.nranks = rank, nranks

    def comm_p2p_setup(self, all_gather, n_slots):
        """Peer-memory gradient allreduce: export this rank's region, exchange the IPC handles with
        `all_gather(bytes) -> list[bytes]` (rank order), import the peers' regions."""
        buf = (C.c_uint8 * 64)()
        L.check(self.lib.dril_comm_p2p_export(self.h, int(n_slots), buf))
        handles = all_gather(bytes(buf))
        assert len(handles) == self.nranks
        blob = (C.c_uint8 * (64 * self.nranks)).from_buffer_copy(b"".join(handles))
        L.check(self.lib.dril_comm_p2p_import(self.h, blob))

    @staticmethod
    def comm_unique_id():
        lib = L.load()
        buf = (C.c_uint8 * 128)()
        L.check(lib.dril_comm_unique_id(buf))
        return bytes(buf)


def set_option(key, value):
    """Process-wide tuning switch of the library (dril_set_option), e.g. set_option("tc", 1)."""
    lib = L.load(require_device=False)
    L.check(lib.dril_set_option(key.encode(), int(value)))


class NormalizeConfig:
    """kwargs of NormalizeWrapperEnv (environment_wrappers/normalizeWrapperEnv.jl:71-80)."""

    def __init__(self, training=True, norm_obs=True, norm_reward=True, clip_obs=10.0, clip_reward=10.0,
                 gamma=0.99, epsilon=1e-8):
        self.training, self.norm_obs, self.norm_reward = training, norm_obs, norm_reward
        self.clip_obs, self.clip_reward, self.gamma, self.epsilon = clip_obs, clip_reward, gamma, epsilon

    def c(self):
        return L.NormCfg(int(self.training), int(self.norm_obs), int(self.norm_reward), self.clip_obs,
                         self.clip_reward, self.gamma, self.epsilon)


class CudaBatchedEnv:
    """AbstractParallelEnv backed by device-resident env state. Replaces
    MultiThreadedParallelEnv(envs) [+ MonitorWrapperEnv + NormalizeWrapperEnv]
    (environment_wrappers/*.jl). Host-copy methods (observe/act) are the slow compatibility
    path used by evaluate_agent and callbacks; training uses the fused device rollout."""

    def __init__(self, kind, n_envs, max_steps=0, obs_dim=0, act_start=1, seed=None, ctx=None,
                 monitor_window=0, normalize=None, gid_offset=0, obs_shape=None, scaling=False, env_params=None,
                 observe_params=False, history_len=1, mask_velocities=False, obs_noise=None, action_delay=0):
        self.kind = kind.lower()
        assert self.kind in ENV_KINDS, f"unknown env kind {kind}"
        self.ctx = ctx or Context.default()
        self.n_envs, self.act_start = int(n_envs), int(act_start)
        self.monitor_window, self.normalize = int(monitor_window), normalize
        self.gid_offset = int(gid_offset)
        if self.kind == "cartpole":
            self.obs_dim, self.max_steps = 4, max_steps or 500
            hi = np.array([4.8, np.inf, 0.41887903, np.inf], dtype=np.float32)
            self._obs_space, self._act_space = Box(-hi, hi), Discrete(2, act_start)
        elif self.kind == "pendulum":
            self.obs_dim, self.max_steps = 3, max_steps or 200
            hi = np.array([1, 1, 8], dtype=np.float32)
            self._obs_space, self._act_space = Box(-hi, hi), Box(np.array([-2.0], np.float32), np.array([2.0], np.float32))
        elif self.kind in ("mountaincar", "mountaincar_continuous"):
            cont = self.kind == "mountaincar_continuous"
            self.obs_dim, self.max_steps = 2, max_steps or (999 if cont else 200)
            self._obs_space = Box(np.array([-1.2, -0.07], np.float32), np.array([0.6, 0.07], np.float32))
            self._act_space = Box(np.array([-1.0], np.float32), np.array([1.0], np.float32)) if cont else Discrete(3, act_start)
        elif self.kind == "acrobot":
            self.obs_dim, self.max_steps = 6, max_steps or 500
            hi = np.array([1, 1, 1, 1, 4 * np.pi, 9 * np.pi], dtype=np.float32)
            self._obs_space, self._act_space = Box(-hi, hi), Discrete(3, act_start)
        else:
            # multi-dimensional Box observations (test/test_buffers.jl:280-314): the feature extractor of the layer is a
            # parameter-free Flatten (layers/layer_helpers.jl:13-25), so the device works on prod(obs_shape) features and only
            # the host-facing arrays carry the shape
            if obs_shape is not None:
                obs_dim = int(np.prod(obs_shape))
            assert obs_dim >= 1
            self.obs_dim, self.max_steps = int(obs_dim), max_steps or 500
            shape = tuple(int(x) for x in obs_shape) if obs_shape is not None else (self.obs_dim,)
            self._obs_space = Box(-np.ones(shape, np.float32), np.ones(shape, np.float32))
            self._act_space = Discrete(2, act_start)
        self.obs_shape = tuple(self._obs_space.size())
        lib = self.ctx.lib
        h = L.P()
        cfg = normalize.c() if normalize is not None else None
        L.check(lib.dril_env_create(self.ctx.h, ENV_KINDS[self.kind], self.n_envs, int(self.max_steps), int(self.obs_dim),
                                    self.act_start, self.gid_offset, C.byref(cfg) if cfg is not None else None,
                                    self.monitor_window, C.byref(h)))
        self.h = h
        self._observe_params = bool(observe_params)
        if self._observe_params:
            # [base observation | the running episode's parameter values]: set before the first observation
            L.check(lib.dril_env_set_observe_params(self.h, 1))
        self.scaling = bool(scaling)
        if self.scaling:
            # ScalingWrapperEnv around every env (scalingWrapperEnv.jl:14-49): spaces become [-1, 1] boxes, the originals are kept
            assert isinstance(self._obs_space, Box) and isinstance(self._act_space, Box), "ScalingWrapperEnv needs Box spaces"
            self.orig_observation_space, self.orig_action_space = self._obs_space, self._act_space
            ol, oh = L.f32(self._obs_space.low).ravel(), L.f32(self._obs_space.high).ravel()
            al, ah = L.f32(self._act_space.low).ravel(), L.f32(self._act_space.high).ravel()
            L.check(lib.dril_env_set_scaling(self.h, 1, L.ptr(ol), L.ptr(oh), L.ptr(al), L.ptr(ah)))
            self._obs_space = Box(-np.ones_like(ol).reshape(self._obs_space.low.shape), np.ones_like(oh).reshape(self._obs_space.low.shape))
            self._act_space = Box(-np.ones_like(al), np.ones_like(ah))
        self._history_len, self._mask_velocities = int(history_len), bool(mask_velocities)
        if self._history_len != 1 or self._mask_velocities:
            # [f_{t-k+1} | ... | f_t], frames without velocities if masked: after Scaling (given the full base bounds above)
            L.check(lib.dril_env_set_obs_history(self.h, self._history_len, int(self._mask_velocities)))
            self._obs_space = observation_space_with_history(self._obs_space, self.kind, self._history_len, self._mask_velocities)
        if self._observe_params:
            self._obs_space = observation_space_with_params(self._obs_space, self.kind)
        if self._observe_params or self._history_len != 1 or self._mask_velocities:
            self.obs_dim = int(self._obs_space.size()[0])
            self.obs_shape = (self.obs_dim,)
            d = L.c_i32(0)
            L.check(lib.dril_env_obs_dim(self.h, C.byref(d)))
            assert d.value == self.obs_dim, (d.value, self.obs_dim)
        self._term = np.zeros(self.n_envs, dtype=bool)
        self._trunc = np.zeros(self.n_envs, dtype=bool)
        self._param_ranges = None
        if env_params:
            self.set_env_params(**env_params)
        self._obs_noise = self._action_delay = None
        if obs_noise is not None:
            self.set_obs_noise(obs_noise)
        if np.any(np.asarray(action_delay) != 0):
            self.set_action_delay(action_delay)
        if seed is not None:
            self.seed(seed)
            self.reset()

    # ---- AbstractParallelEnv interface (interfaces/environments.jl:39-157) ----
    def number_of_envs(self):
        return self.n_envs

    def observation_space(self):
        return self._obs_space

    def action_space(self):
        return self._act_space

    def seed(self, seed):  # Random.seed!(env, seed), wrapper_utils.jl:24-44
        L.check(self.ctx.lib.dril_env_seed(self.h, int(seed)))

    def reset(self):
        L.check(self.ctx.lib.dril_env_reset(self.h))
        self._term[:] = False
        self._trunc[:] = False

    def observe(self):
        out = np.empty((self.n_envs, self.obs_dim), dtype=np.float32)
        L.check(self.ctx.lib.dril_env_observe(self.h, L.ptr(out)))
        return out.reshape((self.n_envs,) + self.obs_shape)

    def act(self, actions):
        """act!(env, actions) -> rewards, terminateds, truncateds, infos (list of dicts)."""
        n = self.n_envs
        if isinstance(self._act_space, Discrete):
            a = np.ascontiguousarray(np.asarray(actions).reshape(n), dtype=np.int64)
        else:
            a = np.ascontiguousarray(np.asarray(actions, dtype=np.float32).reshape(n, -1))
        rewards = np.empty(n, np.float32)
        term = np.empty(n, np.uint8)
        trunc = np.empty(n, np.uint8)
        tobs = np.empty((n, self.obs_dim), np.float32)
        epr = np.empty(n, np.float32)
        epl = np.empty(n, np.int64)
        L.check(self.ctx.lib.dril_env_step(self.h, L.ptr(a), L.ptr(rewards), L.ptr(term), L.ptr(trunc), L.ptr(tobs),
                                           L.ptr(epr), L.ptr(epl)))
        self._term, self._trunc = term.astype(bool), trunc.astype(bool)
        infos = []
        for i in range(n):
            d = {}
            if self._trunc[i]:
                d["terminal_observation"] = tobs[i].reshape(self.obs_shape).copy()
            if self.monitor_window and (self._term[i] or self._trunc[i]):
                d["episode"] = {"r": float(epr[i]), "l": int(epl[i])}
            infos.append(d)
        return rewards, self._term.copy(), self._trunc.copy(), infos

    def terminated(self):
        return self._term.copy()

    def truncated(self):
        return self._trunc.copy()

    def get_info(self):
        return [{} for _ in range(self.n_envs)]

    def is_monitored(self):
        return self.monitor_window > 0

    # ---- wrapper-specific -----------------------------------------------------
    def get_state(self):
        sd = ENV_STATE_DIMS[self.kind]
        st = np.empty((max(sd, 1), self.n_envs), np.float32)
        steps = np.empty(self.n_envs, np.int32)
        L.check(self.ctx.lib.dril_env_get_state(self.h, L.ptr(st), L.ptr(steps)))
        return st[:sd], steps

    def set_state(self, state=None, steps=None):
        st = None if state is None else L.f32(state)
        sp = None if steps is None else np.ascontiguousarray(steps, dtype=np.int32)
        L.check(self.ctx.lib.dril_env_set_state(self.h, L.ptr(st), L.ptr(sp)))

    # ---- observation history ----
    def history_len(self):
        """k of the frame-stacked observation [f_{t-k+1} | ... | f_t] (1: the plain observation)."""
        return self._history_len

    def masks_velocities(self):
        """True if every frame keeps only the non-velocity components (VELOCITY_FREE)."""
        return self._mask_velocities

    # ---- observation noise and action delay ----
    def set_obs_noise(self, std):
        """Per-env observation noise (sensor noise).  `std`: a scalar, an (F0,) vector with one deviation per component of the
        base observation, or an (F0, n_envs) array (F0 = BASE_OBS_DIM[kind]); None turns the noise off.  Component j of every
        observation gets std[j][n] * z added to its raw value (before Scaling, the velocity mask and the history), z ~ N(0, 1)
        a pure function of (seed, env, episode, step, j).  Takes effect at the next observation."""
        if std is None:
            L.check(self.ctx.lib.dril_env_set_obs_noise(self.h, 0, None))
            self._obs_noise = None
            return
        a = np.asarray(std, np.float32)
        if a.ndim == 0:
            a = np.full((BASE_OBS_DIM.get(self.kind, 0), self.n_envs), a, np.float32)
        elif a.ndim == 1:
            a = np.repeat(a[:, None], self.n_envs, axis=1)
        a = np.ascontiguousarray(a, dtype=np.float32)
        assert a.ndim == 2 and a.shape[1] == self.n_envs, f"obs_noise of shape {a.shape}: need (F0, {self.n_envs})"
        L.check(self.ctx.lib.dril_env_set_obs_noise(self.h, a.shape[0], L.ptr(a)))
        self._obs_noise = a.copy()

    def set_action_delay(self, delay):
        """Per-env action delay (actuation delay): an int or an (n_envs,) array of d in [0, MAX_ACTION_DELAY]; env n applies
        the action chosen d steps earlier in its episode (the first action after a reset fills its queue).  None turns the
        delay off.  Restarts every env's queue."""
        if delay is None:
            L.check(self.ctx.lib.dril_env_set_action_delay(self.h, None))
            self._action_delay = None
            return
        d = np.ascontiguousarray(np.broadcast_to(np.asarray(delay, np.int32), (self.n_envs,)), dtype=np.int32)
        L.check(self.ctx.lib.dril_env_set_action_delay(self.h, L.ptr(d)))
        self._action_delay = d.copy()

    def obs_noise(self):
        """(F0, n_envs) float32 standard deviations, or None without observation noise."""
        return None if self._obs_noise is None else self._obs_noise.copy()

    def action_delay(self):
        """(n_envs,) int32 delays, or 0 without action delay."""
        return 0 if self._action_delay is None else self._action_delay.copy()

    # ---- per-env physical parameters ----
    def observes_params(self):
        """True if every observation ends in the running episode's parameter values (observe_params=True)."""
        return self._observe_params

    def set_env_params(self, **kw):
        """Per-env parameter ranges, e.g. set_env_params(length=(0.25, 1.0), masspole=0.2).  Each value is a scalar, an
        (n_envs,) array, or a tuple (lo, hi) of either; every reset draws a value per env from [lo, hi] (a scalar or array is
        a fixed value).  Unnamed parameters keep their defaults (ENV_PARAMS).  With no keyword the env returns to the
        built-in constants (which an env with observe_params=True keeps observing)."""
        names = [nm for nm, _ in ENV_PARAMS[self.kind]]
        unknown = set(kw) - set(names)
        assert not unknown, f"{self.kind} has no parameter(s) {sorted(unknown)}; it has {names}"
        lib, n = self.ctx.lib, self.n_envs
        if not kw:
            if names:
                L.check(lib.dril_env_set_params(self.h, len(names), None, None))
            self._param_ranges = None
            return
        lo = np.empty((len(names), n), np.float32)
        hi = np.empty((len(names), n), np.float32)
        for k, (nm, default) in enumerate(ENV_PARAMS[self.kind]):
            v = kw.get(nm, default)
            a, b = v if isinstance(v, tuple) else (v, v)
            lo[k], hi[k] = np.broadcast_to(np.asarray(a, np.float32), (n,)), np.broadcast_to(np.asarray(b, np.float32), (n,))
        L.check(lib.dril_env_set_params(self.h, len(names), L.ptr(lo), L.ptr(hi)))
        self._param_ranges = {nm: (lo[k].copy(), hi[k].copy()) for k, nm in enumerate(names)}

    def env_param_ranges(self):
        """{name: (lo, hi)} as set by set_env_params, or None for the built-in constants."""
        return None if self._param_ranges is None else dict(self._param_ranges)

    def env_params(self):
        """{name: (n_envs,) float32 array}: each env's parameter values for its running episode."""
        names = [nm for nm, _ in ENV_PARAMS[self.kind]]
        out = np.empty((len(names), self.n_envs), np.float32)
        if names:
            L.check(self.ctx.lib.dril_env_get_params(self.h, len(names), L.ptr(out)))
        return {nm: out[k].copy() for k, nm in enumerate(names)}

    def set_training(self, training):
        L.check(self.ctx.lib.dril_env_set_training(self.h, int(bool(training))))
        if self.normalize is not None:
            self.normalize.training = bool(training)

    def norm_stats(self):
        m = np.empty(self.obs_dim, np.float32)
        v = np.empty(self.obs_dim, np.float32)
        oc, rc = L.c_i64(0), L.c_i64(0)
        rm, rv = L.c_f32(0), L.c_f32(0)
        L.check(self.ctx.lib.dril_env_get_norm_stats(self.h, L.ptr(m), L.ptr(v), C.byref(oc), C.byref(rm), C.byref(rv), C.byref(rc)))
        return dict(obs_mean=m, obs_var=v, obs_count=oc.value, ret_mean=rm.value, ret_var=rv.value, ret_count=rc.value)

    def set_norm_stats(self, s):
        L.check(self.ctx.lib.dril_env_set_norm_stats(self.h, L.ptr(L.f32(s["obs_mean"])), L.ptr(L.f32(s["obs_var"])),
                                                    int(s["obs_count"]), float(s["ret_mean"]), float(s["ret_var"]),
                                                    int(s["ret_count"])))

    def get_original(self):
        o = np.empty((self.n_envs, self.obs_dim), np.float32)
        r = np.empty(self.n_envs, np.float32)
        L.check(self.ctx.lib.dril_env_get_original(self.h, L.ptr(o), L.ptr(r)))
        return o, r

    def monitor_stats(self):
        a, b, n, t = L.c_f32(0), L.c_f32(0), L.c_i64(0), L.c_i64(0)
        L.check(self.ctx.lib.dril_env_monitor_stats(self.h, C.byref(a), C.byref(b), C.byref(n), C.byref(t)))
        return dict(ep_rew_mean=a.value, ep_len_mean=b.value, n_in_window=n.value, total_episodes=t.value)

    def log_stats(self, logger):  # monitorWrapperEnv.jl:64-70
        if not self.monitor_window:
            return
        s = self.monitor_stats()
        if s["n_in_window"] > 0:
            logger.log_scalar("env/ep_rew_mean", s["ep_rew_mean"])
            logger.log_scalar("env/ep_len_mean", s["ep_len_mean"])

    def close(self):
        if self.h:
            self.ctx.lib.dril_env_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DevicePolicy:
    """Device-side actor-critic + optimiser state (the Lux TrainState of the reference)."""

    def __init__(self, ctx, obs_dim, hidden, act_space):
        self.ctx = ctx
        self.obs_dim, self.hidden, self.act_space = int(obs_dim), [int(h) for h in hidden], act_space
        hid = np.asarray(self.hidden, dtype=np.int32)
        h = L.P()
        if isinstance(act_space, Discrete):
            self.act_kind, self.act_n, self.act_elems = 0, act_space.n, 1
            L.check(ctx.lib.dril_policy_create(ctx.h, self.obs_dim, len(self.hidden), L.ptr(hid), 0, act_space.n,
                                               act_space.start, None, None, C.byref(h)))
        else:
            lo, hi = L.f32(act_space.low.reshape(-1)), L.f32(act_space.high.reshape(-1))
            self.act_kind, self.act_n, self.act_elems = 1, lo.size, lo.size
            L.check(ctx.lib.dril_policy_create(ctx.h, self.obs_dim, len(self.hidden), L.ptr(hid), 1, lo.size, 0,
                                               L.ptr(lo), L.ptr(hi), C.byref(h)))
        self.h = h
        n = L.c_i64(0)
        L.check(ctx.lib.dril_policy_num_params(h, C.byref(n)))
        self.n_params = n.value

    def update_path(self):
        """'tensor': the update runs the tcgen05 (3xTF32) loss/grad kernel for this policy; 'mma': the general-shape kernel
        with its wide layers on mma.sync 3xTF32 tiles; 'fp32': the general-shape kernel on FMA tiles only."""
        o = L.c_i32(0)
        L.check(self.ctx.lib.dril_policy_update_path(self.h, C.byref(o)))
        return {1: "tensor", 2: "mma"}.get(o.value, "fp32")

    def set_params(self, flat):
        flat = L.f32(flat)
        L.check(self.ctx.lib.dril_policy_set_params(self.h, L.ptr(flat), flat.size))

    def get_params(self):
        out = np.empty(self.n_params, np.float32)
        L.check(self.ctx.lib.dril_policy_get_params(self.h, L.ptr(out), out.size))
        return out

    def get_opt_state(self):
        m, v = np.empty(self.n_params, np.float32), np.empty(self.n_params, np.float32)
        s = L.c_i64(0)
        L.check(self.ctx.lib.dril_policy_get_opt_state(self.h, L.ptr(m), L.ptr(v), m.size, C.byref(s)))
        return m, v, s.value

    def set_opt_state(self, m, v, step):
        m, v = L.f32(m), L.f32(v)
        L.check(self.ctx.lib.dril_policy_set_opt_state(self.h, L.ptr(m), L.ptr(v), m.size, int(step)))

    def seed(self, seed, step_index=0):
        L.check(self.ctx.lib.dril_policy_seed(self.h, int(seed), int(step_index)))

    def _obs(self, obs):
        return L.f32(np.asarray(obs, dtype=np.float32).reshape(-1, self.obs_dim))

    def _actions_in(self, actions, B):
        if self.act_kind == 0:
            return np.ascontiguousarray(np.asarray(actions).reshape(B), dtype=np.int64)
        return L.f32(np.asarray(actions, dtype=np.float32).reshape(B, self.act_n))

    def forward(self, obs, deterministic=False, env_gids=None):
        obs = self._obs(obs)
        B = obs.shape[0]
        actions = np.empty(B, np.int64) if self.act_kind == 0 else np.empty((B, self.act_n), np.float32)
        values, logp = np.empty(B, np.float32), np.empty(B, np.float32)
        g = None if env_gids is None else np.ascontiguousarray(env_gids, dtype=np.int64)
        L.check(self.ctx.lib.dril_policy_forward(self.h, L.ptr(obs), B, int(deterministic), L.ptr(g), L.ptr(actions),
                                                 L.ptr(values), L.ptr(logp)))
        return actions, values, logp

    def evaluate(self, obs, actions):
        obs = self._obs(obs)
        B = obs.shape[0]
        a = self._actions_in(actions, B)
        v, lp, ent = (np.empty(B, np.float32) for _ in range(3))
        L.check(self.ctx.lib.dril_policy_evaluate(self.h, L.ptr(obs), L.ptr(a), B, L.ptr(v), L.ptr(lp), L.ptr(ent)))
        return v, lp, ent

    def predict_values(self, obs):
        obs = self._obs(obs)
        v = np.empty(obs.shape[0], np.float32)
        L.check(self.ctx.lib.dril_policy_predict_values(self.h, L.ptr(obs), obs.shape[0], L.ptr(v)))
        return v

    def loss_grad(self, obs, actions, adv, ret, old_logp, old_val, hyper):
        obs = self._obs(obs)
        B = obs.shape[0]
        a = self._actions_in(actions, B)
        loss = L.c_f32(0)
        stats = np.zeros(7, np.float32)
        grads = np.zeros(self.n_params, np.float32)
        L.check(self.ctx.lib.dril_ppo_loss_grad(self.h, L.ptr(obs), L.ptr(a), L.ptr(L.f32(adv)), L.ptr(L.f32(ret)),
                                                L.ptr(L.f32(old_logp)), L.ptr(L.f32(old_val)), B, C.byref(hyper),
                                                C.byref(loss), L.ptr(stats), L.ptr(grads)))
        names = ("policy_loss", "value_loss", "entropy_loss", "clip_fraction", "approx_kl_div", "entropy", "ratio")
        return loss.value, dict(zip(names, stats.tolist())), grads

    def optimizer_step(self, grads, hyper):
        g = L.f32(grads)
        norm = L.c_f32(0)
        L.check(self.ctx.lib.dril_optimizer_step(self.h, L.ptr(g), g.size, C.byref(hyper), C.byref(norm)))
        return norm.value

    def close(self):
        if self.h:
            self.ctx.lib.dril_policy_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_BUF_DTYPES = dict(obs=np.float32, rewards=np.float32, values=np.float32, logprobs=np.float32, advantages=np.float32,
                   returns=np.float32, flags=np.uint8, boot=np.float32, last_values=np.float32, episode_r=np.float32,
                   episode_l=np.int32)


class RolloutBuffer:
    """Device-resident RolloutBuffer (buffers/buffer_types.jl:3-15), time-major [n_steps][n_envs]."""

    def __init__(self, observation_space, action_space, gae_lambda, gamma, n_steps, n_envs, ctx=None):
        self.ctx = ctx or Context.default()
        self.gae_lambda, self.gamma, self.n_steps, self.n_envs = float(gae_lambda), float(gamma), int(n_steps), int(n_envs)
        self.obs_dim = int(np.prod(observation_space.size()))
        self.obs_shape = tuple(int(x) for x in observation_space.size())
        self.discrete = isinstance(action_space, Discrete)
        self.act_dim = 1 if self.discrete else int(np.prod(action_space.size()))
        h = L.P()
        L.check(self.ctx.lib.dril_buffer_create(self.ctx.h, self.n_steps, self.n_envs, self.obs_dim,
                                                0 if self.discrete else 1, self.act_dim, C.byref(h)))
        self.h = h

    def __len__(self):
        return self.n_steps * self.n_envs

    def _shape(self, field):
        T, N = self.n_steps, self.n_envs
        if field == "obs":
            return (T, N) + self.obs_shape
        if field == "actions":
            return (T, N, self.act_dim)
        if field == "last_values":
            return (N,)
        return (T, N)

    def download(self, field):
        dt = (np.int32 if self.discrete else np.float32) if field == "actions" else _BUF_DTYPES[field]
        out = np.empty(self._shape(field), dtype=dt)
        L.check(self.ctx.lib.dril_buffer_download(self.h, L.BUF_FIELDS[field], L.ptr(out), out.nbytes))
        return out

    def upload(self, field, arr):
        dt = (np.int32 if self.discrete else np.float32) if field == "actions" else _BUF_DTYPES[field]
        a = np.ascontiguousarray(np.asarray(arr, dtype=dt).reshape(self._shape(field)))
        L.check(self.ctx.lib.dril_buffer_upload(self.h, L.BUF_FIELDS[field], L.ptr(a), a.nbytes))

    def compute_advantages(self, gamma=None, gae_lambda=None):
        L.check(self.ctx.lib.dril_gae(self.h, self.gamma if gamma is None else gamma,
                                      self.gae_lambda if gae_lambda is None else gae_lambda))

    def explained_variance(self):
        out = L.c_f32(0)
        L.check(self.ctx.lib.dril_explained_variance(self.h, C.byref(out)))
        return out.value

    def reference_order(self):
        """Permutation listing time-major sample indices in the reference's trajectory-completion
        order (trajectory.jl:72, rollout_buffer.jl:70-74); for element-wise comparisons only."""
        flags = self.download("flags")
        T, N = flags.shape
        start = np.zeros(N, dtype=np.int64)
        order = []
        for t in range(T):
            for n in range(N):
                if flags[t, n] or t == T - 1:
                    order.extend(range(start[n] * N + n, t * N + n + 1, N))
                    start[n] = t + 1
        return np.asarray(order, dtype=np.int64)

    def close(self):
        if self.h:
            self.ctx.lib.dril_buffer_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def gae_raw(rewards, values, terminated, truncated, boot, last_values, gamma, gae_lambda, ctx=None):
    """Raw-array GAE through dril_gae_raw (parity entry)."""
    ctx = ctx or Context.default()
    r = L.f32(rewards)
    T, N = r.shape
    adv, ret = np.empty((T, N), np.float32), np.empty((T, N), np.float32)
    te = np.ascontiguousarray(terminated, dtype=np.uint8)
    tr = np.ascontiguousarray(truncated, dtype=np.uint8)
    L.check(ctx.lib.dril_gae_raw(ctx.h, L.ptr(r), L.ptr(L.f32(values)), L.ptr(te), L.ptr(tr), L.ptr(L.f32(boot)),
                                 L.ptr(L.f32(last_values)), T, N, gamma, gae_lambda, L.ptr(adv), L.ptr(ret)))
    return adv, ret
