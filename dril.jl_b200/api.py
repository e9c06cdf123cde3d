"""Host-side mirror of the reference's public API for the hot path: ActorCriticLayer, PPO, Agent,
train!, collect_rollout!, evaluate_agent, extract_policy, callbacks and the logger interface.
Names, argument meaning and return values follow the reference (citations per function); Julia's
`f!` spellings drop the bang."""
import ctypes as C
import time
from dataclasses import dataclass, field

import numpy as np

from . import _lib as L
from .core import Context, CudaBatchedEnv, DevicePolicy, NormalizeConfig, RolloutBuffer
from .spaces import Box, Discrete


# ---- wrappers as constructors (environment_wrappers/*.jl): the wrapper stack is fused into the
# ---- device env, so "wrapping" re-creates the batched env with the extra stage switched on ----
def MultiThreadedParallelEnv(kind, n_envs, **kw):
    return CudaBatchedEnv(kind, n_envs, **kw)


BroadcastedParallelEnv = MultiThreadedParallelEnv


def _rewrap(env, **over):
    """The env re-created with `over` switched on: state and step counters are carried over through set_state, which, like
    dril_env_set_state, restarts an observation history from each env's current frame.  Automatic domain randomisation is
    turned on again from its configuration (adr_config): the ranges it reached and its buffers restart at round 0, so wrap
    before training."""
    args = dict(kind=env.kind, n_envs=env.n_envs, max_steps=env.max_steps, obs_dim=env.obs_dim,
                act_start=env.act_start, ctx=env.ctx, monitor_window=env.monitor_window,
                normalize=env.normalize, gid_offset=env.gid_offset, scaling=env.scaling,
                obs_shape=env.obs_shape if len(env.obs_shape) > 1 else None, env_params=env.env_param_ranges(),
                observe_params=env.observes_params(), history_len=env.history_len(),
                mask_velocities=env.masks_velocities(), obs_noise=env.obs_noise(), action_delay=env.action_delay(),
                adr=env.adr_config())
    args.update(over)
    kind, n = args.pop("kind"), args.pop("n_envs")
    st, steps = env.get_state()
    new = CudaBatchedEnv(kind, n, **args)
    new.set_state(st if st.shape[0] else None, steps)
    env.close()
    return new


def MonitorWrapperEnv(env, stats_window=100):
    """monitorWrapperEnv.jl:16-24."""
    return _rewrap(env, monitor_window=stats_window)


def ScalingWrapperEnv(env):
    """scalingWrapperEnv.jl:14-49: observations and actions of a Box/Box env mapped to [-1, 1]; applied per env, i.e. below
    Monitor / Normalize whatever the order of the calls."""
    return _rewrap(env, scaling=True)


def NormalizeWrapperEnv(env, **kw):
    """normalizeWrapperEnv.jl:71-105."""
    return _rewrap(env, normalize=NormalizeConfig(**kw))


# ---- layers (layers/layer_constructors.jl) -----------------------------------------------
def _orthogonal(rng, out_dims, in_dims, gain):
    a = rng.standard_normal((max(out_dims, in_dims), min(out_dims, in_dims)))
    q, r = np.linalg.qr(a)
    q = q * np.sign(np.diag(r))
    if out_dims < in_dims:
        q = q.T
    return (gain * q[:out_dims, :in_dims]).astype(np.float32)


class ActorCriticLayer:
    """ActorCriticLayer(observation_space, action_space; hidden_dims=[64,64], activation=tanh,
    shared_features=true, log_std_init=0) — layer_constructors.jl:3-96. Two independent tanh
    MLPs; `shared_features` only names the (parameter-free) feature extractor."""

    def __init__(self, observation_space, action_space, hidden_dims=(64, 64), activation="tanh",
                 shared_features=True, log_std_init=0.0):
        assert activation in ("tanh", np.tanh), "only tanh is implemented on the device path"
        self.observation_space, self._action_space = observation_space, action_space
        self.hidden_dims = [int(h) for h in hidden_dims]
        self.shared_features, self.log_std_init = shared_features, float(log_std_init)
        self.obs_dim = int(np.prod(observation_space.size()))
        self.discrete = isinstance(action_space, Discrete)
        self.act_n = action_space.n if self.discrete else int(np.prod(action_space.size()))

    def action_space(self):
        return self._action_space

    def layer_dims(self, net):
        out = self.act_n if net == 0 else 1
        if not self.hidden_dims:
            return [(self.obs_dim, 1)]   # layer_helpers.jl:33
        d = [(self.obs_dim, self.hidden_dims[0])]
        d += [(self.hidden_dims[i - 1], self.hidden_dims[i]) for i in range(1, len(self.hidden_dims))]
        return d + [(self.hidden_dims[-1], out)]

    def parameterlength(self):  # layer_lux.jl:82-115
        n = sum(i * o + o for net in (0, 1) for (i, o) in self.layer_dims(net))
        return n + (0 if self.discrete else self.act_n)

    def setup(self, rng):
        """Lux.setup analogue: flat ComponentVector-order parameters. Orthogonal init with gains
        sqrt(2) / 0.01 / 1.0, zero bias (layer_constructors.jl:16-20,61-65)."""
        parts = []
        for net, out_gain in ((0, 0.01), (1, 1.0)):
            dims = self.layer_dims(net)
            for li, (i, o) in enumerate(dims):
                gain = out_gain if li == len(dims) - 1 else np.sqrt(2.0)
                w_oi = _orthogonal(rng, o, i, gain)
                parts += [np.ascontiguousarray(w_oi.T).reshape(-1), np.zeros(o, np.float32)]
        if not self.discrete:
            parts.append(np.full(self.act_n, self.log_std_init, np.float32))
        return np.concatenate(parts).astype(np.float32)

    def param_views(self, flat):
        """NamedTuple-like view (layer_lux.jl:4-52): actor_head/critic_head layer_i (weight (out,in), bias), log_std."""
        out, p = {}, 0
        for net, name in ((0, "actor_head"), (1, "critic_head")):
            layers = {}
            for li, (i, o) in enumerate(self.layer_dims(net)):
                w = flat[p:p + i * o].reshape(i, o).T
                p += i * o
                layers[f"layer_{li + 1}"] = {"weight": w, "bias": flat[p:p + o]}
                p += o
            out[name] = layers
        if not self.discrete:
            out["log_std"] = flat[p:p + self.act_n]
        return out


DiscreteActorCriticLayer = ActorCriticLayer
ContinuousActorCriticLayer = ActorCriticLayer


# ---- PPO (algorithms/ppo.jl:25-40) ---------------------------------------------------------
@dataclass
class PPO:
    gamma: float = 0.99
    gae_lambda: float = 0.95
    clip_range: float = 0.2
    clip_range_vf: float | None = None
    ent_coef: float = 0.0
    vf_coef: float = 0.5
    max_grad_norm: float | None = 0.5
    target_kl: float | None = None
    normalize_advantage: bool = True
    n_steps: int = 2048
    batch_size: int = 64
    epochs: int = 10
    learning_rate: float = 3e-4

    def hyper(self):
        neg = lambda x: -1.0 if x is None else float(x)
        return L.PPOHyper(self.gamma, self.gae_lambda, self.clip_range, neg(self.clip_range_vf), self.ent_coef,
                          self.vf_coef, neg(self.max_grad_norm), neg(self.target_kl), int(self.normalize_advantage),
                          self.learning_rate, 0.9, 0.999, 1e-5)   # Adam(eta, (0.9,0.999), 1e-5): ppo.jl:64-66


def get_hparams(alg):  # logging/logging_utils.jl:11-35
    return {k: getattr(alg, k) for k in ("gamma", "gae_lambda", "clip_range", "ent_coef", "vf_coef", "max_grad_norm",
                                         "n_steps", "batch_size", "epochs", "learning_rate", "normalize_advantage")}


# ---- logging / callbacks (interfaces/logging.jl, callbacks.jl) ----------------------------
class AbstractTrainingLogger:
    def set_step(self, step): pass
    def increment_step(self, n): pass
    def log_scalar(self, key, value): pass
    def log_metrics(self, kv):
        for k, v in kv.items():
            self.log_scalar(k, v)
    def log_hparams(self, hparams, metrics): pass
    def flush(self): pass
    def close(self): pass


class NoTrainingLogger(AbstractTrainingLogger):
    pass


class DictLogger(AbstractTrainingLogger):
    """In-memory logger (stands in for the TensorBoard/Wandb/DearDiary extensions, out of scope)."""

    def __init__(self):
        self.step, self.scalars = 0, {}

    def set_step(self, step):
        self.step = step

    def increment_step(self, n):
        self.step += n

    def log_scalar(self, key, value):
        self.scalars.setdefault(key, []).append((self.step, float(value)))


class AbstractCallback:
    """callbacks.jl:1-15 — every hook receives the driver's locals and returns a Bool."""
    def on_training_start(self, locals_): return True
    def on_rollout_start(self, locals_): return True
    def on_step(self, locals_): return True
    def on_rollout_end(self, locals_): return True
    def on_training_end(self, locals_): return True


@dataclass
class AgentStats:
    steps_taken: int = 0
    gradient_updates: int = 0


class TrainState:
    """Stand-in for Lux.Training.TrainState: `.parameters` is the flat host copy (source of truth
    between train calls), the optimiser state lives on the device."""

    def __init__(self, parameters):
        self.parameters = parameters
        self.states = ()


class Agent:
    """Agent(layer, alg; verbose, logger, rng) — algorithms/ppo.jl:42-62, agents/agent_types.jl:3-69."""

    def __init__(self, layer, alg, verbose=0, logger=None, rng=None, ctx=None, stats_window=100):
        if logger is not None and not isinstance(logger, AbstractTrainingLogger):
            raise TypeError(f"Unsupported logger {type(logger)}")   # interfaces/logging.jl:51-54
        self.layer, self.alg, self.verbose = layer, alg, verbose
        self.logger = logger or NoTrainingLogger()
        self.rng = rng if rng is not None else np.random.default_rng()
        self.ctx = ctx or Context.default()
        self.stats = AgentStats()
        self.stats_window = stats_window
        self.device = DevicePolicy(self.ctx, layer.obs_dim, layer.hidden_dims, layer.action_space())
        assert self.device.n_params == layer.parameterlength()
        self.train_state = TrainState(layer.setup(self.rng))
        self.device.set_params(self.train_state.parameters)
        seed = int(self.rng.integers(0, 2 ** 63 - 1))
        self.device.seed(seed, 0)
        self.shuffle_seed = int(self.rng.integers(0, 2 ** 63 - 1))
        self.epoch_counter = 0

    def set_parameters(self, flat):
        self.train_state.parameters = np.asarray(flat, dtype=np.float32).copy()
        self.device.set_params(self.train_state.parameters)

    def sync_from_device(self):
        self.train_state.parameters = self.device.get_params()
        return self.train_state.parameters


def steps_taken(agent):
    return agent.stats.steps_taken


# agents/agent_methods.jl:19-105
def get_action_and_values(agent, observations):
    a, v, lp = agent.device.forward(observations, deterministic=False)
    return a, v, lp


def predict_values(agent, observations):
    return agent.device.predict_values(observations)


def to_env(action_space, actions):
    """adapters/default_adapters.jl:4-11 (ClampAdapter) / :34-40 (DiscreteAdapter)."""
    if isinstance(action_space, Box):
        return np.clip(actions, action_space.low.reshape(-1), action_space.high.reshape(-1)).astype(np.float32)
    return actions


def predict_actions(agent, observations, deterministic=False, rng=None):
    a, _, _ = agent.device.forward(observations, deterministic=deterministic)
    return to_env(agent.layer.action_space(), a)


def save_policy_params_and_state(agent, path, suffix=".npz"):
    """agents/agent_methods.jl:122-138 — NPZ mirror of the JLD2 dict {"layer","parameters","states","aux"}
    plus the Adam moments the reference does not save."""
    file_path = path if path.endswith(suffix) else path + suffix
    m, v, step = agent.device.get_opt_state()
    np.savez(file_path, parameters=agent.sync_from_device(), hidden_dims=np.asarray(agent.layer.hidden_dims),
             adam_m=m, adam_v=v, adam_step=step)
    return file_path


def load_policy_params_and_state(agent, path, suffix=".npz", restore_optimizer=False):
    """algorithms/ppo.jl:77-94 — parameters restored, optimiser fresh (reference behaviour) unless asked."""
    file_path = path if path.endswith(suffix) else path + suffix
    d = np.load(file_path)
    agent.set_parameters(d["parameters"])
    n = agent.device.n_params
    if restore_optimizer:
        agent.device.set_opt_state(d["adam_m"], d["adam_v"], int(d["adam_step"]))
    else:
        agent.device.set_opt_state(np.zeros(n, np.float32), np.zeros(n, np.float32), 0)
    return agent


# ---- collection (buffers/rollout_buffer.jl:46-90) -----------------------------------------
def collect_rollout(rollout_buffer, agent, alg, env, callbacks=None, forced_actions=None):
    """collect_rollout!(buffer, agent, alg, env) -> (fps, success): fused device rollout + GAE.
    When a callback overrides on_step the rollout runs in chunks of one step (dril_rollout_collect_steps) so that the
    hook of step i sees the env after i - 1 steps and a `false` stops the collection there (trajectory.jl:34-39)."""
    fa = None
    if forced_actions is not None:
        if rollout_buffer.discrete:
            fa = np.ascontiguousarray(np.asarray(forced_actions).reshape(len(rollout_buffer)), dtype=np.int64)
        else:
            fa = L.f32(np.asarray(forced_actions).reshape(len(rollout_buffer), rollout_buffer.act_dim))
    lib = agent.ctx.lib
    active = _on_step_callbacks(callbacks)
    if active:
        n_steps, n_envs = rollout_buffer.n_steps, rollout_buffer.n_envs
        loc = dict(agent=agent, env=env, alg=alg, n_steps=n_steps, n_envs=n_envs, callbacks=callbacks,
                   roll_buffer=rollout_buffer, obs_space=env.observation_space(), act_space=env.action_space())
        t0 = time.time()
        L.check(lib.dril_rollout_collect_steps(env.h, agent.device.h, rollout_buffer.h, 0, 0, 1, None))   # new_obs = observe(env), :32
        for i in range(1, n_steps + 1):
            loc["i"] = i
            if not all(c.on_step(loc) for c in active):
                return 0.0, False
            chunk = None if fa is None else np.ascontiguousarray(fa[(i - 1) * n_envs:i * n_envs])
            L.check(lib.dril_rollout_collect_steps(env.h, agent.device.h, rollout_buffer.h, i - 1, 1, 0, L.ptr(chunk)))
        fps = n_steps * n_envs / max(time.time() - t0, 1e-12)
        rollout_buffer.compute_advantages(alg.gamma, alg.gae_lambda)
        return fps, True
    fps = L.c_f32(0)
    L.check(lib.dril_rollout_collect(env.h, agent.device.h, rollout_buffer.h, L.ptr(fa), C.byref(fps)))
    rollout_buffer.compute_advantages(alg.gamma, alg.gae_lambda)
    return fps.value, True


def _hook(callbacks, name, loc):
    return all(getattr(c, name)(loc) for c in callbacks) if callbacks else True


def _on_step_callbacks(callbacks):
    """Callbacks that override on_step (buffers/trajectory.jl:34-39); the others cost nothing and keep the fused rollout."""
    return [c for c in (callbacks or []) if type(c).on_step is not AbstractCallback.on_step]


LEARN_STATS_KEYS = ("entropy_losses", "policy_losses", "value_losses", "approx_kl_divs", "clip_fractions", "losses",
                    "explained_variances", "fps", "grad_norms", "learning_rates")


def train(agent, env, alg, max_steps, callbacks=None, sync_every_iteration=True):
    """train!(agent, env, alg, max_steps; callbacks) -> (learn_stats, timers) — algorithms/ppo.jl:100-325.
    One dril_ppo_iteration_async per iteration (rollout + GAE + epochs of minibatch updates on the
    device); the host only keeps the reference's bookkeeping. Returns None if a callback aborts."""
    to = {"setup": 0.0, "training_loop": 0.0, "collect_rollout_ms": 0.0, "update_ms": 0.0}
    t_setup = time.time()
    n_steps, n_envs = alg.n_steps, env.number_of_envs()
    # the device buffer is kept on the agent between calls (the reference allocates per train! call;
    # device allocation is the expensive part here) and is fully overwritten by every rollout
    key = (n_steps, n_envs, repr(env.observation_space()), repr(env.action_space()))
    cache = agent.__dict__.setdefault("_roll_buffers", {})
    roll_buffer = cache.get(key)
    if roll_buffer is None or roll_buffer.h is None:
        for old in cache.values():
            old.close()
        cache.clear()
        roll_buffer = RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, n_steps, n_envs,
                                    ctx=agent.ctx)
        cache[key] = roll_buffer
    roll_buffer.gamma, roll_buffer.gae_lambda = float(alg.gamma), float(alg.gae_lambda)
    iterations = max_steps // (n_steps * n_envs)
    total_steps = iterations * n_steps * n_envs
    learn = {k: [] for k in LEARN_STATS_KEYS}
    total_fps = learn["fps"]
    agent.device.set_params(agent.train_state.parameters)     # host parameters are the source of truth
    lib = agent.ctx.lib
    # all lazily made allocations up front (data-parallel callers synchronise their ranks after this: `on_training_start` is the hook)
    L.check(lib.dril_iteration_prepare(env.h, agent.device.h, roll_buffer.h, int(alg.epochs), int(alg.batch_size)))
    to["setup"] = time.time() - t_setup
    if not _hook(callbacks, "on_training_start", dict(locals())):
        return None
    t_loop = time.time()
    # Without callbacks nothing on the host can influence the next iteration, so iteration i+1 is enqueued before
    # the statistics of iteration i are read (the library keeps results in FIFO order): the device never waits for
    # the host.  With callbacks every hook sees the device state of its own iteration, as in the reference.
    pipelined = not callbacks

    def enqueue():
        L.check(lib.dril_ppo_iteration_async(env.h, agent.device.h, roll_buffer.h, C.byref(alg.hyper()), alg.epochs,
                                             alg.batch_size, agent.shuffle_seed, agent.epoch_counter))
        agent.epoch_counter += alg.epochs

    def drain():
        st = L.IterStats()
        while lib.dril_iteration_result(agent.device.h, C.byref(st)) == 0:
            pass

    completed = False
    try:
        for i in range(1, iterations + 1):
            learning_rate = alg.learning_rate                   # Optimisers.adjust! each iteration (ppo.jl:155-157)
            if not _hook(callbacks, "on_rollout_start", dict(locals())):
                return None
            st = L.IterStats()
            if pipelined:
                if i == 1:
                    enqueue()
                if i < iterations:
                    enqueue()
                L.check(lib.dril_iteration_result(agent.device.h, C.byref(st)))
                fps = n_steps * n_envs / max(st.rollout_ms * 1e-3, 1e-12)
            else:
                # with callbacks the iteration is split like the reference's (ppo.jl:160-186): collect_rollout! (on_step
                # hooks inside), bookkeeping, on_rollout_end, and only then the update, so that a hook returning false skips
                # the update and every hook sees the parameters the rollout was collected with
                fps, ok = collect_rollout(roll_buffer, agent, alg, env, callbacks=callbacks)
                if not ok:
                    return None
                ms = env.monitor_stats() if env.is_monitored() else None
            total_fps.append(fps)
            agent.stats.steps_taken += n_steps * n_envs         # add_step! (ppo.jl:173)
            agent.logger.increment_step(n_steps * n_envs)
            agent.logger.log_scalar("env/fps", fps)
            if pipelined:
                if st.episodes_in_window > 0:                   # log_stats(env, logger), monitorWrapperEnv.jl:64-70
                    agent.logger.log_scalar("env/ep_rew_mean", st.ep_rew_mean)
                    agent.logger.log_scalar("env/ep_len_mean", st.ep_len_mean)
            elif ms is not None and ms["n_in_window"] > 0:
                agent.logger.log_scalar("env/ep_rew_mean", ms["ep_rew_mean"])
                agent.logger.log_scalar("env/ep_len_mean", ms["ep_len_mean"])
            if not _hook(callbacks, "on_rollout_end", dict(locals())):
                return None
            if not pipelined:
                rollout_ms = n_steps * n_envs / max(fps, 1e-12) * 1e3
                L.check(lib.dril_ppo_update(agent.device.h, roll_buffer.h, C.byref(alg.hyper()), alg.epochs, alg.batch_size,
                                            agent.shuffle_seed, agent.epoch_counter, C.byref(st)))
                agent.epoch_counter += alg.epochs
                st.rollout_ms = rollout_ms
            agent.stats.gradient_updates += st.n_minibatch_steps
            learn["learning_rates"].append(learning_rate)
            learn["explained_variances"].append(st.explained_variance)
            learn["entropy_losses"].append(st.entropy_loss)
            learn["policy_losses"].append(st.policy_loss)
            learn["value_losses"].append(st.value_loss)
            learn["approx_kl_divs"].append(st.approx_kl_div)
            learn["clip_fractions"].append(st.clip_fraction)
            learn["losses"].append(st.loss)
            learn["grad_norms"].append(st.grad_norm)
            to["collect_rollout_ms"] += st.rollout_ms
            to["update_ms"] += st.update_ms
            lg = agent.logger
            lg.log_scalar("train/entropy_loss", st.entropy_loss)
            lg.log_scalar("train/explained_variance", st.explained_variance)
            lg.log_scalar("train/policy_loss", st.policy_loss)
            lg.log_scalar("train/value_loss", st.value_loss)
            lg.log_scalar("train/approx_kl_div", st.approx_kl_div)
            lg.log_scalar("train/clip_fraction", st.clip_fraction)
            lg.log_scalar("train/loss", st.loss)
            lg.log_scalar("train/grad_norm", st.grad_norm)
            lg.log_scalar("train/learning_rate", learning_rate)
            if st.kl_stopped and agent.verbose:
                print(f"Early stopping at iteration {i} due to reaching max kl")      # ppo.jl:236 @info
            if not agent.layer.discrete and not pipelined:                          # ppo.jl:295-297, every iteration
                lg.log_scalar("train/std", float(np.mean(np.exp(agent.device.get_params()[-agent.layer.act_n:]))))
        completed = True
    finally:
        # an aborted train! keeps the parameters it updated in place (ppo.jl:179-186): whatever the exit path, unread pipelined
        # results are drained and the host copy (the source of truth between calls) follows the device
        if not completed:
            drain()
        params = agent.sync_from_device()                   # copy updated parameters back (SURVEY §8b)
    if not agent.layer.discrete and pipelined:
        agent.logger.log_scalar("train/std", float(np.mean(np.exp(params[-agent.layer.act_n:]))))
    to["training_loop"] = time.time() - t_loop
    learn_stats = {k: np.asarray(v, dtype=np.float32) for k, v in learn.items()}
    if not _hook(callbacks, "on_training_end", dict(locals())):
        return None
    return learn_stats, to


# ---- evaluation (src/evaluation.jl:54-143) -------------------------------------------------
def evaluate_agent(agent, env, n_eval_episodes=10, deterministic=True, reward_threshold=None, return_stats=True,
                   warn=True, rng=None, chunk_steps=None, on_device=True):
    """evaluate_agent(agent, env; n_eval_episodes, deterministic, reward_threshold, return_stats) — src/evaluation.jl:54-143.
    For a CudaBatchedEnv the episode loop runs on the device (dril_evaluate: fused policy + env steps in chunks, one
    device -> host copy of the episode records per chunk); `on_device=False` keeps the step-by-step host loop over the
    AbstractParallelEnv interface (observe / predict_actions / act!), which is what any other env type gets."""
    monitored = env.is_monitored()
    if not monitored and warn:
        import warnings
        warnings.warn("Evaluation environment is not wrapped with a Monitor wrapper. This may result in reporting modified "
                      "episode lengths and rewards, if other wrappers happen to modify these.")
    if on_device and isinstance(env, CudaBatchedEnv):
        er = np.empty(n_eval_episodes, np.float32)
        el = np.empty(n_eval_episodes, np.int64)
        got, steps = L.c_i64(0), L.c_i64(0)
        k = int(chunk_steps or max(1, min(64, env.max_steps)))
        L.check(agent.ctx.lib.dril_evaluate(env.h, agent.device.h, int(n_eval_episodes), int(bool(deterministic)), k,
                                            L.ptr(er), L.ptr(el), C.byref(got), C.byref(steps)))
        assert got.value == n_eval_episodes
    else:
        episode_rewards, episode_lengths = [], []
        n_envs = env.number_of_envs()
        cur_r = np.zeros(n_envs, np.float32)
        cur_l = np.zeros(n_envs, np.int64)
        env.reset()
        obs = env.observe()
        while len(episode_rewards) < n_eval_episodes:
            actions = predict_actions(agent, obs, deterministic=deterministic)
            r, term, trunc, infos = env.act(actions)
            cur_r += r
            cur_l += 1
            obs = env.observe()
            done = term | trunc
            for i in range(n_envs):
                if len(episode_rewards) < n_eval_episodes and done[i]:
                    if monitored and "episode" in infos[i]:
                        episode_rewards.append(infos[i]["episode"]["r"])
                        episode_lengths.append(infos[i]["episode"]["l"])
                    else:
                        episode_rewards.append(float(cur_r[i]))
                        episode_lengths.append(int(cur_l[i]))
                    cur_r[i] = 0
                    cur_l[i] = 0
        er, el = np.asarray(episode_rewards, np.float32), np.asarray(episode_lengths)
    mean_reward = float(er.mean())
    if reward_threshold is not None and mean_reward < reward_threshold:
        raise RuntimeError(f"Mean reward below threshold: {mean_reward:.2f} < {reward_threshold}")
    if return_stats:
        sd = lambda x: float(np.std(x, ddof=1)) if len(x) > 1 else float("nan")
        return dict(mean_reward=mean_reward, std_reward=sd(er), mean_length=float(el.mean()), std_length=sd(el))
    return er, el


# ---- normaliser statistics (environment_wrappers/normalizeWrapperEnv.jl:261-309) -----------
_NORM_KEYS = ("obs_mean", "obs_var", "obs_count", "ret_mean", "ret_var", "ret_count")


def save_normalization_stats(env, filepath):
    """save_normalization_stats(env, filepath): the ten keys of normalizeWrapperEnv.jl:261-277 as an NPZ file (JLD2 on the
    Julia side)."""
    s = env.norm_stats()
    cfg = env.normalize
    path = filepath if filepath.endswith(".npz") else filepath + ".npz"
    np.savez(path, obs_mean=s["obs_mean"], obs_var=s["obs_var"], obs_count=np.int64(s["obs_count"]),
             ret_mean=np.float32(s["ret_mean"]), ret_var=np.float32(s["ret_var"]), ret_count=np.int64(s["ret_count"]),
             clip_obs=np.float32(cfg.clip_obs), clip_reward=np.float32(cfg.clip_reward), gamma=np.float32(cfg.gamma),
             epsilon=np.float32(cfg.epsilon))
    return path


def load_normalization_stats(env, filepath):
    """load_normalization_stats!(env, filepath): running statistics only; clips / gamma / epsilon stay the env's own
    (normalizeWrapperEnv.jl:279-297)."""
    path = filepath if filepath.endswith(".npz") else filepath + ".npz"
    d = np.load(path)
    env.set_norm_stats({k: d[k] for k in _NORM_KEYS})
    return env


def sync_normalization_stats(eval_env, train_env):
    """sync_normalization_stats!(eval_env, train_env): copy the running statistics and zero the eval env's discounted
    returns; the env counts may differ (normalizeWrapperEnv.jl:299-309)."""
    eval_env.set_norm_stats(train_env.norm_stats())
    L.check(eval_env.ctx.lib.dril_env_zero_returns(eval_env.h))


# ---- deployment (src/deployment/deployment_policy.jl:3-71) ---------------------------------
class NeuralPolicy:
    def __init__(self, agent):
        self.layer, self.params = agent.layer, agent.sync_from_device().copy()
        self.action_space = agent.layer.action_space()
        self.device = DevicePolicy(agent.ctx, agent.layer.obs_dim, agent.layer.hidden_dims, self.action_space)
        self.device.set_params(self.params)

    def __call__(self, obs, deterministic=True, rng=None):
        obs = np.asarray(obs, dtype=np.float32)
        single = obs.shape == tuple(self.layer.observation_space.size())
        a, _, _ = self.device.forward(obs.reshape(-1, self.layer.obs_dim), deterministic=deterministic)
        a = to_env(self.action_space, a)
        return a[0] if single else a


class NormWrapperPolicy:
    def __init__(self, policy, obs_mean, obs_var, eps, clip_obs):
        self.policy, self.obs_mean, self.obs_var = policy, obs_mean.copy(), obs_var.copy()
        self.eps, self.clip_obs = np.float32(eps), np.float32(clip_obs)

    def __call__(self, obs, deterministic=True, rng=None):
        obs = np.asarray(obs, dtype=np.float32)
        o = np.clip((obs - self.obs_mean) / np.sqrt(self.obs_var + self.eps), -self.clip_obs, self.clip_obs)
        return self.policy(o.astype(np.float32), deterministic=deterministic, rng=rng)


def extract_policy(agent, norm_env=None):
    p = NeuralPolicy(agent)
    if norm_env is None:
        return p
    s = norm_env.norm_stats()
    return NormWrapperPolicy(p, s["obs_mean"], s["obs_var"], norm_env.normalize.epsilon, norm_env.normalize.clip_obs)
