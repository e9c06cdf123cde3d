"""Observation history on the device (history_len, mask_velocities): the newest frame of a stacked run against a plain run (bit
for bit), the fused fast, cooperative and tcgen05-actor rollouts, the compat path under Monitor, Normalize and Scaling, chunked
collection and dril_evaluate against the oracle (oracle/env_history.py), refills and validation, the update paths at the new
widths, and CartPole without velocities learned from a 4-frame history."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import env_history as EH, env_params as EP, envs as OE, policy as OP, ppo as OO, ppo64 as O64

pytestmark = pytest.mark.gpu
f32 = np.float32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KINDS = ("cartpole", "pendulum", "mountaincar", "mountaincar_continuous", "acrobot")
D0 = EH.BASE_OBS_DIM
CONT = {"pendulum": 2.0, "mountaincar_continuous": 1.0}   # Box(1) envs: action bound
MCC_LOW, MCC_HIGH = np.array([-1.2, -0.07], f32), np.array([0.6, 0.07], f32)
MASKED = {"cartpole": True, "pendulum": False, "mountaincar": True, "mountaincar_continuous": False, "acrobot": True}


@pytest.fixture(scope="module")
def D():
    import __graft_entry__
    __graft_entry__.build()
    import dril_b200
    return dril_b200


def _spec(kind, obs_dim, hidden=(64, 64)):
    if kind in CONT:
        b = CONT[kind]
        return OP.PolicySpec(obs_dim, list(hidden), "continuous", 1, act_low=[-b], act_high=[b])
    return OP.PolicySpec(obs_dim, list(hidden), "discrete", 2 if kind == "cartpole" else 3, act_start=1)


def _actions(kind, rng, shape):
    if kind in CONT:
        return (rng.normal(size=shape + (1,)) * 1.2 * CONT[kind]).astype(f32)
    return rng.integers(1, 3 if kind == "cartpole" else 4, shape)


def _ranges(kind, n, rng, spread=0.5):
    d = np.array([v for _, v in EP.ENV_PARAMS[kind]], dtype=np.float64)[:, None]
    a, b = d * rng.uniform(1 - spread, 1 + spread, (2, len(d), n))
    lo, hi = np.minimum(a, b).astype(f32), np.maximum(a, b).astype(f32)
    hi[:, ::5] = lo[:, ::5]
    return lo, hi


def _kw(kind, lo, hi):
    return {nm: (lo[k], hi[k]) for k, (nm, _) in enumerate(EP.ENV_PARAMS[kind])}


def _flags(buf):
    f = buf.download("flags")
    return (f & 1).astype(bool), ((f >> 1) & 1).astype(bool)


def _params_array(env):
    p = env.env_params()
    return np.stack([p[nm] for nm, _ in EP.ENV_PARAMS[env.kind]])


def _agent(D, env, kind, T, seed=2, hidden=(64, 64)):
    spec = _spec(kind, env.obs_dim, hidden)
    flat = (OP.init_params(spec, seed=seed) + np.random.default_rng(seed).normal(size=spec.n_params()).astype(f32) * 0.05).astype(f32)
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=list(hidden))
    alg = D.PPO(n_steps=T, gamma=0.97, gae_lambda=0.9)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
    agent.set_parameters(flat)
    return spec, flat, agent, alg


def _norm(D, norm):
    return D.NormalizeConfig(norm_obs=norm == "full") if norm else None


# path: (n, T, max_steps, normalize); gtc: >= 96 envs per SM, the actor on tcgen05 (rollout_gtc.cuh) at widths <= 15
PATHS = {"fast": (300, 24, 10, None), "coop": (200, 20, 9, "full"), "gtc": (14208, 4, 3, "ret")}
ENV_FIELDS = ("rewards", "flags", "episode_r", "episode_l")


# ------------------------------------------------------------------------------------------
# 1. the newest frame is free: a k = 3 run's last frame == a plain run, bit for bit
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ranges", [True, False])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("path", list(PATHS))
def test_newest_frame_is_free(D, kind, path, ranges):
    n, T, ms, norm = PATHS[path]
    rng = np.random.default_rng(3)
    lo, hi = _ranges(kind, n, rng)
    mask = MASKED[kind] if ranges else not MASKED[kind]
    pk = _kw(kind, lo, hi) if ranges else None
    envs = [D.CudaBatchedEnv(kind, n, max_steps=ms, seed=9, monitor_window=100, normalize=_norm(D, norm), env_params=pk,
                             history_len=k, mask_velocities=m) for k, m in ((1, False), (3, mask))]
    cols = list(EH.VELOCITY_FREE[kind]) if mask else list(range(D0[kind]))
    F = len(cols)
    assert envs[0].obs_dim == D0[kind] and envs[1].obs_dim == 3 * F
    assert envs[1].history_len() == 3 and envs[1].masks_velocities() == mask
    for rollout in range(3):
        forced = _actions(kind, rng, (T, n))
        outs = []
        for env in envs:
            _, _, agent, alg = _agent(D, env, kind, T)
            assert (agent.device.update_path() == "tensor") == (env.obs_dim <= 15)
            buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
            _, ok = D.collect_rollout(buf, agent, alg, env, forced_actions=forced)
            assert ok
            outs.append({k: buf.download(k) for k in ENV_FIELDS + ("obs",)})
            buf.close()
        what = f"{kind} {path} ranges={ranges} rollout {rollout}"
        np.testing.assert_array_equal(outs[1]["obs"][..., 2 * F:], outs[0]["obs"][..., cols], err_msg=what + ": obs")
        for k in ENV_FIELDS:
            np.testing.assert_array_equal(outs[1][k], outs[0][k], err_msg=f"{what}: {k}")
        assert ((outs[0]["flags"] >> 1) & 1).any()
        for j in range(2):
            np.testing.assert_array_equal(envs[1].get_state()[j], envs[0].get_state()[j])
        np.testing.assert_array_equal(_params_array(envs[1]), _params_array(envs[0]))
        if norm:
            s0, s1 = envs[0].norm_stats(), envs[1].norm_stats()
            for k in s0:
                got = s1[k][2 * F:] if k in ("obs_mean", "obs_var") else s1[k]
                want = s0[k][cols] if k in ("obs_mean", "obs_var") else s0[k]
                np.testing.assert_array_equal(got, want, err_msg=k)


# ------------------------------------------------------------------------------------------
# 2. fused rollout against the oracle
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("path", list(PATHS))
def test_fused_rollout_vs_oracle(D, kind, path):
    n, T, ms, norm = PATHS[path]
    k, mask = 3, MASKED[kind]
    gid = 1000 if path == "fast" else 0
    rng = np.random.default_rng(7)
    lo, hi = _ranges(kind, n, rng)
    env = D.CudaBatchedEnv(kind, n, max_steps=ms, seed=9, monitor_window=100, normalize=_norm(D, norm), gid_offset=gid,
                           env_params=_kw(kind, lo, hi), history_len=k, mask_velocities=mask)
    ob = EH.make(kind, n, k, mask, seed=9, max_steps=ms, gid_offset=gid, param_ranges=(lo, hi))
    o = OE.MonitorWrapper(OE.ParallelEnv(ob))
    if norm:
        o = OE.NormalizeWrapper(o, ob.obs_dim, norm_obs=norm == "full")
    spec, flat, agent, alg = _agent(D, env, kind, T)
    assert spec.obs_dim == EH.history_obs_dim(kind, k, mask)
    tol = dict(rtol=3e-5, atol=3e-4 if kind == "acrobot" else 3e-5) if norm else dict(rtol=1e-5, atol=1e-5)
    cont = kind in CONT
    for rollout in range(2):       # 0: replayed actions, 1: sampled on the device, then replayed through the oracle
        forced = _actions(kind, rng, (T, n)) if rollout == 0 else None
        buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
        _, ok = D.collect_rollout(buf, agent, alg, env, forced_actions=forced)
        assert ok
        acts = buf.download("actions")
        replay = forced if forced is not None else (acts if cont else acts[..., 0])
        eo = OO.collect_rollout_timemajor(o, spec, flat, T, forced_actions=replay)
        te, tr = _flags(buf)
        np.testing.assert_array_equal(te, eo["term"])
        np.testing.assert_array_equal(tr, eo["trunc"])
        np.testing.assert_allclose(buf.download("obs"), eo["obs"], **(tol if norm == "full" else dict(rtol=0, atol=0)))
        np.testing.assert_allclose(buf.download("rewards"), eo["rewards"], **(tol if norm else dict(rtol=0, atol=0)))
        np.testing.assert_allclose(buf.download("values"), eo["values"], **tol)
        np.testing.assert_allclose(buf.download("logprobs"), eo["logprobs"], rtol=1e-4, atol=1e-4)
        np.testing.assert_allclose(buf.download("last_values"), eo["last_values"], **tol)
        np.testing.assert_allclose(np.where(tr, buf.download("boot"), 0), eo["boot"], **tol)
        done = te | tr
        np.testing.assert_allclose(buf.download("episode_r")[done], eo["episode_r"][done], rtol=1e-5)
        np.testing.assert_array_equal(buf.download("episode_l")[done], eo["episode_l"][done])
        np.testing.assert_array_equal(env.get_state()[0], ob.state)
        assert tr.any()
        buf.close()


# ------------------------------------------------------------------------------------------
# 3. compat observe / act! under Monitor, Normalize and Scaling
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,k,mask,norm,scaled", [
    ("cartpole", 4, True, False, False), ("acrobot", 2, False, True, False), ("mountaincar", 3, True, False, False),
    ("pendulum", 3, False, False, True), ("pendulum", 2, True, True, True), ("mountaincar_continuous", 4, True, True, True),
    ("mountaincar_continuous", 2, False, False, True)])
def test_compat_wrappers_vs_oracle(D, kind, k, mask, norm, scaled):
    n, ms, steps = 301, 13, 50
    rng = np.random.default_rng(6)
    lo, hi = _ranges(kind, n, rng)
    env = D.CudaBatchedEnv(kind, n, max_steps=ms, seed=5, monitor_window=100, normalize=D.NormalizeConfig() if norm else None,
                           scaling=scaled, env_params=_kw(kind, lo, hi), history_len=k, mask_velocities=mask)
    assert env.obs_dim == EH.history_obs_dim(kind, k, mask)
    sp = env.observation_space()
    assert sp.size() == (env.obs_dim,)
    if scaled:
        assert (sp.low == -1).all() and (sp.high == 1).all()
    sc = None
    if scaled:
        sc = (OE.PENDULUM_OBS_LOW, OE.PENDULUM_OBS_HIGH) if kind == "pendulum" else (MCC_LOW, MCC_HIGH)
    ob = EH.make(kind, n, k, mask, seed=5, max_steps=ms, param_ranges=(lo, hi), scaling=sc)
    o = OE.MonitorWrapper(OE.ParallelEnv(ob))
    if norm:
        o = OE.NormalizeWrapper(o, ob.obs_dim)
    tol = dict(rtol=3e-5, atol=1e-3 if kind == "acrobot" else 3e-4) if norm else dict(rtol=0, atol=0)
    np.testing.assert_allclose(env.observe(), o.observe(), **tol)
    np.testing.assert_allclose(env.observe(), o.observe(), **tol)      # observe() never moves the history
    n_trunc = 0
    for t in range(steps):
        a = _actions(kind, rng, (n,))
        if scaled:
            a = np.clip(a / CONT[kind], -1, 1).astype(f32)
        r, te, tr, infos = env.act(a)
        ro, teo, tro, info = o.act(a)
        np.testing.assert_array_equal(te, teo)
        np.testing.assert_array_equal(tr, tro)
        np.testing.assert_allclose(r, ro, rtol=3e-5 if norm else 0, atol=0)
        np.testing.assert_allclose(env.observe(), o.observe(), **tol)
        if norm:
            np.testing.assert_array_equal(env.get_original()[0], o.old_obs)
            s = env.norm_stats()
            np.testing.assert_allclose(s["obs_mean"], o.obs_rms.mean, rtol=1e-4, atol=1e-5)
            np.testing.assert_allclose(s["obs_var"], o.obs_rms.var, rtol=1e-3, atol=1e-6)
            assert s["obs_count"] == o.obs_rms.count
        for i in np.nonzero(tro)[0]:
            np.testing.assert_allclose(infos[i]["terminal_observation"], info["terminal_observation"][i], **tol)
        for i in np.nonzero(teo | tro)[0]:
            assert abs(infos[i]["episode"]["r"] - info["episode_r"][i]) <= 1e-5 * max(1.0, abs(info["episode_r"][i]))
            assert infos[i]["episode"]["l"] == info["episode_l"][i]
        n_trunc += tro.sum()
    assert n_trunc > 0


# ------------------------------------------------------------------------------------------
# 4. dril_evaluate against the oracle loop
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
def test_evaluate_vs_oracle_loop(D, kind):
    n, ms, n_eval, k, mask = 37, 40, 60, 4, MASKED[kind]
    rng = np.random.default_rng(8)
    lo, hi = _ranges(kind, n, rng)
    env = D.CudaBatchedEnv(kind, n, max_steps=ms, seed=9, monitor_window=100, env_params=_kw(kind, lo, hi), history_len=k,
                           mask_velocities=mask)
    a0 = _actions(kind, rng, (n,))
    env.act(a0)                              # a history that dril_evaluate's reset must restart
    spec, flat, agent, _ = _agent(D, env, kind, 8, seed=5)
    er, el = D.evaluate_agent(agent, env, n_eval_episodes=n_eval, deterministic=True, return_stats=False, chunk_steps=7)
    ob = EH.make(kind, n, k, mask, seed=9, max_steps=ms, param_ranges=(lo, hi))
    o = OE.MonitorWrapper(OE.ParallelEnv(ob))
    o.act(a0)
    o.reset()     # dril_evaluate resets the env it was handed
    obs = o.observe()
    exp_r, exp_l = [], []
    while len(exp_r) < n_eval:
        a, _, _ = OP.forward(spec, flat, obs, deterministic=True)
        _, term, trunc, infos = o.act(a)
        obs = o.observe()
        for i in range(n):
            if (term[i] or trunc[i]) and len(exp_r) < n_eval:
                exp_r.append(infos["episode_r"][i]); exp_l.append(int(infos["episode_l"][i]))
    np.testing.assert_array_equal(el, np.asarray(exp_l))
    np.testing.assert_allclose(er, np.asarray(exp_r, np.float32), rtol=1e-5)


@pytest.mark.parametrize("kind", KINDS)
def test_frozen_fixtures(D, kind):
    """the compat path against tests/golden/orc_<kind>_history_replay.npz alone"""
    g = np.load(os.path.join(ROOT, "tests", "golden", f"orc_{kind}_history_replay.npz"))
    n = g["obs"].shape[1]
    env = D.CudaBatchedEnv(kind, n, max_steps=int(g["max_steps"]), seed=int(g["seed"]), env_params=_kw(kind, g["lo"], g["hi"]),
                           history_len=int(g["history_len"]), mask_velocities=bool(g["mask_velocities"]),
                           scaling=bool(g["scaling"]))
    np.testing.assert_array_equal(env.observe(), g["obs"][0])
    for t, a in enumerate(g["actions"]):
        r, te, tr, infos = env.act(a)
        np.testing.assert_array_equal(r, g["rewards"][t])
        np.testing.assert_array_equal(te, g["term"][t])
        np.testing.assert_array_equal(tr, g["trunc"][t])
        for i in np.nonzero(tr)[0]:
            np.testing.assert_array_equal(infos[i]["terminal_observation"], g["terminal_obs"][t][i])
        np.testing.assert_array_equal(env.observe(), g["obs"][t + 1])


# ------------------------------------------------------------------------------------------
# 5. chunked collection (on_step, one launch per step) == the fused rollout, across rollouts
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ("cartpole", "acrobot", "pendulum"))
def test_chunked_equals_fused(D, kind):
    n, T, ms = 96, 12, 5
    rng = np.random.default_rng(12)
    lo, hi = _ranges(kind, n, rng)

    class Step(D.AbstractCallback):
        def on_step(self, loc):
            return True

    runs = []
    for chunked in (False, True):
        # a training normaliser keeps both on the general kernel (chunked collection never takes the fast or tcgen05 paths)
        env = D.CudaBatchedEnv(kind, n, max_steps=ms, seed=4, monitor_window=100, normalize=D.NormalizeConfig(),
                               env_params=_kw(kind, lo, hi), history_len=4, mask_velocities=MASKED[kind])
        _, _, agent, alg = _agent(D, env, kind, T, hidden=(16, 16))
        outs = []
        for _ in range(3):
            buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
            _, ok = D.collect_rollout(buf, agent, alg, env, callbacks=[Step()] if chunked else None)
            assert ok
            outs.append({k: buf.download(k) for k in ("obs", "actions", "rewards", "values", "logprobs", "boot", "last_values",
                                                      "flags", "episode_r", "episode_l")})
            outs[-1]["state"], outs[-1]["steps"] = env.get_state()
            outs[-1].update(env.norm_stats())
            buf.close()
        runs.append(outs)
    for r in range(3):
        assert ((runs[0][r]["flags"] >> 1) & 1).any()
        for k in runs[0][r]:
            np.testing.assert_array_equal(runs[1][r][k], runs[0][r][k], err_msg=f"{kind} rollout {r}: {k}")


# ------------------------------------------------------------------------------------------
# 6. refills and validation
# ------------------------------------------------------------------------------------------
def test_reset_set_state_and_rewrap_refill(D):
    n, k = 16, 3
    rng = np.random.default_rng(2)
    env = D.CudaBatchedEnv("pendulum", n, seed=1, history_len=k, mask_velocities=True)
    for _ in range(4):
        env.act(_actions("pendulum", rng, (n,)))
    o = env.observe()
    assert not np.array_equal(o[:, :2], o[:, 4:])            # the frames differ after four steps
    env.set_state(*env.get_state())
    o2 = env.observe()
    np.testing.assert_array_equal(o2, np.tile(o[:, 4:], k))   # set_state: k copies of the current frame
    env.act(_actions("pendulum", rng, (n,)))
    env.reset()
    o3 = env.observe()
    np.testing.assert_array_equal(o3, np.tile(o3[:, 4:], k))
    env.act(_actions("pendulum", rng, (n,)))
    w = D.NormalizeWrapperEnv(D.ScalingWrapperEnv(D.MonitorWrapperEnv(env)))
    assert w.history_len() == k and w.masks_velocities() and w.obs_dim == 6 and w.scaling
    np.testing.assert_array_equal(w.observation_space().low, -np.ones(6, f32))
    w.observe()
    raw = w.get_original()[0]
    np.testing.assert_array_equal(raw, np.tile(raw[:, 4:], k))   # rewrapping restarts the history like set_state


def test_validation(D):
    from dril_b200 import _lib as L
    from dril_b200._lib import DrilError
    lib = D.Context.default().lib
    syn = D.CudaBatchedEnv("synthetic", 4, obs_dim=5)
    assert lib.dril_env_set_obs_history(syn.h, 2, 0) == 3            # DRIL_ERR_UNSUPPORTED
    with pytest.raises(DrilError):
        D.CudaBatchedEnv("synthetic", 4, obs_dim=5, history_len=2)
    # observe_params and history, in either order
    a = D.CudaBatchedEnv("cartpole", 8, seed=1, observe_params=True)
    assert lib.dril_env_set_obs_history(a.h, 2, 0) == 3
    assert lib.dril_env_set_obs_history(a.h, 1, 1) == 3
    assert lib.dril_env_set_obs_history(a.h, 1, 0) == 0               # (1, off) is the plain env: nothing to reject
    b = D.CudaBatchedEnv("cartpole", 8, seed=1, history_len=2)
    assert lib.dril_env_set_observe_params(b.h, 1) == 3
    with pytest.raises(DrilError):
        D.CudaBatchedEnv("cartpole", 8, seed=1, observe_params=True, mask_velocities=True)
    # k outside [1, 4]
    env = D.CudaBatchedEnv("acrobot", 8, seed=1)
    for bad in (0, 5, -1):
        assert lib.dril_env_set_obs_history(env.h, bad, 0) == 1      # DRIL_ERR_INVALID
    with pytest.raises(DrilError):
        D.CudaBatchedEnv("acrobot", 8, seed=1, history_len=5)
    # widths through dril_env_obs_dim; changes only before the first observation (reset and set_state do not count)
    d = L.c_i32(0)
    env.reset()
    env.set_state(*env.get_state())
    for (k, m), w in {(4, 0): 24, (4, 1): 16, (1, 1): 4, (2, 0): 12, (1, 0): 6}.items():
        L.check(lib.dril_env_set_obs_history(env.h, k, m))
        L.check(lib.dril_env_obs_dim(env.h, C.byref(d)))
        assert d.value == w, (k, m, d.value)
    L.check(lib.dril_env_set_obs_history(env.h, 3, 1))
    obs = np.empty((8, 12), f32)
    L.check(lib.dril_env_observe(env.h, L.ptr(obs)))
    np.testing.assert_array_equal(obs, np.tile(obs[:, 8:], 3))
    assert lib.dril_env_set_obs_history(env.h, 2, 1) == 1
    assert lib.dril_env_set_obs_history(env.h, 3, 1) == 0             # unchanged: allowed
    # a policy or buffer built for the base width is rejected
    hist = D.CudaBatchedEnv("cartpole", 16, seed=1, history_len=4, mask_velocities=True)
    base = D.CudaBatchedEnv("cartpole", 16, seed=1)
    layer = D.ActorCriticLayer(base.observation_space(), base.action_space(), hidden_dims=[64, 64])
    alg = D.PPO(n_steps=4)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
    buf = D.RolloutBuffer(base.observation_space(), base.action_space(), 0.95, 0.99, 4, 16)
    with pytest.raises(DrilError):
        D.collect_rollout(buf, agent, alg, hist)
    # set_env_params() with no ranges: back to lo = hi = the defaults
    hist.set_env_params(length=(0.25, 1.0))
    hist.set_env_params()
    assert hist.env_param_ranges() is None and hist.observe().shape == (16, 8)
    np.testing.assert_array_equal(_params_array(hist)[:, 0], np.array([v for _, v in EP.ENV_PARAMS["cartpole"]], f32))


# ------------------------------------------------------------------------------------------
# 7. update paths by shape, the tcgen05 loss/grad kernel at the new widths, one update
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
def test_update_path_by_width(D, kind):
    for mask in (False, True):
        for k in range(1, 5):
            env = D.CudaBatchedEnv(kind, 8, seed=1, history_len=k, mask_velocities=mask)
            layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=[64, 64])
            agent = D.Agent(layer, D.PPO(n_steps=4), rng=np.random.default_rng(0))
            w = env.obs_dim
            assert w == EH.history_obs_dim(kind, k, mask)
            assert agent.device.update_path() == ("tensor" if w <= 15 else "mma"), (kind, k, mask, w)
            env.close()


UPDATE_SHAPES = [(1, [64, 64], "discrete", 3), (8, [64, 64], "discrete", 2), (8, [128, 128, 64], "discrete", 3),
                 (9, [64, 64], "continuous", 1), (9, [128, 128, 64], "continuous", 1), (6, [64, 64], "discrete", 2)]


@pytest.mark.parametrize("obs_dim,hidden,act_kind,n_act", UPDATE_SHAPES)
def test_ftg_loss_grad_vs_fp64(D, obs_dim, hidden, act_kind, n_act):
    if act_kind == "discrete":
        spec = OP.PolicySpec(obs_dim, hidden, "discrete", n_act, act_start=1)
        space = D.Discrete(n_act, 1)
    else:
        spec = OP.PolicySpec(obs_dim, hidden, "continuous", 1, act_low=[-2], act_high=[2])
        space = D.Box(np.array([-2], f32), np.array([2], f32))
    rng = np.random.default_rng(obs_dim * 100 + len(hidden) * 10 + n_act)
    flat = (OP.init_params(spec, seed=4) + rng.normal(size=spec.n_params()).astype(f32) * 0.05).astype(f32)
    p = D.DevicePolicy(D.Context.default(), obs_dim, hidden, space)
    p.set_params(flat)
    assert p.update_path() == "tensor"
    B = D.Context.default().sm_count() * 64 * 2 + 37
    one = np.ones(B)
    for norm, cvf in ((True, None), (False, 0.5)):
        mb = O64.scaled_minibatch(spec, flat, one, one, rng, clip_range_vf=cvf)
        alg = D.PPO(ent_coef=0.0, clip_range_vf=cvf, normalize_advantage=norm)
        cfg = OO.PPOConfig(ent_coef=0.0, clip_range_vf=cvf, normalize_advantage=norm)
        loss, stats, g = p.loss_grad(*mb, alg.hyper())
        eloss, eg, estats = O64.loss64(spec, flat, *mb, cfg)
        assert abs(loss - eloss) <= 1e-4 * max(1.0, abs(eloss)), (loss, eloss)
        for k in O64.STAT_NAMES:
            assert abs(stats[k] - estats[k]) <= 1e-4 * max(1.0, abs(estats[k])), (k, stats[k], estats[k])
        O64.assert_blocks_close(spec, g, eg, 1e-4, what=f"obs_dim {obs_dim} {hidden} {act_kind}({n_act})")
    p.close()


def _relerr(a, b):
    return float(np.linalg.norm(np.asarray(a, np.float64) - b) / max(np.linalg.norm(np.asarray(b, np.float64)), 1e-30))


def test_update_vs_oracle(D):
    """one dril_ppo_update on a CartPole rollout without velocities, 4 frames (width 8: ftg instead of ft)"""
    from dril_b200 import _lib as L
    n, T = 1024, 32
    env = D.CudaBatchedEnv("cartpole", n, seed=5, normalize=D.NormalizeConfig(), history_len=4, mask_velocities=True)
    spec = _spec("cartpole", env.obs_dim)
    flat = OP.init_params(spec, seed=2)
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=spec.hidden)
    alg = D.PPO(n_steps=T, batch_size=T * n // 4, epochs=2, ent_coef=0.01)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
    agent.set_parameters(flat)
    assert agent.device.update_path() == "tensor"
    buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
    D.collect_rollout(buf, agent, alg, env)
    ob = {k: buf.download(k) for k in ("obs", "actions", "rewards", "values", "logprobs", "advantages", "returns")}
    assert ob["obs"].shape[-1] == 8
    st = D.IterStats()
    h = alg.hyper()
    L.check(agent.ctx.lib.dril_ppo_update(agent.device.h, buf.h, C.byref(h), alg.epochs, alg.batch_size, 41, 2, C.byref(st)))
    cfg = OO.PPOConfig(n_steps=T, batch_size=T * n // 4, epochs=2, ent_coef=0.01)
    opt = OO.Adam(flat.size, lr=cfg.learning_rate)
    new_flat, means, _ = OO.ppo_update(spec, flat, opt, ob, cfg, shuffle_seed=41, epoch_counter0=2)
    got = agent.device.get_params()
    assert st.n_minibatch_steps == 8
    assert _relerr(got - flat, new_flat - flat) < 2e-3, _relerr(got - flat, new_flat - flat)
    np.testing.assert_allclose(got, new_flat, rtol=1e-4, atol=2e-6)
    for k in ("policy_loss", "value_loss", "entropy_loss", "approx_kl_div", "clip_fraction", "loss", "grad_norm"):
        assert abs(getattr(st, k) - means[k]) <= 2e-4 * max(1.0, abs(means[k])), (k, getattr(st, k), means[k])
    buf.close()


# ------------------------------------------------------------------------------------------
# 8. learning: CartPole without velocities, from a 4-frame history
# ------------------------------------------------------------------------------------------
LEARN_ITERS, LEARN_TARGET = 150, 475.0


def _cartpole_agent(D, n, T, k):
    env = D.CudaBatchedEnv("cartpole", n, seed=0, monitor_window=100, history_len=k, mask_velocities=True)
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=[64, 64])
    alg = D.PPO(n_steps=T, batch_size=T * n // 4, epochs=4, learning_rate=1e-3, ent_coef=0.0)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
    return env, alg, agent


def _train_best(D, env, alg, agent, n, T, stop):
    best, it = 0.0, 0
    for it in range(LEARN_ITERS):
        D.train(agent, env, alg, n * T)
        best = max(best, env.monitor_stats()["ep_len_mean"])
        if best >= stop:
            break
    return best, it + 1


def test_cartpole_without_velocities_learns_from_history(D):
    n, T = 4096, 128
    env, alg, agent = _cartpole_agent(D, n, T, 4)
    assert env.obs_dim == 8 and agent.device.update_path() == "tensor"
    best, iters = _train_best(D, env, alg, agent, n, T, 499.5)
    env1, alg1, agent1 = _cartpole_agent(D, n, T, 1)
    best1, iters1 = _train_best(D, env1, alg1, agent1, n, T, 499.5)
    print(f"CartPole without velocities: history_len 4 best ep_len_mean {best} after {iters} iterations; "
          f"history_len 1 best {best1} after {iters1} iterations")
    assert best >= LEARN_TARGET, best
    ev = D.CudaBatchedEnv("cartpole", 16, max_steps=500, seed=123, monitor_window=100, history_len=4, mask_velocities=True)
    res = D.evaluate_agent(agent, ev, n_eval_episodes=16, deterministic=True)
    print(f"evaluate_agent on a fresh env: mean return {res['mean_reward']}")
    assert res["mean_reward"] >= LEARN_TARGET, res


def test_cartpole_history_training_is_deterministic(D):
    n, T = 1024, 64
    got = []
    for _ in range(2):
        env, alg, agent = _cartpole_agent(D, n, T, 4)
        for _ in range(4):
            D.train(agent, env, alg, n * T)
        got.append(agent.device.get_params())
        env.close()
    np.testing.assert_array_equal(got[0], got[1])
