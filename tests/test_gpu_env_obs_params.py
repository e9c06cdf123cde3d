"""Parameter-augmented observations on the device (observe_params): the base columns of an augmented run against a plain run
(bit for bit), the fused fast, cooperative and tcgen05-actor rollouts, the compat path under Monitor, Normalize and Scaling and
dril_evaluate against the oracle (oracle/env_obs_params.py), sharding, validation, the tcgen05 loss/grad kernel and update at the
new widths 7, 10 and 12, and CartPole trained on randomised pole lengths and masses with the parameters in its observation."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import env_obs_params as EOP, env_params as EP, envs as OE, policy as OP, ppo as OO, ppo64 as O64

pytestmark = pytest.mark.gpu
f32 = np.float32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KINDS = ("cartpole", "pendulum", "mountaincar", "mountaincar_continuous", "acrobot")
D0 = EOP.BASE_OBS_DIM
CONT = {"pendulum": 2.0, "mountaincar_continuous": 1.0}   # Box(1) envs: action bound
MCC_LOW, MCC_HIGH = np.array([-1.2, -0.07], f32), np.array([0.6, 0.07], f32)


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
    hi[:, ::5] = lo[:, ::5]                        # some envs fixed
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


# path: (n, T, max_steps, normalize); gtc: >= 96 envs per SM, the actor on tcgen05 (rollout_gtc.cuh)
PATHS = {"fast": (300, 24, 10, None), "coop": (200, 20, 9, "full"), "gtc": (14208, 4, 3, "ret")}
ENV_FIELDS = ("rewards", "flags", "episode_r", "episode_l")


# ------------------------------------------------------------------------------------------
# 1. the base columns are free: an augmented run's columns [0, D) == a plain run, bit for bit
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("path", list(PATHS))
def test_base_columns_are_free(D, kind, path):
    n, T, ms, norm = PATHS[path]
    rng = np.random.default_rng(3)
    lo, hi = _ranges(kind, n, rng)
    envs = [D.CudaBatchedEnv(kind, n, max_steps=ms, seed=9, monitor_window=100, normalize=_norm(D, norm), env_params=_kw(kind, lo, hi),
                             observe_params=obs) for obs in (False, True)]
    assert envs[0].obs_dim == D0[kind] and envs[1].obs_dim == EOP.obs_params_dim(kind) and envs[1].observes_params()
    for rollout in range(3):
        forced = _actions(kind, rng, (T, n))
        outs = []
        for env in envs:
            _, _, agent, alg = _agent(D, env, kind, T)
            if path == "gtc" or env.obs_dim > 4:
                assert agent.device.update_path() == "tensor"
            buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
            _, ok = D.collect_rollout(buf, agent, alg, env, forced_actions=forced)
            assert ok
            outs.append({k: buf.download(k) for k in ENV_FIELDS + ("obs",)})
            buf.close()
        np.testing.assert_array_equal(outs[1]["obs"][..., :D0[kind]], outs[0]["obs"], err_msg=f"{kind} {path} {rollout}: obs")
        for k in ENV_FIELDS:
            np.testing.assert_array_equal(outs[1][k], outs[0][k], err_msg=f"{kind} {path} rollout {rollout}: {k}")
        assert ((outs[0]["flags"] >> 1) & 1).any()
        np.testing.assert_array_equal(envs[1].get_state()[0], envs[0].get_state()[0])
        np.testing.assert_array_equal(envs[1].get_state()[1], envs[0].get_state()[1])
        np.testing.assert_array_equal(_params_array(envs[1]), _params_array(envs[0]))
        if norm:
            s0, s1 = envs[0].norm_stats(), envs[1].norm_stats()
            for k in s0:
                got = s1[k][:D0[kind]] if k in ("obs_mean", "obs_var") else s1[k]
                np.testing.assert_array_equal(got, s0[k], err_msg=k)


# ------------------------------------------------------------------------------------------
# 2. fused rollout against the oracle
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("path", list(PATHS))
def test_fused_rollout_vs_oracle(D, kind, path):
    n, T, ms, norm = PATHS[path]
    rng = np.random.default_rng(7)
    lo, hi = _ranges(kind, n, rng)
    env = D.CudaBatchedEnv(kind, n, max_steps=ms, seed=9, monitor_window=100, normalize=_norm(D, norm), env_params=_kw(kind, lo, hi),
                           observe_params=True)
    ob = EOP.make(kind, n, seed=9, max_steps=ms, param_ranges=(lo, hi))
    o = OE.MonitorWrapper(OE.ParallelEnv(ob))
    if norm:
        o = OE.NormalizeWrapper(o, ob.obs_dim, norm_obs=norm == "full")
    spec, flat, agent, alg = _agent(D, env, kind, T)
    assert spec.obs_dim == EOP.obs_params_dim(kind)
    assert agent.device.update_path() == "tensor"
    # (training normaliser on observations: the device's double moment sums vs NumPy's fp32 variance, see test_gpu_envs.py)
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
        np.testing.assert_array_equal(_params_array(env), ob.p)
        np.testing.assert_array_equal(env.get_state()[0], ob.state)
        assert tr.any()
        buf.close()


# ------------------------------------------------------------------------------------------
# 3. compat observe / act! under Monitor, Normalize and Scaling
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,norm,scaled", [
    ("cartpole", False, False), ("acrobot", True, False), ("mountaincar", False, False),
    ("pendulum", False, True), ("pendulum", True, True), ("mountaincar_continuous", True, True),
    ("mountaincar_continuous", False, True)])
def test_compat_wrappers_vs_oracle(D, kind, norm, scaled):
    n, ms, steps = 301, 13, 50
    rng = np.random.default_rng(6)
    lo, hi = _ranges(kind, n, rng)
    # the wrapper stage switched on at construction (MonitorWrapperEnv etc. re-create the env: test_observation_space_and_rewrap)
    env = D.CudaBatchedEnv(kind, n, max_steps=ms, seed=5, monitor_window=100, normalize=D.NormalizeConfig() if norm else None,
                           scaling=scaled, env_params=_kw(kind, lo, hi), observe_params=True)
    assert env.observes_params() and env.obs_dim == EOP.obs_params_dim(kind)
    sp = env.observation_space()
    assert (sp.low[D0[kind]:] == 0).all() and np.isposinf(sp.high[D0[kind]:]).all()
    if scaled:
        assert (sp.low[:D0[kind]] == -1).all() and (sp.high[:D0[kind]] == 1).all()
    sc = None
    if scaled:
        sc = (OE.PENDULUM_OBS_LOW, OE.PENDULUM_OBS_HIGH) if kind == "pendulum" else (MCC_LOW, MCC_HIGH)
    ob = EOP.make(kind, n, seed=5, max_steps=ms, param_ranges=(lo, hi), scaling=sc)
    np.testing.assert_array_equal(_params_array(env), ob.p)
    o = OE.MonitorWrapper(OE.ParallelEnv(ob))
    if norm:
        o = OE.NormalizeWrapper(o, ob.obs_dim)
    # Acrobot's cos(theta1) / cos(theta2) columns start nearly constant: their running variance is tiny, and the last bits in
    # which the device's fp64 moment sums and NumPy's fp32 variance differ show up as ~3e-4 in those normalised columns
    tol = dict(rtol=3e-5, atol=1e-3 if kind == "acrobot" else 3e-4) if norm else dict(rtol=0, atol=0)
    np.testing.assert_allclose(env.observe(), o.observe(), **tol)
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
        for i in np.nonzero(tro)[0]:
            got = infos[i]["terminal_observation"]
            np.testing.assert_allclose(got, info["terminal_observation"][i], **tol)
            if not norm:     # the parameter columns of the ended episode, raw
                np.testing.assert_array_equal(got[D0[kind]:], info["terminal_observation"][i][D0[kind]:])
        for i in np.nonzero(teo | tro)[0]:
            assert abs(infos[i]["episode"]["r"] - info["episode_r"][i]) <= 1e-5 * max(1.0, abs(info["episode_r"][i]))
            assert infos[i]["episode"]["l"] == info["episode_l"][i]
        np.testing.assert_array_equal(_params_array(env), ob.p)
        n_trunc += tro.sum()
    assert n_trunc > 0
    if not norm:
        np.testing.assert_array_equal(env.observe()[:, D0[kind]:], _params_array(env).T)


# ------------------------------------------------------------------------------------------
# 4. dril_evaluate against the oracle loop
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
def test_evaluate_vs_oracle_loop(D, kind):
    n, ms, n_eval = 37, 40, 60
    rng = np.random.default_rng(8)
    lo, hi = _ranges(kind, n, rng)
    env = D.CudaBatchedEnv(kind, n, max_steps=ms, seed=9, monitor_window=100, env_params=_kw(kind, lo, hi), observe_params=True)
    spec, flat, agent, _ = _agent(D, env, kind, 8, seed=5)
    er, el = D.evaluate_agent(agent, env, n_eval_episodes=n_eval, deterministic=True, return_stats=False, chunk_steps=7)
    o = OE.MonitorWrapper(OE.ParallelEnv(EOP.make(kind, n, seed=9, max_steps=ms, param_ranges=(lo, hi))))
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
    """the compat path against tests/golden/orc_<kind>_obs_params_replay.npz alone"""
    g = np.load(os.path.join(ROOT, "tests", "golden", f"orc_{kind}_obs_params_replay.npz"))
    n = g["obs"].shape[1]
    env = D.CudaBatchedEnv(kind, n, max_steps=int(g["max_steps"]), seed=int(g["seed"]), env_params=_kw(kind, g["lo"], g["hi"]),
                           observe_params=True)
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
# 5. sharding
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ("cartpole", "acrobot", "pendulum"))
def test_sharding_invariant(D, kind):
    m, T, ms = 150, 16, 7
    rng = np.random.default_rng(9)
    lo, hi = _ranges(kind, 2 * m, rng)
    whole = D.CudaBatchedEnv(kind, 2 * m, max_steps=ms, seed=3, env_params=_kw(kind, lo, hi), observe_params=True)
    parts = [D.CudaBatchedEnv(kind, m, max_steps=ms, seed=3, gid_offset=m * i, observe_params=True,
                              env_params=_kw(kind, lo[:, m * i:m * (i + 1)], hi[:, m * i:m * (i + 1)])) for i in range(2)]
    for t in range(25):
        a = _actions(kind, rng, (2 * m,))
        rw, tew, trw, iw = whole.act(a)
        got = [p.act(a[m * i:m * (i + 1)]) for i, p in enumerate(parts)]
        np.testing.assert_array_equal(rw, np.concatenate([g[0] for g in got]))
        np.testing.assert_array_equal(trw, np.concatenate([g[2] for g in got]))
        np.testing.assert_array_equal(whole.observe(), np.concatenate([p.observe() for p in parts]))
        for i in np.nonzero(trw)[0]:
            np.testing.assert_array_equal(iw[i]["terminal_observation"], got[i // m][3][i % m]["terminal_observation"])
    forced = _actions(kind, rng, (T, 2 * m))
    outs = []
    for env, sl in [(whole, slice(0, 2 * m))] + [(p, slice(m * i, m * (i + 1))) for i, p in enumerate(parts)]:
        _, _, agent, alg = _agent(D, env, kind, T)
        buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, env.n_envs)
        D.collect_rollout(buf, agent, alg, env, forced_actions=np.ascontiguousarray(forced[:, sl]))
        outs.append({k: buf.download(k) for k in ("obs", "rewards", "flags")})
        buf.close()
    for k in ("obs", "rewards", "flags"):
        np.testing.assert_array_equal(outs[0][k], np.concatenate([outs[1][k], outs[2][k]], axis=1))


# ------------------------------------------------------------------------------------------
# 6. validation
# ------------------------------------------------------------------------------------------
def test_validation(D):
    from dril_b200 import _lib as L
    from dril_b200._lib import DrilError
    lib = D.Context.default().lib
    # the synthetic env has no parameters
    syn = D.CudaBatchedEnv("synthetic", 4, obs_dim=5)
    assert lib.dril_env_set_observe_params(syn.h, 1) == 3            # DRIL_ERR_UNSUPPORTED
    with pytest.raises(DrilError):
        D.CudaBatchedEnv("synthetic", 4, obs_dim=5, observe_params=True)
    # dril_env_obs_dim, and the width only changes before the first observation (reset and set_state do not count)
    env = D.CudaBatchedEnv("acrobot", 8, seed=1)
    d = L.c_i32(0)
    L.check(lib.dril_env_obs_dim(env.h, C.byref(d)))
    assert d.value == 6
    env.reset()
    env.set_state(*env.get_state())
    L.check(lib.dril_env_set_observe_params(env.h, 1))
    L.check(lib.dril_env_obs_dim(env.h, C.byref(d)))
    assert d.value == 12
    L.check(lib.dril_env_set_observe_params(env.h, 0))
    L.check(lib.dril_env_obs_dim(env.h, C.byref(d)))
    assert d.value == 6
    L.check(lib.dril_env_set_observe_params(env.h, 1))
    obs = np.empty((8, 12), f32)
    L.check(lib.dril_env_observe(env.h, L.ptr(obs)))
    np.testing.assert_array_equal(obs[:, 6:], np.broadcast_to(np.array([v for _, v in EP.ENV_PARAMS["acrobot"]], f32), (8, 6)))
    with pytest.raises(DrilError):
        L.check(lib.dril_env_set_observe_params(env.h, 0))
    assert lib.dril_env_set_observe_params(env.h, 0) == 1            # DRIL_ERR_INVALID
    # a policy or buffer built for the base width fails the obs_dim check
    aug = D.CudaBatchedEnv("cartpole", 16, seed=1, observe_params=True)
    base = D.CudaBatchedEnv("cartpole", 16, seed=1)
    layer = D.ActorCriticLayer(base.observation_space(), base.action_space(), hidden_dims=[64, 64])
    alg = D.PPO(n_steps=4)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
    buf = D.RolloutBuffer(base.observation_space(), base.action_space(), 0.95, 0.99, 4, 16)
    with pytest.raises(DrilError):
        D.collect_rollout(buf, agent, alg, aug)
    # set_env_params() with no ranges: back to lo = hi = the defaults, still observed
    aug.set_env_params(length=(0.25, 1.0))
    aug.set_env_params()
    assert aug.env_param_ranges() is None
    o = aug.observe()
    assert o.shape == (16, 10)
    np.testing.assert_array_equal(o[:, 4:], np.broadcast_to(np.array([v for _, v in EP.ENV_PARAMS["cartpole"]], f32), (16, 6)))
    np.testing.assert_array_equal(_params_array(aug), o[:, 4:].T)


def test_observation_space_and_rewrap(D):
    env = D.CudaBatchedEnv("pendulum", 8, seed=1, env_params=dict(l=(0.5, 1.5)), observe_params=True)
    sp = env.observation_space()
    np.testing.assert_array_equal(sp.low, np.array([-1, -1, -8, 0, 0, 0, 0], f32))
    assert np.isposinf(sp.high[3:]).all()
    env.set_env_params(l=(1.0, 2.0))
    assert env.observation_space() == sp
    w = D.NormalizeWrapperEnv(D.ScalingWrapperEnv(D.MonitorWrapperEnv(env)))
    assert w.observes_params() and w.obs_dim == 7
    np.testing.assert_array_equal(w.observation_space().low, np.array([-1, -1, -1, 0, 0, 0, 0], f32))


# ------------------------------------------------------------------------------------------
# 7. the tcgen05 loss/grad kernel and update at the new widths
# ------------------------------------------------------------------------------------------
# (obs_dim, hidden, head, expected update_path): at width 12 a [128,128,64] Discrete(3) policy no longer fits ftg's shared memory
# and takes the mma.sync 3xTF32 kernel
UPDATE_SHAPES = [(10, [64, 64], "discrete", 2, "tensor"), (10, [128, 128, 64], "discrete", 2, "tensor"),
                 (12, [64, 64], "discrete", 3, "tensor"), (12, [128, 128, 64], "discrete", 3, "mma"),
                 (7, [64, 64], "continuous", 1, "tensor"), (7, [128, 128, 64], "continuous", 1, "tensor")]


@pytest.mark.parametrize("obs_dim,hidden,act_kind,n_act,path", UPDATE_SHAPES)
def test_ftg_loss_grad_vs_fp64(D, obs_dim, hidden, act_kind, n_act, path):
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
    assert p.update_path() == path
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


@pytest.mark.parametrize("kind", ("cartpole", "acrobot", "pendulum"))
def test_update_vs_oracle(D, kind):
    """one dril_ppo_update on an augmented rollout (CartPole [64,64] Discrete(2) at width 10 leaves the ft kernel for ftg)"""
    from dril_b200 import _lib as L
    n, T = 1024, 32
    rng = np.random.default_rng(11)
    lo, hi = _ranges(kind, n, rng)
    env = D.CudaBatchedEnv(kind, n, seed=5, normalize=D.NormalizeConfig(), env_params=_kw(kind, lo, hi), observe_params=True)
    spec = _spec(kind, env.obs_dim)
    flat = OP.init_params(spec, seed=2)
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=spec.hidden)
    alg = D.PPO(n_steps=T, batch_size=T * n // 4, epochs=2, ent_coef=0.01)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
    agent.set_parameters(flat)
    assert agent.device.update_path() == "tensor"
    buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
    D.collect_rollout(buf, agent, alg, env)
    ob = {k: buf.download(k) for k in ("obs", "actions", "rewards", "values", "logprobs", "advantages", "returns")}
    assert ob["obs"].shape[-1] == EOP.obs_params_dim(kind)
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
# 8. learning: CartPole on randomised pole length and mass, observing them
# ------------------------------------------------------------------------------------------
RANGES = dict(length=(0.25, 1.0), masspole=(0.05, 0.2))


def _cartpole_agent(D, n, T):
    env = D.CudaBatchedEnv("cartpole", n, seed=0, monitor_window=100, env_params=RANGES, observe_params=True)
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=[64, 64])
    alg = D.PPO(n_steps=T, batch_size=T * n // 4, epochs=4, learning_rate=1e-3, ent_coef=0.0)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
    return env, alg, agent


def test_cartpole_observing_parameters_learns_and_holds_the_corners(D):
    n, T = 4096, 128
    env, alg, agent = _cartpole_agent(D, n, T)
    assert env.obs_dim == 10 and agent.device.update_path() == "tensor"
    best, it = 0.0, 0
    for it in range(150):
        D.train(agent, env, alg, n * T)
        best = max(best, env.monitor_stats()["ep_len_mean"])
        if best >= 499.5:
            break
    print(f"randomised + observed CartPole: best ep_len_mean {best} after {it + 1} iterations")
    assert best >= 499.5, best
    for length in (0.25, 1.0):
        for masspole in (0.05, 0.2):
            ev = D.CudaBatchedEnv("cartpole", 16, max_steps=500, seed=123, monitor_window=100,
                                  env_params=dict(length=length, masspole=masspole), observe_params=True)
            res = D.evaluate_agent(agent, ev, n_eval_episodes=16, deterministic=True)
            print(f"length {length} masspole {masspole}: mean return {res['mean_reward']}")
            assert res["mean_reward"] >= 475, (length, masspole, res)


def test_cartpole_observing_parameters_is_deterministic(D):
    n, T = 1024, 64
    got = []
    for _ in range(2):
        env, alg, agent = _cartpole_agent(D, n, T)
        for _ in range(4):
            D.train(agent, env, alg, n * T)
        got.append(agent.device.get_params())
        env.close()
    np.testing.assert_array_equal(got[0], got[1])
