"""Per-env physical parameters and per-episode domain randomisation on the device: the parametrised kernels at the default values
against the default kernels (bit for bit), against the oracle (oracle/env_params.py) with randomised per-env ranges on the
compat step, the fast, cooperative and tcgen05-actor rollouts and dril_evaluate, against the frozen fixtures alone, sharding,
validation, and CartPole trained on randomised pole lengths and masses holding the pole at the corners of that range."""
import os

import numpy as np
import pytest

from oracle import env_params as EP, envs as OE, policy as OP, ppo as OO

pytestmark = pytest.mark.gpu
f32 = np.float32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KINDS = ("cartpole", "pendulum", "mountaincar", "mountaincar_continuous", "acrobot")
OBS_DIM = {"cartpole": 4, "pendulum": 3, "mountaincar": 2, "mountaincar_continuous": 2, "acrobot": 6}
CONT = {"pendulum": 2.0, "mountaincar_continuous": 1.0}   # Box(1) envs: action bound


@pytest.fixture(scope="module")
def D():
    import __graft_entry__
    __graft_entry__.build()
    import dril_b200
    return dril_b200


@pytest.fixture
def no_tc_rollout(D):
    """CartPole: the default env would take the tensor-core rollout, an env with parameters the fast kernel; compare within the
    same kernel family"""
    D.set_option("tc_rollout", 0)
    yield
    D.set_option("tc_rollout", 1)


def _spec(kind):
    if kind in CONT:
        b = CONT[kind]
        return OP.PolicySpec(OBS_DIM[kind], [64, 64], "continuous", 1, act_low=[-b], act_high=[b])
    return OP.PolicySpec(OBS_DIM[kind], [64, 64], "discrete", 2 if kind == "cartpole" else 3, act_start=1)


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


FIELDS = ("obs", "actions", "rewards", "values", "logprobs", "flags", "boot", "last_values", "episode_r", "episode_l")


def _agent(D, env, kind, T, seed=2):
    spec = _spec(kind)
    flat = (OP.init_params(spec, seed=seed) + np.random.default_rng(seed).normal(size=spec.n_params()).astype(f32) * 0.05).astype(f32)
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=[64, 64])
    alg = D.PPO(n_steps=T, gamma=0.97, gae_lambda=0.9)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
    agent.set_parameters(flat)
    return spec, flat, agent, alg


# path: (n, T, max_steps, normalize)
PATHS = {"fast": (300, 24, 10, None), "coop": (200, 20, 9, "full"), "gtc": (14208, 4, 3, "ret")}


# ------------------------------------------------------------------------------------------
# defaults are free: parametrised kernels at the default values == default kernels, bit for bit
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("path", ["fast", "coop", "gtc"])
def test_defaults_are_free_rollout(D, no_tc_rollout, kind, path):
    n, T, ms, norm = PATHS[path]
    cfg = (lambda: D.NormalizeConfig(norm_obs=norm == "full")) if norm else (lambda: None)
    defaults = {nm: v for nm, v in EP.ENV_PARAMS[kind]}
    envs = [D.CudaBatchedEnv(kind, n, max_steps=ms, seed=9, monitor_window=100, normalize=cfg()),
            D.CudaBatchedEnv(kind, n, max_steps=ms, seed=9, monitor_window=100, normalize=cfg(), env_params=defaults)]
    assert envs[0].env_param_ranges() is None and envs[1].env_param_ranges() is not None
    rng = np.random.default_rng(3)
    for rollout in range(3):
        forced = _actions(kind, rng, (T, n)) if rollout == 0 else None
        outs = []
        for env in envs:
            _, _, agent, alg = _agent(D, env, kind, T)
            buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
            _, ok = D.collect_rollout(buf, agent, alg, env, forced_actions=forced)
            assert ok
            outs.append({k: buf.download(k) for k in FIELDS})
            buf.close()
        for k in FIELDS:
            np.testing.assert_array_equal(outs[0][k], outs[1][k], err_msg=f"{kind} {path} rollout {rollout}: {k}")
        assert _flags_any(outs[0]["flags"])
        np.testing.assert_array_equal(envs[0].get_state()[0], envs[1].get_state()[0])
        if norm:
            s0, s1 = envs[0].norm_stats(), envs[1].norm_stats()
            for k in s0:
                np.testing.assert_array_equal(s0[k], s1[k])
    np.testing.assert_array_equal(_params_array(envs[1]), _params_array(envs[0]))


def _flags_any(f):
    return ((f >> 1) & 1).any()


@pytest.mark.parametrize("kind", KINDS)
def test_defaults_are_free_compat_and_evaluate(D, kind):
    n, ms = 97, 12
    defaults = {nm: v for nm, v in EP.ENV_PARAMS[kind]}
    a = D.CudaBatchedEnv(kind, n, max_steps=ms, seed=4, monitor_window=100)
    b = D.CudaBatchedEnv(kind, n, max_steps=ms, seed=4, monitor_window=100, env_params=defaults)
    rng = np.random.default_rng(5)
    np.testing.assert_array_equal(a.observe(), b.observe())
    for _ in range(30):
        act = _actions(kind, rng, (n,))
        ra, tea, tra, ia = a.act(act)
        rb, teb, trb, ib = b.act(act)
        np.testing.assert_array_equal(ra, rb)
        np.testing.assert_array_equal(tea, teb)
        np.testing.assert_array_equal(tra, trb)
        np.testing.assert_array_equal(a.observe(), b.observe())
        for i in np.nonzero(tra)[0]:
            np.testing.assert_array_equal(ia[i]["terminal_observation"], ib[i]["terminal_observation"])
    res = []
    for env in (a, b):
        _, _, agent, _ = _agent(D, env, kind, 8)
        res.append(D.evaluate_agent(agent, env, n_eval_episodes=150, deterministic=True, return_stats=False, chunk_steps=7))
    np.testing.assert_array_equal(res[0][0], res[1][0])
    np.testing.assert_array_equal(res[0][1], res[1][1])


# ------------------------------------------------------------------------------------------
# replay against the oracle with randomised per-env ranges
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
def test_compat_replay_vs_oracle(D, kind):
    n, ms, steps = 301, 13, 60
    rng = np.random.default_rng(6)
    lo, hi = _ranges(kind, n, rng)
    env = D.CudaBatchedEnv(kind, n, max_steps=ms, seed=5, monitor_window=100, env_params=_kw(kind, lo, hi))
    ob = EP.PARAM_BATCHES[kind](n, seed=5, max_steps=ms, param_ranges=(lo, hi))
    o = OE.MonitorWrapper(OE.ParallelEnv(ob))
    np.testing.assert_array_equal(env.observe(), o.observe())
    np.testing.assert_array_equal(_params_array(env), ob.p)
    for t in range(steps):
        a = _actions(kind, rng, (n,))
        r, te, tr, infos = env.act(a)
        ro, teo, tro, info = o.act(a)
        np.testing.assert_array_equal(te, teo)
        np.testing.assert_array_equal(tr, tro)
        np.testing.assert_array_equal(r, ro)
        np.testing.assert_array_equal(env.observe(), o.observe())
        np.testing.assert_array_equal(_params_array(env), ob.p)      # redrawn exactly at the oracle's resets
        for i in np.nonzero(tro)[0]:
            np.testing.assert_array_equal(infos[i]["terminal_observation"], info["terminal_observation"][i])
        if t == steps // 2:                                           # new ranges mid-episode; then reset!(env)
            lo, hi = _ranges(kind, n, rng)
            env.set_env_params(**_kw(kind, lo, hi))
            ob.set_param_ranges(lo, hi)
            np.testing.assert_array_equal(_params_array(env), ob.p)
    env.reset()
    o.reset()
    np.testing.assert_array_equal(_params_array(env), ob.p)
    np.testing.assert_array_equal(env.observe(), o.observe())


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("path", ["fast", "coop", "gtc"])
def test_fused_rollout_vs_oracle(D, kind, path):
    n, T, ms, norm = PATHS[path]
    rng = np.random.default_rng(7)
    lo, hi = _ranges(kind, n, rng)
    env = D.CudaBatchedEnv(kind, n, max_steps=ms, seed=9, monitor_window=100,
                           normalize=D.NormalizeConfig(norm_obs=norm == "full") if norm else None, env_params=_kw(kind, lo, hi))
    ob = EP.PARAM_BATCHES[kind](n, seed=9, max_steps=ms, param_ranges=(lo, hi))
    o = OE.MonitorWrapper(OE.ParallelEnv(ob))
    if norm:
        o = OE.NormalizeWrapper(o, ob.obs_dim, norm_obs=norm == "full")
    spec, flat, agent, alg = _agent(D, env, kind, T)
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
        np.testing.assert_allclose(np.where(tr, buf.download("boot"), 0), eo["boot"], **tol)
        done = te | tr
        np.testing.assert_allclose(buf.download("episode_r")[done], eo["episode_r"][done], rtol=1e-5)
        np.testing.assert_array_equal(buf.download("episode_l")[done], eo["episode_l"][done])
        np.testing.assert_array_equal(_params_array(env), ob.p)
        np.testing.assert_array_equal(env.get_state()[0], ob.state)
        assert tr.any()
        buf.close()


@pytest.mark.parametrize("kind", KINDS)
def test_evaluate_vs_oracle_loop(D, kind):
    n, ms, n_eval = 37, 40, 60
    rng = np.random.default_rng(8)
    lo, hi = _ranges(kind, n, rng)
    env = D.CudaBatchedEnv(kind, n, max_steps=ms, seed=9, monitor_window=100, env_params=_kw(kind, lo, hi))
    spec, flat, agent, _ = _agent(D, env, kind, 8, seed=5)
    er, el = D.evaluate_agent(agent, env, n_eval_episodes=n_eval, deterministic=True, return_stats=False, chunk_steps=7)
    o = OE.MonitorWrapper(OE.ParallelEnv(EP.PARAM_BATCHES[kind](n, seed=9, max_steps=ms, param_ranges=(lo, hi))))
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
    """the compat path against tests/golden/orc_<kind>_params_replay.npz alone"""
    g = np.load(os.path.join(ROOT, "tests", "golden", f"orc_{kind}_params_replay.npz"))
    n = g["obs"].shape[1]
    env = D.CudaBatchedEnv(kind, n, max_steps=int(g["max_steps"]), seed=int(g["seed"]), env_params=_kw(kind, g["lo"], g["hi"]))
    np.testing.assert_array_equal(env.observe(), g["obs"][0])
    np.testing.assert_array_equal(_params_array(env), g["params"][0])
    for t, a in enumerate(g["actions"]):
        r, te, tr, infos = env.act(a)
        np.testing.assert_array_equal(r, g["rewards"][t])
        np.testing.assert_array_equal(te, g["term"][t])
        np.testing.assert_array_equal(tr, g["trunc"][t])
        for i in np.nonzero(tr)[0]:
            np.testing.assert_array_equal(infos[i]["terminal_observation"], g["terminal_obs"][t][i])
        np.testing.assert_array_equal(env.observe(), g["obs"][t + 1])
        np.testing.assert_array_equal(_params_array(env), g["params"][t + 1])


# ------------------------------------------------------------------------------------------
# sharding, validation, wrappers
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ("cartpole", "acrobot", "pendulum"))
def test_sharding_invariant(D, kind):
    m, T, ms = 150, 16, 7
    rng = np.random.default_rng(9)
    lo, hi = _ranges(kind, 2 * m, rng)
    whole = D.CudaBatchedEnv(kind, 2 * m, max_steps=ms, seed=3, env_params=_kw(kind, lo, hi))
    parts = [D.CudaBatchedEnv(kind, m, max_steps=ms, seed=3, gid_offset=m * i, env_params=_kw(kind, lo[:, m * i:m * (i + 1)], hi[:, m * i:m * (i + 1)]))
             for i in range(2)]
    for t in range(25):
        a = _actions(kind, rng, (2 * m,))
        rw, tew, trw, _ = whole.act(a)
        got = [p.act(a[m * i:m * (i + 1)]) for i, p in enumerate(parts)]
        np.testing.assert_array_equal(rw, np.concatenate([g[0] for g in got]))
        np.testing.assert_array_equal(tew, np.concatenate([g[1] for g in got]))
        np.testing.assert_array_equal(whole.observe(), np.concatenate([p.observe() for p in parts]))
        np.testing.assert_array_equal(_params_array(whole), np.concatenate([_params_array(p) for p in parts], axis=1))
    # fused rollout (fast kernel) with forced actions
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


def test_validation_and_clearing(D):
    from dril_b200._lib import DrilError
    env = D.CudaBatchedEnv("cartpole", 8, seed=1)
    for bad in ({"length": 0.0}, {"masspole": -0.1}, {"tau": float("nan")}, {"gravity": -1.0}, {"length": (1.0, 0.5)},
                {"force_mag": float("inf")}):
        with pytest.raises(DrilError):
            env.set_env_params(**bad)
    with pytest.raises(AssertionError):
        env.set_env_params(pole_length=1.0)
    env.set_env_params(gravity=0.0, force_mag=(0.0, 20.0))     # >= 0 is allowed for gravity and forces
    p = env.env_params()
    assert (p["gravity"] == 0).all() and (p["force_mag"] >= 0).all() and (p["force_mag"] <= 20).all()
    np.testing.assert_array_equal(p["length"], np.full(8, f32(0.5)))
    env.set_env_params()                                        # back to the built-in constants
    assert env.env_param_ranges() is None
    np.testing.assert_array_equal(env.env_params()["masspole"], np.full(8, f32(0.1)))
    for kind, bad in (("pendulum", {"dt": 0.0}), ("mountaincar", {"force": -1e-3}), ("mountaincar_continuous", {"power": float("nan")}),
                      ("acrobot", {"link_moi": 0.0})):
        with pytest.raises(DrilError):
            D.CudaBatchedEnv(kind, 4, env_params=bad)
    syn = D.CudaBatchedEnv("synthetic", 4, obs_dim=5)
    assert syn.env_params() == {}
    from dril_b200 import _lib as L
    lo = np.ones(4, np.float32)
    with pytest.raises(DrilError):                              # the synthetic env has no parameters
        L.check(syn.ctx.lib.dril_env_set_params(syn.h, 1, L.ptr(lo), None))


def test_wrappers_carry_parameters(D):
    rng = np.random.default_rng(10)
    lo, hi = _ranges("mountaincar_continuous", 16, rng)
    env = D.CudaBatchedEnv("mountaincar_continuous", 16, seed=2, env_params=_kw("mountaincar_continuous", lo, hi))
    w = D.NormalizeWrapperEnv(D.ScalingWrapperEnv(D.MonitorWrapperEnv(env)))
    r = w.env_param_ranges()
    np.testing.assert_array_equal(r["power"][0], lo[0])
    np.testing.assert_array_equal(r["gravity"][1], hi[1])
    p = w.env_params()
    assert ((p["power"] >= lo[0]) & (p["power"] <= hi[0])).all()


# ------------------------------------------------------------------------------------------
# learning: CartPole on randomised pole length and mass, evaluated at the corners
# ------------------------------------------------------------------------------------------
def test_cartpole_randomised_holds_the_corners(D):
    n, T = 4096, 128
    env = D.CudaBatchedEnv("cartpole", n, seed=0, monitor_window=100, env_params=dict(length=(0.25, 1.0), masspole=(0.05, 0.2)))
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=[64, 64])
    alg = D.PPO(n_steps=T, batch_size=T * n // 4, epochs=4, learning_rate=1e-3, ent_coef=0.0)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
    best, it = 0.0, 0
    for it in range(150):
        D.train(agent, env, alg, n * T)
        best = max(best, env.monitor_stats()["ep_len_mean"])
        if best >= 499.5:
            break
    print(f"randomised CartPole: best ep_len_mean {best} after {it + 1} iterations")
    assert best >= 499.5, best
    for length in (0.25, 1.0):
        for masspole in (0.05, 0.2):
            ev = D.CudaBatchedEnv("cartpole", 16, max_steps=500, seed=123, monitor_window=100,
                                  env_params=dict(length=length, masspole=masspole))
            res = D.evaluate_agent(agent, ev, n_eval_episodes=16, deterministic=True)
            print(f"length {length} masspole {masspole}: mean return {res['mean_reward']}")
            assert res["mean_reward"] >= 475, (length, masspole, res)
