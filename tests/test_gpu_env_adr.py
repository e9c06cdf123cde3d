"""Automatic domain randomisation on the device (csrc/adr.cuh): forced-action rounds through dril_rollout_collect replayed by the
oracle (oracle/env_adr.py driving oracle/env_params.py) on the fast, cooperative and tcgen05-actor rollouts; the iteration and
chunked paths against the collect path; sharding; ADR with nothing moving against plain ranges; turning it off; observed
parameters, history and noise; error codes; and CartPole learning while ADR widens its pole length and mass."""
import ctypes as C

import numpy as np
import pytest

from oracle import env_adr as EA, env_params as EP, envs as OE, policy as OP, ppo as OO

pytestmark = pytest.mark.gpu
f32 = np.float32
KINDS = ("cartpole", "pendulum", "mountaincar", "mountaincar_continuous", "acrobot")
OBS_DIM = {"cartpole": 4, "pendulum": 3, "mountaincar": 2, "mountaincar_continuous": 2, "acrobot": 6}
CONT = {"pendulum": 2.0, "mountaincar_continuous": 1.0}
ADR_IDX = {"cartpole": (3, 2), "pendulum": (1, 2), "mountaincar": (0, 1), "mountaincar_continuous": (0, 1), "acrobot": (0, 2)}
# path: (n, T, max_steps, normalize): the reward-only normaliser keeps the cooperative / tcgen05-actor kernels with raw observations
PATHS = {"fast": (300, 24, 10, False), "coop": (200, 20, 9, True), "gtc": (14208, 4, 3, True)}
P_BOUNDARY = 0.5
ROUNDS = 5


@pytest.fixture(scope="module")
def D():
    import __graft_entry__
    __graft_entry__.build()
    import dril_b200
    return dril_b200


def _spec(kind):
    if kind in CONT:
        b = CONT[kind]
        return OP.PolicySpec(OBS_DIM[kind], [64, 64], "continuous", 1, act_low=[-b], act_high=[b])
    return OP.PolicySpec(OBS_DIM[kind], [64, 64], "discrete", 2 if kind == "cartpole" else 3, act_start=1)


def _actions(kind, rng, shape):
    if kind in CONT:
        return (rng.normal(size=shape + (1,)) * 1.2 * CONT[kind]).astype(f32)
    return rng.integers(1, 3 if kind == "cartpole" else 4, shape)


def adr_params(kind):
    """two parameters around their defaults: initial [d, 1.1 d], limits [0.5 d, 2 d], step 0.1 d"""
    out = []
    for k in ADR_IDX[kind]:
        d = f32(EP.ENV_PARAMS[kind][k][1])
        out.append(EA.AdrParam(k, d, f32(1.1) * d, f32(0.5) * d, f32(2.0) * d, f32(0.1) * d))
    return out


def _kw(kind, params):
    names = [nm for nm, _ in EP.ENV_PARAMS[kind]]
    return {names[q.index]: dict(init=(q.init_lo, q.init_hi), limits=(q.limit_lo, q.limit_hi), step=q.delta) for q in params}


def scenario(kind, path, seed=9):
    """forced actions of every round, the buffer size and the thresholds: from a pilot run of the oracle at the initial ranges,
    thresholds close enough to the mean return that boundaries both widen and narrow.  Where every episode has the same return
    (all truncated at max_steps, e.g. MountainCar and Acrobot under random actions) every full buffer widens instead."""
    n, T, ms, _ = PATHS[path]
    rng = np.random.default_rng(11)
    forced = [_actions(kind, rng, (T, n)) for _ in range(ROUNDS)]
    spec, flat = _spec(kind), OP.init_params(_spec(kind), seed=2)
    params = adr_params(kind)
    ob = EP.PARAM_BATCHES[kind](n, seed=seed, max_steps=ms)
    o = OE.MonitorWrapper(OE.ParallelEnv(ob))
    eo = OO.collect_rollout_timemajor(o, spec, flat, T, forced_actions=forced[0])
    done = eo["term"] | eo["trunc"]
    r = eo["episode_r"][done].astype(np.float64)
    m = max(4, int(0.6 * done.sum() * P_BOUNDARY / (2 * len(params))))
    if (r == r[0]).all():
        return forced, params, m, float(r[0]) - 1.0, float(r[0])
    sd = r.std() / np.sqrt(m)
    t_high = float(r.max()) if (r == r.max()).mean() > 0.5 else float(r.mean() + 0.41 * sd)   # mostly truncated: widen on those
    return forced, params, m, float(r.mean() - 0.37 * sd), t_high


def oracle_rounds(kind, path, seed=9):
    """the oracle replay of `scenario`: per round the oracle buffer, the batch's parameters and state, and the ADR state"""
    n, T, ms, _ = PATHS[path]
    forced, params, m, t_low, t_high = scenario(kind, path, seed)
    spec, flat = _spec(kind), OP.init_params(_spec(kind), seed=2)
    ob = EP.PARAM_BATCHES[kind](n, seed=seed, max_steps=ms)
    o = OE.MonitorWrapper(OE.ParallelEnv(ob))
    adr = EA.Adr(kind, params, P_BOUNDARY, m, t_low, t_high, seed, np.arange(n))
    adr.attach(ob)
    out = [dict(p=ob.p.copy(), lo=adr.lo.copy(), hi=adr.hi.copy())]
    for fa in forced:
        eo = OO.collect_rollout_timemajor(o, spec, flat, T, forced_actions=fa)
        roll = adr.scan(eo["term"] | eo["trunc"], eo["episode_r"], ob.episode)
        adr.update(*roll)
        adr.write_ranges(ob.plo, ob.phi)
        out.append(dict(eo=eo, p=ob.p.copy(), state=ob.state.copy(), lo=adr.lo.copy(), hi=adr.hi.copy(), sums=adr.sums.copy(),
                        counts=adr.counts.copy(), round=adr.round))
    return out, (forced, params, m, t_low, t_high)


def _device_env(D, kind, path, params, m, t_low, t_high, seed=9, **kw):
    n, T, ms, norm = PATHS[path]
    env = D.CudaBatchedEnv(kind, n, max_steps=ms, seed=seed, monitor_window=100,
                           normalize=D.NormalizeConfig(norm_obs=False) if norm else None, **kw)
    env.set_adr(_kw(kind, params), p_boundary=P_BOUNDARY, buffer_size=m, thresholds=(t_low, t_high))
    return env


def _agent(D, env, kind, T):
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=[64, 64])
    alg = D.PPO(n_steps=T, gamma=0.97, gae_lambda=0.9, batch_size=T * env.n_envs // 2, epochs=1)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
    if env.obs_dim == OBS_DIM[kind]:
        agent.set_parameters(OP.init_params(_spec(kind), seed=2))
    return agent, alg


def _params_array(env):
    p = env.env_params()
    return np.stack([p[nm] for nm, _ in EP.ENV_PARAMS[env.kind]])


def _adr_arrays(env):
    s = env.adr_state()
    names = list(s["ranges"])
    lo = np.array([s["ranges"][k][0] for k in names], f32)
    hi = np.array([s["ranges"][k][1] for k in names], f32)
    counts = np.array([c for k in names for c in s["counts"][k]], np.int64)
    return lo, hi, s["sums"], counts, s["round"]


def _check_adr(env, exp, msg):
    lo, hi, sums, counts, rnd = _adr_arrays(env)
    np.testing.assert_array_equal(lo, exp["lo"], err_msg=msg)
    np.testing.assert_array_equal(hi, exp["hi"], err_msg=msg)
    np.testing.assert_array_equal(counts, exp["counts"], err_msg=msg)
    np.testing.assert_allclose(sums, exp["sums"], rtol=1e-12, atol=0, err_msg=msg)
    assert rnd == exp["round"], msg


# ------------------------------------------------------------------------------------------
# replay against the oracle
# ------------------------------------------------------------------------------------------
def _replay(D, env, kind, path, exp, forced, t_low, t_high):
    n, T, _, _ = PATHS[path]
    np.testing.assert_array_equal(_params_array(env), exp[0]["p"])
    agent, alg = _agent(D, env, kind, T)
    buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
    for r, fa in enumerate(forced):
        e = exp[r + 1]
        _, ok = D.collect_rollout(buf, agent, alg, env, forced_actions=fa)
        assert ok
        msg = f"{kind} {path} round {r}"
        f = buf.download("flags")
        te, tr = (f & 1).astype(bool), ((f >> 1) & 1).astype(bool)
        np.testing.assert_array_equal(te, e["eo"]["term"], err_msg=msg)
        np.testing.assert_array_equal(tr, e["eo"]["trunc"], err_msg=msg)
        np.testing.assert_array_equal(buf.download("obs"), e["eo"]["obs"], err_msg=msg)
        done = te | tr
        np.testing.assert_array_equal(buf.download("episode_r")[done], e["eo"]["episode_r"][done], err_msg=msg)
        np.testing.assert_array_equal(_params_array(env), e["p"], err_msg=msg)
        np.testing.assert_array_equal(env.get_state()[0], e["state"], err_msg=msg)
        _check_adr(env, e, msg)
    widened = any((exp[i + 1]["lo"] < exp[i]["lo"]).any() or (exp[i + 1]["hi"] > exp[i]["hi"]).any() for i in range(ROUNDS))
    narrowed = any((exp[i + 1]["lo"] > exp[i]["lo"]).any() or (exp[i + 1]["hi"] < exp[i]["hi"]).any() for i in range(ROUNDS))
    assert widened, "no boundary widened"
    # Where every episode returns the same value (scenario's t_high - t_low == 1: MountainCar and Acrobot under random actions,
    # and CartPole on the tcgen05-actor path, all truncated at max_steps) a full buffer can only widen, so the replay exercises
    # widening alone.  Narrowing is kind-independent code in adr_update_kernel, replayed here on the kinds whose returns vary.
    assert narrowed or t_high - t_low == 1.0, "no boundary narrowed"
    buf.close()


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("path", ["fast", "coop", "gtc"])
def test_replay_vs_oracle(D, kind, path):
    exp, (forced, params, m, t_low, t_high) = oracle_rounds(kind, path)
    env = _device_env(D, kind, path, params, m, t_low, t_high)
    _replay(D, env, kind, path, exp, forced, t_low, t_high)


@pytest.mark.parametrize("kind", ("cartpole", "pendulum", "acrobot"))
def test_replay_adr_in_constructor_with_seed(D, kind):
    """CudaBatchedEnv(..., seed=s, adr=...) turns ADR on under the context's seed and then seeds the env: the boundary envs
    (a function of the seed) and the attribution must follow the new seed, so the run equals the oracle's under seed s"""
    path, seed = "fast", 9
    assert D.Context.default().seed != seed
    n, T, ms, _ = PATHS[path]
    exp, (forced, params, m, t_low, t_high) = oracle_rounds(kind, path, seed=seed)
    env = D.CudaBatchedEnv(kind, n, max_steps=ms, seed=seed, monitor_window=100,
                           adr=dict(params=_kw(kind, params), p_boundary=P_BOUNDARY, buffer_size=m, thresholds=(t_low, t_high)))
    _replay(D, env, kind, path, exp, forced, t_low, t_high)


def test_reconfigure_unpins_the_previous_parameters(D):
    """turning ADR on again first turns the previous configuration off: a parameter that leaves J keeps [lo_j, hi_j] for every
    env, with no boundary env pinned to lo_j or hi_j"""
    kind, path = "cartpole", "fast"
    n = 4000
    params = [EA.AdrParam(3, 0.5, 0.6, 0.2, 1.0, 0.05), EA.AdrParam(2, 0.1, 0.12, 0.05, 0.2, 0.01)]
    env = D.CudaBatchedEnv(kind, n, max_steps=10, seed=3, monitor_window=100)
    env.set_adr(_kw(kind, params), p_boundary=0.5, buffer_size=8, thresholds=(0.0, 1.0))
    p = _params_array(env)[2]
    assert ((p == f32(0.1)) | (p == f32(0.12))).sum() > n // 8          # boundary envs of masspole are pinned
    env.set_adr(_kw(kind, params[:1]), p_boundary=0.5, buffer_size=8, thresholds=(0.0, 1.0))
    assert list(env.adr_state()["ranges"]) == ["length"]
    env.reset()
    p = _params_array(env)[2]
    assert ((p >= f32(0.1)) & (p <= f32(0.12))).all()
    assert ((p == f32(0.1)) | (p == f32(0.12))).sum() <= 2               # uniform draws from [0.1, 0.12]: no pins left
    env.set_adr(None)
    env.reset()
    p = _params_array(env)[3]
    assert ((p >= f32(0.5)) & (p <= f32(0.6))).all() and ((p == f32(0.5)) | (p == f32(0.6))).sum() <= 2


# ------------------------------------------------------------------------------------------
# the iteration path and chunked collection give the collect path's ADR state
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ("cartpole", "pendulum", "acrobot"))
def test_iteration_and_chunked_paths(D, kind):
    from dril_b200 import _lib as L
    from dril_b200.api import AbstractCallback
    hook = type("Hook", (AbstractCallback,), {"on_step": lambda self, loc: True})()
    _, params, m, t_low, t_high = scenario(kind, "fast")
    n, T, _, _ = PATHS["fast"]
    envs = [_device_env(D, kind, "fast", params, m, t_low, t_high) for _ in range(3)]
    agents = [_agent(D, e, kind, T) for e in envs]
    bufs = [D.RolloutBuffer(e.observation_space(), e.action_space(), 0.9, 0.97, T, n) for e in envs]
    lib = agents[0][0].ctx.lib
    for it in range(ROUNDS):
        agent, alg = agents[0]
        h = alg.hyper()
        L.check(lib.dril_ppo_iteration_async(envs[0].h, agent.device.h, bufs[0].h, C.byref(h), 1, alg.batch_size, 5, it))
        st = D.IterStats()
        L.check(lib.dril_iteration_result(agent.device.h, C.byref(st)))
        acts = bufs[0].download("actions")
        forced = acts if kind in CONT else acts[..., 0]
        D.collect_rollout(bufs[1], agents[1][0], agents[1][1], envs[1], forced_actions=forced)
        D.collect_rollout(bufs[2], agents[2][0], agents[2][1], envs[2], callbacks=[hook], forced_actions=forced)
        ref = _adr_arrays(envs[1])
        for e in (envs[0], envs[2]):
            got = _adr_arrays(e)
            for a, b in zip(got, ref):
                np.testing.assert_array_equal(a, b, err_msg=f"{kind} iteration {it}")
        np.testing.assert_array_equal(_params_array(envs[0]), _params_array(envs[1]))
        np.testing.assert_array_equal(_params_array(envs[2]), _params_array(envs[1]))
    assert ref[-1] == ROUNDS
    for b in bufs:
        b.close()


# ------------------------------------------------------------------------------------------
# sharding, nothing moving, turning off, combinations
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ("cartpole", "acrobot"))
def test_sharding_same_assignment(D, kind):
    m = 500
    params = adr_params(kind)
    kw = dict(p_boundary=0.3, buffer_size=8, thresholds=(0.0, 1.0))
    whole = D.CudaBatchedEnv(kind, 2 * m, seed=3, monitor_window=10)
    whole.set_adr(_kw(kind, params), **kw)
    parts = []
    for i in range(2):
        p = D.CudaBatchedEnv(kind, m, seed=3, monitor_window=10, gid_offset=m * i)
        p.set_adr(_kw(kind, params), **kw)
        parts.append(p)
    pw = _params_array(whole)
    np.testing.assert_array_equal(pw, np.concatenate([_params_array(p) for p in parts], axis=1))
    slots = EA.assign(np.arange(2 * m), 0, 3, 0.3, 4)
    q = params[0]
    np.testing.assert_array_equal(pw[q.index][slots == 0], np.full((slots == 0).sum(), q.init_lo, f32))   # pinned low
    np.testing.assert_array_equal(pw[q.index][slots == 1], np.full((slots == 1).sum(), q.init_hi, f32))   # pinned high
    for e in [whole] + parts:
        e.reset()
    np.testing.assert_array_equal(_params_array(whole), np.concatenate([_params_array(p) for p in parts], axis=1))


@pytest.mark.parametrize("kind", KINDS)
def test_nothing_moving_equals_plain_ranges(D, kind):
    """p_boundary = 0 and thresholds nobody reaches: bit-identical to dril_env_set_params with the initial ranges"""
    n, T, ms, _ = PATHS["fast"]
    params = adr_params(kind)
    names = [nm for nm, _ in EP.ENV_PARAMS[kind]]
    a = D.CudaBatchedEnv(kind, n, max_steps=ms, seed=4, monitor_window=100)
    a.set_adr(_kw(kind, params), p_boundary=0.0, buffer_size=1, thresholds=(-1e30, 1e30))
    b = D.CudaBatchedEnv(kind, n, max_steps=ms, seed=4, monitor_window=100,
                         env_params={names[q.index]: (q.init_lo, q.init_hi) for q in params})
    rng = np.random.default_rng(5)
    for r in range(3):
        forced = _actions(kind, rng, (T, n)) if r < 2 else None
        outs = []
        for env in (a, b):
            agent, alg = _agent(D, env, kind, T)
            buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
            D.collect_rollout(buf, agent, alg, env, forced_actions=forced)
            outs.append({k: buf.download(k) for k in ("obs", "actions", "rewards", "values", "flags", "episode_r")})
            buf.close()
        for k in outs[0]:
            np.testing.assert_array_equal(outs[0][k], outs[1][k], err_msg=f"{kind} rollout {r}: {k}")
        np.testing.assert_array_equal(_params_array(a), _params_array(b))
    lo, hi, _, counts, rnd = _adr_arrays(a)
    assert rnd == 3 and counts.sum() == 0


def test_turning_off_keeps_the_ranges(D):
    kind, path = "cartpole", "fast"
    n, T, ms, _ = PATHS[path]
    exp, (forced, params, m, t_low, t_high) = oracle_rounds(kind, path)
    env = _device_env(D, kind, path, params, m, t_low, t_high)
    agent, alg = _agent(D, env, kind, T)
    buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
    for fa in forced:
        D.collect_rollout(buf, agent, alg, env, forced_actions=fa)
    lo, hi = exp[-1]["lo"], exp[-1]["hi"]
    env.set_adr(None)
    assert env.adr_config() is None
    from dril_b200 import _lib as L
    with pytest.raises(L.DrilError):
        L.check(env.ctx.lib.dril_env_get_adr(env.h, None, None, None, None, None))
    for _ in range(3):        # every reset now draws from [lo_j, hi_j]: no pins, no further moves
        D.collect_rollout(buf, agent, alg, env, forced_actions=forced[0])
        p = _params_array(env)
        for i, q in enumerate(params):
            assert ((p[q.index] >= lo[i]) & (p[q.index] <= hi[i])).all()
            assert (p[q.index] > lo[i]).mean() > 0.9 and (p[q.index] < hi[i]).mean() > 0.9
    env.set_env_params(length=0.5)                      # allowed again
    buf.close()


def test_observed_params_history_and_noise(D):
    """ADR only touches the ranges: with forced actions, an env that observes its parameters, or has a history and sensor
    noise, has the plain ADR env's dynamics and ADR state; the observed values show the pinned boundaries"""
    kind, path = "cartpole", "fast"
    n, T, ms, _ = PATHS[path]
    forced, params, m, t_low, t_high = scenario(kind, path)
    envs = [_device_env(D, kind, path, params, m, t_low, t_high),
            _device_env(D, kind, path, params, m, t_low, t_high, observe_params=True),
            _device_env(D, kind, path, params, m, t_low, t_high, history_len=3, obs_noise=0.05)]
    P = len(EP.ENV_PARAMS[kind])
    for r, fa in enumerate(forced[:3]):
        outs = []
        for env in envs:
            agent, alg = _agent(D, env, kind, T)
            buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
            D.collect_rollout(buf, agent, alg, env, forced_actions=fa)
            outs.append({k: buf.download(k) for k in ("obs", "flags", "episode_r")})
            buf.close()
        for o in outs[1:]:
            np.testing.assert_array_equal(o["flags"], outs[0]["flags"])
            np.testing.assert_array_equal(o["episode_r"], outs[0]["episode_r"])
        for env in envs[1:]:
            for a, b in zip(_adr_arrays(env), _adr_arrays(envs[0])):
                np.testing.assert_array_equal(a, b)
            np.testing.assert_array_equal(_params_array(env), _params_array(envs[0]))
        np.testing.assert_array_equal(envs[0].get_state()[0], envs[2].get_state()[0])
    # observed parameters: after a reset every env observes the values it drew from the current round's ranges; the boundary
    # envs observe their pinned boundary exactly
    envs[1].reset()
    obs = envs[1].observe()
    np.testing.assert_array_equal(obs[:, -P:].T, _params_array(envs[1]))
    lo, hi, _, _, rnd = _adr_arrays(envs[1])
    slots = EA.assign(np.arange(n), rnd, 9, P_BOUNDARY, 4)
    for i, q in enumerate(params):
        col = obs[:, OBS_DIM[kind] + q.index]
        assert (slots == 2 * i).any() and (slots == 2 * i + 1).any()
        np.testing.assert_array_equal(col[slots == 2 * i], np.full((slots == 2 * i).sum(), lo[i], f32))
        np.testing.assert_array_equal(col[slots == 2 * i + 1], np.full((slots == 2 * i + 1).sum(), hi[i], f32))
        assert ((col >= lo[i]) & (col <= hi[i])).all()


def test_error_codes(D):
    from dril_b200 import _lib as L
    INVALID, UNSUP = 1, 3
    lib = D.Context.default().lib
    params = adr_params("cartpole")
    arr = (L.AdrParam * 2)(*[L.AdrParam(q.index, q.init_lo, q.init_hi, q.limit_lo, q.limit_hi, q.delta) for q in params])
    syn = D.CudaBatchedEnv("synthetic", 8, obs_dim=3, monitor_window=10)
    assert lib.dril_env_set_adr(syn.h, 2, arr, 0.2, 8, 0.0, 1.0) == UNSUP
    nomon = D.CudaBatchedEnv("cartpole", 8, seed=1)
    assert lib.dril_env_set_adr(nomon.h, 2, arr, 0.2, 8, 0.0, 1.0) == INVALID
    env = D.CudaBatchedEnv("cartpole", 8, seed=1, monitor_window=10)
    assert lib.dril_env_get_adr(env.h, None, None, None, None, None) == INVALID          # off
    for bad in (dict(p=1.5), dict(m=0), dict(tl=2.0), dict(tl=float("nan")), dict(n=0), dict(n=7)):
        assert lib.dril_env_set_adr(env.h, bad.get("n", 2), arr, bad.get("p", 0.2), bad.get("m", 8), bad.get("tl", 0.0), 1.0) == INVALID
    for field, v in (("index", 6), ("limit_lo", 0.0), ("delta", 0.0), ("init_lo", 0.7), ("limit_hi", float("inf"))):
        a = (L.AdrParam * 1)(L.AdrParam(params[0].index, params[0].init_lo, params[0].init_hi, params[0].limit_lo,
                                        params[0].limit_hi, params[0].delta))
        setattr(a[0], field, v)
        assert lib.dril_env_set_adr(env.h, 1, a, 0.2, 8, 0.0, 1.0) == INVALID, field
    dup = (L.AdrParam * 2)(arr[0], arr[0])
    assert lib.dril_env_set_adr(env.h, 2, dup, 0.2, 8, 0.0, 1.0) == INVALID
    grav = (L.AdrParam * 1)(L.AdrParam(0, 9.8, 9.8, 0.0, 12.0, 0.5))                  # gravity may reach 0
    assert lib.dril_env_set_adr(env.h, 1, grav, 0.2, 8, 0.0, 1.0) == 0
    assert lib.dril_env_set_adr(env.h, 2, arr, 0.2, 8, 0.0, 1.0) == 0                   # reconfigure
    lo = np.ones((6, 8), f32)
    assert lib.dril_env_set_params(env.h, 6, L.ptr(lo), None) == INVALID
    assert lib.dril_env_set_params(env.h, 6, None, None) == INVALID
    assert lib.dril_env_set_adr(env.h, 0, None, 0.0, 1, 0.0, 1.0) == 0
    assert lib.dril_env_set_params(env.h, 6, L.ptr(lo), None) == 0


# ------------------------------------------------------------------------------------------
# learning: CartPole while ADR widens the pole length and mass from the default point
# ------------------------------------------------------------------------------------------
# Measured on an NVIDIA B200 at a 1000 W power limit (README): the first boundary moved after 78 iterations, once the policy held
# the pole at the default point; every side had widened by 4 steps after 84 iterations and by 8 (the low sides' limits) after
# 106, and from the first move to iteration 250 ep_len_mean never fell below 333.8.
LEARN_ITERS = 120
LEARN_MIN_STEPS = 4
LEARN_LEN_FLOOR = 200.0


def test_cartpole_learns_while_adr_widens(D):
    n, T = 4096, 128
    adr = dict(params=dict(length=dict(init=(0.5, 0.5), limits=(0.1, 2.0), step=0.05),
                           masspole=dict(init=(0.1, 0.1), limits=(0.02, 0.5), step=0.01)),
               p_boundary=0.2, buffer_size=64, thresholds=(200.0, 450.0))
    env = D.CudaBatchedEnv("cartpole", n, seed=0, monitor_window=100, observe_params=True, adr=adr)
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=[64, 64])
    alg = D.PPO(n_steps=T, batch_size=T * n // 4, epochs=4, learning_rate=1e-3, ent_coef=0.0)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))

    def steps(s):   # boundary moves so far: length low, high, masspole low, high
        (a, b), (c, d) = s["ranges"]["length"], s["ranges"]["masspole"]
        return (round((0.5 - a) / 0.05), round((b - 0.5) / 0.05), round((0.1 - c) / 0.01), round((d - 0.1) / 0.01))

    first, lens = None, []
    for it in range(LEARN_ITERS):
        D.train(agent, env, alg, n * T)
        s = env.adr_state()
        if first is None and max(steps(s)) > 0:
            first = it
        if first is not None:
            lens.append(env.monitor_stats()["ep_len_mean"])
    s = env.adr_state()
    print(f"ADR CartPole: first move after {first} iterations, ranges {s['ranges']}, steps {steps(s)}, "
          f"ep_len_mean since then min {min(lens) if lens else float('nan'):.1f} last {lens[-1] if lens else float('nan'):.1f}")
    assert min(steps(s)) >= LEARN_MIN_STEPS, steps(s)
    assert min(lens) >= LEARN_LEN_FLOOR, min(lens)
