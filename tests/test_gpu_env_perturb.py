"""Observation noise and action delay on the device: zero noise and zero delay (which run the perturbed kernels) equal the
unperturbed env bit for bit on the fast, cooperative and tcgen05-actor rollouts, compat act!, chunked collection and
dril_evaluate; the frozen fixtures replay bit for bit through compat act! and the fused rollouts; the delay identity through
compat act! and forced-action rollouts; sharding, idempotent observe, mid-run changes and restarts against the oracle
(oracle/env_perturb.py), error codes, and CartPole learned under delay, noise and a 2-frame history."""
import os

import numpy as np
import pytest

from oracle import env_params as EP, env_perturb as PB, envs as OE, policy as OP

pytestmark = pytest.mark.gpu
f32 = np.float32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KINDS = ("cartpole", "pendulum", "mountaincar", "mountaincar_continuous", "acrobot")
D0 = PB.BASE_OBS_DIM
CONT = {"pendulum": 2.0, "mountaincar_continuous": 1.0}   # Box(1) envs: action bound
HISTORY = {False: dict(), True: dict(history_len=3, mask_velocities=True)}


@pytest.fixture(scope="module")
def D():
    import __graft_entry__
    __graft_entry__.build()
    import dril_b200
    return dril_b200


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


def _agent(D, env, kind, T, seed=2, hidden=(64, 64)):
    b = CONT.get(kind)
    spec = (OP.PolicySpec(env.obs_dim, list(hidden), "continuous", 1, act_low=[-b], act_high=[b]) if b else
            OP.PolicySpec(env.obs_dim, list(hidden), "discrete", 2 if kind == "cartpole" else 3, act_start=1))
    flat = (OP.init_params(spec, seed=seed) + np.random.default_rng(seed).normal(size=spec.n_params()).astype(f32) * 0.05).astype(f32)
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=list(hidden))
    alg = D.PPO(n_steps=T, gamma=0.97, gae_lambda=0.9)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
    agent.set_parameters(flat)
    return spec, flat, agent, alg


def _norm(D, norm):
    return D.NormalizeConfig(norm_obs=norm == "full") if norm else None


def _zero(env):
    env.set_obs_noise(0.0)
    env.set_action_delay(np.zeros(env.n_envs, np.int32))


def _rollouts(D, env, kind, T, n, rng_seed, n_roll=2, callbacks=None, forced=True):
    rng = np.random.default_rng(rng_seed)
    _, _, agent, alg = _agent(D, env, kind, T)
    outs = []
    for _ in range(n_roll):
        buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
        fa = _actions(kind, rng, (T, n)) if forced else None
        _, ok = D.collect_rollout(buf, agent, alg, env, callbacks=callbacks, forced_actions=fa)
        assert ok
        outs.append({k: buf.download(k) for k in FIELDS})
        outs[-1]["state"], outs[-1]["steps"] = env.get_state()
        buf.close()
    return outs


FIELDS = ("obs", "actions", "rewards", "values", "logprobs", "boot", "last_values", "flags", "episode_r", "episode_l")
# path: (n, T, max_steps, normalize); gtc: >= 96 envs per SM, the actor on tcgen05 (rollout_gtc.cuh)
PATHS = {"fast": (300, 24, 10, None), "coop": (200, 20, 9, "full"), "gtc": (14208, 4, 3, "ret")}


def _assert_same(a, b, what):
    for r, (x, y) in enumerate(zip(a, b)):
        for k in x:
            assert x[k].tobytes() == y[k].tobytes(), f"{what} rollout {r}: {k}"


# ------------------------------------------------------------------------------------------
# 1. zero perturbation is free
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hist", [False, True])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("path", list(PATHS))
def test_zero_perturbation_rollouts(D, path, kind, hist):
    n, T, ms, norm = PATHS[path]
    lo, hi = _ranges(kind, n, np.random.default_rng(3))
    runs = []
    for zero in (False, True):
        env = D.CudaBatchedEnv(kind, n, max_steps=ms, seed=9, monitor_window=100, normalize=_norm(D, norm),
                               env_params=_kw(kind, lo, hi), **HISTORY[hist])
        if zero:
            _zero(env)
        runs.append(_rollouts(D, env, kind, T, n, 4))
    assert any(((o["flags"] >> 1) & 1).any() for o in runs[0])
    _assert_same(runs[0], runs[1], f"{kind} {path} hist={hist}")


@pytest.mark.parametrize("hist", [False, True])
@pytest.mark.parametrize("kind", KINDS)
def test_zero_perturbation_compat_chunked_evaluate(D, kind, hist):
    n, ms = 97, 11
    lo, hi = _ranges(kind, n, np.random.default_rng(5))

    def make(zero, **kw):
        env = D.CudaBatchedEnv(kind, n, max_steps=ms, seed=7, monitor_window=100, env_params=_kw(kind, lo, hi), **HISTORY[hist], **kw)
        if zero:
            _zero(env)
        return env

    # compat act! under Monitor
    envs = [make(z) for z in (False, True)]
    rng = np.random.default_rng(6)
    for t in range(30):
        a = _actions(kind, rng, (n,))
        o = [e.observe() for e in envs]
        assert o[0].tobytes() == o[1].tobytes()
        s = [e.act(a) for e in envs]
        for x, y in zip(s[0][:3], s[1][:3]):
            assert x.tobytes() == y.tobytes()
        for i, j in zip(s[0][3], s[1][3]):
            assert i.keys() == j.keys() and i.get("episode") == j.get("episode")
            if "terminal_observation" in i:
                assert i["terminal_observation"].tobytes() == j["terminal_observation"].tobytes()

    # chunked collection (training normaliser: the general kernel) == itself unperturbed

    class Step(D.AbstractCallback):
        def on_step(self, loc):
            return True

    runs = [_rollouts(D, make(z, normalize=D.NormalizeConfig()), kind, 8, n, 8, callbacks=[Step()]) for z in (False, True)]
    _assert_same(runs[0], runs[1], f"{kind} chunked hist={hist}")
    # dril_evaluate
    res = []
    for z in (False, True):
        env = make(z)
        _, _, agent, _ = _agent(D, env, kind, 8, seed=5)
        res.append(D.evaluate_agent(agent, env, n_eval_episodes=40, deterministic=True, return_stats=False, chunk_steps=5))
    for x, y in zip(*res):
        assert np.asarray(x).tobytes() == np.asarray(y).tobytes()


# ------------------------------------------------------------------------------------------
# 2. the frozen fixtures
# ------------------------------------------------------------------------------------------
def _fixture_env(D, g, kind, **kw):
    n = g["obs"].shape[1]
    return D.CudaBatchedEnv(kind, n, max_steps=int(g["max_steps"]), seed=int(g["seed"]), env_params=_kw(kind, g["lo"], g["hi"]),
                            history_len=int(g["history_len"]), mask_velocities=bool(g["mask_velocities"]),
                            scaling=bool(g["scaling"]), obs_noise=g["obs_noise"], action_delay=g["action_delay"], **kw)


def _episode_records(rewards, flags):
    """Monitor's records (fp32 running sums) from per-step rewards and done flags"""
    T, n = rewards.shape
    er, el = np.zeros((T, n), f32), np.zeros((T, n), np.int64)
    acc, ln = np.zeros(n, f32), np.zeros(n, np.int64)
    for t in range(T):
        acc = (acc + rewards[t]).astype(f32)
        ln = ln + 1
        d = flags[t] != 0
        er[t][d], el[t][d] = acc[d], ln[d]
        acc[d], ln[d] = 0, 0
    return er, el


@pytest.mark.parametrize("kind", KINDS)
def test_frozen_fixtures(D, kind):
    """compat act! and (Discrete kinds, whose replayed actions need no clamp) the fast and cooperative rollouts against
    tests/golden/orc_<kind>_perturb_replay.npz alone"""
    g = np.load(os.path.join(ROOT, "tests", "golden", f"orc_{kind}_perturb_replay.npz"))
    n, T = g["obs"].shape[1], g["actions"].shape[0]
    flags = g["term"].astype(np.uint8) | (g["trunc"].astype(np.uint8) << 1)
    er, el = _episode_records(g["rewards"], flags)
    env = _fixture_env(D, g, kind, monitor_window=100)
    np.testing.assert_array_equal(env.observe(), g["obs"][0])
    for t, a in enumerate(g["actions"]):
        r, te, tr, infos = env.act(a)
        np.testing.assert_array_equal(r, g["rewards"][t])
        np.testing.assert_array_equal(te, g["term"][t])
        np.testing.assert_array_equal(tr, g["trunc"][t])
        for i in np.nonzero(tr)[0]:
            np.testing.assert_array_equal(infos[i]["terminal_observation"], g["terminal_obs"][t][i])
        for i in np.nonzero(te | tr)[0]:
            assert infos[i]["episode"] == {"r": float(er[t, i]), "l": int(el[t, i])}
        np.testing.assert_array_equal(env.observe(), g["obs"][t + 1])
    if kind in CONT:
        return
    for norm in (None, "ret"):
        env = _fixture_env(D, g, kind, monitor_window=100, normalize=_norm(D, norm))
        _, _, agent, alg = _agent(D, env, kind, T)
        buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
        _, ok = D.collect_rollout(buf, agent, alg, env, forced_actions=g["actions"])
        assert ok
        np.testing.assert_array_equal(buf.download("obs"), g["obs"][:T], err_msg=str(norm))
        np.testing.assert_array_equal(buf.download("flags"), flags, err_msg=str(norm))
        np.testing.assert_array_equal(buf.download("actions").reshape(T, n), g["actions"])   # the chosen actions
        d = flags != 0
        np.testing.assert_array_equal(buf.download("episode_r")[d], er[d])
        np.testing.assert_array_equal(buf.download("episode_l")[d], el[d])
        if norm is None:
            np.testing.assert_array_equal(buf.download("rewards"), g["rewards"])
        buf.close()


# ------------------------------------------------------------------------------------------
# 3. the delay identity: delayed with a_t == undelayed with a_{max(t - d, t0)}
# ------------------------------------------------------------------------------------------
def _ref_actions(acts, flags, delay):
    T, n = acts.shape[:2]
    out = np.empty_like(acts)
    t0 = np.zeros(n, np.int64)
    for t in range(T):
        out[t] = acts[np.maximum(t - delay, t0), np.arange(n)]
        t0 = np.where(flags[t] != 0, t + 1, t0)
    return out


@pytest.mark.parametrize("kind", KINDS)
def test_delay_identity_compat(D, kind):
    n, ms, T = 50, 9, 30
    rng = np.random.default_rng(10)
    lo, hi = _ranges(kind, n, rng)
    delay = np.arange(n) % 5
    acts = _actions(kind, rng, (T, n))
    dl = D.CudaBatchedEnv(kind, n, max_steps=ms, seed=2, env_params=_kw(kind, lo, hi), action_delay=delay)
    un = D.CudaBatchedEnv(kind, n, max_steps=ms, seed=2, env_params=_kw(kind, lo, hi))
    np.testing.assert_array_equal(dl.action_delay(), delay)
    flags = np.zeros((T, n), np.uint8)
    for t in range(T):
        ref = _ref_actions(acts[: t + 1], flags[: t + 1], delay)[t]
        r, te, tr, _ = dl.act(acts[t])
        r2, te2, tr2, _ = un.act(ref)
        flags[t] = te | (tr.astype(np.uint8) << 1)
        for x, y in ((r, r2), (te, te2), (tr, tr2), (dl.observe(), un.observe())):
            np.testing.assert_array_equal(x, y, err_msg=f"step {t}")
    assert (flags != 0).any()


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("path", ["fast", "coop"])
def test_delay_identity_rollouts(D, kind, path):
    n, T, ms, norm = PATHS[path]
    rng = np.random.default_rng(11)
    lo, hi = _ranges(kind, n, rng)
    delay = np.arange(n) % 5
    acts = _actions(kind, rng, (2 * T, n))
    got = {}
    for which in ("delayed", "undelayed"):
        env = D.CudaBatchedEnv(kind, n, max_steps=ms, seed=3, monitor_window=100, normalize=_norm(D, norm),
                               env_params=_kw(kind, lo, hi), action_delay=delay if which == "delayed" else 0)
        _, _, agent, alg = _agent(D, env, kind, T)
        forced = acts if which == "delayed" else _ref_actions(acts, got["delayed"]["flags"], delay)
        outs = []
        for r in range(2):   # the queue continues across rollouts
            buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
            _, ok = D.collect_rollout(buf, agent, alg, env, forced_actions=forced[r * T:(r + 1) * T])
            assert ok
            outs.append({k: buf.download(k) for k in ("obs", "rewards", "flags", "actions", "episode_r", "episode_l")})
            buf.close()
        got[which] = {k: np.concatenate([o[k] for o in outs]) for k in outs[0]}
    assert (got["delayed"]["flags"] != 0).any()
    np.testing.assert_array_equal(got["delayed"]["actions"].reshape(acts.shape), acts)   # the buffer keeps the chosen actions
    for k in ("obs", "rewards", "flags", "episode_r", "episode_l"):
        np.testing.assert_array_equal(got["delayed"][k], got["undelayed"][k], err_msg=k)


# ------------------------------------------------------------------------------------------
# 4. against the oracle: sharding, idempotent observe, mid-run changes, restarts
# ------------------------------------------------------------------------------------------
def _sigma(kind, n, rng):
    s = rng.uniform(0, 0.1, (D0[kind], n)).astype(f32)
    s[:, ::4] = 0
    return s


@pytest.mark.parametrize("kind", KINDS)
def test_oracle_sharding_and_mid_run_changes(D, kind):
    n, ms, T = 64, 10, 36
    rng = np.random.default_rng(12)
    lo, hi = _ranges(kind, n, rng)
    sig, delay = _sigma(kind, n, rng), np.arange(n) % 5
    kw = dict(max_steps=ms, seed=4, monitor_window=100)
    full = D.CudaBatchedEnv(kind, n, env_params=_kw(kind, lo, hi), obs_noise=sig, action_delay=delay, history_len=2, **kw)
    halves = [D.CudaBatchedEnv(kind, n // 2, gid_offset=s.start, env_params=_kw(kind, lo[:, s], hi[:, s]), obs_noise=sig[:, s],
                               action_delay=delay[s], history_len=2, **kw) for s in (slice(0, n // 2), slice(n // 2, n))]
    ob = PB.make(kind, n, sig, delay, 2, seed=4, max_steps=ms, param_ranges=(lo, hi))
    o = OE.ParallelEnv(ob)
    for t in range(T):
        if t == 12:                                   # new deviations: the next observation; new delays: queues restart
            sig, delay = _sigma(kind, n, rng), (np.arange(n) + 2) % 5
            full.set_obs_noise(sig); ob.set_obs_noise(sig)
            full.set_action_delay(delay); ob.set_action_delay(delay)
        if t == 20:
            full.reset(); o.reset()
        if t == 26:                                   # set_state restarts the queue and refills the history
            full.set_state(*full.get_state()); ob.restart_queue(); ob.restart()
        obs = full.observe()
        np.testing.assert_array_equal(obs, full.observe())                # idempotent
        np.testing.assert_array_equal(obs, o.observe(), err_msg=f"step {t}")
        if t < 12:
            np.testing.assert_array_equal(obs, np.concatenate([h.observe() for h in halves]))
        a = _actions(kind, rng, (n,))
        r, te, tr, infos = full.act(a)
        ro, teo, tro, info = o.act(a)
        np.testing.assert_array_equal(r, ro); np.testing.assert_array_equal(te, teo); np.testing.assert_array_equal(tr, tro)
        for i in np.nonzero(tro)[0]:
            np.testing.assert_array_equal(infos[i]["terminal_observation"], info["terminal_observation"][i])
        if t < 12:
            parts = [h.act(a[: n // 2] if i == 0 else a[n // 2:]) for i, h in enumerate(halves)]
            np.testing.assert_array_equal(r, np.concatenate([p[0] for p in parts]))
    # both off: back to the unperturbed kernels, the true state observed
    full.set_obs_noise(None); full.set_action_delay(None)
    st, _ = full.get_state()
    plain = EP.PARAM_BATCHES[kind](n, seed=4)
    plain.state = st.copy()
    k_obs = full.observe()[:, D0[kind]:]
    np.testing.assert_array_equal(k_obs, plain.obs())
    assert full.obs_noise() is None and np.all(full.action_delay() == 0)


def test_noise_statistics_and_true_state(D):
    n = 100_000
    env = D.CudaBatchedEnv("acrobot", n, seed=8)
    clean = env.observe()
    sig = np.linspace(0.05, 0.3, 6, dtype=f32)
    env.set_obs_noise(sig)
    noisy = env.observe()
    z = (noisy.astype(np.float64) - clean) / sig
    assert abs(z.mean()) < 0.01 and abs(z.std() - 1) < 0.01
    st, _ = env.get_state()
    plain = EP.PARAM_BATCHES["acrobot"](n, seed=8)
    np.testing.assert_array_equal(st, plain.state)   # the true state


# ------------------------------------------------------------------------------------------
# 5. error codes
# ------------------------------------------------------------------------------------------
def test_error_codes(D):
    from dril_b200 import _lib as L
    from dril_b200._lib import DrilError
    lib = D.Context.default().lib
    UNSUP, INVALID = 3, 1
    syn = D.CudaBatchedEnv("synthetic", 4, obs_dim=5)
    s = np.zeros((5, 4), f32)
    assert lib.dril_env_set_obs_noise(syn.h, 5, L.ptr(s)) == UNSUP
    assert lib.dril_env_set_action_delay(syn.h, L.ptr(np.zeros(4, np.int32))) == UNSUP
    with pytest.raises(DrilError):
        D.CudaBatchedEnv("synthetic", 4, obs_dim=5, action_delay=1)
    # observe_params, in either order
    a = D.CudaBatchedEnv("cartpole", 8, seed=1, observe_params=True)
    assert lib.dril_env_set_obs_noise(a.h, 4, L.ptr(np.zeros((4, 8), f32))) == UNSUP
    assert lib.dril_env_set_action_delay(a.h, L.ptr(np.ones(8, np.int32))) == UNSUP
    b = D.CudaBatchedEnv("cartpole", 8, seed=1, obs_noise=0.1)
    assert lib.dril_env_set_observe_params(b.h, 1) == UNSUP
    c = D.CudaBatchedEnv("cartpole", 8, seed=1, action_delay=2)
    assert lib.dril_env_set_observe_params(c.h, 1) == UNSUP
    # invalid input
    env = D.CudaBatchedEnv("pendulum", 8, seed=1)
    for bad in (np.full((3, 8), -0.1, f32), np.full((3, 8), np.nan, f32), np.full((3, 8), np.inf, f32)):
        assert lib.dril_env_set_obs_noise(env.h, 3, L.ptr(bad)) == INVALID
    assert lib.dril_env_set_obs_noise(env.h, 2, L.ptr(np.zeros((2, 8), f32))) == INVALID
    for bad in (5, -1):
        d = np.zeros(8, np.int32); d[3] = bad
        assert lib.dril_env_set_action_delay(env.h, L.ptr(d)) == INVALID
    assert env.obs_noise() is None and lib.dril_env_set_obs_noise(env.h, 3, L.ptr(np.zeros((3, 8), f32))) == 0
    # the wrappers carry both options
    env2 = D.CudaBatchedEnv("pendulum", 8, seed=1, obs_noise=[0.1, 0.0, 0.2], action_delay=np.arange(8) % 5)
    w = D.NormalizeWrapperEnv(D.ScalingWrapperEnv(D.MonitorWrapperEnv(env2)))
    np.testing.assert_array_equal(w.obs_noise(), np.repeat(np.array([[0.1], [0.0], [0.2]], f32), 8, axis=1))
    np.testing.assert_array_equal(w.action_delay(), np.arange(8) % 5)


# ------------------------------------------------------------------------------------------
# 6. learning under delay, noise and a 2-frame history
# ------------------------------------------------------------------------------------------
LEARN_ITERS, LEARN_TARGET = 150, 475.0


def test_cartpole_learns_with_delay_noise_and_history(D):
    n, T = 4096, 128
    env = D.CudaBatchedEnv("cartpole", n, seed=0, monitor_window=100, history_len=2, obs_noise=0.01, action_delay=1)
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=[64, 64])
    alg = D.PPO(n_steps=T, batch_size=T * n // 4, epochs=4, learning_rate=1e-3, ent_coef=0.0)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
    best, it = 0.0, 0
    for it in range(LEARN_ITERS):
        D.train(agent, env, alg, n * T)
        best = max(best, env.monitor_stats()["ep_len_mean"])
        if best >= 499.5:
            break
    print(f"CartPole with action_delay 1, obs_noise 0.01, history_len 2: best ep_len_mean {best} after {it + 1} iterations")
    assert best >= LEARN_TARGET, best
