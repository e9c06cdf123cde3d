"""MountainCar, MountainCarContinuous and Acrobot on the device against the oracle: the compat act!/observe path, the fused
rollout on each kernel these envs can take (fast, general cooperative, tcgen05 actor), the tcgen05 loss/grad kernel with a
Discrete(3 | 4) head, one update of Acrobot + NormalizeWrapperEnv, evaluate_agent, and learning on Acrobot."""
import numpy as np
import pytest

from oracle import classic_envs as CE, envs as OE, policy as OP, ppo as OO

pytestmark = pytest.mark.gpu
f32 = np.float32


@pytest.fixture(scope="module")
def D():
    import __graft_entry__
    __graft_entry__.build()
    import dril_b200
    return dril_b200


def _flags(buf):
    f = buf.download("flags")
    return (f & 1).astype(bool), ((f >> 1) & 1).astype(bool)


def _relerr(a, b):
    return np.linalg.norm(a.astype(np.float64) - b) / max(np.linalg.norm(b), 1e-30)


def _batch(kind, n, seed, ms):
    return {"mountaincar": CE.MountainCarBatch, "mountaincar_continuous": CE.MountainCarContinuousBatch,
            "acrobot": CE.AcrobotBatch}[kind](n, seed=seed, max_steps=ms)


def _near_terminal(kind, ob, rng):
    """states that end the episode within a few steps for a third of the envs (random actions rarely reach the goal)"""
    st = ob.state.copy()
    k = np.arange(ob.n) % 3 == 0
    if kind.startswith("mountaincar"):
        st[0, k] = rng.uniform(0.44, 0.5, k.sum())
        st[1, k] = rng.uniform(0.01, 0.07, k.sum())
    else:
        st[0, k] = rng.uniform(2.6, 3.1, k.sum())
        st[1, k] = rng.uniform(-0.3, 0.3, k.sum())
    return st.astype(f32)


# ------------------------------------------------------------------------------------------
# compat path: env.act / env.observe against oracle.envs
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,monitor,norm,scaled", [
    ("mountaincar", False, False, False), ("mountaincar", True, True, False),
    ("mountaincar_continuous", False, False, False), ("mountaincar_continuous", True, True, False),
    ("mountaincar_continuous", True, False, True),
    ("acrobot", False, False, False), ("acrobot", True, True, False)])
def test_env_replay_new_kinds(D, kind, monitor, norm, scaled):
    n, steps, ms = 301, 70, 25
    rng = np.random.default_rng(1)
    ob = _batch(kind, n, 5, ms)
    env = D.CudaBatchedEnv(kind, n, max_steps=ms, seed=5, monitor_window=100 if monitor else 0,
                           normalize=D.NormalizeConfig() if norm else None, scaling=scaled)
    st = _near_terminal(kind, ob, rng)
    env.set_state(st)
    ob.state = st.copy()
    o = OE.ScalingBatch(ob, CE.MOUNTAINCAR_OBS_LOW, CE.MOUNTAINCAR_OBS_HIGH) if scaled else ob
    oenv = OE.ParallelEnv(o)
    if monitor:
        oenv = OE.MonitorWrapper(oenv)
    if norm:
        oenv = OE.NormalizeWrapper(oenv, ob.obs_dim)
    if kind == "mountaincar_continuous":
        act = lambda: rng.uniform(-1.0 if scaled else -1.5, 1.0 if scaled else 1.5, (n, 1)).astype(f32)
    else:
        act = lambda: rng.integers(1, 4, n)
    # Acrobot's cos(theta2) column starts nearly constant: its running variance is tiny, and the last bits in which the device's
    # double moment sums and NumPy's fp32 variance differ show up as ~5e-5 in the normalised column (raw observations: bit-exact)
    tol = dict(rtol=3e-5, atol=3e-4 if kind == "acrobot" else 3e-5) if norm else dict(rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(env.observe(), oenv.observe(), **tol)
    n_term = n_trunc = 0
    for _ in range(steps):
        a = act()
        r, te, tr, infos = env.act(a)
        ro, teo, tro, info = oenv.act(a)
        np.testing.assert_array_equal(te, teo)
        np.testing.assert_array_equal(tr, tro)
        np.testing.assert_allclose(r, ro, rtol=3e-5 if norm else 1e-6, atol=0)
        oo, ooo = env.observe(), oenv.observe()
        if norm:
            np.testing.assert_allclose(oo, ooo, **tol)
            np.testing.assert_array_equal(env.get_original()[0], oenv.old_obs)
        else:
            np.testing.assert_array_equal(oo, ooo)
        for i in np.nonzero(tro)[0]:
            np.testing.assert_allclose(infos[i]["terminal_observation"], info["terminal_observation"][i], **tol)
        assert all(("terminal_observation" in infos[i]) == bool(tro[i]) for i in range(n))
        if monitor:
            for i in np.nonzero(teo | tro)[0]:
                assert abs(infos[i]["episode"]["r"] - info["episode_r"][i]) <= 1e-5 * max(1.0, abs(info["episode_r"][i]))
                assert infos[i]["episode"]["l"] == info["episode_l"][i]
        n_term += teo.sum(); n_trunc += tro.sum()
    assert n_term > 0 and n_trunc > 0
    st_dev, steps_dev = env.get_state()
    np.testing.assert_array_equal(steps_dev, ob.steps)
    assert st_dev.shape == (ob.state.shape[0], n)


def test_spaces_and_defaults(D):
    mc = D.CudaBatchedEnv("mountaincar", 4)
    assert mc.max_steps == 200 and mc.obs_dim == 2
    assert isinstance(mc.action_space(), D.Discrete) and mc.action_space().n == 3 and mc.action_space().start == 1
    np.testing.assert_array_equal(mc.observation_space().low, CE.MOUNTAINCAR_OBS_LOW)
    mcc = D.CudaBatchedEnv("mountaincar_continuous", 4)
    assert mcc.max_steps == 999 and isinstance(mcc.action_space(), D.Box)
    np.testing.assert_array_equal(mcc.action_space().high, [1.0])
    ac = D.MultiThreadedParallelEnv("acrobot", 4, act_start=0)
    assert ac.max_steps == 500 and ac.obs_dim == 6 and ac.action_space().start == 0
    np.testing.assert_array_equal(ac.observation_space().high, CE.ACROBOT_OBS_HIGH)
    assert ac.observe().shape == (4, 6) and ac.get_state()[0].shape == (4, 4)
    sc = D.ScalingWrapperEnv(D.MonitorWrapperEnv(D.MultiThreadedParallelEnv("mountaincar_continuous", 4)))
    np.testing.assert_array_equal(sc.orig_observation_space.high, CE.MOUNTAINCAR_OBS_HIGH)
    with pytest.raises(Exception):
        D.ScalingWrapperEnv(D.MultiThreadedParallelEnv("acrobot", 4))       # Discrete actions: not Box/Box
    env = D.CudaBatchedEnv("acrobot", 8)
    layer = D.ActorCriticLayer(env.observation_space(), D.Discrete(2, 1), hidden_dims=[64, 64])
    alg = D.PPO(n_steps=4)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
    buf = D.RolloutBuffer(env.observation_space(), D.Discrete(2, 1), 0.95, 0.99, 4, 8)
    with pytest.raises(Exception):                                         # Acrobot needs Discrete(3)
        D.collect_rollout(buf, agent, alg, env)


# ------------------------------------------------------------------------------------------
# fused rollout vs the oracle rollout (replayed and sampled actions)
# ------------------------------------------------------------------------------------------
def _spec(kind, hidden, act_start=1):
    if kind == "mountaincar_continuous":
        return OP.PolicySpec(2, hidden, "continuous", 1, act_low=[-1], act_high=[1])
    return OP.PolicySpec(2 if kind == "mountaincar" else 6, hidden, "discrete", 3, act_start=act_start)


@pytest.mark.parametrize("kind,n,T,ms,monitor,norm,scaled", [
    ("mountaincar", 300, 24, 10, True, False, False),             # fast kernel
    ("mountaincar_continuous", 300, 24, 10, True, False, False),
    ("mountaincar_continuous", 257, 20, 9, True, False, True),
    ("acrobot", 333, 24, 11, True, False, False),
    ("acrobot", 4096, 12, 7, False, False, False),
    ("mountaincar", 200, 20, 9, True, True, False),               # general cooperative kernel (training normaliser)
    ("mountaincar_continuous", 200, 20, 9, True, True, True),
    ("acrobot", 500, 20, 9, True, True, False),
    # >= 96 envs per SM: the actor on tcgen05 (rollout_gtc.cuh).  The training normaliser scales rewards only: normalised
    # observations of columns that start nearly constant (Acrobot's cosines, MountainCar's velocity) would compare the oracle's
    # fp32 sums over 14 208 envs rather than the kernel
    ("acrobot", 14208, 4, 3, True, "ret", False),
    ("mountaincar", 14208, 4, 3, False, "ret", False)])
def test_fused_rollout_vs_oracle(D, kind, n, T, ms, monitor, norm, scaled):
    spec = _spec(kind, [64, 64])
    rng = np.random.default_rng(4)
    flat = (OP.init_params(spec, seed=2) + rng.normal(size=spec.n_params()).astype(f32) * 0.05).astype(f32)
    cont = kind == "mountaincar_continuous"
    for opts in ({}, {"tc_actor": 0}, {"defer_critic": 0}):
        if opts and n < 14208:
            continue
        for k, v in opts.items():
            D.set_option(k, v)
        try:
            env = D.CudaBatchedEnv(kind, n, max_steps=ms, seed=9, monitor_window=100 if monitor else 0,
                                   normalize=D.NormalizeConfig(norm_obs=norm != "ret") if norm else None, scaling=scaled)
            ob = _batch(kind, n, 9, ms)
            o = OE.ParallelEnv(OE.ScalingBatch(ob, CE.MOUNTAINCAR_OBS_LOW, CE.MOUNTAINCAR_OBS_HIGH) if scaled else ob)
            if monitor:
                o = OE.MonitorWrapper(o)
            if norm:
                o = OE.NormalizeWrapper(o, spec.obs_dim, norm_obs=norm != "ret")
            layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=spec.hidden)
            alg = D.PPO(n_steps=T, gamma=0.97, gae_lambda=0.9)
            agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
            agent.set_parameters(flat)
            assert agent.device.update_path() == "tensor"
            # (Acrobot + training normaliser: see test_env_replay_new_kinds for the nearly constant cos(theta2) column)
            tol = dict(rtol=3e-5, atol=3e-4 if kind == "acrobot" else 3e-5) if norm else dict(rtol=1e-5, atol=1e-5)
            for rollout in range(2):       # 0: replayed actions, 1: sampled on the device, then replayed through the oracle
                forced = (rng.normal(size=(T, n, 1)).astype(f32) * 1.2 if cont else rng.integers(1, 4, (T, n))) if rollout == 0 else None
                buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
                _, ok = D.collect_rollout(buf, agent, alg, env, forced_actions=forced)
                assert ok
                acts = buf.download("actions")
                replay = forced if forced is not None else (acts if cont else acts[..., 0])
                if forced is None and not cont:
                    assert set(np.unique(replay)) <= {1, 2, 3} and len(np.unique(replay)) == 3
                eo = OO.collect_rollout_timemajor(o, spec, flat, T, forced_actions=replay)
                te, tr = _flags(buf)
                np.testing.assert_array_equal(te, eo["term"])
                np.testing.assert_array_equal(tr, eo["trunc"])
                np.testing.assert_allclose(buf.download("obs"), eo["obs"], **(tol if norm == True else dict(rtol=0, atol=0)))
                np.testing.assert_allclose(buf.download("rewards"), eo["rewards"], **(tol if norm else dict(rtol=1e-6, atol=0)))
                np.testing.assert_allclose(buf.download("values"), eo["values"], **tol)
                np.testing.assert_allclose(buf.download("logprobs"), eo["logprobs"], rtol=1e-4, atol=1e-4)
                np.testing.assert_allclose(buf.download("last_values"), eo["last_values"], **tol)
                np.testing.assert_allclose(np.where(tr, buf.download("boot"), 0), eo["boot"], **tol)
                assert tr.any()
                if monitor:
                    done = te | tr
                    np.testing.assert_allclose(buf.download("episode_r")[done], eo["episode_r"][done], rtol=1e-5)
                    np.testing.assert_array_equal(buf.download("episode_l")[done], eo["episode_l"][done])
                buf.close()
            env.close()
        finally:
            for k in opts:
                D.set_option(k, 1)


# ------------------------------------------------------------------------------------------
# tcgen05 loss/grad kernel with a Discrete(3 | 4) head
# ------------------------------------------------------------------------------------------
def _device_policy(D, spec, flat):
    p = D.DevicePolicy(D.Context.default(), spec.obs_dim, spec.hidden, D.Discrete(spec.act_n, spec.act_start))
    p.set_params(flat)
    return p


def _minibatch(spec, flat, B, rng):
    obs = rng.normal(size=(B, spec.obs_dim)).astype(f32)
    actions = rng.integers(spec.act_start, spec.act_start + spec.act_n, (B, 1))
    v0, lp0, _ = OP.evaluate_actions(spec, flat, obs, actions)
    old_lp = (lp0 + rng.normal(size=B).astype(f32) * 0.2).astype(f32)
    old_v = (v0 + rng.normal(size=B).astype(f32) * 0.3).astype(f32)
    return obs, actions, rng.normal(size=B).astype(f32), rng.normal(size=B).astype(f32), old_lp, old_v


@pytest.mark.parametrize("obs_dim,hidden,n_act", [(6, [64, 64], 3), (2, [64, 64], 4), (6, [128, 128, 64], 3), (2, [128, 128, 64], 4)])
def test_ftg_discrete_head_vs_oracle(D, obs_dim, hidden, n_act):
    """update_ftg.cuh with three or four output columns, on its default path (no option set): loss, statistics and gradients on
    ragged tile counts, many tiles per CTA, large return scales and both loss configurations."""
    spec = OP.PolicySpec(obs_dim, hidden, "discrete", n_act, act_start=1)
    rng = np.random.default_rng(5)
    flat = (OP.init_params(spec, seed=4) + rng.normal(size=spec.n_params()).astype(f32) * 0.05).astype(f32)
    p = _device_policy(D, spec, flat)
    assert p.update_path() == "tensor"
    for B, scale in ((1, 1.0), (63, 1.0), (64, 1.0), (200, 1.0), (1000, 3e4), (148 * 64 * 2 + 17, 1.0)):
        obs, actions, adv, ret, old_lp, old_v = _minibatch(spec, flat, B, rng)
        ret = (ret * scale).astype(f32)
        old_v = (old_v * scale).astype(f32)
        for alg in (D.PPO(ent_coef=0.01, clip_range_vf=0.3 * scale), D.PPO(ent_coef=0.0, normalize_advantage=False, vf_coef=0.7)):
            if B == 1 and alg.normalize_advantage:
                continue
            cfg = OO.PPOConfig(ent_coef=alg.ent_coef, clip_range_vf=alg.clip_range_vf, normalize_advantage=alg.normalize_advantage,
                               vf_coef=alg.vf_coef)
            loss, stats, g = p.loss_grad(obs, actions, adv, ret, old_lp, old_v, alg.hyper())
            eloss, estats, eg = OO.ppo_loss_and_grads(spec, flat, obs, actions, adv, ret, old_lp, old_v, cfg)
            assert abs(loss - eloss) <= 1e-4 * max(1.0, abs(eloss)), (B, loss, eloss)
            for k in estats:
                assert abs(stats[k] - estats[k]) <= 1e-4 * max(1.0, abs(estats[k])), (B, k, stats[k], estats[k])
            assert _relerr(g, eg) < 1e-4, (B, scale, _relerr(g, eg))
    p.close()


def test_acrobot_normalized_update_vs_oracle(D):
    """One update of Acrobot + NormalizeWrapperEnv through the default path (deferred critic, ftg kernel, fused tail) against
    oracle.ppo.ppo_update on the same buffer and the same minibatches."""
    import ctypes as C
    from dril_b200 import _lib as L
    n, T = 1024, 32
    env = D.CudaBatchedEnv("acrobot", n, seed=5, normalize=D.NormalizeConfig())
    spec = _spec("acrobot", [64, 64])
    flat = OP.init_params(spec, seed=2)
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=spec.hidden)
    alg = D.PPO(n_steps=T, batch_size=T * n // 4, epochs=2, ent_coef=0.01)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
    agent.set_parameters(flat)
    assert agent.device.update_path() == "tensor"
    buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
    D.collect_rollout(buf, agent, alg, env)
    ob = {k: buf.download(k) for k in ("obs", "actions", "rewards", "values", "logprobs", "advantages", "returns")}
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


def test_evaluate_agent_mountaincar_vs_oracle_loop(D):
    n = 37
    spec = _spec("mountaincar", [64, 64])
    flat = OP.init_params(spec, seed=5)
    env = D.CudaBatchedEnv("mountaincar", n, max_steps=60, seed=9, monitor_window=100)
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=[64, 64])
    agent = D.Agent(layer, D.PPO(), rng=np.random.default_rng(0))
    agent.set_parameters(flat)
    n_eval = 50
    er, el = D.evaluate_agent(agent, env, n_eval_episodes=n_eval, deterministic=True, return_stats=False, chunk_steps=7)
    o = OE.MonitorWrapper(OE.ParallelEnv(CE.MountainCarBatch(n, seed=9, max_steps=60)))
    o.reset()
    obs = o.observe()
    exp_r, exp_l = [], []
    while len(exp_r) < n_eval:
        a, _, _ = OP.forward(spec, flat, obs, deterministic=True)
        r, term, trunc, infos = o.act(a)
        obs = o.observe()
        for i in range(n):
            if (term[i] or trunc[i]) and len(exp_r) < n_eval:
                exp_r.append(infos["episode_r"][i]); exp_l.append(int(infos["episode_l"][i]))
    np.testing.assert_array_equal(el, np.asarray(exp_l))
    np.testing.assert_allclose(er, np.asarray(exp_r, np.float32), rtol=1e-6)


# ------------------------------------------------------------------------------------------
# learning
# ------------------------------------------------------------------------------------------
# set from a B200 run of this test (1000 W): ep_rew_mean -143 after 9 iterations, -121 after 10, about -92 after 20
ACROBOT_ITERS = 20
ACROBOT_TARGET = -130.0


def test_acrobot_learns(D):
    """PPO with a [64, 64] policy on Acrobot: a random policy scores about -500 (most episodes hit the 500-step limit)."""
    def run():
        n, T = 4096, 128
        env = D.CudaBatchedEnv("acrobot", n, seed=0, monitor_window=100)
        layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=[64, 64])
        alg = D.PPO(n_steps=T, batch_size=T * n // 4, epochs=4, learning_rate=1e-3, ent_coef=0.0)
        agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
        assert agent.device.update_path() == "tensor"
        curve = []
        for _ in range(ACROBOT_ITERS):
            D.train(agent, env, alg, n * T)
            curve.append(env.monitor_stats()["ep_rew_mean"])
        return agent.device.get_params(), curve
    p1, curve = run()
    print("acrobot ep_rew_mean per iteration:", [round(float(c), 1) for c in curve])
    assert np.nanmax(curve) >= ACROBOT_TARGET, curve      # NaN until the first episodes end
    p2, curve2 = run()
    np.testing.assert_array_equal(p1, p2)
