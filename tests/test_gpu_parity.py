"""GPU parity tests: the CUDA path (through the C ABI) against the oracle on the same seeded
inputs. north_star checks: (a) replayed actions -> bit-exact flags, obs <= 1e-6 rel;
(b) GAE <= 1e-5; (c) PPO loss and gradients <= 1e-4 rel; (d) CartPole reaches return 500
(tests/test_gpu_train.py)."""
import numpy as np
import pytest

from oracle import envs as OE, philox as OPH, policy as OP, ppo as OO

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


# ------------------------------------------------------------------------------------------
# (a) env replay through the compat act!/observe path
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,n,steps,max_steps", [("cartpole", 300, 120, 40), ("pendulum", 257, 90, 30),
                                                     ("synthetic", 130, 60, 25), ("cartpole", 1, 30, 500),
                                                     ("pendulum_scaled", 200, 70, 30)])
def test_env_replay_bit_exact_flags(D, kind, n, steps, max_steps):
    rng = np.random.default_rng(0)
    if kind == "cartpole":
        ob = OE.CartPoleBatch(n, seed=5, max_steps=max_steps)
        env = D.CudaBatchedEnv("cartpole", n, max_steps=max_steps, seed=5)
        act = lambda: rng.integers(1, 3, n)
    elif kind == "pendulum":
        ob = OE.PendulumBatch(n, seed=5, max_steps=max_steps)
        env = D.CudaBatchedEnv("pendulum", n, max_steps=max_steps, seed=5)
        act = lambda: rng.uniform(-2.5, 2.5, (n, 1)).astype(f32)
    elif kind == "pendulum_scaled":      # ScalingWrapperEnv (scalingWrapperEnv.jl:94-115) through observe / act!
        ob = OE.ScalingBatch(OE.PendulumBatch(n, seed=5, max_steps=max_steps), OE.PENDULUM_OBS_LOW, OE.PENDULUM_OBS_HIGH)
        env = D.ScalingWrapperEnv(D.MultiThreadedParallelEnv("pendulum", n, max_steps=max_steps))
        env.seed(5); env.reset()
        act = lambda: rng.uniform(-1.0, 1.0, (n, 1)).astype(f32)
    else:
        ob = OE.SyntheticBatch(n, 10, seed=5, max_steps=max_steps)
        env = D.CudaBatchedEnv("synthetic", n, obs_dim=10, max_steps=max_steps, seed=5)
        act = lambda: rng.integers(1, 3, n)
    oenv = OE.ParallelEnv(ob)
    np.testing.assert_array_equal(env.observe(), oenv.observe())
    n_term = n_trunc = 0
    for _ in range(steps):
        a = act()
        r, te, tr, infos = env.act(a)
        ro, teo, tro, info = oenv.act(a)
        np.testing.assert_array_equal(te, teo)
        np.testing.assert_array_equal(tr, tro)
        np.testing.assert_allclose(r, ro, rtol=1e-6, atol=0)
        o, oo = env.observe(), oenv.observe()
        np.testing.assert_allclose(o, oo, rtol=1e-6, atol=1e-7)
        np.testing.assert_array_equal(o, oo)       # in practice bit-exact
        for i in np.nonzero(tro)[0]:
            np.testing.assert_allclose(infos[i]["terminal_observation"], info["terminal_observation"][i], rtol=1e-6)
        assert all(("terminal_observation" in infos[i]) == bool(tro[i]) for i in range(n))
        n_term += teo.sum(); n_trunc += tro.sum()
    assert n == 1 or (n_trunc > 0 and (kind.startswith("pendulum") or n_term > 0))
    st, steps_dev = env.get_state()
    np.testing.assert_array_equal(steps_dev, ob.steps)


def test_env_seeding_and_sharding(D):
    a = D.CudaBatchedEnv("cartpole", 64, seed=11).observe()
    b = D.CudaBatchedEnv("cartpole", 64, seed=11).observe()
    c = D.CudaBatchedEnv("cartpole", 64, seed=12).observe()
    assert (a == b).all() and not (a == c).all()
    d = D.CudaBatchedEnv("cartpole", 32, seed=11, gid_offset=32).observe()
    np.testing.assert_array_equal(d, a[32:])


def test_normalize_monitor_compat_path(D):
    """NormalizeWrapperEnv(MonitorWrapperEnv(parallel env)) step by step vs the oracle."""
    n, ms = 96, 17
    env = D.CudaBatchedEnv("pendulum", n, max_steps=ms, seed=2, monitor_window=100, normalize=D.NormalizeConfig())
    oenv = OE.NormalizeWrapper(OE.MonitorWrapper(OE.ParallelEnv(OE.PendulumBatch(n, seed=2, max_steps=ms))), 3)
    rng = np.random.default_rng(1)
    for t in range(40):
        o, oo = env.observe(), oenv.observe()
        np.testing.assert_allclose(o, oo, rtol=2e-5, atol=2e-5)
        a = rng.uniform(-2, 2, (n, 1)).astype(f32)
        r, te, tr, infos = env.act(a)
        ro, teo, tro, info = oenv.act(a)
        np.testing.assert_array_equal(tr, tro)
        np.testing.assert_allclose(r, ro, rtol=2e-5, atol=2e-5)
        raw_o, raw_r = env.get_original()
        np.testing.assert_allclose(raw_r, oenv.old_rewards, rtol=1e-6)
        for i in np.nonzero(tro)[0]:
            np.testing.assert_allclose(infos[i]["terminal_observation"], info["terminal_observation"][i], rtol=2e-5, atol=2e-5)
            assert abs(infos[i]["episode"]["r"] - info["episode_r"][i]) <= 1e-4 * abs(info["episode_r"][i])
            assert infos[i]["episode"]["l"] == info["episode_l"][i]
    s = env.norm_stats()
    assert s["obs_count"] == oenv.obs_rms.count and s["ret_count"] == oenv.ret_rms.count
    np.testing.assert_allclose(s["obs_mean"], oenv.obs_rms.mean, rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(s["obs_var"], oenv.obs_rms.var, rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(s["ret_var"], oenv.ret_rms.var, rtol=1e-5)
    ms_ = env.monitor_stats()
    exp_r, exp_l = oenv.log_stats()
    assert ms_["n_in_window"] == len(oenv.env.returns)
    assert abs(ms_["ep_rew_mean"] - exp_r) <= 1e-4 * abs(exp_r) and abs(ms_["ep_len_mean"] - exp_l) < 1e-4
    # eval mode freezes statistics (test/test_normalize_wrapper.jl:281-324)
    env.set_training(False); oenv.training = False
    env.observe(); oenv.observe()
    assert env.norm_stats()["obs_count"] == s["obs_count"]


# ------------------------------------------------------------------------------------------
# (b) GAE
# ------------------------------------------------------------------------------------------
def test_gae_closed_form(D):
    """test/test_gae.jl:1-71 through dril_gae_raw."""
    r = np.array([0] * 7 + [1], f32)[:, None]
    v = np.full((8, 1), 0.5, f32)
    term = np.zeros((8, 1), bool); term[-1] = True
    adv, ret = D.gae_raw(r, v, term, np.zeros((8, 1), bool), np.zeros((8, 1), f32), np.zeros(1, f32), 0.99, 0.95)
    gl = 0.99 * 0.95
    closed = np.array([-0.005 * ((1 - gl ** (7 - i)) / (1 - gl)) + gl ** (7 - i) * 0.5 for i in range(7)] + [0.5])
    np.testing.assert_allclose(adv[:, 0], closed, atol=1e-5)
    np.testing.assert_allclose(ret[:, 0], closed + 0.5, atol=1e-5)


@pytest.mark.parametrize("T,N", [(1, 1), (7, 3), (128, 513), (33, 2000)])
def test_gae_random_vs_oracle(D, T, N):
    rng = np.random.default_rng(T * 1000 + N)
    r = rng.normal(size=(T, N)).astype(f32)
    v = rng.normal(size=(T, N)).astype(f32)
    term = rng.random((T, N)) < 0.05
    trunc = rng.random((T, N)) < 0.05
    boot = np.where(trunc, rng.normal(size=(T, N)), 0).astype(f32)
    last = rng.normal(size=N).astype(f32)
    for gamma, lam in ((0.99, 0.95), (1.0, 1.0), (0.9, 0.0)):
        adv, ret = D.gae_raw(r, v, term, trunc, boot, last, gamma, lam)
        ea, er = OO.gae_timemajor(r, v, term, trunc, boot, last, gamma, lam)
        np.testing.assert_allclose(adv, ea, rtol=1e-5, atol=1e-5)
        np.testing.assert_allclose(ret, er, rtol=1e-5, atol=1e-5)
        np.testing.assert_array_equal(adv, ea)   # same op order: bit-exact in practice


# ------------------------------------------------------------------------------------------
# layer application
# ------------------------------------------------------------------------------------------
SPECS = {
    "cartpole": lambda: OP.PolicySpec(4, [64, 64], "discrete", 2, act_start=1),
    "pendulum": lambda: OP.PolicySpec(3, [128, 128, 64], "continuous", 1, act_low=[-2], act_high=[2]),
    "odd": lambda: OP.PolicySpec(10, [24, 12], "discrete", 5, act_start=-2),
    "box3": lambda: OP.PolicySpec(7, [32], "continuous", 3, act_low=[-1, -1, -1], act_high=[1, 1, 1]),
    "nohidden": lambda: OP.PolicySpec(5, [], "continuous", 1, act_low=[-1], act_high=[1]),
}


def _device_policy(D, spec, flat):
    space = D.Discrete(spec.act_n, spec.act_start) if spec.act_kind == "discrete" else D.Box(spec.act_low, spec.act_high)
    p = D.DevicePolicy(D.Context.default(), spec.obs_dim, spec.hidden, space)
    assert p.n_params == spec.n_params()
    p.set_params(flat)
    np.testing.assert_array_equal(p.get_params(), flat)
    return p


@pytest.mark.parametrize("name", list(SPECS))
@pytest.mark.parametrize("B", [1, 77, 1000])
def test_policy_forward_evaluate(D, name, B):
    spec = SPECS[name]()
    rng = np.random.default_rng(3)
    flat = (OP.init_params(spec, seed=1) + rng.normal(size=spec.n_params()).astype(f32) * 0.1).astype(f32)
    p = _device_policy(D, spec, flat)
    obs = rng.normal(size=(B, spec.obs_dim)).astype(f32)
    p.seed(1234, 7)
    a, v, lp = p.forward(obs)
    ea, ev, elp = OP.forward(spec, flat, obs, np.arange(B), 7, 1234)
    np.testing.assert_allclose(v, ev, rtol=1e-5, atol=1e-5)
    if spec.act_kind == "discrete":
        assert a.dtype == np.int64 and a.min() >= spec.act_start and a.max() < spec.act_start + spec.act_n
        # actions follow the same Philox inverse-CDF; allow flips only where u sits on a cumsum boundary
        probs = OP.softmax(OP.mlp_forward(OP.unflatten(spec, flat)["actor"], obs))
        u = OPH.sample_uniform64(np.arange(B), 7, 1234)
        margin = np.abs(np.cumsum(probs, axis=1) - u[:, None]).min(axis=1)
        assert ((a == ea) | (margin < 1e-5)).all()
        same = a == ea
        np.testing.assert_allclose(lp[same], elp[same], rtol=1e-5, atol=1e-5)
    else:
        np.testing.assert_allclose(a, ea, rtol=1e-5, atol=2e-6)
        np.testing.assert_allclose(lp, elp, rtol=1e-4, atol=1e-4)
    # evaluate_actions on the sampled actions reproduces forward (test/test_policies.jl:101-146)
    v2, lp2, ent = p.evaluate(obs, a)
    np.testing.assert_allclose(v2, v, atol=1e-6)
    np.testing.assert_allclose(lp2, lp, atol=1e-5)
    ov, olp, oent = OP.evaluate_actions(spec, flat, obs, a)
    np.testing.assert_allclose(lp2, olp, rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(ent, oent, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(p.predict_values(obs), ev, rtol=1e-5, atol=1e-5)
    # deterministic = mode
    ad, _, _ = p.forward(obs, deterministic=True)
    ed, _, _ = OP.forward(spec, flat, obs, deterministic=True)
    if spec.act_kind == "discrete":
        assert (ad == ed).mean() > 0.995
    else:
        np.testing.assert_allclose(ad, ed, rtol=1e-5, atol=1e-5)


# ------------------------------------------------------------------------------------------
# fused rollout vs oracle (replayed actions)
# ------------------------------------------------------------------------------------------
def _mk(D, kind, n, seed, ms, monitor, norm):
    if kind == "cartpole":
        env = D.CudaBatchedEnv("cartpole", n, max_steps=ms, seed=seed, monitor_window=100 if monitor else 0,
                               normalize=D.NormalizeConfig() if norm else None)
        o = OE.ParallelEnv(OE.CartPoleBatch(n, seed=seed, max_steps=ms)); spec = SPECS["cartpole"]()
    elif kind == "pendulum_scaled":
        # ScalingWrapperEnv around every Pendulum env (scalingWrapperEnv.jl): obs and actions in [-1, 1], below Monitor / Normalize
        env = D.CudaBatchedEnv("pendulum", n, max_steps=ms, seed=seed, monitor_window=100 if monitor else 0,
                               normalize=D.NormalizeConfig() if norm else None, scaling=True)
        assert np.array_equal(env.observation_space().low, -np.ones(3, f32)) and np.array_equal(env.action_space().high, np.ones(1, f32))
        assert np.array_equal(env.orig_action_space.low, [-2.0])
        o = OE.ParallelEnv(OE.ScalingBatch(OE.PendulumBatch(n, seed=seed, max_steps=ms), OE.PENDULUM_OBS_LOW, OE.PENDULUM_OBS_HIGH))
        spec = OP.PolicySpec(3, [64, 32], "continuous", 1, act_low=[-1], act_high=[1])
    else:
        env = D.CudaBatchedEnv("pendulum", n, max_steps=ms, seed=seed, monitor_window=100 if monitor else 0,
                               normalize=D.NormalizeConfig() if norm else None)
        o = OE.ParallelEnv(OE.PendulumBatch(n, seed=seed, max_steps=ms)); spec = SPECS["pendulum"]()
    if monitor:
        o = OE.MonitorWrapper(o)
    if norm:
        o = OE.NormalizeWrapper(o, spec.obs_dim)
    return env, o, spec


@pytest.mark.parametrize("kind,n,T,ms,monitor,norm", [
    ("cartpole", 64, 16, 500, True, False), ("cartpole", 333, 64, 20, True, False), ("cartpole", 4096, 32, 25, False, False),
    ("pendulum", 100, 40, 15, True, True), ("pendulum", 1000, 24, 10, True, True), ("cartpole", 200, 48, 18, True, True),
    ("pendulum", 50, 30, 12, False, False),
    ("pendulum_scaled", 300, 30, 12, True, False), ("pendulum_scaled", 700, 20, 9, True, True),     # fast kernel / cooperative kernel
    ("pendulum", 10240, 5, 3, True, True),      # >= 64 envs per SM with a wide net: 64-env tiles, wide layers on mma.sync tiles
    ("pendulum", 16384, 4, 3, True, True),      # BASELINE config C3's env count (Pendulum + NormalizeWrapperEnv), truncation every 3 steps
    ("cartpole", 14400, 5, 4, True, True),      # general kernel with a [64,64] discrete actor on tcgen05 (rollout_gtc.cuh, two hidden layers)
    ("cartpole", 65536, 6, 4, True, False)])    # BASELINE config C4's env count: 2048 tiles on the tensor-core rollout, truncation list at scale
def test_fused_rollout_replay(D, kind, n, T, ms, monitor, norm):
    env, oenv, spec = _mk(D, kind, n, 9, ms, monitor, norm)
    rng = np.random.default_rng(4)
    flat = (OP.init_params(spec, seed=2) + rng.normal(size=spec.n_params()).astype(f32) * 0.05).astype(f32)
    forced = rng.integers(1, 3, (T, n)) if kind == "cartpole" else rng.normal(size=(T, n, 1)).astype(f32) * 1.5
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=spec.hidden)
    alg = D.PPO(n_steps=T, gamma=0.97, gae_lambda=0.9)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
    agent.set_parameters(flat)
    tol = dict(rtol=3e-5, atol=3e-5) if norm else dict(rtol=1e-5, atol=1e-5)
    for rollout in range(2):           # second rollout continues from the env state (ppo.jl:100-143)
        buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
        fps, ok = D.collect_rollout(buf, agent, alg, env, forced_actions=forced)
        assert ok
        ob = OO.collect_rollout_timemajor(oenv, spec, flat, T, forced_actions=forced)
        te, tr = _flags(buf)
        np.testing.assert_array_equal(te, ob["term"])
        np.testing.assert_array_equal(tr, ob["trunc"])
        np.testing.assert_allclose(buf.download("obs"), ob["obs"], rtol=3e-5 if norm else 1e-6, atol=3e-5 if norm else 1e-7)
        np.testing.assert_allclose(buf.download("rewards"), ob["rewards"], **(tol if norm else dict(rtol=1e-6, atol=0)))
        np.testing.assert_allclose(buf.download("values"), ob["values"], **tol)
        np.testing.assert_allclose(buf.download("logprobs"), ob["logprobs"], rtol=1e-4, atol=1e-4)
        np.testing.assert_allclose(buf.download("last_values"), ob["last_values"], **tol)
        np.testing.assert_allclose(np.where(tr, buf.download("boot"), 0), ob["boot"], **tol)
        if kind == "cartpole":
            np.testing.assert_array_equal(buf.download("actions")[..., 0], forced)
        ea, er = OO.gae_timemajor(ob["rewards"], ob["values"], ob["term"], ob["trunc"], ob["boot"], ob["last_values"], 0.97, 0.9)
        np.testing.assert_allclose(buf.download("advantages"), ea, rtol=1e-4, atol=1e-4)
        np.testing.assert_allclose(buf.download("returns"), buf.download("advantages") + buf.download("values"), atol=1e-6)
        if monitor:
            done = te | tr
            np.testing.assert_allclose(buf.download("episode_r")[done], ob["episode_r"][done], rtol=1e-5)
            np.testing.assert_array_equal(buf.download("episode_l")[done], ob["episode_l"][done])
            mon = oenv.env if norm else oenv
            s = env.monitor_stats()
            assert s["n_in_window"] == len(mon.returns)
            if len(mon.returns):
                assert abs(s["ep_rew_mean"] - np.mean(np.array(mon.returns, f32))) <= 1e-4 * abs(np.mean(mon.returns)) + 1e-5
                assert abs(s["ep_len_mean"] - np.mean(mon.lengths)) < 1e-3
        if norm:
            s = env.norm_stats()
            assert s["obs_count"] == oenv.obs_rms.count and s["ret_count"] == oenv.ret_rms.count
            np.testing.assert_allclose(s["obs_mean"], oenv.obs_rms.mean, rtol=1e-5, atol=1e-6)
            np.testing.assert_allclose(s["obs_var"], oenv.obs_rms.var, rtol=1e-5, atol=1e-6)
            np.testing.assert_allclose([s["ret_mean"], s["ret_var"]], [oenv.ret_rms.mean, oenv.ret_rms.var], rtol=1e-5, atol=1e-6)
        assert (te | tr).any()
        # reference buffer order (rollout_buffer.jl:70-74): the permutation of the device order, element for element
        if T * n <= 40000:
            order = buf.reference_order()
            np.testing.assert_array_equal(order, OO.reference_order(ob["term"], ob["trunc"]))
            assert sorted(order.tolist()) == list(range(T * n))
        buf.close()


@pytest.mark.parametrize("obs_dim,n,T,norm", [(10, 300, 20, False), (64, 130, 12, True), (5, 2000, 8, False)])
def test_fused_rollout_synthetic_env(D, obs_dim, n, T, norm):
    """Rollout-sweep env (SURVEY §8d C5) through the general (cooperative) rollout kernel, replayed actions."""
    ms = 7
    env = D.CudaBatchedEnv("synthetic", n, obs_dim=obs_dim, max_steps=ms, seed=4, monitor_window=100,
                           normalize=D.NormalizeConfig() if norm else None)
    oenv = OE.MonitorWrapper(OE.ParallelEnv(OE.SyntheticBatch(n, obs_dim, seed=4, max_steps=ms)))
    if norm:
        oenv = OE.NormalizeWrapper(oenv, obs_dim)
    spec = OP.PolicySpec(obs_dim, [32, 32], "discrete", 2, act_start=1)
    rng = np.random.default_rng(2)
    flat = (OP.init_params(spec, seed=1) + rng.normal(size=spec.n_params()).astype(f32) * 0.05).astype(f32)
    forced = rng.integers(1, 3, (T, n))
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=[32, 32])
    alg = D.PPO(n_steps=T)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
    agent.set_parameters(flat)
    buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
    D.collect_rollout(buf, agent, alg, env, forced_actions=forced)
    ob = OO.collect_rollout_timemajor(oenv, spec, flat, T, forced_actions=forced)
    te, tr = _flags(buf)
    np.testing.assert_array_equal(te, ob["term"])
    np.testing.assert_array_equal(tr, ob["trunc"])
    tol = dict(rtol=3e-5, atol=3e-5)
    np.testing.assert_allclose(buf.download("obs"), ob["obs"], **tol)
    np.testing.assert_allclose(buf.download("rewards"), ob["rewards"], **tol)
    np.testing.assert_allclose(buf.download("values"), ob["values"], **tol)
    np.testing.assert_allclose(np.where(tr, buf.download("boot"), 0), ob["boot"], **tol)
    np.testing.assert_allclose(buf.download("last_values"), ob["last_values"], **tol)
    assert tr.any() and te.any() if n >= 300 else tr.any()
    buf.close()


@pytest.mark.parametrize("obs_dim,hidden,n,T,per_thread", [(4, [8], 700, 24, 1), (4, [8], 700, 24, 2), (10, [16, 12], 333, 18, 1),
                                                           (64, [8, 8], 130, 12, 2), (16, [6], 5000, 9, 2), (7, [5, 8], 257, 9, 1)])
def test_syn_rollout_kernel_vs_oracle(D, obs_dim, hidden, n, T, per_thread):
    """Thread-per-env rollout of the synthetic env with a small policy (rollout_syn.cuh; SURVEY §8d C5) against the oracle:
    two consecutive rollouts (the state written back by the first feeds the second) with replayed actions are bit-exact on
    flags / observations / rewards, 3e-5 on values, log-probs and both kinds of bootstrap values; Monitor statistics agree;
    a third, SAMPLED rollout follows the Philox stream and matches the general kernel element for element.  `per_thread` = 2
    forces the two-envs-per-thread variant that large batches of narrow nets use."""
    ms = 7
    D.set_option("syn_rollout", per_thread)
    mk = lambda: D.CudaBatchedEnv("synthetic", n, obs_dim=obs_dim, max_steps=ms, seed=4, monitor_window=100)
    env = mk()
    oenv = OE.MonitorWrapper(OE.ParallelEnv(OE.SyntheticBatch(n, obs_dim, seed=4, max_steps=ms)))
    n_a = env.action_space().n
    spec = OP.PolicySpec(obs_dim, hidden, "discrete", n_a, act_start=1)
    rng = np.random.default_rng(2)
    flat = (OP.init_params(spec, seed=1) + rng.normal(size=spec.n_params()).astype(f32) * 0.3).astype(f32)
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=hidden)
    alg = D.PPO(n_steps=T)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
    agent.set_parameters(flat)
    buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
    tol = dict(rtol=3e-5, atol=3e-5)
    for it in range(2):
        forced = rng.integers(1, 1 + n_a, (T, n))
        D.collect_rollout(buf, agent, alg, env, forced_actions=forced)
        ob = OO.collect_rollout_timemajor(oenv, spec, flat, T, forced_actions=forced)
        te, tr = _flags(buf)
        np.testing.assert_array_equal(te, ob["term"])
        np.testing.assert_array_equal(tr, ob["trunc"])
        np.testing.assert_array_equal(buf.download("obs"), ob["obs"])
        np.testing.assert_array_equal(buf.download("rewards"), ob["rewards"])
        np.testing.assert_array_equal(buf.download("actions").reshape(T, n), forced)
        np.testing.assert_allclose(buf.download("values"), ob["values"], **tol)
        np.testing.assert_allclose(buf.download("logprobs"), ob["logprobs"], **tol)
        np.testing.assert_allclose(np.where(tr, buf.download("boot"), 0), ob["boot"], **tol)
        np.testing.assert_allclose(buf.download("last_values"), ob["last_values"], **tol)
        assert tr.any()
        s = env.monitor_stats()
        mon = oenv
        assert s["total_episodes"] == mon.total_episodes
        done = te | tr
        np.testing.assert_array_equal(np.where(done, buf.download("episode_l"), 0), np.where(done, ob["episode_l"], 0))
        np.testing.assert_allclose(np.where(done, buf.download("episode_r"), 0), np.where(done, ob["episode_r"], 0), rtol=1e-6)
    # sampled rollout: the same env state through both kernels
    env2 = mk()
    outs = []
    for e, opt in ((env, 1), (env2, 0)):
        if e is env2:       # bring env2 to the state of env: replaying is cheaper than copying state
            D.set_option("syn_rollout", per_thread)
            e2buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, 2 * T, n)
            alg2 = D.PPO(n_steps=2 * T)
            D.collect_rollout(e2buf, agent, alg2, env2, forced_actions=rng.integers(1, 1 + n_a, (2 * T, n)))
            e2buf.close()
        D.set_option("syn_rollout", per_thread if opt else 0)
        try:
            agent.device.seed(99, 5)
            D.collect_rollout(buf, agent, alg, e)
        finally:
            D.set_option("syn_rollout", 1)
        outs.append({k: buf.download(k) for k in ("obs", "actions", "rewards", "values", "logprobs", "boot", "last_values", "flags")})
    a, b = outs
    for k in ("obs", "actions", "rewards", "flags"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    tr = (a["flags"] & 2) != 0
    for k in ("values", "logprobs", "last_values"):
        np.testing.assert_allclose(a[k], b[k], rtol=1e-5, atol=1e-6, err_msg=k)
    np.testing.assert_allclose(np.where(tr, a["boot"], 0), np.where(tr, b["boot"], 0), rtol=1e-5, atol=1e-6)
    obs, act = a["obs"].reshape(T * n, -1), a["actions"].reshape(T * n)
    probs = OP.softmax(OP.mlp_forward(OP.unflatten(spec, flat)["actor"], obs))
    u = OPH.sample_uniform64(np.tile(np.arange(n), T), 5 + np.repeat(np.arange(T), n), 99)
    ea = OP.categorical_sample(probs, u, spec.act_start)
    margin = np.abs(np.cumsum(probs, axis=1) - u[:, None]).min(axis=1)
    assert ((act == ea) | (margin < 1e-5)).all()
    buf.close()


# ------------------------------------------------------------------------------------------
# (c) PPO loss + gradients, optimiser, full update
# ------------------------------------------------------------------------------------------
def _minibatch(spec, flat, B, rng):
    obs = rng.normal(size=(B, spec.obs_dim)).astype(f32)
    if spec.act_kind == "discrete":
        actions = rng.integers(spec.act_start, spec.act_start + spec.act_n, (B, 1))
    else:
        actions = rng.normal(size=(B, spec.act_n)).astype(f32)
    v0, lp0, _ = OP.evaluate_actions(spec, flat, obs, actions)
    old_lp = (lp0 + rng.normal(size=B).astype(f32) * 0.2).astype(f32)
    old_v = (v0 + rng.normal(size=B).astype(f32) * 0.3).astype(f32)
    return obs, actions, rng.normal(size=B).astype(f32), rng.normal(size=B).astype(f32), old_lp, old_v


def _relerr(a, b):
    return np.linalg.norm(a.astype(np.float64) - b) / max(np.linalg.norm(b), 1e-30)


@pytest.mark.parametrize("name", ["cartpole", "pendulum", "odd", "box3", "nohidden"])
@pytest.mark.parametrize("B", [64, 1000, 4097])
def test_ppo_loss_and_gradients(D, name, B):
    spec = SPECS[name]()
    rng = np.random.default_rng(B)
    flat = (OP.init_params(spec, seed=3) + rng.normal(size=spec.n_params()).astype(f32) * 0.05).astype(f32)
    p = _device_policy(D, spec, flat)
    mb = _minibatch(spec, flat, B, rng)
    for alg in (D.PPO(ent_coef=0.01), D.PPO(ent_coef=0.02, clip_range_vf=0.2, normalize_advantage=False, vf_coef=0.7)):
        cfg = OO.PPOConfig(ent_coef=alg.ent_coef, clip_range_vf=alg.clip_range_vf, normalize_advantage=alg.normalize_advantage,
                           vf_coef=alg.vf_coef)
        loss, stats, g = p.loss_grad(*mb, alg.hyper())
        eloss, estats, eg = OO.ppo_loss_and_grads(spec, flat, *mb, cfg)
        assert abs(loss - eloss) <= 1e-4 * max(1.0, abs(eloss))
        for k in estats:
            assert abs(stats[k] - estats[k]) <= 1e-4 * max(1.0, abs(estats[k])), (k, stats[k], estats[k])
        assert _relerr(g, eg) < 1e-4, _relerr(g, eg)
        np.testing.assert_allclose(g, eg, rtol=1e-3, atol=1e-4 * np.abs(eg).max())


def test_optimizer_step_vs_oracle(D):
    spec = SPECS["cartpole"]()
    rng = np.random.default_rng(0)
    flat = OP.init_params(spec, seed=0)
    p = _device_policy(D, spec, flat)
    opt = OO.Adam(flat.size, lr=3e-4)
    cur = flat
    for it in range(5):
        g = (rng.normal(size=flat.size) * (0.001 if it == 2 else 0.05)).astype(f32)
        gc, norm = OO.clip_grads(g, 0.5)
        cur = opt.step(cur, gc)
        dn = p.optimizer_step(g, D.PPO().hyper())
        assert abs(dn - norm) <= 1e-5 * norm
        np.testing.assert_allclose(p.get_params(), cur, rtol=1e-6, atol=1e-7)
    m, v, step = p.get_opt_state()
    assert step == 5
    np.testing.assert_allclose(m, opt.m, rtol=1e-5, atol=1e-8)
    np.testing.assert_allclose(v, opt.v, rtol=1e-5, atol=1e-10)
    # forward uses the refreshed packed weights
    obs = rng.normal(size=(10, 4)).astype(f32)
    np.testing.assert_allclose(p.predict_values(obs), OP.predict_values(spec, cur, obs), rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("kind,batch", [("cartpole", 256), ("cartpole", 300), ("pendulum", 512)])
def test_ppo_update_vs_oracle(D, kind, batch):
    """Whole epoch/minibatch loop (ppo.jl:188-254) on the same buffer: same Feistel minibatches,
    ragged last batch, clip + Adam. Parameters and per-iteration statistics must agree."""
    n, T = 40, 24
    env, oenv, spec = _mk(D, kind, n, 13, 15, True, False)
    rng = np.random.default_rng(8)
    flat = (OP.init_params(spec, seed=5) + rng.normal(size=spec.n_params()).astype(f32) * 0.02).astype(f32)
    forced = rng.integers(1, 3, (T, n)) if kind == "cartpole" else rng.normal(size=(T, n, 1)).astype(f32)
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=spec.hidden)
    alg = D.PPO(n_steps=T, batch_size=batch, epochs=3, ent_coef=0.01)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
    agent.set_parameters(flat)
    buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
    D.collect_rollout(buf, agent, alg, env, forced_actions=forced)
    ob = {k: buf.download(k) for k in ("obs", "actions", "rewards", "values", "logprobs", "advantages", "returns")}
    import ctypes as C
    st = D.IterStats()
    h = alg.hyper()
    from dril_b200 import _lib as L
    L.check(agent.ctx.lib.dril_ppo_update(agent.device.h, buf.h, C.byref(h), alg.epochs, alg.batch_size, 777, 3, C.byref(st)))
    cfg = OO.PPOConfig(n_steps=T, batch_size=batch, epochs=3, ent_coef=0.01)
    opt = OO.Adam(flat.size, lr=cfg.learning_rate)
    new_flat, means, _ = OO.ppo_update(spec, flat, opt, ob, cfg, shuffle_seed=777, epoch_counter0=3)
    got = agent.device.get_params()
    assert _relerr(got - flat, new_flat - flat) < 2e-3, _relerr(got - flat, new_flat - flat)
    np.testing.assert_allclose(got, new_flat, rtol=1e-4, atol=2e-6)
    n_mb = -(-T * n // batch)
    assert st.n_minibatch_steps == 3 * n_mb and st.kl_stopped == 0
    for k in ("policy_loss", "value_loss", "entropy_loss", "approx_kl_div", "clip_fraction", "loss", "grad_norm"):
        assert abs(getattr(st, k) - means[k]) <= 2e-4 * max(1.0, abs(means[k])), (k, getattr(st, k), means[k])
    assert abs(st.explained_variance - OO.explained_variance(ob["values"], ob["returns"])) < 1e-4
    buf.close()


def test_target_kl_stop(D):
    """ppo.jl:235-238: the KL check comes before the step is applied and stops ALL remaining epochs; grad_norm of the stopping
    minibatch is still recorded; means over the applied minibatches (NaN when none was applied, ppo.jl:257-263).  Stop step,
    parameters and statistics against oracle.ppo.ppo_update on the same buffer."""
    import ctypes as C
    from dril_b200 import _lib as L
    n, T = 32, 16
    for case, target_kl, lr in (("later", 1e-4, 3e-2), ("first", 1e-4, 1e-2)):   # stops after a few applied steps / on the very first minibatch
        env, oenv, spec = _mk(D, "cartpole", n, 1, 500, False, False)
        flat = OP.init_params(spec, seed=1)
        layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=spec.hidden)
        alg = D.PPO(n_steps=T, batch_size=128, epochs=5, target_kl=target_kl, learning_rate=lr)
        agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
        agent.set_parameters(flat)
        buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
        D.collect_rollout(buf, agent, alg, env)
        ob = {k: buf.download(k) for k in ("obs", "actions", "rewards", "values", "logprobs", "advantages", "returns")}
        st = D.IterStats()
        h = alg.hyper()
        if case == "first":       # parameters moved away from the ones the rollout was collected with: the first minibatch trips the stop
            flat = (flat + np.random.default_rng(3).normal(size=flat.size).astype(f32) * 0.05).astype(f32)
            agent.set_parameters(flat)
        L.check(agent.ctx.lib.dril_ppo_update(agent.device.h, buf.h, C.byref(h), alg.epochs, alg.batch_size, 11, 0, C.byref(st)))
        cfg = OO.PPOConfig(n_steps=T, batch_size=128, epochs=5, target_kl=target_kl, learning_rate=lr)
        opt = OO.Adam(flat.size, lr=lr)
        new_flat, means, epochs_run = OO.ppo_update(spec, flat, opt, ob, cfg, shuffle_seed=11, epoch_counter0=0)
        assert st.kl_stopped == 1
        assert st.n_minibatch_steps == opt.t, (st.n_minibatch_steps, opt.t)
        assert st.n_minibatch_steps < 5 * (n * T // 128)
        np.testing.assert_allclose(agent.device.get_params(), new_flat, rtol=2e-4, atol=5e-6)
        for k in ("policy_loss", "value_loss", "approx_kl_div", "loss", "grad_norm"):
            got, exp = getattr(st, k), means[k]
            if np.isnan(exp):
                assert np.isnan(got), (k, got)
            else:
                assert abs(got - exp) <= 5e-4 * max(1.0, abs(exp)), (k, got, exp)
        if case == "first":
            assert opt.t == 0 and np.isnan(st.policy_loss) and np.isfinite(st.grad_norm)   # empty means are NaN, the norm was recorded
            np.testing.assert_array_equal(agent.device.get_params(), flat)
        buf.close()


# ------------------------------------------------------------------------------------------
# full-size properties at the BASELINE config (4096 envs x 128 steps)
# ------------------------------------------------------------------------------------------
def test_full_size_properties(D):
    n, T = 4096, 128
    env = D.CudaBatchedEnv("cartpole", n, seed=0, monitor_window=100)
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=[64, 64])
    alg = D.PPO(n_steps=T, batch_size=T * n // 4, epochs=1)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
    buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
    D.collect_rollout(buf, agent, alg, env)
    adv, ret, val, rew = (buf.download(k) for k in ("advantages", "returns", "values", "rewards"))
    te, tr = _flags(buf)
    assert np.isfinite(adv).all() and (rew == 1).all()
    np.testing.assert_allclose(ret, adv + val, atol=1e-6)
    assert not tr.any() and te.mean() > 0.02        # random policy: ~22-step episodes
    # GAE linearity: scaling rewards/values/bootstraps scales the advantages
    a2, _ = D.gae_raw(2 * rew, 2 * val, te, tr, 2 * buf.download("boot"), 2 * buf.download("last_values"), 0.99, 0.95)
    np.testing.assert_allclose(a2, 2 * adv, rtol=1e-6, atol=1e-6)
    # episode lengths recorded by the monitor equal the gaps between terminations
    el = buf.download("episode_l")
    e0 = np.nonzero(te[:, 0])[0]
    assert (np.diff(e0) == el[e0[1:], 0]).all()
    obs = buf.download("obs")
    assert (np.abs(obs[..., 0]) <= 2.4 + 0.2).all() and (np.abs(obs[..., 2]) <= 0.21 + 0.2).all()
    buf.close()


# ------------------------------------------------------------------------------------------
# kernel-path switches: every combination must agree with the oracle (and hence with each other)
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tc,tail,tc_rollout,persistent", [(1, 1, 1, 1), (1, 1, 1, 0), (1, 0, 1, 1), (0, 0, 0, 1), (1, 1, 0, 1), (0, 0, 1, 1)])
def test_kernel_paths_vs_oracle(D, tc, tail, tc_rollout, persistent):
    """The tensor-core loss/grad kernel (all minibatch steps in one persistent launch, one launch per step with the fused
    reduce/clip/Adam tail, and without the tail), the fp32 CUDA-core kernel, the tensor-core rollout and the general rollout are
    interchangeable: same buffer, same updated parameters."""
    opts = {"tc": tc, "fused_tail": tail, "tc_rollout": tc_rollout, "ftg": 1 if tc else 0, "persistent": persistent}   # tc = 0: the general mma.sync kernel
    try:
        for k, v in opts.items():
            D.set_option(k, v)
        n, T = 96, 20
        env, oenv, spec = _mk(D, "cartpole", n, 31, 12, True, False)
        rng = np.random.default_rng(5)
        flat = (OP.init_params(spec, seed=6) + rng.normal(size=spec.n_params()).astype(f32) * 0.02).astype(f32)
        forced = rng.integers(1, 3, (T, n))
        layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=spec.hidden)
        alg = D.PPO(n_steps=T, batch_size=500, epochs=2, ent_coef=0.01)
        agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
        agent.set_parameters(flat)
        assert agent.device.update_path() == ("tensor" if tc else "mma")    # [64,64] with "tc" off: mma.sync tiles
        buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
        D.collect_rollout(buf, agent, alg, env, forced_actions=forced)
        exp = OO.collect_rollout_timemajor(oenv, spec, flat, T, forced_actions=forced)
        te, tr = _flags(buf)
        np.testing.assert_array_equal(te, exp["term"])
        np.testing.assert_array_equal(tr, exp["trunc"])
        assert tr.any()
        np.testing.assert_allclose(buf.download("obs"), exp["obs"], rtol=1e-6, atol=1e-7)
        np.testing.assert_allclose(buf.download("values"), exp["values"], rtol=1e-5, atol=1e-5)
        np.testing.assert_allclose(buf.download("logprobs"), exp["logprobs"], rtol=1e-4, atol=1e-4)
        np.testing.assert_allclose(np.where(tr, buf.download("boot"), 0), exp["boot"], rtol=1e-5, atol=1e-5)
        np.testing.assert_allclose(buf.download("last_values"), exp["last_values"], rtol=1e-5, atol=1e-5)
        ob = {k: buf.download(k) for k in ("obs", "actions", "rewards", "values", "logprobs", "advantages", "returns")}
        import ctypes as C
        from dril_b200 import _lib as L
        st = D.IterStats()
        h = alg.hyper()
        L.check(agent.ctx.lib.dril_ppo_update(agent.device.h, buf.h, C.byref(h), alg.epochs, alg.batch_size, 99, 0, C.byref(st)))
        cfg = OO.PPOConfig(n_steps=T, batch_size=500, epochs=2, ent_coef=0.01)
        opt = OO.Adam(flat.size, lr=cfg.learning_rate)
        new_flat, means, _ = OO.ppo_update(spec, flat, opt, ob, cfg, shuffle_seed=99, epoch_counter0=0)
        got = agent.device.get_params()
        np.testing.assert_allclose(got, new_flat, rtol=1e-4, atol=2e-6)
        assert st.n_minibatch_steps == 2 * 4
        for k in ("policy_loss", "value_loss", "loss", "grad_norm"):
            assert abs(getattr(st, k) - means[k]) <= 2e-4 * max(1.0, abs(means[k])), (k, getattr(st, k), means[k])
        buf.close()
    finally:
        for k in opts:
            D.set_option(k, 1)


def test_c1_shape_update_vs_oracle(D):
    """BASELINE config C1 (the reference's own CPU-runnable case): 4 envs, n_steps 2048, batch 64 -> 128 Adam steps per
    epoch on half-filled 128-sample tiles, one CTA per launch.  Parameters after one epoch must match the oracle."""
    n, T = 4, 2048
    env, oenv, spec = _mk(D, "cartpole", n, 3, 500, True, False)
    flat = OP.init_params(spec, seed=11)
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=spec.hidden)
    alg = D.PPO(n_steps=T, batch_size=64, epochs=1)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
    agent.set_parameters(flat)
    buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
    D.collect_rollout(buf, agent, alg, env)
    ob = {k: buf.download(k) for k in ("obs", "actions", "rewards", "values", "logprobs", "advantages", "returns")}
    # the rollout itself: stored log-probs / values equal evaluate_actions on the stored (obs, actions)
    v, lp, _ = OP.evaluate_actions(spec, flat, ob["obs"].reshape(T * n, -1), ob["actions"].reshape(T * n, -1))
    np.testing.assert_allclose(ob["logprobs"].reshape(-1), lp, atol=1e-5)
    np.testing.assert_allclose(ob["values"].reshape(-1), v, atol=1e-5)
    import ctypes as C
    from dril_b200 import _lib as L
    st = D.IterStats()
    h = alg.hyper()
    L.check(agent.ctx.lib.dril_ppo_update(agent.device.h, buf.h, C.byref(h), alg.epochs, alg.batch_size, 5, 0, C.byref(st)))
    cfg = OO.PPOConfig(n_steps=T, batch_size=64, epochs=1)
    opt = OO.Adam(flat.size, lr=cfg.learning_rate)
    new_flat, means, _ = OO.ppo_update(spec, flat, opt, ob, cfg, shuffle_seed=5, epoch_counter0=0)
    got = agent.device.get_params()
    assert st.n_minibatch_steps == 128
    np.testing.assert_allclose(got, new_flat, rtol=2e-3, atol=2e-4)
    assert _relerr(got - flat, new_flat - flat) < 2e-2
    for k in ("policy_loss", "value_loss", "loss"):
        assert abs(getattr(st, k) - means[k]) <= 1e-3 * max(1.0, abs(means[k])), (k, getattr(st, k), means[k])
    buf.close()


@pytest.mark.parametrize("n,T,ms", [(33, 6, 1), (64, 1, 500), (5, 40, 2), (1, 9, 3)])
def test_fused_rollout_edge_shapes(D, n, T, ms):
    """Edge cases of the (tensor-core) rollout against the oracle with replayed actions: every step truncates
    (max_steps = 1: back-to-back resets, one terminal observation per sample), a single step, tiny env counts."""
    env, oenv, spec = _mk(D, "cartpole", n, 17, ms, True, False)
    rng = np.random.default_rng(2)
    flat = (OP.init_params(spec, seed=1) + rng.normal(size=spec.n_params()).astype(f32) * 0.05).astype(f32)
    forced = rng.integers(1, 3, (T, n))
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=spec.hidden)
    alg = D.PPO(n_steps=T, gamma=0.97, gae_lambda=0.9)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
    agent.set_parameters(flat)
    for rollout in range(2):
        buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
        D.collect_rollout(buf, agent, alg, env, forced_actions=forced)
        ob = OO.collect_rollout_timemajor(oenv, spec, flat, T, forced_actions=forced)
        te, tr = _flags(buf)
        np.testing.assert_array_equal(te, ob["term"])
        np.testing.assert_array_equal(tr, ob["trunc"])
        np.testing.assert_allclose(buf.download("obs"), ob["obs"], rtol=1e-6, atol=1e-7)
        np.testing.assert_allclose(buf.download("values"), ob["values"], rtol=1e-5, atol=1e-5)
        np.testing.assert_allclose(buf.download("logprobs"), ob["logprobs"], rtol=1e-4, atol=1e-4)
        np.testing.assert_allclose(buf.download("last_values"), ob["last_values"], rtol=1e-5, atol=1e-5)
        np.testing.assert_allclose(np.where(tr, buf.download("boot"), 0), ob["boot"], rtol=1e-5, atol=1e-5)
        ea, er = OO.gae_timemajor(ob["rewards"], ob["values"], ob["term"], ob["trunc"], ob["boot"], ob["last_values"], 0.97, 0.9)
        np.testing.assert_allclose(buf.download("advantages"), ea, rtol=1e-4, atol=1e-4)
        done = te | tr
        if done.any():
            np.testing.assert_array_equal(buf.download("episode_l")[done], ob["episode_l"][done])
        if ms == 1:
            assert tr.all()
        buf.close()


WIDE = {
    "pendulum": lambda: SPECS["pendulum"](),
    "wide_discrete": lambda: OP.PolicySpec(10, [128, 96], "discrete", 5, act_start=0),
    "mid_box": lambda: OP.PolicySpec(6, [64, 32, 16], "continuous", 2, act_low=[-1, -1], act_high=[1, 1]),
    "cartpole_fp32": lambda: SPECS["cartpole"](),
    # activations of one net leave room for less than 128 samples: single-net passes with a 96-sample tile (MMA tiles with
    # 12 sample blocks); without single_net a 48-sample tile of both nets
    "very_wide": lambda: OP.PolicySpec(8, [256, 256], "continuous", 2, act_low=[-1, -1], act_high=[1, 1]),
}


@pytest.mark.parametrize("single,mma", [(1, 1), (1, 0), (0, 1), (0, 0)])
@pytest.mark.parametrize("name", list(WIDE))
def test_wide_net_single_net_passes(D, name, single, mma):
    """General-shape loss/grad kernel: (a) networks too wide for a 128-sample tile of both nets are processed one net per
    pass with shared activation rows (option "single_net"); (b) layers whose padded dims are multiples of 16 run on
    mma.sync 3xTF32 tiles (option "mma").  Both are fixed per policy at creation; every combination meets north_star (c)."""
    spec = WIDE[name]()
    rng = np.random.default_rng(11)
    flat = (OP.init_params(spec, seed=4) + rng.normal(size=spec.n_params()).astype(f32) * 0.05).astype(f32)
    D.set_option("single_net", single); D.set_option("mma", mma); D.set_option("tc", 0); D.set_option("ftg", 0)
    try:
        p = _device_policy(D, spec, flat)
        assert p.update_path() != "tensor"
        for B in (77, 128, 1000):
            mb = _minibatch(spec, flat, B, rng)
            alg = D.PPO(ent_coef=0.01, clip_range_vf=0.3)
            cfg = OO.PPOConfig(ent_coef=0.01, clip_range_vf=0.3)
            loss, stats, g = p.loss_grad(*mb, alg.hyper())
            eloss, estats, eg = OO.ppo_loss_and_grads(spec, flat, *mb, cfg)
            assert abs(loss - eloss) <= 1e-4 * max(1.0, abs(eloss))
            for k in estats:
                assert abs(stats[k] - estats[k]) <= 1e-4 * max(1.0, abs(estats[k])), (k, stats[k], estats[k])
            assert _relerr(g, eg) < 1e-4, _relerr(g, eg)
            print(name, single, mma, B, "grad relerr", _relerr(g, eg))
        p.close()
    finally:
        D.set_option("single_net", 1); D.set_option("mma", 1); D.set_option("tc", 1); D.set_option("ftg", 1)


# ------------------------------------------------------------------------------------------
# many tiles per CTA: the tile loops of the loss/grad kernels (more tiles than SMs) against the oracle
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,B", [("cartpole", 148 * 128 * 4 + 77), ("cartpole", 148 * 64 * 3 + 5), ("pendulum", 148 * 128 * 2 + 33)])
def test_ppo_loss_and_gradients_many_tiles(D, name, B):
    """B large enough that every CTA (and each of its warp groups) processes several sample tiles; the small-B cases of
    test_ppo_loss_and_gradients never leave the first tile of a CTA."""
    spec = SPECS[name]()
    rng = np.random.default_rng(7)
    flat = (OP.init_params(spec, seed=3) + rng.normal(size=spec.n_params()).astype(f32) * 0.05).astype(f32)
    p = _device_policy(D, spec, flat)
    mb = _minibatch(spec, flat, B, rng)
    alg = D.PPO(ent_coef=0.01)
    cfg = OO.PPOConfig(ent_coef=0.01)
    loss, stats, g = p.loss_grad(*mb, alg.hyper())
    eloss, estats, eg = OO.ppo_loss_and_grads(spec, flat, *mb, cfg)
    assert abs(loss - eloss) <= 1e-4 * max(1.0, abs(eloss))
    for k in estats:
        assert abs(stats[k] - estats[k]) <= 1e-4 * max(1.0, abs(estats[k])), (k, stats[k], estats[k])
    assert _relerr(g, eg) < 1e-4, _relerr(g, eg)
    p.close()


@pytest.mark.parametrize("tc,ft", [(1, 1), (1, 0), (0, 0)])
def test_c2_shape_update_vs_oracle(D, tc, ft):
    """BASELINE config C2 at full size (4096 envs x 128 steps, 4 minibatches of 131 072 shuffled samples, 7 tiles per CTA):
    one epoch of the update on the device buffer against the oracle on the same buffer and the same Feistel minibatches."""
    D.set_option("tc", tc)
    D.set_option("ft", ft)
    try:
        n, T = 4096, 128
        env, oenv, spec = _mk(D, "cartpole", n, 5, 500, False, False)
        flat = OP.init_params(spec, seed=2)
        layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=spec.hidden)
        alg = D.PPO(n_steps=T, batch_size=T * n // 4, epochs=1, ent_coef=0.01)
        agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
        agent.set_parameters(flat)
        buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
        D.collect_rollout(buf, agent, alg, env)
        ob = {k: buf.download(k) for k in ("obs", "actions", "rewards", "values", "logprobs", "advantages", "returns")}
        import ctypes as C
        from dril_b200 import _lib as L
        st = D.IterStats()
        h = alg.hyper()
        L.check(agent.ctx.lib.dril_ppo_update(agent.device.h, buf.h, C.byref(h), alg.epochs, alg.batch_size, 41, 2, C.byref(st)))
        cfg = OO.PPOConfig(n_steps=T, batch_size=T * n // 4, epochs=1, ent_coef=0.01)
        opt = OO.Adam(flat.size, lr=cfg.learning_rate)
        new_flat, means, _ = OO.ppo_update(spec, flat, opt, ob, cfg, shuffle_seed=41, epoch_counter0=2)
        got = agent.device.get_params()
        assert st.n_minibatch_steps == 4
        assert _relerr(got - flat, new_flat - flat) < 2e-3, _relerr(got - flat, new_flat - flat)
        np.testing.assert_allclose(got, new_flat, rtol=1e-4, atol=2e-6)
        for k in ("policy_loss", "value_loss", "entropy_loss", "approx_kl_div", "clip_fraction", "loss", "grad_norm"):
            assert abs(getattr(st, k) - means[k]) <= 2e-4 * max(1.0, abs(means[k])), (k, getattr(st, k), means[k])
        buf.close()
    finally:
        D.set_option("tc", 1)
        D.set_option("ft", 1)


@pytest.mark.parametrize("ft", [1, 0])
@pytest.mark.parametrize("B", [1, 63, 64, 65, 1000, 148 * 64 * 2 + 31])
def test_tcgen05_kernels_vs_oracle(D, ft, B):
    """Both tcgen05 loss/grad kernels for the default [64,64] layer (features-on-lanes fp16 hi/lo, option "ft" = 1, and
    samples-on-lanes 3xTF32, "ft" = 0) on ragged tile counts, with large and tiny advantage / return scales applied to the
    whole minibatch (the fp16 kernel scales its deltas by a power of two fixed at a warp group's first tile with a non-zero
    gradient; tiles of different scales: tests/test_gpu_grad_scale.py) and with one action (Discrete(1): zero actor
    gradient)."""
    D.set_option("ft", ft)
    try:
        for name, scale in (("cartpole", 1.0), ("cartpole", 3e4), ("cartpole", 1e-6), ("one_action", 1.0)):
            spec = SPECS["cartpole"]() if name == "cartpole" else OP.PolicySpec(3, [64, 64], "discrete", 1, act_start=0)
            rng = np.random.default_rng(B + int(ft))
            flat = (OP.init_params(spec, seed=3) + rng.normal(size=spec.n_params()).astype(f32) * 0.05).astype(f32)
            p = _device_policy(D, spec, flat)
            assert p.update_path() == "tensor"
            obs, actions, adv, ret, old_lp, old_v = _minibatch(spec, flat, B, rng)
            ret = (ret * scale).astype(f32)
            old_v = (old_v * scale).astype(f32)
            for alg in (D.PPO(ent_coef=0.01), D.PPO(ent_coef=0.0, clip_range_vf=0.2 * scale, normalize_advantage=False, vf_coef=0.7)):
                cfg = OO.PPOConfig(ent_coef=alg.ent_coef, clip_range_vf=alg.clip_range_vf, normalize_advantage=alg.normalize_advantage,
                                   vf_coef=alg.vf_coef)
                a_in = adv if alg.normalize_advantage or B == 1 else (adv * scale).astype(f32)
                if B == 1 and alg.normalize_advantage:
                    continue                      # std of one sample is NaN in the reference as well
                loss, stats, g = p.loss_grad(obs, actions, a_in, ret, old_lp, old_v, alg.hyper())
                eloss, estats, eg = OO.ppo_loss_and_grads(spec, flat, obs, actions, a_in, ret, old_lp, old_v, cfg)
                assert abs(loss - eloss) <= 1e-4 * max(1.0, abs(eloss)), (name, scale, loss, eloss)
                for k in estats:
                    assert abs(stats[k] - estats[k]) <= 1e-4 * max(1.0, abs(estats[k])), (k, stats[k], estats[k])
                assert _relerr(g, eg) < 1e-4, (name, scale, _relerr(g, eg))
            p.close()
    finally:
        D.set_option("ft", 1)


FTG = {
    "pendulum": lambda: SPECS["pendulum"](),                                                        # [128,128,64], Box(1): BASELINE config C3
    "cartpole64": lambda: SPECS["cartpole"](),                                                      # [64,64] through the general kernel (option ftg = 2)
    "wide_discrete": lambda: OP.PolicySpec(10, [128, 128], "discrete", 2, act_start=0),
    "mixed_box2": lambda: OP.PolicySpec(6, [64, 128, 64], "continuous", 2, act_low=[-1, -1], act_high=[1, 1]),
    "narrow_then_wide": lambda: OP.PolicySpec(15, [64, 128], "discrete", 1, act_start=3),
    "three_64": lambda: OP.PolicySpec(3, [64, 64, 64], "continuous", 1, act_low=[-2], act_high=[2]),
}


@pytest.mark.parametrize("name", list(FTG))
def test_general_tcgen05_kernel_vs_oracle(D, name):
    """update_ftg.cuh: the features-on-lanes tcgen05 kernel for two or three hidden layers of width 64 / 128, Discrete(<= 2) or
    Box(<= 2) actions: loss, statistics and gradients against the oracle on ragged tile counts, many tiles per CTA, large
    return scales (the per-pass delta scale) and both loss configurations."""
    spec = FTG[name]()
    D.set_option("ftg", 2)
    try:
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
                assert abs(loss - eloss) <= 1e-4 * max(1.0, abs(eloss)), (name, B, loss, eloss)
                for k in estats:
                    assert abs(stats[k] - estats[k]) <= 1e-4 * max(1.0, abs(estats[k])), (name, B, k, stats[k], estats[k])
                assert _relerr(g, eg) < 1e-4, (name, B, scale, _relerr(g, eg))
        p.close()
    finally:
        D.set_option("ftg", 1)


def test_c3_shape_update_vs_oracle(D):
    """BASELINE config C3 at reduced env count (Pendulum, [128,128,64], NormalizeWrapperEnv): one epoch of the update through the
    general tcgen05 kernel + fused tail against the oracle on the same buffer and the same Feistel minibatches."""
    n, T = 1024, 32
    env, oenv, spec = _mk(D, "pendulum", n, 5, 200, False, True)
    flat = OP.init_params(spec, seed=2)
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=spec.hidden)
    alg = D.PPO(n_steps=T, batch_size=T * n // 4, epochs=2, ent_coef=0.01)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
    agent.set_parameters(flat)
    assert agent.device.update_path() == "tensor"
    buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
    D.collect_rollout(buf, agent, alg, env)
    ob = {k: buf.download(k) for k in ("obs", "actions", "rewards", "values", "logprobs", "advantages", "returns")}
    import ctypes as C
    from dril_b200 import _lib as L
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
