"""Pins the oracle against every closed-form / cross-library check the reference's own tests
hold for the hot path (SURVEY §8c). The reference ships no golden files; each case below
re-runs the reference test's scenario (cited file:line under /root/reference/test) through
the oracle. CPU only."""
import numpy as np
import pytest
from scipy import stats as sps

from oracle import envs as E
from oracle import policy as P
from oracle import ppo as O

f32 = np.float32


def expected_gae(rewards, values, gamma, lam, terminated=True, boot=None):
    """test/test_shared_setup.jl:295-318 (independent restatement used by the reference tests)."""
    n = len(rewards)
    out = np.zeros(n)
    out[-1] = rewards[-1] - values[-1] if (terminated or boot is None) else rewards[-1] + gamma * boot - values[-1]
    for t in range(n - 2, -1, -1):
        out[t] = rewards[t] + gamma * values[t + 1] - values[t] + gamma * lam * out[t + 1]
    return out


def test_gae_analytical():
    """test/test_gae.jl:1-71 — rewards [0x7,1], V=0.5, gamma .99, lambda .95, terminated; closed form."""
    r = np.array([0] * 7 + [1], dtype=f32)
    v = np.full(8, 0.5, dtype=f32)
    adv = O.compute_advantages(r, v, True, None, 0.99, 0.95)
    gl = 0.99 * 0.95
    closed = np.zeros(8)
    closed[-1] = 0.5
    for i in range(7):
        closed[i] = -0.005 * ((1 - gl ** (7 - i)) / (1 - gl)) + gl ** (7 - i) * 0.5
    np.testing.assert_allclose(adv, closed, atol=1e-4)
    # time-major scan agrees
    adv2, ret2 = O.gae_timemajor(r[:, None], v[:, None], np.array([[False]] * 7 + [[True]]),
                                 np.zeros((8, 1), bool), np.zeros((8, 1), f32), np.zeros(1, f32), 0.99, 0.95)
    np.testing.assert_allclose(adv2[:, 0], closed, atol=1e-4)
    np.testing.assert_allclose(ret2[:, 0], closed + 0.5, atol=1e-4)


@pytest.mark.parametrize("gamma,lam", [(0.95, 0.9), (0.99, 0.95), (1.0, 1.0), (0.9, 0.0), (0.8, 0.5)])
def test_gae_parametric(gamma, lam):
    """test/test_gae.jl:73-115."""
    r = np.array([0, 0, 0, 1], dtype=f32)
    v = np.full(4, 0.3, dtype=f32)
    np.testing.assert_allclose(O.compute_advantages(r, v, True, None, gamma, lam),
                               expected_gae(r, v, gamma, lam), atol=1e-4)


def test_gae_multi_episode_mc():
    """test/test_gae.jl:176-220 — 4 episodes of 8 steps in one 32-step rollout, gamma=lambda=1, V=0 -> returns 1."""
    T = 32
    r = np.zeros((T, 1), f32)
    term = np.zeros((T, 1), bool)
    r[7::8] = 1
    term[7::8] = True
    adv, ret = O.gae_timemajor(r, np.zeros((T, 1), f32), term, np.zeros((T, 1), bool), np.zeros((T, 1), f32),
                               np.zeros(1, f32), 1.0, 1.0)
    np.testing.assert_allclose(ret, 1.0, atol=1e-6)


def test_gae_edge_cases():
    """test/test_gae.jl:272-322 — 1-step, gamma=0, lambda=0."""
    np.testing.assert_allclose(O.compute_advantages([1.0], [0.3], True, None, 0.99, 0.95), [0.7], atol=1e-6)
    r = np.array([0.5, 0.2, 1.0], f32)
    v = np.array([0.1, 0.4, 0.3], f32)
    np.testing.assert_allclose(O.compute_advantages(r, v, True, None, 0.0, 0.95), r - v, atol=1e-6)
    np.testing.assert_allclose(O.compute_advantages(r, v, True, None, 0.9, 0.0),
                               expected_gae(r, v, 0.9, 0.0), atol=1e-6)


def test_bootstrap_vs_terminated():
    """test/test_buffers.jl:60-115 — gamma .9, lambda .8, V=.7, bootstrap .2."""
    r = np.array([0, 0, 0, 0, 0, 1], f32)
    v = np.full(6, 0.7, f32)
    a_t = O.compute_advantages(r, v, True, None, 0.9, 0.8)
    a_b = O.compute_advantages(r, v, False, 0.2, 0.9, 0.8)
    np.testing.assert_allclose(a_t, expected_gae(r, v, 0.9, 0.8), atol=1e-4)
    np.testing.assert_allclose(a_b, expected_gae(r, v, 0.9, 0.8, terminated=False, boot=0.2), atol=1e-4)
    assert not np.allclose(a_t, a_b, atol=1e-3)
    # terminated wins over a bootstrap value (trajectory.jl:85)
    np.testing.assert_allclose(O.compute_advantages(r, v, True, 0.2, 0.9, 0.8), a_t)
    # time-major equivalents: truncated with boot, and rollout-limited with last_values
    trunc = np.zeros((6, 1), bool); trunc[-1] = True
    boot = np.zeros((6, 1), f32); boot[-1] = 0.2
    adv, _ = O.gae_timemajor(r[:, None], v[:, None], np.zeros((6, 1), bool), trunc, boot, np.zeros(1, f32), 0.9, 0.8)
    np.testing.assert_allclose(adv[:, 0], a_b, atol=1e-6)
    adv, _ = O.gae_timemajor(r[:, None], v[:, None], np.zeros((6, 1), bool), np.zeros((6, 1), bool),
                             np.zeros((6, 1), f32), np.array([0.2], f32), 0.9, 0.8)
    np.testing.assert_allclose(adv[:, 0], a_b, atol=1e-6)


def test_running_mean_std():
    """test/test_normalize_wrapper.jl:3-38 and :40-70."""
    rms = E.RunningMeanStd((3,))
    assert rms.count == 0 and (rms.mean == 0).all() and (rms.var == 1).all()
    b1 = np.array([[1, 2, 3], [4, 5, 6], [7, 8, 9]], f32)
    rms.update(b1)
    assert rms.count == 3
    np.testing.assert_allclose(rms.mean, b1.mean(1), atol=1e-6)
    np.testing.assert_allclose(rms.var, b1.var(1), atol=1e-6)
    b2 = np.array([[0, 1, 2], [3, 4, 5], [6, 7, 8]], f32)
    rms.update(b2)
    comb = np.hstack([b1, b2])
    assert rms.count == 6
    np.testing.assert_allclose(rms.mean, comb.mean(1), atol=1e-5)
    np.testing.assert_allclose(rms.var, comb.var(1), atol=1e-5)
    z = E.RunningMeanStd((2,))
    z.update(np.array([[5, 5, 5], [3, 3, 3]], f32))
    assert z.count == 3 and np.allclose(z.mean, [5, 3]) and (z.var < 1e-6).all()
    s = E.RunningMeanStd((1,))
    s.update(np.array([[42.0]], f32))
    assert s.count == 1 and np.isclose(s.mean[0], 42) and np.isclose(s.var[0], 0)
    sc = E.RunningMeanStd(())
    sc.update(np.array([[1.0, 2.0, 3.0]], f32))
    assert sc.count == 3 and np.isclose(sc.mean, 2.0) and np.isclose(sc.var, np.var([1.0, 2.0, 3.0]))


def test_diag_gaussian_vs_scipy():
    """test/test_distributions.jl:1-39 (Distributions.MvNormal -> scipy)."""
    rng = np.random.default_rng(0)
    for k in (1, 2, 6, 24):
        for _ in range(20):
            mean = rng.uniform(-1, 1, (1, k)).astype(f32)
            log_std = rng.uniform(-1, 1, k).astype(f32)
            x = rng.uniform(-1, 1, (1, k)).astype(f32)
            mvn = sps.multivariate_normal(mean[0].astype(np.float64), np.diag(np.exp(log_std.astype(np.float64)) ** 2))
            np.testing.assert_allclose(P.gaussian_logpdf(mean, log_std, x)[0], mvn.logpdf(x[0]), rtol=2e-5, atol=2e-5)
            np.testing.assert_allclose(P.gaussian_entropy(log_std, 1)[0], mvn.entropy(), rtol=2e-5, atol=2e-5)


def test_categorical_vs_scipy():
    """test/test_distributions.jl:94-118."""
    rng = np.random.default_rng(1)
    for n in (3, 8):
        for _ in range(50):
            p = rng.random(n).astype(f32)
            p = (p / p.sum()).astype(f32)[None]
            np.testing.assert_allclose(P.categorical_logpdf(p, [1], 1)[0], np.log(p[0, 0]), rtol=1e-6)
            np.testing.assert_allclose(P.categorical_entropy(p)[0], sps.entropy(p[0].astype(np.float64)), rtol=1e-5)
    # start-based env-space actions (test/test_policies.jl:237-283: Discrete(5,-2), Discrete(1,0))
    p = np.array([[0.1, 0.2, 0.3, 0.25, 0.15]], f32)
    assert P.categorical_sample(p, np.array([0.05]), -2)[0] == -2
    assert P.categorical_sample(p, np.array([0.999]), -2)[0] == 2
    assert P.categorical_sample(np.array([[1.0]], f32), np.array([0.5]), 0)[0] == 0


def test_normalize_wrapper_semantics():
    """test/test_normalize_wrapper.jl:141-377 — clipping, eval-mode freeze, terminal obs normalised,
    stats updated on every observe (normalizeWrapperEnv.jl:123-137)."""
    env = E.NormalizeWrapper(E.MonitorWrapper(E.ParallelEnv(E.PendulumBatch(8, seed=3, max_steps=5))), 3)
    o0 = env.observe()
    assert env.obs_rms.count == 8
    assert (np.abs(o0) <= 10).all()
    env.observe()
    assert env.obs_rms.count == 16          # duplicate observe counts again
    for t in range(5):
        r, term, trunc, info = env.act(np.zeros((8, 1), f32))
        assert (np.abs(r) <= 10).all()
    assert trunc.all() and not term.any()
    tobs = info["terminal_observation"]
    assert (np.abs(tobs) <= 10).all()
    assert (env.returns == 0).all()         # zeroed on done (:153-156)
    assert env.ret_rms.count == 40
    # eval mode freezes stats (:281-324)
    env.training = False
    c, m = env.obs_rms.count, env.obs_rms.mean.copy()
    env.observe(); env.act(np.zeros((8, 1), f32))
    assert env.obs_rms.count == c and (env.obs_rms.mean == m).all() and env.ret_rms.count == 40
    # round trip (:141-249): unnormalise recovers raw obs when not clipped
    raw = env.old_obs
    n = env.normalize_obs(raw)
    back = n * np.sqrt(env.obs_rms.var + env.epsilon) + env.obs_rms.mean
    np.testing.assert_allclose(back, raw, atol=1e-5)


class _FixedBatch:
    """One env with a fixed observation that records the last action it received (the ObsTestEnv / ActionTestEnv /
    LargeRangeEnv fixtures of test/test_scaling_wrapper.jl)."""
    n = 1

    def __init__(self, obs, act_low, act_high):
        self._obs = np.asarray(obs, dtype=f32)[None]
        self.act_low, self.act_high = np.asarray(act_low, dtype=f32), np.asarray(act_high, dtype=f32)
        self.last_action = None

    def obs(self):
        return self._obs.copy()

    def step(self, actions):
        self.last_action = np.asarray(actions, dtype=f32).reshape(-1)
        return self.last_action[:1].copy()


def test_scaling_wrapper_reference_scenarios():
    """ScalingWrapperEnv pinned by the reference's own closed-form tests (test/test_scaling_wrapper.jl:42-81 observation
    scaling, :83-129 action scaling, :208-238 large ranges, :178-206 zero-width ranges do not raise)."""
    lo, hi = [0.0, -10.0, 5.0], [10.0, 10.0, 25.0]
    for obs, want in (([5.0, 0.0, 15.0], [0, 0, 0]), (lo, [-1, -1, -1]), (hi, [1, 1, 1])):
        w = E.ScalingBatch(_FixedBatch(obs, [-1.0], [1.0]), lo, hi)
        assert np.abs(w.obs()[0] - np.asarray(want, f32)).max() < 1e-6
        assert w.obs().dtype == f32
    b = _FixedBatch([0.0], [2.0, -5.0, 0.0], [8.0, 15.0, 10.0])
    w = E.ScalingBatch(b, [-1.0], [1.0])
    np.testing.assert_array_equal(w.act_low, [-1, -1, -1]); np.testing.assert_array_equal(w.act_high, [1, 1, 1])
    for a, want in (([0, 0, 0], [5, 5, 5]), ([-1, -1, -1], [2, -5, 0]), ([1, 1, 1], [8, 15, 10])):
        w.step(np.asarray(a, f32))
        assert np.abs(b.last_action - np.asarray(want, f32)).max() < 1e-6
    b = _FixedBatch([500.0, 500.0], [-100.0], [300.0])
    w = E.ScalingBatch(b, [-1000.0, -500.0], [2000.0, 1500.0])
    assert np.abs(w.obs()[0]).max() < 1e-5
    assert abs(float(w.step(np.asarray([0.5], f32))[0]) - 200.0) < 1e-5
    w = E.ScalingBatch(_FixedBatch([0.0, -1.0], [5.0], [5.0]), [0.0, -1.0], [0.0, -1.0])       # zero-width ranges: no exception
    with np.errstate(invalid="ignore", divide="ignore"):
        assert w.obs().shape == (1, 2)
        w.step(np.asarray([0.0], f32))
    # Pendulum through the wrapper: scaled obs in [-1, 1]; a scaled action a reaches the env as the torque 2 a
    pb = E.PendulumBatch(6, seed=3)
    w = E.ScalingBatch(pb, E.PENDULUM_OBS_LOW, E.PENDULUM_OBS_HIGH)
    o = w.obs()
    assert (np.abs(o) <= 1 + 1e-6).all() and np.abs(o[:, 2] * 8 - pb.obs()[:, 2]).max() < 1e-5
    pb2 = E.PendulumBatch(6, seed=3)
    a = np.linspace(-1, 1, 6, dtype=f32)[:, None]
    np.testing.assert_allclose(w.step(a), pb2.step(2 * a), rtol=1e-6)


def test_monitor_wrapper():
    """environment_wrappers/monitorWrapperEnv.jl:44-60 — episode r/l on done, 100-deep window."""
    env = E.MonitorWrapper(E.ParallelEnv(E.PendulumBatch(3, seed=1, max_steps=4)), stats_window=5)
    tot = np.zeros(3, f32)
    for t in range(4):
        r, term, trunc, info = env.act(np.ones((3, 1), f32))
        tot += r
    assert trunc.all()
    np.testing.assert_allclose(info["episode_r"], tot, rtol=1e-6)
    assert (info["episode_l"] == 4).all()
    assert len(env.returns) == 3 and (env.ep_len == 0).all()
    for t in range(4):
        env.act(np.ones((3, 1), f32))
    assert len(env.returns) == 5 and env.total_episodes == 6


def test_auto_reset_terminal_observation():
    """multithreadedParallelEnv.jl:56-71 — flags before reset, terminal obs iff truncated, observe is post-reset."""
    b = E.CartPoleBatch(4, seed=0, max_steps=3)
    env = E.ParallelEnv(b)
    for t in range(3):
        r, term, trunc, info = env.act(np.ones(4, np.int64))
    assert trunc.all()
    assert info["terminal_observation"] is not None
    post = env.observe()
    assert (np.abs(post) <= 0.05).all() and (b.steps == 0).all() and (b.episode == 2).all()
    assert not np.allclose(post, info["terminal_observation"])


def test_seeding_reproducible():
    """test/test_env_seeding.jl:56-105 — same seed -> same streams; sub-env i is its own stream."""
    a = E.CartPoleBatch(6, seed=11).obs()
    b = E.CartPoleBatch(6, seed=11).obs()
    c = E.CartPoleBatch(6, seed=12).obs()
    assert (a == b).all() and not (a == c).all()
    assert len({tuple(r) for r in a}) == 6
    # sharding invariance: global env ids give the same streams on any rank split
    d = E.CartPoleBatch(3, seed=11, gid_offset=3).obs()
    assert (d == a[3:]).all()


def test_forward_vs_evaluate_consistency():
    """test/test_policies.jl:101-146 and test/test_buffers.jl:3-27,166-214."""
    for spec, batch in ((P.PolicySpec(4, [64, 64], "discrete", 2, act_start=1), E.CartPoleBatch(16, seed=0)),
                        (P.PolicySpec(3, [32, 16], "continuous", 1, act_low=[-2], act_high=[2]), E.PendulumBatch(16, seed=0))):
        flat = P.init_params(spec, seed=0)
        assert flat.size == spec.n_params()
        buf = O.collect_rollout_timemajor(E.ParallelEnv(batch), spec, flat, 8)
        v, lp, ent = P.evaluate_actions(spec, flat, buf["obs"].reshape(128, -1), buf["actions"].reshape(128, -1))
        np.testing.assert_allclose(v, buf["values"].reshape(-1), atol=1e-6)
        np.testing.assert_allclose(lp, buf["logprobs"].reshape(-1), atol=1e-5)
        if spec.act_kind == "discrete":
            assert set(np.unique(buf["actions"])) <= {1, 2}


def test_param_counts():
    """SURVEY §8 / test/test_policies.jl:36-64."""
    assert P.PolicySpec(4, [64, 64], "discrete", 2).n_params() == 9155
    assert P.PolicySpec(3, [128, 128, 64], "continuous", 1).n_params() == 50691


def test_reference_order_matches_timemajor():
    """rollout_buffer.jl:70-87: the literal per-trajectory buffer equals the time-major buffer
    permuted by reference_order()."""
    spec = P.PolicySpec(4, [16, 16], "discrete", 2, act_start=1)
    flat = P.init_params(spec, seed=2)
    mk = lambda: E.MonitorWrapper(E.ParallelEnv(E.CartPoleBatch(5, seed=4, max_steps=25)))
    ref = O.collect_rollout_reference(mk(), spec, flat, 80, 0.99, 0.95, policy_seed=7)
    buf = O.collect_rollout_timemajor(mk(), spec, flat, 80, policy_seed=7)
    adv, ret = O.gae_timemajor(buf["rewards"], buf["values"], buf["term"], buf["trunc"], buf["boot"],
                               buf["last_values"], 0.99, 0.95)
    order = O.reference_order(buf["term"], buf["trunc"])
    assert sorted(order) == list(range(400))
    assert buf["trunc"].any() and buf["term"].any()
    np.testing.assert_array_equal(ref["obs"], buf["obs"].reshape(400, -1)[order])
    np.testing.assert_array_equal(ref["actions"].reshape(-1), buf["actions"].reshape(-1)[order])
    np.testing.assert_array_equal(ref["rewards"], buf["rewards"].reshape(-1)[order])
    np.testing.assert_allclose(ref["advantages"], adv.reshape(-1)[order], atol=1e-6)
    np.testing.assert_allclose(ref["returns"], ret.reshape(-1)[order], atol=1e-6)
    np.testing.assert_allclose(ref["returns"], ref["advantages"] + ref["values"], atol=1e-6)  # test_buffers.jl:162-163


@pytest.mark.parametrize("kind", ["discrete", "continuous"])
def test_analytic_gradients_vs_torch_autograd(kind):
    """ppo.jl:365-407 restated in torch fp64 with autograd (oracle/ppo64.py) vs the oracle's hand-written backward."""
    from oracle.ppo64 import loss64
    rng = np.random.default_rng(5)
    if kind == "discrete":
        spec = P.PolicySpec(4, [16, 8], "discrete", 3, act_start=0)
        actions = rng.integers(0, 3, (40, 1))
    else:
        spec = P.PolicySpec(3, [16, 8], "continuous", 2, act_low=[-2, -2], act_high=[2, 2])
        actions = rng.normal(size=(40, 2)).astype(f32)
    flat = (P.init_params(spec, seed=1) + rng.normal(size=spec.n_params()).astype(f32) * 0.05).astype(f32)
    obs = rng.normal(size=(40, spec.obs_dim)).astype(f32)
    adv = rng.normal(size=40).astype(f32)
    ret = rng.normal(size=40).astype(f32)
    v0, lp0, _ = P.evaluate_actions(spec, flat, obs, actions)
    old_lp = (lp0 + rng.normal(size=40).astype(f32) * 0.3).astype(f32)
    old_v = (v0 + rng.normal(size=40).astype(f32) * 0.3).astype(f32)
    for cfg in (O.PPOConfig(ent_coef=0.01), O.PPOConfig(ent_coef=0.02, clip_range_vf=0.2, normalize_advantage=False)):
        loss, stats, g = O.ppo_loss_and_grads(spec, flat, obs, actions, adv, ret, old_lp, old_v, cfg)
        tl, tg, tstats = loss64(spec, flat, obs, actions, adv, ret, old_lp, old_v, cfg)
        assert abs(loss - tl) < 1e-5 * max(1, abs(tl))
        np.testing.assert_allclose(g, tg, rtol=2e-4, atol=2e-6)
        for k in ("clip_fraction", "approx_kl_div", "entropy", "ratio"):
            assert abs(stats[k] - tstats[k]) < 1e-5, k


def test_feistel_is_permutation():
    from oracle import philox
    for n in (1, 2, 7, 64, 1000, 524288 // 64):
        keys = philox.feistel_keys(3, 0, 99)
        perm = philox.feistel_permute(np.arange(n), n, keys)
        assert sorted(perm.tolist()) == list(range(n))
    p1 = philox.feistel_permute(np.arange(1000), 1000, philox.feistel_keys(0, 0, 1))
    p2 = philox.feistel_permute(np.arange(1000), 1000, philox.feistel_keys(1, 0, 1))
    assert (p1 != p2).mean() > 0.9 and (p1 != np.arange(1000)).mean() > 0.9


def test_philox_known_answer():
    """Random123 known-answer vectors for philox4x32-10 (kat_vectors: zero counter/key; all-ones; pi digits)."""
    from oracle import philox
    out = philox.philox4x32(0, 0, 0, 0, 0)
    assert [int(x) for x in out] == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    out = philox.philox4x32(0xffffffff, 0xffffffff, 0xffffffff, 0xffffffff, 0xffffffffffffffff)
    assert [int(x) for x in out] == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    out = philox.philox4x32(0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344, (0x299f31d0 << 32) | 0xa4093822)
    assert [int(x) for x in out] == [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


def test_ppo_learns_tracking_proxy():
    """test/test_ppo_integration.jl:1-40 in spirit: the oracle's PPO improves CartPole episode length
    (small budget so the CPU suite stays fast)."""
    spec = P.PolicySpec(4, [32, 32], "discrete", 2, act_start=1)
    flat = P.init_params(spec, seed=0)
    env = E.MonitorWrapper(E.ParallelEnv(E.CartPoleBatch(8, seed=0)))
    cfg = O.PPOConfig(n_steps=128, batch_size=256, epochs=6, learning_rate=1e-3, ent_coef=0.0)
    flat, ls = O.train(env, spec, flat, cfg, 8 * 128 * 14)
    assert np.mean(list(env.lengths)[-20:]) > 40, np.mean(list(env.lengths)[-20:])
    assert all(np.isfinite(ls["losses"]))
