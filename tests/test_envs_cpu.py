"""MountainCar, MountainCarContinuous and Acrobot in the fp32 oracle (oracle/classic_envs.py), checked against an independent float64
restatement of the Gymnasium equations one step at a time from shared states (Acrobot is chaotic: trajectories diverge, single
steps do not), against closed-form cases, and the env-kind tables of the header, the Python package and the Julia shim."""
import os
import re

import numpy as np
import pytest

from oracle import classic_envs as CE, envs as OE

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
f32 = np.float32
N = 4096


# ---- float64 restatement (Gymnasium classic_control, written independently of the oracle) ----------------------------------
def mc_step64(pos, vel, force, power, goal):
    vel = np.clip(vel + force * power + np.cos(3 * pos) * (-0.0025), -0.07, 0.07)
    pos = np.clip(pos + vel, -1.2, 0.6)
    vel = np.where((pos == -1.2) & (vel < 0), 0.0, vel)
    return pos, vel, (pos >= goal) & (vel >= 0)


def acrobot_dsdt64(s, a):
    m1 = m2 = l1 = 1.0
    lc1 = lc2 = 0.5
    I1 = I2 = 1.0
    g = 9.8
    th1, th2, w1, w2 = s
    d1 = m1 * lc1 ** 2 + m2 * (l1 ** 2 + lc2 ** 2 + 2 * l1 * lc2 * np.cos(th2)) + I1 + I2
    d2 = m2 * (lc2 ** 2 + l1 * lc2 * np.cos(th2)) + I2
    phi2 = m2 * lc2 * g * np.cos(th1 + th2 - np.pi / 2.0)
    phi1 = (-m2 * l1 * lc2 * w2 ** 2 * np.sin(th2) - 2 * m2 * l1 * lc2 * w2 * w1 * np.sin(th2)
            + (m1 * lc1 + m2 * l1) * g * np.cos(th1 - np.pi / 2) + phi2)
    al2 = (a + d2 / d1 * phi1 - m2 * l1 * lc2 * w1 ** 2 * np.sin(th2) - phi2) / (m2 * lc2 ** 2 + I2 - d2 ** 2 / d1)
    al1 = -(d2 * al2 + phi1) / d1
    return np.stack([w1, w2, al1, al2])


def acrobot_rk4_64(s, a, dt=0.2):
    k1 = acrobot_dsdt64(s, a)
    k2 = acrobot_dsdt64(s + dt / 2 * k1, a)
    k3 = acrobot_dsdt64(s + dt / 2 * k2, a)
    k4 = acrobot_dsdt64(s + dt * k3, a)
    return s + dt / 6.0 * (k1 + 2 * k2 + 2 * k3 + k4)


def wrap64(x):
    return (x + np.pi) % (2 * np.pi) - np.pi


def _states_mc(rng):
    return rng.uniform(-1.2, 0.6, N).astype(f32), rng.uniform(-0.07, 0.07, N).astype(f32)


# ---- oracle vs float64 ---------------------------------------------------------------------------------------------------
def test_mountaincar_step_vs_float64():
    rng = np.random.default_rng(0)
    env = CE.MountainCarBatch(N, seed=1)
    pos, vel = _states_mc(rng)
    acts = rng.integers(1, 4, N)
    env.state = np.stack([pos, vel])
    r = env.step(acts)
    p64, v64, t64 = mc_step64(pos.astype(np.float64), vel.astype(np.float64), (acts - 2).astype(np.float64), 0.001, 0.5)
    np.testing.assert_allclose(env.state[0], p64, rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(env.state[1], v64, rtol=1e-5, atol=1e-7)
    clear = np.abs(p64 - 0.5) > 1e-5
    assert (env.terminated[clear] == t64[clear]).all()
    assert (r == -1).all() and r.dtype == f32


def test_mountaincar_continuous_step_vs_float64():
    rng = np.random.default_rng(1)
    env = CE.MountainCarContinuousBatch(N, seed=1)
    pos, vel = _states_mc(rng)
    acts = rng.uniform(-1.5, 1.5, N).astype(f32)          # outside [-1, 1] too: clipped for the force, not for the reward
    env.state = np.stack([pos, vel])
    r = env.step(acts)
    a64 = acts.astype(np.float64)
    p64, v64, t64 = mc_step64(pos.astype(np.float64), vel.astype(np.float64), np.clip(a64, -1, 1), 0.0015, 0.45)
    np.testing.assert_allclose(env.state[0], p64, rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(env.state[1], v64, rtol=1e-5, atol=1e-7)
    clear = np.abs(p64 - 0.45) > 1e-5
    assert (env.terminated[clear] == t64[clear]).all()
    np.testing.assert_allclose(r, np.where(env.terminated, 100.0, 0.0) - 0.1 * a64 ** 2, rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("vscale,tol", [(0.5, 1e-5), (1.0, 1e-3)])
def test_acrobot_step_vs_float64(vscale, tol):
    """Relative error (components below 1 in absolute terms) of one fp32 RK4 step.  With velocities up to half their bounds it
    stays below 1e-5; near the bounds the omega^2 terms (~800) cancel and fp32 rounding of them reaches ~2e-4."""
    rng = np.random.default_rng(2)
    s = np.stack([rng.uniform(-np.pi, np.pi, N), rng.uniform(-np.pi, np.pi, N),
                  rng.uniform(-4 * np.pi, 4 * np.pi, N) * vscale, rng.uniform(-9 * np.pi, 9 * np.pi, N) * vscale]).astype(f32)
    acts = rng.integers(1, 4, N)
    env = CE.AcrobotBatch(N, seed=1)
    env.state = s.copy()
    r = env.step(acts)
    ns = acrobot_rk4_64(s.astype(np.float64), (acts - 2).astype(np.float64))
    ns[2] = np.clip(ns[2], -4 * np.pi, 4 * np.pi)
    ns[3] = np.clip(ns[3], -9 * np.pi, 9 * np.pi)
    d = env.state.astype(np.float64) - ns
    d[:2] = wrap64(d[:2])                                   # the fp64 angles are not wrapped (and a wrap at +-pi may differ)
    assert (np.abs(d) / np.maximum(np.abs(ns), 1.0)).max() <= tol
    assert (np.abs(env.state[:2]) <= np.float32(np.pi)).all()
    th1, th2 = env.state[0].astype(np.float64), env.state[1].astype(np.float64)
    h = -np.cos(th1) - np.cos(th2 + th1)
    clear = np.abs(h - 1.0) > 1e-5
    assert (env.terminated[clear] == (h > 1.0)[clear]).all()
    assert (r == np.where(env.terminated, 0.0, -1.0)).all()
    obs = env.obs()
    np.testing.assert_allclose(obs, np.stack([np.cos(th1), np.sin(th1), np.cos(th2), np.sin(th2), env.state[2], env.state[3]], 1),
                               rtol=0, atol=1e-7)


# ---- closed-form cases ----------------------------------------------------------------------------------------------------
def _mc_dv(pos, idx):
    _, c = OE._sincos32(f32(3.0) * np.array([pos], f32))
    return (f32(idx - 1) * f32(0.001)) + (c[0] * -f32(0.0025))


def test_mountaincar_left_wall():
    env = CE.MountainCarBatch(1)
    env.state = np.array([[-1.19], [-0.05]], f32)
    env.step([1])                                           # push left into the wall
    assert env.state[0, 0] == f32(-1.2) and env.state[1, 0] == 0.0
    assert not env.terminated[0]


def test_mountaincar_goal_exact():
    for vel_extra, want in ((f32(0.0), True), (f32(-1e-4), False)):
        env = CE.MountainCarBatch(1)
        env.state = np.array([[0.5], [-_mc_dv(0.5, 1) + vel_extra]], f32)   # action 2 (no push): velocity lands on 0 exactly
        env.step([2])
        if want:
            assert env.state[0, 0] == f32(0.5) and env.state[1, 0] == 0.0
        else:
            assert env.state[1, 0] < 0
        assert bool(env.terminated[0]) is want


def test_mountaincar_continuous_goal_reward():
    a = f32(0.7)
    _, c = OE._sincos32(f32(3.0) * np.array([0.45], f32))
    dv = (a * f32(0.0015)) - (f32(0.0025) * c[0])
    env = CE.MountainCarContinuousBatch(1)
    env.state = np.array([[0.45], [-dv]], f32)
    r = env.step(np.array([[a]], f32))
    assert env.terminated[0] and env.state[0, 0] == f32(0.45) and env.state[1, 0] == 0.0
    assert r[0] == f32(100.0) - (a * a) * f32(0.1)
    np.testing.assert_allclose(r[0], 100 - 0.1 * 0.7 ** 2, rtol=1e-6)
    # off the goal: only the control cost
    env.state = np.array([[-0.5], [0.0]], f32)
    r = env.step(np.array([[-2.0]], f32))
    assert not env.terminated[0] and r[0] == -(f32(4.0) * f32(0.1))


def test_acrobot_rest_stays_at_rest():
    env = CE.AcrobotBatch(1)
    env.state = np.zeros((4, 1), f32)
    for _ in range(20):
        r = env.step([2])                                   # torque 0
        assert r[0] == -1 and not env.terminated[0]
    assert np.abs(env.state).max() < 1e-5                   # cos(fp32(-pi/2)) is -4.4e-8, not 0: fp32 noise only


@pytest.mark.parametrize("th1,th2,want", [(np.pi, 0.0, True), (0.0, 0.0, False), (np.pi / 2, 0.0, False),
                                          (np.pi, 0.5, True), (2.3, -0.2, True), (1.2, 0.1, False)])
def test_acrobot_terminal_test(th1, th2, want):
    s = np.array([[th1], [th2], [0.0], [0.0]], f32)
    ns, term = CE.AcrobotBatch.advance(s, np.zeros(1, f32))
    h = -np.cos(np.float64(ns[0, 0])) - np.cos(np.float64(ns[1, 0]) + np.float64(ns[0, 0]))
    assert bool(term[0]) == (h > 1.0) == want


def test_acrobot_wrap_at_pi():
    s = np.array([[3.1, -3.1], [-3.1, 3.1], [5.0, -5.0], [-5.0, 5.0]], f32)
    ns, _ = CE.AcrobotBatch.advance(s, np.zeros(2, f32))
    unwrapped = acrobot_rk4_64(s.astype(np.float64), np.zeros(2))
    assert unwrapped[0, 0] > np.pi and unwrapped[0, 1] < -np.pi and unwrapped[1, 0] < -np.pi and unwrapped[1, 1] > np.pi
    assert (np.abs(ns[:2]) <= f32(np.pi)).all()
    np.testing.assert_allclose(ns[:2], wrap64(unwrapped[:2]), atol=1e-5)


def test_acrobot_velocity_clips():
    s = np.array([[0.0, 0.0], [0.0, 0.0], [4 * np.pi, -4 * np.pi], [9 * np.pi, -9 * np.pi]], f32)
    ns, _ = CE.AcrobotBatch.advance(s, np.array([1.0, -1.0], f32))
    unclipped = acrobot_rk4_64(s.astype(np.float64), np.array([1.0, -1.0]))
    assert np.abs(ns[2]).max() <= f32(4 * np.pi) and np.abs(ns[3]).max() <= f32(9 * np.pi)
    for k, lim in ((2, f32(4 * np.pi)), (3, f32(9 * np.pi))):
        over = np.abs(unclipped[k]) > lim
        assert over.any()
        assert (np.abs(ns[k][over]) == lim).all()


def test_reset_distributions():
    mc = CE.MountainCarBatch(N, seed=3)
    assert (mc.state[0] >= -0.6).all() and (mc.state[0] < -0.4).all() and (mc.state[1] == 0).all()
    ac = CE.AcrobotBatch(N, seed=3)
    assert (np.abs(ac.state) <= 0.1).all() and ac.state.std() > 0.05
    mc2 = CE.MountainCarBatch(N, seed=3)
    np.testing.assert_array_equal(mc.state, mc2.state)      # Philox stream: same seed, same resets


def test_wrappers_accept_new_batches():
    """ParallelEnv / Monitor / Normalize / Scaling wrap the new batches unchanged; truncation at the default TimeLimit."""
    rng = np.random.default_rng(4)
    for batch, steps in ((CE.MountainCarBatch(8), 200), (CE.AcrobotBatch(8), 500)):
        env = OE.NormalizeWrapper(OE.MonitorWrapper(OE.ParallelEnv(batch)), batch.obs_dim)
        env.reset()
        for t in range(steps):
            env.observe()
            _, term, trunc, info = env.act(rng.integers(1, 4, 8))
        assert trunc.any() or term.any()
    sb = OE.ScalingBatch(CE.MountainCarContinuousBatch(8), CE.MOUNTAINCAR_OBS_LOW, CE.MOUNTAINCAR_OBS_HIGH)
    env = OE.MonitorWrapper(OE.ParallelEnv(sb))
    env.reset()
    o = env.observe()
    assert o.shape == (8, 2) and (np.abs(o) <= 1).all()
    for _ in range(999):
        _, _, trunc, _ = env.act(rng.uniform(-1, 1, (8, 1)).astype(f32))
    assert trunc.all()


# ---- spaces, defaults and the kind tables ------------------------------------------------------------------------------
def test_oracle_spaces_and_defaults():
    mc, mcc, ac = CE.MountainCarBatch(2), CE.MountainCarContinuousBatch(2), CE.AcrobotBatch(2)
    assert (mc.obs_dim, mc.act_kind, mc.n_actions, mc.max_steps, mc.act_start) == (2, "discrete", 3, 200, 1)
    assert (mcc.obs_dim, mcc.act_kind, mcc.act_dim, mcc.max_steps) == (2, "continuous", 1, 999)
    assert (mcc.act_low[0], mcc.act_high[0]) == (-1.0, 1.0)
    assert (ac.obs_dim, ac.act_kind, ac.n_actions, ac.max_steps, ac.act_start) == (6, "discrete", 3, 500, 1)
    assert mc.obs().shape == (2, 2) and ac.obs().shape == (2, 6)
    np.testing.assert_array_equal(CE.MOUNTAINCAR_OBS_LOW, f32([-1.2, -0.07]))
    np.testing.assert_array_equal(CE.MOUNTAINCAR_OBS_HIGH, f32([0.6, 0.07]))
    np.testing.assert_array_equal(CE.ACROBOT_OBS_HIGH, f32([1, 1, 1, 1, 4 * np.pi, 9 * np.pi]))
    np.testing.assert_array_equal(CE.ACROBOT_OBS_LOW, -CE.ACROBOT_OBS_HIGH)


def test_spaces_module_builds_the_new_spaces():
    from dril_b200.spaces import Box, Discrete
    d = Discrete(3, 1)
    assert d.n == 3 and d.start == 1
    b = Box(CE.ACROBOT_OBS_LOW, CE.ACROBOT_OBS_HIGH)
    assert tuple(b.size()) == (6,)


def _header_kinds():
    hdr = open(os.path.join(ROOT, "include", "dril_b200.h")).read()
    return {m.group(1).lower(): int(m.group(2)) for m in re.finditer(r"DRIL_ENV_([A-Z_]+)\s*=\s*(\d+)", hdr)}


def test_env_kind_tables_agree():
    from dril_b200 import core
    hdr = _header_kinds()
    assert hdr == core.ENV_KINDS
    assert set(core.ENV_STATE_DIMS) == set(hdr)
    assert (core.ENV_STATE_DIMS["mountaincar"], core.ENV_STATE_DIMS["mountaincar_continuous"], core.ENV_STATE_DIMS["acrobot"]) == (2, 2, 4)
    src = open(os.path.join(ROOT, "julia", "DRiLB200.jl")).read()
    m = re.search(r"const ENV_KINDS = Dict\((.*?)\)\n", src)
    jl = {k: int(v) for k, v in re.findall(r":(\w+)\s*=>\s*(\d+)", m.group(1))}
    assert jl == hdr
    for kind in ("mountaincar", "mountaincar_continuous", "acrobot"):
        assert f"kind == :{kind}" in src


@pytest.mark.parametrize("kind,cls", [("mountaincar", CE.MountainCarBatch), ("mountaincar_continuous", CE.MountainCarContinuousBatch),
                                      ("acrobot", CE.AcrobotBatch)])
def test_frozen_replay_fixtures(kind, cls):
    """tests/golden/orc_<kind>_replay.npz: a later edit of the oracle that changes these envs' results is caught here"""
    g = np.load(os.path.join(ROOT, "tests", "golden", f"orc_{kind}_replay.npz"))
    env = OE.ParallelEnv(cls(g["obs"].shape[1], seed=int(g["seed"]), max_steps=int(g["max_steps"])))
    np.testing.assert_array_equal(env.observe(), g["obs"][0])
    for t, a in enumerate(g["actions"]):
        r, te, tr, info = env.act(a)
        np.testing.assert_array_equal(r, g["rewards"][t])
        np.testing.assert_array_equal(te, g["term"][t])
        np.testing.assert_array_equal(tr, g["trunc"][t])
        for i in np.nonzero(tr)[0]:
            np.testing.assert_array_equal(info["terminal_observation"][i], g["terminal_obs"][t][i])
        np.testing.assert_array_equal(env.observe(), g["obs"][t + 1])
    assert g["trunc"].any()
