"""Parameter-augmented observations in the fp32 oracle (oracle/env_obs_params.py): the observation is the base observation
followed by the running episode's parameter values, the terminal observation carries the ended episode's values and the
post-reset observation the new draw, mid-episode range changes, sharding, constant columns under the normaliser, Scaling of the
base components only, the observation space of the Python env, the new C entry points across the header, the Python library
and the Julia shim, and the frozen fixtures."""
import os
import re

import numpy as np
import pytest

from oracle import env_obs_params as EOP, env_params as EP, envs as OE

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
f32 = np.float32
KINDS = ("cartpole", "pendulum", "mountaincar", "mountaincar_continuous", "acrobot")
D0 = {"cartpole": 4, "pendulum": 3, "mountaincar": 2, "mountaincar_continuous": 2, "acrobot": 6}


def _ranges(kind, n, rng, spread=0.5):
    d = np.array([v for _, v in EP.ENV_PARAMS[kind]], dtype=np.float64)[:, None]
    a, b = d * rng.uniform(1 - spread, 1 + spread, (2, len(d), n))
    lo, hi = np.minimum(a, b).astype(f32), np.maximum(a, b).astype(f32)
    hi[:, ::5] = lo[:, ::5]
    return lo, hi


def _actions(kind, rng, n):
    if kind == "cartpole":
        return rng.integers(1, 3, n)
    if kind in ("mountaincar", "acrobot"):
        return rng.integers(1, 4, n)
    return rng.uniform(-2.5, 2.5, (n, 1)).astype(f32)


def test_widths():
    assert {k: EOP.obs_params_dim(k) for k in KINDS} == {"cartpole": 10, "pendulum": 7, "mountaincar": 4,
                                                         "mountaincar_continuous": 4, "acrobot": 12}
    assert max(EOP.obs_params_dim(k) for k in KINDS) <= 15     # FTG_MAX_OBS: the tcgen05 kernels take every width


@pytest.mark.parametrize("kind", KINDS)
def test_observation_is_base_then_values(kind):
    rng = np.random.default_rng(1)
    n = 24
    lo, hi = _ranges(kind, n, rng)
    plain = EP.PARAM_BATCHES[kind](n, seed=3, max_steps=9, param_ranges=(lo, hi))
    aug = EOP.make(kind, n, seed=3, max_steps=9, param_ranges=(lo, hi))
    for _ in range(30):
        o = aug.obs()
        assert o.dtype == f32 and o.shape == (n, EOP.obs_params_dim(kind))
        np.testing.assert_array_equal(o[:, :D0[kind]], plain.obs())
        np.testing.assert_array_equal(o[:, D0[kind]:], plain.p.T)
        a = _actions(kind, rng, n)
        np.testing.assert_array_equal(aug.step(a), plain.step(a))
        done = np.nonzero(aug.terminated | aug.truncated)[0]
        aug.reset_idx(done)
        plain.reset_idx(done)


@pytest.mark.parametrize("kind", KINDS)
def test_terminal_observation_has_the_ended_episode_and_reset_the_new_draw(kind):
    rng = np.random.default_rng(2)
    n = 40
    lo, hi = _ranges(kind, n, rng)
    env = OE.ParallelEnv(EOP.make(kind, n, seed=4, max_steps=6, param_ranges=(lo, hi)))
    seen = 0
    for _ in range(20):
        before = env.b.p.copy()
        _, term, trunc, info = env.act(_actions(kind, rng, n))
        after = env.observe()[:, D0[kind]:]
        for i in np.nonzero(trunc)[0]:
            np.testing.assert_array_equal(info["terminal_observation"][i, D0[kind]:], before[:, i])
            seen += 1
        done = term | trunc
        np.testing.assert_array_equal(after[~done], before.T[~done])
        np.testing.assert_array_equal(after, env.b.p.T)
        exp = EP.env_param_values(env.b.gid, env.b.episode - 1, lo, hi, 4)
        np.testing.assert_array_equal(after, exp.T)          # the new episode's own (gid, e) draw
        redrawn = done & (lo < hi).all(0)
        if redrawn.any():
            assert (after[redrawn] != before.T[redrawn]).any()
    assert seen > n


def test_no_ranges_observes_the_defaults():
    aug = EOP.make("acrobot", 8, seed=1)
    d = np.array([v for _, v in EP.ENV_PARAMS["acrobot"]], dtype=f32)
    np.testing.assert_array_equal(aug.obs()[:, 6:], np.broadcast_to(d, (8, 6)))
    plain = EP.PARAM_BATCHES["acrobot"](8, seed=1)
    np.testing.assert_array_equal(aug.obs()[:, :6], plain.obs())


def test_mid_episode_ranges():
    rng = np.random.default_rng(3)
    n = 32
    aug = EOP.make("cartpole", n, seed=1)
    aug.reset_idx(np.arange(0, n, 2))
    lo, hi = _ranges("cartpole", n, rng)
    aug.set_param_ranges(lo, hi)
    np.testing.assert_array_equal(aug.obs()[:, 4:], EP.env_param_values(aug.gid, aug.episode - 1, lo, hi, 1).T)


@pytest.mark.parametrize("kind", ("cartpole", "acrobot", "pendulum"))
def test_sharding_invariant(kind):
    rng = np.random.default_rng(4)
    m = 24
    lo, hi = _ranges(kind, 2 * m, rng)
    whole = OE.ParallelEnv(EOP.make(kind, 2 * m, seed=2, max_steps=7, param_ranges=(lo, hi)))
    parts = [OE.ParallelEnv(EOP.make(kind, m, seed=2, max_steps=7, gid_offset=m * i,
                                     param_ranges=(lo[:, m * i:m * (i + 1)], hi[:, m * i:m * (i + 1)]))) for i in range(2)]
    for _ in range(20):
        np.testing.assert_array_equal(whole.observe(), np.concatenate([p.observe() for p in parts]))
        a = _actions(kind, rng, 2 * m)
        whole.act(a)
        for i, p in enumerate(parts):
            p.act(a[m * i:m * (i + 1)])


def _device_moments(cols, order):
    """the batch moments as the rollout kernels form them: fp64 sums and sums of squares of the fp32 values (in any order),
    mean = s / N and var = max(q / N - mean^2, 0) in fp64, then rounded to fp32 (csrc/rollout.cuh reduce_and_merge)"""
    x = cols[:, order].astype(np.float64)
    n = x.shape[1]
    s, q = np.zeros(x.shape[0]), np.zeros(x.shape[0])
    for i in range(n):
        s += x[:, i]
        q += x[:, i] * x[:, i]
    bm = s / n
    return bm.astype(f32), np.maximum(q / n - bm * bm, 0.0).astype(f32)


@pytest.mark.parametrize("n", (7, 64, 301))
def test_constant_columns_normalise_to_zero(n):
    """lo == hi everywhere for gravity and tau: from the first update on, the device's statistics of those columns are the
    value itself with variance 0, so they normalise to exactly 0 (every partial sum k * c of an fp32 value is exact in fp64)"""
    rng = np.random.default_rng(5)
    lo, hi = _ranges("cartpole", n, rng)
    for k in (0, 5):
        lo[k] = hi[k] = f32(rng.uniform(0.5, 2.0)) * lo[k, 0]
    env = OE.ParallelEnv(EOP.make("cartpole", n, seed=3, max_steps=8, param_ranges=(lo, hi)))
    rms = OE.RunningMeanStd((10,))
    norm = OE.NormalizeWrapper(env, 10)
    for _ in range(10):
        o = env.observe()
        rms.update_from_moments(*_device_moments(o.T, rng.permutation(n)), n)
        norm.obs_rms = rms
        x = norm.normalize_obs(o)
        assert (x[:, [4, 9]] == 0).all()
        assert (x[:, [6, 7]] != 0).any()
        env.act(rng.integers(1, 3, n))


def test_scaling_maps_base_components_only():
    rng = np.random.default_rng(6)
    n = 16
    lo, hi = _ranges("pendulum", n, rng)
    sc = (OE.PENDULUM_OBS_LOW, OE.PENDULUM_OBS_HIGH)
    aug = EOP.make("pendulum", n, seed=2, param_ranges=(lo, hi), scaling=sc)
    plain = OE.ScalingBatch(EP.PARAM_BATCHES["pendulum"](n, seed=2, param_ranges=(lo, hi)), *sc)
    for _ in range(12):
        o = aug.obs()
        assert o.shape == (n, 7)
        np.testing.assert_array_equal(o[:, :3], plain.obs())
        np.testing.assert_array_equal(o[:, 3:], plain.p.T)
        a = rng.uniform(-1, 1, (n, 1)).astype(f32)
        aug.step(a)
        plain.step(a)


@pytest.mark.parametrize("kind", KINDS)
def test_frozen_obs_param_replay_fixtures(kind):
    """tests/golden/orc_<kind>_obs_params_replay.npz"""
    g = np.load(os.path.join(ROOT, "tests", "golden", f"orc_{kind}_obs_params_replay.npz"))
    n = g["obs"].shape[1]
    env = OE.ParallelEnv(EOP.make(kind, n, seed=int(g["seed"]), max_steps=int(g["max_steps"]), param_ranges=(g["lo"], g["hi"])))
    np.testing.assert_array_equal(env.observe(), g["obs"][0])
    for t, a in enumerate(g["actions"]):
        r, te, tr, info = env.act(a)
        np.testing.assert_array_equal(r, g["rewards"][t])
        np.testing.assert_array_equal(te, g["term"][t])
        np.testing.assert_array_equal(tr, g["trunc"][t])
        for i in np.nonzero(tr)[0]:
            np.testing.assert_array_equal(info["terminal_observation"][i], g["terminal_obs"][t][i])
        np.testing.assert_array_equal(env.observe(), g["obs"][t + 1])
        np.testing.assert_array_equal(env.observe()[:, D0[kind]:], g["params"][t + 1].T)
    assert g["obs"].shape[2] == EOP.obs_params_dim(kind)
    assert g["trunc"].any() and (g["lo"] < g["hi"]).any() and (g["lo"] == g["hi"]).any()
    if kind == "cartpole":
        assert g["term"].any()


@pytest.mark.parametrize("kind", KINDS)
def test_observation_space_bounds(kind):
    from dril_b200 import core
    from dril_b200.spaces import Box
    base = {"cartpole": Box(-np.array([4.8, np.inf, 0.41887903, np.inf], f32), np.array([4.8, np.inf, 0.41887903, np.inf], f32)),
            "pendulum": Box(OE.PENDULUM_OBS_LOW, OE.PENDULUM_OBS_HIGH),
            "mountaincar": Box(np.array([-1.2, -0.07], f32), np.array([0.6, 0.07], f32)),
            "mountaincar_continuous": Box(-np.ones(2, f32), np.ones(2, f32)),    # as ScalingWrapperEnv leaves it
            "acrobot": Box(-np.ones(6, f32), np.ones(6, f32))}[kind]
    sp = core.observation_space_with_params(base, kind)
    P = len(EP.ENV_PARAMS[kind])
    assert sp.size() == (D0[kind] + P,)
    np.testing.assert_array_equal(sp.low[:D0[kind]], base.low)
    np.testing.assert_array_equal(sp.high[:D0[kind]], base.high)
    assert (sp.low[D0[kind]:] == 0).all() and np.isposinf(sp.high[D0[kind]:]).all()
    # every valid range lies inside: the space does not depend on the ranges
    lo, hi = _ranges(kind, 8, np.random.default_rng(7))
    assert ((lo.T >= sp.low[D0[kind]:]) & (hi.T <= sp.high[D0[kind]:])).all()


def test_entry_points_agree():
    hdr = open(os.path.join(ROOT, "include", "dril_b200.h")).read()
    from dril_b200 import _lib as L
    jl = open(os.path.join(ROOT, "julia", "DRiLB200.jl")).read()
    for name in ("dril_env_set_observe_params", "dril_env_obs_dim"):
        m = re.search(r"int32_t " + name + r"\(([^)]*)\);", hdr)
        assert m, name
        n_args = len(m.group(1).split(","))
        assert len(L.PROTOTYPES[name]) == n_args, name
        jm = re.search(r"ccall\(\(:" + name + r", LIB\), Int32, \(([^)]*)\)", jl)
        assert jm, name
        assert len([x for x in jm.group(1).split(",") if x.strip()]) == n_args, name
