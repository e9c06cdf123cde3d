"""Per-env physical parameters in the fp32 oracle (oracle/env_params.py): single steps with non-default parameters against an
independent float64 restatement of the Gymnasium equations, bit-identity with the unparametrised batches at the default
values, the draw rule (inside the range, lo == hi exact, fixed for an episode, redrawn only at a reset, sharding
invariant), validation, the frozen fixtures, and the parameter tables of the header, the Python package and the Julia shim."""
import os
import re

import numpy as np
import pytest

from oracle import env_params as EP, envs as OE
from oracle.classic_envs import AcrobotBatch, MountainCarBatch, MountainCarContinuousBatch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
f32 = np.float32
KINDS = ("cartpole", "pendulum", "mountaincar", "mountaincar_continuous", "acrobot")
PLAIN = {"cartpole": OE.CartPoleBatch, "pendulum": OE.PendulumBatch, "mountaincar": MountainCarBatch,
         "mountaincar_continuous": MountainCarContinuousBatch, "acrobot": AcrobotBatch}


def _ranges(kind, n, rng, spread=0.5):
    d = np.array([v for _, v in EP.ENV_PARAMS[kind]], dtype=np.float64)[:, None]
    a, b = d * rng.uniform(1 - spread, 1 + spread, (2, len(d), n))
    return np.minimum(a, b).astype(f32), np.maximum(a, b).astype(f32)


def _actions(kind, rng, n):
    if kind == "cartpole":
        return rng.integers(1, 3, n)
    if kind in ("mountaincar", "acrobot"):
        return rng.integers(1, 4, n)
    return rng.uniform(-2.5, 2.5, (n, 1)).astype(f32)


# ---- float64 restatement (Gymnasium classic_control with the parameters as attributes, written independently) --------------
def step64(kind, s, a, p):
    s = [np.asarray(x, np.float64) for x in s]
    p = [np.asarray(x, np.float64) for x in p]
    if kind == "cartpole":
        gravity, masscart, masspole, length, force_mag, tau = p
        x, x_dot, th, th_dot = s
        total_mass = masspole + masscart
        pml = masspole * length
        force = np.where(a - 1 == 1, force_mag, -force_mag)
        temp = (force + pml * th_dot ** 2 * np.sin(th)) / total_mass
        thetaacc = (gravity * np.sin(th) - np.cos(th) * temp) / (length * (4.0 / 3.0 - masspole * np.cos(th) ** 2 / total_mass))
        xacc = temp - pml * thetaacc * np.cos(th) / total_mass
        return np.stack([x + tau * x_dot, x_dot + tau * xacc, th + tau * th_dot, th_dot + tau * thetaacc])
    if kind == "pendulum":
        g, m, l, dt = p
        th, thdot = s
        u = np.clip(a.reshape(-1).astype(np.float64), -2.0, 2.0)
        newthdot = np.clip(thdot + (3 * g / (2 * l) * np.sin(th) + 3.0 / (m * l ** 2) * u) * dt, -8.0, 8.0)
        return np.stack([th + newthdot * dt, newthdot])
    if kind in ("mountaincar", "mountaincar_continuous"):
        pos, vel = s
        if kind == "mountaincar":
            force, gravity = p
            vel = vel + (a - 2) * force + np.cos(3 * pos) * (-gravity)
        else:
            power, gravity = p
            vel = vel + np.clip(a.reshape(-1).astype(np.float64), -1.0, 1.0) * power - gravity * np.cos(3 * pos)
        vel = np.clip(vel, -0.07, 0.07)
        pos = np.clip(pos + vel, -1.2, 0.6)
        vel = np.where((pos == -1.2) & (vel < 0), 0.0, vel)
        return np.stack([pos, vel])
    l1, m1, m2, lc1, lc2, I = p
    g, torque = 9.8, (a - 2).astype(np.float64)

    def dsdt(y):
        th1, th2, w1, w2 = y
        d1 = m1 * lc1 ** 2 + m2 * (l1 ** 2 + lc2 ** 2 + 2 * l1 * lc2 * np.cos(th2)) + I + I
        d2 = m2 * (lc2 ** 2 + l1 * lc2 * np.cos(th2)) + I
        phi2 = m2 * lc2 * g * np.cos(th1 + th2 - np.pi / 2.0)
        phi1 = (-m2 * l1 * lc2 * w2 ** 2 * np.sin(th2) - 2 * m2 * l1 * lc2 * w2 * w1 * np.sin(th2)
                + (m1 * lc1 + m2 * l1) * g * np.cos(th1 - np.pi / 2) + phi2)
        al2 = (torque + d2 / d1 * phi1 - m2 * l1 * lc2 * w1 ** 2 * np.sin(th2) - phi2) / (m2 * lc2 ** 2 + I - d2 ** 2 / d1)
        al1 = -(d2 * al2 + phi1) / d1
        return np.stack([w1, w2, al1, al2])

    y0 = np.stack(s)
    k1 = dsdt(y0)
    k2 = dsdt(y0 + 0.1 * k1)
    k3 = dsdt(y0 + 0.1 * k2)
    k4 = dsdt(y0 + 0.2 * k3)
    return y0 + 0.2 / 6.0 * (k1 + 2 * k2 + 2 * k3 + k4)   # (no wrap / clip reached from the states used here)


def _states(kind, rng, n):
    if kind == "cartpole":
        return rng.uniform(-0.2, 0.2, (4, n)).astype(f32)
    if kind == "pendulum":
        return np.stack([rng.uniform(-np.pi, np.pi, n), rng.uniform(-4, 4, n)]).astype(f32)
    if kind in ("mountaincar", "mountaincar_continuous"):
        return np.stack([rng.uniform(-1.1, 0.4, n), rng.uniform(-0.03, 0.03, n)]).astype(f32)
    return np.stack([rng.uniform(-1, 1, n), rng.uniform(-1, 1, n), rng.uniform(-3, 3, n), rng.uniform(-6, 6, n)]).astype(f32)


@pytest.mark.parametrize("kind", KINDS)
def test_nondefault_step_matches_float64(kind):
    rng = np.random.default_rng(11)
    n = 2048
    lo, hi = _ranges(kind, n, rng)
    b = EP.PARAM_BATCHES[kind](n, seed=3, param_ranges=(lo, hi))
    assert not np.array_equal(b.p, EP.default_ranges(kind, n)[0])
    b.state = _states(kind, rng, n)
    s0, p0 = b.state.copy(), b.p.copy()
    a = _actions(kind, rng, n)
    b.step(a)
    ref = step64(kind, s0, np.asarray(a), p0)
    np.testing.assert_allclose(b.state, ref, rtol=2e-5, atol=2e-6 if kind != "acrobot" else 2e-5)


@pytest.mark.parametrize("kind", KINDS)
def test_defaults_bit_identical_to_unparametrised(kind):
    """at the default values every derived coefficient equals the folded constant, so whole replays with resets agree bit
    for bit"""
    rng = np.random.default_rng(12)
    n, steps = 64, 120
    env_p = OE.ParallelEnv(EP.PARAM_BATCHES[kind](n, seed=9, max_steps=40, param_ranges=EP.default_ranges(kind, n)))
    env_0 = OE.ParallelEnv(PLAIN[kind](n, seed=9, max_steps=40))
    for _ in range(steps):
        a = _actions(kind, rng, n)
        r_p, te_p, tr_p, _ = env_p.act(a)
        r_0, te_0, tr_0, _ = env_0.act(a)
        np.testing.assert_array_equal(r_p, r_0)
        np.testing.assert_array_equal(te_p, te_0)
        np.testing.assert_array_equal(tr_p, tr_0)
        np.testing.assert_array_equal(env_p.b.state, env_0.b.state)
        np.testing.assert_array_equal(env_p.observe(), env_0.observe())
    assert env_0.b.episode.max() > 1


def test_acrobot_coefficients_at_defaults_are_the_folded_constants():
    C = EP.AcrobotParamBatch.coef([f32(v) for _, v in EP.ENV_PARAMS["acrobot"]])
    want = dict(a1=0.25, p=1.25, k=1.0, m2=1.0, i=1.0, l2=0.25, q=0.5, h=0.5, h2=1.0, j=1.25)
    for k, v in want.items():
        assert C[k] == f32(v), k
    assert C["g_lc2"] == AcrobotBatch.G_LC2 and C["g_12"] == AcrobotBatch.G_12
    assert float(AcrobotBatch.G_12) == 14.7000007629394531


@pytest.mark.parametrize("kind", KINDS)
def test_draw_rule(kind):
    rng = np.random.default_rng(13)
    n = 256
    lo, hi = _ranges(kind, n, rng)
    hi[:, ::3] = lo[:, ::3]
    env = OE.ParallelEnv(EP.PARAM_BATCHES[kind](n, seed=4, max_steps=15, param_ranges=(lo, hi)))
    b = env.b
    redrawn = 0
    for t in range(60):
        assert ((b.p >= lo) & (b.p <= hi)).all()
        np.testing.assert_array_equal(b.p[:, ::3], lo[:, ::3])
        before, ep_before = b.p.copy(), b.episode.copy()
        env.act(_actions(kind, rng, n))
        reset = b.episode != ep_before
        np.testing.assert_array_equal(b.p[:, ~reset], before[:, ~reset])      # fixed for an episode
        changed = (b.p != before).any(axis=0)
        assert not (changed & ~reset).any()
        redrawn += int(changed.sum())
    assert redrawn > n
    # a pure function of (seed, gid, episode, range)
    np.testing.assert_array_equal(b.p, EP.env_param_values(b.gid, b.episode - 1, lo, hi, 4))


@pytest.mark.parametrize("kind", ("cartpole", "acrobot"))
def test_draws_are_sharding_invariant(kind):
    rng = np.random.default_rng(14)
    m = 32
    lo, hi = _ranges(kind, 2 * m, rng)
    whole = EP.PARAM_BATCHES[kind](2 * m, seed=2, param_ranges=(lo, hi))
    a = EP.PARAM_BATCHES[kind](m, seed=2, gid_offset=0, param_ranges=(lo[:, :m], hi[:, :m]))
    b = EP.PARAM_BATCHES[kind](m, seed=2, gid_offset=m, param_ranges=(lo[:, m:], hi[:, m:]))
    np.testing.assert_array_equal(whole.p, np.concatenate([a.p, b.p], axis=1))


def test_set_ranges_mid_episode_draws_the_running_episode():
    rng = np.random.default_rng(15)
    n = 32
    b = EP.CartPoleParamBatch(n, seed=1, param_ranges=EP.default_ranges("cartpole", n))
    b.reset_idx(np.arange(0, n, 2))
    lo, hi = _ranges("cartpole", n, rng)
    b.set_param_ranges(lo, hi)
    np.testing.assert_array_equal(b.p, EP.env_param_values(b.gid, b.episode - 1, lo, hi, 1))
    b2 = EP.CartPoleParamBatch(n, seed=1, param_ranges=(lo, hi))
    b2.reset_idx(np.arange(0, n, 2))
    np.testing.assert_array_equal(b.p, b2.p)


@pytest.mark.parametrize("kind,name,bad", [
    ("cartpole", "length", 0.0), ("cartpole", "masspole", -0.1), ("cartpole", "tau", np.nan), ("cartpole", "gravity", -1.0),
    ("pendulum", "dt", 0.0), ("pendulum", "l", np.inf), ("mountaincar", "force", -1e-3), ("mountaincar_continuous", "power", np.nan),
    ("acrobot", "link_moi", 0.0), ("acrobot", "link_com_pos_2", -0.5)])
def test_invalid_values_rejected(kind, name, bad):
    lo, hi = EP.default_ranges(kind, 4)
    k = [nm for nm, _ in EP.ENV_PARAMS[kind]].index(name)
    lo[k, 1] = bad
    with pytest.raises(ValueError):
        EP.check_ranges(kind, lo, np.maximum(hi, lo) if np.isfinite(bad) else hi)
    lo, hi = EP.default_ranges(kind, 4)
    hi[k, 2] = lo[k, 2] * f32(0.5)   # lo > hi
    with pytest.raises(ValueError):
        EP.check_ranges(kind, lo, hi)
    lo, hi = EP.default_ranges(kind, 4)
    zero_ok = name not in EP.POSITIVE
    lo[k] = 0.0
    if zero_ok:
        EP.check_ranges(kind, lo, hi)
    else:
        with pytest.raises(ValueError):
            EP.check_ranges(kind, lo, hi)


def _header_params():
    hdr = open(os.path.join(ROOT, "include", "dril_b200.h")).read()
    out = {}
    for m in re.finditer(r"^ \*   (\w+)\s+(\d+):(.*)$", hdr, re.M):
        kind, count, rest = m.group(1), int(m.group(2)), m.group(3).strip()
        pairs = tuple((nm, float(v)) for nm, v in re.findall(r"(\w+) ([-+0-9.e]+)", rest))
        assert len(pairs) == count, kind
        out[kind] = pairs
    return out


def test_parameter_tables_agree_with_env_defaults():
    from dril_b200 import core
    hdr = _header_params()
    assert set(hdr) == set(core.ENV_KINDS)
    for kind in core.ENV_KINDS:
        assert tuple((nm, float(v)) for nm, v in core.ENV_PARAMS[kind]) == hdr[kind], kind
        assert tuple((nm, float(v)) for nm, v in EP.ENV_PARAMS[kind]) == hdr[kind], kind
    assert re.search(r"#define DRIL_ENV_MAX_PARAMS 8\b", open(os.path.join(ROOT, "include", "dril_b200.h")).read())
    assert max(len(v) for v in hdr.values()) <= 8
    # the defaults and counts in the library
    env = open(os.path.join(ROOT, "dril.jl_b200", "csrc", "env.cuh")).read()
    m = re.search(r"k_env_param_default\[6\] = \{(.*?\})\};", env, re.S)
    rows = re.findall(r"\{([^{}]*)\}", m.group(1))
    assert len(rows) == len(core.ENV_KINDS)
    by_id = {v: k for k, v in core.ENV_KINDS.items()}
    for i, row in enumerate(rows):
        vals = [float(x.rstrip("f")) for x in re.findall(r"[-0-9.e]+f", row)]
        assert vals == [v for _, v in hdr[by_id[i]]], by_id[i]
    # Julia
    src = open(os.path.join(ROOT, "julia", "DRiLB200.jl")).read()
    m = re.search(r"const ENV_PARAMS = Dict\((.*?)\n\)\n", src, re.S)
    jl = {}
    for km in re.finditer(r":(\w+)\s*=>\s*\((.*?)\),?\s*$", m.group(1), re.M):
        jl[km.group(1)] = tuple((nm, float(v)) for nm, v in re.findall(r":(\w+)\s*=>\s*([-+0-9.e]+)", km.group(2)))
    assert jl == hdr


@pytest.mark.parametrize("kind", KINDS)
def test_frozen_param_replay_fixtures(kind):
    """tests/golden/orc_<kind>_params_replay.npz: a later edit of the oracle that changes these results is caught here"""
    g = np.load(os.path.join(ROOT, "tests", "golden", f"orc_{kind}_params_replay.npz"))
    n = g["obs"].shape[1]
    env = OE.ParallelEnv(EP.PARAM_BATCHES[kind](n, seed=int(g["seed"]), max_steps=int(g["max_steps"]), param_ranges=(g["lo"], g["hi"])))
    np.testing.assert_array_equal(env.observe(), g["obs"][0])
    np.testing.assert_array_equal(env.b.p, g["params"][0])
    for t, a in enumerate(g["actions"]):
        r, te, tr, info = env.act(a)
        np.testing.assert_array_equal(r, g["rewards"][t])
        np.testing.assert_array_equal(te, g["term"][t])
        np.testing.assert_array_equal(tr, g["trunc"][t])
        for i in np.nonzero(tr)[0]:
            np.testing.assert_array_equal(info["terminal_observation"][i], g["terminal_obs"][t][i])
        np.testing.assert_array_equal(env.observe(), g["obs"][t + 1])
        np.testing.assert_array_equal(env.b.p, g["params"][t + 1])
    assert g["trunc"].any() and (g["lo"] < g["hi"]).any() and (g["lo"] == g["hi"]).any()
