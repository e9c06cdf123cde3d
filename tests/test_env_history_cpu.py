"""Observation history in the fp32 oracle (oracle/env_history.py), checked against an independent NumPy restatement built from
a plain oracle run: oldest-first order, reset padding, the terminal stack of a truncated step and the post-reset stack, for all
five kinds, k = 1 .. 4, with and without velocity masking.  Also: masked columns and Scaling of the kept components, the
observation-space bounds and widths of the Python env, the new C entry point across the header, the Python library and the
Julia shim, and the frozen fixtures."""
import os
import re

import numpy as np
import pytest

from oracle import env_history as EH, env_params as EP, envs as OE

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
f32 = np.float32
KINDS = ("cartpole", "pendulum", "mountaincar", "mountaincar_continuous", "acrobot")
MAX_STEPS = {"cartpole": 9, "pendulum": 7, "mountaincar": 8, "mountaincar_continuous": 6, "acrobot": 8}
WIDTHS = {"cartpole": ((4, 8, 12, 16), (2, 4, 6, 8)), "pendulum": ((3, 6, 9, 12), (2, 4, 6, 8)),
          "mountaincar": ((2, 4, 6, 8), (1, 2, 3, 4)), "mountaincar_continuous": ((2, 4, 6, 8), (1, 2, 3, 4)),
          "acrobot": ((6, 12, 18, 24), (4, 8, 12, 16))}


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


def _restated_stacks(frames, done, tobs_frames, k):
    """stacks from a plain run's per-step frames (T + 1, n, F), done flags (T, n) and terminal frames (T, n, F) alone: the
    episode's frames so far, last k, padded at the front with the episode's first frame"""
    T1, n, F = frames.shape
    obs = np.zeros((T1, n, k * F), f32)
    term = np.zeros((T1 - 1, n, k * F), f32)
    for i in range(n):
        ep = [frames[0, i]]
        for t in range(T1):
            last = ep[-k:]
            obs[t, i] = np.concatenate([last[0]] * (k - len(last)) + last)
            if t == T1 - 1:
                break
            if done[t, i]:
                fin = (ep + [tobs_frames[t, i]])[-k:]
                term[t, i] = np.concatenate([fin[0]] * (k - len(fin)) + fin)
                ep = [frames[t + 1, i]]
            else:
                ep.append(frames[t + 1, i])
    return obs, term


@pytest.mark.parametrize("mask", [False, True])
@pytest.mark.parametrize("k", [1, 2, 3, 4])
@pytest.mark.parametrize("kind", KINDS)
def test_history_matches_restatement(kind, k, mask):
    rng = np.random.default_rng(1)
    n, T = 12, 40
    lo, hi = _ranges(kind, n, rng)
    plain = OE.ParallelEnv(EP.PARAM_BATCHES[kind](n, seed=4, max_steps=MAX_STEPS[kind], param_ranges=(lo, hi)))
    hist = OE.ParallelEnv(EH.make(kind, n, k, mask, seed=4, max_steps=MAX_STEPS[kind], param_ranges=(lo, hi)))
    cols = list(EH.VELOCITY_FREE[kind]) if mask else list(range(EH.BASE_OBS_DIM[kind]))
    frames, done, tf, trunc, got, got_term = [plain.observe()[:, cols]], [], [], [], [hist.observe()], []
    for _ in range(T):
        a = _actions(kind, rng, n)
        r0, te0, tr0, i0 = plain.act(a)
        r1, te1, tr1, i1 = hist.act(a)
        np.testing.assert_array_equal(r0, r1)
        np.testing.assert_array_equal(te0, te1)
        np.testing.assert_array_equal(tr0, tr1)
        done.append(te0 | tr0)
        trunc.append(tr0)
        z = np.zeros((n, len(cols)), f32)
        tf.append(i0["terminal_observation"][:, cols] if tr0.any() else z)
        got_term.append(i1["terminal_observation"] if tr1.any() else np.zeros((n, k * len(cols)), f32))
        frames.append(plain.observe()[:, cols])
        got.append(hist.observe())
    done, trunc = np.array(done), np.array(trunc)
    assert trunc.any()
    obs, term = _restated_stacks(np.array(frames), done, np.array(tf), k)
    got, got_term = np.array(got), np.array(got_term)
    assert got.shape == (T + 1, n, EH.history_obs_dim(kind, k, mask)) == (T + 1, n, WIDTHS[kind][mask][k - 1])
    np.testing.assert_array_equal(got, obs)
    np.testing.assert_array_equal(got_term[trunc], term[trunc])
    # post-reset stacks are k copies of the reset frame; the newest frame is always the plain observation
    F = len(cols)
    for t, i in zip(*np.nonzero(done)):
        np.testing.assert_array_equal(got[t + 1, i], np.tile(got[t + 1, i, -F:], k))
    np.testing.assert_array_equal(got[..., -F:], np.array(frames))


def test_observe_does_not_move_history():
    b = EH.make("cartpole", 4, 3, seed=1)
    b.step(np.array([1, 2, 1, 2]))
    o = b.obs()
    np.testing.assert_array_equal(b.obs(), o)
    np.testing.assert_array_equal(b.obs(), o)
    b.restart()
    np.testing.assert_array_equal(b.obs(), np.tile(o[:, -4:], 3))


@pytest.mark.parametrize("kind", KINDS)
def test_masked_columns(kind):
    n = 8
    full = EH.make(kind, n, 1, False, seed=3)
    masked = EH.make(kind, n, 1, True, seed=3)
    rng = np.random.default_rng(2)
    keep = {"cartpole": [0, 2], "pendulum": [0, 1], "mountaincar": [0], "mountaincar_continuous": [0], "acrobot": [0, 1, 2, 3]}
    for _ in range(5):
        np.testing.assert_array_equal(masked.obs(), full.obs()[:, keep[kind]])
        a = _actions(kind, rng, n)
        full.step(a)
        masked.step(a)


@pytest.mark.parametrize("kind,sc", [("pendulum", (OE.PENDULUM_OBS_LOW, OE.PENDULUM_OBS_HIGH)),
                                     ("mountaincar_continuous", (np.array([-1.2, -0.07], f32), np.array([0.6, 0.07], f32)))])
def test_scaling_maps_kept_components(kind, sc):
    n, k = 8, 2
    rng = np.random.default_rng(5)
    b = EH.make(kind, n, k, True, seed=2, scaling=sc)
    plain = EP.PARAM_BATCHES[kind](n, seed=2)
    cols = list(EH.VELOCITY_FREE[kind])
    lo, hi = sc[0][cols], sc[1][cols]
    prev = None
    for _ in range(6):
        raw = np.asarray(plain.obs(), f32)[:, cols]
        want = (((raw - lo).astype(f32) * (f32(2.0) / (hi - lo)).astype(f32)).astype(f32) - f32(1.0)).astype(f32)
        o = b.obs()
        np.testing.assert_array_equal(o[:, -len(cols):], want)
        if prev is not None:
            np.testing.assert_array_equal(o[:, :len(cols)], prev)
        prev = want
        a = rng.uniform(-1, 1, (n, 1)).astype(f32)
        b.step(a)
        plain.step(b.b.unscale_action(a))


@pytest.mark.parametrize("mask", [False, True])
@pytest.mark.parametrize("kind", KINDS)
def test_observation_space_bounds(kind, mask):
    from dril_b200 import core
    from dril_b200.spaces import Box
    base = {"cartpole": np.array([4.8, np.inf, 0.41887903, np.inf], f32), "pendulum": np.array([1, 1, 8], f32),
            "mountaincar": np.array([0.6, 0.07], f32), "mountaincar_continuous": np.array([0.6, 0.07], f32),
            "acrobot": np.array([1, 1, 1, 1, 4 * np.pi, 9 * np.pi], f32)}[kind]
    space = Box(-base, base)
    assert core.VELOCITY_FREE == EH.VELOCITY_FREE and core.MAX_HISTORY == EH.MAX_HISTORY
    cols = list(EH.VELOCITY_FREE[kind]) if mask else list(range(len(base)))
    for k in range(1, 5):
        sp = core.observation_space_with_history(space, kind, k, mask)
        assert sp.size() == (WIDTHS[kind][mask][k - 1],)
        np.testing.assert_array_equal(sp.high, np.tile(base[cols], k))
        np.testing.assert_array_equal(sp.low, -np.tile(base[cols], k))
    # every width is at most 24, and the tcgen05 kernels' 15-column limit splits them as documented
    assert max(w for ws in WIDTHS[kind] for w in ws) <= 24


def test_entry_point_agrees():
    hdr = open(os.path.join(ROOT, "include", "dril_b200.h")).read()
    from dril_b200 import _lib as L
    jl = open(os.path.join(ROOT, "julia", "DRiLB200.jl")).read()
    name = "dril_env_set_obs_history"
    m = re.search(r"int32_t " + name + r"\(([^)]*)\);", hdr)
    assert m
    n_args = len(m.group(1).split(","))
    assert n_args == 3 and len(L.PROTOTYPES[name]) == n_args
    jm = re.search(r"ccall\(\(:" + name + r", LIB\), Int32, \(([^)]*)\)", jl)
    assert jm and len([x for x in jm.group(1).split(",") if x.strip()]) == n_args
    assert re.search(r"#define DRIL_ENV_MAX_HISTORY 4\b", hdr)


@pytest.mark.parametrize("kind", KINDS)
def test_frozen_history_replay_fixtures(kind):
    """tests/golden/orc_<kind>_history_replay.npz"""
    g = np.load(os.path.join(ROOT, "tests", "golden", f"orc_{kind}_history_replay.npz"))
    n, k, mask = g["obs"].shape[1], int(g["history_len"]), bool(g["mask_velocities"])
    sc = (OE.PENDULUM_OBS_LOW, OE.PENDULUM_OBS_HIGH) if bool(g["scaling"]) else None
    env = OE.ParallelEnv(EH.make(kind, n, k, mask, seed=int(g["seed"]), max_steps=int(g["max_steps"]),
                                 param_ranges=(g["lo"], g["hi"]), scaling=sc))
    np.testing.assert_array_equal(env.observe(), g["obs"][0])
    for t, a in enumerate(g["actions"]):
        r, te, tr, info = env.act(a)
        np.testing.assert_array_equal(r, g["rewards"][t])
        np.testing.assert_array_equal(te, g["term"][t])
        np.testing.assert_array_equal(tr, g["trunc"][t])
        for i in np.nonzero(tr)[0]:
            np.testing.assert_array_equal(info["terminal_observation"][i], g["terminal_obs"][t][i])
        np.testing.assert_array_equal(env.observe(), g["obs"][t + 1])
    assert g["obs"].shape[2] == EH.history_obs_dim(kind, k, mask)
    assert g["trunc"].any() and (g["lo"] < g["hi"]).any()
    if kind == "cartpole":
        assert g["term"].any()
