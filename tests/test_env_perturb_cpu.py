"""Observation noise and action delay in the fp32 oracle (oracle/env_perturb.py): the noise is N(0, sigma^2) and uncorrelated
across components, envs and steps, sigma = 0 and d = 0 are the plain batch bit for bit, observe() is idempotent and results do
not depend on sharding, the delayed batch equals the undelayed one driven by the actions chosen d steps earlier (with the
queue's restart padding), the queue restarts where documented, validation, the new C entry points across the header, the
Python library and the Julia shim, and the frozen fixtures."""
import os
import re

import numpy as np
import pytest
from scipy import stats

from oracle import env_history as EH, env_params as EP, env_perturb as PB, envs as OE

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
f32 = np.float32
KINDS = ("cartpole", "pendulum", "mountaincar", "mountaincar_continuous", "acrobot")
MAX_STEPS = {"cartpole": 9, "pendulum": 7, "mountaincar": 8, "mountaincar_continuous": 6, "acrobot": 8}


def _actions(kind, rng, shape):
    if kind == "cartpole":
        return rng.integers(1, 3, shape)
    if kind in ("mountaincar", "acrobot"):
        return rng.integers(1, 4, shape)
    return rng.uniform(-2.5, 2.5, shape + (1,)).astype(f32)


def _ranges(kind, n):
    lo, hi = EP.default_ranges(kind, n)
    return lo * f32(0.8), hi * f32(1.2)


def _run(env, actions):
    """observations, rewards, flags and terminal observations of a ParallelEnv replay"""
    obs, rew, flags, tobs = [env.observe()], [], [], []
    for a in actions:
        r, te, tr, info = env.act(a)
        rew.append(r); flags.append(te.astype(np.uint8) | (tr.astype(np.uint8) << 1))
        tobs.append(np.where(tr[:, None], info["terminal_observation"], 0) if tr.any() else np.zeros_like(obs[0]))
        obs.append(env.observe())
    return np.stack(obs), np.stack(rew), np.stack(flags), np.stack(tobs)


def test_noise_is_standard_normal_and_uncorrelated():
    n, steps = 6000, 3
    zs = np.stack([PB.noise_z(np.arange(n), np.full(n, 7), np.full(n, s), 6, seed=11) for s in range(steps)])   # (S, n, 6)
    flat = zs.astype(np.float64).ravel()
    assert flat.size >= 100_000
    assert stats.kstest(flat, "norm").pvalue > 1e-3
    for j in range(6):   # every component on its own
        assert stats.kstest(zs[..., j].ravel(), "norm").pvalue > 1e-4
    lim = 5 / np.sqrt(n)
    c = np.corrcoef(zs.reshape(-1, 6).T)                                   # across components
    assert np.abs(c - np.eye(6)).max() < lim
    assert abs(np.corrcoef(zs[0, :-1].ravel(), zs[0, 1:].ravel())[0, 1]) < lim    # across neighbouring envs
    assert abs(np.corrcoef(zs[0].ravel(), zs[1].ravel())[0, 1]) < lim             # across steps
    z_other_ep = PB.noise_z(np.arange(n), np.full(n, 8), np.zeros(n), 6, seed=11)  # across episodes
    assert abs(np.corrcoef(zs[0].ravel(), z_other_ep.ravel())[0, 1]) < lim


@pytest.mark.parametrize("kind", KINDS)
def test_noise_scale_through_batch(kind):
    n = 20000
    d0 = PB.BASE_OBS_DIM[kind]
    sigma = np.repeat(np.linspace(0.01, 0.2, d0, dtype=f32)[:, None], n, axis=1)
    clean = EP.PARAM_BATCHES[kind](n, seed=3)
    noisy = PB.PerturbBatch(EP.PARAM_BATCHES[kind](n, seed=3), sigma)
    diff = (noisy.obs().astype(np.float64) - clean.obs()) / sigma.T
    assert stats.kstest(diff.ravel(), "norm").pvalue > 1e-4
    np.testing.assert_array_equal(noisy.state, clean.state)   # the true state is untouched


@pytest.mark.parametrize("history", [(1, False), (3, True)])
@pytest.mark.parametrize("kind", KINDS)
def test_zero_perturbation_is_plain(kind, history):
    n, T = 24, 30
    rng = np.random.default_rng(1)
    acts = _actions(kind, rng, (T, n))
    k, mask = history
    kw = dict(seed=4, max_steps=MAX_STEPS[kind], param_ranges=_ranges(kind, n))
    plain = OE.ParallelEnv(EH.make(kind, n, k, mask, **kw))
    zero = OE.ParallelEnv(PB.make(kind, n, np.zeros((PB.BASE_OBS_DIM[kind], n), f32), np.zeros(n, np.int32), k, mask, **kw))
    for x, y in zip(_run(plain, acts), _run(zero, acts)):
        assert x.tobytes() == y.tobytes()   # bit for bit, -0 included


def test_zero_sigma_keeps_negative_zero():
    o = np.array([[-0.0, 1.0]], f32)
    out = PB.add_noise(o, np.zeros((2, 1), f32), np.ones((1, 2), f32))
    assert np.signbit(out[0, 0])


@pytest.mark.parametrize("kind", KINDS)
def test_observe_idempotent_and_shard_independent(kind):
    n, T = 16, 20
    rng = np.random.default_rng(2)
    sigma = rng.uniform(0, 0.1, (PB.BASE_OBS_DIM[kind], n)).astype(f32)
    delay = np.arange(n) % 5
    acts = _actions(kind, rng, (T, n))
    kw = dict(seed=9, max_steps=MAX_STEPS[kind])
    full = OE.ParallelEnv(PB.make(kind, n, sigma, delay, **kw))
    halves = [OE.ParallelEnv(PB.make(kind, n // 2, sigma[:, s], delay[s], gid_offset=s.start, **kw))
              for s in (slice(0, n // 2), slice(n // 2, n))]
    o1 = full.observe()
    np.testing.assert_array_equal(o1, full.observe())
    np.testing.assert_array_equal(o1, np.concatenate([h.observe() for h in halves]))
    for a in acts:
        r, te, tr, _ = full.act(a)
        parts = [h.act(a[: n // 2] if i == 0 else a[n // 2:]) for i, h in enumerate(halves)]
        np.testing.assert_array_equal(r, np.concatenate([p[0] for p in parts]))
        np.testing.assert_array_equal(full.observe(), np.concatenate([h.observe() for h in halves]))


def _delayed_reference(acts, flags, delay, restarts=()):
    """the actions an undelayed env must receive: a_{max(t - d, t0)}, t0 = the first step since the queue's restart (after a
    done step, and at the steps in `restarts`)"""
    T, n = acts.shape[:2]
    out = np.empty_like(acts)
    t0 = np.zeros(n, np.int64)
    for t in range(T):
        if t in restarts:
            t0[:] = t
        src = np.maximum(t - delay, t0)
        out[t] = acts[src, np.arange(n)]
        t0 = np.where(flags[t] != 0, t + 1, t0)
    return out


@pytest.mark.parametrize("kind", KINDS)
def test_delay_identity(kind):
    n, T = 20, 40
    rng = np.random.default_rng(3)
    delay = np.arange(n) % 5
    acts = _actions(kind, rng, (T, n))
    kw = dict(seed=5, max_steps=MAX_STEPS[kind], param_ranges=_ranges(kind, n))
    delayed = OE.ParallelEnv(PB.make(kind, n, None, delay, **kw))
    obs, rew, flags, tobs = _run(delayed, acts)
    assert (flags != 0).any()
    ref = OE.ParallelEnv(PB.make(kind, n, **kw))
    for x, y in zip((obs, rew, flags, tobs), _run(ref, _delayed_reference(acts, flags, delay))):
        assert x.tobytes() == y.tobytes()


@pytest.mark.parametrize("how", ["reset", "set_state", "new_delays"])
def test_queue_restarts(how):
    kind, n, T, cut = "pendulum", 10, 24, 11
    rng = np.random.default_rng(4)
    delay = np.arange(n) % 5
    acts = _actions(kind, rng, (T, n))
    kw = dict(seed=6, max_steps=50)
    b = PB.make(kind, n, None, delay, **kw)
    env = OE.ParallelEnv(b)
    ref_b = PB.make(kind, n, **kw)
    ref = OE.ParallelEnv(ref_b)
    flags = np.zeros((T, n), np.uint8)
    for t in range(T):
        if t == cut:
            if how == "reset":
                env.reset(); ref.reset()
            elif how == "set_state":
                b.restart_queue()   # the device's dril_env_set_state
            else:
                b.set_action_delay(delay)
        ref_acts = _delayed_reference(acts[: t + 1], flags[: t + 1], delay, restarts=(cut,))
        r, te, tr, _ = env.act(acts[t])
        r2, te2, tr2, _ = ref.act(ref_acts[t])
        flags[t] = te | (tr.astype(np.uint8) << 1)
        np.testing.assert_array_equal(r, r2)
        np.testing.assert_array_equal(env.observe(), ref.observe())


def test_validation():
    n = 4
    with pytest.raises(ValueError):
        PB.check_noise("cartpole", np.zeros((3, n)), n)                    # wrong component count
    with pytest.raises(ValueError):
        PB.check_noise("cartpole", np.full((4, n), -0.1), n)               # negative
    with pytest.raises(ValueError):
        PB.check_noise("acrobot", np.full((6, n), np.nan), n)              # non-finite
    with pytest.raises(ValueError):
        PB.check_noise("pendulum", np.full((3, n), np.inf), n)
    with pytest.raises(ValueError):
        PB.check_delay([0, 1, 5, 2], n)
    with pytest.raises(ValueError):
        PB.check_delay([0, -1, 0, 2], n)
    PB.check_noise("mountaincar", np.zeros((2, n)), n)
    PB.check_delay([0, 4, 3, 2], n)


def test_entry_points_agree():
    hdr = open(os.path.join(ROOT, "include", "dril_b200.h")).read()
    from dril_b200 import _lib as L
    jl = open(os.path.join(ROOT, "julia", "DRiLB200.jl")).read()
    for name, n_args in (("dril_env_set_obs_noise", 3), ("dril_env_set_action_delay", 2)):
        m = re.search(r"int32_t " + name + r"\(([^)]*)\);", hdr)
        assert m and len(m.group(1).split(",")) == n_args and len(L.PROTOTYPES[name]) == n_args
        for jm in re.finditer(r"ccall\(\(:" + name + r", LIB\), Int32, \(([^)]*)\)", jl):
            assert len([x for x in jm.group(1).split(",") if x.strip()]) == n_args
    assert re.search(r"#define DRIL_ENV_MAX_ACTION_DELAY 4\b", hdr)


def replay_fixture(g, kind):
    n = g["obs"].shape[1]
    sc = (OE.PENDULUM_OBS_LOW, OE.PENDULUM_OBS_HIGH) if bool(g["scaling"]) else None
    return OE.ParallelEnv(PB.make(kind, n, g["obs_noise"], g["action_delay"], int(g["history_len"]), bool(g["mask_velocities"]),
                                  seed=int(g["seed"]), max_steps=int(g["max_steps"]), param_ranges=(g["lo"], g["hi"]), scaling=sc))


@pytest.mark.parametrize("kind", KINDS)
def test_frozen_perturb_replay_fixtures(kind):
    """tests/golden/orc_<kind>_perturb_replay.npz"""
    g = np.load(os.path.join(ROOT, "tests", "golden", f"orc_{kind}_perturb_replay.npz"))
    env = replay_fixture(g, kind)
    np.testing.assert_array_equal(env.observe(), g["obs"][0])
    for t, a in enumerate(g["actions"]):
        r, te, tr, info = env.act(a)
        np.testing.assert_array_equal(r, g["rewards"][t])
        np.testing.assert_array_equal(te, g["term"][t])
        np.testing.assert_array_equal(tr, g["trunc"][t])
        for i in np.nonzero(tr)[0]:
            np.testing.assert_array_equal(info["terminal_observation"][i], g["terminal_obs"][t][i])
        np.testing.assert_array_equal(env.observe(), g["obs"][t + 1])
    assert g["trunc"].any() and (g["lo"] < g["hi"]).any()
    assert (g["obs_noise"] == 0).any() and (g["obs_noise"] > 0).any()
    assert set(np.unique(g["action_delay"])) == {0, 1, 2, 3, 4}
    if kind == "cartpole":
        assert g["term"].any()
