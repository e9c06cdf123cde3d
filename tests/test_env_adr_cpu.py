"""Automatic domain randomisation, CPU side: the oracle's update rule on hand-built scenarios, attribution across host resets and
episodes that span rounds, the boundary assignment over many envs, configuration validation, and the Julia binding's ccalls."""
import os
import re

import numpy as np
import pytest

from oracle import env_adr as EA, env_params as EP

f32 = np.float32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LEN = EA.AdrParam(3, 0.5, 0.6, 0.1, 0.8, 0.25)        # cartpole length
MP = EA.AdrParam(2, 0.1, 0.1, 0.05, 0.2, 0.02)        # cartpole masspole


def _decide(params, lo, hi, sums, counts, m=4, t=(10.0, 20.0)):
    return EA.decide(params, np.array(lo, f32), np.array(hi, f32), np.array(sums, float), np.array(counts, np.int64), m, *t)


def test_update_widen_narrow_and_clamp():
    # low side widens (mean 25 >= 20), high side narrows (mean 5 <= 10)
    lo, hi, s, c = _decide([LEN], [0.5], [0.7], [100.0, 20.0], [4, 4])
    assert lo[0] == f32(f32(0.5) - f32(0.25)) and hi[0] == f32(0.6)           # hi clamped at init_hi, not 0.45
    assert (s == 0).all() and (c == 0).all()
    # widening clamps at the limits
    lo, hi, _, _ = _decide([LEN], [0.2], [0.7], [100.0, 100.0], [4, 4])
    assert lo[0] == f32(0.1) and hi[0] == f32(0.8)
    # narrowing clamps at the initial range
    lo, hi, _, _ = _decide([LEN], [0.4], [0.8], [0.0, 0.0], [4, 4])
    assert lo[0] == f32(0.5) and hi[0] == f32(0.6)
    lo, hi, _, _ = _decide([EA.AdrParam(3, 0.5, 0.6, 0.1, 2.0, 0.25)], [0.1], [1.5], [0.0, 0.0], [4, 4])
    assert lo[0] == f32(f32(0.1) + f32(0.25)) and hi[0] == f32(f32(1.5) - f32(0.25))
    # between the thresholds: nothing moves, the buffer still restarts
    lo, hi, s, c = _decide([LEN], [0.4], [0.7], [60.0, 60.0], [4, 4])
    assert lo[0] == f32(0.4) and hi[0] == f32(0.7) and (c == 0).all() and (s == 0).all()


def test_update_below_buffer_size_and_two_parameters():
    lo, hi, s, c = _decide([LEN, MP], [0.5, 0.1], [0.6, 0.1], [100.0, 3.0, 200.0, 0.0], [3, 1, 5, 4])
    assert lo[0] == f32(0.5) and hi[0] == f32(0.6)                          # below m: untouched, kept
    np.testing.assert_array_equal(s[:2], [100.0, 3.0])
    np.testing.assert_array_equal(c[:2], [3, 1])
    assert lo[1] == f32(f32(0.1) - f32(0.02)) and hi[1] == f32(0.1)         # mean 40 widens, mean 0 narrows at init
    assert c[2] == 0 and c[3] == 0
    # fp32 subtraction and addition, rounded once
    lo, hi, _, _ = _decide([MP], [0.1], [0.1], [1e3, 1e3], [4, 4])
    assert lo[0] == f32(0.1) - f32(0.02) and hi[0] == f32(0.1) + f32(0.02)


def test_update_accumulates_until_m():
    a = EA.Adr("cartpole", [LEN], 0.5, 4, 10.0, 20.0, seed=1, gid=np.arange(8))
    a.update(np.array([50.0, 0.0]), np.array([2, 0]))
    assert a.counts[0] == 2 and a.lo[0] == f32(0.5)
    a.update(np.array([50.0, 0.0]), np.array([2, 0]))
    assert a.counts[0] == 0 and a.lo[0] == f32(0.25) and a.round == 2


class _Counters:
    """just the reset counters of a batch"""

    def __init__(self, n):
        self.n = n
        self.episode = np.ones(n, dtype=np.int64)


def test_attribution_spanning_rounds_and_host_resets():
    n, T = 4, 6
    a = EA.Adr("cartpole", [LEN], 1.0, 1, 10.0, 20.0, seed=3, gid=np.arange(n))   # every env a boundary env
    b = _Counters(n)
    a.ep_mark, a.run_slot = b.episode.copy(), a.slots(0)
    s0 = a.slots(0)
    # round 0: env 0 ends two episodes, env 1 none, env 2 one, env 3 none
    done = np.zeros((T, n), bool)
    done[1, 0] = done[4, 0] = done[2, 2] = True
    r = np.zeros((T, n), f32)
    r[1, 0], r[4, 0], r[2, 2] = 5.0, 7.0, 11.0
    b.episode += done.sum(0)
    sums, counts = a.scan(done, r, b.episode)
    exp = np.zeros(2)
    np.add.at(exp, [s0[0], s0[0], s0[2]], [5.0, 7.0, 11.0])
    np.testing.assert_array_equal(sums, exp)
    assert counts.sum() == 3
    np.testing.assert_array_equal(a.run_slot, s0)        # envs 0, 2 started round-0 episodes; 1, 3 still run their first
    a.round = 1
    s1 = a.slots(1)
    # between rounds: host reset of every env (those episodes end outside a rollout: not counted), then env 1's new episode
    # ends in round 1, and env 3 (reset too) ends one
    b.episode += 1
    done = np.zeros((T, n), bool)
    done[0, 1] = done[3, 3] = True
    r = np.zeros((T, n), f32)
    r[0, 1], r[3, 3] = 2.0, 3.0
    b.episode += done.sum(0)
    sums, counts = a.scan(done, r, b.episode)
    exp = np.zeros(2)
    np.add.at(exp, [s1[1], s1[3]], [2.0, 3.0])           # started by the host reset during round 1: round 1's slots
    np.testing.assert_array_equal(sums, exp)


def test_attribution_episode_spanning_a_round():
    n, T = 3, 4
    a = EA.Adr("cartpole", [LEN, MP], 1.0, 1, 10.0, 20.0, seed=11, gid=np.arange(n))
    b = _Counters(n)
    a.ep_mark, a.run_slot = b.episode.copy(), a.slots(0)
    s0 = a.slots(0)
    a.scan(np.zeros((T, n), bool), np.zeros((T, n), f32), b.episode)     # round 0: nothing ends
    a.round = 1
    done = np.zeros((T, n), bool)
    done[2, :] = True
    r = np.full((T, n), 4.0, f32)
    b.episode += 1
    sums, counts = a.scan(done, r, b.episode)
    exp = np.zeros(4, np.int64)
    np.add.at(exp, s0, 1)                                # the episodes drawn in round 0 count for round 0's slots
    np.testing.assert_array_equal(counts, exp)
    np.testing.assert_array_equal(a.run_slot, a.slots(1))


def test_assignment_fraction_and_uniform_slots():
    n = 400_000
    for p, S in ((0.2, 4), (0.05, 16), (1.0, 2)):
        s = EA.assign(np.arange(n), 7, 12345, p, S)
        frac = (s >= 0).mean()
        assert abs(frac - p) < 4 * np.sqrt(p * (1 - p) / n) + 1e-9, (p, frac)
        cnt = np.bincount(s[s >= 0], minlength=S)
        e = (s >= 0).sum() / S
        chi2 = ((cnt - e) ** 2 / e).sum()
        assert chi2 < S + 6 * np.sqrt(2 * S), (p, S, chi2)
    assert (EA.assign(np.arange(1000), 0, 1, 0.0, 4) == -1).all()
    a, b = EA.assign(np.arange(100), 3, 9, 0.5, 4), EA.assign(np.arange(100), 4, 9, 0.5, 4)
    assert (a != b).any()                                # a new draw every round
    np.testing.assert_array_equal(EA.assign(np.arange(50, 100), 3, 9, 0.5, 4), a[50:])   # a pure function of the gid


def test_config_validation():
    ok = dict(p_boundary=0.2, buffer_size=8, t_low=10.0, t_high=20.0)
    EA.check_config("cartpole", [LEN, MP], **ok)
    bad = [
        ([EA.AdrParam(6, 1, 1, 1, 1, 1)], ok),                          # index out of range
        ([LEN, LEN], ok),                                             # repeated
        ([EA.AdrParam(3, 0.5, 0.6, 0.0, 0.8, 0.1)], ok),                # length must stay > 0
        ([EA.AdrParam(3, 0.5, 0.6, 0.55, 0.8, 0.1)], ok),               # limit_lo > init_lo
        ([EA.AdrParam(3, 0.7, 0.6, 0.1, 0.8, 0.1)], ok),                # init_lo > init_hi
        ([EA.AdrParam(3, 0.5, 0.6, 0.1, 0.8, 0.0)], ok),                # delta 0
        ([EA.AdrParam(3, 0.5, 0.6, 0.1, float("inf"), 0.1)], ok),       # not finite
        ([LEN], dict(ok, p_boundary=1.5)), ([LEN], dict(ok, buffer_size=0)), ([LEN], dict(ok, t_low=20.0)),
        ([], ok),
    ]
    for params, kw in bad:
        with pytest.raises(ValueError):
            EA.check_config("cartpole", params, **kw)
    EA.check_config("cartpole", [EA.AdrParam(0, 9.8, 9.8, 0.0, 12.0, 0.5)], **ok)   # gravity may reach 0
    with pytest.raises(ValueError):
        EA.check_config("cartpole", [LEN], **ok, monitor=False)
    with pytest.raises(ValueError):
        EA.check_config("synthetic", [LEN], **ok)


def test_oracle_ranges_and_attach():
    n = 64
    a = EA.Adr("acrobot", [EA.AdrParam(0, 0.9, 1.1, 0.5, 2.0, 0.1)], 0.5, 4, -400.0, -100.0, seed=5, gid=np.arange(n))
    b = EP.PARAM_BATCHES["acrobot"](n, seed=5)
    a.attach(b)
    s = a.slots()
    assert (s >= 0).any() and (s < 0).any()
    np.testing.assert_array_equal(b.plo[0], np.where(s == 1, f32(1.1), f32(0.9)))
    np.testing.assert_array_equal(b.phi[0], np.where(s == 0, f32(0.9), f32(1.1)))
    np.testing.assert_array_equal(b.plo[1:], b.phi[1:])                 # outside J: the defaults
    assert ((b.p[0] >= b.plo[0]) & (b.p[0] <= b.phi[0])).all()           # running episodes redrawn
    a.detach(b)
    assert (b.plo[0] == f32(0.9)).all() and (b.phi[0] == f32(1.1)).all()


def test_julia_binding_arities():
    src = open(os.path.join(ROOT, "julia", "DRiLB200.jl")).read()
    for sym, arity in (("dril_env_set_adr", 7), ("dril_env_get_adr", 6)):
        m = re.search(r"ccall\(\(:%s, LIB\), Int32,\s*\(([^)]*)\)" % sym, src)
        assert m, f"{sym} is not bound"
        assert len([t for t in m.group(1).split(",") if t.strip()]) == arity, (sym, m.group(1))
    hdr = open(os.path.join(ROOT, "include", "dril_b200.h")).read()
    for sym, arity in (("dril_env_set_adr", 7), ("dril_env_get_adr", 6)):
        m = re.search(r"int32_t %s\(([^)]*)\)" % sym, hdr)
        assert m and len(m.group(1).split(",")) == arity
