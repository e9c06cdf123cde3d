"""CPU checks of the float64 reference's helpers (oracle/ppo64.py) that tests/test_gpu_grad_scale.py relies on: the
parameter-block splitter and the minibatch generator with per-tile gradient magnitudes and branch margins."""
import numpy as np
import pytest

from oracle import policy as OP, ppo as OO
from oracle import ppo64 as O64

f32 = np.float32

# every shape the loss/grad parity tests run (tests/test_gpu_parity.py SPECS / FTG, tests/test_gpu_grad_scale.py PATHS)
SHAPES = [
    OP.PolicySpec(4, [64, 64], "discrete", 2, act_start=1),
    OP.PolicySpec(3, [128, 128, 64], "continuous", 1, act_low=[-2], act_high=[2]),
    OP.PolicySpec(10, [24, 12], "discrete", 5, act_start=-2),
    OP.PolicySpec(7, [32], "continuous", 3, act_low=[-1, -1, -1], act_high=[1, 1, 1]),
    OP.PolicySpec(5, [], "continuous", 1, act_low=[-1], act_high=[1]),
    OP.PolicySpec(10, [128, 128], "discrete", 2, act_start=0),
    OP.PolicySpec(6, [64, 128, 64], "continuous", 2, act_low=[-1, -1], act_high=[1, 1]),
    OP.PolicySpec(15, [64, 128], "discrete", 1, act_start=3),
    OP.PolicySpec(3, [64, 64, 64], "continuous", 1, act_low=[-2], act_high=[2]),
    OP.PolicySpec(6, [64, 64], "discrete", 3, act_start=0),
    OP.PolicySpec(2, [128, 128, 64], "discrete", 3, act_start=0),
    OP.PolicySpec(4, [64, 64], "discrete", 4, act_start=1),
    OP.PolicySpec(5, [128, 128, 64], "discrete", 4, act_start=0),
]


@pytest.mark.parametrize("i", range(len(SHAPES)))
def test_grad_blocks_cover_flat_vector_once(i):
    spec = SHAPES[i]
    n = spec.n_params()
    hits = np.zeros(n, np.int64)
    blocks = O64.grad_blocks(spec)
    for _, _, s in blocks:
        hits[s] += 1
    assert (hits == 1).all()
    # same order and shapes as the oracle's unflatten: actor W / b per layer, critic W / b per layer, log_std
    flat = np.arange(n, dtype=f32)
    params = OP.unflatten(spec, flat)
    want = [np.asarray(x).reshape(-1) for name in ("actor", "critic") for (W, b) in params[name] for x in (W, b)]
    if spec.act_kind == "continuous":
        want.append(params["log_std"])
    assert len(want) == len(blocks)
    for (name, net, s), w in zip(blocks, want):
        np.testing.assert_array_equal(flat[s], w)
        assert net == (1 if name.startswith("critic") else 0)


def test_block_errors_floor_and_nonfinite():
    spec = OP.PolicySpec(3, [8, 8], "discrete", 1, act_start=0)        # Discrete(1): the actor's gradient is zero
    g64 = np.zeros(spec.n_params())
    crit = [s for name, net, s in O64.grad_blocks(spec) if net == 1]
    for s in crit:
        g64[s] = 1.0
    g = g64.copy()
    g[0] = 1e-12                                                        # tiny against the floor: accepted
    O64.assert_blocks_close(spec, g, g64)
    g[0] = 1e-3
    with pytest.raises(AssertionError):
        O64.assert_blocks_close(spec, g, g64)
    g[0] = np.nan
    with pytest.raises(AssertionError, match="non-finite"):
        O64.assert_blocks_close(spec, g, g64)


PATTERNS = [("step", 2.0 ** 16), ("step", 2.0 ** 40), ("step", 2.0 ** -20), "tiny", "outliers", "zero"]


@pytest.mark.parametrize("spec_i", [0, 1, 9])
@pytest.mark.parametrize("pattern", PATTERNS)
def test_generator_tile_ratios_and_margins(spec_i, pattern):
    spec = SHAPES[spec_i]
    rng = np.random.default_rng(3)
    flat = (OP.init_params(spec, seed=4) + rng.normal(size=spec.n_params()).astype(f32) * 0.05).astype(f32)
    B, lead = 64 * 40 + 37, 64 * 16
    mag, zero = O64.tile_magnitudes(pattern, B, lead, rng)
    for net in ("actor", "critic"):
        one, none = np.ones(B), np.zeros(B, bool)
        cvf, c = 0.5, 0.2
        a_mag, c_mag, a_zero, c_zero = (mag, one, zero, none) if net == "actor" else (one, mag, none, zero)
        obs, actions, adv, ret, old_lp, old_v = O64.scaled_minibatch(spec, flat, a_mag, c_mag, rng, clip_range=c, clip_range_vf=cvf,
                                                                     actor_zero=a_zero, critic_zero=c_zero)
        out, v = O64.forward64(spec, flat, obs)
        # magnitudes: |adv| (actor) and ret - v (critic) within [1/8, 2] x the sample's magnitude (float32 rounding aside)
        if net == "actor":
            x, m = np.abs(adv.astype(np.float64)), a_mag
            paired = slice(0, 2 * (B // 2))
            assert np.array_equal(adv[paired][0::2], -adv[paired][1::2])
            assert adv[paired].astype(np.float64).sum() == 0.0
        else:
            x, m = ret.astype(np.float64) - v, c_mag
            if m.min() >= 1e-3:                                     # not at float32's resolution of v
                assert (x > 0).all()
        sel = m >= 1e-3 if net == "critic" else np.arange(B) < 2 * (B // 2)     # an odd last sample has no pair: adv 0
        ratio_x = x[sel] / m[sel]
        assert ratio_x.min() >= 0.125 * (1 - 1e-6) and ratio_x.max() <= 2.0 * (1 + 1e-6)
        # per-tile ratios: the leading tiles' largest magnitude against the rest's is the pattern's ratio within 16x
        if isinstance(pattern, tuple) and not (net == "critic" and pattern[1] < 1e-3):
            r = np.abs(x[lead:]).max() / np.abs(x[:lead]).max()
            assert pattern[1] / 16 <= r <= pattern[1] * 16, r
        if pattern == "tiny" and net == "actor":
            assert np.abs(x[:lead]).max() <= 2.01e-30 and np.abs(x[lead:-1]).min() >= 0.1
        if pattern == "outliers":
            big = m > 1
            assert abs(big.mean() - 0.01) < 0.002 and (x[big].min() >= 0.99 * 2.0 ** 17)
        # branch margins
        ratio = np.exp(O64.logp64(spec, flat, out, actions) - old_lp.astype(np.float64))
        for edge in (1 - c, 1 + c):
            assert np.abs(ratio - edge).min() >= (O64.RATIO_MARGIN - 1e-3) * c
        dv = v - old_v.astype(np.float64)
        assert np.abs(np.abs(dv) - cvf).min() >= (O64.VF_MARGIN - 1e-3) * cvf
        if spec.act_kind == "discrete" and spec.act_n > 1:
            assert np.diff(np.sort(out, axis=1), axis=1).min() >= O64.TIE_GAP
        # zero-gradient samples: clipped on the side that zeroes their gradient
        if net == "actor" and zero.any():
            s = np.sign(adv[zero])
            assert ((s > 0) & (ratio[zero] > 1 + c) | (s < 0) & (ratio[zero] < 1 - c) | (s == 0)).all()
        if net == "critic" and zero.any():
            assert (np.abs(dv[zero]) > cvf).all()
        # and the float64 reference sees exactly zero gradient from them
        if zero.any():
            cfg = OO.PPOConfig(ent_coef=0.0, clip_range=c, clip_range_vf=cvf, normalize_advantage=False)
            keep = ~zero
            sub = lambda a: a[keep]
            full = O64.loss64(spec, flat, obs, actions, adv, ret, old_lp, old_v, cfg)[1] * B
            part = O64.loss64(spec, flat, *(sub(a) for a in (obs, actions, adv, ret, old_lp, old_v)), cfg)[1] * keep.sum()
            net_s = [s for _, n_, s in O64.grad_blocks(spec) if n_ == (0 if net == "actor" else 1)]
            for s in net_s:
                np.testing.assert_allclose(full[s], part[s], rtol=1e-9, atol=1e-12 * np.abs(part[s]).max())


def test_fp64_reference_matches_oracle_at_benign_inputs():
    """The float64 reference and the float32 oracle agree on an ordinary minibatch (the hand-written backward pin of
    tests/test_oracle_pins.py at a tile-structured minibatch)."""
    spec = SHAPES[1]
    rng = np.random.default_rng(9)
    flat = (OP.init_params(spec, seed=2) + rng.normal(size=spec.n_params()).astype(f32) * 0.05).astype(f32)
    B = 64 * 5 + 3
    mb = O64.scaled_minibatch(spec, flat, np.ones(B), np.ones(B), rng, clip_range_vf=0.5)
    cfg = OO.PPOConfig(clip_range_vf=0.5)
    eloss, estats, eg = OO.ppo_loss_and_grads(spec, flat, *mb, cfg)
    loss, g, stats = O64.loss64(spec, flat, *mb, cfg)
    assert abs(loss - eloss) <= 1e-5 * max(1.0, abs(loss))
    for k in O64.STAT_NAMES:
        assert abs(stats[k] - estats[k]) <= 1e-5 * max(1.0, abs(stats[k])), k
    O64.assert_blocks_close(spec, eg, g, 1e-4)
