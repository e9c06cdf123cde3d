"""Loss/grad kernels against the float64 reference (oracle/ppo64.py) per parameter block, on minibatches whose 64-sample
tiles differ in gradient magnitude by many orders.

The fp16 hi/lo kernels (update_ft.cuh, update_ftg.cuh) feed the backward deltas to the tensor cores scaled by one power of
two per CTA and warp group / net pass, chosen at the first tile with a non-zero gradient; dW accumulates in TMEM over all
the CTA's tiles.  Through DevicePolicy.loss_grad the samples stay in order: tile t holds samples [64 t, 64 t + 64), CTA c
processes tiles c, c + G, ... with G = min(tiles, SMs), and in update_ft.cuh its two warp groups alternate over them.  The
first 2 G tiles are therefore the first tile of every CTA and group, and the patterns below set their magnitude apart from
the rest's.  The 3xTF32, mma.sync and fp32 kernels have no delta scale and serve as controls."""
import ctypes as C
import zlib

import numpy as np
import pytest

from oracle import policy as OP, ppo as OO
from oracle import ppo64 as O64

pytestmark = pytest.mark.gpu
f32 = np.float32


@pytest.fixture(scope="module")
def D():
    import __graft_entry__
    __graft_entry__.build()
    import dril_b200
    return dril_b200


# name -> (spec, options, expected update_path); options are set before the policy is created and restored afterwards
PATHS = {
    "ft": (lambda: OP.PolicySpec(4, [64, 64], "discrete", 2, act_start=1), {}, "tensor"),
    "ftg_64": (lambda: OP.PolicySpec(4, [64, 64], "discrete", 2, act_start=1), {"ftg": 2}, "tensor"),
    "ftg_c3": (lambda: OP.PolicySpec(3, [128, 128, 64], "continuous", 1, act_low=[-2], act_high=[2]), {}, "tensor"),
    "ftg_box2": (lambda: OP.PolicySpec(6, [64, 128, 64], "continuous", 2, act_low=[-1, -1], act_high=[1, 1]), {}, "tensor"),
    "ftg_d3_64": (lambda: OP.PolicySpec(6, [64, 64], "discrete", 3, act_start=0), {}, "tensor"),
    "ftg_d3_128": (lambda: OP.PolicySpec(2, [128, 128, 64], "discrete", 3, act_start=0), {}, "tensor"),
    "ftg_d4_64": (lambda: OP.PolicySpec(4, [64, 64], "discrete", 4, act_start=1), {}, "tensor"),
    "ftg_d4_128": (lambda: OP.PolicySpec(5, [128, 128, 64], "discrete", 4, act_start=0), {}, "tensor"),
    # controls without a delta scale
    "tf32": (lambda: OP.PolicySpec(4, [64, 64], "discrete", 2, act_start=1), {"ft": 0}, "tensor"),
    "mma": (lambda: OP.PolicySpec(3, [128, 128, 64], "continuous", 1, act_low=[-2], act_high=[2]),
            {"tc": 0, "ftg": 0, "mma": 1}, "mma"),
    "fp32": (lambda: OP.PolicySpec(4, [64, 64], "discrete", 2, act_start=1), {"tc": 0, "ftg": 0, "mma": 0}, "fp32"),
}
_DEFAULTS = {"tc": 1, "ft": 1, "ftg": 1, "mma": 1, "persistent": 1}

PATTERNS = {
    "step_2^10": ("step", 2.0 ** 10),       # inside the first tile's headroom: the scale does not move
    "step_2^16": ("step", 2.0 ** 16),
    "step_2^24": ("step", 2.0 ** 24),
    "step_2^40": ("step", 2.0 ** 40),
    "tiny_lead": "tiny",
    "step_down_2^-20": ("step", 2.0 ** -20),
    "outliers": "outliers",
    "zero_lead": "zero",
}

# largest per-block error against float64, loss and statistics: north_star (c)
RTOL = 1e-4


def _policy(D, spec, flat, opts):
    for k, v in opts.items():
        D.set_option(k, v)
    space = D.Discrete(spec.act_n, spec.act_start) if spec.act_kind == "discrete" else D.Box(spec.act_low, spec.act_high)
    p = D.DevicePolicy(D.Context.default(), spec.obs_dim, spec.hidden, space)
    p.set_params(flat)
    return p


def _restore(D):
    for k, v in _DEFAULTS.items():
        D.set_option(k, v)


@pytest.mark.parametrize("net", ["actor", "critic"])
@pytest.mark.parametrize("pattern", list(PATTERNS))
@pytest.mark.parametrize("path", list(PATHS))
def test_loss_grad_tile_scales_vs_fp64(D, path, pattern, net):
    mk, opts, expect = PATHS[path]
    spec = mk()
    rng = np.random.default_rng(zlib.crc32(f"{path} {pattern} {net}".encode()))
    flat = (OP.init_params(spec, seed=4) + rng.normal(size=spec.n_params()).astype(f32) * 0.05).astype(f32)
    sms = D.Context.default().sm_count()
    B = sms * 64 * 6 + 37
    lead = 2 * min((B + 63) // 64, sms) * 64
    mag, zero = O64.tile_magnitudes(PATTERNS[pattern], B, lead, rng)
    one, none = np.ones(B), np.zeros(B, bool)
    try:
        p = _policy(D, spec, flat, opts)
        assert p.update_path() == expect
        # (normalize_advantage, clip_range_vf): the critic's zero-gradient lead needs the value clip
        cfgs = [(True, None), (False, 0.5)]
        if pattern == "zero_lead" and net == "critic":
            cfgs = [(True, 0.5), (False, 0.5)]
        for norm, cvf in cfgs:
            a_mag, c_mag = (mag, one) if net == "actor" else (one, mag)
            a_zero, c_zero = (zero, none) if net == "actor" else (none, zero)
            mb = O64.scaled_minibatch(spec, flat, a_mag, c_mag, rng, clip_range_vf=cvf, actor_zero=a_zero, critic_zero=c_zero)
            alg = D.PPO(ent_coef=0.0, clip_range_vf=cvf, normalize_advantage=norm)
            cfg = OO.PPOConfig(ent_coef=0.0, clip_range_vf=cvf, normalize_advantage=norm)
            what = f"{path} {pattern} {net} normalize={norm} clip_range_vf={cvf}"
            loss, stats, g = p.loss_grad(*mb, alg.hyper())
            eloss, eg, estats = O64.loss64(spec, flat, *mb, cfg)
            assert np.isfinite(loss) and abs(loss - eloss) <= RTOL * max(1.0, abs(eloss)), (what, loss, eloss)
            for k in O64.STAT_NAMES:
                assert abs(stats[k] - estats[k]) <= RTOL * max(1.0, abs(estats[k])), (what, k, stats[k], estats[k])
            errs = O64.assert_blocks_close(spec, g, eg, RTOL, what=what)
            print(f"GRADSCALE {path} {pattern} {net} norm={int(norm)} cvf={cvf} max_block_err={max(errs.values()):.3e}")
        p.close()
    finally:
        _restore(D)


# ------------------------------------------------------------------------------------------
# end to end: sparse large returns through the whole update
# ------------------------------------------------------------------------------------------
E2E = {
    # MountainCarContinuous: obs (position, velocity), Box(1) -> update_ftg.cuh
    "mountaincar_continuous": (lambda: OP.PolicySpec(2, [64, 64], "continuous", 1, act_low=[-1], act_high=[1]),
                               ([-1.2, -0.07], [0.6, 0.07])),
    # CartPole: Discrete(2) -> update_ft.cuh
    "cartpole": (lambda: OP.PolicySpec(4, [64, 64], "discrete", 2, act_start=1), ([-2.4, -3.0, -0.2, -3.0], [2.4, 3.0, 0.2, 3.0])),
}


@pytest.mark.parametrize("persistent", [1, 0])
@pytest.mark.parametrize("name", list(E2E))
def test_update_sparse_goal_returns_vs_oracle(D, name, persistent):
    """A rollout buffer whose returns are costs of order 1e-2 with +100 at 0.5 % of the samples (a sparse goal bonus, like
    MountainCarContinuous's), uploaded as is: 2 epochs x 4 minibatches of Feistel-shuffled samples through dril_ppo_update
    against the oracle's update.  The critic's output layer starts small, so the value errors of the cost steps are four
    orders of magnitude below the bonus."""
    mk, (lo, hi) = E2E[name]
    spec = mk()
    T, N = 64, 2048
    n = T * N
    rng = np.random.default_rng(17)
    flat = OP.init_params(spec, seed=6)
    out_layer = (f"critic.W{len(spec.hidden)}", f"critic.b{len(spec.hidden)}")
    for blk, _, s in O64.grad_blocks(spec):
        if blk in out_layer:
            flat[s] *= f32(1e-3)
    obs = rng.uniform(lo, hi, size=(n, spec.obs_dim)).astype(f32)
    if spec.act_kind == "discrete":
        actions = rng.integers(spec.act_start, spec.act_start + spec.act_n, (n, 1)).astype(np.int32)
    else:
        actions = rng.uniform(-1, 1, size=(n, spec.act_n)).astype(f32)
    out, v = O64.forward64(spec, flat, obs)
    logp = O64.logp64(spec, flat, out, actions)
    ret = -rng.uniform(0.0, 2e-2, n)
    ret[rng.random(n) < 0.005] = 100.0
    values = (v + rng.normal(size=n) * 1e-3).astype(f32)
    ob = {"obs": obs.reshape(T, N, spec.obs_dim), "actions": actions.reshape(T, N, -1),
          "rewards": np.zeros((T, N), f32), "values": values.reshape(T, N),
          "logprobs": (logp + rng.normal(size=n) * 0.05).astype(f32).reshape(T, N),
          "returns": ret.astype(f32).reshape(T, N)}
    ob["advantages"] = (ob["returns"] - ob["values"]).astype(f32)
    space = D.Discrete(spec.act_n, spec.act_start) if spec.act_kind == "discrete" else D.Box(spec.act_low, spec.act_high)
    try:
        p = _policy(D, spec, flat, {"persistent": persistent})
        assert p.update_path() == "tensor"
        buf = D.RolloutBuffer(D.Box(lo, hi), space, 0.95, 0.99, T, N)
        for k in ("obs", "actions", "values", "logprobs", "advantages", "returns"):
            buf.upload(k, ob[k])
        alg = D.PPO(n_steps=T, batch_size=n // 4, epochs=2, ent_coef=0.0)
        from dril_b200 import _lib as L
        st = D.IterStats()
        h = alg.hyper()
        L.check(p.ctx.lib.dril_ppo_update(p.h, buf.h, C.byref(h), alg.epochs, alg.batch_size, 29, 1, C.byref(st)))
        cfg = OO.PPOConfig(n_steps=T, batch_size=n // 4, epochs=2, ent_coef=0.0)
        opt = OO.Adam(flat.size, lr=cfg.learning_rate)
        new_flat, means, _ = OO.ppo_update(spec, flat, opt, ob, cfg, shuffle_seed=29, epoch_counter0=1)
        got = p.get_params()
        assert np.isfinite(got).all()
        assert st.n_minibatch_steps == 8
        rel = np.linalg.norm((got - flat).astype(np.float64) - (new_flat - flat)) / np.linalg.norm((new_flat - flat).astype(np.float64))
        assert rel < 2e-3, rel
        np.testing.assert_allclose(got, new_flat, rtol=1e-4, atol=2e-6)
        for k in ("policy_loss", "value_loss", "entropy_loss", "approx_kl_div", "clip_fraction", "loss", "grad_norm"):
            assert abs(getattr(st, k) - means[k]) <= 2e-4 * max(1.0, abs(means[k])), (k, getattr(st, k), means[k])
        buf.close()
        p.close()
    finally:
        _restore(D)
