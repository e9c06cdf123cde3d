"""The float64 sampling reference (oracle/ppo64.py sample_ref64) against the fp32 oracle policy (oracle/policy.py forward),
and the terminal observations of truncated samples that oracle.ppo.collect_rollout_timemajor returns (term_obs)."""
import numpy as np
import pytest

from oracle import envs as OE, policy as OP, ppo as OO
from oracle import ppo64 as O64

f32 = np.float32
SEED = (1 << 40) + 12345          # both Philox key words non-zero

SPECS = {
    "cartpole": lambda: OP.PolicySpec(4, [64, 64], "discrete", 2, act_start=1),
    "acrobot_start-1": lambda: OP.PolicySpec(6, [64, 64], "discrete", 3, act_start=-1),
    "d5_start0": lambda: OP.PolicySpec(7, [32], "discrete", 5, act_start=0),
    "pendulum": lambda: OP.PolicySpec(3, [128, 128, 64], "continuous", 1, act_low=[-2], act_high=[2]),
    "box3": lambda: OP.PolicySpec(5, [32, 16], "continuous", 3, act_low=[-1] * 3, act_high=[1] * 3),
}


def _flat(spec, seed):
    rng = np.random.default_rng(seed)
    flat = OP.init_params(spec, seed=seed)
    # larger actor outputs than the init's gain of 0.01, so that the probabilities are far from uniform
    return (flat + rng.normal(size=spec.n_params()).astype(f32) * 0.3).astype(f32)


@pytest.mark.parametrize("name", list(SPECS))
@pytest.mark.parametrize("step0", [5, 2 ** 32 - 3])
def test_sample_ref64_matches_fp32_oracle(name, step0):
    spec = SPECS[name]()
    flat = _flat(spec, 3)
    rng = np.random.default_rng(7)
    N, T = 257, 8
    obs = rng.normal(size=(T * N, spec.obs_dim)).astype(f32)
    gid = np.tile(np.arange(N) + 1_000_003, T)
    step = (step0 + np.repeat(np.arange(T), N)) % 2 ** 32
    a32 = np.concatenate([OP.forward(spec, flat, obs[t * N:(t + 1) * N], gid[:N], (step0 + t) % 2 ** 32, SEED)[0].reshape(N, -1)
                          for t in range(T)])
    ref = O64.sample_ref64(spec, flat, obs, gid, step, SEED, actions=a32)
    # a step index past 2**32 is the same draw as its residue
    ref_wrapped = O64.sample_ref64(spec, flat, obs, gid, step + 2 ** 32, SEED)
    np.testing.assert_array_equal(ref_wrapped["actions"], ref["actions"])
    v32, lp32, _ = OP.evaluate_actions(spec, flat, obs, a32)
    np.testing.assert_allclose(ref["values"], v32, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(ref["logp"], lp32, rtol=1e-4, atol=1e-5)
    if spec.act_kind == "discrete":
        ok = ref["margin"] >= 1e-5
        assert (~ok).sum() <= max(4, 1e-4 * T * N)
        np.testing.assert_array_equal(a32[ok, 0], ref["actions"][ok])
        assert set(np.unique(ref["actions"])) == set(range(spec.act_start, spec.act_start + spec.act_n))
    else:
        np.testing.assert_allclose(a32, ref["actions"], rtol=1e-5, atol=1e-5)
        sigma = np.exp(flat[-spec.act_n:].astype(np.float64))
        res = (ref["actions"] - ref["out"]) / sigma
        assert abs(res.mean()) < 0.05 and abs(res.std() - 1) < 0.05


def test_sample_ref64_stream_positions_differ():
    """The reference follows the stream: another step, another env id or another key word gives other actions."""
    spec = SPECS["acrobot_start-1"]()
    flat = _flat(spec, 1)
    obs = np.random.default_rng(2).normal(size=(4000, spec.obs_dim)).astype(f32)
    gid, step = np.arange(4000), np.full(4000, 9)
    base = O64.sample_ref64(spec, flat, obs, gid, step, SEED)["actions"]
    for g, s, k in ((gid, step + 1, SEED), (gid + 1, step, SEED), (gid, step, SEED & 0xFFFFFFFF), (gid, step, SEED >> 32 << 32)):
        assert (O64.sample_ref64(spec, flat, obs, g, s, k)["actions"] != base).mean() > 0.2


def test_term_obs_holds_terminal_observations():
    """term_obs[t, n] is info["terminal_observation"][n] where sample (t, n) truncated and zero elsewhere; boot is the
    critic of exactly those rows."""
    spec = SPECS["cartpole"]()
    flat = _flat(spec, 5)
    n, T, ms = 37, 23, 4
    forced = np.random.default_rng(0).integers(1, 3, (T, n))
    mk = lambda: OE.MonitorWrapper(OE.ParallelEnv(OE.CartPoleBatch(n, seed=3, max_steps=ms)))
    ob = OO.collect_rollout_timemajor(mk(), spec, flat, T, forced_actions=forced)
    assert ob["term_obs"].shape == (T, n, spec.obs_dim)
    env = mk()
    env.observe()
    for t in range(T):
        _, term, trunc, info = env.act(forced[t])
        env.observe()
        np.testing.assert_array_equal(ob["trunc"][t], trunc)
        exp = np.where(trunc[:, None], info["terminal_observation"], 0) if trunc.any() else np.zeros((n, spec.obs_dim), f32)
        np.testing.assert_array_equal(ob["term_obs"][t], exp)
    assert ob["trunc"].sum() > 10
    tr = ob["trunc"]
    np.testing.assert_allclose(ob["boot"][tr], OP.predict_values(spec, flat, ob["term_obs"][tr]), rtol=1e-6, atol=1e-7)
    assert not ob["term_obs"][~tr].any()
