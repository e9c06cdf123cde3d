"""Sampled rollouts on every rollout kernel against the float64 policy and the Philox SAMPLE stream.

Training never replays actions: every rollout samples them.  The action of env gid at step t of a rollout comes from
Philox block (gid, step0 + t mod 2**32, 0, SAMPLE) under the policy's 64-bit seed: Discrete heads take the first action
whose fp32 cumulative probability is >= the fp64 uniform u, Box heads store mean + exp(log_std) z.  A kernel that drew from
the wrong stream position, used 1 - u, mixed up the env id or picked the wrong CDF bucket would still fill a self-consistent
buffer (its log-probs and values are those of the action it stored), and PPO would still train, only worse.  So each case
here collects two consecutive sampled rollouts (the second continues the stream at step0 + T) and compares every row with
oracle/ppo64.py sample_ref64 on the stored observations (the normalised ones each kernel fed its actor):

  Discrete actions   equal to the fp64 reference wherever u is at least 1e-5 from every cumulative probability (margin);
                     at most max(8, 2e-4 T N) samples are that close (the count depends on u and the fp64 reference
                     only, not on the kernel: about (2A - 1) 1e-5 T N for A actions, so the bound keeps the test from
                     passing vacuously and is 4 standard deviations clear at the largest rows); every action value occurs
  Box actions        raw (unclamped), within 1e-5 (1 + |ref|) of mean64 + exp(log_std) z; (a - mean64) / sigma over the
                     buffer has |mean| < 0.05 and |std - 1| < 0.05
  log-probs          within 1e-4 max(1, |logp64|) of logp64 of the stored action
  values             within 3e-5 max(1, |V64|) of the fp64 critic on the stored observations
  last_values, boot  the fp64 critic of last_obs / term_obs of an oracle replay of the device's actions, at the same bound
                     (plus 3e-5 absolute where a training normaliser makes the replay's observations match to 3e-5 only);
                     the replay's flags equal the device's, its observations and rewards match at the replay tests' bounds

N derives from the SM count S so that every case lands on its kernel with a ragged last tile; test_sampling_kernel_routing
profiles one rollout of each case and checks the kernel (and, where the tile width shows in the grid, the grid).
"""
import json
import os
import re
import tempfile
import zlib

import numpy as np
import pytest

from oracle import classic_envs as CE, envs as OE, policy as OP, ppo as OO
from oracle import ppo64 as O64

pytestmark = pytest.mark.gpu
f32 = np.float32
SEED = (1 << 40) + 12345          # both Philox key words matter
STEP0 = 5
WRAP = 2 ** 32 - 3                # the first rollout crosses the wrap of the 32-bit sample counter
GID = 1_000_003
_DEFAULTS = {"tc_rollout": 1, "tc_actor": 1}


@pytest.fixture(scope="module")
def D():
    import __graft_entry__
    __graft_entry__.build()
    import dril_b200
    return dril_b200


@pytest.fixture(scope="module")
def S(D):
    return D.Context.default().sm_count()


def _spec(kind, hidden, act_start=1, obs_dim=None):
    if kind == "cartpole":
        return OP.PolicySpec(obs_dim or 4, hidden, "discrete", 2, act_start=act_start)
    if kind == "pendulum":
        return OP.PolicySpec(obs_dim or 3, hidden, "continuous", 1, act_low=[-2], act_high=[2])
    if kind == "mountaincar_continuous":
        return OP.PolicySpec(obs_dim or 2, hidden, "continuous", 1, act_low=[-1], act_high=[1])
    return OP.PolicySpec(obs_dim or (2 if kind == "mountaincar" else 6), hidden, "discrete", 3, act_start=act_start)


def _oracle_env(kind, n, seed, ms, gid_offset, act_start, scaling, norm, obs_dim):
    if kind == "cartpole":
        b = OE.CartPoleBatch(n, seed=seed, max_steps=ms, gid_offset=gid_offset, act_start=act_start)
    elif kind == "pendulum":
        b = OE.PendulumBatch(n, seed=seed, max_steps=ms, gid_offset=gid_offset)
    elif kind == "mountaincar":
        b = CE.MountainCarBatch(n, seed=seed, max_steps=ms, gid_offset=gid_offset, act_start=act_start)
    elif kind == "mountaincar_continuous":
        b = CE.MountainCarContinuousBatch(n, seed=seed, max_steps=ms, gid_offset=gid_offset)
    else:
        b = CE.AcrobotBatch(n, seed=seed, max_steps=ms, gid_offset=gid_offset, act_start=act_start)
    if scaling:
        b = OE.ScalingBatch(b, CE.MOUNTAINCAR_OBS_LOW, CE.MOUNTAINCAR_OBS_HIGH)
    o = OE.MonitorWrapper(OE.ParallelEnv(b))
    return OE.NormalizeWrapper(o, obs_dim) if norm else o


class Case:
    """One sampled-rollout configuration.  n is a function of the SM count S.  kernel: regex of the rollout kernel's name
    (demangled); critic: regex of the batched critic pass behind it, or None; tile: envs per CTA where the grid shows it;
    threads: the block size where it tells the fast kernel's 8x8 register tiles (128 threads for a 64-env tile) from its
    4x4 ones (256)."""

    def __init__(self, kind, hidden, n, T, ms, kernel, critic=None, tile=None, threads=None, norm=False, opts=None, act_start=1,
                 gid_offset=0, step0=STEP0, scaling=False, replay=True, chunked=False, env_kw=None):
        self.kind, self.hidden, self.n, self.T, self.ms = kind, hidden, n, T, ms
        self.kernel, self.critic, self.tile, self.threads, self.norm = kernel, critic, tile, threads, norm
        self.opts, self.act_start, self.gid_offset, self.step0 = opts or {}, act_start, gid_offset, step0
        self.scaling, self.replay, self.chunked, self.env_kw = scaling, replay, chunked, env_kw or {}


TC = r"rollout_tc_kernel<{}>"
FAST = r"rollout_fast_kernel<(true|false), [^,>]+>"
COOP = r"rollout_kernel<(true|false), [^,>]+>"
GTC = r"rollout_gtc_kernel<{}, [^,>]+, {}>"
FTG_CRITIC = r"critic_values_ftg_kernel<\d>"

CASES = {
    # Kernels as a profile of one rollout on an NVIDIA B200 (148 SMs) named them; test_sampling_kernel_routing checks them.
    # C2: the tensor-core CartPole rollout, actor only, then one batched critic pass.
    # rollout_tc_kernel<1> + critic_values_tc_kernel
    "tc1": Case("cartpole", [64, 64], lambda S: 333, 40, 20, TC.format(1), r"critic_values_tc_kernel", step0=WRAP),
    # C4's regime: at least two 32-env tiles per SM -> the 64-register two-CTAs-per-SM build.
    # rollout_tc_kernel<2> (grid 2 S) + critic_values_tc_kernel
    "tc2": Case("cartpole", [64, 64], lambda S: 64 * S + 17, 6, 4, TC.format(2), r"critic_values_tc_kernel", step0=WRAP),
    # the sampled counterparts of test_fused_rollout_edge_shapes: a single env; every step truncates.
    # rollout_tc_kernel<1> + critic_values_tc_kernel
    "tc_edge_1": Case("cartpole", [64, 64], lambda S: 1, 9, 3, TC.format(1), r"critic_values_tc_kernel"),
    "tc_edge_33": Case("cartpole", [64, 64], lambda S: 33, 6, 1, TC.format(1), r"critic_values_tc_kernel"),
    # the fast kernel (no training normaliser): 4x4 register tiles at 8 / 16 / 32 / 64 envs per CTA, 8x8 tiles.
    # rollout_fast_kernel<true, 63u> (fast32: <true, 7u>), grid ceil(N / tile)
    "fast8": Case("mountaincar", [64, 64], lambda S: 2 * S + 5, 12, 7, FAST, tile=8),
    "fast16": Case("acrobot", [64, 64], lambda S: 24 * S + 3, 8, 5, FAST, tile=16, act_start=-1),
    "fast32": Case("cartpole", [64, 64], lambda S: 48 * S + 7, 8, 5, FAST, tile=32, act_start=0, opts={"tc_rollout": 0}),
    "fast64": Case("acrobot", [64, 64], lambda S: 80 * S + 9, 6, 4, FAST, tile=64, threads=256, act_start=-1,
                   gid_offset=GID, step0=WRAP),
    "fast_t8": Case("acrobot", [64, 64], lambda S: 96 * S + 13, 4, 3, FAST, tile=64, threads=128),
    # Box(1) on the fast kernel: weights in shared memory / streamed; the clamp goes to the env, the raw action to the buffer.
    # rollout_fast_kernel<true, 63u> / rollout_fast_kernel<false, 7u>
    "fast_box_mcc": Case("mountaincar_continuous", [64, 64], lambda S: 300, 24, 10, FAST, scaling=True),
    "fast_box_pendulum": Case("pendulum", [128, 128, 64], lambda S: 300, 24, 10, FAST),
    # the cooperative kernel with a training normaliser, critic in the step loop (nets the tcgen05 kernels do not cover).
    # rollout_kernel<true, 7u>
    "coop_cartpole": Case("cartpole", [64, 32], lambda S: 200, 20, 9, COOP, norm=True, step0=WRAP),
    "coop_pendulum": Case("pendulum", [64, 32], lambda S: 200, 20, 9, COOP, norm=True),
    # ... with the critic deferred to one batched pass.  rollout_kernel<true, 63u | 7u> + critic_values_ftg_kernel
    "coop_defer_mountaincar": Case("mountaincar", [64, 64], lambda S: 700, 20, 9, COOP, FTG_CRITIC, norm=True),
    "coop_defer_pendulum": Case("pendulum", [64, 64], lambda S: 700, 20, 9, COOP, FTG_CRITIC, norm=True),
    # ... with the wide layers on mma.sync tiles, 128-env tiles (the tcgen05 actor switched off).
    # rollout_kernel<false, 7u> + critic_values_ftg_kernel
    "coop_mma": Case("pendulum", [128, 128, 64], lambda S: 96 * S + 5, 4, 3, COOP, FTG_CRITIC, norm=True, opts={"tc_actor": 0}),
    # the actor on tcgen05 inside the general step loop.  rollout_gtc_kernel<2, 7u, 2>, <3, 7u, 2> (C3), <2, 63u, 4>,
    # <3, 63u, 4>, each + critic_values_ftg_kernel
    "gtc2": Case("cartpole", [64, 64], lambda S: 96 * S + 7, 6, 4, GTC.format(2, 2), FTG_CRITIC, norm=True, step0=WRAP),
    "gtc3_box": Case("pendulum", [128, 128, 64], lambda S: 16384, 4, 3, GTC.format(3, 2), FTG_CRITIC, norm=True),   # C3
    "gtc_d3_acrobot": Case("acrobot", [64, 64], lambda S: 96 * S + 7, 4, 3, GTC.format(2, 4), FTG_CRITIC, norm=True,
                           gid_offset=GID),
    "gtc_d3_mountaincar": Case("mountaincar", [128, 128, 64], lambda S: 96 * S + 7, 4, 3, GTC.format(3, 4), FTG_CRITIC,
                               norm=True),
    # kind-set instantiations added with the env features: policy-side checks only.  rollout_fast_kernel<true, 65539u>,
    # rollout_gtc_kernel<2, 196667u, 4>, rollout_fast_kernel<true, 327683u>, rollout_fast_kernel<true, 589883u>,
    # rollout_gtc_kernel<2, 589883u, 4>
    "ks_params_fast": Case("cartpole", [64, 64], lambda S: 333, 12, 9, FAST, replay=False,
                           env_kw=dict(env_params=dict(length=(0.25, 1.0), masspole=(0.05, 0.2)))),
    "ks_obs_params_gtc": Case("acrobot", [64, 64], lambda S: 96 * S + 7, 4, 3, GTC.format(2, 4), FTG_CRITIC, norm=True,
                              replay=False, env_kw=dict(env_params=dict(link_mass_1=(0.8, 1.2)), observe_params=True)),
    "ks_history_fast": Case("cartpole", [64, 64], lambda S: 333, 12, 9, FAST, replay=False,
                            env_kw=dict(history_len=4, mask_velocities=True)),
    "ks_perturb_fast": Case("acrobot", [64, 64], lambda S: 333, 12, 9, FAST, replay=False,
                            env_kw=dict(obs_noise=0.01, action_delay=2)),
    "ks_perturb_gtc": Case("acrobot", [64, 64], lambda S: 96 * S + 7, 4, 3, GTC.format(2, 4), FTG_CRITIC, norm=True,
                           replay=False, env_kw=dict(obs_noise=0.01, action_delay=2)),
    # chunked collection (an on_step callback): dril_rollout_collect_steps over buffer views, one step per chunk.
    # rollout_fast_kernel<true, 7u> / rollout_kernel<true, 7u> per chunk (and rollout_kernel<false, 7u> for the first
    # observation's statistics update)
    "chunked_cartpole": Case("cartpole", [64, 64], lambda S: 333, 12, 7, FAST, chunked=True, step0=WRAP),
    "chunked_pendulum": Case("pendulum", [64, 64], lambda S: 256, 16, 7, COOP, norm=True, chunked=True),
}
# Acrobot's and MountainCar's normalised observations of columns that start nearly constant match the oracle's over ~14 000
# envs only to its fp32 sums (test_fused_rollout_vs_oracle): their replays check flags and rewards only
REPLAY_FLAGS_ONLY = {"gtc_d3_acrobot", "gtc_d3_mountaincar"}


def _make(D, case, S):
    n = case.n(S)
    norm = D.NormalizeConfig() if case.norm else None
    env = D.CudaBatchedEnv(case.kind, n, max_steps=case.ms, seed=9, monitor_window=100, normalize=norm,
                           act_start=case.act_start, gid_offset=case.gid_offset, scaling=case.scaling, **case.env_kw)
    spec = _spec(case.kind, case.hidden, case.act_start, env.obs_dim)
    rng = np.random.default_rng(zlib.crc32(case.kind.encode()))
    flat = (OP.init_params(spec, seed=2) + rng.normal(size=spec.n_params()).astype(f32) * 0.05).astype(f32)
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=case.hidden)
    alg = D.PPO(n_steps=case.T, gamma=0.97, gae_lambda=0.9)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
    agent.set_parameters(flat)
    agent.device.seed(SEED, case.step0)
    oenv = None
    if case.replay:
        oenv = _oracle_env(case.kind, n, 9, case.ms, case.gid_offset, case.act_start, case.scaling, case.norm, spec.obs_dim)
    return env, oenv, spec, flat, agent, alg


def _callbacks(D, case):
    """A callback that overrides on_step: collect_rollout then runs one step per chunk."""
    if not case.chunked:
        return None

    class Hook(D.AbstractCallback):
        def on_step(self, loc):
            return True
    return [Hook()]


def _collect(D, case, env, agent, alg):
    buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, case.T, env.n_envs)
    _, ok = D.collect_rollout(buf, agent, alg, env, callbacks=_callbacks(D, case))
    assert ok
    out = {k: buf.download(k) for k in ("obs", "actions", "logprobs", "values", "last_values", "boot", "flags", "rewards")}
    buf.close()
    return out


def _rel(err, ref):
    return np.abs(err) / np.maximum(1.0, np.abs(ref))


def _check_rollout(name, case, spec, flat, out, step0, oenv, acc):
    T, N = out["rewards"].shape
    obs = out["obs"].reshape(T * N, -1)
    acts = out["actions"].reshape(T * N, -1)
    gid = case.gid_offset + np.tile(np.arange(N), T)
    step = (step0 + np.repeat(np.arange(T), N)) % 2 ** 32
    ref = O64.sample_ref64(spec, flat, obs, gid, step, SEED, actions=acts)
    err = {}
    if spec.act_kind == "discrete":
        a = acts[:, 0]
        ok = ref["margin"] >= 1e-5
        bad = np.flatnonzero(ok & (a != ref["actions"]))
        assert bad.size == 0, (f"{name}: {bad.size} sampled actions differ from the stream, first (t, n) = "
                               f"{[(int(i // N), int(i % N)) for i in bad[:5]]}: got {a[bad[:5]].tolist()}, "
                               f"want {ref['actions'][bad[:5]].tolist()}")
        err["exempt"] = int((~ok).sum())
        assert err["exempt"] <= max(8, 2e-4 * T * N), (name, err["exempt"])
        acc.setdefault("values_seen", set()).update(np.unique(a).tolist())
    else:
        e = np.abs(acts - ref["actions"]) / (1 + np.abs(ref["actions"]))
        err["act"] = float(e.max())
        assert err["act"] <= 1e-5, (name, err["act"], np.unravel_index(e.argmax(), e.shape))
        sigma = np.exp(np.asarray(flat[-spec.act_n:], np.float64))
        acc.setdefault("resid", []).append(((acts - ref["out"]) / sigma).reshape(-1))
    e = _rel(out["logprobs"].reshape(-1) - ref["logp"], ref["logp"])
    err["logp"] = float(e.max())
    assert err["logp"] <= 1e-4, (name, err["logp"], int(e.argmax()))
    e = _rel(out["values"].reshape(-1) - ref["values"], ref["values"])
    err["value"] = float(e.max())
    assert err["value"] <= 3e-5, (name, err["value"], int(e.argmax()))
    if oenv is None:
        return err
    # replay the device's actions (raw; the oracle clamps Box actions to the space like the kernels) through the oracle env
    replay = acts.reshape(T, N) if spec.act_kind == "discrete" else acts.reshape(T, N, -1)
    eo = OO.collect_rollout_timemajor(oenv, spec, flat, T, forced_actions=replay)
    te, tr = (out["flags"] & 1).astype(bool), ((out["flags"] >> 1) & 1).astype(bool)
    np.testing.assert_array_equal(te, eo["term"], err_msg=f"{name}: terminated")
    np.testing.assert_array_equal(tr, eo["trunc"], err_msg=f"{name}: truncated")
    assert tr.any(), name
    ntol = dict(rtol=3e-5, atol=3e-4 if case.kind == "acrobot" else 3e-5)
    np.testing.assert_allclose(out["rewards"], eo["rewards"], **(ntol if case.norm else dict(rtol=1e-6, atol=0)),
                               err_msg=f"{name}: rewards")
    if name in REPLAY_FLAGS_ONLY:
        return err
    np.testing.assert_allclose(out["obs"], eo["obs"], **(ntol if case.norm else dict(rtol=1e-6, atol=1e-7)),
                               err_msg=f"{name}: observations")
    slack = 3e-5 if case.norm else 0.0
    _, lv64 = O64.forward64(spec, flat, eo["last_obs"])
    d, bound = np.abs(out["last_values"] - lv64), 3e-5 * np.maximum(1.0, np.abs(lv64)) + slack
    err["last"] = float((d / np.maximum(1.0, np.abs(lv64))).max())
    assert (d <= bound).all(), (name, err["last"], int((d - bound).argmax()))
    _, bv64 = O64.forward64(spec, flat, eo["term_obs"][tr])
    d, bound = np.abs(out["boot"][tr] - bv64), 3e-5 * np.maximum(1.0, np.abs(bv64)) + slack
    err["boot"] = float((d / np.maximum(1.0, np.abs(bv64))).max())
    assert (d <= bound).all(), (name, err["boot"], int((d - bound).argmax()))
    return err


@pytest.mark.parametrize("name", list(CASES))
def test_sampled_rollout_vs_fp64(D, S, name):
    case = CASES[name]
    try:
        for k, v in case.opts.items():
            D.set_option(k, v)
        env, oenv, spec, flat, agent, alg = _make(D, case, S)
        acc = {}
        for r in range(2):
            step0 = (case.step0 + r * case.T) % 2 ** 32
            out = _collect(D, case, env, agent, alg)
            err = _check_rollout(name, case, spec, flat, out, step0, oenv, acc)
            print(f"SAMPLING {name} rollout={r} N={env.n_envs} T={case.T} step0={step0} "
                  + " ".join(f"{k}={v:.3e}" if isinstance(v, float) else f"{k}={v}" for k, v in err.items()))
        if spec.act_kind == "discrete":
            assert acc["values_seen"] == set(range(spec.act_start, spec.act_start + spec.act_n)), (name, acc["values_seen"])
        else:
            res = np.concatenate(acc["resid"])
            assert abs(res.mean()) < 0.05 and abs(res.std() - 1) < 0.05, (name, res.mean(), res.std())
        env.close()
    finally:
        for k in case.opts:
            D.set_option(k, _DEFAULTS[k])


def _kernel_launches(fn):
    """[(kernel name, grid, block)] of the CUDA kernels launched while fn() runs (torch.profiler, CUDA activities)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as fh:
            ev = json.load(fh)["traceEvents"]
    return [(e["name"], tuple(e["args"].get("grid", ())), tuple(e["args"].get("block", ())))
            for e in ev if e.get("cat") == "kernel"]


@pytest.mark.parametrize("name", list(CASES))
def test_sampling_kernel_routing(D, S, name):
    """The kernel each case of test_sampled_rollout_vs_fp64 is meant to reach, read from a profile of one rollout."""
    case = CASES[name]
    try:
        for k, v in case.opts.items():
            D.set_option(k, v)
        env, _, _, _, agent, alg = _make(D, case, S)
        _collect(D, case, env, agent, alg)           # module loads and first-launch work outside the profile
        launches = _kernel_launches(lambda: _collect(D, case, env, agent, alg))
        names = [nm for nm, _, _ in launches]
        roll = [x for x in launches if re.search(r"rollout_\w*kernel", x[0])]
        print(f"ROUTING {name} N={env.n_envs}: " + ", ".join(sorted({re.sub(r"\(.*", "", nm) for nm, _, _ in roll}))
              + f" grid={roll[0][1] if roll else None} block={roll[0][2] if roll else None}")
        assert roll and all(re.search(case.kernel, nm) for nm, _, _ in roll), (name, case.kernel, names)
        if case.chunked:        # one launch per step (and the first observe's statistics update under a training normaliser)
            assert len(roll) == case.T + (1 if case.norm else 0), (name, len(roll))
        if case.critic is not None:
            assert any(re.search(case.critic, nm) for nm in names), (name, case.critic, names)
        else:
            assert not any("critic_values" in nm for nm in names), (name, names)
        if case.tile is not None:
            assert roll[0][1][0] == -(-env.n_envs // case.tile), (name, roll[0][1], case.tile)
        if case.threads is not None:
            assert roll[0][2][0] == case.threads, (name, roll[0][2], case.threads)
        env.close()
    finally:
        for k in case.opts:
            D.set_option(k, _DEFAULTS[k])
