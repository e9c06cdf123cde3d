"""The kernels between a rollout and its update: the Monitor ring push (one CTA per buffer row), the GAE pass that also
writes the sample records of a tcgen05 update, and the minibatch advantage moments finished inside the all-epochs permute
launch.  Each is checked against the code it replaces: the single-CTA ring push (restated below), ft_pack_records_kernel
(dril_ppo_update packs the records itself) and adv_stats_finalize_kernel (the per-epoch staging path still runs it)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def D():
    import __graft_entry__
    __graft_entry__.build()
    import dril_b200
    return dril_b200


def _ring_push(ring_r, ring_l, head, flags, ep_r, ep_l, window):
    """The single-CTA ring push this library ran before: rows from t0 on, in chunks, keeping the last `window` of a chunk."""
    done = (flags & 3) != 0
    dc = done.sum(axis=1)
    cum, t0 = 0, done.shape[0]
    while t0 > 0 and cum < window:
        t0 -= 1
        cum += dc[t0]
    for t in range(t0, done.shape[0]):
        idx = np.nonzero(done[t])[0]
        for k, n in enumerate(idx):
            if k >= len(idx) - window:
                ring_r[(head + k) % window] = ep_r[t, n]
                ring_l[(head + k) % window] = ep_l[t, n]
        head += len(idx)
    return head


def _window_stats(ring_r, ring_l, head, window):
    """dril_env_monitor_stats: fp32 sum of the returns and fp64 sum of the lengths, slot order."""
    cnt = min(head, window)
    if cnt == 0:
        return None
    sr, sl = np.float32(0), 0.0
    for i in range(cnt):
        sr = np.float32(sr + ring_r[i])
        sl += float(ring_l[i])
    return np.float32(sr / np.float32(cnt)), np.float32(sl / cnt), cnt


# (kind, n_envs, n_steps, max_steps, window): Pendulum episodes end together at max_steps with distinct fp32 returns, so the
# slot-order fp32 sum sees the order of the ring; CartPole episodes end at scattered steps and envs
@pytest.mark.parametrize("kind,n,T,ms,window", [
    ("pendulum", 37, 16, 10, 1000),       # fewer than `window` episodes per rollout
    ("pendulum", 37, 10, 10, 37),         # exactly `window` per rollout, all in one row
    ("pendulum", 1100, 8, 3, 5),          # a row holds many more than `window`: wraps
    ("pendulum", 1100, 12, 5, 1500),      # a long window filled over rows and rollouts
    ("cartpole", 1000, 40, 500, 100),     # scattered terminations
    ("cartpole", 1029, 24, 500, 7),
])
def test_monitor_ring_matches_single_cta_push(D, kind, n, T, ms, window):
    env = D.CudaBatchedEnv(kind, n, max_steps=ms, seed=11, monitor_window=window)
    hidden = [64, 64]
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=hidden)
    alg = D.PPO(n_steps=T, batch_size=n * T, epochs=1)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(3))
    buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
    ring_r, ring_l, head = np.zeros(window, np.float32), np.zeros(window, np.int64), 0
    for _ in range(4):
        _, ok = D.collect_rollout(buf, agent, alg, env)
        assert ok
        head = _ring_push(ring_r, ring_l, head, buf.download("flags"), buf.download("episode_r"), buf.download("episode_l"), window)
        got = env.monitor_stats()
        exp = _window_stats(ring_r, ring_l, head, window)
        assert exp is not None
        assert got["n_in_window"] == exp[2]
        assert np.float32(got["ep_rew_mean"]).tobytes() == exp[0].tobytes(), (got, exp)
        assert np.float32(got["ep_len_mean"]).tobytes() == exp[1].tobytes(), (got, exp)
    buf.close()
    env.close()


def _train_two_ways(D, kind, n, T, hidden, epochs, n_mb):
    """Two identical agents: one runs dril_ppo_iteration_async (the GAE pass writes the sample records), the other
    dril_rollout_collect + dril_gae + dril_ppo_update (ft_pack_records_kernel packs them).  Returns both parameter vectors."""
    from dril_b200 import _lib as L
    out = []
    for fused in (True, False):
        env = D.CudaBatchedEnv(kind, n, seed=5, monitor_window=100)
        layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=hidden)
        alg = D.PPO(n_steps=T, batch_size=n * T // n_mb, epochs=epochs)
        agent = D.Agent(layer, alg, rng=np.random.default_rng(7))
        assert agent.device.update_path() == "tensor"
        buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
        lib, h = agent.ctx.lib, alg.hyper()
        for it in range(3):
            if fused:
                L.check(lib.dril_ppo_iteration_async(env.h, agent.device.h, buf.h, C.byref(h), epochs, alg.batch_size, 123, it * epochs))
                st = D.IterStats()
                L.check(lib.dril_iteration_result(agent.device.h, C.byref(st)))
            else:
                fps = C.c_float(0)
                L.check(lib.dril_rollout_collect(env.h, agent.device.h, buf.h, None, C.byref(fps)))
                L.check(lib.dril_gae(buf.h, C.c_float(alg.gamma), C.c_float(alg.gae_lambda)))
                st = D.IterStats()
                L.check(lib.dril_ppo_update(agent.device.h, buf.h, C.byref(h), epochs, alg.batch_size, 123, it * epochs, C.byref(st)))
            assert st.n_minibatch_steps > 0
        out.append(agent.device.get_params())
        buf.close()
        env.close()
    return out


@pytest.mark.parametrize("kind,n,T,hidden", [
    ("cartpole", 4096, 128, [64, 64]),           # the [64,64] Discrete(2) kernel (update_ft.cuh), C2 shape
    ("pendulum", 1000, 24, [128, 128, 64]),      # the general kernel (update_ftg.cuh), Box actions, N not a multiple of 32
])
def test_gae_records_equal_packed_records(D, kind, n, T, hidden):
    """Every field of a record feeds the update, so bit-identical parameters after three iterations mean the records the GAE
    pass wrote are those ft_pack_records_kernel writes."""
    a, b = _train_two_ways(D, kind, n, T, hidden, epochs=2, n_mb=4)
    assert a.tobytes() == b.tobytes()


_CHILD = r"""
import sys
sys.path.insert(0, sys.argv[1])
import numpy as np
import __graft_entry__
__graft_entry__.build()
import dril_b200 as D
D.set_option("persistent", 0)
env = D.CudaBatchedEnv("cartpole", 1000, seed=9, monitor_window=100)
layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=[64, 64])
alg = D.PPO(n_steps=32, batch_size=32000 // 5, epochs=3)
agent = D.Agent(layer, alg, rng=np.random.default_rng(2))
assert agent.device.update_path() == "tensor"
D.train(agent, env, alg, 32000 * 3)
np.save(sys.argv[2], agent.device.get_params())
"""


def test_fused_moment_finalize_equals_separate_kernel(D, tmp_path):
    """With every epoch staged by one permute launch the minibatch advantage moments are finished in that launch; with a
    staging budget of 0 MB the update stages epoch by epoch and runs adv_stats_kernel + adv_stats_finalize_kernel.  One
    launch per minibatch step in both, so the moments are the only difference: the parameters must agree bit for bit."""
    got = []
    for budget in (None, "0"):
        envv = dict(os.environ)
        envv.pop("DRIL_STAGE_ALL_MB", None)
        if budget is not None:
            envv["DRIL_STAGE_ALL_MB"] = budget
        out = tmp_path / f"params_{budget}.npy"
        subprocess.run([sys.executable, "-c", _CHILD, ROOT, str(out)], check=True, env=envv, cwd=str(tmp_path), timeout=600)
        got.append(np.load(out))
    assert got[0].tobytes() == got[1].tobytes()
