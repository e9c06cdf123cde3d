"""Automatic domain randomisation in a data-parallel run, world_size 2, one process per GPU (needs 2 GPUs; skipped on a machine
with one): forced-action rollouts on two shards of one CartPole batch, through the NCCL and the peer-memory exchange, through
dril_rollout_collect, chunked collection and dril_ppo_iteration_async.  Both ranks must hold identical ADR state every round, equal
to the oracle (oracle/env_adr.py) run over the union of the envs."""
import os
import socket

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N_LOCAL, T, MS, ROUNDS, SEED = 150, 24, 10, 4, 9
ADR = dict(length=dict(init=(0.5, 0.55), limits=(0.25, 1.0), step=0.05),
           masspole=dict(init=(0.1, 0.11), limits=(0.05, 0.2), step=0.01))
P_BOUNDARY, M, THRESHOLDS = 0.5, 40, (9.978, 10.0)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _forced(r):
    return np.random.default_rng(1000 + r).integers(1, 3, (T, 2 * N_LOCAL))


def _worker(rank, world, port, out):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    import ctypes as C
    import dril_b200 as D
    from dril_b200 import _lib as L

    def all_gather(b):
        o = [None] * world
        dist.all_gather_object(o, b)
        return o

    class Hook(D.AbstractCallback):
        def on_step(self, loc):
            return True

    res = {}
    sl = slice(rank * N_LOCAL, (rank + 1) * N_LOCAL)
    for path in ("collect_nccl", "collect_p2p", "chunked", "iteration"):
        ctx = D.Context(device=rank, seed=0)
        uid = [D.Context.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.comm_init(rank, world, uid[0])
        env = D.CudaBatchedEnv("cartpole", N_LOCAL, max_steps=MS, seed=SEED, ctx=ctx, monitor_window=100, gid_offset=rank * N_LOCAL)
        env.set_adr(ADR, p_boundary=P_BOUNDARY, buffer_size=M, thresholds=THRESHOLDS)
        layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=[64, 64])
        alg = D.PPO(n_steps=T, batch_size=T * N_LOCAL // 2, epochs=1)
        agent = D.Agent(layer, alg, rng=np.random.default_rng(0), ctx=ctx)
        if path != "collect_nccl":
            ctx.comm_p2p_setup(all_gather, agent.device.n_params + 8)
        buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, N_LOCAL, ctx=ctx)
        L.check(ctx.lib.dril_iteration_prepare(env.h, agent.device.h, buf.h, alg.epochs, alg.batch_size))
        dist.barrier()
        states, actions = [], []
        for r in range(ROUNDS):
            if path == "iteration":
                h = alg.hyper()
                L.check(ctx.lib.dril_ppo_iteration_async(env.h, agent.device.h, buf.h, C.byref(h), 1, alg.batch_size, 5, r))
                st = D.IterStats()
                L.check(ctx.lib.dril_iteration_result(agent.device.h, C.byref(st)))
                actions.append(buf.download("actions")[..., 0])
            else:
                fa = np.ascontiguousarray(_forced(r)[:, sl])
                D.collect_rollout(buf, agent, alg, env, callbacks=[Hook()] if path == "chunked" else None, forced_actions=fa)
            s = env.adr_state()
            states.append(dict(ranges=s["ranges"], counts=s["counts"], sums=s["sums"], round=s["round"]))
        res[path] = dict(states=states, actions=actions)
        buf.close(); env.close(); agent.device.close()
    np.save(out + f".rank{rank}.npy", res, allow_pickle=True)
    dist.barrier()
    dist.destroy_process_group()


def _oracle(forced_rounds):
    from oracle import env_adr as EA, env_params as EP, envs as OE, policy as OP, ppo as OO
    n = 2 * N_LOCAL
    params = [EA.AdrParam(3, 0.5, 0.55, 0.25, 1.0, 0.05), EA.AdrParam(2, 0.1, 0.11, 0.05, 0.2, 0.01)]
    ob = EP.PARAM_BATCHES["cartpole"](n, seed=SEED, max_steps=MS)
    o = OE.MonitorWrapper(OE.ParallelEnv(ob))
    adr = EA.Adr("cartpole", params, P_BOUNDARY, M, *THRESHOLDS, SEED, np.arange(n))
    adr.attach(ob)
    spec = OP.PolicySpec(4, [64, 64], "discrete", 2, act_start=1)
    flat = OP.init_params(spec, seed=0)
    out = []
    for fa in forced_rounds:
        eo = OO.collect_rollout_timemajor(o, spec, flat, T, forced_actions=fa)
        adr.after_rollout(ob, eo["term"] | eo["trunc"], eo["episode_r"])
        out.append(dict(lo=adr.lo.copy(), hi=adr.hi.copy(), sums=adr.sums.copy(), counts=adr.counts.copy(), round=adr.round))
    return out


def _arrays(s):
    names = ("length", "masspole")
    return (np.array([s["ranges"][k][0] for k in names], np.float32), np.array([s["ranges"][k][1] for k in names], np.float32),
            np.asarray(s["sums"]), np.array([c for k in names for c in s["counts"][k]]), s["round"])


def test_dp_adr_vs_oracle(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    out = str(tmp_path / "dp_adr")
    mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    R = [np.load(out + f".rank{r}.npy", allow_pickle=True).item() for r in range(2)]
    exp = _oracle([_forced(r) for r in range(ROUNDS)])
    for path in ("collect_nccl", "collect_p2p", "chunked"):
        for r in range(ROUNDS):
            a0, a1 = _arrays(R[0][path]["states"][r]), _arrays(R[1][path]["states"][r])
            for x, y in zip(a0, a1):
                np.testing.assert_array_equal(x, y, err_msg=f"{path} round {r}: ranks differ")
            lo, hi, sums, counts, rnd = a0
            e = exp[r]
            np.testing.assert_array_equal(lo, e["lo"], err_msg=f"{path} round {r}")
            np.testing.assert_array_equal(hi, e["hi"], err_msg=f"{path} round {r}")
            np.testing.assert_array_equal(counts, e["counts"], err_msg=f"{path} round {r}")
            np.testing.assert_allclose(sums, e["sums"], rtol=1e-12, atol=0, err_msg=f"{path} round {r}")
            assert rnd == e["round"]
    moved = [(exp[r]["lo"] != exp[r - 1]["lo"]).any() or (exp[r]["hi"] != exp[r - 1]["hi"]).any() for r in range(1, ROUNDS)]
    assert any(moved)
    # the iteration path sampled its actions: the oracle replays the union of both ranks' actions
    acts = [np.concatenate([R[0]["iteration"]["actions"][r], R[1]["iteration"]["actions"][r]], axis=1) for r in range(ROUNDS)]
    exp = _oracle(acts)
    for r in range(ROUNDS):
        a0, a1 = _arrays(R[0]["iteration"]["states"][r]), _arrays(R[1]["iteration"]["states"][r])
        for x, y in zip(a0, a1):
            np.testing.assert_array_equal(x, y, err_msg=f"iteration round {r}: ranks differ")
        np.testing.assert_array_equal(a0[0], exp[r]["lo"])
        np.testing.assert_array_equal(a0[1], exp[r]["hi"])
        np.testing.assert_array_equal(a0[3], exp[r]["counts"])
        np.testing.assert_allclose(a0[2], exp[r]["sums"], rtol=1e-12, atol=0)
