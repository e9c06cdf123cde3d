"""Data-parallel CUDA path (SURVEY §8e) against the oracle, world_size 2, one process per GPU (needs 2 GPUs; skipped on a
machine with one).  Both gradient exchanges — the NVLink peer-memory push inside the loss/grad
kernel's fused tail and the NCCL allreduce — must
  * leave bit-identical parameters on the two ranks,
  * match oracle.ppo run on the UNION minibatches (per-minibatch advantage normalisation over the global minibatch,
    ppo.jl:350-356; clip + Adam on the global mean gradient),
and a data-parallel Pendulum + NormalizeWrapperEnv rollout must end with identical normaliser statistics on both ranks that
equal the Chan merge (normalizeWrapperEnv.jl:37-48) over all shards."""
import os
import socket

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


N_LOCAL, T, EPOCHS, SEED = 96, 20, 2, 777


def _worker(rank, world, port, out):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ.setdefault("NCCL_DEBUG", "WARN")
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    import ctypes as C
    import dril_b200 as D
    from dril_b200 import _lib as L
    from oracle import policy as OP

    def all_gather(b):
        o = [None] * world
        dist.all_gather_object(o, b)
        return o

    res = {}
    for path in ("nccl", "p2p", "p2p_persistent"):
        # "p2p_persistent": the exchange inside the persistent step loop (option "persistent" = 2; off by default in data-parallel runs)
        D.set_option("persistent", 2 if path == "p2p_persistent" else 1)
        ctx = D.Context(device=rank, seed=0)
        uid = [D.Context.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.comm_init(rank, world, uid[0])
        spec = OP.PolicySpec(4, [64, 64], "discrete", 2, act_start=1)
        flat = OP.init_params(spec, seed=6)
        env = D.CudaBatchedEnv("cartpole", N_LOCAL, max_steps=12, seed=31, ctx=ctx, monitor_window=100, gid_offset=rank * N_LOCAL)
        layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=[64, 64])
        alg = D.PPO(n_steps=T, batch_size=T * N_LOCAL // 2, epochs=EPOCHS, ent_coef=0.01)
        agent = D.Agent(layer, alg, rng=np.random.default_rng(0), ctx=ctx)
        agent.set_parameters(flat)
        if path != "nccl":
            ctx.comm_p2p_setup(all_gather, agent.device.n_params + 8)
        forced = np.random.default_rng(100 + rank).integers(1, 3, (T, N_LOCAL))
        buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, N_LOCAL, ctx=ctx)
        D.collect_rollout(buf, agent, alg, env, forced_actions=forced)
        shard = {k: buf.download(k) for k in ("obs", "actions", "rewards", "values", "logprobs", "advantages", "returns")}
        st = D.IterStats()
        h = alg.hyper()
        L.check(ctx.lib.dril_ppo_update(agent.device.h, buf.h, C.byref(h), alg.epochs, alg.batch_size, SEED, 3, C.byref(st)))
        res[path] = dict(params=agent.device.get_params(), shard=shard, stats=st.as_dict(), monitor=env.monitor_stats())
        buf.close(); env.close(); agent.device.close()
    D.set_option("persistent", 1)
    # ---- data-parallel Pendulum + NormalizeWrapperEnv: one rollout with replayed actions, then the merged statistics --------
    ctx = D.Context(device=rank, seed=0)
    uid = [D.Context.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    ctx.comm_init(rank, world, uid[0])
    n, Tp = 64, 10
    env = D.CudaBatchedEnv("pendulum", n, max_steps=7, seed=5, ctx=ctx, monitor_window=100, gid_offset=rank * n, normalize=D.NormalizeConfig())
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=[16, 16])
    alg = D.PPO(n_steps=Tp, batch_size=Tp * n, epochs=1)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0), ctx=ctx)
    ctx.comm_p2p_setup(all_gather, agent.device.n_params + 8)
    forced = np.random.default_rng(200 + rank).normal(size=(Tp, n, 1)).astype(np.float32)
    buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, Tp, n, ctx=ctx)
    D.collect_rollout(buf, agent, alg, env, forced_actions=forced)
    res["norm"] = dict(stats=env.norm_stats(), forced=forced, monitor=env.monitor_stats(), rewards=buf.download("rewards"))
    # a full train! on top (sampled actions): statistics stay identical across ranks, parameters too
    out_t = D.train(agent, env, alg, 2 * Tp * n)
    res["norm_train"] = dict(stats=env.norm_stats(), params=agent.train_state.parameters.copy(), ok=out_t is not None)
    np.save(out + f".rank{rank}.npy", res, allow_pickle=True)
    dist.barrier()
    dist.destroy_process_group()


def _relerr(a, b):
    return np.linalg.norm(a.astype(np.float64) - b) / max(np.linalg.norm(b), 1e-30)


def test_dp_cuda_paths_vs_oracle(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from oracle import envs as OE, policy as OP, ppo as OO
    out = str(tmp_path / "dp")
    mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    R = [np.load(out + f".rank{r}.npy", allow_pickle=True).item() for r in range(2)]
    spec = OP.PolicySpec(4, [64, 64], "discrete", 2, act_start=1)
    flat = OP.init_params(spec, seed=6)
    for path in ("nccl", "p2p", "p2p_persistent"):
        np.testing.assert_array_equal(R[0][path]["params"], R[1][path]["params"], err_msg=f"{path}: ranks differ")
        shards = [R[r][path]["shard"] for r in range(2)]
        n_tot = T * N_LOCAL
        bs = n_tot // 2
        cfg = OO.PPOConfig(n_steps=T, batch_size=2 * bs, epochs=EPOCHS, ent_coef=0.01)
        opt = OO.Adam(flat.size, lr=cfg.learning_rate)
        cur = flat.copy()
        rec = {k: [] for k in ("policy_loss", "value_loss", "loss", "grad_norm")}
        flatten = lambda s, k: s[k].reshape(n_tot, -1) if k in ("obs", "actions") else s[k].reshape(n_tot)
        for e in range(EPOCHS):
            idx = [OO.minibatch_indices(n_tot, bs, 3 + e, r, SEED) for r in range(2)]
            for i in range(len(idx[0])):
                cat = lambda k: np.concatenate([flatten(shards[r], k)[idx[r][i]] for r in range(2)])
                loss, stats, g = OO.ppo_loss_and_grads(spec, cur, cat("obs"), cat("actions"), cat("advantages"), cat("returns"),
                                                       cat("logprobs"), cat("values"), cfg)
                g, norm = OO.clip_grads(g, cfg.max_grad_norm)
                cur = opt.step(cur, g)
                rec["policy_loss"].append(stats["policy_loss"]); rec["value_loss"].append(stats["value_loss"])
                rec["loss"].append(loss); rec["grad_norm"].append(norm)
        got = R[0][path]["params"]
        assert _relerr(got - flat, cur - flat) < 2e-3, (path, _relerr(got - flat, cur - flat))
        np.testing.assert_allclose(got, cur, rtol=1e-4, atol=2e-6, err_msg=path)
        st = R[0][path]["stats"]
        assert st["n_minibatch_steps"] == EPOCHS * 2
        for k, v in rec.items():
            m = float(np.mean(np.asarray(v, np.float32)))
            assert abs(st[k] - m) <= 2e-4 * max(1.0, abs(m)), (path, k, st[k], m)
    assert np.abs(R[0]["nccl"]["params"] - R[0]["p2p"]["params"]).max() <= 1e-6
    np.testing.assert_array_equal(R[0]["p2p"]["params"], R[0]["p2p_persistent"]["params"])     # same kernel, same order of sums
    # ---- normaliser merge: both ranks hold the Chan merge over all shards ------------------------------------------------------
    s0, s1 = R[0]["norm"]["stats"], R[1]["norm"]["stats"]
    for k in ("obs_mean", "obs_var"):
        np.testing.assert_array_equal(s0[k], s1[k])
    assert (s0["obs_count"], s0["ret_count"], s0["ret_mean"], s0["ret_var"]) == (s1["obs_count"], s1["ret_count"], s1["ret_mean"], s1["ret_var"])
    n, Tp = 64, 10
    assert s0["obs_count"] == 2 * n * (Tp + 1) and s0["ret_count"] == 2 * n * Tp
    # single-process oracle over all 2 n envs with the same replayed actions: the raw trajectories do not depend on the
    # normaliser, so its sequentially merged statistics equal the merged per-rollout moments up to rounding
    o = OE.NormalizeWrapper(OE.MonitorWrapper(OE.ParallelEnv(OE.PendulumBatch(2 * n, seed=5, max_steps=7))), 3)
    forced = np.concatenate([R[0]["norm"]["forced"], R[1]["norm"]["forced"]], axis=1)
    pspec = OP.PolicySpec(3, [16, 16], "continuous", 1, act_low=[-2], act_high=[2])
    OO.collect_rollout_timemajor(o, pspec, OP.init_params(pspec, seed=0), Tp, forced_actions=forced)
    np.testing.assert_allclose(s0["obs_mean"], o.obs_rms.mean, rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(s0["obs_var"], o.obs_rms.var, rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose([s0["ret_mean"], s0["ret_var"]], [o.ret_rms.mean, o.ret_rms.var], rtol=1e-4, atol=1e-5)
    # Monitor sums are global: both ranks report the same episode totals, and they equal the oracle's
    assert R[0]["norm"]["monitor"]["total_episodes"] == R[1]["norm"]["monitor"]["total_episodes"] == o.env.total_episodes
    t0, t1 = R[0]["norm_train"], R[1]["norm_train"]
    assert t0["ok"] and t1["ok"]
    np.testing.assert_array_equal(t0["params"], t1["params"])
    np.testing.assert_array_equal(t0["stats"]["obs_mean"], t1["stats"]["obs_mean"])
    assert t0["stats"]["obs_count"] == t1["stats"]["obs_count"] == 2 * n * (Tp + 1) * 3
