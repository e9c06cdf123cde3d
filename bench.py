#!/usr/bin/env python
"""bench.py — end-to-end PPO env-steps/s (BASELINE.json metric) on N B200s of one node.

A "step" is one PPO iteration of the hot path: fused rollout (n_steps x n_envs env steps with the
actor-critic in the loop) -> GAE -> `epochs` x `n_minibatches` fused loss/grad + clip + Adam
updates, over synthetic env batches of the named shape with random-init weights.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--repeats R] [--impl ours|reference] [--workload c2|c3|c4|c5]
                  [--dump-outputs DIR]

The default line measures C2 (BASELINE configs[1]) as `value` and carries C4 (65 536 envs/GPU, every N) and C3 (one GPU) under
`workloads`; --workload c5 runs the rollout-only sweep.

The timed steps of a workload are exactly K iterations, after a fixed number of untimed ones (the workload's `warmup`, or W if
larger), so the state every step starts from depends only on the arguments.  --dump-outputs DIR writes what the last timed
step of the main workload returned (dump_outputs()), to compare two builds output for output.

N > 1 is launched with torch.distributed.run (one rank per GPU): envs shard across
ranks (weak scaling: per-GPU env count fixed), gradients are allreduced over NVLink peer memory per minibatch
(NCCL fallback with DRIL_NO_P2P=1).
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True        # the benchmark leaves the source tree as it found it (it may be read-only)

# warmup: untimed iterations before the timed steps, about 0.3 s of work on one B200 (sustained clocks, steady-state enqueue
# path).  A fixed count, not a time, because what an iteration costs depends on how far training has come: on a B200 at its
# 1000 W limit a C2 iteration takes 1.61 ms after 3 iterations and 1.67 ms after 190.
WORKLOADS = {
    # BASELINE.json configs[1]: the configuration the metric is quoted on (fits one GPU)
    "c2": dict(name="PPO CartPole, 4096 batched envs/GPU, n_steps=128, hidden [64,64], discrete categorical policy",
               kind="cartpole", n_envs=4096, n_steps=128, hidden=[64, 64], normalize=False, warmup=190),
    "c3": dict(name="PPO Pendulum diag-Gaussian, 16384 envs/GPU, n_steps=128, hidden [128,128,64], NormalizeWrapperEnv obs+reward",
               kind="pendulum", n_envs=16384, n_steps=128, hidden=[128, 128, 64], normalize=True, warmup=15),
    "c4": dict(name="PPO CartPole, 65536 envs/GPU data-parallel, n_steps=128, hidden [64,64]",
               kind="cartpole", n_envs=65536, n_steps=128, hidden=[64, 64], normalize=False, warmup=18),
}
EPOCHS, N_MINIBATCHES = 4, 4          # BASELINE.json does not fix these (SURVEY §8d); stated with every number
METRIC, UNIT = "end-to-end PPO env-steps/sec", "env-steps/s"
DUMP_BYTES = 64 * 10 ** 6             # --dump-outputs: the whole dump stays below this


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], bf16_burst=d["bf16_tflops"], bf16_sustained=d["bf16_tflops_sustained"],
                    sm_max_mhz=d.get("sm_max_mhz", 1965.0), source="measured")
    return dict(hbm=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, sm_max_mhz=1965.0, source="fallback")


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region through NVML (a polling thread in this
    process; an external `nvidia-smi -lms` loop measurably slowed the timed kernels)."""

    def __init__(self, gpu_index):
        self.idx, self.samples, self.stop_flag, self.th, self.err = gpu_index, [], False, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.idx]) if vis and vis.split(",")[self.idx].isdigit() else self.idx
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.mx = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def _poll(self):
        # every NVML query stalls the GPU front end for ~1.5 ms (measured: 4 samples cost 13 % of a 50 ms region), so the
        # region is sampled sparsely: once 10 ms after the start, then every 100 ms; the max clock is read before it
        nv = self.nv
        time.sleep(0.01)
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((sm, self.mx, rs, None))
            except Exception as e:  # pragma: no cover
                self.err = repr(e)
                return
            for _ in range(10):
                if self.stop_flag:
                    break
                time.sleep(0.01)

    def stop(self):
        if self.th is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: %s" % self.err]}
        self.stop_flag = True
        self.th.join(timeout=1.0)
        nv = self.nv
        names = {getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
                 getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                 getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                 getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap"}
        reasons = set()
        for (_, _, rs, _) in self.samples:
            for bit, name in names.items():
                if rs & bit:
                    reasons.add(name)
        sm = [x[0] for x in self.samples]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(x[1] for x in self.samples) if sm else None,
                "reasons": sorted(reasons), "samples": len(sm),
                "how": "NVML (clock + event reasons) inside the timed region: 10 ms after its start, then every 100 ms"}


def dist_setup(n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        # NCCL writes its version banner / debug lines to stdout by default: stdout carries ONE JSON line only
        os.environ.setdefault("NCCL_DEBUG", "WARN")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        return rank, world, local, dist
    return rank, world, local, None


def dump_outputs(out_dir, agent, buf, stats):
    """Writes what one PPO iteration hands its caller, as out_dir/<name>.npy in float32 or float64: the updated policy
    parameters (params), the iteration statistics without its two timings (stat_<field>) and every rollout buffer field
    (buf_<field>, time-major [n_steps, n_envs, ...]).  When the buffer would take the dump above DUMP_BYTES, its fields keep a
    fixed, seeded sample of env columns; env_index lists the columns kept."""
    os.makedirs(out_dir, exist_ok=True)
    out = {"params": agent.device.get_params()}
    out.update({"stat_" + k: np.array([v], np.float64) for k, v in stats.as_dict().items() if k not in ("rollout_ms", "update_ms")})
    fields = {f: buf.download(f) for f in ("obs", "actions", "rewards", "values", "logprobs", "advantages", "returns", "flags",
                                           "boot", "last_values", "episode_r", "episode_l")}
    n_envs = buf.n_envs
    per_env = 8 + sum(4 * a.size // n_envs for a in fields.values())                # float32 columns + their env_index entry
    fixed = sum(a.nbytes for a in out.values()) + 128 * (len(out) + len(fields) + 1)  # + one .npy header per file
    keep = min(n_envs, (DUMP_BYTES - fixed) // per_env)
    idx = np.arange(n_envs) if keep == n_envs else np.sort(np.random.default_rng(0).choice(n_envs, keep, replace=False))
    out["env_index"] = idx.astype(np.float64)
    for f, a in fields.items():
        out["buf_" + f] = (a[idx] if f == "last_values" else a[:, idx]).astype(np.float32)   # flags, actions, lengths: exact
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measure(D, ctx, dist, rank, world, local, wname, steps, repeats, warmup, p2p_state, clock_sampler=None, dump_dir=None):
    """One workload on this rank's GPU: `steps` timed PPO iterations in `repeats` (or fewer) equal blocks (CUDA events on the
    library's stream, L2 flushed before every iteration, max over ranks per block, median over blocks), the same through
    train! (wall clock), and a per-kernel CUDA-event profile.  With dump_dir, rank 0 writes what the last timed iteration
    returned there.  Returns a dict; every rank must call it with the same arguments."""
    import ctypes as C
    from dril_b200 import _lib as L
    w = WORKLOADS[wname]
    n_envs, n_steps = w["n_envs"], w["n_steps"]
    env = D.CudaBatchedEnv(w["kind"], n_envs, seed=0, ctx=ctx, monitor_window=100, gid_offset=rank * n_envs,
                           normalize=D.NormalizeConfig() if w["normalize"] else None)
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=w["hidden"])
    batch = n_steps * n_envs // N_MINIBATCHES                      # per-rank minibatch; global = batch * world
    alg = D.PPO(n_steps=n_steps, batch_size=batch, epochs=EPOCHS)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0), ctx=ctx)   # same init on every rank
    comm = "single GPU"
    if world > 1:
        comm = "NCCL allreduce of the flat gradient per minibatch"
        if os.environ.get("DRIL_NO_P2P", "0") != "1":
            if p2p_state.get("slots", 0) < agent.device.n_params + 8:
                def all_gather(b):
                    out = [None] * world
                    dist.all_gather_object(out, b)
                    return out
                ctx.comm_p2p_setup(all_gather, agent.device.n_params + 8)
                p2p_state["slots"] = agent.device.n_params + 8
            comm = ("one-shot NVLink peer-memory allreduce (push) of the flat gradient inside the loss/grad kernel's fused tail; "
                    "advantage / explained-variance / normaliser moments through a second small peer-memory kernel; no NCCL on the data path")
    buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, n_steps, n_envs, ctx=ctx)
    lib, hyper = ctx.lib, alg.hyper()
    steps_per_iter = n_steps * n_envs
    pending = [0]
    last_stats = [None]

    def read_result():
        s_ = L.IterStats()
        L.check(lib.dril_iteration_result(agent.device.h, C.byref(s_)))
        pending[0] -= 1
        last_stats[0] = s_
        return s_

    def iteration_async():
        # results are read in FIFO order and at most 4 iterations may be in flight: reading an OLD result waits on that
        # iteration's event only, so the host stays ahead of the device and the stream never drains inside a timed loop
        if pending[0] >= int(os.environ.get('BENCH_PENDING', '3')):
            read_result()
        L.check(lib.dril_ppo_iteration_async(env.h, agent.device.h, buf.h, C.byref(hyper), alg.epochs, alg.batch_size,
                                             agent.shuffle_seed, agent.epoch_counter))
        agent.epoch_counter += alg.epochs
        pending[0] += 1

    def drain():
        while pending[0] > 0:
            read_result()
        return last_stats[0]

    def barrier():
        ctx.synchronize()
        if dist:
            dist.barrier()
        ctx.synchronize()

    def max_over_ranks(x):
        if not dist:
            return x
        import torch
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # every allocation up front, then all ranks together: no rank sits in a cudaMalloc while a peer's GPU already spins in an exchange
    L.check(lib.dril_iteration_prepare(env.h, agent.device.h, buf.h, int(alg.epochs), int(alg.batch_size)))
    barrier()
    # ---- warm-up: max(W, the workload's warm-up) untimed steps, each like a timed one (the first flush allocates its buffer).
    # A fixed count: the timed steps start from a state that depends on the arguments only ----------------------------------
    n_w = max(warmup, w["warmup"])
    for _ in range(n_w):
        ctx.flush_l2()
        iteration_async()
    drain()
    # ---- value: K iterations resident on the device in up to `repeats` equal blocks, CUDA events on the launching stream ----
    n_blocks = max(b for b in range(1, max(repeats, 1) + 1) if steps % b == 0)
    per_block = steps // n_blocks
    barrier()
    if clock_sampler is not None:
        clock_sampler.start()
    launches0 = ctx.launch_count()
    block_ms = []
    for _ in range(n_blocks):
        barrier()
        ctx.event_record(0)
        for _ in range(per_block):
            ctx.flush_l2()                  # inside the timed region: nothing stays L2-hot from the previous step
            iteration_async()
        ctx.event_record(1)
        barrier()
        block_ms.append(max_over_ranks(ctx.event_elapsed_ms(0, 1)))
    clocks = clock_sampler.stop() if clock_sampler is not None else None
    launches = (ctx.launch_count() - launches0) // n_blocks
    st = drain()
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, agent, buf, st)
    ms = float(np.median(block_ms))
    value = steps_per_iter * world * per_block / (ms * 1e-3)

    # ---- e2e: the public API call (train!) with host parameters in and statistics out (no L2 flush on this path) -------
    D.train(agent, env, alg, steps_per_iter * 3)       # warm-up of the public path (its rollout buffer is allocated once per agent)
    e2e_s = []
    for _ in range(min(repeats, 3)):
        barrier()
        t0 = time.perf_counter()
        out = D.train(agent, env, alg, steps_per_iter * steps)
        ctx.synchronize()
        e2e_s.append(max_over_ranks(time.perf_counter() - t0))
        assert out is not None and np.isfinite(out[0]["losses"]).all()
    e2e_value = steps_per_iter * world * steps / float(np.median(e2e_s))
    n_params = agent.device.n_params
    h2d = int(n_params * 4 / steps + C.sizeof(L.PPOHyper))       # parameters once per train! + hyper per iteration
    d2h = int(n_params * 4 / steps + C.sizeof(L.IterStats) + 64)

    # ---- per-kernel CUDA-event profile of the same steps (roofline) ---------------------------------------------------
    ctx.set_profiling(True)
    ctx.reset_profile()
    for _ in range(steps):
        ctx.flush_l2()
        iteration_async()
    ctx.synchronize()
    prof = ctx.profile()
    ctx.set_profiling(False)
    st = drain()
    barrier()
    total_prof_ms = sum(v[0] for v in prof.values()) or 1.0
    kern = {}
    for name, (tms, n) in prof.items():
        if n:
            kern[name] = {"ms_per_step": tms / steps, "launches_per_step": n / steps, "share": tms / total_prof_ms}
    res = dict(workload=w["name"], value=value, ms_per_step=ms / per_block, block_ms=block_ms, repeats=n_blocks, steps=steps,
               per_block=per_block, e2e=e2e_value, h2d=h2d, d2h=d2h, launches=int(launches), clocks=clocks, kernels=kern, comm=comm,
               batch=batch, steps_per_iter=steps_per_iter, warmup_run=n_w, path=agent.device.update_path(),
               layer_dims=[layer.layer_dims(0), layer.layer_dims(1)], obs_dim=env.obs_dim,
               last=({k: (v if np.isfinite(v) else None) for k, v in st.as_dict().items()}))
    buf.close(); env.close(); agent.device.close()
    for b in getattr(agent, "_roll_buffers", {}).values():
        b.close()
    return res


def rooflines_of(res, pk):
    """Per-kernel rooflines of one measured workload (algorithmic bytes / flops per iteration: SURVEY §8d, DESIGN.md §4)."""
    kern, spi = res["kernels"], res["steps_per_iter"]
    D_obs = res["obs_dim"]
    fwd_flops = 2 * sum(i * o for net in (0, 1) for (i, o) in res["layer_dims"][net])
    hid_flops = 2 * sum(i * o for net in (0, 1) for (i, o) in res["layer_dims"][net][1:-1])
    ro = kern.get("rollout", {"ms_per_step": float("nan")})
    lg = kern.get("loss_grad", {"ms_per_step": float("nan")})
    gae = kern.get("gae", {"ms_per_step": float("nan")})
    pm = kern.get("permute")
    fp32_peak = 148 * 128 * 2 * pk["sm_max_mhz"] * 1e6 / 1e12
    lg_flops = 3 * fwd_flops * spi * EPOCHS
    lg_bytes = (4 * D_obs + 4 + 12) * spi * EPOCHS
    t_lg = lg["ms_per_step"] * 1e-3
    r = {
        "rollout": {"bound": "hbm", "achieved": (4 * D_obs + 17) * spi / (ro["ms_per_step"] * 1e-3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                    "fp32_tflops": fwd_flops * spi / (ro["ms_per_step"] * 1e-3) / 1e12, "share": ro.get("share")},
        "gae": {"bound": "hbm", "achieved": 17 * spi / (gae["ms_per_step"] * 1e-3) / 1e9, "peak": pk["hbm"], "unit": "GB/s", "share": gae.get("share")},
        "loss_grad": {"bound": "tensor", "achieved": lg_flops / t_lg / 1e12, "peak": pk["bf16_sustained"], "unit": "TFLOP/s",
                      "hbm_gbs": lg_bytes / t_lg / 1e9, "frac_of_fp32_fma_peak": lg_flops / t_lg / 1e12 / fp32_peak,
                      "share": lg.get("share"), "path": res["path"],
                      # the hidden GEMMs (fwd, dH, dW) are issued three times (hi*hi + lo*hi + hi*lo)
                      "tensor_issued_tflops": 3 * 3 * hid_flops * spi * EPOCHS / t_lg / 1e12 if res["path"] in ("tensor", "mma") else 0.0},
    }
    if pm:
        r["permute"] = {"bound": "hbm", "achieved": 2 * (4 * D_obs + 20) * spi * EPOCHS / (pm["ms_per_step"] * 1e-3) / 1e9, "peak": pk["hbm"],
                        "unit": "GB/s", "share": pm.get("share")}
    for x in r.values():
        x["frac"] = x["achieved"] / x["peak"]
    return r


def run_ours(args):
    import dril_b200 as D
    import __graft_entry__
    rank, world, local, dist = dist_setup(args.gpus)
    if rank == 0:
        __graft_entry__.build()
    if dist:
        dist.barrier()
    ctx = D.Context(device=local, seed=0)
    if world > 1:
        uid = [D.Context.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.comm_init(rank, world, uid[0])
    if args.workload == "c5":
        return run_c5(args, D, ctx, dist, rank, world, local)
    p2p_state = {}
    sampler = ClockSampler(local) if rank == 0 and not os.environ.get('BENCH_NO_SAMPLER') else None
    main_w = args.workload
    res = measure(D, ctx, dist, rank, world, local, main_w, args.steps, args.repeats, args.warmup, p2p_state, sampler,
                  dump_dir=args.dump_outputs)
    # the other BASELINE configs ride along in the same line (a plain `--gpus/--steps/--warmup` run reports them too): C4
    # (65 536 envs/GPU, the data-parallel config) at every N, C3 (Pendulum, wide net, normaliser) on one GPU
    extra = {}
    if main_w == "c2" and not args.no_extra:
        extra["c4"] = measure(D, ctx, dist, rank, world, local, "c4", max(2, args.steps // 4), min(args.repeats, 3), 3, p2p_state)
        if world == 1:
            extra["c3"] = measure(D, ctx, dist, rank, world, local, "c3", max(2, args.steps // 8), min(args.repeats, 3), 3, p2p_state)
    if rank != 0:
        if dist:
            dist.barrier()
            dist.destroy_process_group()
        return
    pk = peaks()
    rooflines = rooflines_of(res, pk)
    kern = res["kernels"]
    dominant = max(kern, key=lambda k: kern[k]["share"])
    roof = dict(rooflines.get(dominant, rooflines["loss_grad"]))
    lg_path = res["path"]
    if lg_path == "tensor":
        note = ("loss_grad: features-on-lanes tcgen05 kernel (update_ft.cuh): all GEMMs of both nets (layer 0 included) on tcgen05.mma "
                "kind::f16 with the fp16 hi/lo split (hi*hi + lo*hi + hi*lo, fp32 accumulation in TMEM, 22 significant bits, gradient "
                "error ~1e-6 vs the oracle), deltas rescaled per tile by a power of two; achieved = fp32-equivalent algorithmic FLOPs "
                "(fwd + 2x bwd) / time, peak = measured dense bf16 by contract; tensor_issued_tflops counts the three issued products; "
                "one persistent cooperative launch runs all minibatch steps of the iteration (Adam and the gradient exchange in its tail); "
                "the kernel is bound by the shared-memory pipe (UMMA operand reads + LDS/STS of the CUDA-core phases), see DESIGN.md")
    elif lg_path == "mma":
        note = ("general-shape loss_grad kernel: hidden GEMMs on warp-level tensor-core tiles (mma.sync m16n8k8 TF32, 3xTF32 split, "
                "fp32-level accuracy), thin layers and loss head on CUDA cores; achieved = fp32-equivalent algorithmic FLOPs / time, "
                "peak = measured dense bf16 (tcgen05 path) by contract")
    else:
        note = ("fp32 CUDA-core kernels; frac is against the tensor peak by contract, frac_of_fp32_fma_peak is the pipe it actually runs on")
    # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` captures of workload C2
    # (profiles/r02_lossgrad_ft_summary.txt, profiles/r01_rollout_tc_final_summary.txt); null for other workloads
    # (the loss/grad launch is the persistent kernel: one launch = the 16 minibatch steps of an iteration, 76.2 MB read + 3.7 MB written
    # against 75.5 MB of algorithmic record bytes)
    traffic_c2 = {"loss_grad": 76.2e6 + 3.7e6, "rollout": 192.3e3} if (main_w == "c2" and lg_path == "tensor") else {}
    roof.update({"kernel": dominant, "traffic": traffic_c2.get(dominant),
                 "peak_source": pk["source"] + (" sustained bf16" if roof["bound"] == "tensor" else " copy"), "note": note})
    w = WORKLOADS[main_w]
    cfg_of = lambda r: {"workload": r["workload"], "epochs": EPOCHS, "minibatches_per_epoch": N_MINIBATCHES, "batch_size_per_gpu": r["batch"],
                        "env_steps_per_step_per_gpu": r["steps_per_iter"], "adam_steps_per_step": EPOCHS * N_MINIBATCHES,
                        "l2": "value: flushed (256 MB memset on the stream before every timed step, inside the timed region); e2e (train!) "
                              "does not pay the flush", "warmup_iterations_run": r["warmup_run"],
                        "timing": f"{r['steps']} timed steps: median of {r['repeats']} blocks of {r['per_block']} steps (CUDA events, "
                                  "max over ranks per block)",
                        "parallelism": f"dp{world} over envs, {r['comm']}" if world > 1 else "single GPU"}
    line = {
        "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": res["warmup_run"],
        "repeats": res["repeats"], "block_ms": res["block_ms"],
        "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic (on-device env batches of the named shape, orthogonal random-init weights, seed 0)",
        "config": cfg_of(res),
        "e2e": {"value": res["e2e"], "unit": UNIT, "h2d_bytes_per_step": res["h2d"], "d2h_bytes_per_step": res["d2h"],
                "api": "dril_b200.train (train!): host parameters in, per-iteration learn_stats + final parameters out, wall clock, "
                       "median of 3 calls"},
        "gpu_launches": res["launches"] * res["repeats"],
        "gpu_launches_per_block": res["launches"],
        "clocks": res["clocks"],
        "roofline": roof,
        "rooflines": rooflines,
        "kernels": kern,
        "last_iteration": res["last"],
    }
    if extra:
        line["workloads"] = {}
        for k, r in extra.items():
            rf = rooflines_of(r, pk)
            line["workloads"][k] = {"value": r["value"], "unit": UNIT, "ms_per_step": r["ms_per_step"], "steps": r["steps"], "repeats": r["repeats"],
                                    "block_ms": r["block_ms"], "e2e": r["e2e"], "config": cfg_of(r), "kernels": r["kernels"],
                                    "rooflines": rf, "gpu_launches_per_block": r["launches"], "update_path": r["path"]}
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(main_w)
    print(json.dumps(line), flush=True)
    if dist:
        dist.barrier()
        dist.destroy_process_group()


def run_c5(args, D, ctx, dist, rank, world, local):
    """BASELINE config C5: synthetic rollout-only sweep (policy forward + env step + GAE, no update), n_envs 2^10..2^20 x obs_dim
    4..64 per GPU; reports env-steps/s and the rollout kernel's HBM fraction (algorithmic 4 D + 17 B per env-step written, 17 B
    read + 8 B written by GAE) per point; `value` is the best point's throughput."""
    import ctypes as C
    from dril_b200 import _lib as L
    pk = peaks()
    hidden = [int(x) for x in os.environ.get("C5_HIDDEN", "8").split(",") if x]
    points = []
    n_steps = 128
    grid = [(o, l) for o in (4, 16, 64) for l in (10, 14, 17, 20)]
    if os.environ.get("C5_POINTS"):                      # e.g. "16:17,64:17" (obs_dim:log2 n_envs): profiling single points
        grid = [tuple(int(v) for v in q.split(":")) for q in os.environ["C5_POINTS"].split(",")]
    for obs_dim, lg_n in grid:
        if True:
            n_envs = 1 << lg_n
            env = D.CudaBatchedEnv("synthetic", n_envs, obs_dim=obs_dim, seed=0, ctx=ctx, monitor_window=0, gid_offset=rank * n_envs)
            layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=hidden)
            alg = D.PPO(n_steps=n_steps)
            agent = D.Agent(layer, alg, rng=np.random.default_rng(0), ctx=ctx)
            buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, n_steps, n_envs, ctx=ctx)
            fps = L.c_f32(0)
            for _ in range(3):
                L.check(ctx.lib.dril_rollout_collect(env.h, agent.device.h, buf.h, None, C.byref(fps)))
                buf.compute_advantages()
            ctx.set_profiling(True); ctx.reset_profile()
            reps = 5 if lg_n < 20 else 3
            for _ in range(reps):
                ctx.flush_l2()
                L.check(ctx.lib.dril_rollout_collect(env.h, agent.device.h, buf.h, None, C.byref(fps)))
                buf.compute_advantages()
            ctx.synchronize()
            prof = ctx.profile(); ctx.set_profiling(False)
            ro_ms, gae_ms = prof["rollout"][0] / reps, prof["gae"][0] / reps
            spi = n_steps * n_envs
            points.append({"n_envs": n_envs, "obs_dim": obs_dim, "rollout_ms": ro_ms, "gae_ms": gae_ms,
                           "env_steps_per_s": spi / ((ro_ms + gae_ms) * 1e-3),
                           "rollout_gbs": (4 * obs_dim + 17) * spi / (ro_ms * 1e-3) / 1e9,
                           "rollout_hbm_frac": (4 * obs_dim + 17) * spi / (ro_ms * 1e-3) / 1e9 / pk["hbm"],
                           "gae_gbs": 17 * spi / (gae_ms * 1e-3) / 1e9, "gae_hbm_frac": 17 * spi / (gae_ms * 1e-3) / 1e9 / pk["hbm"]})
            buf.close(); env.close(); agent.device.close()
    if rank != 0:
        return
    best = max(points, key=lambda p: p["rollout_hbm_frac"])
    line = {"metric": "rollout-only env-steps/sec (synthetic sweep, C5)", "value": best["env_steps_per_s"] * world, "unit": UNIT, "n_gpus": world,
            "steps": 5, "warmup": 3, "ms_per_step": best["rollout_ms"] + best["gae_ms"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic env (Philox observations / rewards / terminations)",
            "config": {"workload": "Synthetic rollout-only sweep: 1k-1M envs/GPU, obs_dim 4-64, policy forward + GAE", "hidden": hidden,
                       "n_steps": n_steps, "l2": "flushed before every timed rollout"},
            "roofline": {"bound": "hbm", "achieved": best["rollout_gbs"], "peak": pk["hbm"], "unit": "GB/s", "frac": best["rollout_hbm_frac"],
                         "kernel": "rollout", "traffic": None, "peak_source": pk["source"] + " copy", "point": best},
            "sweep": points}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the restated CPU reference (oracle/, NumPy + threaded BLAS).
# DRiL.jl itself cannot run here: there is no Julia toolchain in the image (SURVEY §8c).
# ---------------------------------------------------------------------------------------------
def _oracle_iteration_rate(workload, sample_envs, iterations):
    from oracle import envs as OE, policy as OP, ppo as OO
    w = WORKLOADS[workload]
    n_steps = w["n_steps"]
    if w["kind"] == "cartpole":
        spec = OP.PolicySpec(4, w["hidden"], "discrete", 2, act_start=1)
        env = OE.MonitorWrapper(OE.ParallelEnv(OE.CartPoleBatch(sample_envs, seed=0)))
    else:
        spec = OP.PolicySpec(3, w["hidden"], "continuous", 1, act_low=[-2], act_high=[2])
        env = OE.MonitorWrapper(OE.ParallelEnv(OE.PendulumBatch(sample_envs, seed=0)))
        if w["normalize"]:
            env = OE.NormalizeWrapper(env, 3)
    flat = OP.init_params(spec, seed=0)
    cfg = OO.PPOConfig(n_steps=n_steps, batch_size=n_steps * sample_envs // N_MINIBATCHES, epochs=EPOCHS)
    OO.train(env, spec, flat, cfg, n_steps * sample_envs)              # warm-up iteration
    t0 = time.perf_counter()
    OO.train(env, spec, flat, cfg, n_steps * sample_envs * iterations)
    dt = time.perf_counter() - t0
    return n_steps * sample_envs * iterations / dt, dt


def _oracle_c1_rate():
    """BASELINE configs[0], the reference's own CPU-runnable quick-start shape (SURVEY §8d): CartPole, 4 envs, n_steps 2048,
    batch 64, epochs 10, default [64,64] layer; one warm-up iteration + one timed iteration of the restated reference."""
    from oracle import envs as OE, policy as OP, ppo as OO
    spec = OP.PolicySpec(4, [64, 64], "discrete", 2, act_start=1)
    env = OE.MonitorWrapper(OE.ParallelEnv(OE.CartPoleBatch(4, seed=0)))
    flat = OP.init_params(spec, seed=0)
    cfg = OO.PPOConfig(n_steps=2048, batch_size=64, epochs=10)
    OO.train(env, spec, flat, cfg, 2048 * 4)
    t0 = time.perf_counter()
    OO.train(env, spec, flat, cfg, 2048 * 4)
    dt = time.perf_counter() - t0
    return 2048 * 4 / dt, dt


def julia_probe():
    import shutil
    exe = shutil.which("julia")
    if not exe:
        return "julia not found on PATH: DRiL.jl itself cannot be timed on this box (no Julia toolchain in the image, no network)"
    try:
        return subprocess.run([exe, "--version"], capture_output=True, text=True, timeout=20).stdout.strip()
    except Exception as e:  # pragma: no cover
        return f"julia at {exe} did not answer: {e!r}"


def cpu_baseline(workload):
    sample_envs = max(64, WORKLOADS[workload]["n_envs"] // 8)
    rate, dt = _oracle_iteration_rate(workload, sample_envs, 2)
    c1_rate, c1_dt = _oracle_c1_rate()
    return {"value": rate, "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
            "sample": f"restated reference (Python/NumPy, threaded BLAS), not DRiL.jl: 2 PPO iterations of {sample_envs} envs x "
                      f"{WORKLOADS[workload]['n_steps']} steps, epochs {EPOCHS}, {N_MINIBATCHES} minibatches ({dt:.1f} s)",
            "c1": {"value": c1_rate, "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
                   "sample": f"BASELINE configs[0] shape: CartPole, 4 envs, n_steps 2048, batch 64, epochs 10, hidden [64,64]: one PPO "
                             f"iteration of the restated reference ({c1_dt:.1f} s)"},
            "julia": julia_probe()}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = WORKLOADS[args.workload]
    sample_envs = max(64, w["n_envs"] // 8)
    from oracle import envs as OE, policy as OP, ppo as OO  # noqa: F401
    rates = []
    _oracle_iteration_rate(args.workload, sample_envs, 1)             # warm-up
    t_all = time.perf_counter()
    for _ in range(args.steps):
        r, _ = _oracle_iteration_rate(args.workload, sample_envs, 1)
        rates.append(r)
    total = time.perf_counter() - t_all
    value = float(np.mean(rates))
    sample = (f"restated reference (Python/NumPy oracle port), not DRiL.jl (no Julia toolchain): each step = 1 PPO iteration of "
              f"{sample_envs} envs x {w['n_steps']} steps (1/8 of the per-GPU workload), epochs {EPOCHS}, {N_MINIBATCHES} minibatches")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total / max(args.steps, 1) * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": w["name"], "epochs": EPOCHS, "minibatches_per_epoch": N_MINIBATCHES},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": sample, "julia": julia_probe()},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed PPO iterations")
    ap.add_argument("--warmup", type=int, default=3, help="untimed iterations before the timed ones (at least the workload's own)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=list(WORKLOADS) + ["c5"])
    ap.add_argument("--repeats", type=int, default=5,
                    help="the --steps iterations run in this many equal blocks (fewer if it does not divide --steps); "
                         "the median block is reported")
    ap.add_argument("--no-extra", action="store_true", help="C2 only: skip the C4 / C3 blocks under `workloads`")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed iteration of the main workload returned as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.workload is None:
        args.workload = "c2"
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload == "c5"):
        ap.error("--dump-outputs needs --impl ours and a PPO workload (c2, c3, c4)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
