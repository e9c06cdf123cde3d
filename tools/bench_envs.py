"""PPO throughput per classic-control env: one JSON line per env, env count and (with --randomize) parameter setting.

    python tools/bench_envs.py [--envs cartpole,pendulum,mountaincar,mountaincar_continuous,acrobot] [--n-envs 4096,65536]
                               [--steps 20] [--normalize] [--randomize] [--observe-params] [--history K]
                               [--mask-velocities] [--obs-noise SIGMA] [--action-delay D] [--adr] [--repeats 1]

--randomize runs every configuration twice, alternating: with the built-in constants and with per-env parameters drawn at every
reset from +-50 % of each default (set_env_params), --repeats times.  --observe-params adds a third run in the alternation: the
same randomised parameters, observed by the policy (observe_params=True: obs_dim = base + parameter count).  --history K adds
a run with a K-frame observation history (history_len=K: obs_dim = K * base), --mask-velocities one with velocity-free frames
(history_len 1) and, with --history, one with K velocity-free frames; all with the built-in constants.  --obs-noise SIGMA and
--action-delay D add runs with observation noise (SIGMA on every component of every env), with every env's actions delayed
by D steps, and with both.  --adr adds a run with the --randomize ranges and automatic domain randomisation on the kind's first
two parameters (set_adr: initial range the randomised one, p_boundary 0.2, buffer 64, thresholds nothing reaches, so the ranges
stay put and every iteration pays the full ADR pass); its adr_ms is the pass's own time (the "env" profile kind, which nothing
else uses inside an iteration).

Each run: [64, 64] policy, n_steps 128, 4 epochs x 4 minibatches; warm-up iterations, then --steps iterations timed with CUDA events
on the library's stream, L2 overwritten before every iteration (as bench.py does), then the same iterations again with the
per-kernel profile on for the rollout / update split.  Reports env-steps/s, ms per iteration, the loss/grad kernel path, the rollout
kernel the library's dispatch rule picks for the configuration, and the card name and power limit read in the same run."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception as e:                  # the numbers still stand; say that the card could not be read
        return f"unknown ({e})", "unknown"


def rollout_kernel(kind, n, sms, normalize, act_n, randomize, obs_dim):
    """launch_rollout's choice (csrc/api.cu) for a [64, 64] policy: CartPole without normaliser, per-env parameters, history,
    noise or delay (randomize) the tensor-core rollout; otherwise without a training normaliser the fast kernel; with one the cooperative
    general kernel, its actor on tcgen05 (rollout_gtc.cuh) from 64 envs per SM on at widths <= 15"""
    if not normalize:
        return "tc" if kind == "cartpole" and not randomize else "fast"
    return "gtc" if n >= 64 * sms and obs_dim <= 15 else "general"


def run(D, kind, n, steps, warmup, normalize, randomize, observe_params=False, history_len=1, mask_velocities=False,
        obs_noise=0.0, action_delay=0, adr=False):
    from dril_b200 import _lib as L
    from dril_b200.core import ENV_PARAMS
    T = 128
    params = {nm: (0.5 * d, 1.5 * d) for nm, d in ENV_PARAMS[kind]} if randomize else None
    env = D.CudaBatchedEnv(kind, n, seed=0, monitor_window=100, normalize=D.NormalizeConfig() if normalize else None,
                           env_params=params, observe_params=observe_params, history_len=history_len,
                           mask_velocities=mask_velocities, obs_noise=obs_noise or None, action_delay=action_delay)
    if adr:
        env.set_adr({nm: dict(init=params[nm], limits=(0.25 * d, 2.0 * d), step=0.05 * d) for nm, d in ENV_PARAMS[kind][:2]},
                    p_boundary=0.2, buffer_size=64, thresholds=(-1e30, 1e30))
    layer = D.ActorCriticLayer(env.observation_space(), env.action_space(), hidden_dims=[64, 64])
    alg = D.PPO(n_steps=T, batch_size=T * n // 4, epochs=4)
    agent = D.Agent(layer, alg, rng=np.random.default_rng(0))
    ctx = agent.ctx
    lib = ctx.lib
    buf = D.RolloutBuffer(env.observation_space(), env.action_space(), alg.gae_lambda, alg.gamma, T, n)
    hyper = alg.hyper()
    L.check(lib.dril_iteration_prepare(env.h, agent.device.h, buf.h, int(alg.epochs), int(alg.batch_size)))

    def iterate(k):
        for _ in range(k):
            ctx.flush_l2()
            L.check(lib.dril_ppo_iteration_async(env.h, agent.device.h, buf.h, C.byref(hyper), alg.epochs, alg.batch_size,
                                                 agent.shuffle_seed, agent.epoch_counter))
            agent.epoch_counter += alg.epochs
            st = L.IterStats()
            L.check(lib.dril_iteration_result(agent.device.h, C.byref(st)))

    iterate(warmup)
    ctx.synchronize()
    ctx.event_record(0)
    iterate(steps)
    ctx.event_record(1)
    ctx.synchronize()
    ms = ctx.event_elapsed_ms(0, 1) / steps
    ctx.set_profiling(True)
    ctx.reset_profile()
    iterate(steps)
    ctx.synchronize()
    prof = ctx.profile()
    ctx.set_profiling(False)
    upd = sum(prof.get(k, (0.0, 0))[0] for k in ("loss_grad", "grad_reduce", "adam", "permute", "adv_stats")) / steps
    sms = ctx.sm_count()
    act = env.action_space()
    res = dict(env=kind, n_envs=n, n_steps=T, hidden=[64, 64], epochs=4, minibatches=4, normalize=bool(normalize),
               randomize=bool(randomize), observe_params=bool(observe_params), history_len=history_len,
               mask_velocities=bool(mask_velocities), obs_noise=obs_noise, action_delay=action_delay, obs_dim=env.obs_dim,
               env_steps_per_s=n * T / (ms * 1e-3), ms_per_iter=ms,
               rollout_ms=prof.get("rollout", (0.0, 0))[0] / steps, update_ms=upd, adr=bool(adr),
               adr_ms=prof.get("env", (0.0, 0))[0] / steps,
               update_path=agent.device.update_path(),
               rollout_kernel=rollout_kernel(kind, n, sms, normalize, getattr(act, "n", 1),
                                             randomize or history_len > 1 or mask_velocities or obs_noise or action_delay,
                                             env.obs_dim),
               ep_rew_mean=env.monitor_stats()["ep_rew_mean"], timed_iters=steps, warmup_iters=warmup)
    buf.close()
    env.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", default="mountaincar,mountaincar_continuous,acrobot")
    ap.add_argument("--n-envs", default="4096,65536")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--normalize", action="store_true")
    ap.add_argument("--randomize", action="store_true", help="alternate built-in constants and +-50 %% per-env parameters")
    ap.add_argument("--observe-params", action="store_true", help="also randomised parameters observed by the policy")
    ap.add_argument("--history", type=int, default=1, help="also a run with this many frames of observation history")
    ap.add_argument("--mask-velocities", action="store_true", help="also runs with velocity-free frames")
    ap.add_argument("--obs-noise", type=float, default=0.0, help="also runs with this observation-noise deviation")
    ap.add_argument("--action-delay", type=int, default=0, help="also runs with this action delay")
    ap.add_argument("--adr", action="store_true", help="also randomised parameters with automatic domain randomisation")
    ap.add_argument("--repeats", type=int, default=1)
    args = ap.parse_args()
    import __graft_entry__
    __graft_entry__.build()
    import dril_b200 as D
    name, power = card()
    for kind in args.envs.split(","):
        for n in (int(x) for x in args.n_envs.split(",")):
            for _ in range(args.repeats):
                # (randomize, observe_params, history_len, mask_velocities, obs_noise, action_delay, adr)
                variants = [(False, False, 1, False, 0.0, 0, False)] + \
                    ([(True, False, 1, False, 0.0, 0, False)] if args.randomize or args.adr else []) + \
                    ([(True, False, 1, False, 0.0, 0, True)] if args.adr else []) + \
                    ([(True, True, 1, False, 0.0, 0, False)] if args.observe_params else []) + \
                    ([(False, False, args.history, False, 0.0, 0, False)] if args.history > 1 else []) + \
                    ([(False, False, 1, True, 0.0, 0, False)] if args.mask_velocities else []) + \
                    ([(False, False, args.history, True, 0.0, 0, False)] if args.mask_velocities and args.history > 1 else []) + \
                    ([(False, False, 1, False, args.obs_noise, 0, False)] if args.obs_noise else []) + \
                    ([(False, False, 1, False, 0.0, args.action_delay, False)] if args.action_delay else []) + \
                    ([(False, False, 1, False, args.obs_noise, args.action_delay, False)] if args.obs_noise and args.action_delay else [])
                for randomize, observe, k, mask, sigma, delay, adr in variants:
                    r = run(D, kind, n, args.steps, args.warmup, args.normalize, randomize, observe, k, mask, sigma, delay, adr)
                    r.update(card=name, power_limit=power)
                    print(json.dumps(r), flush=True)


if __name__ == "__main__":
    main()
