"""Oracle (test infrastructure): rollout collection, GAE, PPO loss/gradients, Adam, train loop.

Follows:
  collect_trajectories      buffers/trajectory.jl:22-78   (literal, per-trajectory, small cases)
  compute_advantages!       buffers/trajectory.jl:80-102
  collect_rollout!          buffers/rollout_buffer.jl:46-90 (trajectory-completion order)
  loss functor              algorithms/ppo.jl:365-407; normalize! :350-356; clip_range :344-346
  grad clip / KL stop       algorithms/ppo.jl:209-239; utils/optimization_utils.jl:74-107
  Adam                      algorithms/ppo.jl:64-66 (Optimisers.Adam(eta, (0.9,0.999), 1e-5)); third-party
                            rule restated from Optimisers.jl 0.4 — PARITY UNPINNED
  train!                    algorithms/ppo.jl:100-325
  minibatching              algorithms/ppo.jl:188-195 (MLUtils DataLoader: reshuffle per epoch,
                            partial last batch) with the Feistel permutation of philox.py
"""
import time
from dataclasses import dataclass

import numpy as np

from . import philox
from . import policy as P

f32 = np.float32


@dataclass
class PPOConfig:  # algorithms/ppo.jl:25-40
    gamma: float = 0.99
    gae_lambda: float = 0.95
    clip_range: float = 0.2
    clip_range_vf: float | None = None
    ent_coef: float = 0.0
    vf_coef: float = 0.5
    max_grad_norm: float = 0.5
    target_kl: float | None = None
    normalize_advantage: bool = True
    n_steps: int = 2048
    batch_size: int = 64
    epochs: int = 10
    learning_rate: float = 3e-4


# --------------------------------------------------------------------------------------
# GAE
# --------------------------------------------------------------------------------------
def compute_advantages(rewards, values, terminated, bootstrap_value, gamma, gae_lambda):
    """buffers/trajectory.jl:80-102, one trajectory."""
    gamma, lam = f32(gamma), f32(gae_lambda)
    rewards = np.asarray(rewards, dtype=f32)
    values = np.asarray(values, dtype=f32)
    n = len(rewards)
    adv = np.zeros(n, dtype=f32)
    if terminated or bootstrap_value is None:
        delta = rewards[-1] - values[-1]
    else:
        delta = rewards[-1] + gamma * f32(bootstrap_value) - values[-1]
    adv[-1] = delta
    for i in range(n - 2, -1, -1):
        delta = rewards[i] + gamma * values[i + 1] - values[i]
        adv[i] = delta + gamma * lam * adv[i + 1]
    return adv


def gae_timemajor(rewards, values, term, trunc, boot, last_values, gamma, gae_lambda):
    """Per-env reverse scan on time-major [T,N] arrays; equivalent to compute_advantages on
    every trajectory (SURVEY Appendix A.11). boot[t,n] = V(terminal_obs) where truncated;
    last_values[n] = V(new_obs) after the final step."""
    gamma, lam = f32(gamma), f32(gae_lambda)
    T, N = rewards.shape
    adv = np.zeros((T, N), dtype=f32)
    a_next = np.zeros(N, dtype=f32)
    v_next = np.zeros(N, dtype=f32)
    for t in range(T - 1, -1, -1):
        done = term[t] | trunc[t]
        last = done | (t == T - 1)
        # value that follows this step inside the same trajectory, or the bootstrap
        boot_t = np.where(term[t], f32(0), np.where(trunc[t], boot[t], last_values if t == T - 1 else f32(0)))
        use_boot = last & ~term[t]
        nv = np.where(last, np.where(use_boot, boot_t, f32(0)), v_next).astype(f32)
        has_next = ~last | use_boot
        delta = np.where(has_next, rewards[t] + gamma * nv - values[t], rewards[t] - values[t]).astype(f32)
        an = np.where(last, f32(0), a_next)
        adv[t] = np.where(last, delta, delta + gamma * lam * an).astype(f32)
        a_next = adv[t]
        v_next = values[t]
    return adv, (adv + values).astype(f32)


# --------------------------------------------------------------------------------------
# Rollout collection
# --------------------------------------------------------------------------------------
def collect_rollout_timemajor(env, spec, flat, n_steps, policy_seed=0, step0=0, env_gid=None,
                              forced_actions=None):
    """Time-major restatement of trajectory.jl:22-78 (the device layout). Returns a dict of
    [T,N,...] arrays + boot + last_values + last_obs; term_obs [T,N,D] holds the terminal observation of
    every truncated sample (zero elsewhere). `env` exposes observe()/act() (oracle.envs)."""
    N = env.n
    if env_gid is None:
        env_gid = np.arange(N)
    D = spec.obs_dim
    A = 1 if spec.act_kind == "discrete" else spec.act_n
    buf = dict(
        obs=np.zeros((n_steps, N, D), dtype=f32),
        actions=np.zeros((n_steps, N, A), dtype=np.int64 if spec.act_kind == "discrete" else f32),
        rewards=np.zeros((n_steps, N), dtype=f32), values=np.zeros((n_steps, N), dtype=f32),
        logprobs=np.zeros((n_steps, N), dtype=f32),
        term=np.zeros((n_steps, N), dtype=bool), trunc=np.zeros((n_steps, N), dtype=bool),
        boot=np.zeros((n_steps, N), dtype=f32), term_obs=np.zeros((n_steps, N, D), dtype=f32),
        episode_r=np.zeros((n_steps, N), dtype=f32), episode_l=np.zeros((n_steps, N), dtype=np.int64),
    )
    new_obs = env.observe()                                         # trajectory.jl:32
    for t in range(n_steps):
        obs = new_obs
        fa = None if forced_actions is None else forced_actions[t]
        actions, values, logp = P.forward(spec, flat, obs, env_gid, step0 + t, policy_seed,
                                          forced_actions=fa)          # :41
        rewards, term, trunc, info = env.act(P.to_env(spec, actions))  # :42-44
        new_obs = env.observe()                                       # :45
        buf["obs"][t] = obs
        buf["actions"][t] = np.asarray(actions).reshape(N, A)
        buf["rewards"][t] = rewards
        buf["values"][t] = values
        buf["logprobs"][t] = logp
        buf["term"][t] = term
        buf["trunc"][t] = trunc
        if info.get("episode_r") is not None:
            buf["episode_r"][t] = info["episode_r"]
            buf["episode_l"][t] = info["episode_l"]
        if trunc.any() and info.get("terminal_observation") is not None:   # :57-61
            tv = P.predict_values(spec, flat, info["terminal_observation"])
            buf["boot"][t] = np.where(trunc, tv, f32(0))
            buf["term_obs"][t] = np.where(trunc[:, None], info["terminal_observation"], f32(0))
    buf["last_values"] = P.predict_values(spec, flat, new_obs)            # :65-70
    buf["last_obs"] = new_obs
    return buf


def reference_order(term, trunc):
    """Indices (t*N+n) of the time-major buffer listed in the reference's buffer order:
    trajectories appended in (step i, env j) completion order, each laid out contiguously
    (trajectory.jl:72, rollout_buffer.jl:70-74)."""
    T, N = term.shape
    start = np.zeros(N, dtype=np.int64)
    order = []
    for t in range(T):
        for n in range(N):
            if term[t, n] or trunc[t, n] or t == T - 1:
                order.extend(range(start[n] * N + n, t * N + n + 1, N))
                start[n] = t + 1
    return np.array(order, dtype=np.int64)


def collect_rollout_reference(env, spec, flat, n_steps, gamma, gae_lambda, policy_seed=0, step0=0,
                              env_gid=None, forced_actions=None):
    """Literal restatement of collect_trajectories + collect_rollout! (per-trajectory lists,
    trajectory-completion order). Small cases only."""
    N = env.n
    if env_gid is None:
        env_gid = np.arange(N)
    cur = [dict(obs=[], act=[], rew=[], logp=[], val=[]) for _ in range(N)]
    trajs = []
    new_obs = env.observe()
    for i in range(n_steps):
        obs = new_obs
        fa = None if forced_actions is None else forced_actions[i]
        actions, values, logp = P.forward(spec, flat, obs, env_gid, step0 + i, policy_seed, forced_actions=fa)
        rewards, term, trunc, info = env.act(P.to_env(spec, actions))
        new_obs = env.observe()
        for j in range(N):
            c = cur[j]
            c["obs"].append(obs[j]); c["act"].append(np.asarray(actions)[j]); c["rew"].append(rewards[j])
            c["logp"].append(logp[j]); c["val"].append(values[j])
            if term[j] or trunc[j] or i == n_steps - 1:
                c["terminated"] = bool(term[j]); c["truncated"] = bool(trunc[j]); c["boot"] = None
                if trunc[j] and info.get("terminal_observation") is not None:
                    c["boot"] = P.predict_values(spec, flat, info["terminal_observation"][j:j + 1])[0]
                if (not term[j]) and (not trunc[j]) and i == n_steps - 1:
                    c["boot"] = P.predict_values(spec, flat, new_obs[j:j + 1])[0]
                trajs.append(c)
                cur[j] = dict(obs=[], act=[], rew=[], logp=[], val=[])
    out = dict(obs=[], actions=[], rewards=[], logprobs=[], values=[], advantages=[], returns=[])
    for tr in trajs:
        adv = compute_advantages(tr["rew"], tr["val"], tr["terminated"], tr["boot"], gamma, gae_lambda)
        out["obs"] += tr["obs"]; out["actions"] += tr["act"]; out["rewards"] += tr["rew"]
        out["logprobs"] += tr["logp"]; out["values"] += tr["val"]
        out["advantages"] += list(adv)
        out["returns"] += list(adv + np.asarray(tr["val"], dtype=f32))
    return {k: np.asarray(v) for k, v in out.items()}


# --------------------------------------------------------------------------------------
# Loss + analytic gradients
# --------------------------------------------------------------------------------------
def normalize_adv(adv):  # ppo.jl:350-356 (Bessel-corrected std, eps 1e-8)
    adv = np.asarray(adv, dtype=f32)
    m = adv.mean(dtype=f32)
    s = adv.std(ddof=1, dtype=f32) if adv.size > 1 else f32(np.nan)
    return ((adv - m) / (s + f32(1e-8))).astype(f32)


def ppo_loss_and_grads(spec, flat, obs, actions, advantages, returns, old_logprobs, old_values, cfg,
                       want_grads=True):
    """(alg::PPO)(layer, ps, st, batch) ppo.jl:365-407 and its reverse pass.
    Returns loss, stats dict, flat gradient (ComponentVector order)."""
    params = P.unflatten(spec, flat)
    obs = np.asarray(obs, dtype=f32)
    B = obs.shape[0]
    adv = np.asarray(advantages, dtype=f32)
    if cfg.normalize_advantage:
        adv = normalize_adv(adv)
    returns = np.asarray(returns, dtype=f32)
    old_logp = np.asarray(old_logprobs, dtype=f32)
    old_values = np.asarray(old_values, dtype=f32)

    a_out, a_acts = P.mlp_forward(params["actor"], obs, keep=True)
    c_out, c_acts = P.mlp_forward(params["critic"], obs, keep=True)
    values_raw = c_out.reshape(B)
    if spec.act_kind == "discrete":
        probs = P.softmax(a_out)
        idx = np.asarray(actions).astype(np.int64).reshape(B) - spec.act_start
        logp = np.log(probs[np.arange(B), idx]).astype(f32)
        logprobs_all = np.log(probs).astype(f32)
        ent = (-(probs * logprobs_all).sum(axis=1, dtype=f32)).astype(f32)
    else:
        a = np.asarray(actions, dtype=f32).reshape(B, spec.act_n)
        log_std = params["log_std"]
        logp = P.gaussian_logpdf(a_out, log_std, a)
        ent = P.gaussian_entropy(log_std, B)
    if cfg.clip_range_vf is not None:
        c = f32(cfg.clip_range_vf)
        values = (old_values + np.clip(values_raw - old_values, -c, c)).astype(f32)
    else:
        values = values_raw
    eps = f32(cfg.clip_range)
    log_ratio = (logp - old_logp).astype(f32)
    r = np.exp(log_ratio).astype(f32)
    r_c = np.clip(r, f32(1) - eps, f32(1) + eps).astype(f32)
    s1, s2 = r * adv, r_c * adv
    p_loss = -np.minimum(s1, s2).mean(dtype=f32)
    ent_loss = -ent.mean(dtype=f32)
    v_loss = ((values - returns) ** 2).mean(dtype=f32)
    loss = f32(p_loss + f32(cfg.ent_coef) * ent_loss + f32(cfg.vf_coef) * v_loss)
    stats = dict(policy_loss=float(p_loss), value_loss=float(v_loss), entropy_loss=float(ent_loss),
                 clip_fraction=float((r != r_c).mean()),
                 approx_kl_div=float((np.exp(log_ratio) - 1 - log_ratio).mean(dtype=f32)),
                 entropy=float(ent.mean(dtype=f32)), ratio=float(r.mean(dtype=f32)))
    if not want_grads:
        return float(loss), stats, None

    invB = f32(1.0 / B)
    # min(s1,s2) = ifelse(s2 < s1, s2, s1): ties route the gradient to s1 = r*A
    g_logp = np.where(s2 < s1, f32(0), -invB * adv * r).astype(f32)
    g_ent = np.full(B, -f32(cfg.ent_coef) * invB, dtype=f32)
    g_val = (f32(cfg.vf_coef) * f32(2) * (values - returns) * invB).astype(f32)
    if cfg.clip_range_vf is not None:
        d = values_raw - old_values
        g_val = np.where((d >= -c) & (d <= c), g_val, f32(0)).astype(f32)

    grads = {"actor": None, "critic": None}
    if spec.act_kind == "discrete":
        onehot = np.zeros_like(probs)
        onehot[np.arange(B), idx] = 1
        dz = g_logp[:, None] * (onehot - probs) + g_ent[:, None] * (-probs * (logprobs_all + ent[:, None]))
    else:
        var_inv = np.exp(f32(-2) * log_std).astype(f32)
        diff = a - a_out
        dz = g_logp[:, None] * diff * var_inv
        g_ls = (g_logp[:, None] * (f32(-1) + diff * diff * var_inv)).sum(axis=0, dtype=f32) + g_ent.sum(dtype=f32)
        grads["log_std"] = g_ls.astype(f32)
    grads["actor"] = _mlp_backward(params["actor"], a_acts, dz.astype(f32))
    grads["critic"] = _mlp_backward(params["critic"], c_acts, g_val.reshape(B, 1))
    return float(loss), stats, P.flatten(spec, grads)


def _mlp_backward(layers, acts, dout):
    grads = [None] * len(layers)
    dz = dout
    for li in range(len(layers) - 1, -1, -1):
        W, _ = layers[li]
        h_in = acts[li]
        grads[li] = ((h_in.T @ dz).astype(f32), dz.sum(axis=0, dtype=f32))
        if li > 0:
            dh = (dz @ W.T).astype(f32)
            dz = (dh * (f32(1) - h_in * h_in)).astype(f32)
    return grads


# --------------------------------------------------------------------------------------
# Optimiser
# --------------------------------------------------------------------------------------
class Adam:
    """Optimisers.jl 0.4 Adam rule as configured at ppo.jl:64-66 (eta=lr, beta=(0.9,0.999),
    epsilon=1e-5), bias-corrected; state m, v and step t. PARITY UNPINNED (third-party)."""

    def __init__(self, n, lr=3e-4, beta1=0.9, beta2=0.999, eps=1e-5):
        self.m = np.zeros(n, dtype=f32)
        self.v = np.zeros(n, dtype=f32)
        self.t = 0
        self.lr, self.b1, self.b2, self.eps = lr, beta1, beta2, eps

    def step(self, flat, g):
        self.t += 1
        b1, b2 = f32(self.b1), f32(self.b2)
        self.m = (b1 * self.m + (f32(1) - b1) * g).astype(f32)
        self.v = (b2 * self.v + (f32(1) - b2) * g * g).astype(f32)
        c1 = f32(1.0 - float(self.b1) ** self.t)
        c2 = f32(1.0 - float(self.b2) ** self.t)
        upd = (self.m / c1) / (np.sqrt(self.v / c2) + f32(self.eps)) * f32(self.lr)
        return (flat - upd).astype(f32)


def clip_grads(g, max_grad_norm):
    """ppo.jl:216-232 + optimization_utils.jl:74-107: scale by max/norm (no eps) if norm > max.
    Returns (clipped grads, pre-clip norm)."""
    norm = f32(np.sqrt((g.astype(f32) ** 2).sum(dtype=f32)))
    if max_grad_norm is not None and norm > f32(max_grad_norm):
        g = (g * (f32(max_grad_norm) / norm)).astype(f32)
    return g, float(norm)


# --------------------------------------------------------------------------------------
# train!
# --------------------------------------------------------------------------------------
def minibatch_indices(n_total, batch_size, epoch_counter, rank, seed):
    keys = philox.feistel_keys(epoch_counter, rank, seed)
    perm = philox.feistel_permute(np.arange(n_total), n_total, keys)
    return [perm[s:s + batch_size] for s in range(0, n_total, batch_size)]


def ppo_update(spec, flat, opt, buf, cfg, shuffle_seed=0, epoch_counter0=0, rank=0):
    """One iteration's epoch/minibatch loop (ppo.jl:205-254) on a time-major buffer dict with
    advantages/returns filled. Returns new flat params, per-iteration stats, epochs consumed."""
    T, N = buf["rewards"].shape
    n_total = T * N
    obs = buf["obs"].reshape(n_total, -1)
    actions = buf["actions"].reshape(n_total, -1)
    adv = buf["advantages"].reshape(n_total)
    ret = buf["returns"].reshape(n_total)
    logp = buf["logprobs"].reshape(n_total)
    val = buf["values"].reshape(n_total)
    rec = {k: [] for k in ("entropy_loss", "policy_loss", "value_loss", "approx_kl_div",
                           "clip_fraction", "loss", "grad_norm")}
    cont = True
    epochs_run = 0
    for epoch in range(cfg.epochs):
        epochs_run += 1
        for idx in minibatch_indices(n_total, cfg.batch_size, epoch_counter0 + epoch, rank, shuffle_seed):
            loss, stats, g = ppo_loss_and_grads(spec, flat, obs[idx], actions[idx], adv[idx], ret[idx],
                                                logp[idx], val[idx], cfg)
            g, norm = clip_grads(g, cfg.max_grad_norm)
            rec["grad_norm"].append(norm)
            if cfg.target_kl is not None and stats["approx_kl_div"] > 1.5 * cfg.target_kl:
                cont = False
                break
            flat = opt.step(flat, g)
            for k in ("entropy_loss", "policy_loss", "value_loss", "approx_kl_div", "clip_fraction"):
                rec[k].append(stats[k])
            rec["loss"].append(loss)
        if not cont:
            break
    means = {k: (float(np.mean(np.asarray(v, dtype=f32))) if len(v) else float("nan")) for k, v in rec.items()}
    return flat, means, epochs_run


def explained_variance(values, returns):  # ppo.jl:256 (Bessel-corrected var)
    v = np.asarray(values, dtype=f32).reshape(-1)
    r = np.asarray(returns, dtype=f32).reshape(-1)
    return float(1 - np.var(v - r, ddof=1, dtype=f32) / np.var(r, ddof=1, dtype=f32))


def train(env, spec, flat, cfg, max_steps, policy_seed=0, shuffle_seed=0, opt=None, env_gid=None):
    """train! ppo.jl:100-325 (no callbacks/logging). Returns (flat, learn_stats dict)."""
    N = env.n
    iterations = max_steps // (cfg.n_steps * N)
    if opt is None:
        opt = Adam(flat.size, lr=cfg.learning_rate)
    keys = ("entropy_losses", "policy_losses", "value_losses", "approx_kl_divs", "clip_fractions",
            "losses", "explained_variances", "fps", "grad_norms", "learning_rates")
    ls = {k: [] for k in keys}
    step0 = 0
    epoch_counter = 0
    for _ in range(iterations):
        opt.lr = cfg.learning_rate
        t0 = time.time()
        buf = collect_rollout_timemajor(env, spec, flat, cfg.n_steps, policy_seed, step0, env_gid)
        adv, ret = gae_timemajor(buf["rewards"], buf["values"], buf["term"], buf["trunc"], buf["boot"],
                                 buf["last_values"], cfg.gamma, cfg.gae_lambda)
        buf["advantages"], buf["returns"] = adv, ret
        fps = cfg.n_steps * N / max(time.time() - t0, 1e-9)
        step0 += cfg.n_steps
        flat, means, epochs_run = ppo_update(spec, flat, opt, buf, cfg, shuffle_seed, epoch_counter)
        epoch_counter += cfg.epochs
        ls["explained_variances"].append(explained_variance(buf["values"], buf["returns"]))
        ls["entropy_losses"].append(means["entropy_loss"]); ls["policy_losses"].append(means["policy_loss"])
        ls["value_losses"].append(means["value_loss"]); ls["approx_kl_divs"].append(means["approx_kl_div"])
        ls["clip_fractions"].append(means["clip_fraction"]); ls["losses"].append(means["loss"])
        ls["grad_norms"].append(means["grad_norm"]); ls["fps"].append(fps)
        ls["learning_rates"].append(cfg.learning_rate)
    return flat, ls
