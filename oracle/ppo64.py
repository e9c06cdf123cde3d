"""Oracle (test infrastructure): the PPO loss of algorithms/ppo.jl:365-407 restated in torch float64 with autograd.

It is the high-precision reference the loss/grad kernels are compared with block by block: ``loss64`` evaluates the loss,
the seven statistics ``DevicePolicy.loss_grad`` returns and the flat gradient in float64 from the float32 inputs;
``grad_blocks`` splits a flat gradient into its parameter blocks (ComponentVector order of policy.py) and
``assert_blocks_close`` compares every block with its own relative bound.
"""
import numpy as np

STAT_NAMES = ("policy_loss", "value_loss", "entropy_loss", "clip_fraction", "approx_kl_div", "entropy", "ratio")


def _nets(spec, t):
    p = 0
    nets = []
    for net in (0, 1):
        layers = []
        for (i, o) in spec.layer_dims(net):
            W = t[p:p + i * o].reshape(i, o); p += i * o
            b = t[p:p + o]; p += o
            layers.append((W, b))
        nets.append(layers)
    return nets, p


def _mlp(layers, x):
    import torch
    for li, (W, b) in enumerate(layers):
        x = x @ W + b
        if li < len(layers) - 1:
            x = torch.tanh(x)
    return x


def forward64(spec, flat, obs):
    """float64 actor outputs (logits or means) [B][act_n] and values [B] of the float32 parameters."""
    import torch
    with torch.no_grad():
        t = torch.tensor(np.asarray(flat, dtype=np.float32).astype(np.float64))
        nets, _ = _nets(spec, t)
        x = torch.tensor(np.asarray(obs, dtype=np.float32).astype(np.float64))
        return _mlp(nets[0], x).numpy(), _mlp(nets[1], x).reshape(-1).numpy()


def logp64(spec, flat, out, actions):
    """float64 log-probabilities of `actions` under actor outputs `out` (forward64)."""
    out = np.asarray(out, dtype=np.float64)
    if spec.act_kind == "discrete":
        z = out - out.max(axis=1, keepdims=True)
        lsm = z - np.log(np.exp(z).sum(axis=1, keepdims=True))
        idx = np.asarray(actions).reshape(-1).astype(np.int64) - spec.act_start
        return lsm[np.arange(len(idx)), idx]
    ls = np.asarray(flat, dtype=np.float32)[spec.n_params() - spec.act_n:].astype(np.float64)
    a = np.asarray(actions, dtype=np.float32).reshape(len(out), spec.act_n).astype(np.float64)
    k = spec.act_n
    return -0.5 * (2 * ls.sum() + ((a - out) ** 2 * np.exp(-2 * ls)).sum(1) + k * np.log(2 * np.pi))


def loss64(spec, flat, obs, actions, adv, ret, old_lp, old_v, cfg):
    """Loss, flat gradient and statistics (STAT_NAMES) of ppo.jl:365-407 in float64 autograd; cfg: oracle.ppo.PPOConfig."""
    import torch
    t = torch.tensor(np.asarray(flat, dtype=np.float32).astype(np.float64), requires_grad=True)
    nets, p = _nets(spec, t)
    x = torch.tensor(np.asarray(obs, dtype=np.float32).astype(np.float64))
    out = _mlp(nets[0], x)
    values = _mlp(nets[1], x).reshape(-1)
    A = torch.tensor(np.asarray(adv, dtype=np.float32).astype(np.float64))
    if cfg.normalize_advantage:
        A = (A - A.mean()) / (A.std(unbiased=True) + 1e-8)
    if spec.act_kind == "discrete":
        probs = torch.softmax(out, dim=1)
        idx = torch.tensor(np.asarray(actions).reshape(-1).astype(np.int64) - spec.act_start)
        logp = torch.log(probs[torch.arange(len(idx)), idx])
        ent = -(probs * torch.log(probs)).sum(1)
    else:
        ls = t[p:p + spec.act_n]
        a = torch.tensor(np.asarray(actions, dtype=np.float32).astype(np.float64).reshape(len(x), spec.act_n))
        k = spec.act_n
        logp = -0.5 * (2 * ls.sum() + ((a - out) ** 2 * torch.exp(-2 * ls)).sum(1) + k * np.log(2 * np.pi))
        ent = (0.5 * k * (1 + np.log(2 * np.pi)) + ls.sum()) * torch.ones(len(a), dtype=torch.float64)
    ov = torch.tensor(np.asarray(old_v, dtype=np.float32).astype(np.float64))
    if cfg.clip_range_vf is not None:
        values = ov + torch.clamp(values - ov, -cfg.clip_range_vf, cfg.clip_range_vf)
    lr = logp - torch.tensor(np.asarray(old_lp, dtype=np.float32).astype(np.float64))
    r = torch.exp(lr)
    rc = torch.clamp(r, 1 - cfg.clip_range, 1 + cfg.clip_range)
    p_loss = -torch.minimum(r * A, rc * A).mean()
    ent_loss = -ent.mean()
    v_loss = ((values - torch.tensor(np.asarray(ret, dtype=np.float32).astype(np.float64))) ** 2).mean()
    loss = p_loss + cfg.ent_coef * ent_loss + cfg.vf_coef * v_loss
    loss.backward()
    p_loss, v_loss, ent_loss, r, lr, ent = (x.detach() for x in (p_loss, v_loss, ent_loss, r, lr, ent))
    st = dict(policy_loss=float(p_loss), value_loss=float(v_loss), entropy_loss=float(ent_loss),
              clip_fraction=float((r != rc).double().mean()), approx_kl_div=float((torch.exp(lr) - 1 - lr).mean()),
              entropy=float(ent.mean()), ratio=float(r.mean()))
    return float(loss.detach()), t.grad.numpy(), st


def grad_blocks(spec):
    """[(name, net, slice)] of the flat parameter vector: actor W / b per layer, critic W / b per layer, then log_std."""
    blocks = []
    p = 0
    for net, nn in ((0, "actor"), (1, "critic")):
        for li, (i, o) in enumerate(spec.layer_dims(net)):
            blocks.append((f"{nn}.W{li}", net, slice(p, p + i * o))); p += i * o
            blocks.append((f"{nn}.b{li}", net, slice(p, p + o))); p += o
    if spec.act_kind == "continuous":
        blocks.append(("log_std", 0, slice(p, p + spec.act_n))); p += spec.act_n
    assert p == spec.n_params()
    return blocks


def block_errors(spec, g, g64, floor=1e-6):
    """{block: relative error} of gradient g against the float64 gradient g64.  A block's error is ||g - g64|| over
    max(||g64||, floor * ||g64 of its net||): a block whose reference is (nearly) zero is compared absolutely against
    that floor.  A net whose whole reference gradient is zero, like the actor of Discrete(1), takes the floor from the
    full gradient instead.  log_std counts to the actor."""
    g = np.asarray(g, dtype=np.float64)
    g64 = np.asarray(g64, dtype=np.float64)
    blocks = grad_blocks(spec)
    net_norm = [np.sqrt(sum(np.sum(g64[s] ** 2) for _, n, s in blocks if n == net)) for net in (0, 1)]
    net_norm = [x if x > 0 else np.linalg.norm(g64) for x in net_norm]
    errs = {}
    for name, net, s in blocks:
        den = max(np.linalg.norm(g64[s]), floor * net_norm[net], 1e-300)
        errs[name] = float(np.linalg.norm(g[s] - g64[s]) / den)
    return errs


def assert_blocks_close(spec, g, g64, rtol=1e-4, floor=1e-6, what=""):
    """Every entry of g finite and every parameter block within rtol of the float64 gradient (block_errors)."""
    g = np.asarray(g)
    bad = np.flatnonzero(~np.isfinite(g))
    assert bad.size == 0, f"{what}: {bad.size} non-finite gradient entries, first at {bad[:5].tolist()}"
    errs = block_errors(spec, g, g64, floor)
    worst = max(errs, key=errs.get)
    assert errs[worst] <= rtol, f"{what}: block {worst} relative error {errs[worst]:.3e} > {rtol:.0e} ({errs})"
    return errs


# --------------------------------------------------------------------------------------
# minibatches with chosen per-sample gradient magnitudes
# --------------------------------------------------------------------------------------
RATIO_MARGIN = 0.25        # of clip_range: no sample's ratio within 0.25 * clip_range of 1 +- clip_range
VF_MARGIN = 0.25           # of clip_range_vf: no sample's v - old_v within 0.25 * clip_range_vf of +-clip_range_vf
TIE_GAP = 1e-3             # no two logits of a sample closer than this


def tile_magnitudes(pattern, B, lead, rng):
    """Per-sample gradient magnitudes of a named pattern over B samples in order, and the mask of samples whose gradient
    must be exactly zero.  `lead` (even) samples lead: the first tile of every CTA / warp group of a loss/grad kernel.
      ("step", R)   the lead at 1, the rest at R
      "tiny"        the lead at 1e-30, the rest at 1
      "outliers"    1, with 1 % of the sample pairs, placed at random, at 2^20
      "zero"        the lead clipped (zero gradient), the rest at 1
    Magnitudes are set per sample pair (2k, 2k + 1) so that advantages can cancel in pairs (scaled_minibatch)."""
    mag = np.ones(B)
    zero = np.zeros(B, bool)
    lead = min(lead, B)
    if isinstance(pattern, tuple) and pattern[0] == "step":
        mag[lead:] = pattern[1]
    elif pattern == "tiny":
        mag[:lead] = 1e-30
    elif pattern == "outliers":
        pairs = rng.choice(B // 2, size=max(1, B // 200), replace=False)
        mag[2 * pairs] = mag[2 * pairs + 1] = 2.0 ** 20
    elif pattern == "zero":
        zero[:lead] = True
    else:
        raise ValueError(pattern)
    return mag, zero


def scaled_minibatch(spec, flat, actor_mag, critic_mag, rng, clip_range=0.2, clip_range_vf=None, actor_zero=None,
                     critic_zero=None):
    """float32 minibatch (obs, actions, adv, ret, old_lp, old_v) whose per-sample gradient magnitudes follow actor_mag
    (through the advantages) and critic_mag (ret = v + critic_mag * z, v the float64 value), with every sample clear of
    the branches the kernels decide in float32 and the reference in float64:
      * ratio = exp(logp - old_lp) inside 1 +- 0.75 clip_range or outside 1 +- 1.25 clip_range;
      * v - old_v inside +-0.75 clip_range_vf or outside +-1.25 clip_range_vf;
      * no two logits of a sample within TIE_GAP.
    Samples of actor_zero are clipped on the side that zeroes their gradient (ratio beyond 1 + clip_range with a positive
    advantage, below 1 - clip_range with a negative one); samples of critic_zero have |v - old_v| > clip_range_vf.
    Advantages come in pairs (a, -a) of sample 2k and 2k + 1, so the minibatch mean is about zero and advantage
    normalisation keeps the ratios between tiles.  ret - v has one sign: the critic's bias gradient is then a
    well-conditioned sum (terms that cancel would measure float32 summation, not the kernels).  Magnitude 1 means |adv| and
    ret - v in [1/8, 2]."""
    B = len(actor_mag)
    actor_zero = np.zeros(B, bool) if actor_zero is None else np.asarray(actor_zero, bool)
    critic_zero = np.zeros(B, bool) if critic_zero is None else np.asarray(critic_zero, bool)
    assert not critic_zero.any() or clip_range_vf is not None
    obs = rng.normal(size=(B, spec.obs_dim)).astype(np.float32)
    if spec.act_kind == "discrete":
        actions = rng.integers(spec.act_start, spec.act_start + spec.act_n, (B, 1))
    else:
        actions = rng.normal(size=(B, spec.act_n)).astype(np.float32)
    out, v = forward64(spec, flat, obs)
    if spec.act_kind == "discrete" and spec.act_n > 1:
        for _ in range(50):
            s = np.sort(out, axis=1)
            tie = np.flatnonzero(np.diff(s, axis=1).min(axis=1) < TIE_GAP)
            if tie.size == 0:
                break
            obs[tie] = rng.normal(size=(tie.size, spec.obs_dim)).astype(np.float32)
            out, v = forward64(spec, flat, obs)
        else:
            raise RuntimeError("could not separate the logits")
    logp = logp64(spec, flat, out, actions)
    # advantages: +-k/8 * magnitude, k in 1..16, in cancelling pairs (an odd last sample gets 0: no gradient)
    amag = np.asarray(actor_mag, np.float64)
    npair = B // 2
    assert np.array_equal(amag[0:2 * npair:2], amag[1:2 * npair:2]), "magnitudes must be set per sample pair"
    a = amag[0:2 * npair:2] * rng.integers(1, 17, npair) / 8.0 * rng.choice([-1.0, 1.0], npair)
    adv = np.zeros(B)
    adv[0:2 * npair:2], adv[1:2 * npair:2] = a, -a
    adv = adv.astype(np.float32)
    # ratios
    c = clip_range
    inside = rng.random(B) < 0.7
    ratio = np.where(inside, 1 + rng.uniform(-0.75, 0.75, B) * c,
                     1 + rng.choice([-1.0, 1.0], B) * rng.uniform(1.25, 2.0, B) * c)
    sgn = np.sign(adv)
    zsel = actor_zero & (sgn != 0)
    ratio[zsel] = 1 + sgn[zsel] * rng.uniform(1.25, 2.0, zsel.sum()) * c
    old_lp = (logp - np.log(ratio)).astype(np.float32)
    # critic
    cm = np.asarray(critic_mag, np.float64)
    ret = (v + cm * rng.integers(1, 17, B) / 8.0).astype(np.float32)
    if clip_range_vf is None:
        dv = rng.normal(size=B) * 0.3
    else:
        dv = rng.choice([-1.0, 1.0], B) * np.where(critic_zero, rng.uniform(1.25, 2.0, B), rng.uniform(0.0, 0.75, B)) * clip_range_vf
    old_v = (v - dv).astype(np.float32)
    return obs, actions, adv, ret, old_lp, old_v
