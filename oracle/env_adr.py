"""Oracle (test infrastructure): automatic domain randomisation (include/dril_b200.h, csrc/adr.cuh) restated in NumPy: the
assignment of boundary envs, the ranges each round writes, the attribution of finished episodes to boundary slots and the
update of the boundaries.  It drives the *ParamBatch classes of oracle/env_params.py through their plo / phi arrays, so a
forced-action run over several rounds can be replayed on the CPU.

Slots: 2 i + 0 is the low, 2 i + 1 the high side of the i-th ADR parameter.  In round r env gid is a boundary env when
u01_f32(w0) < p_boundary, w = Philox block (gid, r mod 2^32, 0, TAG_ADR = 8); its slot is w1 mod 2 |J|.
"""
from dataclasses import dataclass

import numpy as np

from . import philox
from .env_params import ENV_PARAMS, POSITIVE

f32 = np.float32
TAG_ADR = 8


@dataclass
class AdrParam:
    index: int
    init_lo: float
    init_hi: float
    limit_lo: float
    limit_hi: float
    delta: float


def check_config(kind, params, p_boundary, buffer_size, t_low, t_high, monitor=True):
    """the validation of dril_env_set_adr; raises ValueError"""
    names = [nm for nm, _ in ENV_PARAMS[kind]]
    if not names:
        raise ValueError(f"{kind} has no parameters")
    if not monitor:
        raise ValueError("ADR needs a Monitor")
    if not 1 <= len(params) <= len(names):
        raise ValueError("need 1 .. P parameters")
    if not (np.isfinite(p_boundary) and 0 <= p_boundary <= 1):
        raise ValueError("p_boundary outside [0, 1]")
    if buffer_size < 1:
        raise ValueError("buffer_size < 1")
    if not (np.isfinite(t_low) and np.isfinite(t_high) and t_low < t_high):
        raise ValueError("need finite t_low < t_high")
    seen = set()
    for q in params:
        if not 0 <= q.index < len(names) or q.index in seen:
            raise ValueError(f"bad or repeated index {q.index}")
        seen.add(q.index)
        v = np.array([q.init_lo, q.init_hi, q.limit_lo, q.limit_hi, q.delta], dtype=f32)
        if not np.isfinite(v).all():
            raise ValueError("values must be finite")
        if not (v[2] <= v[0] <= v[1] <= v[3]):
            raise ValueError("need limit_lo <= init_lo <= init_hi <= limit_hi")
        if not (v[2] > 0 if names[q.index] in POSITIVE else v[2] >= 0):
            raise ValueError("limit_lo violates the parameter's sign rule")
        if not v[4] > 0:
            raise ValueError("delta must be > 0")


def assign(gid, rnd, seed, p_boundary, n_slots):
    """slot of each env gid (n,) in round rnd: -1 for a plain env"""
    x = philox.philox4x32(np.asarray(gid, dtype=np.int64), np.int64(rnd) & 0xFFFFFFFF, 0, TAG_ADR, seed)
    boundary = philox.u01_f32(x[0]) < f32(p_boundary)
    return np.where(boundary, (np.asarray(x[1], dtype=np.int64) % n_slots), -1).astype(np.int64)


def decide(params, lo, hi, sums, counts, m, t_low, t_high):
    """one update from the state (lo, hi float32 (|J|,), sums float64 (2|J|,), counts int64 (2|J|,)) after the rollout's sums
    were added: (lo, hi, sums, counts) after it"""
    lo, hi, sums, counts = lo.copy(), hi.copy(), sums.copy(), counts.copy()
    lo0, hi0 = lo.copy(), hi.copy()
    for s in range(2 * len(params)):
        if counts[s] < m:
            continue
        mean = sums[s] / counts[s]
        i, q = s // 2, params[s // 2]
        d = f32(q.delta)
        if mean >= np.float64(f32(t_high)):
            if s & 1:
                hi[i] = min(f32(q.limit_hi), f32(hi0[i] + d))
            else:
                lo[i] = max(f32(q.limit_lo), f32(lo0[i] - d))
        elif mean <= np.float64(f32(t_low)):
            if s & 1:
                hi[i] = max(f32(q.init_hi), f32(hi0[i] - d))
            else:
                lo[i] = min(f32(q.init_lo), f32(lo0[i] + d))
        sums[s], counts[s] = 0.0, 0
    return lo, hi, sums, counts


class Adr:
    """ADR over the envs with global ids `gid` of one batch (or the union of all shards): attach() turns it on for an oracle
    *ParamBatch, after_rollout() is the device's pass after a collected rollout."""

    def __init__(self, kind, params, p_boundary, buffer_size, t_low, t_high, seed, gid):
        check_config(kind, params, p_boundary, buffer_size, t_low, t_high)
        self.kind, self.params = kind, list(params)
        self.p_boundary, self.m, self.t_low, self.t_high = f32(p_boundary), int(buffer_size), t_low, t_high
        self.seed, self.gid = seed, np.asarray(gid, dtype=np.int64)
        k = len(self.params)
        self.lo = np.array([q.init_lo for q in self.params], dtype=f32)
        self.hi = np.array([q.init_hi for q in self.params], dtype=f32)
        self.sums, self.counts = np.zeros(2 * k), np.zeros(2 * k, dtype=np.int64)
        self.round = 0
        self.ep_mark = self.run_slot = None

    def slots(self, rnd=None):
        return assign(self.gid, self.round if rnd is None else rnd, self.seed, self.p_boundary, 2 * len(self.params))

    def write_ranges(self, plo, phi, slots=None):
        """the ranges of the current round (slots=-1 everywhere: without pins) into plo / phi (P, n), in place"""
        slots = self.slots() if slots is None else slots
        for i, q in enumerate(self.params):
            plo[q.index] = np.where(slots == 2 * i + 1, self.hi[i], self.lo[i])
            phi[q.index] = np.where(slots == 2 * i, self.lo[i], self.hi[i])

    def attach(self, batch):
        """turn ADR on for an oracle *ParamBatch (ranges outside J kept, the defaults without ranges); running episodes
        redrawn; attribution words started"""
        if batch.p is None:
            d = np.array([v for _, v in ENV_PARAMS[self.kind]], dtype=f32)[:, None]
            plo, phi = np.repeat(d, batch.n, axis=1), np.repeat(d, batch.n, axis=1)
        else:
            plo, phi = batch.plo.copy(), batch.phi.copy()
        self.write_ranges(plo, phi)
        batch.set_param_ranges(plo, phi)
        self.ep_mark = batch.episode.astype(np.int64).copy()
        self.run_slot = self.slots()

    def scan(self, done, episode_r, episode):
        """attribution of a rollout's done flags / Monitor returns (T, n) given the reset counters (n,) at its end ->
        per-slot (sums, counts) of the rollout; advances ep_mark / run_slot"""
        S = 2 * len(self.params)
        cur = self.slots()
        sums, counts = np.zeros(S), np.zeros(S, dtype=np.int64)
        episode = np.asarray(episode, dtype=np.int64)
        d = done.sum(axis=0)
        k = np.cumsum(done, axis=0) - 1                       # index of each done among the env's dones
        idx = episode[None, :] - 1 - d[None, :] + k           # the episode each done ends
        slot = np.where(idx >= self.ep_mark[None, :], cur[None, :], self.run_slot[None, :])
        sel = done & (slot >= 0)
        np.add.at(sums, slot[sel], episode_r[sel].astype(np.float64))
        np.add.at(counts, slot[sel], 1)
        self.run_slot = np.where(episode - 1 >= self.ep_mark, cur, self.run_slot)
        self.ep_mark = episode.copy()
        return sums, counts

    def update(self, sums, counts):
        """add the rollout's (global) sums and counts, decide, advance the round"""
        self.lo, self.hi, self.sums, self.counts = decide(self.params, self.lo, self.hi, self.sums + sums, self.counts + counts,
                                                          self.m, self.t_low, self.t_high)
        self.round += 1

    def after_rollout(self, batch, done, episode_r):
        """the device's pass after a collected rollout of `batch`: scan, update, next round's ranges (no redraw)"""
        self.update(*self.scan(done, episode_r, batch.episode))
        self.write_ranges(batch.plo, batch.phi)

    def detach(self, batch):
        """ADR off: every env at [lo_j, hi_j] without pins"""
        self.write_ranges(batch.plo, batch.phi, slots=np.full(batch.n, -1))
