"""CPU restatement of n-step returns as the CUDA sample kernel computes them (include/dmdqn_b200.h, dmdqn_sample with
hp->n_step > 1): the lookahead length m, the return R, the discount and the bootstrap row, plus a stacked learn step whose
TD targets take a discount per row.

Like oracle/, this is test infrastructure.  It builds on oracle/replay.py and tests/per_oracle.py without changing them.
Every float64 operation below is one IEEE operation in the kernel's order (multiply and add kept apart), so the sampled
returns and discounts can be compared bit for bit.
"""
from __future__ import annotations

import numpy as np
import torch

from oracle.replay import RingReplay
from per_oracle import WeightedStackedOracle


def batch_stats(rewards: np.ndarray) -> tuple[float, float]:
    """(mean, std + 1e-8) of the first-step rewards ``[B]`` with the kernel's canonical tree (oracle/replay.py
    zscore_canonical): lane l adds elements l, l+32, ... in order, then an xor butterfly (16, 8, 4, 2, 1)."""
    r = np.asarray(rewards, np.float64)
    b = r.shape[0]

    def tree_sum(x):
        acc = [0.0] * 32
        for i in range(b):
            acc[i % 32] = acc[i % 32] + float(x[i])
        for off in (16, 8, 4, 2, 1):
            acc = [acc[l] + acc[l ^ off] for l in range(32)]
        return acc[0]

    mean = tree_sum(r) / b
    var = tree_sum([(float(v) - mean) * (float(v) - mean) for v in r]) / b
    return mean, float(np.sqrt(var)) + 1e-8


def lookahead(done: np.ndarray, n_written: int, capacity: int, slot: int, n: int) -> tuple[int, int, bool]:
    """(m, bootstrap slot, terminal) for the row in physical ``slot`` of one agent's ring (``done[C]``)."""
    size = min(n_written, capacity)
    j = (slot - (n_written - size)) % capacity                    # logical index of the drawn row
    lim = min(max(n, 1), size - j)
    m = lim
    for k in range(lim):
        if done[(slot + k) % capacity]:
            m = k + 1
            break
    last = (slot + m - 1) % capacity
    return m, last, bool(done[last])          # the scan stops on the first done, so the last row is done iff one was met


def nstep_batch(ring: RingReplay, agents: np.ndarray, slots: np.ndarray, n: int, gamma: float,
                normalize_rewards: bool = True):
    """The sample kernel's outputs for one network's batch of rows ``(agents[i], slots[i])``: a dict of
    ``r_hat`` (R, float32), ``discount`` (float32), ``done`` (terminal flag of the return, float32), ``next_slot`` (the
    bootstrap row's physical slot) and ``m``.  ``n`` of 0 or 1 gives the one-step target."""
    agents, slots = np.asarray(agents, np.int64), np.asarray(slots, np.int64)
    b = slots.shape[0]
    c = ring.c
    r0 = ring.rew[agents, slots]
    mean, denom = batch_stats(r0) if normalize_rewards else (0.0, 1.0)
    z = (lambda r: (float(r) - mean) / denom) if normalize_rewards else float
    out = {k: np.zeros(b, np.float32) for k in ("r_hat", "discount", "done")}
    out["next_slot"] = np.zeros(b, np.int64)
    out["m"] = np.zeros(b, np.int64)
    for i in range(b):
        a, s = int(agents[i]), int(slots[i])
        if n <= 1:
            d = np.float32(1.0 if ring.done[a, s] else 0.0)
            m, last, disc = 1, s, np.float32(gamma) * (np.float32(1.0) - d)
        else:
            m, last, term = lookahead(ring.done[a], int(ring.n_written[a]), c, s, n)
            gm = gamma
            for _ in range(1, m):
                gm = gm * gamma
            d = np.float32(1.0 if term else 0.0)
            disc = np.float32(0.0) if term else np.float32(gm)
        ret, g = z(r0[i]), 1.0
        for k in range(1, m):
            g = g * gamma
            ret = ret + g * z(ring.rew[a, (s + k) % c])
        out["r_hat"][i] = np.float32(ret)
        out["discount"][i] = disc
        out["done"][i] = d
        out["next_slot"][i] = last
        out["m"][i] = m
    return out


class NStepStackedOracle(WeightedStackedOracle):
    """WeightedStackedOracle whose TD targets take a discount per row: y = R + discount * Q_tgt(s') (with every discount
    equal to gamma * (1 - done) this is the one-step target of StackedOracle, bit for bit)."""

    _discounts = None

    def td_targets(self, rewards, next_states, dones):
        if self._discounts is None:
            return super().td_targets(rewards, next_states, dones)
        r = torch.as_tensor(rewards, dtype=torch.float32)
        s2 = torch.as_tensor(next_states, dtype=torch.float32)
        disc = torch.as_tensor(np.asarray(self._discounts, np.float32))
        with torch.no_grad():
            tq_all = self.forward(self.target, s2)
            q_next = self.forward(self.online, s2)
            if self.double_dqn:
                tq = torch.gather(tq_all, 2, torch.argmax(q_next, dim=2, keepdim=True))[..., 0]
            else:
                tq = tq_all.max(dim=2).values
            y = r + disc * tq
        return y, q_next, tq_all

    def learn_on_batch(self, states, actions, rewards, next_states, dones, active=None, is_weights=None, discounts=None):
        """As WeightedStackedOracle.learn_on_batch; ``discounts[N, B]`` (None = gamma * (1 - dones)) replaces the one-step
        discount, and ``rewards`` are the n-step returns."""
        self._discounts = discounts
        try:
            return super().learn_on_batch(states, actions, rewards, next_states, dones, active, is_weights)
        finally:
            self._discounts = None
