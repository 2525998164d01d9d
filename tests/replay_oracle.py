"""CPU restatement of what the CUDA sample kernel and the learn step compute beyond oracle/ (include/dmdqn_b200.h):

* proportional prioritized experience replay (Schaul et al. 2016, DMDQN_SAMPLE_PRIORITIZED): the canonical priority sum,
  the stratified draw, the importance weights, the beta schedule, the priority rule and a ring with priorities;
* n-step returns (dmdqn_sample, hp->n_step): the lookahead length m, the return R, the discount and the bootstrap row;
* a stacked learn step that weights every row's loss term by an importance weight and takes a discount per row.

Like oracle/, this is test infrastructure, built on oracle/replay.py and oracle/dqn.py.  Every float64 operation below is
one IEEE operation in the kernel's order (multiply and add kept apart), so the drawn slots, returns and discounts can be
compared bit for bit.
"""
from __future__ import annotations

import numpy as np
import torch

from oracle.dqn import StackedOracle, adam_scalars, adam_update_, loss_and_grad
from oracle.replay import RingReplay, zscore_stats

CHUNK = 128


def chunk_totals(priority: np.ndarray) -> np.ndarray:
    """Float64 total of every chunk of 128 consecutive slots: lane l (0..31) adds slots l, l+32, l+64, l+96 in order,
    then the lanes are combined by an xor butterfly (16, 8, 4, 2, 1).  Slots past the ring count as 0."""
    p = np.asarray(priority, np.float32).astype(np.float64)
    nch = -(-p.shape[0] // CHUNK)
    x = np.concatenate([p, np.zeros(nch * CHUNK - p.shape[0])]).reshape(nch, 4, 32)    # [chunk][k][lane]
    acc = np.zeros((nch, 32))
    for k in range(4):
        acc = acc + x[:, k, :]
    lanes = np.arange(32)
    for off in (16, 8, 4, 2, 1):
        acc = acc + acc[:, lanes ^ off]
    return acc[:, 0]


def chunk_prefixes(priority: np.ndarray) -> np.ndarray:
    """[nch + 1] exclusive prefixes of the chunk totals, summed in chunk order; the last entry is the total S."""
    tot = chunk_totals(priority)
    out = np.zeros(tot.shape[0] + 1)
    run = 0.0
    for c in range(tot.shape[0]):
        run = run + float(tot[c])
        out[c + 1] = run
    return out


def stratified_u(total: float, words: np.ndarray) -> np.ndarray:
    """u_k = ((k + w_k * 2^-32) * S) / B, float64, left to right."""
    w = np.asarray(words, np.uint32)
    b = w.shape[0]
    return np.array([((k + float(w[k]) * 2.0 ** -32) * total) / b for k in range(b)])


def draw_from_u(priority: np.ndarray, u: np.ndarray) -> np.ndarray:
    """The slot of every u: the last chunk whose exclusive prefix is <= u, then the first slot of that chunk whose running
    sum (starting at the prefix) exceeds u.  A walk that rounding carries past the chunk ends on the last slot of the ring
    with a non-zero priority (slot 0 if there is none)."""
    p = np.asarray(priority, np.float32)
    prefix = chunk_prefixes(p)
    nch = prefix.shape[0] - 1
    nz = np.nonzero(p > 0)[0]
    last = int(nz[-1]) if nz.size else 0
    out = np.empty(len(u), np.int32)
    for i, ui in enumerate(u):
        c = int(np.searchsorted(prefix[:nch], ui, side="right")) - 1
        run, slot = float(prefix[c]), -1
        for s in range(c * CHUNK, min((c + 1) * CHUNK, p.shape[0])):
            run = run + float(p[s])
            if run > ui:
                slot = s
                break
        out[i] = slot if slot >= 0 else last
    return out


def prioritized_indices(priority: np.ndarray, words: np.ndarray) -> np.ndarray:
    """Physical slots drawn from one ring's priorities ``[C]`` with the uint32 words ``[B]``."""
    return draw_from_u(priority, stratified_u(float(chunk_prefixes(priority)[-1]), words))


def beta_schedule(t: int, beta0: float, beta_steps: int) -> float:
    """beta_t = min(1, beta0 + (1 - beta0) * t / beta_steps); beta0 when beta_steps <= 0."""
    if beta_steps <= 0:
        return beta0
    return min(1.0, beta0 + (1.0 - beta0) * t / beta_steps)


def is_weights(priority: np.ndarray, slots: np.ndarray, beta: float) -> np.ndarray:
    """(p_min / p_i)^beta in float64 rounded to float32, p_min = the smallest drawn priority (1 where p_i is 0)."""
    p = np.asarray(priority, np.float32)[np.asarray(slots)].astype(np.float64)
    pmin = p.min()
    with np.errstate(divide="ignore", invalid="ignore"):
        w = np.where(p > 0, np.power(pmin / np.where(p > 0, p, 1.0), beta), 1.0)
    return w.astype(np.float32)


def priority_of(delta: np.ndarray, alpha: float, eps: float) -> np.ndarray:
    """(float)pow(|delta| + eps, alpha) in float64."""
    return np.power(np.abs(np.asarray(delta, np.float32).astype(np.float64)) + eps, alpha).astype(np.float32)


class PrioritizedRing(RingReplay):
    """RingReplay with ``priority[N, C]`` (p^alpha per physical slot, 0 = never written) and ``priority_max[N]``: a push
    gives the written slot the agent's ``priority_max``; masked-out agents are untouched."""

    def __init__(self, n_agents: int, capacity: int, obs_dim: int):
        super().__init__(n_agents, capacity, obs_dim)
        self.priority = np.zeros((n_agents, capacity), np.float32)
        self.priority_max = np.ones((n_agents,), np.float32)

    def push(self, obs, act, rew, next_obs, done, mask=None) -> None:
        slots = self.n_written % self.c
        before = self.n_written.copy()
        super().push(obs, act, rew, next_obs, done, mask)
        for a in np.nonzero(self.n_written != before)[0]:
            self.priority[a, slots[a]] = self.priority_max[a]

    def update(self, agent: int, slots: np.ndarray, delta: np.ndarray, alpha: float, eps: float) -> None:
        """The learn step's priority rule for one agent's drawn slots (non-finite priorities are not stored)."""
        p = priority_of(delta, alpha, eps)
        ok = np.isfinite(p)
        self.priority[agent, np.asarray(slots)[ok]] = p[ok]
        if ok.any():
            self.priority_max[agent] = max(self.priority_max[agent], p[ok].max())


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
    mean, denom = zscore_stats(r0) if normalize_rewards else (0.0, 1.0)
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



class ReplayStackedOracle(StackedOracle):
    """StackedOracle whose learn step weights every row's loss term by an importance weight and whose TD targets take a
    discount per row."""

    def td_targets(self, rewards, next_states, dones, discounts=None):
        """y = R + discount * Q_tgt(s'); ``discounts[N, B]`` None = gamma * (1 - dones), StackedOracle's one-step target
        (with every discount equal to gamma * (1 - done) the two agree bit for bit)."""
        if discounts is None:
            return super().td_targets(rewards, next_states, dones)
        r = torch.as_tensor(rewards, dtype=torch.float32)
        s2 = torch.as_tensor(next_states, dtype=torch.float32)
        disc = torch.as_tensor(np.asarray(discounts, np.float32))
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
        """As StackedOracle.learn_on_batch; ``is_weights[N, B]`` (None = 1) multiplies each row's loss term, so the loss
        is mean_i(w_i * term_i) and its gradient is that of the weighted loss; ``discounts[N, B]`` (None =
        gamma * (1 - dones)) replaces the one-step discount, and ``rewards`` are then the n-step returns.  Also returns
        ``delta`` = q(s)[a] - y."""
        n = self.n
        active = np.ones((n,), bool) if active is None else np.asarray(active, bool)
        s = torch.as_tensor(states, dtype=torch.float32)
        a = torch.as_tensor(actions, dtype=torch.int64)
        y, q_next, tq_all = self.td_targets(rewards, next_states, dones, discounts)
        params = [p.detach().requires_grad_(True) for p in self.online]
        q_all = self.forward(params, s)
        pred = torch.gather(q_all, 2, a[..., None])[..., 0]
        terms, _ = loss_and_grad(pred, y, self.loss_kind)
        if is_weights is not None:
            terms = torch.as_tensor(np.asarray(is_weights, np.float32)) * terms
        loss = terms.mean(dim=1)
        grads = torch.autograd.grad(loss.sum(), params)
        act_t = torch.as_tensor(active)
        with torch.no_grad():
            for i in np.nonzero(active)[0]:
                self.learn_step[i] += 1
                alpha, eps = adam_scalars(int(self.learn_step[i]), self.lr, self.adam_form)
                for p, g, m, v in zip(self.online, grads, self.adam_m, self.adam_v):
                    adam_update_(p[i], g[i], m[i], v[i], alpha, eps)
                if self.tau is not None:
                    tau = np.float32(self.tau)
                    for t, o in zip(self.target, self.online):
                        t[i].copy_(tau * o[i] + (np.float32(1.0) - tau) * t[i])
                elif self.learn_step[i] % self.freq == 0:
                    for t, o in zip(self.target, self.online):
                        t[i].copy_(o[i])
        return {
            "loss": torch.where(act_t, loss.detach(), torch.zeros_like(loss)).numpy(),
            "y": y.numpy(), "q_all": q_all.detach().numpy(), "q_next": q_next.numpy(),
            "tq_all": tq_all.numpy(), "grads": [g.numpy() for g in grads],
            "delta": (pred.detach() - y).numpy(),
        }
