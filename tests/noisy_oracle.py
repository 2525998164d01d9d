"""CPU restatement of noisy networks (config ``noisy``, Fortunato et al. 2018, factorized Gaussian noise; include/dmdqn_b200.h
dmdqn_noisy): the Philox4x32-10 counter-based generator, the Box-Muller factors f(z) = sgn(z) sqrt|z|, the noise of a
parameter block, the fold eff = mu + sigma * eps in the header's fp32 order, and a stacked learn step on noisy layers
W = mu + sigma * eps with gradients for mu and sigma from torch.autograd.  Test infrastructure, built on
tests/replay_oracle.py and oracle/dqn.py."""
from __future__ import annotations

import numpy as np
import torch

from oracle.dqn import adam_scalars, adam_update_, loss_and_grad
from replay_oracle import ReplayStackedOracle

_M32 = np.uint64(0xFFFFFFFF)
NOIS = 0x6e6f6973


def philox4x32_10(ctr, key):
    """Random123's Philox4x32-10 on uint32 counters ``ctr`` (four arrays or ints) and key ``(k0, k1)``: four uint32 arrays."""
    c0, c1, c2, c3 = (np.asarray(x, np.uint64) & _M32 for x in ctr)
    k0, k1 = np.uint64(key[0]) & _M32, np.uint64(key[1]) & _M32
    for r in range(10):
        if r:
            k0, k1 = (k0 + np.uint64(0x9E3779B9)) & _M32, (k1 + np.uint64(0xBB67AE85)) & _M32
        p0, p1 = c0 * np.uint64(0xD2511F53), c2 * np.uint64(0xCD9E8D57)
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _M32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _M32
    return tuple(x.astype(np.uint32) for x in (c0, c1, c2, c3))


def box_muller(x, y) -> np.ndarray:
    """z = sqrt(-2 ln((x + 0.5) 2^-32)) cos(2 pi y 2^-32) in float64, rounded to fp32."""
    u1 = (np.asarray(x, np.float64) + 0.5) * 2.0 ** -32
    u2 = np.asarray(y, np.float64) * 2.0 ** -32
    return (np.sqrt(-2.0 * np.log(u1)) * np.cos(2 * np.pi * u2)).astype(np.float32)


def factor(z) -> np.ndarray:
    z = np.asarray(z, np.float32)
    return np.where(z >= 0, np.sqrt(np.abs(z)), -np.sqrt(np.abs(z))).astype(np.float32)


def factor_vector(key: int, vec: int, s: int, t: int, n: int, valid: int) -> np.ndarray:
    """Entries 0..n of factor vector ``vec`` (2 * layer + side) of set ``s`` at step ``t``; entries >= valid are 0."""
    i = np.arange(n, dtype=np.uint64)
    x, y, _, _ = philox4x32_10((i, ((vec >> 1) << 2) | ((vec & 1) << 1) | s, t, NOIS), (key & 0xFFFFFFFF, key >> 32))
    f = factor(box_muller(x, y))
    f[valid:] = 0
    return f


def record_offsets(rec) -> list[int]:
    """The nine offsets of a NoiseRecord (eight vectors and the end) as ints."""
    names = ("w1_in", "w1_out", "w2_in", "w2_out", "w3_in", "w3_out", "v_in", "v_out")
    off = [int(getattr(rec, k)) for k in names]
    return off + [off[-1] + 4]


def noise_record(key: int, t: int, s: int, rec, obs_dim: int, n_actions: int) -> np.ndarray:
    """One set's noise record [rec.stride] (fp32)."""
    off = record_offsets(rec)
    out = np.zeros(int(rec.stride), np.float32)
    for v in range(8):
        n = off[v + 1] - off[v]
        valid = obs_dim if v == 0 else n_actions if v == 5 else 1 if v == 7 else n
        out[off[v]:off[v + 1]] = factor_vector(key, v, s, t, n, valid)
    return out


def factors(record: np.ndarray, rec) -> list[np.ndarray]:
    off = record_offsets(rec)
    return [np.asarray(record[off[v]:off[v + 1]], np.float32) for v in range(8)]


def eps_block(record: np.ndarray, rec, layout, hidden: int, dueling: bool) -> np.ndarray:
    """The noise of every float of a parameter block [layout.stride]: fin[i] * fout[j] (one fp32 product) for weights,
    fout[j] for biases, 0 on padding."""
    f = factors(record, rec)
    L, H = layout, hidden
    e = np.zeros(int(L.stride), np.float32)
    e[L.w1:L.b1] = np.multiply.outer(f[0], f[1]).reshape(-1)
    e[L.b1:L.w2] = f[1]
    e[L.w2:L.b2] = np.multiply.outer(f[2], f[3]).reshape(-1)
    e[L.b2:L.w3] = f[3]
    e[L.w3:L.b3] = np.multiply.outer(f[4], f[5]).reshape(-1)
    e[L.b3:L.b3 + 4] = f[5]
    if dueling:
        e[L.wv:L.wv + H] = f[6] * f[7][0]
        e[L.bv:L.bv + 4] = f[7]
    return e


def fold_np(mu: np.ndarray, sigma: np.ndarray, eps: np.ndarray) -> np.ndarray:
    """eff = mu + sigma * eps: one fp32 product, then one fp32 sum."""
    return (np.asarray(mu, np.float32) + np.asarray(sigma, np.float32) * np.asarray(eps, np.float32)).astype(np.float32)


def eps_params(record: np.ndarray, rec, state_size: int, action_size: int, dueling: bool) -> list[torch.Tensor]:
    """The noise of each parameter tensor in Keras order ([W1, b1, W2, b2, W3, b3] (+ [Wv, bv]))."""
    f = factors(record, rec)
    d, a = state_size, action_size
    out = [np.multiply.outer(f[0][:d], f[1]), f[1], np.multiply.outer(f[2], f[3]), f[3], np.multiply.outer(f[4], f[5][:a]),
           f[5][:a]]
    if dueling:
        out += [np.multiply.outer(f[6], f[7][:1]), f[7][:1]]
    return [torch.as_tensor(np.ascontiguousarray(x, np.float32)) for x in out]


class NoisyStackedOracle(ReplayStackedOracle):
    """ReplayStackedOracle over noisy networks: ``online`` / ``target`` hold mu, ``sigma`` / ``sigma_tgt`` sigma (the same
    Keras-ordered lists, plain or dueling heads), both learned by Adam and synchronised to the target.  ``learn_on_batch``
    takes the step's noise per network as stacked parameter-shaped tensors: ``eps_online`` for Q(s) and the argmax at s',
    ``eps_target`` for the target network."""

    def __init__(self, n_nets, state_size, nn_layers, action_size, *, dueling=False, **kw):
        super().__init__(n_nets, state_size, nn_layers, action_size, **kw)
        self.dueling = dueling

    def set_state(self, mu, sigma, mu_tgt, sigma_tgt, m, v, sm, sv):
        self.online, self.sigma, self.target, self.sigma_tgt = mu, sigma, mu_tgt, sigma_tgt
        self.adam_m, self.adam_v, self.sigma_m, self.sigma_v = m, v, sm, sv

    def forward(self, params, x):
        if not self.dueling:
            return ReplayStackedOracle.forward(params, x)
        w1, b1, w2, b2, w3, b3, wv, bv = params
        h = torch.relu(torch.baddbmm(b1[:, None, :], x, w1))
        h = torch.relu(torch.baddbmm(b2[:, None, :], h, w2))
        adv = torch.baddbmm(b3[:, None, :], h, w3)
        return torch.baddbmm(bv[:, None, :], h, wv) + adv - adv.mean(dim=2, keepdim=True)

    @staticmethod
    def effective(mu, sigma, eps):
        return [m + s * e for m, s, e in zip(mu, sigma, eps)]

    def learn_on_batch(self, states, actions, rewards, next_states, dones, eps_online, eps_target, active=None,
                       is_weights=None, discounts=None):
        n = self.n
        active = np.ones((n,), bool) if active is None else np.asarray(active, bool)
        s = torch.as_tensor(states, dtype=torch.float32)
        a = torch.as_tensor(actions, dtype=torch.int64)
        r = torch.as_tensor(rewards, dtype=torch.float32)
        s2 = torch.as_tensor(next_states, dtype=torch.float32)
        disc = torch.as_tensor(np.asarray(discounts, np.float32)) if discounts is not None else \
            np.float32(self.gamma) * (1 - torch.as_tensor(dones, dtype=torch.float32))
        with torch.no_grad():
            tq_all = self.forward(self.effective(self.target, self.sigma_tgt, eps_target), s2)
            q_next = self.forward(self.effective(self.online, self.sigma, eps_online), s2)
            if self.double_dqn:
                tq = torch.gather(tq_all, 2, torch.argmax(q_next, dim=2, keepdim=True))[..., 0]
            else:
                tq = tq_all.max(dim=2).values
            y = r + disc * tq
        mu = [p.detach().requires_grad_(True) for p in self.online]
        sg = [p.detach().requires_grad_(True) for p in self.sigma]
        q_all = self.forward(self.effective(mu, sg, eps_online), s)
        pred = torch.gather(q_all, 2, a[..., None])[..., 0]
        terms, _ = loss_and_grad(pred, y, self.loss_kind)
        if is_weights is not None:
            terms = torch.as_tensor(np.asarray(is_weights, np.float32)) * terms
        loss = terms.mean(dim=1)
        grads = torch.autograd.grad(loss.sum(), mu + sg)
        g_mu, g_sg = grads[:len(mu)], grads[len(mu):]
        with torch.no_grad():
            for i in np.nonzero(active)[0]:
                self.learn_step[i] += 1
                alpha, eps = adam_scalars(int(self.learn_step[i]), self.lr, self.adam_form)
                for ps, gs, ms, vs in ((self.online, g_mu, self.adam_m, self.adam_v),
                                       (self.sigma, g_sg, self.sigma_m, self.sigma_v)):
                    for p, g, m, v in zip(ps, gs, ms, vs):
                        adam_update_(p[i], g[i], m[i], v[i], alpha, eps)
                for tgt, src in ((self.target, self.online), (self.sigma_tgt, self.sigma)):
                    if self.tau is not None:
                        tau = np.float32(self.tau)
                        for t, o in zip(tgt, src):
                            t[i].copy_(tau * o[i] + (np.float32(1.0) - tau) * t[i])
                    elif self.learn_step[i] % self.freq == 0:
                        for t, o in zip(tgt, src):
                            t[i].copy_(o[i])
        return {"loss": np.where(active, loss.detach().numpy(), 0), "y": y.numpy(), "q_all": q_all.detach().numpy(),
                "q_next": q_next.numpy(), "tq_all": tq_all.numpy(), "g_mu": [g.numpy() for g in g_mu],
                "g_sigma": [g.numpy() for g in g_sg]}
