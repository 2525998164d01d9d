"""CPU restatement of implicit quantile networks (IQN) of include/dmdqn_b200.h (dmdqn_iqn): the device-drawn fractions, the
cosine features, the forward pass, the K-midpoint policy, the target samples, the pair terms with sampled fractions and a
stacked learn step whose parameter gradients back-propagate the closed-form quantile gradient through the network.

The fractions are the Philox restatement of tests/noisy_oracle.py; the midpoints, the expected values and the pair-term
order are those of tests/quantile_oracle.py; importance weights and per-row discounts come from the caller as in
tests/replay_oracle.py.  Every step after the head is one rounded float32 operation in the header's order (no FMA).
"""
from __future__ import annotations

import math

import numpy as np
import torch

import quantile_oracle as QO
from noisy_oracle import philox4x32_10
from oracle.dqn import adam_scalars, adam_update_
from replay_oracle import priority_of  # noqa: F401  (re-exported for the tests)

F32 = np.float32
IQN_TAG = 0x69716E00


def fractions(key: int, rows, n: int, t: int, s: int) -> np.ndarray:
    """[len(rows), n] float32: fraction i of row r, ((x >> 9) + 0.5) * 2^-23 with x the first Philox word of counter
    {r, i, t, 0x69716e00 | s} under the key's low and high words."""
    rows = np.asarray(rows, np.uint64)
    r = np.repeat(rows[:, None], n, 1)
    i = np.repeat(np.arange(n, dtype=np.uint64)[None, :], rows.shape[0], 0)
    x = philox4x32_10((r, i, np.full(r.shape, t, np.uint64), np.full(r.shape, IQN_TAG | s, np.uint64)),
                      (key & 0xFFFFFFFF, key >> 32))[0]
    return ((x >> np.uint32(9)).astype(F32) + F32(0.5)) * F32(2.0 ** -23)


def cos_features(tau, n_cos: int) -> np.ndarray:
    """[..., n_cos] float32: cos(pi * m * tau) in float64 (pi * m first), rounded."""
    tau = np.asarray(tau, F32).astype(np.float64)
    m = np.arange(n_cos)
    return np.cos((np.pi * m) * tau[..., None]).astype(F32)


def init_params(seed: int, state_size: int, hidden: int, action_size: int, n_cos: int) -> list[torch.Tensor]:
    """dmdqn_b200.group.keras_init with the cosine embedding, restated: [W1, b1, W2, b2, W3, b3, Wphi, bphi]."""
    gen = torch.Generator().manual_seed(int(seed))
    out = []
    for fi, fo in ((state_size, hidden), (hidden, hidden)):
        std = math.sqrt(2.0 / fi) / 0.87962566103423978
        w = torch.empty(fi, fo)
        torch.nn.init.trunc_normal_(w, 0.0, std, -2 * std, 2 * std, generator=gen)
        out += [w, torch.zeros(fo)]
    limit = math.sqrt(6.0 / (hidden + action_size))
    out += [(torch.rand(hidden, action_size, generator=gen) * 2 - 1) * limit, torch.zeros(action_size)]
    std = math.sqrt(2.0 / n_cos) / 0.87962566103423978
    w = torch.empty(n_cos, hidden)
    torch.nn.init.trunc_normal_(w, 0.0, std, -2 * std, 2 * std, generator=gen)
    return out + [w, torch.zeros(hidden)]


def forward(params, s, tau) -> torch.Tensor:
    """Z [G, B, M, A] for stacked params (leading network axis), states s [G, B, D] and fractions tau [G, B, M]."""
    w1, b1, w2, b2, w3, b3, wp, bp = params
    s = torch.as_tensor(np.asarray(s, F32))
    c = torch.as_tensor(cos_features(tau, wp.shape[1]))
    h1 = torch.relu(torch.einsum("gbd,gdh->gbh", s, w1) + b1[:, None])
    phi = torch.relu(torch.einsum("gbmc,gch->gbmh", c, wp) + bp[:, None, None])
    z = h1[:, :, None] * phi
    h2 = torch.relu(torch.einsum("gbmh,ghk->gbmk", z, w2) + b2[:, None, None])
    return torch.einsum("gbmh,gha->gbma", h2, w3) + b3[:, None, None]


def pair_terms(theta, t, tau, kappa: float):
    """(rho, drho) [..., N(i), N'(j)] float32: quantile_oracle.pair_terms with the fractions tau [..., N] as w's source."""
    theta, t, tau = np.asarray(theta, F32), np.asarray(t, F32), np.asarray(tau, F32)[..., :, None]
    u = (t[..., None, :] - theta[..., :, None]).astype(F32)
    w = np.where(u < 0, (F32(1.0) - tau).astype(F32), tau).astype(F32)
    k = F32(kappa)
    if k > 0:
        au = np.abs(u)
        quad = ((F32(0.5) * (u * u).astype(F32)).astype(F32) / k).astype(F32)
        lin = (au - (F32(0.5) * k).astype(F32)).astype(F32)
        rho = (w * np.where(au <= k, quad, lin)).astype(F32)
        drho = ((-w * np.minimum(np.maximum(u, -k), k)).astype(F32) / k).astype(F32)
    else:
        rho = (w * np.abs(u)).astype(F32)
        drho = np.where(u > 0, -w, np.where(u < 0, w, F32(0.0))).astype(F32)
    return rho, drho


def row_loss_and_grad(theta, t, tau, kappa: float):
    """(L [...], g [..., N]): L = (sum_i (sum_j rho_ij, j order), i order) / N', g_i = (sum_j drho_ij) / N'."""
    rho, drho = pair_terms(theta, t, tau, kappa)
    n, n_p = rho.shape[-2], rho.shape[-1]
    lp = np.zeros(rho.shape[:-1], F32)
    gs = np.zeros(rho.shape[:-1], F32)
    for j in range(n_p):
        lp = (lp + rho[..., j]).astype(F32)
        gs = (gs + drho[..., j]).astype(F32)
    L = np.zeros(lp.shape[:-1], F32)
    for i in range(n):
        L = (L + lp[..., i]).astype(F32)
    return (L / F32(n_p)).astype(F32), (gs / F32(n_p)).astype(F32)


def mean_over(z: torch.Tensor) -> np.ndarray:
    """Z [G, B, M, A] -> the mean over the M fractions in order, [G, B, A] (quantile_oracle.expected_q)."""
    return QO.expected_q(np.moveaxis(z.detach().numpy(), 2, 3))


class IqnOracle:
    """Stacked IQN networks: ``online`` / ``target`` / ``adam_m`` / ``adam_v`` hold [W1, b1, W2, b2, W3 [H, A], b3 [A],
    Wphi [n_cos, H], bphi [H]] with a leading network axis."""

    def __init__(self, n_nets, state_size, hidden, action_size, n_cos=64, n_tau=8, n_tau_prime=8, n_policy=32, kappa=1.0,
                 gamma=0.99, learning_rate=1e-3, target_update_frequency=1000, tau=None, double_dqn=True, seed0=0,
                 adam_form="keras"):
        self.n, self.a, self.n_cos = n_nets, action_size, n_cos
        self.n_tau, self.n_tau_prime, self.n_policy, self.kappa = n_tau, n_tau_prime, n_policy, kappa
        self.gamma, self.lr, self.freq, self.tau, self.double_dqn, self.adam_form = (
            gamma, learning_rate, target_update_frequency, tau, double_dqn, adam_form)
        per = [init_params(seed0 + g, state_size, hidden, action_size, n_cos) for g in range(n_nets)]
        self.online = [torch.stack(x) for x in zip(*per)]
        self.target = [p.clone() for p in self.online]
        self.adam_m = [torch.zeros_like(p) for p in self.online]
        self.adam_v = [torch.zeros_like(p) for p in self.online]
        self.learn_step = np.zeros(n_nets, np.int64)

    def policy_q(self, params, s) -> np.ndarray:
        """The K-midpoint Q [G, B, A]."""
        s = np.asarray(s, F32)
        mid = np.broadcast_to(QO.midpoints(self.n_policy), s.shape[:2] + (self.n_policy,))
        with torch.no_grad():
            return mean_over(forward(params, s, mid))

    def learn_on_batch(self, states, actions, rewards, next_states, discounts, tau, tau_p, is_weights=None, loss_batch=None,
                       active=None, apply=True):
        """One step on batches [G, B, ...] with the fractions tau [G, B, N] / tau_p [G, B, N'] (as the device drew them)."""
        g, b = np.asarray(actions).shape
        lb = b if loss_batch is None else loss_batch
        active = np.ones((g,), bool) if active is None else np.asarray(active, bool)
        q_on = self.policy_q(self.online, next_states)
        q_tg = self.policy_q(self.target, next_states)
        q_next = q_on if self.double_dqn else q_tg
        best = np.argmax(q_next, axis=2)
        with torch.no_grad():
            zt = forward(self.target, next_states, tau_p).numpy()          # [G, B, N', A]
        th_t = np.take_along_axis(zt, best[..., None, None], 3)[..., 0]
        r, d = np.asarray(rewards, F32), np.asarray(discounts, F32)
        t = (r[..., None] + (d[..., None] * th_t).astype(F32)).astype(F32)
        tq_all = QO.expected_q(np.moveaxis(zt, 2, 3))
        params = [p.detach().requires_grad_(True) for p in self.online]
        z = forward(params, states, tau)                                   # [G, B, N, A]
        zn = z.detach().numpy()
        q_all = QO.expected_q(np.moveaxis(zn, 2, 3))
        a = np.asarray(actions, np.int64)
        theta = np.take_along_axis(zn, a[..., None, None], 3)[..., 0]
        row, gi = row_loss_and_grad(theta, t, tau, self.kappa)
        w = np.ones((g, b), F32) if is_weights is None else np.asarray(is_weights, F32)
        grad = ((w[..., None] * gi).astype(F32) / F32(lb)).astype(F32)
        dz = np.zeros(zn.shape, F32)
        np.put_along_axis(dz, a[..., None, None], grad[..., None], 3)
        grads = torch.autograd.grad((z * torch.as_tensor(dz)).sum(), params)
        loss = np.where(active, (w * row).astype(F32).sum(axis=1, dtype=np.float64) / lb, 0.0)
        if apply:
            with torch.no_grad():
                for i in np.nonzero(active)[0]:
                    self.learn_step[i] += 1
                    alpha, eps = adam_scalars(int(self.learn_step[i]), self.lr, self.adam_form)
                    for prm, gg, mm, v in zip(self.online, grads, self.adam_m, self.adam_v):
                        adam_update_(prm[i], gg[i], mm[i], v[i], alpha, eps)
                    if self.tau is not None:
                        tt = F32(self.tau)
                        for x, o in zip(self.target, self.online):
                            x[i].copy_(tt * o[i] + (F32(1.0) - tt) * x[i])
                    elif self.learn_step[i] % self.freq == 0:
                        for x, o in zip(self.target, self.online):
                            x[i].copy_(o[i])
        return {"loss": loss, "T": t, "best": best, "q_all": q_all, "q_next": q_next, "tq_all": tq_all, "theta": theta,
                "grad": grad, "row_loss": row, "grads": [x.numpy() for x in grads]}

    def act(self, obs, eps, w_explore, w_action):
        from oracle.dqn import explore_decision, random_action
        q = self.policy_q(self.online, np.asarray(obs, F32)[:, None])[:, 0]     # network g acts on observation g
        greedy = np.argmax(q, axis=1).astype(np.int32)
        explore = explore_decision(w_explore, eps)
        return np.where(explore, random_action(w_action, self.a), greedy).astype(np.int32), q
