"""CPU restatement of the quantile regression (QR-DQN) learn step and act of include/dmdqn_b200.h (dmdqn_quantile).

The midpoints, the expected values, the target samples and the pairwise quantile Huber terms follow the header's
operation order in float32 (every product, quotient and sum rounded on its own, no FMA); the trunk and the head run the
oracle's float32 forward.  The logit gradient is the closed form (w_r g_i) / loss_batch, and the parameter gradients are
its back-propagation through the network.  Built on tests/replay_oracle.py (importance weights, per-row discounts).
"""
from __future__ import annotations

import numpy as np
import torch

from oracle.dqn import adam_scalars, adam_update_
from replay_oracle import ReplayStackedOracle

F32 = np.float32


def midpoints(n: int) -> np.ndarray:
    """tau_i = (float)((2 i + 1) / (2.0 N)), the division in float64."""
    return np.array([(2 * i + 1) / (2.0 * n) for i in range(n)], np.float64).astype(F32)


def expected_q(x: np.ndarray) -> np.ndarray:
    """x[..., N] float32 -> (sum_i x_i in i order) / N."""
    x = np.asarray(x, F32)
    s = np.zeros(x.shape[:-1], F32)
    for i in range(x.shape[-1]):
        s = (s + x[..., i]).astype(F32)
    return (s / F32(x.shape[-1])).astype(F32)


def pair_terms(theta: np.ndarray, t: np.ndarray, kappa: float):
    """(rho, drho) [..., N(i), N(j)] float32 for quantiles theta [..., N] and target samples t [..., N]."""
    theta, t = np.asarray(theta, F32), np.asarray(t, F32)
    n = theta.shape[-1]
    tau = midpoints(n)[:, None]
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


def row_loss_and_grad(theta: np.ndarray, t: np.ndarray, kappa: float):
    """(L [...], g [..., N]) float32: L = (sum_i (sum_j rho_ij) in i order) / N, g_i = (sum_j drho_ij) / N."""
    rho, drho = pair_terms(theta, t, kappa)
    n = rho.shape[-1]
    lp = np.zeros(rho.shape[:-1], F32)
    gs = np.zeros(rho.shape[:-1], F32)
    for j in range(n):
        lp = (lp + rho[..., j]).astype(F32)
        gs = (gs + drho[..., j]).astype(F32)
    L = np.zeros(lp.shape[:-1], F32)
    for i in range(n):
        L = (L + lp[..., i]).astype(F32)
    return (L / F32(n)).astype(F32), (gs / F32(n)).astype(F32)


class QuantileOracle(ReplayStackedOracle):
    """ReplayStackedOracle with QR-DQN heads: ``online`` / ``target`` hold [W1, b1, W2, b2, W3 [H, A*N], b3 [A*N]] stacks
    (the host weight list), column a*N + i = quantile i of action a."""

    def __init__(self, n_nets, state_size, nn_layers, action_size, n_quantiles=50, kappa=1.0, **kw):
        super().__init__(n_nets, state_size, nn_layers, action_size * n_quantiles, **kw)
        self.a, self.n_quantiles, self.kappa = action_size, n_quantiles, kappa

    def quantiles(self, params, x) -> torch.Tensor:
        """[N, B, A, N] float32."""
        out = self.forward(params, torch.as_tensor(np.asarray(x, F32)))
        return out.reshape(out.shape[0], out.shape[1], self.a, self.n_quantiles)

    def q_values(self, obs) -> torch.Tensor:
        with torch.no_grad():
            x = self.quantiles(self.online, np.asarray(obs, F32)[:, None, :])[:, 0].numpy()
        return torch.as_tensor(expected_q(x))

    def targets(self, rewards, next_states, discounts):
        """(T [N, B, N], a* [N, B], q_next [N, B, A], tq_all [N, B, A]) from the online / target quantiles at s'."""
        with torch.no_grad():
            xo = self.quantiles(self.online, next_states).numpy()
            xt = self.quantiles(self.target, next_states).numpy()
        q_next, tq_all = expected_q(xo), expected_q(xt)
        best = np.argmax(q_next if self.double_dqn else tq_all, axis=2)
        th = np.take_along_axis(xt, best[..., None, None], 2)[:, :, 0]
        r, d = np.asarray(rewards, F32), np.asarray(discounts, F32)
        t = (r[..., None] + (d[..., None] * th).astype(F32)).astype(F32)
        return t, best, q_next, tq_all

    def learn_on_batch(self, states, actions, rewards, next_states, dones, active=None, is_weights=None, discounts=None,
                       loss_batch=None, apply=True):
        """One step on batches ``[N, B, ...]``; ``rewards`` are the returns R, ``discounts`` the per-row d (None =
        gamma * (1 - dones)).  Returns the targets, views, the row losses, the logit gradient and the parameter gradients
        (float32, before Adam); ``apply`` runs Adam and the target sync."""
        n, b = np.asarray(actions).shape
        active = np.ones((n,), bool) if active is None else np.asarray(active, bool)
        lb = b if loss_batch is None else loss_batch
        if discounts is None:
            discounts = (F32(self.gamma) * (F32(1.0) - np.asarray(dones, F32))).astype(F32)
        t, best, q_next, tq_all = self.targets(rewards, next_states, discounts)
        params = [p.detach().requires_grad_(True) for p in self.online]
        xt = self.quantiles(params, states)
        x = xt.detach().numpy()
        q_all = expected_q(x)
        a = np.asarray(actions, np.int64)
        xa = np.take_along_axis(x, a[..., None, None], 2)[:, :, 0]
        row, g = row_loss_and_grad(xa, t, self.kappa)
        w = np.ones((n, b), F32) if is_weights is None else np.asarray(is_weights, F32)
        terms = (w * row).astype(F32)
        dx = np.zeros(x.shape, F32)
        da = ((w[..., None] * g).astype(F32) / F32(lb)).astype(F32)
        np.put_along_axis(dx, a[..., None, None], da[:, :, None, :], 2)
        grads = torch.autograd.grad((xt * torch.as_tensor(dx)).sum(), params)   # back-propagation of dX
        loss = np.where(active, terms.sum(axis=1, dtype=np.float64) / lb, 0.0)
        if apply:
            with torch.no_grad():
                for i in np.nonzero(active)[0]:
                    self.learn_step[i] += 1
                    alpha, eps = adam_scalars(int(self.learn_step[i]), self.lr, self.adam_form)
                    for prm, gg, mm, v in zip(self.online, grads, self.adam_m, self.adam_v):
                        adam_update_(prm[i], gg[i], mm[i], v[i], alpha, eps)
                    if self.tau is not None:
                        tau = F32(self.tau)
                        for tt, o in zip(self.target, self.online):
                            tt[i].copy_(tau * o[i] + (F32(1.0) - tau) * tt[i])
                    elif self.learn_step[i] % self.freq == 0:
                        for tt, o in zip(self.target, self.online):
                            tt[i].copy_(o[i])
        return {"loss": loss, "T": t, "best": best, "q_all": q_all, "q_next": q_next, "tq_all": tq_all, "row_loss": row,
                "dlogits": dx, "grads": [gg.numpy() for gg in grads]}

    def act(self, obs, eps, w_explore, w_action):
        from oracle.dqn import explore_decision, random_action
        q = self.q_values(obs).numpy()
        greedy = np.argmax(q, axis=1).astype(np.int32)
        explore = explore_decision(w_explore, eps)
        return np.where(explore, random_action(w_action, self.a), greedy).astype(np.int32), q
