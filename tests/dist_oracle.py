"""CPU restatement of the distributional (C51) learn step and act of include/dmdqn_b200.h (dmdqn_dist).

The support, the softmax statistics, the expected values and the projection follow the header's operation order in
float32 (every product and sum rounded on its own, ``fmaf`` where the header says so); the trunk and the head run the
oracle's float32 forward.  The logit gradient is the explicit (w_i (p_j - m_j)) / loss_batch, and the parameter gradients
are its back-propagation through the network.  Built on tests/replay_oracle.py (importance weights, per-row discounts).
"""
from __future__ import annotations

import numpy as np
import torch

from oracle.dqn import adam_scalars, adam_update_
from replay_oracle import ReplayStackedOracle

F32 = np.float32


def support(n: int, v_min: float, v_max: float):
    """(z[N] float32, lo, hi, dz): z_j = (float)(v_min + j * dz64), dz64 = (v_max - v_min) / (N - 1) in float64."""
    dz64 = (v_max - v_min) / (n - 1)
    z = np.array([v_min + j * dz64 for j in range(n)], np.float64).astype(F32)
    return z, F32(v_min), F32(v_max), F32(dz64)


def fmaf(a, b, c):
    """fp32 fused multiply-add: the product of two floats is exact in float64, one rounding of the sum (the float64 sum
    rounds first, which differs from a true fmaf in rare double-rounding cases far below the test tolerances)."""
    return (np.asarray(a, np.float64) * np.asarray(b, np.float64) + np.asarray(c, np.float64)).astype(F32)


def softmax_stats(x: np.ndarray):
    """x[..., N] float32 -> (mx, S): S summed in j order."""
    x = np.asarray(x, F32)
    mx = x.max(axis=-1)
    s = np.zeros(x.shape[:-1], F32)
    for j in range(x.shape[-1]):
        s = (s + np.exp(x[..., j] - mx)).astype(F32)
    return mx, s


def expected_q(x: np.ndarray, z: np.ndarray) -> np.ndarray:
    """Q = sum_j p_j z_j with fmaf in j order, p_j = expf(x_j - mx) / S."""
    x = np.asarray(x, F32)
    mx, s = softmax_stats(x)
    q = np.zeros(x.shape[:-1], F32)
    for j in range(x.shape[-1]):
        p = (np.exp(x[..., j] - mx) / s).astype(F32)
        q = fmaf(p, z[j], q)
    return q


def probs(x: np.ndarray) -> np.ndarray:
    mx, s = softmax_stats(x)
    return (np.exp(np.asarray(x, F32) - mx[..., None]) / s[..., None]).astype(F32)


def log_probs(x: np.ndarray) -> np.ndarray:
    mx, s = softmax_stats(x)
    return ((np.asarray(x, F32) - mx[..., None]) - np.log(s)[..., None]).astype(F32)


def project(p: np.ndarray, r: float, d: float, z: np.ndarray, lo, hi, dz) -> np.ndarray:
    """The header's projection of one row: p[N] onto the support after t = R + d z_j, in j order, float32."""
    n = z.shape[0]
    m = np.zeros(n, F32)
    r, d = F32(r), F32(d)
    for j in range(n):
        t = min(max(F32(r + F32(d * z[j])), lo), hi)
        b = min(F32(F32(t - lo) / dz), F32(n - 1))
        l, u = np.floor(b), np.ceil(b)
        li, ui = int(l), int(u)
        if li == ui:
            m[li] = F32(m[li] + p[j])
        else:
            m[li] = F32(m[li] + F32(p[j] * F32(u - b)))
            m[ui] = F32(m[ui] + F32(p[j] * F32(b - l)))
    return m


def project_float64(p: np.ndarray, r: float, d: float, z: np.ndarray, v_min: float, v_max: float) -> np.ndarray:
    """Algorithm 1 of Bellemare, Dabney & Munos (2017) in float64, independent of the header's statement."""
    n = z.shape[0]
    dz = (v_max - v_min) / (n - 1)
    zz = v_min + np.arange(n) * dz
    m = np.zeros(n)
    for j in range(n):
        tz = min(max(r + d * zz[j], v_min), v_max)
        b = (tz - v_min) / dz
        l, u = int(np.floor(b)), int(np.ceil(b))
        if l == u:
            m[l] += p[j]
        else:
            m[l] += p[j] * (u - b)
            m[u] += p[j] * (b - l)
    return m


class DistOracle(ReplayStackedOracle):
    """ReplayStackedOracle with C51 heads: ``online`` / ``target`` hold [W1, b1, W2, b2, W3 [H, A*N], b3 [A*N]] stacks (the
    host weight list), column a*N + j = atom j of action a."""

    def __init__(self, n_nets, state_size, nn_layers, action_size, n_atoms=51, v_min=-10.0, v_max=10.0, **kw):
        super().__init__(n_nets, state_size, nn_layers, action_size * n_atoms, **kw)
        self.a, self.n_atoms = action_size, n_atoms
        self.v_min, self.v_max = v_min, v_max
        self.z, self.lo, self.hi, self.dz = support(n_atoms, v_min, v_max)

    def logits(self, params, x) -> torch.Tensor:
        """[N, B, A, N] float32."""
        out = self.forward(params, torch.as_tensor(np.asarray(x, F32)))
        return out.reshape(out.shape[0], out.shape[1], self.a, self.n_atoms)

    def q_values(self, obs) -> torch.Tensor:
        with torch.no_grad():
            x = self.logits(self.online, np.asarray(obs, F32)[:, None, :])[:, 0].numpy()
        return torch.as_tensor(expected_q(x, self.z))

    def targets(self, rewards, next_states, discounts):
        """(m [N, B, N], a* [N, B], q_next [N, B, A], tq_all [N, B, A]) from the online / target logits at s'."""
        with torch.no_grad():
            xo = self.logits(self.online, next_states).numpy()
            xt = self.logits(self.target, next_states).numpy()
        q_next, tq_all = expected_q(xo, self.z), expected_q(xt, self.z)
        best = np.argmax(q_next if self.double_dqn else tq_all, axis=2)
        pt = probs(np.take_along_axis(xt, best[..., None, None], 2)[:, :, 0])
        r, d = np.asarray(rewards, F32), np.asarray(discounts, F32)
        m = np.zeros(pt.shape, F32)
        for g in range(m.shape[0]):
            for i in range(m.shape[1]):
                m[g, i] = project(pt[g, i], r[g, i], d[g, i], self.z, self.lo, self.hi, self.dz)
        return m, best, q_next, tq_all

    def learn_on_batch(self, states, actions, rewards, next_states, dones, active=None, is_weights=None, discounts=None,
                       loss_batch=None, apply=True):
        """One step on batches ``[N, B, ...]``; ``rewards`` are the returns R, ``discounts`` the per-row d (None =
        gamma * (1 - dones)).  Returns the targets, views, the cross-entropy, the logit gradient and the parameter
        gradients (float32, before Adam); ``apply`` runs Adam and the target sync."""
        n, b = np.asarray(actions).shape
        active = np.ones((n,), bool) if active is None else np.asarray(active, bool)
        lb = b if loss_batch is None else loss_batch
        if discounts is None:
            discounts = (F32(self.gamma) * (F32(1.0) - np.asarray(dones, F32))).astype(F32)
        m, best, q_next, tq_all = self.targets(rewards, next_states, discounts)
        params = [p.detach().requires_grad_(True) for p in self.online]
        xt = self.logits(params, states)
        x = xt.detach().numpy()
        q_all = expected_q(x, self.z)
        a = np.asarray(actions, np.int64)
        xa = np.take_along_axis(x, a[..., None, None], 2)[:, :, 0]
        lp, p = log_probs(xa), probs(xa)
        ce = np.zeros((n, b), F32)
        for j in range(self.n_atoms):
            ce = fmaf(m[..., j], lp[..., j], ce)
        ce = -ce
        w = np.ones((n, b), F32) if is_weights is None else np.asarray(is_weights, F32)
        terms = (w * ce).astype(F32)
        dx = np.zeros(x.shape, F32)
        da = ((w[..., None] * (p - m)).astype(F32) / F32(lb)).astype(F32)
        np.put_along_axis(dx, a[..., None, None], da[:, :, None, :], 2)
        grads = torch.autograd.grad((xt * torch.as_tensor(dx)).sum(), params)   # back-propagation of dX
        loss = np.where(active, terms.sum(axis=1, dtype=np.float64) / lb, 0.0)
        if apply:
            with torch.no_grad():
                for i in np.nonzero(active)[0]:
                    self.learn_step[i] += 1
                    alpha, eps = adam_scalars(int(self.learn_step[i]), self.lr, self.adam_form)
                    for prm, g, mm, v in zip(self.online, grads, self.adam_m, self.adam_v):
                        adam_update_(prm[i], g[i], mm[i], v[i], alpha, eps)
                    if self.tau is not None:
                        tau = F32(self.tau)
                        for t, o in zip(self.target, self.online):
                            t[i].copy_(tau * o[i] + (F32(1.0) - tau) * t[i])
                    elif self.learn_step[i] % self.freq == 0:
                        for t, o in zip(self.target, self.online):
                            t[i].copy_(o[i])
        return {"loss": loss, "m": m, "best": best, "q_all": q_all, "q_next": q_next, "tq_all": tq_all, "ce": ce,
                "dlogits": dx, "grads": [g.numpy() for g in grads]}

    def act(self, obs, eps, w_explore, w_action):
        from oracle.dqn import explore_decision, random_action
        q = self.q_values(obs).numpy()
        greedy = np.argmax(q, axis=1).astype(np.int32)
        explore = explore_decision(w_explore, eps)
        return np.where(explore, random_action(w_action, self.a), greedy).astype(np.int32), q
