"""CPU restatement of Rainbow networks (config ``rainbow``; include/dmdqn_b200.h dmdqn_rainbow_layout): C51 heads with a
per-atom dueling fold on noisy layers.  Built from tests/dist_oracle.py (the C51 step), tests/noisy_oracle.py (Philox, the
factors and the fold eff = mu + sigma * eps) and tests/dueling_oracle.py (the fold and projection of one row of four
advantage values), applied per atom.  Test infrastructure."""
from __future__ import annotations

import numpy as np
import torch

import dist_oracle as DO
import dueling_oracle as DU
import noisy_oracle as NO
from oracle.dqn import adam_scalars, adam_update_

F32 = np.float32


def noise_record(key: int, t: int, s: int, rec, obs_dim: int, n_actions: int, n_atoms: int) -> np.ndarray:
    """One set's Rainbow noise record [rec.stride]: output factor a * Np + j of W3 is 0 unless a < A and j < N, value output
    j is 0 for j >= N; every other vector is noisy_oracle's."""
    off = NO.record_offsets(rec)
    off[8] = int(rec.v_out) + (off[5 + 1] - off[5]) // 4          # v_out is Np long (w3_out is 4 * Np)
    npad = (off[6] - off[5]) // 4
    out = np.zeros(int(rec.stride), np.float32)
    for v in range(8):
        n = off[v + 1] - off[v]
        f = NO.factor_vector(key, v, s, t, n, n)
        if v == 0:
            f[obs_dim:] = 0
        elif v == 5:
            col = np.arange(n)
            f[(col // npad >= n_actions) | (col % npad >= n_atoms)] = 0
        elif v == 7:
            f[n_atoms:] = 0
        out[off[v]:off[v + 1]] = f
    return out


def factors(record: np.ndarray, rec) -> list[np.ndarray]:
    off = NO.record_offsets(rec)
    off[8] = int(rec.v_out) + (off[6] - off[5]) // 4
    return [np.asarray(record[off[v]:off[v + 1]], np.float32) for v in range(8)]


def eps_block(record: np.ndarray, rec, layout, hidden: int) -> np.ndarray:
    """The noise of every float of a Rainbow block [layout.stride]: fin[k] * fout[col] for weights, fout[col] for biases."""
    f = factors(record, rec)
    L = layout
    e = np.zeros(int(L.stride), np.float32)
    e[L.w1:L.b1] = np.multiply.outer(f[0], f[1]).reshape(-1)
    e[L.b1:L.w2] = f[1]
    e[L.w2:L.b2] = np.multiply.outer(f[2], f[3]).reshape(-1)
    e[L.b2:L.w3] = f[3]
    e[L.w3:L.b3] = np.multiply.outer(f[4], f[5]).reshape(-1)
    e[L.b3:L.wv] = f[5]
    e[L.wv:L.bv] = np.multiply.outer(f[6], f[7]).reshape(-1)
    e[L.bv:L.end] = f[7]
    return e


def fold_heads(blk: np.ndarray, layout, hidden: int, n_actions: int, n_atoms: int) -> np.ndarray:
    """W3e | b3e [(H + 1) * 4 * Np] of a Rainbow block: dueling_oracle.fold_np per atom (fp32, the header's order)."""
    L, H = layout, hidden
    npad = (n_atoms + 3) // 4 * 4
    w3 = np.asarray(blk[L.w3:L.b3], F32).reshape(H, 4, npad)
    b3 = np.asarray(blk[L.b3:L.wv], F32).reshape(4, npad)
    wv = np.asarray(blk[L.wv:L.bv], F32).reshape(H, npad)
    bv = np.asarray(blk[L.bv:L.end], F32)
    out = np.zeros((H + 1, 4, npad), F32)
    for j in range(n_atoms):
        ew, eb = DU.fold_np(w3[:, :, j], b3[:, j], wv[:, j], bv[j], n_actions)
        out[:H, :, j], out[H, :, j] = ew, eb
    return out.reshape(-1)


def project_heads(g: np.ndarray, layout, hidden: int, n_actions: int, n_atoms: int) -> np.ndarray:
    """The Rainbow gradient block from the gradient G of W3e | b3e in a block's W3 / b3 region (the rest is copied):
    dueling_oracle.project_np per atom; Wv / bv get the sums, atoms j >= N get 0."""
    L, H = layout, hidden
    npad = (n_atoms + 3) // 4 * 4
    out = np.array(g, F32, copy=True)
    g3 = out[L.w3:L.b3].reshape(H, 4, npad).copy()
    gb = out[L.b3:L.wv].reshape(4, npad).copy()
    w3 = np.zeros_like(g3); b3 = np.zeros_like(gb)
    wv = np.zeros((H, npad), F32); bv = np.zeros(npad, F32)
    for j in range(n_atoms):
        w3[:, :, j], b3[:, j], wv[:, j], bv[j] = DU.project_np(g3[:, :, j], gb[:, j], n_actions)
    out[L.w3:L.b3], out[L.b3:L.wv] = w3.reshape(-1), b3.reshape(-1)
    out[L.wv:L.bv], out[L.bv:L.end] = wv.reshape(-1), bv
    return out


def c51_block(eff: np.ndarray, head: np.ndarray, layout, dist_stride: int) -> np.ndarray:
    """The C51 block [dist_stride] holding eff's trunk and the folded head (the same offsets up to b3 + 4 * Np)."""
    out = np.zeros(dist_stride, F32)
    out[:layout.w3] = eff[:layout.w3]
    out[layout.w3:layout.wv] = head
    return out


class RainbowOracle(DO.DistOracle):
    """DistOracle on Rainbow networks: ``online`` / ``target`` hold mu and ``sigma`` / ``sigma_tgt`` sigma as the host's
    weight lists [W1, b1, W2, b2, W3 [H, A*N], b3 [A*N], Wv [H, N], bv [N]].  The head's logits are
    x_{a,j} = V_j + Adv_{a,j} - mean_b Adv_{b,j}.  ``learn_on_batch`` runs DistOracle's step on eff = mu + sigma * eps (the
    step's noise per network as stacked parameter-shaped tensors), then Adam on mu with g and on sigma with g * eps."""

    def set_state(self, mu, sigma, mu_tgt, sigma_tgt, m, v, sm, sv):
        self.online, self.sigma, self.target, self.sigma_tgt = mu, sigma, mu_tgt, sigma_tgt
        self.adam_m, self.adam_v, self.sigma_m, self.sigma_v = m, v, sm, sv

    def forward(self, params, x):
        w1, b1, w2, b2, w3, b3, wv, bv = params
        h = torch.relu(torch.baddbmm(b1[:, None, :], x, w1))
        h = torch.relu(torch.baddbmm(b2[:, None, :], h, w2))
        adv = torch.baddbmm(b3[:, None, :], h, w3)
        adv = adv.reshape(adv.shape[0], adv.shape[1], self.a, self.n_atoms)
        v = torch.baddbmm(bv[:, None, :], h, wv)[:, :, None, :]
        return (v + adv - adv.mean(dim=2, keepdim=True)).reshape(adv.shape[0], adv.shape[1], -1)

    def learn_on_batch(self, states, actions, rewards, next_states, dones, eps_online=None, eps_target=None, active=None,
                       is_weights=None, discounts=None, loss_batch=None, apply=True):
        n = np.asarray(actions).shape[0]
        active = np.ones((n,), bool) if active is None else np.asarray(active, bool)
        mu, mu_t = self.online, self.target
        self.online = NO.NoisyStackedOracle.effective(mu, self.sigma, eps_online)
        self.target = NO.NoisyStackedOracle.effective(mu_t, self.sigma_tgt, eps_target)
        try:
            out = DO.DistOracle.learn_on_batch(self, states, actions, rewards, next_states, dones, active=active,
                                               is_weights=is_weights, discounts=discounts, loss_batch=loss_batch, apply=False)
        finally:
            self.online, self.target = mu, mu_t
        g_mu = [torch.as_tensor(g) for g in out["grads"]]
        g_sg = [g * e for g, e in zip(g_mu, eps_online)]
        out["g_mu"], out["g_sigma"] = [g.numpy() for g in g_mu], [g.numpy() for g in g_sg]
        if apply:
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
                            tau = F32(self.tau)
                            for t, o in zip(tgt, src):
                                t[i].copy_(tau * o[i] + (F32(1.0) - tau) * t[i])
                        elif self.learn_step[i] % self.freq == 0:
                            for t, o in zip(tgt, src):
                                t[i].copy_(o[i])
        return out


def eps_params(record: np.ndarray, rec, state_size: int, action_size: int, n_atoms: int) -> list[torch.Tensor]:
    """The noise of each parameter tensor in the host's order [W1, b1, W2, b2, W3 [H, A*N], b3 [A*N], Wv [H, N], bv [N]]."""
    f = factors(record, rec)
    d, a, n = state_size, action_size, n_atoms
    npad = (n + 3) // 4 * 4
    fo = f[5].reshape(4, npad)[:a, :n].reshape(-1)
    out = [np.multiply.outer(f[0][:d], f[1]), f[1], np.multiply.outer(f[2], f[3]), f[3], np.multiply.outer(f[4], fo), fo,
           np.multiply.outer(f[6], f[7][:n]), f[7][:n]]
    return [torch.as_tensor(np.ascontiguousarray(x, np.float32)) for x in out]
