"""CPU restatement of the dueling Q-network (config ``dueling``, Wang et al. 2016): the textbook two-stream head
Q = V + Adv - mean_a Adv on the shared trunk, with gradients by torch.autograd.  It restates the model, not the folded
head the kernels use.  Test infrastructure, built on tests/replay_oracle.py and oracle/dqn.py."""
from __future__ import annotations

import numpy as np
import torch

from oracle.dqn import glorot_uniform, he_normal
from replay_oracle import ReplayStackedOracle


def dueling_init(seed: int, state_size: int, hidden: int, action_size: int) -> list[torch.Tensor]:
    """[W1, b1, W2, b2, W3, b3, Wv [H, 1], bv [1]]: oracle.dqn.init_params' draws, then Wv GlorotUniform(H, 1) from the
    same generator."""
    gen = torch.Generator().manual_seed(int(seed))
    w1 = he_normal(gen, state_size, hidden)
    w2 = he_normal(gen, hidden, hidden)
    w3 = glorot_uniform(gen, hidden, action_size)
    wv = glorot_uniform(gen, hidden, 1)
    return [w1, torch.zeros(hidden), w2, torch.zeros(hidden), w3, torch.zeros(action_size), wv, torch.zeros(1)]


class DuelingStackedOracle(ReplayStackedOracle):
    """ReplayStackedOracle over dueling networks: 8 parameter tensors per network, every one of them learned by Adam
    and synchronised to the target."""

    def __init__(self, n_nets: int, state_size: int, nn_layers, action_size: int, *, seed0: int = 0, **kw):
        super().__init__(n_nets, state_size, nn_layers, action_size, seed0=seed0, **kw)
        per = [dueling_init(seed0 + i, state_size, nn_layers[0], action_size) for i in range(n_nets)]
        self.online = [torch.stack([p[k] for p in per]) for k in range(8)]
        self.target = [p.clone() for p in self.online]
        self.adam_m = [torch.zeros_like(p) for p in self.online]
        self.adam_v = [torch.zeros_like(p) for p in self.online]

    @staticmethod
    def forward(params, x: torch.Tensor) -> torch.Tensor:
        w1, b1, w2, b2, w3, b3, wv, bv = params
        h = torch.relu(torch.baddbmm(b1[:, None, :], x, w1))
        h = torch.relu(torch.baddbmm(b2[:, None, :], h, w2))
        adv = torch.baddbmm(b3[:, None, :], h, w3)                  # [N, B, A]
        v = torch.baddbmm(bv[:, None, :], h, wv)                    # [N, B, 1]
        return v + adv - adv.mean(dim=2, keepdim=True)


# The folded head the kernels use (include/dmdqn_b200.h), restated in numpy fp32 with the header's arithmetic order for the
# bit-exact checks: sums left to right, an IEEE division by A, then (w - mean) + v.
def fold_np(w3: np.ndarray, b3: np.ndarray, wv: np.ndarray, bv, n_actions: int) -> tuple[np.ndarray, np.ndarray]:
    """W3 [H, 4], b3 [4], wv [H], bv -> W3e [H, 4], b3e [4] (fp32; columns >= A are 0)."""
    rows = np.concatenate([np.asarray(w3, np.float32).reshape(-1, 4), np.asarray(b3, np.float32).reshape(1, 4)])
    v = np.concatenate([np.asarray(wv, np.float32).reshape(-1), np.asarray(bv, np.float32).reshape(1)])
    s = rows[:, 0].copy()
    for b in range(1, n_actions):
        s = s + rows[:, b]
    mean = s / np.float32(n_actions)
    out = np.zeros_like(rows)
    for a in range(n_actions):
        out[:, a] = (rows[:, a] - mean) + v
    return out[:-1], out[-1]


def project_np(g3: np.ndarray, gb3: np.ndarray, n_actions: int) -> tuple[np.ndarray, np.ndarray, np.ndarray, np.float32]:
    """The folded head's gradient G [H, 4], Gb [4] -> (dW3 [H, 4], db3 [4], dwv [H], dbv) (fp32; columns >= A are 0)."""
    rows = np.concatenate([np.asarray(g3, np.float32).reshape(-1, 4), np.asarray(gb3, np.float32).reshape(1, 4)])
    s = rows[:, 0].copy()
    for b in range(1, n_actions):
        s = s + rows[:, b]
    mean = s / np.float32(n_actions)
    out = np.zeros_like(rows)
    for a in range(n_actions):
        out[:, a] = rows[:, a] - mean
    return out[:-1], out[-1], s[:-1], s[-1]
