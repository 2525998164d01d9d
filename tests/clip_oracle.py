"""CPU restatement of global-norm gradient clipping (dmdqn_clip_adam_apply, config ``global_clipnorm``): the float64 norm
and fp32 scale of one network's gradient, and a stacked learn step that clips each network's gradient before its Adam
step.  Test infrastructure, built on tests/replay_oracle.py and oracle/dqn.py."""
from __future__ import annotations

import numpy as np
import torch

from oracle.dqn import adam_scalars, adam_update_
from replay_oracle import ReplayStackedOracle


def clip_scale(grads, c: float) -> tuple[float, np.float32]:
    """Global-norm clipping of one network's gradient tensors (tf.clip_by_global_norm, dmdqn_clip_adam_apply): the
    float64 norm n of all elements and the fp32 scale (float)(c / max(n, c)), 1 when n is not finite."""
    sq = sum(float(np.sum(np.square(np.asarray(g, np.float32).astype(np.float64)))) for g in grads)
    n = float(np.sqrt(sq))
    return n, (np.float32(c / max(n, c)) if np.isfinite(n) else np.float32(1.0))


class ClipStackedOracle(ReplayStackedOracle):
    """ReplayStackedOracle whose learn step can clip each learning network's gradient to a global norm."""

    def learn_on_batch(self, states, actions, rewards, next_states, dones, active=None, is_weights=None, discounts=None,
                       global_clipnorm=None):
        """As ReplayStackedOracle.learn_on_batch; ``global_clipnorm`` c (None = no clipping, the parent's step) scales
        each learning network's gradient by ``clip_scale`` before its Adam step and target sync.  Also returns
        ``norms[N]``: the float64 norm before clipping, 0 for an inactive network (zeros without clipping)."""
        n = self.n
        if global_clipnorm is None:
            out = super().learn_on_batch(states, actions, rewards, next_states, dones, active, is_weights, discounts)
            out["norms"] = np.zeros((n,))
            return out
        saved = [[p.clone() for p in ps] for ps in (self.online, self.target, self.adam_m, self.adam_v)]
        step0 = self.learn_step.copy()
        out = super().learn_on_batch(states, actions, rewards, next_states, dones, active, is_weights, discounts)
        for ps, ss in zip((self.online, self.target, self.adam_m, self.adam_v), saved):   # undo the unclipped update
            for p, s in zip(ps, ss):
                p.copy_(s)
        self.learn_step[:] = step0
        active = np.ones((n,), bool) if active is None else np.asarray(active, bool)
        grads = [torch.as_tensor(g) for g in out["grads"]]
        norms = np.zeros((n,))
        with torch.no_grad():
            for i in np.nonzero(active)[0]:
                self.learn_step[i] += 1
                alpha, eps = adam_scalars(int(self.learn_step[i]), self.lr, self.adam_form)
                gi = [g[i] for g in grads]
                norms[i], scale = clip_scale(gi, global_clipnorm)
                if scale != 1:
                    gi = [g * scale for g in gi]
                for p, g, m, v in zip(self.online, gi, self.adam_m, self.adam_v):
                    adam_update_(p[i], g, m[i], v[i], alpha, eps)
                if self.tau is not None:
                    tau = np.float32(self.tau)
                    for t, o in zip(self.target, self.online):
                        t[i].copy_(tau * o[i] + (np.float32(1.0) - tau) * t[i])
                elif self.learn_step[i] % self.freq == 0:
                    for t, o in zip(self.target, self.online):
                        t[i].copy_(o[i])
        out["norms"] = norms
        return out
