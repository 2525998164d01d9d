"""Per-agent facade with the reference's names: ``DQNAgent`` and ``ReplayBuffer``.

Mirrors reference src/agents/dqn_agent.py member for member (ctor :97-151, select_action
:246-274, store_experience :306-310, remember :312-325, learn :328-380,
update_target_network :382-387, update_target_network_soft :389-399, save_model/load_model
:401-422, get_epsilon :424-426, replay :428-434) plus ``select_greedy_action`` from
src/experimental/agent.py:148-152 (src/scripts/test.py:88 calls it).  Each object is a
1-agent view (offset pointers) onto an :class:`AgentGroup`; the arithmetic runs in
libdmdqn_b200.so.  Host-side randomness follows the reference exactly -- ``np.random`` for
the explore draw (:263-265) and ``random.sample`` for the replay indices (:63) -- so a
seeded reference run and a seeded facade run pick the same actions and transitions.  With
``sample_mode: prioritized`` ``learn()`` draws its batch on the device from the ring's priorities
instead (the reference has no prioritized replay, so there is no index stream to follow).
"""
from __future__ import annotations

import logging
import random

import numpy as np
import torch

from . import epsilon as epsilon_schedules
from .group import AgentGroup


logger = logging.getLogger("dmdqn_logger")        # the reference's logger name (log_config.py)


class ReplayBuffer:
    """``deque(maxlen=buffer_size)`` semantics on a device ring (dqn_agent.py:27-89)."""

    def __init__(self, buffer_size: int, _group: AgentGroup | None = None, state_size: int = 89,
                 batch_size: int = 128):
        self._g = _group if _group is not None else AgentGroup(
            1, {"replay_buffer_size": buffer_size, "batch_size": batch_size}, state_size)
        self.buffer_size = buffer_size

    def add(self, experience: tuple) -> None:
        state, action, reward, next_state, done = experience
        s = torch.as_tensor(np.asarray(state) if not isinstance(state, torch.Tensor) else state)
        s2 = torch.as_tensor(np.asarray(next_state) if not isinstance(next_state, torch.Tensor) else next_state)
        s, s2 = s.reshape(1, -1), s2.reshape(1, -1)      # np.squeeze(axis=0) of [1,D] (:45-46)
        if s.shape[1] != s2.shape[1]:                    # :50-54
            return
        self._g.push(s, [int(action)], [float(reward)], s2, [bool(done)])

    def sample(self, batch_size: int):
        """Five device tensors (states, actions i32, z-scored rewards, next_states, dones) or
        None while the buffer holds fewer than ``batch_size`` transitions (:61-62).  Indices
        come from ``random.sample`` exactly like the reference (:63)."""
        size = len(self)
        if size < batch_size:
            return None
        if batch_size != self._g.batch_size:
            raise ValueError(f"batch_size={batch_size} differs from the configured {self._g.batch_size}")
        idx = random.sample(range(size), batch_size)
        s, a, r, s2, d, _ = self._g.sample(np.asarray(idx, np.int32)[None], sample_mode="indices")
        return s[0], a[0], r[0], s2[0], d[0]

    def __len__(self) -> int:
        return int(min(self._g.n_written_host[0], self._g.capacity))


class _Network:
    """Stand-in for the Keras model attributes ``online_network`` / ``target_network``."""

    def __init__(self, group: AgentGroup, which: str):
        self._g, self._which = group, which

    def get_weights(self):
        return [w.numpy() for w in self._g.get_weights(0, self._which)]

    def set_weights(self, weights) -> None:
        self._g.set_weights(0, weights, self._which)

    def __call__(self, states) -> torch.Tensor:
        """Q-values ``[n, A]`` for ``states [n, D]`` (one act-kernel launch per row)."""
        x = torch.as_tensor(states, dtype=torch.float32).reshape(-1, self._g.state_size)
        target = self._which == "target"
        return torch.stack([self._g.act(row[None], return_q=True, target=target, noisy=False)[1][0, : self._g.action_size]
                            for row in x])


class DQNAgent:
    def __init__(self, state_size: int = 89, action_size: int = 4, agent_id: str = "J_0_0", config: dict | None = None,
                 _group: AgentGroup | None = None, _index: int = 0):
        config = dict(config or {})
        self.agent_id = agent_id
        self.state_size = int(state_size)       # the reference hard-codes 89/4 (:108-109); args honoured here
        self.action_size = int(action_size)
        self.learning_rate = config.get("learning_rate", 0.001)
        self.gamma = config.get("gamma", 0.99)
        self.epsilon = config.get("epsilon_start", 1.0)
        self.epsilon_min = config.get("epsilon_min", 0.01)
        self.epsilon_decay_steps = config.get("epsilon_decay_steps", 100000)
        self.epsilon_decay_rate = ((self.epsilon - self.epsilon_min) / self.epsilon_decay_steps
                                   if self.epsilon_decay_steps > 0 else 0)      # experimental/agent.py:82-84
        # 'reference' = the hard-coded exponential schedule of src/agents (:258-261, yaml epsilon_* keys ignored);
        # 'linear' = the variant's decay after every action (experimental/agent.py:140-144)
        self.epsilon_schedule = config.get("epsilon_schedule", "reference")
        if self.epsilon_schedule not in epsilon_schedules.KINDS:
            raise ValueError(f"epsilon_schedule={self.epsilon_schedule!r}: expected 'reference' or 'linear'")
        self.buffer_size = config.get("replay_buffer_size", 10000)
        self.batch_size = config.get("batch_size", 128)
        self.target_update_frequency = config.get("target_update_frequency", 1000)
        self.nn_layers = config.get("nn_layers", [64, 64])
        self.tau = config.get("tau", None)
        if _group is None:
            _group = AgentGroup(1, config, self.state_size, self.action_size, seed=config.get("seed", 0))
        self._g = _group.agent_view(_index)
        if self._g.noisy:       # noisy networks explore through their learned noise: no epsilon-greedy
            self.epsilon = self.epsilon_min = 0.0
        self.online_network = _Network(self._g, "online")
        self.target_network = _Network(self._g, "target")
        self.replay_buffer = ReplayBuffer(self.buffer_size, _group=self._g)
        self.global_step_count = 0
        self.learn_step_counter = 0
        self.last_metrics = None

    # -- act -----------------------------------------------------------------------------
    def update_epsilon_before_action(self) -> float:
        """The src/agents schedule, evaluated before the explore draw (:258-261); a no-op for 'linear'.  Always 0 for
        noisy networks."""
        if self._g.noisy:
            return self.epsilon
        self.epsilon = epsilon_schedules.before_action(self.epsilon_schedule, self.epsilon, self.epsilon_min,
                                                       self.global_step_count)
        return self.epsilon

    def update_epsilon_after_action(self) -> float:
        """The variant's linear decay, applied after the action was chosen (experimental/agent.py:140-144)."""
        if self._g.noisy:
            return self.epsilon
        self.epsilon = epsilon_schedules.after_action(self.epsilon_schedule, self.epsilon, self.epsilon_min,
                                                      self.epsilon_decay_rate)
        return self.epsilon

    def select_action(self, state_tensor) -> int:
        """Epsilon-greedy on the online network; with ``noisy: true`` greedy on the noisy online network (the noise of the
        next learn step), with no epsilon draw."""
        if self._g.noisy:
            return int(self._g.act(torch.as_tensor(state_tensor, dtype=torch.float32).reshape(1, -1)).item())
        self.update_epsilon_before_action()
        if np.random.rand() < self.epsilon:                                 # :263-265
            action = np.random.randint(0, self.action_size)
        else:
            action = self.select_greedy_action(state_tensor)
        self.update_epsilon_after_action()
        return action

    def select_greedy_action(self, state_tensor) -> int:
        """Greedy on the online network; for noisy networks on the mean weights mu alone (greedy evaluation)."""
        return int(self._g.act(torch.as_tensor(state_tensor, dtype=torch.float32).reshape(1, -1), noisy=False).item())

    # -- remember ------------------------------------------------------------------------
    def store_experience(self, experience) -> None:                        # :306-310
        self.replay_buffer.add(experience)
        self.global_step_count += 1

    def remember(self, state, action, reward, next_state, done) -> None:   # :312-325
        self.replay_buffer.add((state, action, reward, next_state, done))

    # -- learn ---------------------------------------------------------------------------
    def learn(self):
        """Loss as a 0-dim device tensor, or None while the buffer is short (:333-335)."""
        size = len(self.replay_buffer)
        if size < self.batch_size:
            return None
        if self._g.prioritized:     # proportional prioritized replay: the kernel draws from device words
            metrics = self._g.learn()
        else:
            idx = np.asarray(random.sample(range(size), self.batch_size), np.int32)[None]   # :63
            metrics = self._g.learn(idx, sample_mode="indices")
        self.learn_step_counter += 1                                        # :359
        self.last_metrics = metrics[0]
        return metrics[0, 0].clone()

    def replay(self):                                                       # :428-434
        loss = self.learn()
        return 0 if loss is None else loss

    def update_target_network(self) -> None:                                # :382-387
        self._g.sync_target()

    def update_target_network_soft(self) -> None:                           # :389-399 (tau made real)
        self._g.sync_target(tau=0.005 if self.tau is None else self.tau)

    # -- checkpoint ----------------------------------------------------------------------
    def save_model(self, filepath) -> None:                                 # :401-409 (online weights only)
        try:
            torch.save({"weights": self._g.get_weights(0), "nn_layers": self.nn_layers}, filepath)
        except Exception as exc:                                            # the reference logs and carries on (:408-409)
            logger.error("Agent %s: error saving model to %s: %s", self.agent_id, filepath, exc)

    def load_model(self, filepath) -> bool:                                 # :411-422
        try:
            blob = torch.load(filepath, weights_only=True)
            self._g.set_weights(0, blob["weights"], sync_target=True)
            return True
        except Exception as exc:
            logger.error("Agent %s: error loading model from %s: %s", self.agent_id, filepath, exc)
            return False

    def get_epsilon(self) -> float:                                         # :424-426
        return self.epsilon


def create_agents(tl_junctions, agent_config: dict, state_size: int = 89, action_size: int = 4,
                  seed: int = 0) -> tuple[dict, AgentGroup]:
    """``agents`` dict of the reference's train.py:109-127, all backed by ONE group so the
    batched calls and the per-agent facade see the same device state."""
    group = AgentGroup(len(tl_junctions), agent_config, state_size, action_size, seed=seed)
    agents = {j: DQNAgent(state_size, action_size, j, agent_config, _group=group, _index=i)
              for i, j in enumerate(tl_junctions)}
    return agents, group
