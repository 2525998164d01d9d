"""Oracle: replay buffer, sampling-index contracts and reward z-score.

TEST INFRASTRUCTURE (see oracle/__init__.py).  Restates, on the CPU:

* ``ReplayBuffer.__init__/add/__len__``  reference src/agents/dqn_agent.py:27-57,87-89
* ``ReplayBuffer.sample``                 reference src/agents/dqn_agent.py:59-85
* the ``deque(maxlen=C)`` <-> ring mapping used by the device ring
  (SURVEY.md App. A.5): logical j (0 = oldest) <-> physical
  ``(n_written - size + j) mod C``.
* the "supplied draws" index contracts (SURVEY.md App. A.6) -- these are NEW
  contracts (the reference draws with CPython ``random.sample``); the
  reference-exact stream is available through explicit-index mode, see
  :func:`cpython_sample_indices`.
"""
from __future__ import annotations

import random
from collections import deque

import numpy as np

MASK32 = (1 << 32) - 1


# ----------------------------------------------------------------------------
# Faithful single-agent buffer (deque + random.sample), numpy outputs.
# ----------------------------------------------------------------------------
class FaithfulReplayBuffer:
    """Line-by-line behavioural restatement of reference ``ReplayBuffer``
    (src/agents/dqn_agent.py:27-89) with numpy in place of ``tf.convert_to_tensor``.

    ``rng`` is a ``random.Random`` (defaults to the module-global generator the
    reference uses).  ``normalize_rewards`` exists only so tests can look at raw
    rewards; the reference always normalises (dqn_agent.py:66-69).
    """

    def __init__(self, buffer_size: int, rng: random.Random | None = None):
        self.buffer = deque(maxlen=buffer_size)  # dqn_agent.py:29
        self._rng = rng

    def add(self, experience: tuple) -> None:
        state, action, reward, next_state, done = experience
        state_copy = np.array(state, copy=True)  # dqn_agent.py:39-40
        next_state_copy = np.array(next_state, copy=True)
        state_copy = np.squeeze(state_copy, axis=0)  # dqn_agent.py:45-46 ([1,D] -> [D])
        next_state_copy = np.squeeze(next_state_copy, axis=0)
        if len(state_copy) != len(next_state_copy):  # dqn_agent.py:50-54 (drop)
            return
        self.buffer.append((state_copy, action, reward, next_state_copy, done))

    def sample(self, batch_size: int, normalize_rewards: bool = True):
        if len(self.buffer) < batch_size:  # dqn_agent.py:61-62
            return None
        sampler = self._rng.sample if self._rng is not None else random.sample
        batch = sampler(self.buffer, batch_size)  # dqn_agent.py:63
        states, actions, rewards, next_states, dones = map(np.array, zip(*batch))
        if normalize_rewards:
            rewards = zscore(rewards)  # dqn_agent.py:66-69
        return (
            np.asarray(states, dtype=np.float32),
            np.asarray(actions, dtype=np.int32),
            np.asarray(rewards, dtype=np.float32),
            np.asarray(next_states, dtype=np.float32),
            np.asarray(dones, dtype=np.float32),
        )

    def __len__(self) -> int:
        return len(self.buffer)


def zscore(rewards: np.ndarray) -> np.ndarray:
    """``(r - mean) / (std_pop + 1e-8)`` in float64 -- dqn_agent.py:66-69, numpy order."""
    r = np.asarray(rewards, dtype=np.float64)
    return (r - np.mean(r)) / (np.std(r) + 1e-8)


def _tree_sum(x: np.ndarray) -> np.ndarray:
    """Canonical float64 sum over the last axis: lane l (0..31) adds x[l], x[l+32], ... in
    order, then the lanes are combined with an xor butterfly (offsets 16,8,4,2,1)."""
    pad = (-x.shape[-1]) % 32
    if pad:
        x = np.concatenate([x, np.zeros(x.shape[:-1] + (pad,), np.float64)], axis=-1)
    x = x.reshape(x.shape[:-1] + (-1, 32))
    acc = np.zeros(x.shape[:-2] + (32,), np.float64)
    for row in range(x.shape[-2]):
        acc = acc + x[..., row, :]
    lanes = np.arange(32)
    for off in (16, 8, 4, 2, 1):
        acc = acc + acc[..., lanes ^ off]
    return acc[..., 0]


def zscore_stats(rewards: np.ndarray) -> tuple[np.ndarray, np.ndarray]:
    """``(mean, std + 1e-8)`` of ``[..., B]`` float64 rewards with the CUDA kernel's fixed
    summation tree (:func:`_tree_sum`): mean = total / B; the squared deviations
    ``(r-mean)*(r-mean)`` (multiply rounded, then added: no FMA) go through the same tree;
    std = sqrt(total / B).  The n-step returns normalise every reward with these."""
    r = np.asarray(rewards, dtype=np.float64)
    b = r.shape[-1]
    mean = _tree_sum(r) / b
    dev = r - mean[..., None]
    var = _tree_sum(dev * dev) / b
    return mean, np.sqrt(var) + 1e-8


def zscore_canonical(rewards: np.ndarray) -> np.ndarray:
    """Same statistic as :func:`zscore` with the FIXED summation tree the CUDA kernel uses
    (:func:`zscore_stats`), so the device result can be compared bit-for-bit (float64 ops
    are IEEE on both sides): out = (r - mean) / (std + 1e-8).

    ``rewards`` is ``[..., B]`` float64; leading dims are independent batches.
    """
    r = np.asarray(rewards, dtype=np.float64)
    mean, denom = zscore_stats(r)
    return (r - mean[..., None]) / denom[..., None]


# ----------------------------------------------------------------------------
# Ring <-> deque mapping (device layout) for N agents.
# ----------------------------------------------------------------------------
def ring_physical(n_written: int, capacity: int, logical: np.ndarray) -> np.ndarray:
    """Physical ring slot of logical index j (0 = oldest) -- SURVEY.md App. A.5."""
    size = min(n_written, capacity)
    return (n_written - size + np.asarray(logical, dtype=np.int64)) % capacity


class RingReplay:
    """Array-of-rings replay for N agents with the device layout
    (``obs[N,C,D]``, ``next_obs[N,C,D]``, ``act[N,C]`` i32, ``rew[N,C]`` f64,
    ``done[N,C]`` u8, ``n_written[N]`` i64).  ``deque(maxlen=C)`` semantics
    (dqn_agent.py:29,56): append at the head, overwrite the oldest when full."""

    def __init__(self, n_agents: int, capacity: int, obs_dim: int):
        self.n, self.c, self.d = n_agents, capacity, obs_dim
        self.obs = np.zeros((n_agents, capacity, obs_dim), np.float32)
        self.next_obs = np.zeros((n_agents, capacity, obs_dim), np.float32)
        self.act = np.zeros((n_agents, capacity), np.int32)
        self.rew = np.zeros((n_agents, capacity), np.float64)
        self.done = np.zeros((n_agents, capacity), np.uint8)
        self.n_written = np.zeros((n_agents,), np.int64)

    def size(self) -> np.ndarray:
        return np.minimum(self.n_written, self.c)

    def push(self, obs, act, rew, next_obs, done, mask=None) -> None:
        """One transition per agent (rows of the ``[N,...]`` inputs); ``mask[N]``
        selects which agents store (dqn_agent.py:312-325 called per agent)."""
        for a in range(self.n):
            if mask is not None and not mask[a]:
                continue
            slot = int(self.n_written[a] % self.c)
            self.obs[a, slot] = obs[a]
            self.next_obs[a, slot] = next_obs[a]
            self.act[a, slot] = act[a]
            self.rew[a, slot] = rew[a]
            self.done[a, slot] = 1 if done[a] else 0
            self.n_written[a] += 1

    def logical_to_slot(self, agent: int, logical: np.ndarray) -> np.ndarray:
        return ring_physical(int(self.n_written[agent]), self.c, logical)

    def gather(self, agent: int, logical: np.ndarray, normalize_rewards: bool = True,
               canonical: bool = True):
        """The five ``sample`` outputs (dqn_agent.py:64-85) for given logical indices."""
        slot = self.logical_to_slot(agent, logical)
        r = self.rew[agent, slot]
        if normalize_rewards:
            r = zscore_canonical(r) if canonical else zscore(r)
        return (
            self.obs[agent, slot].copy(),
            self.act[agent, slot].copy(),
            r.astype(np.float32),
            self.next_obs[agent, slot].copy(),
            self.done[agent, slot].astype(np.float32),
        )


# ----------------------------------------------------------------------------
# Index contracts.
# ----------------------------------------------------------------------------
def cpython_sample_indices(rng: random.Random, size: int, batch: int) -> np.ndarray:
    """Reference-exact logical indices: ``random.sample(deque, B)`` (dqn_agent.py:63)
    picks positions exactly as ``random.sample(range(len), B)`` does (CPython's
    ``sample`` only indexes the population), so explicit-index mode fed with this
    reproduces the reference's stream for a given ``random.seed``."""
    return np.asarray(rng.sample(range(size), batch), dtype=np.int32)


def fisher_yates_indices(words: np.ndarray, size: int) -> np.ndarray:
    """"Draws, without replacement" contract (SURVEY.md App. A.6 (ii)): sparse
    partial Fisher-Yates restating CPython's pool path (random.py ``sample``:
    ``j = randbelow(n-i); result[i] = pool[j]; pool[j] = pool[n-i-1]``) with
    ``randbelow(m) := (w_i * m) >> 32`` on the supplied uint32 word ``w_i``.
    Returns B distinct logical indices in [0, size)."""
    words = np.asarray(words, dtype=np.uint64)
    b = words.shape[0]
    assert b <= size
    pool: dict[int, int] = {}
    out = np.empty((b,), np.int32)
    for i in range(b):
        m = size - i
        j = (int(words[i]) * m) >> 32
        out[i] = pool.get(j, j)
        pool[j] = pool.get(m - 1, m - 1)
    return out


def replacement_indices(words: np.ndarray, size: int) -> np.ndarray:
    """"Draws, with replacement" contract (App. A.6 (iii)): ``(w_i * size) >> 32``.
    A flagged deviation from the reference (which samples distinct items)."""
    w = np.asarray(words, dtype=np.uint64)
    return ((w * np.uint64(size)) >> np.uint64(32)).astype(np.int32)


def explore_decision(w_explore: np.ndarray, eps: np.ndarray) -> np.ndarray:
    """``u < eps`` with ``u = w / 2**32`` (dqn_agent.py:263), evaluated exactly in
    float64 as ``w < eps * 2**32``."""
    return np.asarray(w_explore, np.float64) < np.asarray(eps, np.float64) * 4294967296.0


def random_action(w_action: np.ndarray, n_actions: int) -> np.ndarray:
    """Uniform action in [0, A) from a uint32 word (dqn_agent.py:265 analogue)."""
    w = np.asarray(w_action, dtype=np.uint64)
    return ((w * np.uint64(n_actions)) >> np.uint64(32)).astype(np.int32)
