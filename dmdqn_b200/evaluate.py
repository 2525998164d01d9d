"""Evaluation rollouts -- the reference's src/scripts/test.py (``run_evaluation_episode`` :48-150, ``main_eval``
:153-260) on the device path: greedy actions from ``select_greedy_action`` / one batched ``AgentGroup.act`` launch,
``random`` and ``fixed`` (fixed-time cycle) baselines, one CSV row per (mode, seed).

    python -m dmdqn_b200.evaluate --modes dqn random fixed --num_eval_episodes 2 --model_dir models/

The reference script drives a ``SumoTrafficEnvironment``; here ``TraciGridEnv`` offers the same four calls
(``reset(sumo_seed)``, ``step(actions) -> (obs, rewards, done, info)``, ``get_controlled_intersection_ids()``,
``get_action_size(id)``) over TraCI -- real SUMO when ``traci`` imports, the seeded queue model otherwise --
with the 89-dim observation ``DQNAgent`` is built for (order_lanes.py:502-555) and train.py's reward.  Noisy networks
(``noisy: true``) are evaluated greedily on their mean weights mu, without noise."""
from __future__ import annotations

import argparse
import csv
import json
import os
import sys
from collections import deque

import numpy as np
import torch

from .train import (ACTION_MAP, MAX_SIM_TIME, STEP_DURATION, get_traci, initialize_environment, load_config, read_traci,
                    set_seeds)


class TraciGridEnv:
    def __init__(self, config: dict, group=None, live_signal: bool = False, seed: int = 0):
        self.config, self.live_signal = dict(config), live_signal
        self.traci, self.is_fake = get_traci(self.config, seed)
        self.ids, self.table, self.nbr = initialize_environment(self.traci, self.config)
        self.group = group
        self.step_duration = float(self.config.get("step_duration", STEP_DURATION))
        self.max_sim_time = float(self.config.get("max_sim_time", MAX_SIM_TIME))
        self.lw = float(self.config.get("local_reward_weight", 0.3)); self.gw = float(self.config.get("global_reward_weight", 0.7))
        self.time = 0.0

    def get_controlled_intersection_ids(self):
        return list(self.ids)

    def get_action_size(self, agent_id):
        return len(ACTION_MAP)

    def _observe(self):
        rd = read_traci(self.traci, self.ids, self.table, self.live_signal)
        obs, _, reward, _ = self.group.featurize(*rd[:4], self.time, rd[4], self.nbr, local_weight=self.lw, global_weight=self.gw)
        self.obs_dev, self._reward_dev = obs, reward            # reward of THESE readings = pre-step reward of the next step
        host = obs[:, :89].cpu().numpy()
        return {j: host[i] for i, j in enumerate(self.ids)}

    def reset(self, sumo_seed: int = 0):
        if self.is_fake:
            self.traci.seed = int(sumo_seed)
        self.traci.load(["-c", self.config.get("sumo_cfg_path", ""), "--seed", str(sumo_seed)])
        self.time = float(self.traci.simulation.getTime())
        return self._observe()

    def step(self, actions: dict):
        for j in self.ids:
            self.traci.trafficlight.setPhase(j, ACTION_MAP[int(actions.get(j, 0))])     # train.py:225-226
        reward = self._reward_dev.cpu().numpy()                                           # train.py:241: pre-step readings
        target, done = self.time + self.step_duration, False
        while self.time < target:
            self.traci.simulationStep()
            self.time = float(self.traci.simulation.getTime())
            done = self.traci.simulation.getMinExpectedNumber() == 0 or self.time >= self.max_sim_time
        obs = self._observe()
        return obs, {j: float(reward[i]) for i, j in enumerate(self.ids)}, bool(done), {}

    def close(self):
        self.traci.close()


def run_evaluation_episode(env, config, episode_seed, mode="dqn", agents=None, eval_epsilon=0.01, fixed_cycle=None,
                           batched: bool = True):
    """test.py:48-150.  ``batched`` answers every greedy agent of a step with one ``AgentGroup.act`` launch; the
    numpy draws (explore test, random action) are made per agent in the reference's order either way."""
    set_seeds(episode_seed)
    observations = env.reset(sumo_seed=episode_seed)
    ids = env.get_controlled_intersection_ids()
    done, step = False, 0
    episode_rewards = {a: 0.0 for a in ids}
    all_step_queues = deque(maxlen=config.get("max_steps_per_episode", 1000) * len(ids))
    fixed_state = {}
    if mode == "fixed":
        if not fixed_cycle:
            print("Error: Fixed mode selected but no fixed_cycle definition provided.")
            return None
        fixed_state = {a: {"phase_idx": 0, "time_in_phase": 0.0} for a in ids}
    while not done:
        step += 1
        actions, greedy = {}, []
        for a in ids:
            if mode == "dqn":
                if agents and a in agents:
                    if np.random.rand() < eval_epsilon:
                        actions[a] = int(np.random.randint(0, env.get_action_size(a)))
                    elif batched and getattr(env, "group", None) is not None:
                        greedy.append(a)
                    else:
                        actions[a] = int(agents[a].select_greedy_action(torch.as_tensor(observations[a][None])))
                else:
                    actions[a] = int(np.random.randint(0, env.get_action_size(a)))
            elif mode == "random":
                actions[a] = int(np.random.randint(0, env.get_action_size(a)))
            else:                                               # fixed-time cycle: [(action, seconds), ...] per agent
                st, cyc = fixed_state[a], fixed_cycle[a]
                if st["time_in_phase"] >= cyc[st["phase_idx"]][1]:
                    st["phase_idx"] = (st["phase_idx"] + 1) % len(cyc)
                    st["time_in_phase"] = 0.0
                actions[a] = int(cyc[st["phase_idx"]][0])
                st["time_in_phase"] += config.get("step_duration", STEP_DURATION)
        if greedy:
            acts = env.group.act(env.obs_dev, noisy=False).cpu().numpy()     # greedy for all on mu, one launch
            for a in greedy:
                actions[a] = int(acts[ids.index(a)])
        next_observations, rewards, done, _ = env.step(actions)
        for a in ids:
            episode_rewards[a] += rewards.get(a, 0)
            all_step_queues.append(float(np.sum(observations[a][:12])))
        observations = next_observations
        if step >= config.get("max_steps_per_episode", 1000):
            done = True
    total = float(sum(episode_rewards.values()))
    return {"mode": mode, "seed": episode_seed, "total_reward": total,
            "avg_reward_per_agent": total / len(episode_rewards) if episode_rewards else 0.0,
            "avg_step_queue_sum": float(np.mean(all_step_queues)) if all_step_queues else 0.0, "steps": step}


def main_eval(args):
    """test.py:153-260: every mode over the same seeds, detailed CSV + per-mode means."""
    from .agent import create_agents
    paths = {k: v for k, v in (("agent_yaml_path", args.agent_config), ("env_yaml_path", args.env_config)) if v}
    config = load_config(**paths)
    config.update({k: v for k, v in vars(args).items() if v is not None})
    probe = TraciGridEnv(config, seed=args.eval_seed_start)
    agents, group = create_agents(probe.ids, config, seed=0)
    probe.group = group
    env = probe
    loaded = 0
    if args.model_dir:
        for j in env.ids:
            loaded += bool(agents[j].load_model(os.path.join(args.model_dir, f"{j}_online.weights.pt")))
    print(f"{loaded} of {len(env.ids)} agent models loaded from {args.model_dir!r}")
    fixed_cycle = {j: [(a, 30.0) for a in range(len(ACTION_MAP))] for j in env.ids}
    rows = []
    for mode in args.modes:
        for e in range(args.num_eval_episodes):
            r = run_evaluation_episode(env, config, args.eval_seed_start + e, mode, agents, args.eval_epsilon, fixed_cycle)
            if r:
                rows.append(r)
    env.close()
    if rows:
        with open(args.output_csv, "w", newline="") as f:
            w = csv.DictWriter(f, fieldnames=list(rows[0]))
            w.writeheader(); w.writerows(rows)
    summary = {m: {k: float(np.mean([r[k] for r in rows if r["mode"] == m])) for k in ("total_reward", "avg_step_queue_sum", "steps")}
               for m in args.modes if any(r["mode"] == m for r in rows)}
    print(json.dumps(summary))
    return rows


def parse_args(argv=None):
    ap = argparse.ArgumentParser(description="Evaluate DQN agents against random / fixed-time control")
    ap.add_argument("--agent_config", default=None); ap.add_argument("--env_config", default=None)
    ap.add_argument("--model_dir", default=None)
    ap.add_argument("--num_eval_episodes", type=int, default=2)
    ap.add_argument("--eval_seed_start", type=int, default=1000)
    ap.add_argument("--eval_epsilon", type=float, default=0.01)
    ap.add_argument("--modes", nargs="+", default=["dqn", "random"])
    ap.add_argument("--output_csv", default="evaluation_results.csv")
    ap.add_argument("--max_sim_time", type=float, default=None)
    return ap.parse_args(argv)


if __name__ == "__main__":
    sys.exit(0 if main_eval(parse_args()) else 1)
