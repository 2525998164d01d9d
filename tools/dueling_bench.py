"""Cost of dueling Q-networks (config ``dueling``) on one GPU.

* cfg3 (256 agents, batch 256, hidden [256, 256], capacity 30 000, full rings, precision tf32x3): device-resident learn
  sweeps of a plain and a dueling group with the same seeded rings and trunk weights, alternated in one process,
  ``--rounds`` rounds of ``--steps`` timed sweeps after ``--warmup`` untimed ones, CUDA events around each run of sweeps.
  The dueling sweep adds the fold kernel and H + 4 Adam elements per network.
* cfg2 (16 agents, batch 64) the same way, each sweep one CUDA graph replay (``capture_learn``): there the extra launch
  counts.
* Where the cfg3 difference goes: each stage of ``dmdqn_learn_stages`` (sample -- in dueling mode the fold kernel and the
  sample kernel --, K3, K4a, K4b) issued as its own call, CUDA events between the calls, dueling against plain.
* The fold kernel alone at cfg3: its device time from ``torch.profiler`` over ``--steps`` dueling learn sweeps, in a pass
  of its own after the timed ones.
* ``dmdqn_act`` against ``dmdqn_act_dueling`` on 768 agents (greedy, hidden 256).

The card's name, power limit and maximum SM clock are read in the same run.  Prints one JSON object; ``--out FILE`` also
writes it there.

    python tools/dueling_bench.py --out profiles/r07_dueling_cfg3.json
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

import torch  # noqa: E402

from dmdqn_b200 import _native as N  # noqa: E402
from dmdqn_b200.group import AgentGroup  # noqa: E402
from tools.sample_bench import card, timed  # noqa: E402

D, A = 89, 4
CFG3 = dict(agents=256, batch=256, hidden=256, capacity=30000)
CFG2 = dict(agents=16, batch=64, hidden=256, capacity=30000)
STAGES = {"sample": 1, "target": 2, "online": 4, "wgrad": 8}


def make_group(w, dueling, seed=11):
    cfg = {"nn_layers": [w["hidden"], w["hidden"]], "replay_buffer_size": w["capacity"], "batch_size": w["batch"],
           "learning_rate": 5e-4, "target_update_frequency": 1000, "dueling": dueling}
    grp = AgentGroup(w["agents"], cfg, D, A, seed=seed)
    n, cap = grp.n_agents, grp.capacity
    gen = torch.Generator(device=grp.device).manual_seed(seed)
    grp.obs[:, :, :D] = torch.randint(-1, 20, (n, cap, D), device=grp.device, generator=gen).float()
    grp.next_obs[:, :, :D] = torch.randint(-1, 20, (n, cap, D), device=grp.device, generator=gen).float()
    grp.act_ring.copy_(torch.randint(0, A, (n, cap), device=grp.device, generator=gen).int())
    grp.rew_ring.copy_(-torch.randint(0, 5000, (n, cap), device=grp.device, generator=gen).double() * 0.7)
    grp.done_ring.copy_((torch.rand((n, cap), device=grp.device, generator=gen) < 0.05).to(torch.uint8))
    grp.n_written.fill_(cap); grp.n_written_host[:] = cap
    return grp


def sweeps(groups, draws, args, replay=None):
    """Median us per sweep of every group over alternating rounds; ``replay[k]`` (a graph replay) replaces learn()."""
    for k, g in groups.items():
        for i in range(args.warmup):
            if replay:
                replay[k][1].copy_(draws[i])
                replay[k][0]()
            else:
                g.learn(draws[i])
    torch.cuda.synchronize()
    res = {k: [] for k in groups}
    for _ in range(args.rounds):
        for k, g in groups.items():
            if replay:
                fn, buf = replay[k]
                res[k].append(timed(lambda d, fn=fn, buf=buf: (buf.copy_(d), fn()), draws, args.warmup))
            else:
                res[k].append(timed(lambda d, g=g: g.learn(d), draws, args.warmup))
    for g in groups.values():
        g.check_errors()
    return {k: {"median": statistics.median(v), "rounds": v} for k, v in res.items()}


def stage_times(grp, draws, start):
    """us per call of each learn stage, issued one stage per call with an event before and after each."""
    stream = torch.cuda.current_stream()
    tot = dict.fromkeys(STAGES, 0.0)
    for i in range(start, draws.shape[0]):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(STAGES) + 1)]
        ev[0].record(stream)
        for k, (name, bit) in enumerate(STAGES.items()):
            N.check(grp.lib.dmdqn_learn_stages(C.byref(grp.dims), C.byref(grp.hp), C.byref(grp.replay), C.byref(grp.nets),
                                               draws[i].data_ptr(), None, grp.metrics.data_ptr(), grp.workspace.data_ptr(),
                                               grp.workspace.numel(), bit, stream.cuda_stream))
            ev[k + 1].record(stream)
        ev[-1].synchronize()
        for k, name in enumerate(STAGES):
            tot[name] += ev[k].elapsed_time(ev[k + 1]) * 1e3
    return {k: v / (draws.shape[0] - start) for k, v in tot.items()}


def fold_kernel_us(grp, draws, start):
    """Mean device time of fold_kernel over the learn sweeps, from torch.profiler (a pass of its own)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(start, draws.shape[0]):
            grp.learn(draws[i])
        torch.cuda.synchronize()
    times = [e.device_time for e in prof.events() if "fold_kernel" in e.name]          # us per launch
    if not times:
        raise RuntimeError("torch.profiler recorded no fold_kernel launch")
    return {"median": statistics.median(times), "launches": len(times)}


def act_only(grp, obs):
    def run(_):
        grp.act(obs)
    return run


def alternate(fns, draws, args):
    res = {k: [] for k in fns}
    for _ in range(args.rounds):
        for k, fn in fns.items():
            res[k].append(timed(fn, draws, args.warmup))
    return {k: {"median": statistics.median(v), "rounds": v} for k, v in res.items()}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("dueling_bench.py measures on a CUDA device; none is visible")
    g3 = {"plain": make_group(CFG3, False), "dueling": make_group(CFG3, True)}
    draws = g3["plain"].draw_words((args.warmup + args.steps, CFG3["agents"], CFG3["batch"]))
    cfg3 = sweeps(g3, draws, args)
    per_stage = {k: [] for k in g3}
    for _ in range(args.rounds):
        for k, g in g3.items():
            per_stage[k].append(stage_times(g, draws, args.warmup))
    per_stage = {k: {s: statistics.median(r[s] for r in v) for s in STAGES} for k, v in per_stage.items()}
    fold = fold_kernel_us(g3["dueling"], draws, args.warmup)
    for g in g3.values():
        g.check_errors()
    precision = list(N.PRECISION)[g3["plain"].hp.precision]
    del g3, draws
    torch.cuda.empty_cache()

    g2 = {"plain": make_group(CFG2, False), "dueling": make_group(CFG2, True)}
    replay = {k: g.capture_learn() for k, g in g2.items()}       # (replay, draws buffer)
    draws2 = g2["plain"].draw_words((args.warmup + args.steps, CFG2["agents"], CFG2["batch"]))
    cfg2 = sweeps(g2, draws2, args, replay)
    del g2, replay, draws2
    torch.cuda.empty_cache()

    wa = dict(agents=768, batch=64, hidden=256, capacity=64)
    ga = {"plain": make_group(wa, False), "dueling": make_group(wa, True)}
    obs = torch.randint(-1, 20, (768, 96), device="cuda").float()
    obs[:, D:] = 0
    adraws = torch.zeros((args.warmup + args.steps, 1), device="cuda")
    for g in ga.values():
        for _ in range(args.warmup):
            g.act(obs)
    act = alternate({k: act_only(g, obs) for k, g in ga.items()}, adraws, args)

    out = {
        "what": "dueling Q-networks: learn sweeps and act with dueling heads against the plain head",
        "workload": f"cfg3: {CFG3['agents']} agents, batch {CFG3['batch']}, hidden [256,256], obs 89, actions 4, capacity "
                    f"{CFG3['capacity']} (rings full, 5 % done), independent networks, precision {precision}; cfg2: "
                    f"{CFG2['agents']} agents, batch {CFG2['batch']}, one CUDA graph replay per sweep; act: 768 agents, "
                    "hidden 256, greedy",
        "card": card(),
        "method": f"{args.rounds} alternating rounds x {args.steps} timed calls after {args.warmup} warm-up calls, CUDA "
                  "events",
        "cfg3_sweep_us": cfg3,
        "cfg3_sweep_extra_us": cfg3["dueling"]["median"] - cfg3["plain"]["median"],
        "cfg3_stage_us": per_stage,
        "cfg3_stage_extra_us": {s: per_stage["dueling"][s] - per_stage["plain"][s] for s in STAGES},
        "stage_method": "each stage of dmdqn_learn_stages as its own call, CUDA events between the calls (no chaining, so "
                        "the stages add up to more than the chained sweep); median over the rounds of the mean per sweep",
        "fold_kernel_us_cfg3": fold,
        "fold_method": "torch.profiler device time of fold_kernel in dueling learn sweeps (a pass of its own)",
        "fold_bytes_cfg3": 2 * 256 * (5 * 256 + 5 + 4 * 256 + 4) * 4,
        "cfg2_graph_sweep_us": cfg2,
        "cfg2_sweep_extra_us": cfg2["dueling"]["median"] - cfg2["plain"]["median"],
        "act_768_us": act,
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
