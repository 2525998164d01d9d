"""Cost of global-norm gradient clipping (config ``global_clipnorm``: dmdqn_learn_grads + dmdqn_clip_adam_apply) on one GPU.

* cfg3 (256 agents, batch 256, hidden [256, 256], capacity 30 000, full rings): device-resident learn sweeps of three
  groups with the same seeded rings and weights, alternated in one process: the unclipped ``dmdqn_learn``, clipping
  where every network clips (c = 1e-6), and clipping where none does (c = 1e30).  ``--rounds`` rounds of ``--steps``
  timed sweeps after ``--warmup`` untimed ones, CUDA events around each run of sweeps.
* cfg2 (16 agents, batch 64) the same way, each sweep one CUDA graph replay (``capture_learn``): there the extra launch
  counts.
* The clip kernel alone at cfg3 (``dmdqn_clip_adam_apply`` on the last step's gradient block), its time and its rate on
  its algorithmic bytes: per network the gradient read once, theta / m / v read and written, 28 bytes per parameter of
  the block [0, b3 + 4) (no target sync in the timed window: target_update_frequency is 1000).

The card's name, power limit and maximum SM clock are read in the same run.  Prints one JSON object; ``--out FILE`` also
writes it there.

    python tools/clip_bench.py --out profiles/r06_clip_cfg3.json
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
from tools.sample_bench import card, make_group, timed  # noqa: E402

CFG3 = dict(agents=256, batch=256, hidden=256, capacity=30000)
CFG2 = dict(agents=16, batch=64, hidden=256, capacity=30000)
VARIANTS = {"unclipped": None, "clip_every_network": 1e-6, "clip_no_network": 1e30}


def groups_for(w):
    out = {}
    for k, c in VARIANTS.items():
        g = make_group("fisher_yates", 1, w, 11)
        g.global_clipnorm = c
        if c is not None:
            g.grads = torch.zeros_like(g.theta)
            g.grad_norms = torch.zeros((g.n_nets,), dtype=torch.float32, device=g.device)
        out[k] = g
    return out


def clip_only(grp):
    def run(_):
        N.check(grp.lib.dmdqn_clip_adam_apply(C.byref(grp.dims), C.byref(grp.hp), C.byref(grp.nets), grp.grads.data_ptr(),
                                              grp.global_clipnorm, grp.grad_norms.data_ptr(), grp.workspace.data_ptr(),
                                              grp.workspace.numel(), torch.cuda.current_stream().cuda_stream))
    return run


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


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("clip_bench.py measures on a CUDA device; none is visible")
    g3 = groups_for(CFG3)
    draws = g3["unclipped"].draw_words((args.warmup + args.steps, CFG3["agents"], CFG3["batch"]))
    cfg3 = sweeps(g3, draws, args)
    clip_us = []
    grp = g3["clip_every_network"]
    for _ in range(args.rounds):
        clip_us.append(timed(clip_only(grp), draws, args.warmup))
    grp.check_errors()
    norms = grp.grad_norms.cpu()
    p_block = int(grp.layout.b3) + 4
    clip_bytes = 28 * p_block * grp.n_nets
    clip_med = statistics.median(clip_us)
    del g3, draws, grp
    torch.cuda.empty_cache()

    g2 = groups_for(CFG2)
    replay = {k: g.capture_learn() for k, g in g2.items()}       # (replay, draws buffer)
    draws2 = g2["unclipped"].draw_words((args.warmup + args.steps, CFG2["agents"], CFG2["batch"]))
    cfg2 = sweeps(g2, draws2, args, replay)

    base3, base2 = cfg3["unclipped"]["median"], cfg2["unclipped"]["median"]
    out = {
        "what": "global-norm gradient clipping: learn sweeps with dmdqn_learn_grads + dmdqn_clip_adam_apply against the "
                "unclipped dmdqn_learn, and the clip kernel alone",
        "workload": f"cfg3: {CFG3['agents']} agents, batch {CFG3['batch']}, hidden [256,256], obs 89, actions 4, capacity "
                    f"{CFG3['capacity']} (rings full, 5 % done), independent networks, precision "
                    f"{list(N.PRECISION)[g2['unclipped'].hp.precision]}; cfg2: {CFG2['agents']} agents, batch {CFG2['batch']}, "
                    "one CUDA graph replay per sweep",
        "card": card(),
        "method": f"{args.rounds} alternating rounds x {args.steps} timed sweeps after {args.warmup} warm-up sweeps, CUDA "
                  "events; theta, m, v and the gradient block are 94 MB each at cfg3, 376 MB together, far more than L2",
        "cfg3_sweep_us": cfg3,
        "cfg2_graph_sweep_us": cfg2,
        "cfg3_sweep_extra_us": {k: cfg3[k]["median"] - base3 for k in VARIANTS if k != "unclipped"},
        "cfg2_sweep_extra_us": {k: cfg2[k]["median"] - base2 for k in VARIANTS if k != "unclipped"},
        "clip_kernel_cfg3": {"us": {"median": clip_med, "rounds": clip_us}, "algorithmic_bytes": clip_bytes,
                             "tb_per_s": clip_bytes / (clip_med * 1e-6) / 1e12,
                             "bytes_rule": "28 per parameter of [0, b3 + 4): gradient read, theta / m / v read and written",
                             "block_floats": p_block, "median_norm": float(norms.median())},
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
