"""Cost of Rainbow networks (config ``rainbow``: C51 with 51 atoms, dueling streams, noisy layers) on one GPU.

* cfg3 (256 agents, batch 256, hidden [256, 256], capacity 30 000, full rings): device-resident learn sweeps alternated in
  one process, ``--rounds`` rounds of ``--steps`` timed sweeps after ``--warmup`` untimed ones, CUDA events around each run
  of sweeps: Rainbow (``dmdqn_learn_grads_rainbow`` + ``dmdqn_adam_apply_rainbow``), C51 (``dmdqn_learn_grads_dist`` +
  ``dmdqn_adam_apply_dist``) and fp32 plain ``dmdqn_learn``.
* Each kernel of the Rainbow and C51 steps alone at cfg3: device time from ``torch.profiler`` over ``--steps`` sweeps (a
  pass of its own), with the bytes the HBM-bound new kernels must move and the rate that gives.
* cfg2 (16 agents, batch 64) the same three steps, each sweep one CUDA graph replay.
* ``dmdqn_act_rainbow`` (noisy, and greedy on mu) against ``dmdqn_act_dist`` on 768 agents (hidden 256).

The card's name, power limit and maximum SM clock are read in the same run.  Prints one JSON object; ``--out FILE`` also
writes it there.

    python tools/rainbow_bench.py --out profiles/r12_rainbow_cfg3.json
"""
from __future__ import annotations

import argparse
import json
import os
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

import torch  # noqa: E402

from tools.dist_bench import group  # noqa: E402
from tools.dueling_bench import alternate  # noqa: E402
from tools.noisy_bench import kernel_us  # noqa: E402
from tools.sample_bench import card  # noqa: E402

D, A, ATOMS = 89, 4, 51
CFG3 = dict(agents=256, batch=256, hidden=256, capacity=30000)
CFG2 = dict(agents=16, batch=64, hidden=256, capacity=30000)
RAINBOW_KERNELS = ("noisy_fold_kernel", "head_fold_kernel", "rainbow_target_kernel", "rainbow_online_kernel",
                   "dist_wgrad_kernel", "rainbow_project_kernel", "noisy_adam_apply_kernel")
DIST_KERNELS = ("dist_target_kernel", "dist_online_kernel", "dist_wgrad_kernel", "adam_apply_kernel")


def hbm_bytes(grp):
    """Bytes each HBM-bound Rainbow kernel has to move per sweep (every network learning)."""
    L, n, h = grp.layout, grp.n_nets, grp.hidden
    npad = grp.atom_stride
    rows, nh = h + 1, 4 * npad
    return {
        "noisy_fold_kernel": 2 * n * L.stride * 12,                               # per set: mu + sigma read, eff written
        "head_fold_kernel": 2 * n * rows * (nh + npad + nh) * 4,                  # per set: W3 | b3 and Wv | bv read, W3e written
        "rainbow_project_kernel": n * rows * (2 * nh + npad) * 4,                 # W3 | b3 read and written, Wv | bv written
        "noisy_adam_apply_kernel": n * L.end * 52,                                 # g; mu, m, v and sigma, m, v read and written
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rainbow_bench.py measures on a CUDA device; none is visible")

    g3 = {"rainbow": group(CFG3, rainbow=True, num_atoms=ATOMS), "dist": group(CFG3, distributional=True, num_atoms=ATOMS),
          "fp32_learn": group(CFG3, precision="fp32")}
    draws = g3["rainbow"].draw_words((args.warmup + args.steps, CFG3["agents"], CFG3["batch"]))
    fns = {k: (lambda d, g=g: g.learn(d)) for k, g in g3.items()}
    for fn in fns.values():
        for i in range(args.warmup):
            fn(draws[i])
    cfg3 = alternate(fns, draws, args)
    kern = kernel_us(g3["rainbow"], draws, args.warmup, RAINBOW_KERNELS)
    kern_dist = kernel_us(g3["dist"], draws, args.warmup, DIST_KERNELS)
    nbytes = hbm_bytes(g3["rainbow"])
    for name, b in nbytes.items():
        kern[name].update(bytes=b, tb_per_s=b / (kern[name]["median_us"] * 1e-6) / 1e12)
    for g in g3.values():
        g.check_errors()
    losses = g3["rainbow"].metrics[:, 0].cpu()
    assert torch.isfinite(losses).all(), "non-finite Rainbow loss"
    del g3, draws, fns
    torch.cuda.empty_cache()

    g2 = {"rainbow": group(CFG2, rainbow=True, num_atoms=ATOMS), "dist": group(CFG2, distributional=True, num_atoms=ATOMS),
          "fp32_learn": group(CFG2, precision="fp32")}
    replay = {k: g.capture_learn() for k, g in g2.items()}
    draws2 = g2["rainbow"].draw_words((args.warmup + args.steps, CFG2["agents"], CFG2["batch"]))
    fns2 = {k: (lambda d, fn=fn, buf=buf: (buf.copy_(d), fn())) for k, (fn, buf) in replay.items()}
    for fn in fns2.values():
        for i in range(args.warmup):
            fn(draws2[i])
    cfg2 = alternate(fns2, draws2, args)
    for g in g2.values():
        g.check_errors()
    del g2, replay, draws2, fns2
    torch.cuda.empty_cache()

    wa = dict(agents=768, batch=64, hidden=256, capacity=64)
    ga = {"rainbow": group(wa, rainbow=True, num_atoms=ATOMS), "dist": group(wa, distributional=True, num_atoms=ATOMS)}
    obs = torch.randint(-1, 20, (768, 96), device="cuda").float()
    obs[:, D:] = 0
    adraws = torch.zeros((args.warmup + args.steps, 1), device="cuda")
    acts = {"rainbow_noisy": lambda _: ga["rainbow"].act(obs), "rainbow_greedy_mu": lambda _: ga["rainbow"].act(obs, noisy=False),
            "dist": lambda _: ga["dist"].act(obs)}
    for fn in acts.values():
        for _ in range(args.warmup):
            fn(None)
    act = alternate(acts, adraws, args)

    out = {
        "what": "Rainbow (C51 with 51 atoms, dueling streams, noisy layers): learn sweeps, its kernels, and act, against C51 "
                "and the plain fp32 network",
        "workload": f"cfg3: {CFG3['agents']} agents, batch {CFG3['batch']}, hidden [256,256], obs 89, actions 4, capacity "
                    f"{CFG3['capacity']} (rings full, 5 % done), independent networks; cfg2: {CFG2['agents']} agents, batch "
                    f"{CFG2['batch']}, one CUDA graph replay per sweep; act: 768 agents, hidden 256, greedy (noisy or mu)",
        "card": card(),
        "method": f"{args.rounds} alternating rounds x {args.steps} timed calls after {args.warmup} warm-up calls, CUDA "
                  "events; kernels: torch.profiler device time in a pass of its own; bytes counted from the layout",
        "cfg3_sweep_us": cfg3,
        "cfg3_rainbow_over": {k: cfg3["rainbow"]["median"] / cfg3[k]["median"] for k in ("dist", "fp32_learn")},
        "cfg3_rainbow_kernels": kern,
        "cfg3_dist_kernels": kern_dist,
        "cfg2_graph_sweep_us": cfg2,
        "cfg2_rainbow_over_dist": cfg2["rainbow"]["median"] / cfg2["dist"]["median"],
        "act_768_us": act,
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
