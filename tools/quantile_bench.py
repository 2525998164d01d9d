"""Cost of quantile regression DQN (config ``quantile``, QR-DQN with 50 quantiles) on one GPU, against C51 (51 atoms)
and the plain network.

* cfg3 (256 agents, batch 256, hidden [256, 256], capacity 30 000, full rings): device-resident learn sweeps alternated in
  one process, ``--rounds`` rounds of ``--steps`` timed sweeps after ``--warmup`` untimed ones, CUDA events around each run
  of sweeps: fp32 plain ``dmdqn_learn``, C51 (``dmdqn_learn_grads_dist`` + ``dmdqn_adam_apply_dist``) and QR-DQN
  (``dmdqn_learn_grads_quantile`` + ``dmdqn_adam_apply_dist``), all fp32.
* cfg2 (16 agents, batch 64) the same three sweeps, each sweep one CUDA graph replay.
* Each kernel of the quantile step alone at cfg3, and the C51 target / online kernels for comparison: device time from
  ``torch.profiler`` over ``--steps`` sweeps (passes of their own).
* ``dmdqn_act``, ``dmdqn_act_dist`` and ``dmdqn_act_quantile`` on 768 agents (greedy, hidden 256).

The card's name, power limit and maximum SM clock are read in the same run.  Prints one JSON object; ``--out FILE`` also
writes it there.

    python tools/quantile_bench.py --out profiles/r10_quantile_cfg3.json
"""
from __future__ import annotations

import argparse
import json
import os
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

import torch  # noqa: E402

from tools.dueling_bench import alternate, make_group  # noqa: E402
from tools.noisy_bench import kernel_us  # noqa: E402
from tools.sample_bench import card  # noqa: E402

D, A, ATOMS, QUANTILES = 89, 4, 51, 50
CFG3 = dict(agents=256, batch=256, hidden=256, capacity=30000)
CFG2 = dict(agents=16, batch=64, hidden=256, capacity=30000)
KERNELS = ("quantile_target_kernel", "quantile_online_kernel", "dist_wgrad_kernel", "adam_apply_kernel")
C51_KERNELS = ("dist_target_kernel", "dist_online_kernel")


def group(w, seed=11, **extra):
    """make_group's rings and trunk in a group built with ``extra`` config keys."""
    from dmdqn_b200.group import AgentGroup
    plain = make_group(w, False, seed)
    cfg = dict(plain.config, precision="auto")
    cfg.update(extra)
    grp = AgentGroup(w["agents"], cfg, D, A, seed=seed)
    for name in ("obs", "next_obs", "act_ring", "rew_ring", "done_ring", "n_written"):
        getattr(grp, name).copy_(getattr(plain, name))
    grp.n_written_host[:] = plain.n_written_host
    del plain
    return grp


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("quantile_bench.py measures on a CUDA device; none is visible")

    g3 = {"fp32_learn": group(CFG3, precision="fp32"), "c51": group(CFG3, distributional=True, num_atoms=ATOMS),
          "quantile": group(CFG3, quantile=True, num_quantiles=QUANTILES)}
    draws = g3["quantile"].draw_words((args.warmup + args.steps, CFG3["agents"], CFG3["batch"]))
    fns = {k: (lambda d, g=g: g.learn(d)) for k, g in g3.items()}
    for fn in fns.values():
        for i in range(args.warmup):
            fn(draws[i])
    cfg3 = alternate(fns, draws, args)
    kern = kernel_us(g3["quantile"], draws, args.warmup, KERNELS)
    kern_c51 = kernel_us(g3["c51"], draws, args.warmup, C51_KERNELS)
    for g in g3.values():
        g.check_errors()
    losses = g3["quantile"].metrics[:, 0].cpu()
    assert torch.isfinite(losses).all(), "non-finite quantile loss"
    del g3, draws, fns
    torch.cuda.empty_cache()

    g2 = {"fp32_learn": group(CFG2, precision="fp32"), "c51": group(CFG2, distributional=True, num_atoms=ATOMS),
          "quantile": group(CFG2, quantile=True, num_quantiles=QUANTILES)}
    replay = {k: g.capture_learn() for k, g in g2.items()}
    draws2 = g2["quantile"].draw_words((args.warmup + args.steps, CFG2["agents"], CFG2["batch"]))
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
    ga = {"plain": group(wa, precision="fp32"), "c51": group(wa, distributional=True, num_atoms=ATOMS),
          "quantile": group(wa, quantile=True, num_quantiles=QUANTILES)}
    obs = torch.randint(-1, 20, (768, 96), device="cuda").float()
    obs[:, D:] = 0
    adraws = torch.zeros((args.warmup + args.steps, 1), device="cuda")
    for g in ga.values():
        for _ in range(args.warmup):
            g.act(obs)
    act = alternate({k: (lambda _, g=g: g.act(obs)) for k, g in ga.items()}, adraws, args)

    out = {
        "what": "quantile regression DQN (QR-DQN, 50 quantiles, kappa 1): learn sweeps, its kernels, and act, against C51 "
                "(51 atoms) and the plain network",
        "workload": f"cfg3: {CFG3['agents']} agents, batch {CFG3['batch']}, hidden [256,256], obs 89, actions 4, capacity "
                    f"{CFG3['capacity']} (rings full, 5 % done), independent networks; cfg2: {CFG2['agents']} agents, batch "
                    f"{CFG2['batch']}, one CUDA graph replay per sweep; act: 768 agents, hidden 256, greedy",
        "card": card(),
        "method": f"{args.rounds} alternating rounds x {args.steps} timed calls after {args.warmup} warm-up calls, CUDA "
                  "events; kernels: torch.profiler device time in passes of their own",
        "quantile_pair_terms_per_sweep": CFG3["agents"] * CFG3["batch"] * QUANTILES * QUANTILES,
        "cfg3_sweep_us": cfg3,
        "cfg3_quantile_over": {k: cfg3["quantile"]["median"] / cfg3[k]["median"] for k in ("fp32_learn", "c51")},
        "cfg3_kernels": kern,
        "cfg3_c51_kernels": kern_c51,
        "cfg2_graph_sweep_us": cfg2,
        "cfg2_quantile_over": {k: cfg2["quantile"]["median"] / cfg2[k]["median"] for k in ("fp32_learn", "c51")},
        "act_768_us": act,
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
