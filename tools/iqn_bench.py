"""Cost of implicit quantile networks (config ``iqn`` at its defaults: N = N' = 8 sampled fractions, K = 32 policy midpoints,
64 cosine features) on one GPU, against QR-DQN (50 quantiles) and the plain network.

* cfg3 (256 agents, batch 256, hidden [256, 256], capacity 30 000, full rings): device-resident learn sweeps alternated in
  one process, ``--rounds`` rounds of ``--steps`` timed sweeps after ``--warmup`` untimed ones, CUDA events around each run
  of sweeps: fp32 plain ``dmdqn_learn``, QR-DQN (``dmdqn_learn_grads_quantile`` + ``dmdqn_adam_apply_dist``) and IQN
  (``dmdqn_learn_grads_iqn`` + ``dmdqn_adam_apply_iqn``), all fp32.
* Each kernel of the IQN step alone at cfg3: device time from ``torch.profiler`` over ``--steps`` sweeps (a pass of its
  own), with the multiply-adds each learn kernel does per sweep (counted from the shapes below) and its FFMA rate.
* cfg2 (16 agents, batch 64) the same three sweeps, each sweep one CUDA graph replay.
* ``dmdqn_act``, ``dmdqn_act_quantile`` and ``dmdqn_act_iqn`` on 768 agents (greedy, hidden 256).

The card's name, power limit and maximum SM clock are read in the same run.  Prints one JSON object; ``--out FILE`` also
writes it there.

    python tools/iqn_bench.py --out profiles/r11_iqn_cfg3.json
"""
from __future__ import annotations

import argparse
import json
import os
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

import torch  # noqa: E402

from tools.dueling_bench import alternate  # noqa: E402
from tools.noisy_bench import kernel_us  # noqa: E402
from tools.quantile_bench import CFG2, CFG3, D, group  # noqa: E402
from tools.sample_bench import card  # noqa: E402

QUANTILES = 50
N_TAU, N_TAU_P, K_POLICY, N_COS = 8, 8, 32, 64
KERNELS = ("iqn_target_kernel", "iqn_online_kernel", "iqn_wgrad_kernel", "adam_apply_kernel")


def macs(agents: int, batch: int, h: int, dp: int = 96, n: int = N_TAU, n_p: int = N_TAU_P, k: int = K_POLICY,
         n_cos: int = N_COS, bm: int = 64) -> dict:
    """Multiply-adds per learn sweep of each IQN kernel as the kernels run them (double DQN; layer 1 over the padded
    observation width dp, head 4 wide), and the plain step's work by DESIGN.md section 4's count (4M + H^2 + HA)."""
    rows = agents * batch
    tiles = agents * -(-batch // bm)
    per_pass = h * h + 4 * h                       # layer 2 and the head of one (row, fraction)
    target = rows * (2 * dp * h + k * per_pass + n_p * (n_cos * h + per_pass)) + tiles * k * n_cos * h
    online = rows * (dp * h + n * (n_cos * h + per_pass) + n * (h * h + 4 * h))   # forward, then dz = dh2 W2^T and the head
    wgrad = rows * (n * h * h + n * n_cos * h + dp * h)
    m = D * h + h * h + h * 4                     # DESIGN.md section 4: one forward of a sample, M = D*H + H*H + H*A
    return {"iqn_target_kernel": target, "iqn_online_kernel": online, "iqn_wgrad_kernel": wgrad,
            "total": target + online + wgrad, "plain_step": rows * (4 * m + h * h + h * 4)}


def iqn_group(w, **extra):
    return group(w, iqn=True, iqn_num_tau=N_TAU, iqn_num_tau_prime=N_TAU_P, iqn_num_policy_tau=K_POLICY,
                 iqn_embedding_dim=N_COS, **extra)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("iqn_bench.py measures on a CUDA device; none is visible")

    g3 = {"fp32_learn": group(CFG3, precision="fp32"), "quantile": group(CFG3, quantile=True, num_quantiles=QUANTILES),
          "iqn": iqn_group(CFG3)}
    draws = g3["iqn"].draw_words((args.warmup + args.steps, CFG3["agents"], CFG3["batch"]))
    fns = {k: (lambda d, g=g: g.learn(d)) for k, g in g3.items()}
    for fn in fns.values():
        for i in range(args.warmup):
            fn(draws[i])
    cfg3 = alternate(fns, draws, args)
    kern = kernel_us(g3["iqn"], draws, args.warmup, KERNELS)
    count = macs(CFG3["agents"], CFG3["batch"], CFG3["hidden"])
    rate = {k: 2 * count[k] / (kern[k]["median_us"] * 1e-6) / 1e12 for k in KERNELS[:3]}   # TFLOP/s, one FFMA = 2 flops
    for g in g3.values():
        g.check_errors()
    losses = g3["iqn"].metrics[:, 0].cpu()
    assert torch.isfinite(losses).all(), "non-finite IQN loss"
    del g3, draws, fns
    torch.cuda.empty_cache()

    g2 = {"fp32_learn": group(CFG2, precision="fp32"), "quantile": group(CFG2, quantile=True, num_quantiles=QUANTILES),
          "iqn": iqn_group(CFG2)}
    replay = {k: g.capture_learn() for k, g in g2.items()}
    draws2 = g2["iqn"].draw_words((args.warmup + args.steps, CFG2["agents"], CFG2["batch"]))
    fns2 = {k: (lambda d, fn=fn, buf=buf: (buf.copy_(d), fn())) for k, (fn, buf) in replay.items()}
    for fn in fns2.values():
        for i in range(args.warmup):
            fn(draws2[i])
    cfg2 = alternate(fns2, draws2, args)
    del g2, replay, draws2, fns2
    torch.cuda.empty_cache()

    wa = dict(agents=768, batch=64, hidden=256, capacity=64)
    ga = {"plain": group(wa, precision="fp32"), "quantile": group(wa, quantile=True, num_quantiles=QUANTILES),
          "iqn": iqn_group(wa)}
    obs = torch.randint(-1, 20, (768, 96), device="cuda").float()
    obs[:, D:] = 0
    adraws = torch.zeros((args.warmup + args.steps, 1), device="cuda")
    for g in ga.values():
        for _ in range(args.warmup):
            g.act(obs)
    act = alternate({k: (lambda _, g=g: g.act(obs)) for k, g in ga.items()}, adraws, args)

    out = {
        "what": f"implicit quantile networks (IQN, N = N' = {N_TAU}, K = {K_POLICY}, n_cos = {N_COS}, kappa 1): learn sweeps, "
                "its kernels, and act, against QR-DQN (50 quantiles) and the plain network",
        "workload": f"cfg3: {CFG3['agents']} agents, batch {CFG3['batch']}, hidden [256,256], obs 89, actions 4, capacity "
                    f"{CFG3['capacity']} (rings full, 5 % done), independent networks; cfg2: {CFG2['agents']} agents, batch "
                    f"{CFG2['batch']}, one CUDA graph replay per sweep; act: 768 agents, hidden 256, greedy",
        "card": card(),
        "method": f"{args.rounds} alternating rounds x {args.steps} timed calls after {args.warmup} warm-up calls, CUDA "
                  "events; kernels: torch.profiler device time in a pass of its own",
        "cfg3_macs_per_sweep": count,
        "cfg3_sweep_us": cfg3,
        "cfg3_iqn_over": {k: cfg3["iqn"]["median"] / cfg3[k]["median"] for k in ("fp32_learn", "quantile")},
        "cfg3_kernels": kern,
        "cfg3_kernel_ffma_tflops": rate,
        "cfg2_graph_sweep_us": cfg2,
        "act_768_us": act,
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
