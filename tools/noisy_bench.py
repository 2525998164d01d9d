"""Cost of noisy networks (config ``noisy``) on one GPU.

* cfg3 (256 agents, batch 256, hidden [256, 256], capacity 30 000, full rings, precision tf32x3): device-resident learn
  sweeps alternated in one process, ``--rounds`` rounds of ``--steps`` timed sweeps after ``--warmup`` untimed ones, CUDA
  events around each run of sweeps: plain ``dmdqn_learn``, plain ``dmdqn_learn_grads`` + ``dmdqn_adam_apply`` (the same
  two-call split without noise), and the noisy step (``dmdqn_learn_grads_noisy`` + ``dmdqn_noisy_adam_apply``).
* cfg2 (16 agents, batch 64) the same way, each sweep one CUDA graph replay (``capture_learn``).
* The fold kernel and the noisy Adam kernel alone at cfg3: device time from ``torch.profiler`` over ``--steps`` noisy sweeps
  (a pass of its own), and the achieved rate on their algorithmic bytes (fold: mu and sigma read, eff written, for both
  sets; Adam: g read, theta / m / v of mu and of sigma read and written; the target copy, every 1000 steps here, is left out).
* ``dmdqn_act`` against ``dmdqn_act_noisy`` on 768 agents (greedy, hidden 256): 4P against 8P weight bytes per action.

The card's name, power limit and maximum SM clock are read in the same run.  Prints one JSON object; ``--out FILE`` also
writes it there.

    python tools/noisy_bench.py --out profiles/r08_noisy_cfg3.json
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
from tools.dueling_bench import alternate, make_group  # noqa: E402
from tools.sample_bench import card, timed  # noqa: E402

D, A = 89, 4
CFG3 = dict(agents=256, batch=256, hidden=256, capacity=30000)
CFG2 = dict(agents=16, batch=64, hidden=256, capacity=30000)


def noisy_group(w, seed=11):
    """make_group's rings and trunk with the noisy blocks allocated (make_group's groups are plain)."""
    from dmdqn_b200.group import AgentGroup
    plain = make_group(w, False, seed)
    cfg = dict(plain.config, noisy=True, precision=list(N.PRECISION)[plain.hp.precision])
    grp = AgentGroup(w["agents"], cfg, D, A, seed=seed)
    for name in ("obs", "next_obs", "act_ring", "rew_ring", "done_ring", "n_written"):
        getattr(grp, name).copy_(getattr(plain, name))
    grp.n_written_host[:] = plain.n_written_host
    del plain
    return grp


def grads_then_adam(grp, grads):
    """Plain dmdqn_learn_grads + dmdqn_adam_apply on one stream: the two-call split the noisy step also has."""
    def run(d):
        s = torch.cuda.current_stream().cuda_stream
        ws, nws = grp.workspace.data_ptr(), grp.workspace.numel()
        N.check(grp.lib.dmdqn_learn_grads(C.byref(grp.dims), C.byref(grp.hp), C.byref(grp.replay), C.byref(grp.nets),
                                          d.data_ptr(), None, grp.batch_size, grads.data_ptr(), grp.metrics.data_ptr(), ws, nws, s))
        N.check(grp.lib.dmdqn_adam_apply(C.byref(grp.dims), C.byref(grp.hp), C.byref(grp.nets), grads.data_ptr(), ws, nws, s))
    return run


def kernel_us(grp, draws, start, names):
    """Median device time per launch of each named kernel over noisy learn sweeps, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(start, draws.shape[0]):
            grp.learn(draws[i])
        torch.cuda.synchronize()
    out = {}
    for name in names:
        times = [e.device_time for e in prof.events() if name in e.name]
        if not times:
            raise RuntimeError(f"torch.profiler recorded no {name} launch")
        out[name] = {"median_us": statistics.median(times), "launches": len(times)}
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("noisy_bench.py measures on a CUDA device; none is visible")

    g3 = {"learn": make_group(CFG3, False), "grads_adam": make_group(CFG3, False), "noisy": noisy_group(CFG3)}
    grads = torch.zeros_like(g3["grads_adam"].theta)
    draws = g3["learn"].draw_words((args.warmup + args.steps, CFG3["agents"], CFG3["batch"]))
    fns = {"learn": lambda d: g3["learn"].learn(d), "grads_adam": grads_then_adam(g3["grads_adam"], grads),
           "noisy": lambda d: g3["noisy"].learn(d)}
    for fn in fns.values():
        for i in range(args.warmup):
            fn(draws[i])
    cfg3 = alternate(fns, draws, args)
    kern = kernel_us(g3["noisy"], draws, args.warmup, ("noisy_fold_kernel", "noisy_adam_apply_kernel"))
    for g in g3.values():
        g.check_errors()
    gn = g3["noisy"]
    stride, end, nets = int(gn.layout.stride), int(gn.layout.b3) + 4, gn.n_nets
    fold_bytes = nets * 2 * stride * 12
    adam_bytes = nets * end * 4 * 13
    kern["noisy_fold_kernel"].update(bytes=fold_bytes, gbps=fold_bytes / kern["noisy_fold_kernel"]["median_us"] / 1e3)
    kern["noisy_adam_apply_kernel"].update(bytes=adam_bytes, gbps=adam_bytes / kern["noisy_adam_apply_kernel"]["median_us"] / 1e3)
    precision = list(N.PRECISION)[g3["learn"].hp.precision]
    del g3, draws, grads, fns
    torch.cuda.empty_cache()

    g2 = {"learn": make_group(CFG2, False), "noisy": noisy_group(CFG2)}
    replay = {k: g.capture_learn() for k, g in g2.items()}
    draws2 = g2["learn"].draw_words((args.warmup + args.steps, CFG2["agents"], CFG2["batch"]))
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
    ga = {"plain": make_group(wa, False), "noisy": noisy_group(wa)}
    obs = torch.randint(-1, 20, (768, 96), device="cuda").float()
    obs[:, D:] = 0
    adraws = torch.zeros((args.warmup + args.steps, 1), device="cuda")
    for g in ga.values():
        for _ in range(args.warmup):
            g.act(obs)
    act = alternate({k: (lambda _, g=g: g.act(obs)) for k, g in ga.items()}, adraws, args)
    p_bytes = int(ga["plain"].layout.b3 + 4) * 4
    act_bytes = {"plain": 768 * p_bytes, "noisy": 768 * 2 * p_bytes}

    out = {
        "what": "noisy networks: learn sweeps, the fold and noisy Adam kernels, and act, against the plain network",
        "workload": f"cfg3: {CFG3['agents']} agents, batch {CFG3['batch']}, hidden [256,256], obs 89, actions 4, capacity "
                    f"{CFG3['capacity']} (rings full, 5 % done), independent networks, precision {precision}; cfg2: "
                    f"{CFG2['agents']} agents, batch {CFG2['batch']}, one CUDA graph replay per sweep; act: 768 agents, "
                    "hidden 256, greedy",
        "card": card(),
        "method": f"{args.rounds} alternating rounds x {args.steps} timed calls after {args.warmup} warm-up calls, CUDA "
                  "events; kernels: torch.profiler device time in a pass of its own",
        "cfg3_sweep_us": cfg3,
        "cfg3_noisy_extra_us": {k: cfg3["noisy"]["median"] - cfg3[k]["median"] for k in ("learn", "grads_adam")},
        "cfg3_kernels": kern,
        "cfg2_graph_sweep_us": cfg2,
        "cfg2_noisy_extra_us": cfg2["noisy"]["median"] - cfg2["learn"]["median"],
        "act_768_us": act,
        "act_weight_bytes": act_bytes,
        "act_gbps": {k: act_bytes[k] / act[k]["median"] / 1e3 for k in act},
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
