"""Cost of the sample kernel's variants at cfg3 (256 agents, batch 256, hidden [256, 256], capacity 30 000) on one GPU:
uniform (fisher_yates) draws at n_step 1, 3 and 8, and prioritized replay at n_step 1 and 3.

Five groups with the same seeded rings (5 % of the transitions done; spread-out priorities on the prioritized ones) and
weights run device-resident learn sweeps alternately in one process: ``--rounds`` rounds of ``--steps`` timed sweeps
after ``--warmup`` untimed ones, CUDA events around each run of sweeps.  The sample stage alone (dmdqn_learn_stages with
the sample bit only) is timed the same way.  The card's name, power limit and maximum SM clock are read in the same run.
Prints one JSON object; ``--out FILE`` also writes it there.  Only the API of AgentGroup and dmdqn_learn_stages is used,
so the script also times older trees of this project.

    python tools/sample_bench.py --out profiles/r05_sample_cfg3.json
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

import torch  # noqa: E402

from dmdqn_b200 import _native as N  # noqa: E402
from dmdqn_b200.group import AgentGroup  # noqa: E402

D, A = 89, 4
CFG3 = dict(agents=256, batch=256, hidden=256, capacity=30000)
VARIANTS = {"uniform_n1": ("fisher_yates", 1), "uniform_n3": ("fisher_yates", 3), "uniform_n8": ("fisher_yates", 8),
            "prioritized_n1": ("prioritized", 1), "prioritized_n3": ("prioritized", 3)}


def card():
    """Name and power limit of the current device (nvidia-smi, read only)."""
    idx = torch.cuda.current_device()
    out = {"name": torch.cuda.get_device_name(idx)}
    try:
        q = subprocess.run(["nvidia-smi", f"--id={idx}", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        name, limit, clk = (v.strip() for v in q.stdout.strip().split(","))
        out.update(nvidia_smi_name=name, power_limit=limit, max_sm_clock=clk)
    except Exception as exc:                  # the timing is still valid; say why the limit is missing
        out["power_limit"] = f"unavailable ({exc})"
    return out


def make_group(sample_mode, n_step, w, seed):
    cfg = {"nn_layers": [w["hidden"], w["hidden"]], "replay_buffer_size": w["capacity"], "batch_size": w["batch"],
           "learning_rate": 5e-4, "target_update_frequency": 1000, "sample_mode": sample_mode, "n_step": n_step}
    grp = AgentGroup(w["agents"], cfg, D, A, seed=seed)
    n, cap = grp.n_agents, grp.capacity
    gen = torch.Generator(device=grp.device).manual_seed(seed)
    grp.obs[:, :, :D] = torch.randint(-1, 20, (n, cap, D), device=grp.device, generator=gen).float()
    grp.next_obs[:, :, :D] = torch.randint(-1, 20, (n, cap, D), device=grp.device, generator=gen).float()
    grp.act_ring.copy_(torch.randint(0, A, (n, cap), device=grp.device, generator=gen).int())
    grp.rew_ring.copy_(-torch.randint(0, 5000, (n, cap), device=grp.device, generator=gen).double() * 0.7)
    grp.done_ring.copy_((torch.rand((n, cap), device=grp.device, generator=gen) < 0.05).to(torch.uint8))
    grp.n_written.fill_(cap); grp.n_written_host[:] = cap
    if grp.priority is not None:              # a ring that has been learning a while: spread-out priorities
        grp.priority.copy_(torch.rand((n, cap), device=grp.device, generator=gen) * 2 + 0.01)
        grp.priority_max.copy_(grp.priority.max(1).values)
    return grp


def timed(fn, draws, start):
    stream = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(draws.shape[0] - start):
        fn(draws[start + i])
    e1.record(stream)
    e1.synchronize()
    return e0.elapsed_time(e1) / (draws.shape[0] - start) * 1e3        # us per sweep


def sample_only(grp):
    def run(d):
        N.check(grp.lib.dmdqn_learn_stages(C.byref(grp.dims), C.byref(grp.hp), C.byref(grp.replay), C.byref(grp.nets),
                                           d.data_ptr(), None, grp.metrics.data_ptr(), grp.workspace.data_ptr(),
                                           grp.workspace.numel(), 1,          # DMDQN_STAGE_SAMPLE
                                           torch.cuda.current_stream().cuda_stream))
    return run


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sample_bench.py measures on a CUDA device; none is visible")
    w = CFG3
    groups = {k: make_group(mode, n, w, 11) for k, (mode, n) in VARIANTS.items()}
    draws = groups["uniform_n1"].draw_words((args.warmup + args.steps, w["agents"], w["batch"]))
    sweep = {k: [] for k in groups}
    sample = {k: [] for k in groups}
    for g in groups.values():                 # warm-up of every shape the timed runs use
        for i in range(args.warmup):
            g.learn(draws[i])
            sample_only(g)(draws[i])
    torch.cuda.synchronize()
    for _ in range(args.rounds):              # alternate the groups: drift of the shared host hits them all alike
        for k, g in groups.items():
            sweep[k].append(timed(lambda d, g=g: g.learn(d), draws, args.warmup))
        for k, g in groups.items():
            sample[k].append(timed(sample_only(g), draws, args.warmup))
    for g in groups.values():
        g.check_errors()
    med = {k: statistics.median(v) for k, v in sweep.items()}
    med_s = {k: statistics.median(v) for k, v in sample.items()}
    out = {
        "what": "sample kernel variants: device-resident learn sweeps (dmdqn_learn: sample + K3 + K4a + K4b for every "
                "network), and the sample kernel alone",
        "workload": f"cfg3: {w['agents']} agents, batch {w['batch']}, hidden [{w['hidden']},{w['hidden']}], obs 89, actions 4, "
                    f"replay capacity {w['capacity']} (rings full, 5 % done), independent networks, precision "
                    f"{list(N.PRECISION)[groups['uniform_n1'].hp.precision]}",
        "card": card(),
        "method": f"{args.rounds} alternating rounds x {args.steps} timed sweeps after {args.warmup} warm-up sweeps, CUDA "
                  "events; the ring (5.9 GB per group) is far larger than L2",
        "sweep_us": {k: {"median": med[k], "rounds": v} for k, v in sweep.items()},
        "sample_stage_us": {k: {"median": med_s[k], "rounds": v} for k, v in sample.items()},
        "sweep_over_uniform_n1": {k: med[k] / med["uniform_n1"] for k in groups if k != "uniform_n1"},
        "sample_extra_us": {k: med_s[k] - med_s["uniform_n1"] for k in groups if k != "uniform_n1"},
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
