#!/usr/bin/env python
"""bench.py -- agent-updates/s of the Double-DQN learn step (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload cfg3] [--dump-outputs DIR]

A "step" is one learn sweep: every agent of the workload runs one ``learn()`` (sample B
transitions from its ring, target + online forward, backward, Adam, target sync).
Workloads (BASELINE.json configs; synthetic replay, observation-shaped integers, rings full):
  cfg2  16 agents,  B=64,  H=256      cfg3  256 agents, B=256, H=256  (default, per GPU)
  cfg4  512 agents, B=512, H=256 per GPU (4096 over 8 GPUs)
N>1 shards agents across ranks with no collective (independent networks): weak scaling,
every rank holds the per-GPU workload.  The same JSON line carries, under "blocks", the other configurations
BASELINE.json names: cfg3 strong-scaled (256 agents in total over the ranks), cfg4 (512 agents per GPU, batch 512)
and cfg5 (one shared network, hidden 512, global batch 1024, gradient reduction over the ranks); "act" is measured
on a working set larger than the L2.  One JSON line on stdout (rank 0).
--dump-outputs DIR writes what the last timed learn sweep left to its caller as DIR/<name>.npy (learn_outputs); every
input is seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import random
import statistics
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries exactly ONE JSON line.  Libraries write there too (NCCL prints "NCCL version ..." on stdout at
# init), so the real stdout is kept on a private descriptor for the result and fd 1 is pointed at stderr.
_JSON_FD = os.dup(1)
os.dup2(2, 1)


def emit(obj) -> None:
    os.write(_JSON_FD, (json.dumps(obj) + "\n").encode())

WORKLOADS = {
    "cfg2": dict(agents=16, batch=64, hidden=256, capacity=30000, grid="4x4"),
    "cfg3": dict(agents=256, batch=256, hidden=256, capacity=30000, grid="16x16"),
    "cfg4": dict(agents=512, batch=512, hidden=256, capacity=30000, grid="64x64 city grid / 8 GPUs"),
}
D, A = 89, 4


def workload_name(key):
    w = WORKLOADS[key]
    return (f"{key}: {w['agents']} agents/GPU ({w['grid']}), batch {w['batch']}, hidden [{w['hidden']},{w['hidden']}], obs 89, "
            f"actions 4, replay capacity {w['capacity']}, independent networks")


def agent_cfg(w, precision="fp32"):
    return {"learning_rate": 5e-4, "gamma": 0.99, "replay_buffer_size": w["capacity"], "batch_size": w["batch"],
            "target_update_frequency": 1000, "nn_layers": [w["hidden"], w["hidden"]],    # config/agent_config.yaml
            "precision": precision}


def flops_bytes(w):
    """Algorithmic work per agent-update (SURVEY.md section 8 D-roofline, DESIGN.md)."""
    b, h = w["batch"], w["hidden"]
    m = D * h + h * h + h * A
    p = m + h + h + A
    k = {"target": dict(flops=2 * 2 * b * m, bytes=b * (D + 2) * 4 + 8 * p),
         "online": dict(flops=2 * b * m + 2 * b * (h * h + h * A), bytes=b * (D + 1) * 4 + 4 * p),
         "wgrad_adam": dict(flops=2 * b * m, bytes=24 * p),      # theta, m, v read AND written back (theta_tgt on sync steps: +4P)
         "sample": dict(flops=0, bytes=b * 13 + b * 16)}
    return {"flops": 2 * b * (4 * m + h * h + h * A), "bytes": b * (2 * D + 3) * 4 + 24 * p, "params": p, "kernels": k}


# ------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """SM clock, power and throttle reasons sampled WHILE the timed region runs: NVML every 10 ms
    (nvidia_ml_py), or nvidia-smi every 200 ms when NVML cannot be loaded."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    NAMES = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt, self.how = index, [], threading.Event(), "nvidia-smi"
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.how = "nvml"
        except Exception:
            self.nv = None

    @staticmethod
    def _physical_index(local):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v for v in vis.split(",") if v.strip()]
            if local < len(ids) and ids[local].strip().isdigit():
                return int(ids[local])
        return local

    def _nvml_row(self):
        nv = self.nv
        bits = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
            else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        flags = (getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8), getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20), getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4))
        return [float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)), self.max_sm, nv.nvmlDeviceGetPowerUsage(self.h) / 1e3] + \
               ["Active" if bits & f else "Not Active" for f in flags]

    def run(self):
        import subprocess
        while not self._stop_evt.is_set():
            try:
                if self.nv is not None:
                    self.rows.append(self._nvml_row())
                else:
                    out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                    f = [x.strip() for x in out.strip().split(",")]
                    if len(f) >= 7:
                        self.rows.append(f)
            except Exception:
                pass
            self._stop_evt.wait(0.01 if self.nv is not None else 0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = [float(r[0]) for r in self.rows]
        reasons = [n for i, n in enumerate(self.NAMES, 3) if any(str(r[i]).lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": float(self.rows[0][1]), "samples": len(sm), "how": self.how,
                "power_w_max": max(float(r[2]) for r in self.rows), "reasons": reasons}


def ncu_traffic(workload, precision, kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed `ncu --set full`
    capture of this workload (profiles/ncu_traffic.json names the capture each figure comes from); None when
    this workload / precision has not been captured."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        return t[f"{workload}/{precision}"][kernel]["dram_bytes"]
    except Exception:
        return None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return {"hbm_gbs": j["hbm_gbs"], "bf16_tflops": j["bf16_tflops"], "bf16_tflops_sustained": j["bf16_tflops_sustained"],
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


# ------------------------------------------------------------------------------------------
def synth_fill(grp, seed):
    """Full rings of featuriser-shaped data: queue counts 0..19 as floats, -1 padding,
    rewards 0.3*local + 0.7*global (float64), dones ~ 1/240 (SURVEY.md D-inputs)."""
    n, c = grp.n_agents, grp.capacity
    gen = torch.Generator(device=grp.device).manual_seed(seed)
    chunk = max(1, (1 << 28) // (c * D))
    for a0 in range(0, n, chunk):
        a1 = min(n, a0 + chunk)
        for ring in (grp.obs, grp.next_obs):
            v = torch.randint(-1, 20, (a1 - a0, c, D), device=grp.device, generator=gen).float()
            ring[a0:a1, :, :D] = v
    grp.act_ring.copy_(torch.randint(0, A, (n, c), device=grp.device, generator=gen).int())
    loc = torch.randint(0, 240, (n, c), device=grp.device, generator=gen).double()
    glob = torch.randint(0, 240 * 256, (1, c), device=grp.device, generator=gen).double()
    grp.rew_ring.copy_(-0.3 * loc - 0.7 * glob)
    grp.done_ring.copy_((torch.rand((n, c), device=grp.device, generator=gen) < 1 / 240).to(torch.uint8))
    grp.n_written.fill_(c + 777)
    grp.n_written_host[:] = c + 777


DUMP_SAMPLE, DUMP_SEED, DUMP_LIMIT = 1 << 20, 0, 64 << 20


def learn_outputs(grp, metrics):
    """What a caller of AgentGroup.learn holds after the call: the metrics it returns ([G, 8] float32: loss, q mean, q std,
    action histogram, learned flag) and the network state it updated (online and target weights, Adam moments).  Those
    four are sampled at DUMP_SAMPLE positions drawn with DUMP_SEED from every network's parameters in AgentGroup.unpack's
    (Keras) order, layout padding left out: the same positions for the same workload, whatever the parameter layout."""
    logical = torch.cat([t.reshape(-1) for t in grp.unpack(torch.arange(grp.layout.stride, dtype=torch.float64))]).long()
    per_net = logical.numel()
    pick = np.sort(np.random.default_rng(DUMP_SEED).choice(grp.n_nets * per_net, min(grp.n_nets * per_net, DUMP_SAMPLE), replace=False))
    net, j = np.divmod(pick, per_net)
    flat = (torch.as_tensor(net) * grp.layout.stride + logical[torch.as_tensor(j)]).to(grp.device)
    out = {"metrics": metrics.cpu().numpy()}
    for name, t in (("theta", grp.theta), ("theta_target", grp.theta_tgt), ("adam_m", grp.adam_m), ("adam_v", grp.adam_v)):
        out[f"{name}_sample"] = t.reshape(-1)[flat].cpu().numpy()
    return out


def dump_outputs(path, arrays):
    os.makedirs(path, exist_ok=True)
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_LIMIT
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), a)


def _events(n):
    return [torch.cuda.Event(enable_timing=True) for _ in range(n)]


def _barrier(world):
    torch.cuda.synchronize()
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def _max_over_ranks(vals, world, device):
    if world == 1:
        return list(vals)
    import torch.distributed as dist
    t = torch.tensor(list(vals), device=device, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(x) for x in t]


def time_learn(grp, draws, K, W, world):
    """K learn sweeps after W warm-up sweeps: CUDA events on the launching stream, barrier + synchronize on both
    sides, max over ranks.  Returns ms for the K sweeps."""
    stream = torch.cuda.current_stream()
    for i in range(W):
        grp.learn(draws[i])
    _barrier(world)
    e0, e1 = _events(2)
    e0.record(stream)
    for i in range(K):
        grp.learn(draws[W + i])
    e1.record(stream)
    _barrier(world)
    return _max_over_ranks([e0.elapsed_time(e1)], world, grp.device)[0]


STAGE_NAMES = ["sample", "target", "online", "wgrad_adam"]


def roofline_of(kernel, kt, pk, precision, ffma_peak, runner_up=None):
    """The roof that binds `kernel`.  K4b (weight gradients + Adam) moves 24 bytes per parameter for 2 B M flops per network:
    its HBM floor (84 us at cfg3) is twice its tensor floor, so it is reported against the measured HBM rate; K3 / K4a are
    GEMM chains with almost no HBM traffic and are reported against the measured bf16 tensor rate (of which 3xTF32 can reach 1/6)."""
    e = kt[kernel]
    if kernel == "wgrad_adam":
        out = {"bound": "hbm", "kernel": kernel, "achieved": e["gbs"], "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": e["gbs"] / pk["hbm_gbs"],
               "traffic": e["traffic"], "algorithmic_bytes": e["algorithmic_bytes"], "peak_source": pk["source"],
               "note": "algorithmic bytes = 24 P per network (theta / m / v read and written) + the gathered rows; the same kernel against the "
                       f"tensor roof: {e['tflops']:.1f} TFLOP/s = {e['tflops'] / pk['bf16_tflops_sustained']:.3f} of the measured bf16 rate"}
    else:
        ach_tf = e["tflops"]
        out = {"bound": "tensor", "kernel": kernel, "achieved": ach_tf, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
               "frac": ach_tf / pk["bf16_tflops_sustained"], "traffic": e["traffic"], "algorithmic_bytes": e["algorithmic_bytes"],
               "peak_source": pk["source"], "frac_of_burst_peak": ach_tf / pk["bf16_tflops"],
               "note": (f"fp32 FFMA kernel: fraction of the fp32 FFMA peak at the sampled clock = {ach_tf / ffma_peak:.3f} of "
                        f"{ffma_peak:.1f} TFLOP/s") if precision == "fp32" else
                       ("tcgen05 kind::tf32; achieved counts ALGORITHMIC flops (each product is issued as "
                        f"{3 if precision == 'tf32x3' else 1} MMA(s)); peak is the measured bf16 figure (tf32 dense peak is half of it), so the "
                        f"ceiling of this precision is frac = {1 / (6 if precision == 'tf32x3' else 2):.3f}")}
    if runner_up and runner_up != kernel:
        r = roofline_of(runner_up, kt, pk, precision, ffma_peak)
        out["runner_up"] = {k: r[k] for k in ("bound", "kernel", "achieved", "peak", "unit", "frac")}
        out["runner_up"]["ms"] = kt[runner_up]["ms"]
    out["ms"] = e["ms"]
    return out


def _with_chain_note(roof, dom, kt, stage_ms, ms_step, pk):
    """`roof` describes the dominant kernel launched ALONE (one stage per call).  Inside dmdqn_learn the kernels overlap
    (programmatic dependent launches), so their durations cannot be separated by events; what can be stated is the step's
    time that is not covered by the other kernels' stand-alone durations -- an upper bound of the dominant kernel's exclusive
    share of the chained step -- and the rate of its algorithmic bytes / flops over that share."""
    others = sum(v for k, v in stage_ms.items() if k != dom)
    excl = ms_step - others
    if excl > 0 and excl < stage_ms[dom]:
        e = kt[dom]
        ach = (e["algorithmic_bytes"] / (excl / 1e3) / 1e9) if roof["bound"] == "hbm" else e["tflops"] * stage_ms[dom] / excl
        roof["in_chain"] = {"exclusive_ms": excl, "achieved": ach, "frac": ach / roof["peak"],
                            "note": "step time minus the other kernels' stand-alone durations: the part of the chained step only this kernel "
                                    "accounts for (its first CTAs run under the previous kernel's last round); derived, not a separate measurement"}
    return roof


def stage_times(grp, draws, K):
    """The same sweep issued one stage per call (dmdqn_learn_stages) with events in between: mean ms per kernel."""
    from dmdqn_b200 import _native as N
    import ctypes as C
    stream = torch.cuda.current_stream()
    evs = [_events(5) for _ in range(K)]
    for i in range(K):
        d = draws[i]
        for s in range(4):
            evs[i][s].record(stream)
            N.check(grp.lib.dmdqn_learn_stages(C.byref(grp.dims), C.byref(grp.hp), C.byref(grp.replay), C.byref(grp.nets),
                                               d.data_ptr(), None, grp.metrics.data_ptr(), grp.workspace.data_ptr(),
                                               grp.workspace.numel(), 1 << s, stream.cuda_stream))
        evs[i][4].record(stream)
    torch.cuda.synchronize()
    grp.learn_step_host += K
    return {nm: statistics.mean(evs[i][s].elapsed_time(evs[i][s + 1]) for i in range(K)) for s, nm in enumerate(STAGE_NAMES)}


def kernel_table(w, n, stage_ms, workload, precision):
    """Per kernel: duration, algorithmic flops / bytes per launch, achieved rates, ncu DRAM traffic per launch."""
    fb = flops_bytes(w)
    pk = peaks()
    out = {}
    for k_ in STAGE_NAMES:
        ms, kf = stage_ms[k_], fb["kernels"][k_]
        out[k_] = {"ms": ms, "tflops": n * kf["flops"] / (ms / 1e3) / 1e12, "algorithmic_bytes": n * kf["bytes"],
                   "gbs": n * kf["bytes"] / (ms / 1e3) / 1e9, "hbm_frac": n * kf["bytes"] / (ms / 1e3) / 1e9 / pk["hbm_gbs"],
                   "traffic": ncu_traffic(workload, precision, k_)}
    return out


def timed(fn, reps, stream):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b_ = _events(2)
    a.record(stream)
    for _ in range(reps):
        fn()
    b_.record(stream)
    torch.cuda.synchronize()
    return a.elapsed_time(b_) / reps


def graph_timed(fn, launches, replays, stream):
    """Device time of `fn` without the Python call overhead: `launches` calls captured in a CUDA graph, replayed."""
    side = torch.cuda.Stream()
    side.wait_stream(stream)
    with torch.cuda.stream(side):
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            for i in range(launches):
                fn(i)
        for _ in range(3):
            graph.replay()
        side.synchronize()
        a_, b_ = _events(2)
        a_.record(side)
        for _ in range(replays):
            graph.replay()
        b_.record(side)
        side.synchronize()
        ms = a_.elapsed_time(b_) / (replays * launches)
    stream.wait_stream(side)
    return ms


# ---- blocks: the other configurations north_star names, inside the same JSON line ---------------------------
def block_act(args, rank, world, local):
    """actions/s with a working set LARGER than the 126 MB L2: 768 agents x 4P bytes = 276 MB of weights are streamed
    per launch (cyclic access over 2.2x the L2 capacity: no reuse between launches), next to the 256-agent launch
    whose 92 MB stay L2-resident between replays (the figure round 1 reported)."""
    from dmdqn_b200.group import AgentGroup
    w = WORKLOADS["cfg3"]
    p = flops_bytes(w)["params"]
    stream = torch.cuda.current_stream()
    out = {}
    for tag, n in (("hbm_768_agents", 768), ("l2_resident_256_agents", 256)):
        grp = AgentGroup(n, dict(agent_cfg(w, args.precision), replay_buffer_size=4, batch_size=4), D, A, seed=7 + rank)
        obs = torch.randint(-1, 20, (n, D), device=grp.device).float()
        eps0 = torch.zeros(n, dtype=torch.float64, device=grp.device)
        wz = torch.zeros(n, dtype=torch.int32, device=grp.device)
        api_ms = timed(lambda: grp.act(obs, eps0, wz, wz), 200, stream)
        try:
            ms = graph_timed(lambda i: grp.act(obs, eps0, wz, wz), 16, 20, stream)
        except Exception as exc:                                                   # noqa: BLE001
            print(f"act graph timing unavailable ({exc}); reporting the API loop", file=sys.stderr)
            ms = api_ms
        ms = _max_over_ranks([ms], world, grp.device)[0]
        gbs = n * 4 * p / (ms / 1e3) / 1e9
        out[tag] = {"agents_per_gpu": n, "value": n * world / (ms / 1e3), "unit": "actions/s", "ms": ms, "api_ms": api_ms,
                    "weight_bytes_per_launch": n * 4 * p, "hbm_gbs": gbs, "hbm_frac": gbs / peaks()["hbm_gbs"]}
        del grp, obs
        torch.cuda.empty_cache()
    head = out["hbm_768_agents"]
    return {"value": head["value"], "unit": "actions/s", "ms": head["ms"], "eps": 0.0, "bytes_per_action": 4 * p,
            "hbm_gbs": head["hbm_gbs"], "hbm_frac": head["hbm_frac"],
            "timing": "16 launches captured in a CUDA graph, replayed 20x (device time); api_ms = the same call from Python; "
                      "eps = 0 so every agent runs its network",
            "cold_ncu_us_256_agents": (ncu_traffic("cfg3", args.precision, "act") and
                                       json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
                                       [f"cfg3/{args.precision}"]["act"]["ncu_duration_us"]),
            **out}


def block_cfg2(args, rank, world, local, K, W):
    """BASELINE cfg2: 16 agents (4x4 grid), batch 64 on one GPU -- a launch/latency-bound shape (each kernel runs one short item per
    CTA on 16-48 of the 148 SMs).  Measured twice: the plain dmdqn_learn call per step, and the step captured once as a CUDA graph
    (AgentGroup.capture_learn) and replayed.  Every rank runs its own copy; rank 0's numbers are reported."""
    from dmdqn_b200.group import AgentGroup
    w = WORKLOADS["cfg2"]
    grp = AgentGroup(w["agents"], agent_cfg(w, args.precision), D, A, seed=77)
    synth_fill(grp, seed=5)
    n, b = grp.n_agents, grp.batch_size
    draws = grp.draw_words((K + W, n, b))
    ms_plain = time_learn(grp, draws, K, W, world)
    replay, dbuf = grp.capture_learn()
    stream = torch.cuda.current_stream()
    for i in range(W):
        dbuf.copy_(draws[i]); replay()
    _barrier(world)
    e0, e1 = _events(2)
    e0.record(stream)
    for i in range(K):
        dbuf.copy_(draws[W + i]); replay()
    e1.record(stream)
    _barrier(world)
    ms_graph = e0.elapsed_time(e1)
    stage_ms = stage_times(grp, draws[W:], min(K, 20))
    grp.check_errors()
    del grp, draws
    torch.cuda.empty_cache()
    return {"workload": workload_name("cfg2"), "value": n * K / (ms_graph / 1e3), "unit": "agent-updates/s", "ms_per_step": ms_graph / K,
            "how": "one CUDA-graph replay per step (sample, K3, K4a, K4b captured once; the draws buffer refilled before each replay)",
            "plain_calls": {"value": n * K / (ms_plain / 1e3), "ms_per_step": ms_plain / K}, "steps": K,
            "kernels_ms_rank0": stage_ms}


def block_strong_cfg3(args, rank, world, local, K, W):
    """BASELINE cfg3 'then sharded 2/4/8': 256 agents in TOTAL, split by contiguous agent range over the ranks
    (parallel.shard_range), no collective.  value = 256 agents x steps / max-over-ranks time."""
    from dmdqn_b200.group import AgentGroup
    from dmdqn_b200.parallel import shard_range
    w = WORKLOADS["cfg3"]
    lo, hi = shard_range(w["agents"], world, rank)
    grp = AgentGroup(hi - lo, agent_cfg(w, args.precision), D, A, seed=1000 + lo)
    synth_fill(grp, seed=100 + rank)
    draws = grp.draw_words((K + W, grp.n_agents, grp.batch_size))
    ms = time_learn(grp, draws, K, W, world)
    st = stage_times(grp, draws[W:], min(K, 20))
    del grp
    torch.cuda.empty_cache()
    return {"workload": "cfg3 strong: 256 agents total, batch 256, hidden 256, agent ranges over the ranks, no collective",
            "agents_total": w["agents"], "agents_this_rank": hi - lo, "value": w["agents"] * K / (ms / 1e3),
            "unit": "agent-updates/s", "ms_per_step": ms / K, "scaling": "strong", "steps": K,
            "kernels_ms_rank0": st}


def block_cfg4(args, rank, world, local, K, W):
    """BASELINE cfg4: 4096 agents (64x64 city grid), batch 512, sharded 512 per GPU with no collective (weak: the
    per-GPU shard is the unit; 8 GPUs hold the whole grid)."""
    from dmdqn_b200.group import AgentGroup
    w = WORKLOADS["cfg4"]
    grp = AgentGroup(w["agents"], agent_cfg(w, args.precision), D, A, seed=5000 + 1000 * rank)
    synth_fill(grp, seed=200 + rank)
    draws = grp.draw_words((K + W, grp.n_agents, grp.batch_size))
    ms = time_learn(grp, draws, K, W, world)
    st = stage_times(grp, draws[W:], min(K, 10))
    fb = flops_bytes(w)
    n = grp.n_agents
    del grp
    torch.cuda.empty_cache()
    return {"workload": workload_name("cfg4"), "agents_total": n * world, "value": n * world * K / (ms / 1e3),
            "unit": "agent-updates/s", "ms_per_step": ms / K, "scaling": "weak", "steps": K,
            "tflops_per_gpu": n * fb["flops"] / (ms / K / 1e3) / 1e12, "kernels_ms_rank0": st}


def block_cfg5(args, rank, world, local, K, W):
    """BASELINE cfg5: ONE network (hidden 512) shared by 1024 agents; every learn step draws a global batch of 1024
    transitions, 1024/N per GPU from that GPU's rings (1024/N agents each), gradients summed over the ranks
    (parallel.SharedParameterStep: NCCL all-reduce of the 4P-byte block, or the fused peer-memory reduce + Adam
    when the library offers it), identical Adam on every replica.  value = shared updates/s x 1024 agents served
    (SURVEY.md section 8 D-inputs); raw updates/s and samples/s alongside."""
    from dmdqn_b200.group import AgentGroup
    from dmdqn_b200.parallel import SharedParameterStep
    import torch.distributed as dist
    agents_total, batch_global, hidden, cap = 1024, 1024, 512, 4096
    if agents_total % world or batch_global % world:
        return {"skipped": f"world size {world} does not divide 1024"}
    cfg = {"learning_rate": 5e-4, "gamma": 0.99, "replay_buffer_size": cap, "batch_size": batch_global // world,
           "target_update_frequency": 1000, "nn_layers": [hidden, hidden], "share_parameters": True, "precision": "auto"}
    grp = AgentGroup(agents_total // world, cfg, D, A, seed=42)            # same seed: replicas start identical
    synth_fill(grp, seed=300 + rank)
    fused_note = None
    try:
        step = SharedParameterStep.for_group(grp)                          # world > 1: fused peer-memory reduce + Adam
    except Exception as exc:                                               # CUDA IPC refused on this box: measure the NCCL path, say so
        fused_note = f"peer-memory exchange unavailable ({type(exc).__name__}: {str(exc)[:120]}): NCCL all_reduce path measured instead"
        step = SharedParameterStep.for_group(grp, fused=False)
    stream = torch.cuda.current_stream()

    def run_steps(st):
        for _ in range(W):
            st.step()
        _barrier(world)
        e0, e1 = _events(2)
        e0.record(stream)
        for _ in range(K):
            st.step()
        e1.record(stream)
        _barrier(world)
        return _max_over_ranks([e0.elapsed_time(e1)], world, grp.device)[0]
    ms = run_steps(step)
    ms_nccl = run_steps(SharedParameterStep.for_group(grp, fused=False)) if world > 1 else None
    # phase split of one step: local gradients | reduction | Adam
    ev = [_events(4) for _ in range(min(K, 20))]
    for e in ev:
        e[0].record(stream)
        grads, _ = step.local_grads(step.local_batch * world)
        e[1].record(stream)
        if world > 1:
            dist.all_reduce(grads)
        e[2].record(stream)
        step.apply(grads)
        e[3].record(stream)
    torch.cuda.synchronize()
    phases = {nm: statistics.mean(e[i].elapsed_time(e[i + 1]) for e in ev) for i, nm in enumerate(("local_grads", "allreduce", "adam"))}
    identical = True
    if world > 1:
        chk = grp.theta.double().sum().reshape(1)
        lo_, hi_ = chk.clone(), chk.clone()
        dist.all_reduce(lo_, op=dist.ReduceOp.MIN); dist.all_reduce(hi_, op=dist.ReduceOp.MAX)
        identical = bool((lo_ == hi_).item())
    p = hidden * D + hidden * hidden + hidden * A + 2 * hidden + A
    ups = K / (ms / 1e3)
    del grp
    torch.cuda.empty_cache()
    return {"workload": f"cfg5: one shared network, hidden [512,512], 1024 agents, global batch 1024 ({batch_global // world} per GPU), "
                        f"replay capacity {cap} per agent, gradient all-reduce of {4 * p} bytes",
            "value": ups * agents_total, "unit": "agent-updates/s (shared updates/s x 1024 agents served)",
            "shared_updates_per_s": ups, "samples_per_s": ups * batch_global, "ms_per_step": ms / K, "scaling": "strong",
            "steps": K, "phases_ms_rank0": phases, "replicas_identical": identical,
            "reduction": "none (1 GPU)" if world == 1 else (fused_note or "dmdqn_allreduce_adam: flag exchange + peer loads over NVLink (CUDA IPC) + Adam in one kernel"),
            "nccl_baseline": None if ms_nccl is None else {"ms_per_step": ms_nccl / K, "value": K / (ms_nccl / 1e3) * agents_total,
                                                          "what": "torch.distributed all_reduce (NCCL) between dmdqn_learn_grads and dmdqn_adam_apply; phases_ms_rank0 splits this path"}}


def block_gather_featurize(grp, world, K):
    """K1b's stand-alone gather (ReplayBuffer.sample's five tensors) and K0, with achieved GB/s on algorithmic bytes."""
    from dmdqn_b200.parallel import grid_neighbor_table
    stream = torch.cuda.current_stream()
    n, b = grp.n_agents, grp.batch_size
    draws = grp.draw_words((n, b))
    sample_ms = timed(lambda: grp.sample(draws), 30, stream)            # sample + gather + the output allocations
    # the gather kernel alone: the workspace already holds the sampled rows
    from dmdqn_b200 import _native as N
    import ctypes as C
    states = torch.zeros((n, b, D), device=grp.device); nxt = torch.zeros_like(states)
    acts = torch.zeros((n, b), dtype=torch.int32, device=grp.device); rew = torch.zeros((n, b), device=grp.device)
    dn = torch.zeros((n, b), device=grp.device)
    gather_ms = timed(lambda: N.check(grp.lib.dmdqn_gather(C.byref(grp.dims), C.byref(grp.replay), grp.workspace.data_ptr(),
                                                           grp.workspace.numel(), states.data_ptr(), acts.data_ptr(), rew.data_ptr(),
                                                           nxt.data_ptr(), dn.data_ptr(), None, stream.cuda_stream)), 50, stream)
    g_bytes = n * b * 724 * 2                                                # 724 B read + 724 B written per sampled transition
    halting = torch.randint(0, 20, (n, 12), dtype=torch.int32, device=grp.device)
    zi = torch.zeros(n, dtype=torch.int32, device=grp.device); zd = torch.zeros(n, dtype=torch.float64, device=grp.device)
    zv = torch.zeros(n, dtype=torch.uint8, device=grp.device)
    side = max(r for r in range(1, int(n ** 0.5) + 1) if n % r == 0)          # this GPU's shard of the grid: side x n/side
    nbr = torch.as_tensor(grid_neighbor_table(side, n // side)).to(grp.device)
    feat_ms = timed(lambda: grp.featurize(halting, zi, zd, zd, 0.0, zv, nbr), 200, stream)
    f_bytes = n * (64 + 96 * 4 + 17 * 8 + 8)
    pk = peaks()["hbm_gbs"]
    return {"gather": {"ms": gather_ms, "api_sample_ms": sample_ms, "bytes_per_transition": 724, "algorithmic_bytes": g_bytes,
                       "gbs": g_bytes / (gather_ms / 1e3) / 1e9, "hbm_frac": g_bytes / (gather_ms / 1e3) / 1e9 / pk,
                       "note": "dmdqn_gather alone (rows already sampled): B x 724 B read from the rings + the same written densely"},
            "featurize": {"ms": feat_ms, "agents_per_s": n * world / (feat_ms / 1e3), "bytes_per_agent": 64 + 96 * 4 + 17 * 8 + 8,
                          "gbs": f_bytes / (feat_ms / 1e3) / 1e9, "hbm_frac": f_bytes / (feat_ms / 1e3) / 1e9 / pk,
                          "note": "launch bound: a few hundred KB per call"}}


def run_ours(args):
    from dmdqn_b200.group import AgentGroup
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    w = WORKLOADS[args.workload]
    fb = flops_bytes(w)
    grp = AgentGroup(w["agents"], agent_cfg(w, args.precision), D, A, seed=1000 * rank)
    synth_fill(grp, seed=rank)
    n, b = grp.n_agents, grp.batch_size
    K, W = args.steps, args.warmup
    draws = grp.draw_words((K + W, n, b))
    stream = torch.cuda.current_stream()

    # ---- device-resident throughput: K learn sweeps, inputs already in HBM ----------------
    sampler = ClockSampler(local)
    for i in range(W):
        grp.learn(draws[i])
    _barrier(world)
    sampler.start()
    e0, e1 = _events(2)
    e0.record(stream)
    for i in range(K):
        metrics = grp.learn(draws[W + i])
    e1.record(stream)
    _barrier(world)
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:                        # before anything below moves the weights on
        dump_outputs(args.dump_outputs, learn_outputs(grp, metrics))

    # ---- per-kernel durations: same sweep, one stage per call, events in between ----------
    stage_ms = stage_times(grp, draws[W:], K)

    # ---- end to end: host transitions + draws in, losses out, every step ------------------
    # dmdqn_step_host (include/dmdqn_b200.h): the step's inputs sit in ONE pinned host block (struct of arrays);
    # the call queues one H2D copy, push, learn and the copy of the metrics back; the caller synchronises and reads.
    sb = grp.make_step_block()
    hv = sb["host"]
    hv["obs"].copy_(torch.randint(0, 20, (n, D)).float()); hv["next_obs"].copy_(torch.randint(0, 20, (n, D)).float())
    hv["act"].copy_(torch.randint(0, A, (n,), dtype=torch.int32)); hv["rew"].copy_(-torch.rand(n, dtype=torch.float64) * 100)
    hv["done"].zero_(); hv["draws"].copy_(torch.randint(0, 2**31, (n, b), dtype=torch.int32))
    h2d = sb["bytes"]
    d2h = sb["metrics_host"].numel() * sb["metrics_host"].element_size()

    def e2e_step():
        m = grp.step_host(sb)                                  # remember + replay (train.py:274-292), host buffers
        stream.synchronize()                                   # the caller reads the losses
        return float(m[0, 0])
    for _ in range(W):
        e2e_step()
    _barrier(world)
    e0.record(stream)
    for _ in range(K):
        e2e_step()
    e1.record(stream)
    _barrier(world)
    ms_e2e_plain = e0.elapsed_time(e1)
    # the same step as ONE CUDA-graph launch (AgentGroup.capture_step_host: the copy in, push, the learn chain and the copy of
    # the losses out captured once; same host block, same bits): what a training loop that keeps its step block would call
    replay_step = grp.capture_step_host(sb)

    def e2e_graph_step():
        m = replay_step()
        stream.synchronize()
        return float(m[0, 0])
    for _ in range(W):
        e2e_graph_step()
    _barrier(world)
    e0.record(stream)
    for _ in range(K):
        e2e_graph_step()
    e1.record(stream)
    _barrier(world)
    ms_e2e = e0.elapsed_time(e1)
    grp.check_errors()                                         # raises if a tcgen05 kernel's bounded wait expired
    ms, ms_e2e, ms_e2e_plain = _max_over_ranks([ms, ms_e2e, ms_e2e_plain], world, grp.device)

    extra = block_gather_featurize(grp, world, K)
    del grp, draws
    torch.cuda.empty_cache()

    # ---- the other configurations north_star names --------------------------------------------
    blocks = {}
    want = set(args.blocks.split(",")) if args.blocks not in ("all", "none") else (
        {"act", "cfg2", "strong_cfg3", "cfg4", "cfg5"} if args.blocks == "all" else set())
    bk, bw = max(3, min(K, args.block_steps)), 3
    if "act" in want:
        extra["act"] = block_act(args, rank, world, local)
    if "cfg2" in want:
        blocks["cfg2"] = block_cfg2(args, rank, world, local, bk, bw)
    if "strong_cfg3" in want:
        blocks["strong_cfg3"] = block_strong_cfg3(args, rank, world, local, bk, bw)
    if "cfg4" in want:
        blocks["cfg4"] = block_cfg4(args, rank, world, local, max(3, bk // 3), bw)
    if "cfg5" in want:
        blocks["cfg5"] = block_cfg5(args, rank, world, local, bk, bw)

    total_agents = n * world
    value = total_agents * K / (ms / 1e3)
    pk = peaks()
    dom = max(("target", "online", "wgrad_adam"), key=lambda k_: stage_ms[k_])
    kt = kernel_table(w, n, stage_ms, args.workload, args.precision)
    ffma_peak = 148 * 128 * 2 * (clocks["sm_mhz"] or 1965.0) * 1e6 / 1e12
    launches_per_step = 4
    out = {
        "metric": "agent-updates/sec", "value": value, "unit": "agent-updates/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic replay (observation-shaped integers, full rings), random-init weights",
        "config": {"workload": workload_name(args.workload)},
        "details": {"precision": args.precision, "agents_total": total_agents,
                    "sharding": "agent ranges, no collectives" if world > 1 else "single GPU",
                    "l2_policy": "working set (replay ring 5.9 GB, theta/m/v 368 MB, scratch 200 MB at cfg3) exceeds the 126 MB L2",
                    "sample_mode": "fisher_yates (device draws)"},
        "e2e": {"value": total_agents * K / (ms_e2e / 1e3), "unit": "agent-updates/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / K,
                "what": "AgentGroup.capture_step_host: dmdqn_step_host (one pinned host block with the transition of every agent + the draws -> one H2D copy -> push -> learn chain -> losses to pinned host memory) captured once and replayed as ONE CUDA-graph launch per step; the host block is the step's input, the stream is synchronised and the loss read every step",
                "plain_call": {"value": total_agents * K / (ms_e2e_plain / 1e3), "ms_per_step": ms_e2e_plain / K,
                               "what": "the same step through AgentGroup.step_host (six operations enqueued per step instead of one graph launch)"}},
        "gpu_launches": launches_per_step * K,
        "clocks": clocks,
        "roofline": _with_chain_note(roofline_of(dom, kt, pk, args.precision, ffma_peak, runner_up=sorted(("target", "online", "wgrad_adam"), key=lambda k_: -stage_ms[k_])[1]),
                                     dom, kt, stage_ms, ms / K, pk),
        "kernels": kt,
        **extra,
        "step": {"flops_per_agent_update": fb["flops"], "bytes_per_agent_update": fb["bytes"],
                 "tflops": n * fb["flops"] / (ms / K / 1e3) / 1e12, "hbm_gbs_algorithmic": n * fb["bytes"] / (ms / K / 1e3) / 1e9,
                 "hbm_frac": n * fb["bytes"] / (ms / K / 1e3) / 1e9 / pk["hbm_gbs"]},
        "blocks": blocks,
    }
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(w, budget_s=args.cpu_budget)
        emit(out)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------
def build_oracle_agents(w, n_agents, seed=0):
    """Faithful per-agent oracle objects with full deque buffers (reference structure:
    one DQNAgent per intersection, train.py:109-127)."""
    from oracle.dqn import OracleDQNAgent
    rng = np.random.default_rng(seed)
    agents = []
    c = w["capacity"]
    for i in range(n_agents):
        ag = OracleDQNAgent(D, A, f"J_{i}", dict(agent_cfg(w), seed=i))
        s = rng.integers(-1, 20, (c, 1, D)).astype(np.float32); s2 = rng.integers(-1, 20, (c, 1, D)).astype(np.float32)
        a = rng.integers(0, A, c); r = -0.3 * rng.integers(0, 240, c) - 0.7 * rng.integers(0, 240 * 256, c)
        dn = rng.random(c) < 1 / 240
        for t in range(c):
            ag.replay_buffer.buffer.append((s[t, 0], int(a[t]), float(r[t]), s2[t, 0], bool(dn[t])))
        agents.append(ag)
    return agents


def cpu_baseline(w, budget_s=15.0, sample_agents=None):
    """The oracle's sequential per-agent learn loop (train.py:274-292 + dqn_agent.py:328-380)
    on this box's host cores, bounded to ~budget_s of CPU work."""
    sample_agents = sample_agents or min(w["agents"], 16)
    random.seed(0)
    agents = build_oracle_agents(w, sample_agents)
    for ag in agents[:2]:
        ag.replay()                                   # warm-up
    t0 = time.perf_counter(); sweeps = 0
    while True:
        for ag in agents:
            ag.replay()
        sweeps += 1
        el = time.perf_counter() - t0
        if el > budget_s or sweeps >= 200:
            break
    return {"value": sample_agents * sweeps / el, "unit": "agent-updates/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{sample_agents} of {w['agents']} agents (full {w['capacity']}-deep deque buffers), {sweeps} learn sweeps, "
                      f"{el:.1f} s; sequential per-agent loop of the CPU PyTorch oracle (reference is TensorFlow: not installable)",
            "host_cpus": os.cpu_count()}


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port; oracle/_ref does not exist because
    TensorFlow/Keras cannot be installed) on the host cores, same workload/metric."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    w = WORKLOADS[args.workload]
    sample_agents = min(w["agents"], 16)
    random.seed(0)
    agents = build_oracle_agents(w, sample_agents)
    K, W = args.steps, args.warmup
    for _ in range(min(W, 3)):
        for ag in agents:
            ag.replay()
    t0 = time.perf_counter()
    for _ in range(K):
        for ag in agents:
            ag.replay()
    el = time.perf_counter() - t0
    v = sample_agents * K / el
    sample = (f"each step = one learn sweep over {sample_agents} of {w['agents']} agents (full {w['capacity']}-deep deque buffers); "
              "sequential per-agent loop")
    emit({
        "impl": "reference", "metric": "agent-updates/sec", "value": v, "unit": "agent-updates/s",
        "n_gpus": int(os.environ.get("WORLD_SIZE", 1)), "steps": K, "warmup": W, "ms_per_step": el / K * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic replay",
        "config": {"workload": workload_name(args.workload)},
        "cpu_baseline": {"value": v, "unit": "agent-updates/s", "cores": torch.get_num_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "agent-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="tf32x3", choices=["fp32", "tf32x3", "tf32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--blocks", default="all", help="all | none | comma list of act,cfg2,strong_cfg3,cfg4,cfg5")
    ap.add_argument("--block-steps", type=int, default=30)
    ap.add_argument("--cpu-budget", type=float, default=15.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed learn sweep (rank 0) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
