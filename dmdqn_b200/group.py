"""AgentGroup: all intersection agents of one GPU behind batched calls.

The reference keeps ``agents: dict[str, DQNAgent]`` and walks it sequentially
(src/scripts/train.py:109-127,211-292).  Here the same state lives in a handful of device
tensors (layout: include/dmdqn_b200.h) and every step of the hot path is one native call
over all agents:

    featurize  -> K0   (order_lanes.py:392-555, train.py:159-165,241-254)
    act        -> K2   (dqn_agent.py:246-274)
    push       -> K1a  (dqn_agent.py:31-57,306-325)
    sample     -> K1b  (dqn_agent.py:59-85)
    learn      -> K1b+K3+K4 (dqn_agent.py:328-380)

PyTorch is only the allocator / stream provider; the arithmetic is in
libdmdqn_b200.so.  ``agent_view(i)`` gives a 1-agent group on the same storage (offset
pointers), which is what the per-agent ``DQNAgent`` facade (agent.py) drives.
"""
from __future__ import annotations

import ctypes as C
import functools
import math
import numbers

import numpy as np
import torch

from . import _native as N

DEFAULTS = {  # DQNAgent defaults, dqn_agent.py:112-127
    "learning_rate": 0.001, "gamma": 0.99, "epsilon_start": 1.0, "epsilon_min": 0.01,
    "epsilon_decay_steps": 100000, "replay_buffer_size": 10000, "batch_size": 128,
    "target_update_frequency": 1000, "nn_layers": [64, 64],
    # new keys (SURVEY.md section 5 "Config / flags"); defaults = reference behaviour
    "tau": None, "loss": "mse", "normalize_rewards": True, "double_dqn": True, "adam_form": "keras",
    "share_parameters": False, "precision": "auto", "sample_mode": "fisher_yates",
    # prioritized replay (sample_mode "prioritized"): priority exponent, initial importance exponent (annealed to 1 over
    # per_beta_steps learn steps), priority offset
    "per_alpha": 0.6, "per_beta": 0.4, "per_beta_steps": 100000, "per_eps": 1e-6,
    # n-step returns: transitions per TD target (1 = the reference's one-step target), at most N.MAX_NSTEP
    "n_step": 1,
    # global-norm gradient clipping (Keras global_clipnorm): None, or c > 0 to scale each network's gradient to a norm <= c
    "global_clipnorm": None,
    # dueling Q-networks (Wang et al. 2016): value and advantage heads on the shared trunk, Q = V + Adv - mean(Adv)
    "dueling": False,
    # noisy networks (Fortunato et al. 2018): factorized Gaussian noise on every layer replaces epsilon-greedy exploration;
    # sigma starts at noisy_sigma0 / sqrt(fan_in)
    "noisy": False, "noisy_sigma0": 0.5,
}


def _ptr(t: torch.Tensor | None) -> int | None:
    return None if t is None else t.data_ptr()


def _on_device(method):
    """Native calls launch on the CURRENT device with the stream they are handed: make the group's device current
    for the duration of the call, so a process that holds groups on several GPUs launches each on its own."""
    @functools.wraps(method)
    def wrapper(self, *args, **kwargs):
        if torch.cuda.current_device() == self.device.index:
            return method(self, *args, **kwargs)
        with torch.cuda.device(self.device):
            return method(self, *args, **kwargs)
    return wrapper


def keras_init(seed: int, state_size: int, hidden: int, action_size: int, dueling: bool = False) -> list[torch.Tensor]:
    """HeNormal hidden kernels, GlorotUniform head, zero biases (dqn_agent.py:166-181), as
    [W1,b1,W2,b2,W3,b3] in Keras ``get_weights()`` order, kernels ``[in,out]``.  ``dueling`` appends the value head
    [Wv [H,1], bv [1]], Wv GlorotUniform drawn from the same generator after W3 (the other draws do not change)."""
    gen = torch.Generator().manual_seed(int(seed))
    out = []
    dims = [state_size, hidden, hidden]
    for i in range(2):
        std = math.sqrt(2.0 / dims[i]) / 0.87962566103423978
        w = torch.empty(dims[i], dims[i + 1])
        torch.nn.init.trunc_normal_(w, 0.0, std, -2 * std, 2 * std, generator=gen)
        out += [w, torch.zeros(dims[i + 1])]
    limit = math.sqrt(6.0 / (hidden + action_size))
    out += [(torch.rand(hidden, action_size, generator=gen) * 2 - 1) * limit, torch.zeros(action_size)]
    if dueling:
        limit = math.sqrt(6.0 / (hidden + 1))
        out += [(torch.rand(hidden, 1, generator=gen) * 2 - 1) * limit, torch.zeros(1)]
    return out


def noise_key(seed: int) -> int:
    """The 64-bit Philox key of a noisy network from its init seed (``seed + g``, the seed ``keras_init`` takes): splitmix64,
    so a network's noise depends on its global index only, not on how the agents are sharded."""
    m = (1 << 64) - 1
    z = (int(seed) + 0x9E3779B97F4A7C15) & m
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & m
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & m
    return z ^ (z >> 31)


class AgentGroup:
    def __init__(self, n_agents: int, config: dict | None = None, state_size: int = 89, action_size: int = 4,
                 device: str | torch.device | None = None, seed: int = 0, _parent: "AgentGroup | None" = None,
                 _index: int = 0):
        cfg = dict(DEFAULTS)
        cfg.update(config or {})
        self.config = cfg
        layers = list(cfg["nn_layers"])
        if len(layers) != 2 or layers[0] != layers[1]:
            raise ValueError(f"nn_layers={layers}: the CUDA path supports two equal hidden layers [H, H]")
        self.n_agents = int(n_agents)
        self.shared = bool(cfg["share_parameters"])
        self.prioritized = cfg["sample_mode"] == "prioritized"
        if self.prioritized and self.shared:
            raise ValueError("sample_mode='prioritized' serves independent networks only: it cannot be combined with "
                             "share_parameters=true")
        self.n_step = int(cfg["n_step"])
        if not 1 <= self.n_step <= N.MAX_NSTEP:
            raise ValueError(f"n_step={cfg['n_step']}: must be in [1, {N.MAX_NSTEP}] (1 = one-step TD targets)")
        clip = cfg["global_clipnorm"]
        if clip is not None and (isinstance(clip, bool) or not isinstance(clip, numbers.Real) or not math.isfinite(clip)
                                 or clip <= 0):
            raise ValueError(f"global_clipnorm={clip!r}: must be None (no clipping) or a positive finite number")
        self.global_clipnorm = None if clip is None else float(clip)
        if cfg["dueling"] not in (True, False):
            raise ValueError(f"dueling={cfg['dueling']!r}: must be true or false")
        self.dueling = bool(cfg["dueling"])
        if not isinstance(cfg["noisy"], (bool, np.bool_)):
            raise ValueError(f"noisy={cfg['noisy']!r}: must be true or false")
        self.noisy = bool(cfg["noisy"])
        s0 = cfg["noisy_sigma0"]
        if isinstance(s0, bool) or not isinstance(s0, numbers.Real) or not math.isfinite(s0) or s0 < 0:
            raise ValueError(f"noisy_sigma0={s0!r}: must be a finite number >= 0")
        self.noisy_sigma0 = float(s0)
        if self.noisy and self.global_clipnorm is not None:
            raise ValueError("noisy=true cannot be combined with global_clipnorm yet: the global norm over the mean and the "
                             "sigma gradients is not implemented")
        self.n_nets = 1 if self.shared else self.n_agents
        self.state_size, self.action_size = int(state_size), int(action_size)
        self.obs_stride = (self.state_size + 15) // 16 * 16
        self.hidden = int(layers[0])
        self.batch_size = int(cfg["batch_size"])
        self.capacity = int(cfg["replay_buffer_size"])
        self.lib = N.lib()  # raises if the extension is missing: no fallback
        if not torch.cuda.is_available():
            raise N.NativeError("dmdqn_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())

        self.dims = N.Dims(self.n_agents, self.n_nets, self.state_size, self.obs_stride, self.hidden,
                           self.action_size, self.batch_size, self.capacity)
        if self.dueling:        # W1 | b1 | W2 | b2 | W3 | b3 | wv | bv: the same offsets up to b3, a longer stride
            self.layout = N.DuelingLayout()
            N.check(self.lib.dmdqn_param_layout_dueling(C.byref(self.dims), C.byref(self.layout)))
        else:
            self.layout = N.Layout()
            N.check(self.lib.dmdqn_param_layout(C.byref(self.dims), C.byref(self.layout)))
        self.noise_record = N.NoiseRecord()
        N.check(self.lib.dmdqn_noise_layout(C.byref(self.dims), C.byref(self.noise_record)))
        if cfg["precision"] == "auto":   # fp32-class either way (same 1e-5 bar): tcgen05 3xTF32 where that path is built, FFMA elsewhere
            cfg["precision"] = "tf32x3" if (self.hidden == 256 and self.obs_stride in (32, 64, 96) and self.batch_size % 4 == 0
                                            and self.batch_size <= 4096) else "fp32"
        self.hp = N.HParams(
            float(cfg["gamma"]), float(cfg["learning_rate"]), 0.9, 0.999,
            1e-7 if cfg["adam_form"] == "keras" else 1e-8,
            -1.0 if cfg["tau"] is None else float(cfg["tau"]),
            int(cfg["target_update_frequency"]), N.LOSS[cfg["loss"]], int(bool(cfg["normalize_rewards"])),
            int(bool(cfg["double_dqn"])), N.ADAM[cfg["adam_form"]], N.SAMPLE[cfg["sample_mode"]],
            N.PRECISION[cfg["precision"]], float(cfg["per_alpha"]), float(cfg["per_beta"]), float(cfg["per_eps"]),
            int(cfg["per_beta_steps"]), self.n_step, dueling=int(self.dueling))

        dev, n, c, dp, g = self.device, self.n_agents, self.capacity, self.obs_stride, self.n_nets
        for name in self._NOISY_PTRS:
            setattr(self, name, None)
        if _parent is None:
            self.obs = torch.zeros((n, c, dp), dtype=torch.float32, device=dev)
            self.next_obs = torch.zeros((n, c, dp), dtype=torch.float32, device=dev)
            self.act_ring = torch.zeros((n, c), dtype=torch.int32, device=dev)
            self.rew_ring = torch.zeros((n, c), dtype=torch.float64, device=dev)
            self.done_ring = torch.zeros((n, c), dtype=torch.uint8, device=dev)
            self.n_written = torch.zeros((n,), dtype=torch.int64, device=dev)
            self.theta = torch.zeros((g, self.layout.stride), dtype=torch.float32, device=dev)
            self.theta_tgt = torch.zeros_like(self.theta)
            self.adam_m = torch.zeros_like(self.theta)
            self.adam_v = torch.zeros_like(self.theta)
            self.learn_step = torch.zeros((g,), dtype=torch.int32, device=dev)
            # prioritized replay: p^alpha per physical slot (0 = never written) and each ring's largest priority
            self.priority = torch.zeros((n, c), dtype=torch.float32, device=dev) if self.prioritized else None
            self.priority_max = torch.ones((n,), dtype=torch.float32, device=dev) if self.prioritized else None
            # gradient clipping: the raw gradient blocks of a step and each network's norm before clipping (last step)
            self.grads = torch.zeros_like(self.theta) if self.global_clipnorm is not None else None
            self.grad_norms = torch.zeros((g,), dtype=torch.float32, device=dev) if self.global_clipnorm is not None else None
            if self.noisy:      # sigma with its target and moments, the effective blocks, the gradient and the noise record
                self.sigma, self.sigma_tgt = torch.zeros_like(self.theta), torch.zeros_like(self.theta)
                self.sigma_m, self.sigma_v = torch.zeros_like(self.theta), torch.zeros_like(self.theta)
                self.eff, self.eff_tgt = torch.zeros_like(self.theta), torch.zeros_like(self.theta)
                self.grads = torch.zeros_like(self.theta)
                self.noise = torch.zeros((g, 2, int(self.noise_record.stride)), dtype=torch.float32, device=dev)
                self.key = torch.zeros((g,), dtype=torch.int64, device=dev)
            self.n_written_host = np.zeros((n,), np.int64)       # host mirrors: no device sync
            self.learn_step_host = np.zeros((g,), np.int64)
        else:
            p, i = _parent, _index
            j = 0 if p.shared else i
            self.obs, self.next_obs = p.obs[i:i + 1], p.next_obs[i:i + 1]
            self.act_ring, self.rew_ring, self.done_ring = p.act_ring[i:i + 1], p.rew_ring[i:i + 1], p.done_ring[i:i + 1]
            self.n_written = p.n_written[i:i + 1]
            self.priority = None if p.priority is None else p.priority[i:i + 1]
            self.priority_max = None if p.priority_max is None else p.priority_max[i:i + 1]
            self.theta, self.theta_tgt = p.theta[j:j + 1], p.theta_tgt[j:j + 1]
            self.adam_m, self.adam_v = p.adam_m[j:j + 1], p.adam_v[j:j + 1]
            self.learn_step = p.learn_step[j:j + 1]
            self.grads = None if p.grads is None else p.grads[j:j + 1]
            self.grad_norms = None if p.grad_norms is None else p.grad_norms[j:j + 1]
            if self.noisy:
                for name in self._NOISY:
                    setattr(self, name, getattr(p, name)[j:j + 1])
            self.n_written_host = p.n_written_host[i:i + 1]
            self.learn_step_host = p.learn_step_host[j:j + 1]
        self.replay = N.Replay(_ptr(self.obs), _ptr(self.next_obs), _ptr(self.act_ring), _ptr(self.rew_ring),
                               _ptr(self.done_ring), _ptr(self.n_written), _ptr(self.priority), _ptr(self.priority_max))
        self.nets = N.Nets(_ptr(self.theta), _ptr(self.theta_tgt), _ptr(self.adam_m), _ptr(self.adam_v),
                           _ptr(self.learn_step))
        self.noisy_ptrs = N.Noisy(*(_ptr(getattr(self, k)) for k in self._NOISY_PTRS)) if self.noisy else None
        nbytes = C.c_size_t()
        N.check(self.lib.dmdqn_workspace_bytes(C.byref(self.dims), C.byref(nbytes)))
        self.workspace = torch.zeros((nbytes.value,), dtype=torch.uint8, device=dev)
        dv = N.DebugViews()
        N.check(self.lib.dmdqn_debug(C.byref(self.dims), _ptr(self.workspace), self.workspace.numel(), C.byref(dv)))
        self._tc_error_offset = dv.tc_error - self.workspace.data_ptr()
        self.metrics = torch.zeros((g, N.METRICS_STRIDE), dtype=torch.float32, device=dev)
        self._feat_scratch = torch.zeros((2,), dtype=torch.int64, device=dev)
        self._zero_eps = torch.zeros((n,), dtype=torch.float64, device=dev)
        self._zero_words = torch.zeros((n,), dtype=torch.int32, device=dev)
        self._gen = torch.Generator(device=dev)
        self._gen.manual_seed(int(seed) + 0x5EED)
        self._views: dict[int, AgentGroup] = {}
        if _parent is None:
            self.init_weights(seed)

    # the noisy tensors: the dmdqn_noisy fields in order, and the gradient block of the noisy learn step
    _NOISY_PTRS = ("sigma", "sigma_tgt", "sigma_m", "sigma_v", "eff", "eff_tgt", "noise", "key")
    _NOISY = _NOISY_PTRS + ("grads",)

    # ------------------------------------------------------------------ helpers ---------
    @property
    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def _dev(self, x, dtype) -> torch.Tensor:
        # np.asarray first: torch.as_tensor on a list of Python floats makes a float32 tensor, which would round the
        # float64 rewards the reference keeps as Python floats (dqn_agent.py:43) before they reach the ring
        t = x if isinstance(x, torch.Tensor) else torch.as_tensor(np.asarray(x))
        return t.to(device=self.device, dtype=dtype, non_blocking=True).contiguous()

    def agent_view(self, i: int) -> "AgentGroup":
        """1-agent group over agent i's slices of this group's storage."""
        if self.n_agents == 1:
            return self
        if i not in self._views:
            self._views[i] = AgentGroup(1, dict(self.config, share_parameters=False), self.state_size,
                                        self.action_size, self.device, _parent=self, _index=i)
        return self._views[i]

    def sizes_host(self) -> np.ndarray:
        return np.minimum(self.n_written_host, self.capacity)

    # ------------------------------------------------------------------ weights ---------
    def pack(self, weights) -> torch.Tensor:
        """[W1,b1,W2,b2,W3,b3] (Keras order, kernels [in,out]; dueling: + [Wv [H,1], bv [1]]) -> one parameter block."""
        L, H, A = self.layout, self.hidden, self.action_size
        ws = [torch.as_tensor(np.asarray(w), dtype=torch.float32) for w in weights]
        if len(ws) != (8 if self.dueling else 6):
            raise ValueError(f"expected {8 if self.dueling else 6} weight tensors, got {len(ws)}")
        w1, b1, w2, b2, w3, b3 = ws[:6]
        blk = torch.zeros((L.stride,), dtype=torch.float32)
        blk[L.w1:L.w1 + self.obs_stride * H].view(self.obs_stride, H)[: self.state_size] = w1
        blk[L.b1:L.b1 + H] = b1
        blk[L.w2:L.w2 + H * H] = w2.reshape(-1)
        blk[L.b2:L.b2 + H] = b2
        blk[L.w3:L.w3 + H * 4].view(H, 4)[:, :A] = w3
        blk[L.b3:L.b3 + A] = b3
        if self.dueling:
            blk[L.wv:L.wv + H] = ws[6].reshape(H)
            blk[L.bv:L.bv + 1] = ws[7].reshape(1)
        return blk

    def unpack(self, blk: torch.Tensor) -> list[torch.Tensor]:
        L, H, A = self.layout, self.hidden, self.action_size
        blk = blk.detach().cpu()
        out = [blk[L.w1:L.w1 + self.obs_stride * H].view(self.obs_stride, H)[: self.state_size].clone(),
               blk[L.b1:L.b1 + H].clone(), blk[L.w2:L.w2 + H * H].view(H, H).clone(),
               blk[L.b2:L.b2 + H].clone(), blk[L.w3:L.w3 + H * 4].view(H, 4)[:, :A].clone(),
               blk[L.b3:L.b3 + A].clone()]
        if self.dueling:
            out += [blk[L.wv:L.wv + H].view(H, 1).clone(), blk[L.bv:L.bv + 1].clone()]
        return out

    def sigma_init(self) -> list[torch.Tensor]:
        """Initial sigma of a noisy network in ``keras_init``'s order: noisy_sigma0 / sqrt(fan_in) for every weight and bias
        of a layer (Fortunato et al.'s factorized rule), fan_in = state_size for layer 1 and H after it."""
        d, h, a = self.state_size, self.hidden, self.action_size
        s1, s2 = np.float32(self.noisy_sigma0 / math.sqrt(d)), np.float32(self.noisy_sigma0 / math.sqrt(h))
        shapes = [((d, h), s1), ((h,), s1), ((h, h), s2), ((h,), s2), ((h, a), s2), ((a,), s2)]
        if self.dueling:
            shapes += [((h, 1), s2), ((1,), s2)]
        return [torch.full(shape, float(v), dtype=torch.float32) for shape, v in shapes]

    def init_weights(self, seed: int = 0) -> None:
        """Per-network Keras-style init (seed + g), target = online, Adam state zero
        (dqn_agent.py:129-137).  Noisy networks: sigma from ``sigma_init``, the Philox key ``noise_key(seed + g)``."""
        blocks = torch.stack([self.pack(keras_init(seed + g, self.state_size, self.hidden, self.action_size, self.dueling))
                              for g in range(self.n_nets)])
        self.theta.copy_(blocks)
        self.theta_tgt.copy_(blocks)
        self.adam_m.zero_(); self.adam_v.zero_(); self.learn_step.zero_()
        self.learn_step_host[:] = 0
        if self.noisy:
            sig = self.pack(self.sigma_init()).to(self.device)
            self.sigma.copy_(sig.expand_as(self.sigma)); self.sigma_tgt.copy_(self.sigma)
            self.sigma_m.zero_(); self.sigma_v.zero_()
            keys = [noise_key(seed + g) for g in range(self.n_nets)]
            self.key.copy_(torch.tensor([k - (1 << 64) if k >= 1 << 63 else k for k in keys], dtype=torch.int64))

    def _blocks(self, which: str) -> list[torch.Tensor]:
        t = {"online": (self.theta, self.sigma), "target": (self.theta_tgt, self.sigma_tgt), "m": (self.adam_m, self.sigma_m),
             "v": (self.adam_v, self.sigma_v)}[which]
        return list(t) if self.noisy else [t[0]]

    def set_weights(self, net: int, weights, which: str = "online", sync_target: bool = False) -> None:
        """``weights`` as ``get_weights`` returns them: noisy networks take the mu list followed by the sigma list."""
        weights = list(weights)
        blocks = self._blocks(which)
        k = len(weights) // len(blocks)
        if k * len(blocks) != len(weights):
            raise ValueError(f"expected {len(blocks)} equal lists of weight tensors, got {len(weights)} tensors")
        for i, (t, tg) in enumerate(zip(blocks, self._blocks("target"))):
            t[net].copy_(self.pack(weights[i * k:(i + 1) * k]))
            if sync_target:
                tg[net].copy_(t[net])

    def get_weights(self, net: int, which: str = "online") -> list[torch.Tensor]:
        """[W1, b1, W2, b2, W3, b3] (+ [Wv, bv] with dueling heads); noisy networks: the mu list, then the sigma list."""
        return [w for t in self._blocks(which) for w in self.unpack(t[net])]

    # ------------------------------------------------------------------ K0 --------------
    @_on_device
    def featurize(self, halting, phase, next_switch, phase_dur, sim_time, signal_valid, nbr_idx,
                  phase_lut=None, snapshot=None, local_weight=0.3, global_weight=0.7, obs_out=None):
        """Returns (obs[N,obs_stride] f32, own[N,17] f64, reward[N] f64, global_reward[1] f64), all on
        the device.  obs[:, :89] is the reference's build_state_vector output."""
        n = self.n_agents
        halting = self._dev(halting, torch.int32); phase = self._dev(phase, torch.int32)
        next_switch = self._dev(next_switch, torch.float64); phase_dur = self._dev(phase_dur, torch.float64)
        signal_valid = self._dev(signal_valid, torch.uint8); nbr_idx = self._dev(nbr_idx, torch.int32)
        if phase_lut is None:
            phase_lut = torch.tensor([0, 1, 2, 3] + [-1] * 12, dtype=torch.int32)   # PHASE_ENCODING
        phase_lut = self._dev(phase_lut, torch.int32)
        snapshot = None if snapshot is None else self._dev(snapshot, torch.float64)
        obs = obs_out if obs_out is not None else torch.empty((n, self.obs_stride), dtype=torch.float32, device=self.device)
        own = torch.empty((n, 17), dtype=torch.float64, device=self.device)
        reward = torch.empty((n,), dtype=torch.float64, device=self.device)
        glob = torch.empty((1,), dtype=torch.float64, device=self.device)
        N.check(self.lib.dmdqn_featurize(n, _ptr(halting), _ptr(phase), _ptr(next_switch), _ptr(phase_dur),
                                         float(sim_time), _ptr(signal_valid), _ptr(nbr_idx), _ptr(phase_lut),
                                         _ptr(snapshot), float(local_weight), float(global_weight), _ptr(own),
                                         _ptr(obs), obs.shape[1], _ptr(reward), _ptr(glob),
                                         _ptr(self._feat_scratch), self._stream))
        return obs, own, reward, glob

    @_on_device
    def featurize_alt(self, halting_nesw, phase, next_switch, sim_time, nbr_idx_nesw, signal_valid=None, prev_own=None,
                      obs_stride: int = 76):
        """The SumoTrafficEnvironment contract (sumo_env.py:532-679): returns (obs[N,obs_stride] f32 whose first 74
        columns are ``_get_observations``' vector, own[N,14] f64 to pass as ``prev_own`` next step, reward[N] f64 =
        ``_calculate_rewards`` (0 on the first step)), all on the device.  Queue codes: -2 = PAD lane, -1 = failed read."""
        n = self.n_agents
        halting = self._dev(halting_nesw, torch.int32); phase = self._dev(phase, torch.int32)
        next_switch = self._dev(next_switch, torch.float64); nbr_idx = self._dev(nbr_idx_nesw, torch.int32)
        signal_valid = torch.ones((n,), dtype=torch.uint8, device=self.device) if signal_valid is None \
            else self._dev(signal_valid, torch.uint8)
        prev = None if prev_own is None else self._dev(prev_own, torch.float64)
        obs = torch.empty((n, obs_stride), dtype=torch.float32, device=self.device)
        own = torch.empty((n, 14), dtype=torch.float64, device=self.device)
        reward = torch.empty((n,), dtype=torch.float64, device=self.device)
        N.check(self.lib.dmdqn_featurize_alt(n, _ptr(halting), _ptr(phase), _ptr(next_switch), _ptr(signal_valid),
                                             float(sim_time), _ptr(nbr_idx), _ptr(prev), _ptr(own), _ptr(obs), obs.shape[1],
                                             _ptr(reward), self._stream))
        return obs, own, reward

    # ------------------------------------------------------------------ K2 --------------
    @_on_device
    def act(self, obs, eps=None, w_explore=None, w_action=None, return_q: bool = False, target: bool = False,
            noisy: bool | None = None):
        """Batched epsilon-greedy (dqn_agent.py:263-274).  ``eps`` None -> greedy for all.
        Draws default to the group's device generator.  Returns actions[N] int32 (device)
        and, if asked, q[N,4] (rows of exploring agents are NaN: no forward pass ran).
        ``target=True`` runs the same kernel on the target parameters (``target_network(x)``).
        Noisy networks act on mu + sigma * eps with the online noise of the next learn step (``dmdqn_act_noisy``);
        ``noisy=False`` acts on mu alone (greedy evaluation).  The target network is always read without noise."""
        n = self.n_agents
        obs = self._dev(obs, torch.float32)
        if obs.dim() == 3:
            obs = obs.reshape(n, -1)
        if eps is None:
            eps_t, w1, w2 = self._zero_eps, self._zero_words, self._zero_words
        else:
            eps_t = self._dev(eps, torch.float64).expand(n).contiguous() if torch.as_tensor(eps).dim() == 0 \
                else self._dev(eps, torch.float64)
            w1 = self.draw_words((n,)) if w_explore is None else self._words(w_explore)
            w2 = self.draw_words((n,)) if w_action is None else self._words(w_action)
        actions = torch.empty((n,), dtype=torch.int32, device=self.device)
        q = torch.full((n, 4), float("nan"), dtype=torch.float32, device=self.device) if return_q else None
        nets = self.nets if not target else N.Nets(_ptr(self.theta_tgt), _ptr(self.theta_tgt), _ptr(self.adam_m),
                                                   _ptr(self.adam_v), _ptr(self.learn_step))
        args = (_ptr(obs), obs.shape[1], _ptr(eps_t), _ptr(w1), _ptr(w2), _ptr(actions), _ptr(q), self._stream)
        if self.noisy and noisy is not False and not target:
            N.check(self.lib.dmdqn_act_noisy(C.byref(self.dims), C.byref(nets), C.byref(self.noisy_ptrs), int(self.dueling),
                                             *args))
        else:
            act = self.lib.dmdqn_act_dueling if self.dueling else self.lib.dmdqn_act
            N.check(act(C.byref(self.dims), C.byref(nets), *args))
        return (actions, q) if return_q else actions

    def draw_words(self, shape) -> torch.Tensor:
        """Uniform 32-bit words from the group's device generator (bit pattern of an int32)."""
        w = torch.randint(0, 2**32, shape, dtype=torch.int64, device=self.device, generator=self._gen)
        return (w - 2**31).to(torch.int32)

    def _words(self, w) -> torch.Tensor:
        if isinstance(w, torch.Tensor):
            return w.to(self.device).contiguous().view(torch.int32) if w.dtype in (torch.int32, torch.uint32) \
                else w.to(self.device, torch.int64).to(torch.int32).contiguous()
        return torch.from_numpy(np.ascontiguousarray(np.asarray(w).astype(np.uint32)).view(np.int32)).to(self.device)

    # ------------------------------------------------------------------ K1a -------------
    @_on_device
    def push(self, obs, act, rew, next_obs, done, mask=None) -> None:
        """One transition per agent (dqn_agent.py:312-325 for every agent at once)."""
        n = self.n_agents
        obs = self._dev(obs, torch.float32).reshape(n, -1)
        next_obs = self._dev(next_obs, torch.float32).reshape(n, -1)
        if obs.shape[1] != next_obs.shape[1]:
            return  # dqn_agent.py:50-54: inconsistent sizes -> the transition is dropped
        act = self._dev(act, torch.int32).reshape(n)
        rew = self._dev(rew, torch.float64).reshape(n)
        done = self._dev(done, torch.uint8).reshape(n)
        mask_t = None if mask is None else self._dev(mask, torch.uint8)
        N.check(self.lib.dmdqn_push(C.byref(self.dims), C.byref(self.replay), _ptr(obs), _ptr(act), _ptr(rew),
                                    _ptr(next_obs), _ptr(done), obs.shape[1], _ptr(mask_t), self._stream))
        if mask is None:
            self.n_written_host += 1
        else:
            self.n_written_host += np.asarray(torch.as_tensor(mask).cpu()).astype(np.int64).reshape(n)

    # ------------------------------------------------------------------ K1b -------------
    def _draws(self, draws, mode):
        if draws is None:
            if mode == N.SAMPLE["indices"]:
                raise ValueError("sample_mode='indices' needs explicit logical indices")
            return self.draw_words((self.n_nets, self.batch_size))
        if mode == N.SAMPLE["indices"]:
            return self._dev(draws, torch.int32).reshape(self.n_nets, self.batch_size)
        return self._words(draws).reshape(self.n_nets, self.batch_size)

    def _hp_for(self, sample_mode):
        if sample_mode is None:
            return self.hp
        hp = N.HParams.from_buffer_copy(self.hp)
        hp.sample_mode = N.SAMPLE[sample_mode]
        return hp

    def active_host(self, mask=None) -> np.ndarray:
        """Which networks learn this step (dqn_agent.py:333-335), from the host mirrors."""
        if self.shared:
            on = np.array([int(self.sizes_host()[0]) * self.n_agents >= self.batch_size])
        else:
            on = self.sizes_host() >= self.batch_size
        if mask is not None:
            on = on & np.asarray(torch.as_tensor(mask).cpu()).astype(bool).reshape(self.n_nets)
        return on

    @_on_device
    def sample(self, draws=None, sample_mode: str | None = None):
        """ReplayBuffer.sample for every network (dqn_agent.py:59-85).  Returns
        (states[G,B,D], actions[G,B] i32, rewards[G,B], next_states[G,B,D], dones[G,B], active[G])
        on the device; rows of inactive networks are zero."""
        hp = self._hp_for(sample_mode)
        d = self._draws(draws, hp.sample_mode)
        g, b, dd = self.n_nets, self.batch_size, self.state_size
        N.check(self.lib.dmdqn_sample(C.byref(self.dims), C.byref(hp), C.byref(self.replay), C.byref(self.nets),
                                      _ptr(d), None, 0, _ptr(self.workspace), self.workspace.numel(), self._stream))
        states = torch.zeros((g, b, dd), dtype=torch.float32, device=self.device)
        next_states = torch.zeros_like(states)
        actions = torch.zeros((g, b), dtype=torch.int32, device=self.device)
        rewards = torch.zeros((g, b), dtype=torch.float32, device=self.device)
        dones = torch.zeros((g, b), dtype=torch.float32, device=self.device)
        active = torch.zeros((g,), dtype=torch.int32, device=self.device)
        N.check(self.lib.dmdqn_gather(C.byref(self.dims), C.byref(self.replay), _ptr(self.workspace),
                                      self.workspace.numel(), _ptr(states), _ptr(actions), _ptr(rewards),
                                      _ptr(next_states), _ptr(dones), _ptr(active), self._stream))
        return states, actions, rewards, next_states, dones, active

    # ------------------------------------------------------------------ K1b+K3+K4 -------
    def _learn_call(self, hp, draws_ptr, mask_ptr, stream_ptr) -> None:
        """The learn step's native calls: ``dmdqn_learn``, or with ``global_clipnorm`` set the raw gradients
        (``dmdqn_learn_grads``) followed by the clipped Adam step (``dmdqn_clip_adam_apply``, norms -> ``grad_norms``), or with
        ``noisy`` set ``dmdqn_learn_grads_noisy`` followed by ``dmdqn_noisy_adam_apply``."""
        ws, nws = _ptr(self.workspace), self.workspace.numel()
        if self.noisy:          # gradient of the effective weights, then Adam on mu and sigma
            N.check(self.lib.dmdqn_learn_grads_noisy(C.byref(self.dims), C.byref(hp), C.byref(self.replay), C.byref(self.nets),
                                                     C.byref(self.noisy_ptrs), draws_ptr, mask_ptr, self.batch_size,
                                                     _ptr(self.grads), _ptr(self.metrics), ws, nws, stream_ptr))
            N.check(self.lib.dmdqn_noisy_adam_apply(C.byref(self.dims), C.byref(hp), C.byref(self.nets), C.byref(self.noisy_ptrs),
                                                    _ptr(self.grads), ws, nws, stream_ptr))
            return
        if self.global_clipnorm is None:
            N.check(self.lib.dmdqn_learn(C.byref(self.dims), C.byref(hp), C.byref(self.replay), C.byref(self.nets),
                                         draws_ptr, mask_ptr, _ptr(self.metrics), ws, nws, stream_ptr))
            return
        N.check(self.lib.dmdqn_learn_grads(C.byref(self.dims), C.byref(hp), C.byref(self.replay), C.byref(self.nets),
                                           draws_ptr, mask_ptr, self.batch_size, _ptr(self.grads), _ptr(self.metrics), ws, nws,
                                           stream_ptr))
        N.check(self.lib.dmdqn_clip_adam_apply(C.byref(self.dims), C.byref(hp), C.byref(self.nets), _ptr(self.grads),
                                               self.global_clipnorm, _ptr(self.grad_norms), ws, nws, stream_ptr))

    @_on_device
    def learn(self, draws=None, mask=None, sample_mode: str | None = None) -> torch.Tensor:
        """One Double-DQN step for every network whose ring holds >= batch transitions
        (dqn_agent.py:328-380).  Returns metrics[G,8] on the device: loss, q_mean, q_std,
        action histogram[4], learned flag.  No host sync."""
        hp = self._hp_for(sample_mode)
        d = self._draws(draws, hp.sample_mode)
        mask_t = None if mask is None else self._dev(mask, torch.uint8)
        self._learn_call(hp, _ptr(d), _ptr(mask_t), self._stream)
        self.learn_step_host += self.active_host(mask).astype(np.int64)
        return self.metrics

    @_on_device
    def capture_learn(self, sample_mode: str | None = None):
        """The learn step as a CUDA graph (sample -> K3 -> K4a -> K4b captured once, replayed with one launch): what a
        small grid wants, where the four launches cost as much as the kernels (BASELINE cfg2: 16 agents, B = 64).
        Returns ``(replay, draws)``: refill ``draws`` (int32 [n_nets, B] on the device: uniform words, or logical indices
        in 'indices' mode) and call ``replay()`` -> metrics[G,8] (device, no host sync).  The library keeps no state, so the
        graph is just the four kernels with their arguments; the step counters live on the device as always."""
        hp = self._hp_for(sample_mode)
        draws = self.draw_words((self.n_nets, self.batch_size)).contiguous()
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))

        def launch(stream_ptr, advance_host):
            self._learn_call(hp, _ptr(draws), None, stream_ptr)
            if advance_host:
                self.learn_step_host += self.active_host().astype(np.int64)
        with torch.cuda.stream(side):           # warm-up outside the capture: per-device launch attributes are set here
            launch(side.cuda_stream, True)
        torch.cuda.current_stream(self.device).wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            launch(torch.cuda.current_stream(self.device).cuda_stream, False)

        def replay() -> torch.Tensor:
            graph.replay()
            self.learn_step_host += self.active_host().astype(np.int64)
            return self.metrics
        return replay, draws

    # ------------------------------------------------------------------ host-buffer step ----
    def make_step_block(self):
        """Pinned host block + device mirror for ``step_host``: typed views ``host[name]`` / ``dev[name]`` for
        obs, next_obs [N,obs_dim] f32, act [N] i32, rew [N] f64, done [N] u8, draws [n_nets,B] i32, laid out as one
        struct of arrays so a step is one H2D copy (include/dmdqn_b200.h dmdqn_step_block)."""
        n, d, g, b = self.n_agents, self.state_size, self.n_nets, self.batch_size
        fields = [("obs", torch.float32, (n, d)), ("next_obs", torch.float32, (n, d)), ("rew", torch.float64, (n,)),
                  ("act", torch.int32, (n,)), ("draws", torch.int32, (g, b)), ("done", torch.uint8, (n,))]
        offs, off = {}, 0
        for name, dt, shape in fields:
            off = (off + 15) // 16 * 16
            nbytes = int(np.prod(shape)) * torch.empty((), dtype=dt).element_size()
            offs[name] = (off, nbytes, dt, shape); off += nbytes
        off = (off + 15) // 16 * 16
        host = torch.zeros(off, dtype=torch.uint8).pin_memory()
        dev = torch.zeros(off, dtype=torch.uint8, device=self.device)
        view = lambda blk, k: blk[offs[k][0]:offs[k][0] + offs[k][1]].view(offs[k][2]).view(offs[k][3])
        blk = N.StepBlock(off, offs["obs"][0], offs["next_obs"][0], offs["act"][0], offs["rew"][0], offs["done"][0],
                          offs["draws"][0], d)
        return {"desc": blk, "host_block": host, "dev_block": dev, "bytes": off,
                "host": {k: view(host, k) for k in offs}, "dev": {k: view(dev, k) for k in offs},
                "metrics_host": torch.zeros((g, N.METRICS_STRIDE), dtype=torch.float32).pin_memory()}

    def _step_host_call(self, hp, sb, stream_ptr) -> None:
        """``dmdqn_step_host``; with ``global_clipnorm`` set the same step from its parts on the same stream (the current
        one, ``stream_ptr``): the H2D copy of the block, ``dmdqn_push``, the clipped learn calls and the metrics D2H copy; the
        same with ``noisy`` set and the noisy learn calls."""
        if self.global_clipnorm is None and not self.noisy:
            N.check(self.lib.dmdqn_step_host(C.byref(self.dims), C.byref(hp), C.byref(self.replay), C.byref(self.nets),
                                             C.byref(sb["desc"]), sb["host_block"].data_ptr(), sb["dev_block"].data_ptr(),
                                             _ptr(self.metrics), sb["metrics_host"].data_ptr(), _ptr(self.workspace),
                                             self.workspace.numel(), stream_ptr))
            return
        desc, dev = sb["desc"], sb["dev_block"].data_ptr()
        sb["dev_block"].copy_(sb["host_block"], non_blocking=True)
        N.check(self.lib.dmdqn_push(C.byref(self.dims), C.byref(self.replay), dev + desc.obs_off, dev + desc.act_off,
                                    dev + desc.rew_off, dev + desc.next_obs_off, dev + desc.done_off, desc.in_stride, None,
                                    stream_ptr))
        self._learn_call(hp, dev + desc.draws_off, None, stream_ptr)
        sb["metrics_host"].copy_(self.metrics, non_blocking=True)

    @_on_device
    def step_host(self, sb) -> torch.Tensor:
        """remember + replay for every agent from the HOST block ``sb`` (``make_step_block``): one H2D copy, push, learn,
        metrics back to ``sb["metrics_host"]`` -- all queued on the current stream by ONE library call
        (train.py:274-292).  Synchronise the stream before reading the returned pinned tensor."""
        self._step_host_call(self._hp_for(None), sb, self._stream)
        self.n_written_host += 1
        self.learn_step_host += self.active_host().astype(np.int64)
        return sb["metrics_host"]

    def capture_step_host(self, sb):
        """``step_host`` as a CUDA graph: the H2D copy of the pinned block, push, the learn chain and the copy of the metrics
        back to pinned host memory are captured once and replayed with ONE launch per step (the block and the metrics buffer
        are the fixed addresses of ``sb``; refill ``sb["host"]`` before each replay).  Returns ``replay`` -> the pinned
        metrics tensor; synchronise the stream before reading it.  Same results as ``step_host``, bit for bit."""
        hp = self._hp_for(None)
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))

        def launch(stream_ptr):
            self._step_host_call(hp, sb, stream_ptr)
        with torch.cuda.stream(side):           # warm-up outside the capture (per-device launch attributes): one real step
            launch(side.cuda_stream)
            self.n_written_host += 1
            self.learn_step_host += self.active_host().astype(np.int64)
        torch.cuda.current_stream(self.device).wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            launch(torch.cuda.current_stream(self.device).cuda_stream)

        def replay() -> torch.Tensor:
            graph.replay()
            self.n_written_host += 1
            self.learn_step_host += self.active_host().astype(np.int64)
            return sb["metrics_host"]
        return replay

    def check_errors(self) -> None:
        """Raise if a tcgen05 kernel reported an expired mbarrier wait since the last check (the kernels then skip
        the weight update instead of applying garbage; learned flag metrics[:, 7] < 0).  Reads one int from the
        device: call it where the host synchronises anyway (after reading the losses)."""
        off = self._tc_error_offset
        code = int(self.workspace[off:off + 4].view(torch.int32).item())
        if code:
            self.workspace[off:off + 4].zero_()
            raise N.NativeError(f"a tcgen05 learn kernel timed out on an mbarrier (code {code}); the step was not applied")

    def debug_views(self) -> dict:
        """Intermediate results of the last learn() as device tensors (parity tests)."""
        v = N.DebugViews()
        N.check(self.lib.dmdqn_debug(C.byref(self.dims), _ptr(self.workspace), self.workspace.numel(), C.byref(v)))
        base = self.workspace.data_ptr()
        g, b = self.n_nets, self.batch_size

        def view(ptr, dtype, shape):
            off = ptr - base
            nbytes = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
            return self.workspace[off:off + nbytes].view(dtype).view(*shape)
        nv = N.NStepViews()
        N.check(self.lib.dmdqn_debug_nstep(C.byref(self.dims), _ptr(self.workspace), self.workspace.numel(), C.byref(nv)))
        out = {"y": view(v.y, torch.float32, (g, b)), "q_all": view(v.q_all, torch.float32, (g, b, 4)),
               "q_next": view(v.q_next, torch.float32, (g, b, 4)), "tq_all": view(v.tq_all, torch.float32, (g, b, 4)),
               "rows": view(v.rows, torch.int32, (g, b)), "r_hat": view(v.r_hat, torch.float32, (g, b)),
               "active": view(v.active, torch.int32, (g,)), "tc_error": view(v.tc_error, torch.int32, (1,)),
               "is_weights": view(v.is_w, torch.float32, (g, b)),
               "next_rows": view(nv.next_rows, torch.int32, (g, b)), "discount": view(nv.discount, torch.float32, (g, b))}
        if self.noisy:           # factor vectors [network][set][record] and effective blocks of the last fold
            out["noise"], out["eff"], out["eff_tgt"] = self.noise, self.eff, self.eff_tgt
        if self.dueling:         # the folded heads W3e[H][4] | b3e[4] of the last learn step, online (0) and target (1)
            dv = N.DuelingViews()
            N.check(self.lib.dmdqn_debug_dueling(C.byref(self.dims), _ptr(self.workspace), self.workspace.numel(), C.byref(dv)))
            out["head"] = view(dv.head, torch.float32, (2, g, 4 * self.hidden + 4))
        if self.hp.precision != 0:
            # the tcgen05 path keeps its activation scratch transposed ([feature][batch]) and never
            # materialises dh2: "dh2" is relu'(h2) as 0/1 here (its non-zero pattern is what the tests use)
            out["dh1"] = view(v.dh1, torch.float32, (g, self.hidden, b)).transpose(1, 2)
            bits = view(v.relu2_bits, torch.int32, (g, b, self.hidden // 32))      # [network][batch row][word]
            sh = torch.arange(32, device=bits.device, dtype=torch.int32).view(1, 1, 1, 32)
            out["dh2"] = ((bits.unsqueeze(3) >> sh) & 1).reshape(g, b, self.hidden).float()
        else:
            out["dh1"] = view(v.dh1, torch.float32, (g, b, self.hidden))
            out["dh2"] = view(v.dh2, torch.float32, (g, b, self.hidden))
        return out

    @_on_device
    def sync_target(self, mask=None, tau: float | None = None) -> None:
        """update_target_network (tau None, dqn_agent.py:382-384) / soft update (:389-399)."""
        mask_t = None if mask is None else self._dev(mask, torch.uint8)
        tau = -1.0 if tau is None else float(tau)
        if self.noisy:           # mu and sigma
            N.check(self.lib.dmdqn_sync_target_noisy(C.byref(self.dims), C.byref(self.nets), C.byref(self.noisy_ptrs),
                                                     int(self.dueling), _ptr(mask_t), tau, self._stream))
            return
        sync = self.lib.dmdqn_sync_target_dueling if self.dueling else self.lib.dmdqn_sync_target
        N.check(sync(C.byref(self.dims), C.byref(self.nets), _ptr(mask_t), tau, self._stream))
