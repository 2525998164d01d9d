"""ctypes binding of libdmdqn_b200.so (include/dmdqn_b200.h).  Loading fails loudly: the
product path has no CPU or PyTorch fallback."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libdmdqn_b200.so")

OK, ERR_ARG, ERR_CUDA, ERR_WORKSPACE = 0, -1, -2, -3
LOSS = {"mse": 0, "huber": 1}
SAMPLE = {"indices": 0, "fisher_yates": 1, "replacement": 2, "prioritized": 3}
PER_MAX_CAPACITY = 8192 * 128
MAX_NSTEP = 16
ADAM = {"keras": 0, "torch": 1}
PRECISION = {"fp32": 0, "tf32": 1, "tf32x3": 2}
METRICS_STRIDE = 8


class Dims(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("n_agents", "n_nets", "obs_dim", "obs_stride", "hidden",
                                          "n_actions", "batch", "capacity")]


class Layout(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("w1", "b1", "w2", "b2", "w3", "b3", "stride")]


class DuelingLayout(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("w1", "b1", "w2", "b2", "w3", "b3", "wv", "bv", "stride")]


class Replay(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("obs", "next_obs", "act", "rew", "done", "n_written", "priority", "priority_max")]


class Nets(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("theta", "theta_tgt", "adam_m", "adam_v", "learn_step")]


class HParams(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("gamma", "learning_rate", "beta1", "beta2", "adam_eps", "tau")] + \
               [(n, C.c_int32) for n in ("target_update_frequency", "loss", "normalize_rewards", "double_dqn",
                                         "adam_form", "sample_mode", "precision")] + \
               [("dueling", C.c_int32)] + \
               [(n, C.c_double) for n in ("per_alpha", "per_beta0", "per_eps")] + [("per_beta_steps", C.c_int32)] + \
               [("n_step", C.c_int32)]      # in what was tail padding: sizeof stays 112
    # dueling sits at offset 76 (interior padding), between precision and per_alpha.  It is keyword-only, so positional
    # constructions keep the order of every field before it; later fields are keyword-only as well.
    _ARGS = ("gamma", "learning_rate", "beta1", "beta2", "adam_eps", "tau", "target_update_frequency", "loss",
             "normalize_rewards", "double_dqn", "adam_form", "sample_mode", "precision", "per_alpha", "per_beta0", "per_eps",
             "per_beta_steps", "n_step")

    def __init__(self, *args, **kwargs):
        if len(args) > len(self._ARGS):
            raise TypeError(f"HParams takes at most {len(self._ARGS)} positional arguments; dueling is keyword-only")
        super().__init__(**dict(zip(self._ARGS, args)), **kwargs)


assert C.sizeof(HParams) == 112 and HParams.dueling.offset == 76, "dmdqn_hparams layout (include/dmdqn_b200.h)"


class DebugViews(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("y", "q_all", "q_next", "tq_all", "rows", "r_hat", "active", "tc_error", "dh1", "dh2", "relu2_bits", "is_w")]


class NStepViews(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("next_rows", "discount")]


class DuelingViews(C.Structure):
    _fields_ = [("head", C.c_void_p)]


class Noisy(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("sigma", "sigma_tgt", "sigma_m", "sigma_v", "eff", "eff_tgt", "noise", "key")]


class NoiseRecord(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("w1_in", "w1_out", "w2_in", "w2_out", "w3_in", "w3_out", "v_in", "v_out", "stride")]


MAX_PEERS, PEER_BLOCKS, PEER_TIMEOUT = 8, 128, 77


class Peers(C.Structure):
    _fields_ = [("grads", C.c_void_p * MAX_PEERS), ("loss", C.c_void_p * MAX_PEERS), ("flags", C.c_void_p * MAX_PEERS),
                ("rank", C.c_int32), ("world", C.c_int32), ("epoch", C.c_uint32)]


class StepBlock(C.Structure):
    _fields_ = [(n, C.c_size_t) for n in ("bytes", "obs_off", "next_obs_off", "act_off", "rew_off", "done_off", "draws_off")] + \
               [("in_stride", C.c_int32)]


# name -> (restype, argtypes); mirrors include/dmdqn_b200.h one to one
_P = C.c_void_p
SIGNATURES = {
    "dmdqn_last_error": (C.c_char_p, []),
    "dmdqn_abi_version": (C.c_int, []),
    "dmdqn_param_layout": (C.c_int, [C.POINTER(Dims), C.POINTER(Layout)]),
    "dmdqn_param_layout_dueling": (C.c_int, [C.POINTER(Dims), C.POINTER(DuelingLayout)]),
    "dmdqn_workspace_bytes": (C.c_int, [C.POINTER(Dims), C.POINTER(C.c_size_t)]),
    "dmdqn_featurize": (C.c_int, [C.c_int32, _P, _P, _P, _P, C.c_double, _P, _P, _P, _P, C.c_double,
                                  C.c_double, _P, _P, C.c_int32, _P, _P, _P, _P]),
    "dmdqn_featurize_alt": (C.c_int, [C.c_int32, _P, _P, _P, _P, C.c_double, _P, _P, _P, _P, C.c_int32, _P, _P]),
    "dmdqn_act": (C.c_int, [C.POINTER(Dims), C.POINTER(Nets), _P, C.c_int32, _P, _P, _P, _P, _P, _P]),
    "dmdqn_act_dueling": (C.c_int, [C.POINTER(Dims), C.POINTER(Nets), _P, C.c_int32, _P, _P, _P, _P, _P, _P]),
    "dmdqn_push": (C.c_int, [C.POINTER(Dims), C.POINTER(Replay), _P, _P, _P, _P, _P, C.c_int32, _P, _P]),
    "dmdqn_sample": (C.c_int, [C.POINTER(Dims), C.POINTER(HParams), C.POINTER(Replay), C.POINTER(Nets), _P, _P,
                               C.c_int32, _P, C.c_size_t, _P]),
    "dmdqn_gather": (C.c_int, [C.POINTER(Dims), C.POINTER(Replay), _P, C.c_size_t, _P, _P, _P, _P, _P, _P, _P]),
    "dmdqn_learn": (C.c_int, [C.POINTER(Dims), C.POINTER(HParams), C.POINTER(Replay), C.POINTER(Nets), _P, _P,
                              _P, _P, C.c_size_t, _P]),
    "dmdqn_learn_stages": (C.c_int, [C.POINTER(Dims), C.POINTER(HParams), C.POINTER(Replay), C.POINTER(Nets), _P, _P,
                                     _P, _P, C.c_size_t, C.c_int32, _P]),
    "dmdqn_step_host": (C.c_int, [C.POINTER(Dims), C.POINTER(HParams), C.POINTER(Replay), C.POINTER(Nets), C.POINTER(StepBlock),
                                 _P, _P, _P, _P, _P, C.c_size_t, _P]),
    "dmdqn_learn_grads": (C.c_int, [C.POINTER(Dims), C.POINTER(HParams), C.POINTER(Replay), C.POINTER(Nets), _P, _P,
                                    C.c_int32, _P, _P, _P, C.c_size_t, _P]),
    "dmdqn_adam_apply": (C.c_int, [C.POINTER(Dims), C.POINTER(HParams), C.POINTER(Nets), _P, _P, C.c_size_t, _P]),
    "dmdqn_clip_adam_apply": (C.c_int, [C.POINTER(Dims), C.POINTER(HParams), C.POINTER(Nets), _P, C.c_double, _P, _P,
                                        C.c_size_t, _P]),
    "dmdqn_allreduce_adam":(C.c_int, [C.POINTER(Dims), C.POINTER(HParams), C.POINTER(Nets), C.POINTER(Peers), _P, _P, _P,
                                       C.c_size_t, _P]),
    "dmdqn_ipc_export": (C.c_int, [_P, _P, C.POINTER(C.c_uint64)]),
    "dmdqn_ipc_open": (C.c_int, [_P, C.c_uint64, C.POINTER(C.c_void_p)]),
    "dmdqn_ipc_close": (C.c_int, [_P, C.c_uint64]),
    "dmdqn_debug": (C.c_int, [C.POINTER(Dims), _P, C.c_size_t, C.POINTER(DebugViews)]),
    "dmdqn_debug_nstep": (C.c_int, [C.POINTER(Dims), _P, C.c_size_t, C.POINTER(NStepViews)]),
    "dmdqn_debug_dueling": (C.c_int, [C.POINTER(Dims), _P, C.c_size_t, C.POINTER(DuelingViews)]),
    "dmdqn_sync_target": (C.c_int, [C.POINTER(Dims), C.POINTER(Nets), _P, C.c_double, _P]),
    "dmdqn_sync_target_dueling": (C.c_int, [C.POINTER(Dims), C.POINTER(Nets), _P, C.c_double, _P]),
    "dmdqn_noise_layout": (C.c_int, [C.POINTER(Dims), C.POINTER(NoiseRecord)]),
    "dmdqn_noisy_fold": (C.c_int, [C.POINTER(Dims), C.POINTER(HParams), C.POINTER(Nets), C.POINTER(Noisy), _P]),
    "dmdqn_learn_grads_noisy": (C.c_int, [C.POINTER(Dims), C.POINTER(HParams), C.POINTER(Replay), C.POINTER(Nets),
                                          C.POINTER(Noisy), _P, _P, C.c_int32, _P, _P, _P, C.c_size_t, _P]),
    "dmdqn_noisy_adam_apply": (C.c_int, [C.POINTER(Dims), C.POINTER(HParams), C.POINTER(Nets), C.POINTER(Noisy), _P, _P,
                                         C.c_size_t, _P]),
    "dmdqn_act_noisy": (C.c_int, [C.POINTER(Dims), C.POINTER(Nets), C.POINTER(Noisy), C.c_int32, _P, C.c_int32, _P, _P, _P,
                                  _P, _P, _P]),
    "dmdqn_sync_target_noisy": (C.c_int, [C.POINTER(Dims), C.POINTER(Nets), C.POINTER(Noisy), C.c_int32, _P, C.c_double, _P]),
}

_lib = None


class NativeError(RuntimeError):
    pass


def lib() -> C.CDLL:
    """The loaded library; raises if it has not been built (``python -m dmdqn_b200.build``)."""
    global _lib
    if _lib is None:
        path = LIB_PATH
        prof = os.environ.get("DMDQN_PROFILING_LIB")  # phase-stamp / debug builds live in their own file (build.py); never the default
        if prof:
            path = os.path.join(os.path.dirname(LIB_PATH), prof if prof.endswith(".so") else "libdmdqn_b200_timing.so")
        if not os.path.exists(path):
            raise NativeError(
                f"{path} is missing: build it with `python -m dmdqn_b200.build` "
                "(nvcc, sm_100a). dmdqn_b200 has no CPU fallback.")
        handle = C.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the .so does not export it
            fn.restype, fn.argtypes = res, args
        if handle.dmdqn_abi_version() != 3:      # 3: + prioritized replay fields at the end of the replay / hparams / debug structs
            raise NativeError("libdmdqn_b200.so ABI version mismatch: rebuild")
        _lib = handle
    return _lib


def check(rc: int) -> None:
    if rc != OK:
        msg = lib().dmdqn_last_error().decode("utf-8", "replace")
        raise NativeError(f"dmdqn_b200 native call failed ({rc}): {msg}")
