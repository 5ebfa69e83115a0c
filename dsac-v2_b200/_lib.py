"""ctypes binding of libdsact.so (C ABI declared in include/dsact.h).

The CUDA library is the product; there is no CPU fallback.  Importing this
module without the built library raises, and so does every call on a machine
without a CUDA device.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# DSACT_LIB: kernel-development aid (A/B of two builds on one GPU box); the product is libdsact.so beside this file
LIB_PATH = os.environ.get("DSACT_LIB") or os.path.join(_HERE, "libdsact.so")

ABI_VERSION = 1
MAX_HIDDEN = 6
NUM_STATS = 16

ACTIVATIONS = {"linear": 0, "relu": 1, "gelu": 2, "tanh": 3, "sigmoid": 4, "elu": 5, "selu": 6}
GEMM_MODES = {"fp32": 0, "bf16x3": 1, "bf16": 2}
ACT_DISTS = {"TanhGaussDistribution": 0, "GaussDistribution": 1}   # utils/act_distribution_cls.py

# state slots, include/dsact.h
STATE_STDSUM = 4
STATE_ACC = 16
STATE_STATS = 48


class Config(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("obs_dim", C.c_int32), ("act_dim", C.c_int32),
        ("n_hidden_q", C.c_int32), ("n_hidden_pi", C.c_int32),
        ("hidden_q", C.c_int32 * MAX_HIDDEN), ("hidden_pi", C.c_int32 * MAX_HIDDEN),
        ("act_q", C.c_int32), ("act_pi", C.c_int32), ("max_batch", C.c_int32),
        ("auto_alpha", C.c_int32), ("delay_update", C.c_int32), ("gemm_mode", C.c_int32),
        ("use_graph", C.c_int32), ("act_dist", C.c_int32),
        ("gamma", C.c_double), ("tau", C.c_double), ("tau_b", C.c_double), ("alpha_fixed", C.c_double),
        ("lr_q", C.c_double), ("lr_pi", C.c_double), ("lr_alpha", C.c_double),
        ("min_log_std", C.c_double), ("max_log_std", C.c_double),
        ("adam_beta1", C.c_double), ("adam_beta2", C.c_double), ("adam_eps", C.c_double),
    ]


MAX_CONV = 8


class CnnConfig(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("channels", C.c_int32), ("height", C.c_int32), ("width", C.c_int32),
        ("act_dim", C.c_int32), ("n_conv", C.c_int32),
        ("conv_kernel", C.c_int32 * MAX_CONV), ("conv_channels", C.c_int32 * MAX_CONV), ("conv_stride", C.c_int32 * MAX_CONV),
        ("n_hidden", C.c_int32), ("hidden", C.c_int32 * MAX_HIDDEN), ("act_hidden", C.c_int32),
        ("max_batch", C.c_int32), ("auto_alpha", C.c_int32), ("delay_update", C.c_int32),
        ("q_heads", C.c_int32), ("act_dist", C.c_int32), ("pi_std", C.c_int32), ("algo", C.c_int32), ("v1_bound", C.c_int32),
        ("gamma", C.c_double), ("tau", C.c_double), ("tau_b", C.c_double), ("alpha_fixed", C.c_double),
        ("lr_q", C.c_double), ("lr_pi", C.c_double), ("lr_alpha", C.c_double),
        ("min_log_std", C.c_double), ("max_log_std", C.c_double),
        ("adam_beta1", C.c_double), ("adam_beta2", C.c_double), ("adam_eps", C.c_double), ("td_bound", C.c_double),
    ]


class Layout(C.Structure):
    _fields_ = [("n_q", C.c_int64), ("n_pi", C.c_int64), ("n_params", C.c_int64), ("n_targets", C.c_int64),
                ("workspace_bytes", C.c_int64), ("state_floats", C.c_int64), ("max_batch", C.c_int64)]


_fp = C.c_void_p  # device pointers travel as integers


class Buffers(C.Structure):
    _fields_ = [("params", _fp), ("targets", _fp), ("grads", _fp), ("adam_m", _fp), ("adam_v", _fp),
                ("act_high", _fp), ("act_low", _fp), ("state", _fp), ("workspace", _fp)]


class Batch(C.Structure):
    _fields_ = [("obs", _fp), ("act", _fp), ("rew", _fp), ("obs2", _fp), ("done", _fp), ("batch", C.c_int32),
                ("logp", _fp)]


class Noise(C.Structure):
    _fields_ = [("eps1", _fp), ("eps2", _fp), ("z3", _fp), ("z4", _fp)]


class Profile(C.Structure):
    _fields_ = [("ms", C.c_double * 4), ("flops", C.c_double * 4), ("launches", C.c_int32 * 4), ("total_ms", C.c_double)]


class Replay(C.Structure):
    _fields_ = [("obs", _fp), ("obs2", _fp), ("act", _fp), ("rew", _fp), ("done", _fp), ("logp", _fp),
                ("capacity", C.c_int64)]


class ReplayU8(C.Structure):
    """dsact_replay_u8: obs / obs2 hold one uint8 code per pixel (the pixel is float32(k) / 255)."""
    _fields_ = [("obs", _fp), ("obs2", _fp), ("act", _fp), ("rew", _fp), ("done", _fp), ("logp", _fp),
                ("capacity", C.c_int64)]


# every symbol include/dsact.h declares: (restype, argtypes)
IPC_HANDLE_BYTES = 64   # DSACT_IPC_HANDLE_BYTES
DP_MAX_RANKS = 8        # DSACT_DP_MAX_RANKS

SYMBOLS = {
    "dsact_last_error": (C.c_char_p, []),
    "dsact_abi_version": (C.c_int, []),
    "dsact_query_layout": (C.c_int, [C.POINTER(Config), C.POINTER(Layout)]),
    "dsact_create": (C.c_int, [C.POINTER(Config), C.c_int, C.POINTER(C.c_void_p)]),
    "dsact_destroy": (None, [C.c_void_p]),
    "dsact_bind": (C.c_int, [C.c_void_p, C.POINTER(Buffers)]),
    "dsact_seed": (C.c_int, [C.c_void_p, C.c_uint64]),
    "dsact_set_carry": (C.c_int, [C.c_void_p, C.c_float, C.c_float, C.c_int64, C.c_int64, C.c_void_p]),
    "dsact_step": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.POINTER(Noise), C.c_int64, C.c_void_p]),
    "dsact_step_host": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.POINTER(Noise), C.c_int64, C.c_void_p]),
    "dsact_stage_host": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.POINTER(Batch), C.c_void_p]),
    "dsact_stage_release": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dsact_grad_phase1": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.POINTER(Noise), C.c_void_p]),
    "dsact_grad_phase2": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p]),
    "dsact_compute_grads": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.POINTER(Noise), C.c_void_p]),
    "dsact_apply": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p]),
    "dsact_read_stats": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "dsact_replay_bind": (C.c_int, [C.c_void_p, C.POINTER(Replay)]),
    "dsact_replay_add": (C.c_int, [C.c_void_p] + [C.c_void_p] * 6 + [C.c_int64, C.c_int64, C.c_void_p]),
    "dsact_replay_sample": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.POINTER(Batch), C.c_void_p]),
    "dsact_replay_step": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.POINTER(Noise), C.c_int64, C.c_void_p]),
    "dsact_dp_export": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_int64)]),
    "dsact_dp_connect": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "dsact_dp_step": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.POINTER(Noise), C.c_int64, C.c_int64, C.c_void_p]),
    "dsact_dp_replay_step": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.POINTER(Noise), C.c_int64, C.c_int64,
                                       C.c_void_p]),
    "dsact_cnn_query_layout": (C.c_int, [C.POINTER(CnnConfig), C.POINTER(Layout)]),
    "dsact_cnn_create": (C.c_int, [C.POINTER(CnnConfig), C.c_int, C.POINTER(C.c_void_p)]),
    "dsact_cnn_destroy": (None, [C.c_void_p]),
    "dsact_cnn_bind": (C.c_int, [C.c_void_p, C.POINTER(Buffers)]),
    "dsact_cnn_set_carry": (C.c_int, [C.c_void_p, C.c_float, C.c_float, C.c_int64, C.c_int64, C.c_void_p]),
    "dsact_cnn_replay_bind": (C.c_int, [C.c_void_p, C.POINTER(Replay)]),
    "dsact_cnn_replay_add": (C.c_int, [C.c_void_p] + [C.c_void_p] * 6 + [C.c_int64, C.c_int64, C.c_void_p]),
    "dsact_cnn_replay_sample": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.POINTER(Batch), C.c_void_p]),
    "dsact_cnn_replay_bind_u8": (C.c_int, [C.c_void_p, C.POINTER(ReplayU8)]),
    "dsact_cnn_replay_add_u8": (C.c_int, [C.c_void_p] + [C.c_void_p] * 6 + [C.c_int64, C.c_int64, C.c_void_p]),
    "dsact_cnn_seed": (C.c_int, [C.c_void_p, C.c_uint64]),
    "dsact_cnn_step": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.POINTER(Noise), C.c_int64, C.c_void_p]),
    "dsact_cnn_grad_phase1": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.POINTER(Noise), C.c_void_p]),
    "dsact_cnn_grad_phase2": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p]),
    "dsact_cnn_compute_grads": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.POINTER(Noise), C.c_void_p]),
    "dsact_cnn_apply": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p]),
    "dsact_cnn_read_stats": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "dsact_profile_step": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.POINTER(Noise), C.c_int64, C.c_void_p, C.POINTER(Profile)]),
    "dsact_launch_count": (C.c_int64, [C.c_void_p]),
    "dsact_last_call_launches": (C.c_int32, [C.c_void_p]),
    "dsact_test_gemm": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p,
                                  C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
}

_lib = None


class DsactError(RuntimeError):
    pass


def load() -> C.CDLL:
    """dlopen libdsact.so and type every entry point.  Raises if it was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DsactError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no CPU fallback for the DSAC-T update path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.dsact_abi_version() != ABI_VERSION:
        raise DsactError(f"libdsact.so ABI {lib.dsact_abi_version()} != binding ABI {ABI_VERSION}")
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        raise DsactError(f"libdsact error {rc}: {load().dsact_last_error().decode()}")
