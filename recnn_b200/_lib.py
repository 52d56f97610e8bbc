"""ctypes binding of the C ABI in include/recnn_b200.h.

The library is mandatory: there is no CPU or eager-PyTorch fallback behind
these calls.  ``lib()`` raises if librecnn_b200.so is missing or was built from
different sources (run ``python -m recnn_b200.build`` or
``__graft_entry__.build()``).
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

PH_VALUE_GRAD, PH_VALUE_OPT, PH_POLICY_LOSS, PH_POLICY_GRAD, PH_POLICY_OPT, PH_SOFT_UPDATE, PH_GATHER = \
    1, 2, 4, 8, 16, 32, 64
PH_FINISH = 128
PH_ALL = 255
ALGO_DDPG, ALGO_TD3 = 0, 1
OPT_EXTERNAL, OPT_SGD, OPT_ADAM, OPT_RANGER = 0, 1, 2, 3
METRIC_L2, METRIC_IP, METRIC_COS = 0, 1, 2
REINFORCE_BASIC, REINFORCE_CORRECTED, REINFORCE_TOPK = 0, 1, 2


class Dims(C.Structure):
    _fields_ = [("state_dim", C.c_int32), ("action_dim", C.c_int32), ("hidden", C.c_int32),
                ("reserved", C.c_int32)]


class DiscreteDims(C.Structure):
    _fields_ = [("state_dim", C.c_int32), ("hidden", C.c_int32), ("num_items", C.c_int32), ("reserved", C.c_int32)]


class Net(C.Structure):
    _fields_ = [("params", C.c_void_p), ("grads", C.c_void_p), ("opt_m", C.c_void_p),
                ("opt_v", C.c_void_p), ("opt_t", C.c_void_p), ("opt_slow", C.c_void_p)]


class Optim(C.Structure):
    _fields_ = [("kind", C.c_int32), ("k", C.c_int32), ("lr", C.c_double), ("beta1", C.c_double),
                ("beta2", C.c_double), ("eps", C.c_double), ("weight_decay", C.c_double),
                ("momentum", C.c_double), ("alpha", C.c_double), ("n_sma_threshold", C.c_double)]


class StepArgs(C.Structure):
    _fields_ = [
        ("algo", C.c_int32), ("phases", C.c_int32), ("learn", C.c_int32), ("do_policy_step", C.c_int32),
        ("dims", Dims),
        ("n_rows", C.c_int64), ("n_rows_global", C.c_int64),
        ("state", C.c_void_p), ("next_state", C.c_void_p), ("action", C.c_void_p),
        ("table", C.c_void_p), ("n_items", C.c_int64), ("frame", C.c_int32), ("emb_dim", C.c_int32),
        ("items", C.c_void_p), ("ratings", C.c_void_p), ("reward", C.c_void_p), ("done", C.c_void_p),
        ("policy", Net), ("target_policy", Net), ("value", Net * 2), ("target_value", Net * 2),
        ("policy_optim", Optim), ("value_optim", Optim),
        ("gamma", C.c_float), ("min_value", C.c_float), ("max_value", C.c_float),
        ("noise_std", C.c_float), ("noise_clip", C.c_float), ("dropout", C.c_int32),
        ("soft_tau", C.c_double),
        ("masks", C.c_void_p * 8), ("noise", C.c_void_p), ("seed", C.c_uint64), ("rng_step", C.c_void_p),
        ("losses", C.c_void_p), ("losses_host", C.c_void_p), ("next_action_out", C.c_void_p), ("gen_action_out", C.c_void_p),
        ("next_action_in", C.c_void_p),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_int64),
        ("comm", C.c_void_p),
    ]


_PROBE_FIELDS = ["dims", "n_rows", "table", "policy", "policy_optim", "gamma", "soft_tau", "masks", "seed",
                 "losses", "workspace_bytes", "comm"]

# name -> (restype, argtypes); every symbol include/recnn_b200.h declares
SIGNATURES = {
    "recnn_b200_abi_version": (C.c_int, []),
    "recnn_b200_last_error": (C.c_char_p, []),
    "recnn_b200_launch_count": (C.c_int64, []),
    "recnn_sizeof_step_args": (C.c_int64, []),
    "recnn_offsetof_step_args": (C.c_int64, [C.c_int]),
    "recnn_frame_gather": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "recnn_done_from_sizes": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int64, C.c_void_p]),
    "recnn_window_gather_users": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                            C.c_int64, C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_void_p]),
    "recnn_window_gather_ids": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p,
                                          C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p]),
    "recnn_actor_param_count": (C.c_int64, [C.POINTER(Dims)]),
    "recnn_critic_param_count": (C.c_int64, [C.POINTER(Dims)]),
    "recnn_net_layout": (C.c_int, [C.POINTER(Dims), C.c_int, C.POINTER(C.c_int64)]),
    "recnn_forward_scratch_floats": (C.c_int64, [C.POINTER(Dims), C.c_int64, C.c_int]),
    "recnn_actor_forward": (C.c_int, [C.POINTER(Dims), C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                      C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "recnn_critic_forward": (C.c_int, [C.POINTER(Dims), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "recnn_linear_forward": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                       C.c_void_p, C.c_void_p]),
    "recnn_gemm_tf32x3": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int64,
                                    C.c_int, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "recnn_gemm_fp32": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int64,
                                  C.c_int, C.c_void_p, C.c_int64, C.c_void_p]),
    "recnn_polyak_update": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_double, C.c_void_p]),
    "recnn_step_workspace_bytes": (C.c_int64, [C.POINTER(Dims), C.c_int64, C.c_int32]),
    "recnn_ddpg_step": (C.c_int, [C.POINTER(StepArgs), C.c_void_p]),
    "recnn_td3_step": (C.c_int, [C.POINTER(StepArgs), C.c_void_p]),
    "recnn_optimizer_step": (C.c_int, [C.POINTER(Optim), C.POINTER(Net), C.c_int64, C.c_void_p, C.c_void_p]),
    "recnn_item_norms": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "recnn_retrieve_workspace_bytes": (C.c_int64, [C.c_int64, C.c_int64, C.c_int32]),
    "recnn_retrieve_topk": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32,
                                      C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "recnn_discrete_layout": (C.c_int, [C.POINTER(DiscreteDims), C.POINTER(C.c_int64)]),
    "recnn_discrete_scratch_floats": (C.c_int64, [C.POINTER(DiscreteDims), C.c_int64, C.c_int32]),
    "recnn_discrete_forward": (C.c_int, [C.POINTER(DiscreteDims), C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p,
                                         C.c_void_p, C.c_void_p]),
    "recnn_categorical_sample": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_void_p, C.c_uint64,
                                           C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "recnn_categorical_log_prob": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p]),
    "recnn_reinforce_policy_grad": (C.c_int, [C.POINTER(DiscreteDims), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p,
                                              C.c_void_p, C.c_void_p]),
    "recnn_reinforce_streamed_scratch_floats": (C.c_int64, [C.POINTER(DiscreteDims), C.c_int64, C.c_int32]),
    "recnn_reinforce_policy_grad_streamed": (C.c_int, [C.POINTER(DiscreteDims), C.c_void_p, C.c_void_p, C.c_void_p,
                                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32,
                                                       C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "recnn_comm_create": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, C.POINTER(C.c_void_p)]),
    "recnn_comm_handle_bytes": (C.c_int32, []),
    "recnn_comm_local_handle": (C.c_int, [C.c_void_p, C.c_void_p]),
    "recnn_comm_connect": (C.c_int, [C.c_void_p, C.c_void_p]),
    "recnn_comm_allreduce": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "recnn_comm_destroy": (C.c_int, [C.c_void_p]),
}

_LIB = None


class RecnnError(RuntimeError):
    pass


def lib_path() -> str:
    return _build.LIB


def lib():
    """The loaded shared library (built on first use if a compiler is present)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.isfile(path):
        try:
            _build.build()
        except Exception as exc:  # no silent fallback: the CUDA library is the product
            raise RecnnError("librecnn_b200.so is missing and could not be built: %s" % exc) from exc
    handle = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(handle, name)
        except AttributeError as exc:
            raise RecnnError("librecnn_b200.so does not export %s (stale build?)" % name) from exc
        fn.restype = res
        fn.argtypes = args
    if handle.recnn_sizeof_step_args() != C.sizeof(StepArgs):
        raise RecnnError("recnn_step_args layout mismatch: C %d bytes, ctypes %d bytes"
                         % (handle.recnn_sizeof_step_args(), C.sizeof(StepArgs)))
    for i, f in enumerate(_PROBE_FIELDS):
        if handle.recnn_offsetof_step_args(i) != getattr(StepArgs, f).offset:
            raise RecnnError("recnn_step_args.%s offset mismatch" % f)
    _LIB = handle
    return handle


def check(status: int):
    if status != 0:
        msg = lib().recnn_b200_last_error()
        raise RecnnError("recnn_b200 call failed (%d): %s" % (status, (msg or b"").decode()))


def ptr(t):
    """Device/host pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def stream_ptr(device=None):
    import torch
    return torch.cuda.current_stream(device).cuda_stream
