"""ctypes binding of libsacb200.so (C ABI declared in include/sacb200.h).

There is NO CPU fallback: importing works anywhere (so the "library loads and exports every symbol"
check can run on a CPU box) but every compute entry point needs a B200; `create` raises otherwise.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SACB_LIB") or os.path.join(_HERE, "libsacb200.so")      # SACB_LIB: an experiment build of the same sources (A/B timing)

c_f32p = ctypes.POINTER(ctypes.c_float)
c_f64p = ctypes.POINTER(ctypes.c_double)
c_i64p = ctypes.POINTER(ctypes.c_int64)

OK, ERR_ARG, ERR_DEVICE, ERR_STATE, ERR_NOMEM = 0, -1, -2, -3, -4
MATH_FP32, MATH_BF16X3 = 0, 1
LAUNCH_STAGED, LAUNCH_PERSISTENT = 0, 1
NET_POLICY, NET_Q1, NET_Q2, NET_Q1_TARGET, NET_Q2_TARGET = range(5)
SLOT_PARAM, SLOT_ADAM_M, SLOT_ADAM_V, SLOT_GRAD = range(4)
REPLAY_UNIFORM, REPLAY_PER = 0, 1
USE_LAST_SAMPLE, NO_LOSS_READBACK, EXPORT_GRADS, DEVICE_INDICES, WRITE_BACK_TD = 1, 2, 4, 8, 16


class Config(ctypes.Structure):
    _fields_ = [
        ("obs_dim", ctypes.c_int32), ("act_dim", ctypes.c_int32), ("hidden_dim", ctypes.c_int32), ("n_hidden", ctypes.c_int32),
        ("gamma", ctypes.c_float), ("tau", ctypes.c_float), ("lr", ctypes.c_float), ("alpha0", ctypes.c_float),
        ("auto_entropy", ctypes.c_int32), ("action_scale", ctypes.c_float), ("action_bias", ctypes.c_float),
        ("replay_kind", ctypes.c_int32), ("capacity", ctypes.c_int64),
        ("per_alpha", ctypes.c_float), ("per_beta_start", ctypes.c_float), ("per_beta_frames", ctypes.c_int64),
        ("max_batch", ctypes.c_int32), ("n_agents", ctypes.c_int32), ("math_mode", ctypes.c_int32), ("launch_mode", ctypes.c_int32),
        ("device", ctypes.c_int32), ("seed", ctypes.c_uint64), ("per_weighted_loss", ctypes.c_int32), ("layer_norm", ctypes.c_int32), ("reserved", ctypes.c_int32 * 6),
    ]


class Scalars(ctypes.Structure):
    _fields_ = [("log_alpha", ctypes.c_float), ("alpha", ctypes.c_float), ("log_alpha_m", ctypes.c_float), ("log_alpha_v", ctypes.c_float),
                ("step_policy", ctypes.c_int64), ("step_q1", ctypes.c_int64), ("step_q2", ctypes.c_int64), ("step_alpha", ctypes.c_int64),
                ("n_updates", ctypes.c_int64), ("act_counter", ctypes.c_int64)]


class PerStats(ctypes.Structure):
    _fields_ = [("frame", ctypes.c_int64), ("pos", ctypes.c_int64), ("len", ctypes.c_int64), ("n_fine", ctypes.c_int64),
                ("n_flagged", ctypes.c_int64), ("n_exact_fallbacks", ctypes.c_int64), ("total_f32", ctypes.c_float), ("cdf_last", ctypes.c_double)]


class Stats(ctypes.Structure):
    _fields_ = [("kernel_launches", ctypes.c_int64), ("n_stages", ctypes.c_int32), ("n_tasks", ctypes.c_int32), ("n_tiles", ctypes.c_int32),
                ("grid", ctypes.c_int32), ("block", ctypes.c_int32), ("smem_bytes", ctypes.c_int32), ("sm_count", ctypes.c_int32),
                ("n_programs", ctypes.c_int32)]


class Hparams(ctypes.Structure):
    _fields_ = [("lr", ctypes.c_float), ("gamma", ctypes.c_float), ("tau", ctypes.c_float), ("target_entropy", ctypes.c_float)]


H = ctypes.c_void_p
I, I64, U32 = ctypes.c_int, ctypes.c_int64, ctypes.c_uint32

# name -> (restype, argtypes): every symbol include/sacb200.h declares
SIGNATURES = {
    "sacb_default_config": (None, [ctypes.POINTER(Config)]),
    "sacb_last_error": (ctypes.c_char_p, []),
    "sacb_version": (ctypes.c_char_p, []),
    "sacb_device_count": (I, []),
    "sacb_create": (I, [ctypes.POINTER(Config), ctypes.POINTER(H)]),
    "sacb_destroy": (I, [H]),
    "sacb_synchronize": (I, [H]),
    "sacb_num_tensors": (I, [H, I]),
    "sacb_tensor_info": (I, [H, I, I, c_i64p, c_i64p, c_i64p]),
    "sacb_tensor_dev": (I, [H, I, I, I, I, ctypes.POINTER(ctypes.c_void_p)]),
    "sacb_import_tensor": (I, [H, I, I, I, I, c_f32p, I64]),
    "sacb_export_tensor": (I, [H, I, I, I, I, c_f32p, I64]),
    "sacb_get_scalars": (I, [H, I, ctypes.POINTER(Scalars)]),
    "sacb_set_scalars": (I, [H, I, ctypes.POINTER(Scalars)]),
    "sacb_set_lr": (I, [H, ctypes.c_float]),
    "sacb_get_hparams": (I, [H, I, ctypes.POINTER(Hparams)]),
    "sacb_set_hparams": (I, [H, I, ctypes.POINTER(Hparams)]),
    "sacb_copy_agents": (I, [H, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32), I]),
    "sacb_invalidate_shadows": (I, [H]),
    "sacb_push": (I, [H, I, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, I64]),
    "sacb_push_rows": (I, [H, I, c_f32p, I64]),
    "sacb_row_floats": (I64, [H]),
    "sacb_host_first_distinct": (I64, [ctypes.c_char_p, I64, ctypes.c_uint64, I, c_i64p, I64, I64]),      # words: a bytes object, passed without a copy
    "sacb_len": (I64, [H, I]),
    "sacb_read_transitions": (I, [H, I, c_i64p, I64, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p]),
    "sacb_clear_replay": (I, [H, I]),
    "sacb_sample_uniform": (I, [H, I, c_i64p, I64, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p]),
    "sacb_per_sample": (I, [H, I, c_f64p, I64, c_i64p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p]),
    "sacb_per_sample_all": (I, [H, c_f64p, I64, c_i64p, c_f32p]),
    "sacb_per_update": (I, [H, I, c_i64p, c_f32p, I64]),
    "sacb_per_update_final": (I, [H, I, c_i64p, c_f32p, I64]),
    "sacb_per_update_from_td": (I, [H, I, I64]),
    "sacb_per_step": (I, [H, I64, c_f32p, U32]),
    "sacb_per_get_priorities": (I, [H, I, c_f32p, I64]),
    "sacb_per_set_priorities": (I, [H, I, c_f32p, c_f32p, I64]),
    "sacb_per_get_stats": (I, [H, I, ctypes.POINTER(PerStats)]),
    "sacb_per_set_frame": (I, [H, I, I64]),
    "sacb_update": (I, [H, I64, c_i64p, c_f32p, c_f32p, c_f32p, U32]),
    "sacb_update_steps": (I, [H, I64, I, c_f32p, U32]),
    "sacb_update_batch": (I, [H, I64, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, U32]),
    "sacb_stage_indices": (I, [H, c_i64p, I64, I64]),
    "sacb_get_losses": (I, [H, I, c_f32p]),
    "sacb_get_losses_all": (I, [H, c_f32p]),
    "sacb_select_action": (I, [H, I, c_f32p, I, c_f32p, c_f32p]),
    "sacb_select_action_batch": (I, [H, c_f32p, I, c_f32p, c_f32p]),
    "sacb_q_forward": (I, [H, I, I, c_f32p, c_f32p, I64, c_f32p]),
    "sacb_policy_forward": (I, [H, I, c_f32p, I64, c_f32p, c_f32p]),
    "sacb_policy_sample": (I, [H, I, c_f32p, I64, c_f32p, c_f32p, c_f32p]),
    "sacb_dp_backward": (I, [H, I, I64, c_i64p, c_f32p, c_f32p]),
    "sacb_dp_apply": (I, [H, I]),
    "sacb_dp_ipc_handle": (I, [H, ctypes.c_void_p]),
    "sacb_dp_connect": (I, [H, I, I, ctypes.c_void_p]),
    "sacb_dp_exchange_apply": (I, [H, I]),
    "sacb_dp_get_losses": (I, [H, c_f32p]),
    "sacb_dp_grad_buffer": (I, [H, I, ctypes.POINTER(ctypes.c_void_p), c_i64p]),
    "sacb_get_stream": (I, [H, ctypes.POINTER(ctypes.c_void_p)]),
    "sacb_get_stats": (I, [H, ctypes.POINTER(Stats)]),
    "sacb_timer_start": (I, [H]),
    "sacb_timer_stop": (I, [H, c_f32p]),
    "sacb_time_update": (I, [H, I64, I, c_f32p]),
    "sacb_time_stages": (I, [H, I64, c_f32p, I]),
    "sacb_debug_read_slots": (I, [H, I, ctypes.POINTER(ctypes.c_int32), I64]),
    "sacb_debug_read_activation": (I, [H, I, I, I, I, I64, c_f32p]),
    "sacb_selftest_gemm": (I, [I, I, I, I, I, I, I, c_f32p]),
    "sacb_selftest_gemm_stream": (I, [I, I, I, I, I, I, I, I, I, c_f32p]),
    "sacb_selftest_gemm_tile": (I, [I, I, I, I, I, I, I, I, I, c_f32p]),
}

_lib = None


def lib():
    """Loads the CUDA library; fails loudly (no CPU path exists) if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python humanoid-walking-with-sac_b200/build.py` "
                "(nvcc, sm_100a). This package has no CPU or PyTorch fallback.")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)      # AttributeError here = header / library mismatch
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


class SacbError(RuntimeError):
    pass


def check(rc):
    if rc >= 0:
        return rc
    msg = lib().sacb_last_error().decode()
    if rc in (ERR_ARG, ERR_STATE):
        raise ValueError(msg)
    if rc == ERR_NOMEM:
        raise MemoryError(msg)
    raise SacbError(msg)


def f32(a):
    """C-contiguous float32 view/copy of an array-like (the cast of sac_imp.py:81-85)."""
    return np.ascontiguousarray(a, dtype=np.float32)


def ptr(a, ctype=ctypes.c_float):
    # ctypes.cast on the raw address: about 3x cheaper than ndarray.ctypes.data_as, and this sits on the per-step path
    if a is None:
        return None
    p = ctypes.cast(a.__array_interface__["data"][0], ctypes.POINTER(ctype))
    p._owner = a      # keeps a temporary array alive for as long as the pointer object lives (what data_as does)
    return p


def default_config():
    c = Config()
    lib().sacb_default_config(ctypes.byref(c))
    return c


def create(cfg):
    h = H()
    check(lib().sacb_create(ctypes.byref(cfg), ctypes.byref(h)))
    return h


class DevArray:
    """Zero-copy view of device memory for torch.as_tensor (CUDA array interface v3)."""

    def __init__(self, ptr_value, shape, owner):
        self._owner = owner      # keeps the handle alive
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<f4", "data": (int(ptr_value), False), "version": 3, "strides": None}
