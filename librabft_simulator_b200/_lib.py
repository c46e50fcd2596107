"""ctypes binding of the C ABI declared in ``include/lbft.h`` (the product's only native entry).

There is deliberately no fallback: if ``csrc/liblbft_b200.so`` is missing or no CUDA device is usable,
importing this module / creating a simulator raises.
"""
import ctypes
import os

from ._build import LIB_PATH

c_u32, c_u64, c_i32, c_i64, c_f64 = ctypes.c_uint32, ctypes.c_uint64, ctypes.c_int32, ctypes.c_int64, ctypes.c_double


class LbftConfig(ctypes.Structure):
    """``lbft_config`` of include/lbft.h (field order and types must match exactly)."""
    _fields_ = [
        ("struct_size", c_u32), ("num_instances", c_u32), ("num_nodes", c_u32), ("delay_kind", c_u32),
        ("seeds", ctypes.c_void_p), ("max_clock", c_i64), ("delay_mean", c_f64), ("delay_variance", c_f64),
        ("delay_lo", c_i64), ("delay_hi", c_i64), ("target_commit_interval", c_i64), ("delta", c_i64),
        ("gamma", c_f64), ("lambda_", c_f64), ("commands_per_epoch", c_u64), ("voting_rights", ctypes.c_void_p),
        ("silent", ctypes.c_void_p), ("partition_windows", c_u32), ("partition_max_len", c_u32),
        ("device", c_i32), ("round_cap", c_u32), ("queue_cap", c_u32), ("payload_cap", c_u32),
        ("flags", c_u32), ("reserved", c_u32),
    ]


class LbftParamSet(ctypes.Structure):
    """``lbft_param_set`` of include/lbft.h: one parameter set of a sweep (``lbft_create_sweep``)."""
    _fields_ = [
        ("struct_size", c_u32), ("delay_kind", c_u32), ("delay_mean", c_f64), ("delay_variance", c_f64),
        ("delay_lo", c_i64), ("delay_hi", c_i64), ("target_commit_interval", c_i64), ("delta", c_i64),
        ("gamma", c_f64), ("lambda_", c_f64), ("silent_mask", c_u64),
    ]


MAX_PARAM_SETS = 4096  # LBFT_MAX_PARAM_SETS


class LbftCommit(ctypes.Structure):
    _fields_ = [("proposer", c_u32), ("index", c_u32), ("time", c_i64)]


class LbftRoundSwitch(ctypes.Structure):
    """include/lbft.h lbft_round_switch (data_writer.rs:14)"""
    _fields_ = [("node", c_u32), ("round", c_u32), ("time", c_i64)]


FLAG_ROUND_SWITCHES = 1  # LBFT_FLAG_ROUND_SWITCHES
FLAG_RESUMABLE = 2  # LBFT_FLAG_RESUMABLE
FLAG_TRUE_DATA_SYNC = 4  # LBFT_FLAG_TRUE_DATA_SYNC (non-parity variant)


class LbftTiming(ctypes.Structure):
    _fields_ = [("init_ms", c_f64), ("sim_ms", c_f64), ("finalize_ms", c_f64), ("h2d_ms", c_f64), ("d2h_ms", c_f64),
                ("h2d_bytes", c_u64), ("d2h_bytes", c_u64), ("kernel_launches", c_u32), ("reserved", c_u32)]


LBFT_OK = 0
LBFT_ERR_CAPACITY = -4
ST_DONE, ST_ROUND_OVERFLOW, ST_QUEUE_OVERFLOW, ST_PAYLOAD_OVERFLOW = 1, 2, 4, 8
ST_INVARIANT, ST_EPOCH_CHANGE, ST_DELAY_NEAR_INT, ST_TIME_OVERFLOW = 16, 32, 64, 128
ST_ERROR_MASK = ST_ROUND_OVERFLOW | ST_QUEUE_OVERFLOW | ST_PAYLOAD_OVERFLOW | ST_INVARIANT | ST_TIME_OVERFLOW

EXPORTS = [
    "lbft_create", "lbft_create_sweep", "lbft_run", "lbft_run_async", "lbft_wait", "lbft_commit_logs", "lbft_upload", "lbft_run_device", "lbft_download", "lbft_commit_counts",
    "lbft_last_states", "lbft_commit_log", "lbft_round_switches", "lbft_active_rounds", "lbft_counters", "lbft_status", "lbft_timing_info",
    "lbft_memory_info", "lbft_kernel_info", "lbft_run_until", "lbft_snapshot_size", "lbft_snapshot_save", "lbft_snapshot_load", "lbft_set_seeds", "lbft_device_buffer", "lbft_destroy", "lbft_last_error", "lbft_abi_version",
]

_lib = None


class LbftError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("lbft error %d: %s" % (code, message))
        self.code = code


def load():
    """Load ``liblbft_b200.so`` (fails loudly if it has not been built)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "%s is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback for the product path)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    P = ctypes.c_void_p
    lib.lbft_create.argtypes = [ctypes.POINTER(LbftConfig), ctypes.POINTER(P)]
    lib.lbft_create_sweep.argtypes = [ctypes.POINTER(LbftConfig), ctypes.POINTER(LbftParamSet), c_u32, P, ctypes.POINTER(P)]
    for name in ("lbft_run", "lbft_run_async", "lbft_wait", "lbft_upload", "lbft_run_device", "lbft_download"):
        getattr(lib, name).argtypes = [P]
    for name in ("lbft_commit_counts", "lbft_last_states", "lbft_active_rounds", "lbft_counters", "lbft_status"):
        getattr(lib, name).argtypes = [P, P]
    lib.lbft_commit_log.argtypes = [P, c_u32, c_u32, ctypes.POINTER(LbftCommit), ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t)]
    lib.lbft_commit_logs.argtypes = [P, P, ctypes.c_size_t, P]
    lib.lbft_round_switches.argtypes = [P, c_u32, ctypes.POINTER(LbftRoundSwitch), ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t)]
    lib.lbft_timing_info.argtypes = [P, ctypes.POINTER(LbftTiming)]
    lib.lbft_run_until.argtypes = [P, c_i64]
    lib.lbft_snapshot_size.argtypes = [P, ctypes.POINTER(ctypes.c_size_t)]
    lib.lbft_snapshot_save.argtypes = [P, P, ctypes.c_size_t]
    lib.lbft_snapshot_load.argtypes = [P, P, ctypes.c_size_t]
    lib.lbft_memory_info.argtypes = [P, ctypes.POINTER(c_u64), ctypes.POINTER(c_u32)]
    lib.lbft_kernel_info.argtypes = [P, ctypes.c_char_p, ctypes.c_size_t]
    lib.lbft_set_seeds.argtypes = [P, P]
    lib.lbft_device_buffer.argtypes = [P, c_u32, ctypes.POINTER(P), ctypes.POINTER(ctypes.c_size_t)]
    lib.lbft_destroy.argtypes = [P]
    lib.lbft_destroy.restype = None
    lib.lbft_last_error.restype = ctypes.c_char_p
    lib.lbft_abi_version.restype = c_u32
    _lib = lib
    return lib


def check(code, allow=()):
    if code != LBFT_OK and code not in allow:
        raise LbftError(code, load().lbft_last_error().decode())
    return code
