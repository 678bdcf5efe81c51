"""ctypes binding of libnig_b200.so (C ABI declared in include/nig_b200.h).

The library is the ONLY implementation of the step path: if it is missing, or if no sm_100 device is
visible, everything here raises -- there is no CPU fallback and nothing under oracle/ is ever imported.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG_DIR)                       # neorl-industrial-gym_b200/
LIB_PATH = os.environ.get("NIG_LIB_PATH") or os.path.join(_ROOT, "libnig_b200.so")   # (override: A/B builds, tools/ab_build.sh)
CSRC_DIR = os.path.join(_ROOT, "csrc")

ABI_VERSION = 6
MAX_CONSTRAINTS = 8
STATS_SLOTS = 32

OK, ERR_INVALID, ERR_CUDA, ERR_NO_DEVICE, ERR_UNSUPPORTED = 0, 1, 2, 3, 4
ENV_CHEMICAL_REACTOR, ENV_POWER_GRID, ENV_ROBOT_ASSEMBLY = 0, 1, 2
CON_BUILTIN, CON_BOUND, CON_HOSTMASK = 0, 1, 2
F_TERMINATED, F_TRUNCATED, F_CRITICAL, F_RESET, F_INACTIVE = 1, 2, 4, 8, 128
LAYOUT_SOA, LAYOUT_AOS = 0, 1
POLICY_ACTIONS, POLICY_UNIFORM, POLICY_ZERO, POLICY_PCTRL, POLICY_BASELINE, POLICY_MLP = 0, 1, 2, 3, 4, 5
MLP_OUT_IDENTITY, MLP_OUT_TANH = 0, 1
BASELINE_RANDOM, BASELINE_PID, BASELINE_MPC, BASELINE_CONSTANT = 0, 1, 2, 3
ROLLOUT_USE_TMA = 1
ROLLOUT_ACCUMULATE = 2
ST_STEPS, ST_EPISODES, ST_TERMINATED, ST_TRUNCATED, ST_CRITICAL, ST_VIOLATIONS, ST_SUCCESSES, ST_EP_LEN_SUM = range(8)
ST_CON0 = 8
ST_EP_LEN_SQ = 16
ST_F_RETURN_SUM, ST_F_RETURN_SQ, ST_F_REWARD_SUM = 24, 25, 26


class Constraint(C.Structure):
    _fields_ = [("kind", C.c_int32), ("id", C.c_int32), ("si", C.c_int32), ("ai", C.c_int32),
                ("coef", C.c_float), ("lo", C.c_float), ("hi", C.c_float), ("penalty", C.c_float),
                ("critical", C.c_int32)]


class EnvSpec(C.Structure):
    _fields_ = [("state_dim", C.c_int32), ("action_dim", C.c_int32), ("noise_dim", C.c_int32),
                ("max_episode_steps", C.c_int32), ("n_constraints", C.c_int32), ("reserved", C.c_int32),
                ("constraints", Constraint * MAX_CONSTRAINTS)]


class Config(C.Structure):
    _fields_ = [("env_kind", C.c_int32), ("device", C.c_int32), ("n_envs", C.c_int64),
                ("env_id_offset", C.c_int64), ("seed", C.c_uint64), ("max_episode_steps", C.c_int32),
                ("auto_reset", C.c_int32), ("n_constraints", C.c_int32), ("reserved", C.c_int32),
                ("constraints", Constraint * MAX_CONSTRAINTS)]


class StepIO(C.Structure):
    _fields_ = [("actions", C.c_void_p), ("noise", C.c_void_p), ("reset_states", C.c_void_p),
                ("hostmask", C.c_void_p), ("obs", C.c_void_p), ("next_obs", C.c_void_p),
                ("reward", C.c_void_p), ("flags", C.c_void_p), ("viol_mask", C.c_void_p),
                ("action_layout", C.c_int32), ("aux_layout", C.c_int32),
                ("terminated", C.c_void_p), ("truncated", C.c_void_p)]


class Baseline(C.Structure):
    _fields_ = [("kind", C.c_int32), ("reserved", C.c_int32), ("kp", C.c_double), ("ki", C.c_double), ("kd", C.c_double),
                ("setpoint", C.c_double * 8)]


class PolicyParams(C.Structure):
    _fields_ = [("p_ctrl", C.c_float), ("uniform_scale", C.c_float), ("store_clip", C.c_float), ("mode", C.c_int32),
                ("gain", (C.c_float * 2) * 8), ("sigma", C.c_float * 8), ("baseline", Baseline)]


class Rollout(C.Structure):
    _fields_ = [("n_steps", C.c_int32), ("policy", C.c_int32), ("flags", C.c_int32), ("reserved", C.c_int32),
                ("actions", C.c_void_p), ("noise", C.c_void_p), ("pp", PolicyParams),
                ("reward_sum", C.c_void_p), ("viol_count", C.c_void_p), ("done_count", C.c_void_p)]


class Trajectory(C.Structure):
    """nig_trajectory_t: the per-step device arrays of nig_rollout_record, time-major [K][n][dim] (NULL = not recorded)."""
    _fields_ = [("obs", C.c_void_p), ("actions", C.c_void_p), ("rewards", C.c_void_p), ("flags", C.c_void_p),
                ("viol_mask", C.c_void_p), ("terminated", C.c_void_p), ("truncated", C.c_void_p), ("next_obs", C.c_void_p)]


class RolloutHost(C.Structure):
    _fields_ = [("n_steps", C.c_int32), ("steps_per_launch", C.c_int32), ("policy", C.c_int32), ("reset_first", C.c_int32),
                ("init_states", C.c_void_p), ("actions", C.c_void_p), ("noise", C.c_void_p), ("pp", PolicyParams),
                ("reward_sum", C.c_void_p), ("viol_count", C.c_void_p), ("done_count", C.c_void_p),
                ("final_obs", C.c_void_p), ("counters24", C.c_void_p), ("sums8", C.c_void_p)]


class DatasetOut(C.Structure):
    _fields_ = [("observations", C.c_void_p), ("actions", C.c_void_p), ("rewards", C.c_void_p),
                ("terminals", C.c_void_p), ("timeouts", C.c_void_p), ("next_observations", C.c_void_p),
                ("safety", C.c_void_p), ("capacity", C.c_int64), ("terminals_include_truncation", C.c_int32),
                ("reserved", C.c_int32)]


class Mlp(C.Structure):
    _fields_ = [("n_hidden", C.c_int32), ("hidden", C.c_int32 * 2), ("output_activation", C.c_int32), ("in_dim", C.c_int32),
                ("out_dim", C.c_int32), ("weight", C.c_void_p * 3), ("bias", C.c_void_p * 3), ("obs_mean", C.c_void_p),
                ("obs_inv_std", C.c_void_p)]


# every symbol include/nig_b200.h declares: (restype, argtypes)
_VP, _I32, _I64, _U32, _U64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_uint64
SYMBOLS = {
    "nig_abi_version": (C.c_int, []),
    "nig_last_error": (C.c_char_p, []),
    "nig_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "nig_env_spec": (C.c_int, [C.c_int, C.POINTER(EnvSpec)]),
    "nig_create": (C.c_int, [C.POINTER(Config), C.POINTER(_VP)]),
    "nig_destroy": (C.c_int, [_VP]),
    "nig_pitch": (_I64, [_VP]),
    "nig_num_envs": (_I64, [_VP]),
    "nig_set_constraints": (C.c_int, [_VP, C.POINTER(Constraint), _I32]),
    "nig_reset": (C.c_int, [_VP, _VP, _VP, _I32, _VP]),
    "nig_reset_host": (C.c_int, [_VP, _VP, _VP, _VP]),
    "nig_step": (C.c_int, [_VP, C.POINTER(StepIO), _VP]),
    "nig_step_host": (C.c_int, [_VP, C.POINTER(StepIO)]),
    "nig_rollout": (C.c_int, [_VP, C.POINTER(Rollout), _VP]),
    "nig_rollout_record": (C.c_int, [_VP, C.POINTER(Rollout), C.POINTER(Trajectory), _VP]),
    "nig_rollout_steps": (C.c_int, [_VP, _VP, C.c_int32, _VP]),
    "nig_rollout_host": (C.c_int, [_VP, C.POINTER(RolloutHost)]),
    "nig_reset_policy_state": (C.c_int, [_VP, _VP]),
    "nig_set_mlp_policy": (C.c_int, [_VP, C.POINTER(Mlp)]),
    "nig_selftest_mlp": (C.c_int, [_VP, _VP, _I64, _VP]),
    "nig_dataset": (C.c_int, [_VP, _I64, _I32, _I32, C.POINTER(PolicyParams), C.POINTER(DatasetOut), C.POINTER(_I64), _VP]),
    "nig_dataset_size": (C.c_int, [_VP, _I64, _I32, _I32, C.POINTER(PolicyParams), C.POINTER(_I64), _VP]),
    "nig_get_state": (C.c_int, [_VP, _VP, _I32, _VP, _VP, _VP, _VP]),
    "nig_set_state": (C.c_int, [_VP, _VP, _I32, _VP, _VP, _VP, _VP]),
    "nig_get_state_host": (C.c_int, [_VP, _VP, _VP, _VP, _VP]),
    "nig_set_state_host": (C.c_int, [_VP, _VP, _VP, _VP, _VP]),
    "nig_state_ptr": (C.c_int, [_VP, C.POINTER(_VP), C.POINTER(_VP)]),
    "nig_get_tick": (C.c_int, [_VP, C.POINTER(_U32), C.POINTER(_U32)]),
    "nig_set_tick": (C.c_int, [_VP, _U32, _U32]),
    "nig_use_device_tick": (C.c_int, [_VP, _I32]),
    "nig_commit_ticks": (C.c_int, [_VP, _VP]),
    "nig_set_seed": (C.c_int, [_VP, _U64]),
    "nig_stats_ptr": (C.c_int, [_VP, C.POINTER(_VP)]),
    "nig_fold_stats": (C.c_int, [_VP, _VP]),
    "nig_read_stats": (C.c_int, [_VP, _VP, _VP]),
    "nig_clear_stats": (C.c_int, [_VP, _VP]),
    "nig_allreduce_stats": (C.c_int, [_VP, _VP, _VP]),
    "nig_nccl_unique_id": (C.c_int, [_VP]),
    "nig_nccl_comm_init": (C.c_int, [C.POINTER(_VP), _I32, _VP, _I32, _I32]),
    "nig_nccl_comm_destroy": (C.c_int, [_VP]),
    "nig_track_extrema": (C.c_int, [_VP, C.c_int32]),
    "nig_track_returns": (C.c_int, [_VP, C.c_int32]),
    "nig_track_step_stats": (C.c_int, [_VP, C.c_int32]),
    "nig_extrema_ptr": (C.c_int, [_VP, C.POINTER(_VP)]),
    "nig_read_extrema": (C.c_int, [_VP, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(_I32)]),
    "nig_decode_extrema": (C.c_int, [_VP, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(_I32)]),
    "nig_sync": (C.c_int, [_VP]),
    "nig_host_alloc": (C.c_int, [C.c_size_t, C.POINTER(_VP)]),
    "nig_host_free": (C.c_int, [_VP]),
    "nig_launch_count": (_I64, [_VP]),
    "nig_fp32_probe": (C.c_int, [C.c_int, _I32, C.POINTER(C.c_double), _VP]),
    "nig_selftest_division": (C.c_int, [C.c_int, _I64, _U64, C.POINTER(_I64), C.POINTER(_I64)]),
    "nig_selftest_normal": (C.c_int, [C.c_int, C.c_uint32, C.c_uint32, C.c_int64, C.POINTER(C.c_uint64)]),
    "nig_selftest_policy": (C.c_int, [C.c_int, C.c_int32, C.c_int32, C.c_void_p, _I64, C.c_int32, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p]),
}


class NativeLibraryMissing(ImportError):
    pass


def build_native(verbose: bool = False) -> str:
    """Compile libnig_b200.so for sm_100a with nvcc (csrc/Makefile). Explicit -- never run implicitly."""
    out = None if verbose else subprocess.DEVNULL
    subprocess.check_call(["make", "-C", CSRC_DIR], stdout=out)
    return LIB_PATH


_lib = None


def lib():
    """Load the CUDA library; raises loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeLibraryMissing(
                f"{LIB_PATH} not found. neorl_industrial (B200) has no CPU fallback: build the CUDA "
                f"extension first (python -c 'import __graft_entry__ as g; g.build()' or make -C {CSRC_DIR}).")
        h = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(h, name)          # AttributeError if the .so does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        if h.nig_abi_version() != ABI_VERSION:
            raise NativeLibraryMissing(f"{LIB_PATH}: ABI version {h.nig_abi_version()} != {ABI_VERSION}; rebuild it")
        _lib = h
    return _lib


def check(rc: int) -> None:
    if rc == OK:
        return
    msg = lib().nig_last_error().decode("utf-8", "replace")
    if rc in (ERR_INVALID,):
        raise ValueError(msg)
    if rc == ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise RuntimeError(msg)          # CUDA failure / no sm_100 device: never falls back to a CPU path


def env_spec(kind: int) -> EnvSpec:
    s = EnvSpec()
    check(lib().nig_env_spec(kind, C.byref(s)))
    return s


def device_count() -> int:
    n = C.c_int(0)
    rc = lib().nig_device_count(C.byref(n))
    return n.value if rc == OK else 0


class PinnedArray:
    """A page-locked host numpy array (cudaHostAlloc through the C ABI)."""

    def __init__(self, shape, dtype):
        self.shape = tuple(int(x) for x in np.atleast_1d(shape))
        self.dtype = np.dtype(dtype)
        nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        p = C.c_void_p()
        check(lib().nig_host_alloc(max(nbytes, 1), C.byref(p)))
        self._ptr = p.value
        buf = (C.c_char * max(nbytes, 1)).from_address(self._ptr)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(np.prod(self.shape))).reshape(self.shape)

    @property
    def ptr(self) -> int:
        return self._ptr

    def __del__(self):
        try:
            if getattr(self, "_ptr", None):
                self.array = None
                lib().nig_host_free(self._ptr)
                self._ptr = None
        except Exception:
            pass


def ptr_of(x) -> int | None:
    """Raw address of a numpy array (host) or a torch tensor (device or host); None passes through."""
    if x is None:
        return None
    if isinstance(x, np.ndarray):
        if not x.flags["C_CONTIGUOUS"]:
            raise ValueError("array must be C-contiguous")
        return x.ctypes.data
    if hasattr(x, "data_ptr"):
        if not x.is_contiguous():
            raise ValueError("tensor must be contiguous")
        return x.data_ptr()
    raise TypeError(f"cannot take the address of {type(x)}")
