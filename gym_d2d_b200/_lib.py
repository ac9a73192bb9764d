"""ctypes binding of libd2d_b200.so (include/d2d_b200.h).

There is deliberately no fallback: if the shared library is missing or a call fails, this raises.  The
product path never touches oracle/ or any CPU implementation.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

from .build import LIB

ABI_VERSION = 5
STATS_REPLICAS = 1024
NUM_STATS = 8
STAT_NAMES = ('sum_reward', 'sum_capacity_mbps', 'sum_reward_sq', 'env_steps', 'penalties', 'rescues', 'ticket_timeouts')

PL_LOG_DISTANCE, PL_FREE_SPACE, PL_COST_HATA, PL_SHADOWING = 0, 1, 2, 3
OBS_LINEAR = 0
REWARD_SYSTEM_CAPACITY, REWARD_SHANNON, REWARD_CUE_SINR_SHANNON = 0, 1, 2
LINK_UPLINK, LINK_DOWNLINK, LINK_SIDELINK = 1, 2, 3

OK, ERR_INVALID_ARG, ERR_UNSUPPORTED, ERR_CUDA, ERR_STATE = 0, -1, -2, -3, -4


class D2DConfig(C.Structure):
    _fields_ = [('abi_version', C.c_int32), ('cuda_device', C.c_int32), ('num_envs', C.c_int64),
                ('num_rbs', C.c_int32), ('num_cues', C.c_int32), ('num_due_pairs', C.c_int32),
                ('n_pwr_cue', C.c_int32), ('n_pwr_due', C.c_int32), ('episode_length', C.c_int32),
                ('path_loss_model', C.c_int32), ('obs_fn', C.c_int32), ('reward_fn', C.c_int32),
                ('num_downlinks', C.c_int32), ('n_pwr_mbs', C.c_int32), ('reserved0', C.c_int32),
                ('carrier_freq_GHz', C.c_double), ('ple', C.c_double), ('cell_radius_m', C.c_double),
                ('d2d_radius_m', C.c_double), ('min_capacity_mbps', C.c_double), ('reward_param', C.c_double),
                ('shadow_d0_m', C.c_double), ('shadow_chi_dB', C.c_double), ('rng_seed', C.c_uint64), ('first_global_env', C.c_uint64)]


class D2DLink(C.Structure):
    _fields_ = [('tx_eirp_offset_dB', C.c_double), ('rx_offset_dB', C.c_double), ('rx_noise_dBm', C.c_double),
                ('rx_sensitivity_dBm', C.c_double), ('tx_rb_bandwidth_kHz', C.c_double),
                ('link_type', C.c_int32), ('reserved0', C.c_int32), ('path_loss_const_dB', C.c_double)]


class D2DStepIO(C.Structure):
    _fields_ = [('actions', C.c_void_p), ('obs', C.c_void_p), ('capacity_mbps', C.c_void_p),
                ('reward', C.c_void_p), ('done', C.c_void_p), ('rate_bps', C.c_void_p),
                ('rb', C.c_void_p), ('tx_pwr_dBm', C.c_void_p), ('agent_reward', C.c_void_p),
                ('obs_dyn', C.c_void_p), ('actions_out', C.c_void_p), ('flags', C.c_uint32), ('reserved0', C.c_uint32)]


STEP_INPUTS_STABLE = 1          # d2d_step_io.flags (include/d2d_b200.h, "Ordering rule")
STEP_ACTIONS_I16 = 2            # d2d_step_host*: `actions` is int16 [E][N]
STEP_AUTORESET = 4              # d2d_step: next-step auto-reset of envs whose previous step returned done
EPISODE_DRAW_ACTIONS = 1        # d2d_episode flags
OUT_OBS, OUT_CAPACITY, OUT_REWARD, OUT_DONE, OUT_RATE, OUT_RB, OUT_TX_PWR, OUT_AGENT_REWARD, OUT_OBS_DYN = (
    1, 2, 4, 8, 16, 32, 64, 128, 256)


class D2DError(RuntimeError):
    """A libd2d_b200 call failed (CUDA error or library state)."""


class D2DUnsupportedError(ValueError):
    """The configuration is outside what the sm_100a kernels implement."""


# every symbol include/d2d_b200.h declares: (name, restype, argtypes)
_vp, _i64, _u64, _i32 = C.c_void_p, C.c_int64, C.c_uint64, C.c_int32
SIGNATURES = {
    'd2d_abi_version': (C.c_int, []),
    'd2d_last_error': (C.c_char_p, []),
    'd2d_create': (C.c_int, [C.POINTER(D2DConfig), C.POINTER(D2DLink), C.POINTER(_vp)]),
    'd2d_destroy': (C.c_int, [_vp]),
    'd2d_state_bytes': (C.c_int, [_vp, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    'd2d_bind_state': (C.c_int, [_vp, _vp, _vp, _vp]),
    'd2d_bind_positions_f64': (C.c_int, [_vp, _vp]),
    'd2d_bind_autoreset': (C.c_int, [_vp, _vp, _u64]),
    'd2d_set_positions': (C.c_int, [_vp, _vp, C.c_int, _i64, _i64, _vp]),
    'd2d_reset': (C.c_int, [_vp, _u64, _u64, _vp, _vp]),
    'd2d_get_positions': (C.c_int, [_vp, _vp, C.c_int, _i64, _i64, _vp]),
    'd2d_sample_actions': (C.c_int, [_vp, _vp, _u64, C.c_uint32, _vp]),
    'd2d_step': (C.c_int, [_vp, C.POINTER(D2DStepIO), _vp]),
    'd2d_episode': (C.c_int, [_vp, C.POINTER(D2DStepIO), _i32, _u64, _u64, C.c_uint32, _vp]),
    'd2d_rollout': (C.c_int, [_vp, C.POINTER(D2DStepIO), _i32, _u64, C.c_uint32, _vp]),
    'd2d_host_slot_buffers': (C.c_int, [_vp, C.c_int, C.c_uint32, C.POINTER(D2DStepIO)]),
    'd2d_step_many': (C.c_int, [_vp, C.POINTER(D2DStepIO), _i32, _vp]),
    'd2d_step_host': (C.c_int, [_vp, C.POINTER(D2DStepIO), _vp]),
    'd2d_step_host_async': (C.c_int, [_vp, C.POINTER(D2DStepIO), C.c_int, _vp]),
    'd2d_step_host_wait': (C.c_int, [_vp, C.c_int]),
    'd2d_per_agent_obs': (C.c_int, [_vp, _vp, _vp, _i64, _vp]),
    'd2d_stats_reset': (C.c_int, [_vp, _vp]),
    'd2d_launch_count': (_i64, [_vp]),
    'd2d_step_geometry': (C.c_int, [_vp, C.POINTER(_i32), C.POINTER(_i32), C.POINTER(_i32), C.POINTER(_i32)]),
}

_lib = None


def lib_path() -> Path:
    """The in-tree library; D2D_B200_LIB points tuning runs at an alternative build of the same sources."""
    import os
    return Path(os.environ.get('D2D_B200_LIB', LIB))


def load():
    """dlopen libd2d_b200.so.  Raises if it has not been built - there is no CPU fallback."""
    global _lib
    if _lib is None:
        LIB_ = lib_path()
        if not LIB_.exists():
            raise D2DError(f'{LIB_} is missing: build it with `python -m gym_d2d_b200.build` (needs nvcc). '
                           'gym_d2d_b200 has no CPU fallback.')
        lib = C.CDLL(str(LIB_))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        if lib.d2d_abi_version() != ABI_VERSION:
            raise D2DError(f'libd2d_b200.so ABI {lib.d2d_abi_version()} != binding ABI {ABI_VERSION}: rebuild')
        _lib = lib
    return _lib


def check(rc: int) -> None:
    if rc == OK:
        return
    msg = (load().d2d_last_error() or b'').decode('utf-8', 'replace')
    if rc == ERR_UNSUPPORTED:
        raise D2DUnsupportedError(msg)
    if rc == ERR_INVALID_ARG:
        raise ValueError(msg)
    raise D2DError(f'libd2d_b200 error {rc}: {msg}')
