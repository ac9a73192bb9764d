"""Which step kernel d2d_create picks for a configuration, restated from the sources so that a test can say which
instantiation it means to run and check it through VecD2DEnv.step_geometry() before it compares anything.

Every rule below cites the line of gym_d2d_b200/csrc it restates.  tests/test_host_logic.py compiles the real host
functions of the three shared-memory layouts with nvcc and checks the formulas here against them, so a change of a layout
that is not mirrored here fails on the CPU tier already.

expected_kernel(kw, E) -> dict(family, lpt, bt, wpb, spec, block, smem)
    family  'warp' | 'dense' | 'sorting' | 'general' | 'unsupported'
    lpt     links per thread (dense / sorting kernel), 0 otherwise
    bt      threads per block of the dense kernel, 0 otherwise
    wpb     warps per block of the warp kernel, 0 otherwise
    spec    the instantiation specialised for one shape (warp: the default 25/25/25 EnvConfig, dense: 100/100/500)
    block   threads per block: what step_geometry()['block'] reports
    smem    dynamic shared memory per block: what step_geometry()['smem_bytes'] reports
"""
from __future__ import annotations

import math
import os
from typing import Mapping, Optional

from gym_d2d_b200 import _lib
from gym_d2d_b200.config import EnvConfig, link_table, to_c_config

MAX_PWR_LEVELS = 128               # d2d_common.cuh:22 D2D_MAX_PWR_LEVELS
BLOCK_THREADS = 256                # d2d_internal.h:211 D2D_BLOCK_THREADS
BLOCK_MAX_LPT = 4                  # d2d_internal.h:212 D2D_BLOCK_MAX_LPT
BLOCK_RESQ = 32                    # d2d_step_block.cuh:225 D2D_BLOCK_RESQ
LATENCY_ENVS = 2048                # d2d_internal.h:191 D2D_LATENCY_ENVS
DENSE_MAX_WARPS = 16               # d2d_step_dense.cuh:31 D2D_DENSE_MAX_WARPS
DENSE_RC_BYTES = 136               # sizeof(D2DDenseRC), d2d_step_dense.cuh:38-46 (checked by tests/test_host_logic.py)
DENSE_SMEM_CAP = 75 * 1024         # d2d_abi.cu:269 (three blocks per SM)
DENSE_MAX_RBS = 512                # d2d_abi.cu:268 (9 bits of the packed link state)
SMEM_LIMIT = 227 * 1024            # d2d_abi.cu:278
WARP_BIN_CAP = 8                   # d2d_step_warp.cuh:66 D2D_BIN_CAP


def _al(x: int, a: int) -> int:
    return (x + a - 1) // a * a


# ---- shared-memory layouts -----------------------------------------------------------------------------------------------------
def warp_smem(R: int, wpb: int) -> int:
    """d2d_step_warp.cuh:78-86 d2d_warp_smem_bytes."""
    blk = MAX_PWR_LEVELS * 4 + 64 * 16 + 64 * 8                                   # D2D_BLK_BYTES
    per_warp = R * (WARP_BIN_CAP * 16 + 16) + 528 + _al(R * 8, 16)               # d2d_warp_smem_per_warp
    return blk + wpb * per_warp


def dense_bin_cap(N: int, R: int) -> int:
    """d2d_step_dense.cuh:74-80 d2d_dense_bin_cap: mean + 3.5 sigma of the per-RB load, a multiple of 8."""
    m = N / max(R, 1)
    cap = int(m + 3.5 * math.sqrt(m) + 1.0)
    cap = max(min(cap, N), 8)
    return _al(cap, 8)


def dense_smem(N: int, R: int, cap: int, bt: int, V: int) -> int:
    """d2d_step_dense.cuh:52-70 d2d_dense_layout(...).total."""
    b = MAX_PWR_LEVELS * 8 + MAX_PWR_LEVELS * 4                                   # pwr_d, pwr
    b += 2 * 4 * DENSE_MAX_WARPS * 4 + 8 * 8 + _al(DENSE_RC_BYTES, 16) + 16        # red, sst, rc, mbar
    b += _al(N * 4, 16) + 16 + _al(V * 8, 16) + 16                               # sact, spos
    b += 2 * bt * 4                                                               # grp
    b += 3 * _al(R + 2, 4) * 4                                                    # cnt
    b = _al(b, 128)
    b += 2 * R * cap * 16                                                         # bins
    return b + 112


def block2_smem(N: int, R: int) -> int:
    """d2d_step_block.cuh:227-235 d2d_block2_smem_bytes (the sorting block kernel)."""
    return (N * 16 + MAX_PWR_LEVELS * 4 + _al((R + 1) * 2 * 4, 16) + _al(N * 4, 16)
            + 2 * (BLOCK_RESQ * 8 + 4) * 4 + 2 * 32 * 4)


def block_smem(N: int, R: int) -> int:
    """d2d_step_block.cuh:33-42 d2d_block_smem_bytes (the general-topology kernel)."""
    return 4 * N * 16 + MAX_PWR_LEVELS * 4 + 2 * R * 4 + N * 4 + 32 * 4 + _al(N * 2, 16)


# ---- the dispatch of d2d_create ----------------------------------------------------------------------------------------------------
def _uniform(config: EnvConfig) -> bool:
    """d2d_abi.cu:179-184: one set of link constants per link type (no per-device override changed one) and no downlinks.
    Restated on the unfolded link rows: equal rows fold to equal constants."""
    if config.downlinks:
        return False
    rows = link_table(config)
    keys = ('tx_eirp_offset_dB', 'rx_offset_dB', 'rx_noise_dBm', 'rx_sensitivity_dBm', 'tx_rb_bandwidth_kHz', 'path_loss_const_dB')
    C = config.num_cues
    return all(tuple(r[k] for k in keys) == tuple(rows[0 if j < C else C][k] for k in keys) for j, r in enumerate(rows))


def expected_kernel(kw: Mapping, E: int, env: Optional[Mapping[str, str]] = None, downlink: bool = False) -> dict:
    """The step kernel d2d_create (d2d_abi.cu:223-279) selects for VecD2DEnv(E, kw, downlink=downlink).  `env` is the process
    environment the handle is created under (default os.environ): the knobs D2D_B200_WPB, D2D_B200_DENSE=0 and D2D_B200_SPEC."""
    env = os.environ if env is None else env
    kw = {k: v for k, v in kw.items() if k not in ('reward_fn', 'obs_fn')}
    config = EnvConfig(**kw)
    config.downlinks = bool(downlink)
    cc = to_c_config(config, E, 0, 0, 0, 0.0)
    R, C, D = cc.num_rbs, cc.num_cues, cc.num_due_pairs
    N = config.num_links
    V = config.num_devices
    ple2 = cc.ple == 2.0                                                          # d2d_abi.cu:119,130
    uniform = _uniform(config)
    cost_hata = cc.path_loss_model == _lib.PL_COST_HATA
    general = bool(downlink) or cc.path_loss_model == _lib.PL_SHADOWING          # d2d_abi.cu:225
    out = dict(family='', lpt=0, bt=0, wpb=0, spec=False, block=0, smem=0, ple2=ple2, uniform=uniform, N=N)
    if C <= 32 and D <= 32 and R <= 64 and not general:                           # d2d_abi.cu:226
        wpb = 2 if E <= LATENCY_ENVS else 4                                       # d2d_abi.cu:240
        if 'D2D_B200_WPB' in env:                                                 # d2d_abi.cu:239-240
            v = int(env['D2D_B200_WPB'] or 0)
            wpb = 8 if v == 8 else 2 if v == 2 else 4
        spec = (ple2 and uniform and not cost_hata and R == 25 and C == 25 and D == 25      # d2d_abi.cu:232-233, 242-243
                and cc.n_pwr_cue == 24 and cc.n_pwr_due == 21)
        if 'D2D_B200_SPEC' in env:
            spec = spec and int(env['D2D_B200_SPEC'] or 0) != 0
        return dict(out, family='warp', wpb=wpb, spec=spec, block=32 * wpb, smem=warp_smem(R, wpb))
    lpt = (N + BLOCK_THREADS - 1) // BLOCK_THREADS if N <= BLOCK_THREADS * BLOCK_MAX_LPT and not general else 0   # d2d_abi.cu:260-261
    cap = dense_bin_cap(N, R)                                                     # d2d_abi.cu:262
    dn = env.get('D2D_B200_DENSE')
    bt = 320 if ((N + 319) // 320) * 10 < ((N + 255) // 256) * 8 and (N + 319) // 320 <= 3 else 256   # d2d_abi.cu:267
    dense = (lpt > 0 and R <= DENSE_MAX_RBS and dense_smem(N, R, cap, bt, V) <= DENSE_SMEM_CAP        # d2d_abi.cu:268-269
             and not (dn is not None and int(dn or 0) == 0))
    if dense:
        lpt = (N + bt - 1) // bt                                                  # d2d_abi.cu:272
        spec = (ple2 and bt == 320 and N == 600 and C == 100 and R == 100 and cap == 16      # d2d_abi.cu:232-233, 274-275
                and cc.n_pwr_cue == 24 and cc.n_pwr_due == 21)
        if 'D2D_B200_SPEC' in env:
            spec = spec and int(env['D2D_B200_SPEC'] or 0) != 0
        smem = dense_smem(N, R, cap, bt, V)
        out = dict(out, family='dense', lpt=lpt, bt=bt, spec=spec, block=bt, smem=smem)
    else:
        smem = block2_smem(N, R) if lpt else block_smem(N, R)                     # d2d_abi.cu:277, d2d_tu_block.cu:6
        out = dict(out, family='sorting' if lpt else 'general', lpt=lpt, block=BLOCK_THREADS, smem=smem)
    if out['smem'] > SMEM_LIMIT:                                                  # d2d_abi.cu:278
        out['family'] = 'unsupported'
    return out
