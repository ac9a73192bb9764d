"""CPU tier: host-side logic of the product package and the shape of the C ABI (no compute calls)."""
import ctypes as C
import functools
import json
import math
import re
from pathlib import Path

import numpy as np
import pytest
from hypothesis import given, settings, strategies as st

import gym_d2d_b200 as G
from gym_d2d_b200 import _lib, config as cfgmod, plugins
from oracle import d2d_oracle as O

ROOT = Path(__file__).resolve().parent.parent


# ---- C ABI ---------------------------------------------------------------------------------------------
def _declared_symbols():
    text = (ROOT / 'include' / 'd2d_b200.h').read_text()
    return sorted(set(re.findall(r'^D2D_API\s+[\w\s\*]+?\b(d2d_\w+)\s*\(', text, flags=re.M)))


def test_library_exports_every_declared_symbol():
    declared = _declared_symbols()
    assert len(declared) >= 14 and 'd2d_step' in declared and 'd2d_step_host' in declared
    lib = C.CDLL(str(_lib.lib_path()))
    for name in declared:
        assert hasattr(lib, name), f'{name} is declared in include/d2d_b200.h but not exported'
    assert sorted(_lib.SIGNATURES) == declared        # the ctypes binding covers exactly the header
    assert _lib.load().d2d_abi_version() == _lib.ABI_VERSION


def test_struct_layouts_match_header(tmp_path):
    """sizeof / offsetof of every ABI struct as a C compiler sees include/d2d_b200.h against the ctypes mirrors."""
    import subprocess
    assert C.sizeof(_lib.D2DConfig) == 2 * 4 + 8 + 12 * 4 + 10 * 8
    assert C.sizeof(_lib.D2DLink) == 5 * 8 + 2 * 4 + 8
    assert C.sizeof(_lib.D2DStepIO) == 11 * C.sizeof(C.c_void_p) + 8
    structs = {'d2d_config_t': _lib.D2DConfig, 'd2d_link_t': _lib.D2DLink, 'd2d_step_io_t': _lib.D2DStepIO}
    lines = ['#include <stddef.h>', '#include <stdio.h>', f'#include "{ROOT / "include" / "d2d_b200.h"}"', 'int main(void) {']
    for cname, cls in structs.items():
        lines.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'  printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    consts = {'D2D_STEP_INPUTS_STABLE': _lib.STEP_INPUTS_STABLE, 'D2D_STEP_ACTIONS_I16': _lib.STEP_ACTIONS_I16,
              'D2D_OUT_OBS': _lib.OUT_OBS, 'D2D_OUT_CAPACITY': _lib.OUT_CAPACITY, 'D2D_OUT_REWARD': _lib.OUT_REWARD, 'D2D_OUT_DONE': _lib.OUT_DONE,
              'D2D_OUT_RATE': _lib.OUT_RATE, 'D2D_OUT_RB': _lib.OUT_RB, 'D2D_OUT_TX_PWR': _lib.OUT_TX_PWR,
              'D2D_OUT_AGENT_REWARD': _lib.OUT_AGENT_REWARD, 'D2D_OUT_OBS_DYN': _lib.OUT_OBS_DYN}
    for cname in consts:                                      # flag / mask constants of the binding against the header's
        lines.append(f'  printf("{cname} %d\\n", (int){cname});')
    lines += ['  printf("abi %d\\n", D2D_ABI_VERSION);', '  return 0;', '}']
    src = tmp_path / 'layout.c'
    src.write_text('\n'.join(lines))
    subprocess.run(['gcc', '-std=c99', '-o', str(tmp_path / 'layout'), str(src)], check=True)
    got = dict(l.rsplit(' ', 1) for l in subprocess.run([str(tmp_path / 'layout')], check=True, capture_output=True,
                                                        text=True).stdout.strip().splitlines())
    assert int(got['abi']) == _lib.ABI_VERSION
    for cname, value in consts.items():
        assert int(got[cname]) == value, cname
    for cname, cls in structs.items():
        assert int(got[cname]) == C.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert int(got[f'{cname}.{fname}']) == getattr(cls, fname).offset, f'{cname}.{fname}'


def test_error_paths_without_gpu():
    """Argument errors are reported through codes + d2d_last_error, never by aborting."""
    lib = _lib.load()
    assert lib.d2d_create(None, None, None) == _lib.ERR_INVALID_ARG
    assert b'null' in lib.d2d_last_error()
    cfg = cfgmod.to_c_config(G.EnvConfig(), 4, 0, 0, 0, 0.0)
    links = (_lib.D2DLink * 50)(*[_lib.D2DLink(**r) for r in cfgmod.link_table(G.EnvConfig())])
    h = C.c_void_p()
    cfg.abi_version = 99
    assert lib.d2d_create(C.byref(cfg), links, C.byref(h)) == _lib.ERR_INVALID_ARG
    cfg.abi_version = _lib.ABI_VERSION
    cfg.path_loss_model = 7
    assert lib.d2d_create(C.byref(cfg), links, C.byref(h)) == _lib.ERR_UNSUPPORTED
    assert lib.d2d_step(None, None, None) == _lib.ERR_INVALID_ARG
    assert lib.d2d_launch_count(None) == -1


def test_product_never_imports_the_oracle():
    for py in (ROOT / 'gym_d2d_b200').glob('*.py'):
        src = py.read_text()
        assert 'oracle' not in re.sub(r'""".*?"""', '', src, flags=re.S).replace('# oracle', ''), py.name


def test_no_gpu_means_loud_failure():
    import torch
    if torch.cuda.is_available():
        pytest.skip('a GPU is present')
    with pytest.raises(Exception):
        G.VecD2DEnv(4, {})
    with pytest.raises(_lib.D2DError):
        G.VecD2DEnv(4, {}, device='cpu')


# ---- EnvConfig surface (envs/env_config.py:12-27) -------------------------------------------------------------
def test_env_config_defaults_and_keys():
    c = G.EnvConfig()
    expect = dict(num_rbs=25, num_cues=25, num_due_pairs=25, cell_radius_m=500.0, d2d_radius_m=20.0,
                  due_min_tx_power_dBm=0, due_max_tx_power_dBm=20, cue_max_tx_power_dBm=23, mbs_max_tx_power_dBm=46,
                  carrier_freq_GHz=2.1, num_subcarriers=12, subcarrier_spacing_kHz=15, channel_bandwidth_MHz=20.0,
                  device_config_file=None)
    for k, v in expect.items():
        assert getattr(c, k) == v
    assert c.path_loss_model is G.LogDistancePathLoss and c.traffic_model is G.UplinkTrafficModel
    assert c.num_pwr_actions == {'due': 21, 'cue': 24, 'mbs': 47}           # envs/d2d_env.py:31-35
    with pytest.raises(TypeError):
        G.EnvConfig(unknown_key=1)


def test_device_and_link_order():
    """test/gym_d2d/test_simulator.py:5-18 + devices.py:20-25 + envs/d2d_env.py:55-60"""
    c = G.EnvConfig(num_cues=3, num_due_pairs=2)
    assert c.device_ids() == ['mbs', 'cue00', 'cue01', 'cue02', 'due00', 'due01', 'due02', 'due03']
    assert c.link_keys() == ['cue00:mbs', 'cue01:mbs', 'cue02:mbs', 'due00:due01', 'due02:due03']
    assert c.device_ids() == O.OracleConfig(num_cues=3, num_due_pairs=2).device_ids()
    wide = G.EnvConfig(num_cues=1, num_due_pairs=500)
    assert wide.link_keys()[-1] == 'due998:due999'
    cfgs = c.device_configs()
    assert cfgs['cue00']['max_tx_power_dBm'] == 23 and cfgs['due00']['max_tx_power_dBm'] == 20
    assert cfgs['mbs']['max_tx_power_dBm'] == 46.0                            # Appendix B.5: not propagated


def test_link_table_matches_oracle_device_arithmetic(golden_dir):
    """The product folds device.py's link budget per link; the oracle evaluates it per call.  Same numbers."""
    dev = json.loads((golden_dir / 'overrides_device_config.json').read_text())
    for kw, overrides, path in [({}, {}, None),
                                (dict(num_rbs=3, num_cues=3, num_due_pairs=4), {k: v['config'] for k, v in dev.items()},
                                 golden_dir / 'overrides_device_config.json')]:
        c = G.EnvConfig(**kw, device_config_file=path)
        oc = O.OracleConfig(**kw, device_overrides=overrides)
        devs, L = O.device_table(oc), O.lib()
        for j, row in enumerate(cfgmod.link_table(c)):
            t = 1 + j if j < c.num_cues else 1 + c.num_cues + 2 * (j - c.num_cues)
            r = 0 if j < c.num_cues else t + 1
            assert row['tx_eirp_offset_dB'] == pytest.approx(L.d2d_oracle_eirp_dBm(C.byref(devs[t]), 0.0), abs=1e-12)
            assert row['rx_offset_dB'] == pytest.approx(L.d2d_oracle_rx_signal_level_dBm(C.byref(devs[r]), 0.0, 0.0), abs=1e-12)
            assert row['rx_noise_dBm'] == devs[r].thermal_noise_dBm
            assert row['rx_sensitivity_dBm'] == pytest.approx(L.d2d_oracle_rx_sensitivity_dBm(C.byref(devs[r])), abs=1e-12)
            assert row['tx_rb_bandwidth_kHz'] == L.d2d_oracle_rb_bandwidth_kHz(C.byref(devs[t]))
    t0 = cfgmod.link_table(G.EnvConfig())
    assert (t0[0]['tx_eirp_offset_dB'], t0[0]['rx_offset_dB'], t0[0]['rx_sensitivity_dBm']) == (-6.0, 17.5, pytest.approx(-123.4))
    assert (t0[-1]['rx_offset_dB'], t0[-1]['rx_noise_dBm'], t0[-1]['rx_sensitivity_dBm']) == (-3.0, -104.5, -107.5)


# ---- plugin resolution ------------------------------------------------------------------------------------------
def test_supported_plugins_resolve():
    assert plugins.resolve_path_loss(G.LogDistancePathLoss) == (_lib.PL_LOG_DISTANCE, 2.0)
    assert plugins.resolve_path_loss(G.FreeSpacePathLoss) == (_lib.PL_FREE_SPACE, 2.0)
    assert plugins.resolve_path_loss(functools.partial(G.LogDistancePathLoss, ple=3.5)) == (_lib.PL_LOG_DISTANCE, 3.5)
    assert plugins.resolve_obs_fn(G.LinearObsFunction) == _lib.OBS_LINEAR
    assert plugins.resolve_reward_fn(G.SystemCapacityRewardFunction) == (_lib.REWARD_SYSTEM_CAPACITY, 0.0)
    assert plugins.resolve_reward_fn(functools.partial(G.SystemCapacityRewardFunction, min_capacity_mbps=0.5))[1] == 0.5
    # SURVEY 8(f)-3 plugins: parameters and defaults of envs/reward_fn.py:48,61 and path_loss.py:91
    assert plugins.resolve_reward_fn(G.ShannonRewardFunction) == (_lib.REWARD_SHANNON, -70.0)
    assert plugins.resolve_reward_fn(functools.partial(G.CueSinrShannonRewardFunction, sinr_threshold_dB=3.0)) == (_lib.REWARD_CUE_SINR_SHANNON, 3.0)
    assert plugins.resolve_path_loss(G.CostHataPathLoss) == (_lib.PL_COST_HATA, float(G.AreaType.SUBURBAN.value))
    assert plugins.resolve_path_loss(functools.partial(G.CostHataPathLoss, area_type=G.AreaType.URBAN))[1] == 2.0


def test_cost_hata_fold_matches_the_oracle_restatement():
    """config.cost_hata_fold turns CostHataPathLoss (path_loss.py:90-123) into (exponent, per-receiver constant); the pair must
    reproduce the oracle's restatement of the reference formula at any distance, for both receiver classes and area types."""
    L = O.lib()
    for area in (G.AreaType.RURAL, G.AreaType.SUBURBAN, G.AreaType.URBAN):
        c = G.EnvConfig(num_rbs=3, num_cues=2, num_due_pairs=2, path_loss_model=functools.partial(G.CostHataPathLoss, area_type=area))
        ple, consts = cfgmod.cost_hata_fold(c)
        for rx, h_rx in [('mbs', 23.0), ('due01', 1.5)]:
            for d in (3.0, 77.0, 499.0):
                want = L.d2d_oracle_cost_hata_pl(d, 2.1, area.value, 1.5, h_rx)
                assert 10 * ple * math.log10(d) + consts[rx] == pytest.approx(want, rel=1e-12)
    rows = cfgmod.link_table(c)
    assert rows[0]['path_loss_const_dB'] == consts['mbs'] and rows[-1]['path_loss_const_dB'] == consts['due03']
    assert cfgmod.cost_hata_fold(G.EnvConfig()) is None


def test_reference_classes_are_accepted_by_identity():
    from oracle import ref_runner as R
    if R.import_reference() is None:
        pytest.skip('reference not importable here')
    from gym_d2d.envs.obs_fn import LinearObsFunction as RefObs
    from gym_d2d.envs.reward_fn import ShannonRewardFunction as RefShannon, SystemCapacityRewardFunction as RefRew
    from gym_d2d.path_loss import CostHataPathLoss as RefHata, LogDistancePathLoss as RefLD
    assert plugins.resolve_path_loss(RefLD) == (_lib.PL_LOG_DISTANCE, 2.0)
    assert plugins.resolve_obs_fn(RefObs) == _lib.OBS_LINEAR
    assert plugins.resolve_reward_fn(RefRew) == (_lib.REWARD_SYSTEM_CAPACITY, 0.0)
    from gym_d2d.path_loss import AreaType as RefArea, ShadowingPathLoss as RefShadow
    assert plugins.resolve_path_loss(RefShadow) == (_lib.PL_SHADOWING, 2.0) and plugins.shadowing_params(RefShadow) == (100.0, 2.7)
    assert plugins.resolve_path_loss(RefHata) == (_lib.PL_COST_HATA, 1.0)
    assert plugins.resolve_path_loss(functools.partial(RefHata, area_type=RefArea.URBAN)) == (_lib.PL_COST_HATA, 2.0)
    assert plugins.resolve_reward_fn(RefShannon) == (_lib.REWARD_SHANNON, -70.0)
    assert plugins.shadowing_params(functools.partial(RefShadow, chi_dB=3.5, d0_m=50.0)) == (50.0, 3.5)


def test_custom_and_unimplemented_plugins_are_rejected():
    class CustomPathLoss(G.LogDistancePathLoss):      # examples/custom_path_loss.py
        def __call__(self, tx, rx):
            return 100.0

    class CustomObs(G.LinearObsFunction):
        pass

    for bad in (CustomPathLoss, functools.partial(G.ShadowingPathLoss, sigma=1.0), functools.partial(G.CostHataPathLoss, ple=3.0),
                functools.partial(G.FreeSpacePathLoss, ple=3.0)):
        with pytest.raises(G.UnsupportedPluginError):
            plugins.resolve_path_loss(bad)
    with pytest.raises(G.UnsupportedPluginError):
        plugins.resolve_obs_fn(CustomObs)
    class CustomReward(G.ShannonRewardFunction):
        pass

    for bad in (CustomReward, functools.partial(G.ShannonRewardFunction, min_capacity_mbps=1.0)):
        with pytest.raises(G.UnsupportedPluginError):
            plugins.resolve_reward_fn(bad)
    with pytest.raises(TypeError):
        plugins.resolve_path_loss(G.LogDistancePathLoss(2.1))   # an instance, not a class


def test_make_rejects_unknown_id():
    with pytest.raises(ValueError):
        G.make('NotAnEnv-v0')


# ---- the integer decode the kernel uses (envs/d2d_env.py:93-101) ----------------------------------------------------
def _kernel_decode(a: int, n: int):
    """Bit-for-bit model of the device code (d2d_div_magic / d2d_div in csrc/d2d_common.cuh):
    rb = umulhi(a, ceil(2^32 / n)) for n > 1, a for n == 1; p = a - rb * n."""
    magic = 0 if n <= 1 else ((1 << 32) + n - 1) // n
    assert magic < 1 << 32
    rb = (a * magic) >> 32 if magic else a
    return rb, a - rb * n


@settings(max_examples=400, deadline=None)
@given(n=st.integers(1, 128), a=st.integers(0, 2 ** 24))
def test_magic_division_is_exact(n, a):
    assert _kernel_decode(a, n) == (a // n, a % n)


def test_magic_division_exhaustive_for_default_spaces():
    for n, hi in ((21, 25 * 21), (24, 25 * 24), (47, 25 * 47), (24, 100 * 24), (21, 100 * 21)):
        a = np.arange(hi, dtype=np.int64)
        magic = ((1 << 32) + n - 1) // n
        rb = (a * magic) >> 32
        assert (rb == a // n).all() and (a - rb * n == a % n).all()


def test_shard_range_partitions_the_batch():
    from gym_d2d_b200.dist import shard_range
    for total, world in [(1048576, 8), (4096, 3), (5, 8), (1000, 7)]:
        spans = [shard_range(total, r, world) for r in range(world)]
        assert spans[0][0] == 0 and sum(c for _, c in spans) == total
        for (f0, c0), (f1, _c1) in zip(spans, spans[1:]):
            assert f0 + c0 == f1
        assert max(c for _, c in spans) - min(c for _, c in spans) <= 1


def test_dict_views_follow_the_reference_layout():
    """D2DEnv's dict building (cached index tables, one gather) against a per-key restatement of envs/obs_fn.py:43-53 (own 6-tuple, then
    every other present link's in the action dict's order), envs/d2d_env.py:103-116 (info) and simulator.py:77-87 (state keys) - on
    synthetic host arrays, no GPU: a full agent set, a shuffled subset, and the first set again (served from the cache)."""
    from gym_d2d_b200.d2d_env import D2DEnv
    rng = np.random.default_rng(3)
    N = 12
    env = object.__new__(D2DEnv)
    keys_all = [f'cue{i:02d}:mbs' for i in range(5)] + [f'due{2 * i:02d}:due{2 * i + 1:02d}' for i in range(7)]
    env._link_index = {k: i for i, k in enumerate(keys_all)}
    env._views = {}
    env._host = {'obs': rng.normal(size=(1, N, 6)).astype(np.float32), 'rate_bps': rng.random((1, N)).astype(np.float32),
                 'capacity_mbps': rng.random((1, N)).astype(np.float32), 'rb': rng.integers(0, 25, (1, N)).astype(np.int16),
                 'tx_pwr_dbm': rng.integers(0, 24, (1, N)).astype(np.int16)}
    table = env._host['obs'][0].astype(np.float64)
    for keys in (keys_all, [keys_all[i] for i in rng.permutation(N)[:7]], keys_all):
        obs, state, acts = env._obs_dict(keys), env._state(keys), env._actions_view(keys)
        assert list(obs) == keys and list(acts) == keys
        rows = [env._link_index[k] for k in keys]
        for pos, k in enumerate(keys):
            expect = np.concatenate([table[rows[pos]]] + [table[r] for q, r in enumerate(rows) if q != pos])
            np.testing.assert_array_equal(obs[k], expect)
            assert obs[k].dtype == np.float64 and obs[k].shape == (6 * len(keys),)
            pair = tuple(k.split(':'))
            assert state['sinrs_db'][pair] == float(env._host['obs'][0, rows[pos], 4]) and isinstance(state['sinrs_db'][pair], float)
            assert state['snrs_db'][pair] == float(env._host['obs'][0, rows[pos], 5])
            assert state['rate_bps'][pair] == float(env._host['rate_bps'][0, rows[pos]])
            assert state['capacity_mbps'][pair] == float(env._host['capacity_mbps'][0, rows[pos]])
            assert acts[k] == (int(env._host['rb'][0, rows[pos]]), int(env._host['tx_pwr_dbm'][0, rows[pos]]))
            assert all(isinstance(v, int) for v in acts[k])
        assert list(state['sinrs_db']) == [tuple(k.split(':')) for k in keys]
    assert len(env._views) == 2


# ---- the step-kernel dispatch restated in tests/_kernel_dispatch.py, against the real host functions ---------------------------
_LAYOUT_PROBE = r'''
#include "d2d_internal.h"
#include "d2d_step_dense.cuh"
#include "d2d_step_block.cuh"
#include "d2d_step_warp.cuh"
#include <cstdio>
int main() {
    std::printf("rc %zu\n", sizeof(D2DDenseRC));
    int N, R, V, bt;
    while (std::scanf("%d %d %d %d", &N, &R, &V, &bt) == 4) {
        const int cap = d2d_dense_bin_cap(N, R);
        std::printf("%d %d %d %d %d %u %zu %zu %u %u %u\n", N, R, V, bt, cap, d2d_dense_layout(N, R, cap, bt, V).total,
                    d2d_block2_smem_bytes(N, R), d2d_block_smem_bytes(N, R), d2d_warp_smem_bytes(R, 2), d2d_warp_smem_bytes(R, 4),
                    d2d_warp_smem_bytes(R, 8));
    }
    return 0;
}
'''


def test_restated_kernel_layouts_match_the_host_functions(tmp_path):
    """tests/_kernel_dispatch.py restates the bin capacity and the shared-memory layouts of the dense, sorting, general and warp
    kernels; the GPU matrix (tests/test_kernel_matrix.py) asserts step_geometry() against them.  Here the real host functions
    (d2d_dense_bin_cap, d2d_dense_layout, d2d_block2_smem_bytes, d2d_block_smem_bytes, d2d_warp_smem_bytes) are compiled into a
    host-only program and must agree byte for byte over a sweep of link and RB counts."""
    import shutil
    import subprocess
    from tests import _kernel_dispatch as KD
    nvcc = shutil.which('nvcc') or ('/usr/local/cuda/bin/nvcc' if Path('/usr/local/cuda/bin/nvcc').exists() else None)
    if nvcc is None:
        pytest.skip('nvcc not found')
    src = tmp_path / 'layout_probe.cu'
    src.write_text(_LAYOUT_PROBE)
    exe = tmp_path / 'layout_probe'
    subprocess.run([nvcc, '-gencode', 'arch=compute_100a,code=sm_100a', '-std=c++17', '-diag-suppress', '159',
                    '-I', str(ROOT / 'gym_d2d_b200' / 'csrc'), '-o', str(exe), str(src)], check=True, capture_output=True)
    cases = []
    for N in (1, 64, 65, 100, 255, 256, 257, 300, 320, 321, 512, 600, 640, 641, 700, 768, 769, 800, 960, 961, 1000, 1024, 1025,
              2000, 3000, 3300, 4000):
        for R in (1, 4, 25, 64, 100, 300, 512, 600, 3000):
            for D in {0, N // 5, (4 * N) // 5, N}:
                cases.append((N, R, 1 + N + D, 256 if (N + R + D) % 2 else 320))
    res = subprocess.run([str(exe)], input=''.join(f'{n} {r} {v} {b}\n' for n, r, v, b in cases), check=True, capture_output=True, text=True)
    lines = res.stdout.strip().splitlines()
    assert lines[0] == f'rc {KD.DENSE_RC_BYTES}'
    assert len(lines) == 1 + len(cases)
    for (N, R, V, bt), line in zip(cases, lines[1:]):
        got = [int(x) for x in line.split()]
        assert got[:4] == [N, R, V, bt]
        cap = KD.dense_bin_cap(N, R)
        want = [cap, KD.dense_smem(N, R, cap, bt, V), KD.block2_smem(N, R), KD.block_smem(N, R),
                KD.warp_smem(R, 2), KD.warp_smem(R, 4), KD.warp_smem(R, 8)]
        assert got[4:] == want, (N, R, V, bt)


@pytest.mark.parametrize('R,C,D,E,env,family,lpt,bt,wpb', [
    (64, 32, 32, 1024, {}, 'warp', 0, 0, 2), (64, 32, 32, 5000, {}, 'warp', 0, 0, 4),
    (64, 32, 32, 100, {'D2D_B200_WPB': '8'}, 'warp', 0, 0, 8), (16, 24, 40, 96, {}, 'dense', 1, 256, 0),
    (65, 32, 32, 64, {}, 'dense', 1, 256, 0), (64, 33, 32, 64, {}, 'dense', 1, 256, 0),
    (50, 60, 240, 64, {}, 'dense', 1, 320, 0), (40, 80, 320, 64, {}, 'dense', 2, 256, 0), (60, 100, 500, 64, {}, 'dense', 2, 320, 0),
    (30, 140, 560, 64, {}, 'dense', 3, 256, 0), (25, 160, 640, 64, {}, 'dense', 3, 320, 0), (25, 224, 800, 64, {}, 'dense', 4, 256, 0),
    (600, 40, 160, 64, {}, 'sorting', 1, 0, 0), (300, 100, 500, 64, {}, 'sorting', 3, 0, 0), (600, 224, 800, 64, {}, 'sorting', 4, 0, 0),
    (60, 100, 500, 64, {'D2D_B200_DENSE': '0'}, 'sorting', 3, 0, 0), (25, 225, 800, 64, {}, 'general', 0, 0, 0),
    (100, 600, 2400, 64, {}, 'general', 0, 0, 0), (100, 800, 3200, 64, {}, 'unsupported', 0, 0, 0)])
def test_restated_dispatch_picks_the_documented_family(R, C, D, E, env, family, lpt, bt, wpb):
    """Spot checks of the restated dispatch at the edges of each family: C, D <= 32 and R <= 64 for the warp kernel; N = 1024
    as the largest dense / sorting shape; R > 512 or a dense layout over 75 KB for the sorting kernel; past 227 KB refused."""
    from tests._kernel_dispatch import expected_kernel
    k = expected_kernel(dict(num_rbs=R, num_cues=C, num_due_pairs=D), E, env=env)
    assert (k['family'], k['lpt'], k['bt'], k['wpb']) == (family, lpt, bt, wpb)
    assert expected_kernel(dict(num_rbs=4, num_cues=5, num_due_pairs=6), 64, env={}, downlink=True)['family'] == 'general'
    assert expected_kernel(dict(num_rbs=25), 512, env={})['spec'] and not expected_kernel(dict(num_rbs=25), 512, env={'D2D_B200_SPEC': '0'})['spec']
    assert expected_kernel(dict(num_rbs=100, num_cues=100, num_due_pairs=500), 64, env={})['spec']
