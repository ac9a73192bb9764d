"""GPU tier (-m gpu): every step-kernel instantiation d2d_create can pick, held to the float64 oracle.

d2d_create (gym_d2d_b200/csrc/d2d_abi.cu:223-279) sends a configuration to one of four kernel families - the warp kernel
(2-, 4- or 8-warp blocks), the dense kernel (seven (links per thread, threads per block) shapes plus the instantiation for
100 RBs / 100 CUEs / 500 DUE pairs), the sorting block kernel (1-4 links per thread) and the general-topology kernel - each
instantiated for ple == 2 or not, and the dense and warp kernels also for the core-output (FULL) and fp64-shadow (EXACT)
variants.  tests/_kernel_dispatch.py restates that dispatch; every cell here first asserts from step_geometry() that the
library picked the kernel the cell is named after, so a cell that silently lands on another family fails, and only then
compares two consecutive steps with the oracle: rb and Tx power bit-exact, everything else within RTOL (tests/_util.py).
"""
import functools
import json
import zlib

import numpy as np
import pytest

from oracle import d2d_oracle as O
from tests._kernel_dispatch import expected_kernel
from tests._util import RTOL, assert_rel, check_against_oracle

torch = pytest.importorskip('torch')
pytestmark = pytest.mark.gpu

# name: (num_rbs, num_cues, num_due_pairs, num_envs, environment knobs, (family, links per thread, dense threads, warps per block))
SHAPES = {
    'warp_2w': (64, 32, 32, 1024, {}, ('warp', 0, 0, 2)),                      # both lane slots full, 64 RBs
    'warp_4w': (64, 32, 32, 5000, {}, ('warp', 0, 0, 4)),
    'warp_8w': (64, 32, 32, 1024, {'D2D_B200_WPB': '8'}, ('warp', 0, 0, 8)),
    'warp_1rb': (1, 32, 32, 256, {}, ('warp', 0, 0, 2)),                       # 64 links on one RB: the all-pairs path
    'dense_1x256': (4, 40, 60, 128, {}, ('dense', 1, 256, 0)),
    'dense_1x320': (50, 60, 240, 128, {}, ('dense', 1, 320, 0)),
    'dense_2x256': (40, 80, 320, 96, {}, ('dense', 2, 256, 0)),
    'dense_2x320': (60, 100, 500, 64, {}, ('dense', 2, 320, 0)),
    'dense_2x320_spec': (100, 100, 500, 64, {}, ('dense', 2, 320, 0)),         # SPEC at ple = 2
    'dense_3x256': (30, 140, 560, 64, {}, ('dense', 3, 256, 0)),
    'dense_3x320': (25, 160, 640, 64, {}, ('dense', 3, 320, 0)),
    'dense_4x256': (20, 200, 800, 48, {}, ('dense', 4, 256, 0)),
    'dense_4x256_n1024': (25, 224, 800, 48, {}, ('dense', 4, 256, 0)),       # the largest dense N
    'dense_4x256_one_rb': (1, 224, 800, 48, {}, ('dense', 4, 256, 0)),       # ... with every link on one RB: 1023 interferers
    'dense_3x256_cue_heavy': (30, 560, 140, 64, {}, ('dense', 3, 256, 0)),   # CUE links in slots k >= 1
    'dense_1x320_due_only': (40, 0, 320, 96, {}, ('dense', 1, 320, 0)),
    'sorting_1': (600, 40, 160, 64, {}, ('sorting', 1, 0, 0)),                 # R > 512
    'sorting_2': (600, 80, 320, 64, {}, ('sorting', 2, 0, 0)),
    'sorting_3': (600, 140, 560, 48, {}, ('sorting', 3, 0, 0)),
    'sorting_3_big_bins': (300, 100, 500, 48, {}, ('sorting', 3, 0, 0)),      # R <= 512, but the dense layout is over 75 KB
    'sorting_4': (600, 200, 800, 32, {}, ('sorting', 4, 0, 0)),
    'sorting_4_n1024': (600, 224, 800, 32, {}, ('sorting', 4, 0, 0)),
    'sorting_3_cue_heavy': (600, 560, 140, 48, {}, ('sorting', 3, 0, 0)),
    'sorting_2_due_only': (600, 0, 400, 64, {}, ('sorting', 2, 0, 0)),
    'general_n1025': (25, 225, 800, 32, {}, ('general', 0, 0, 0)),
    'general_n2000': (100, 400, 1600, 32, {}, ('general', 0, 0, 0)),
    'general_n3000': (100, 600, 2400, 32, {}, ('general', 0, 0, 0)),
    'general_n3300': (100, 1100, 2200, 32, {}, ('general', 0, 0, 0)),         # exactly 227 KB of shared memory
}


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.fail('the gpu tier needs a CUDA device (no CPU fallback exists)')


def _device_overrides(cfg, rng):
    """Per-device 'config' entries for about one UE in seven (simulator.py:31: such an entry replaces the env-level dict)."""
    ids = cfg.device_ids()[1:]
    out = {}
    for i in rng.choice(len(ids), size=max(2, len(ids) // 7), replace=False):
        out[ids[i]] = dict(tx_antenna_gain_dBi=float(rng.uniform(-3, 5)), rx_antenna_gain_dBi=float(rng.uniform(-3, 5)),
                           thermal_noise_dBm=float(rng.uniform(-110, -100)), noise_figure_dB=float(rng.uniform(5, 9)),
                           sinr_dB=float(rng.uniform(-12, -8)), body_loss_dB=float(rng.uniform(0, 4)),
                           num_subcarriers=int(rng.choice([12, 24])), subcarrier_spacing_kHz=15)
    return out


def _setup(monkeypatch, tmp_path, shape, ple=2.0, cost_hata=False, overrides=False, seed_tag=''):
    """(VecD2DEnv kwargs, oracle config, E, rng) of a cell; applies the shape's environment knobs."""
    import gym_d2d_b200 as G
    R, C, D, E, knobs, _ = SHAPES[shape]
    kw = dict(num_rbs=R, num_cues=C, num_due_pairs=D)
    okw = dict(kw)
    if cost_hata:
        kw['path_loss_model'] = G.CostHataPathLoss
        okw['path_loss_model'] = 'cost_hata'
    elif ple != 2.0:
        kw['path_loss_model'] = functools.partial(G.LogDistancePathLoss, ple=ple)
        okw['ple'] = ple
    rng = np.random.default_rng(zlib.crc32(f'{shape}/{ple}/{cost_hata}/{overrides}/{seed_tag}'.encode()))
    if overrides:
        ov = _device_overrides(O.OracleConfig(**okw), rng)
        f = tmp_path / 'device_config.json'
        f.write_text(json.dumps({k: {'config': v} for k, v in ov.items()}))
        kw['device_config_file'] = f
        okw['device_overrides'] = ov
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    return kw, O.OracleConfig(**okw), E, rng


def _make_env(shape, kw, E, info, exact=False):
    """The env, after asserting that the library picked the shape's kernel (step_geometry against tests/_kernel_dispatch.py)."""
    import gym_d2d_b200 as G
    _need_gpu()
    want = expected_kernel(kw, E)
    assert (want['family'], want['lpt'], want['bt'], want['wpb']) == SHAPES[shape][5], (shape, want)
    env = G.VecD2DEnv(E, dict(kw), device='cuda', info=info, exact_positions=exact)
    geo = env.step_geometry()
    assert (geo['block'], geo['smem_bytes']) == (want['block'], want['smem']), (shape, want, geo)
    return env, want


def _npw(cfg):
    return np.where(np.arange(cfg.num_links) < cfg.num_cues, cfg.cue_max_tx_power_dBm + 1,
                    cfg.due_max_tx_power_dBm - cfg.due_min_tx_power_dBm + 1)


def _actions(cfg, E, rng):
    """Uniform actions; every fifth env crowds all its links onto 3 RBs (long walks, overflowing dense bins)."""
    act = O.random_actions(cfg, E, rng)
    crowded = np.arange(E) % 5 == 2
    act[crowded] = act[crowded] % (min(3, cfg.num_rbs) * _npw(cfg))
    return act


def _absent(E, N, rng):
    """~30 % of the agents absent; env 1 has a single agent."""
    active = (rng.random((E, N)) >= 0.3).astype(np.uint8)
    active[1] = 0
    active[1, int(rng.integers(N))] = 1
    return active


def _step(env, act, active=None):
    a = act if active is None else np.where(active > 0, act, -1)
    obs, reward, done, info = env.step(torch.as_tensor(a, dtype=torch.int32, device='cuda').contiguous())
    torch.cuda.synchronize()
    out = dict(obs=obs.cpu().numpy(), reward=reward.cpu().numpy(), done=done.cpu().numpy(), capacity_mbps=info['capacity_mbps'].cpu().numpy())
    if env.want_info:
        out.update(rate_bps=info['rate_bps'].cpu().numpy(), rb=info['rb'].cpu().numpy().astype(np.int32),
                   tx_pwr_dbm=info['tx_pwr_dbm'].cpu().numpy().astype(np.int32))
    return out


def _compare(out, ref, info):
    if info:
        check_against_oracle(out, ref)
    else:       # the core outputs only: the FULL instantiations write nothing else
        assert_rel(out['obs'][..., 4], ref['sinr_db'], RTOL, 'sinr_db')
        assert_rel(out['obs'][..., 5], ref['snr_db'], RTOL, 'snr_db')
        assert_rel(out['obs'][..., :4], ref['obs'][..., :4], RTOL, 'obs positions')
        assert_rel(out['capacity_mbps'], ref['capacity_mbps'], RTOL, 'capacity_mbps')
        assert_rel(out['reward'], ref['reward'], RTOL, 'reward')


def _run_cell(monkeypatch, tmp_path, shape, ple=2.0, info=True, exact=False, cost_hata=False, overrides=False, absent=False):
    kw, cfg, E, rng = _setup(monkeypatch, tmp_path, shape, ple, cost_hata, overrides, seed_tag=f'{info}/{exact}/{absent}')
    env, want = _make_env(shape, kw, E, info, exact)
    pos = O.random_positions(cfg, E, rng, fp32_exact=not exact)
    if exact and cfg.num_due_pairs:
        # every 7th env's first D2D pair 5 cm .. 1 m apart: the worst case of rounding positions to fp32
        C = cfg.num_cues
        pos[::7, 2 + C] = pos[::7, 1 + C] + rng.uniform(0.05, 1.0, (len(pos[::7]), 1)) * np.array([0.6, 0.8])
    env.set_positions(pos)
    env.reset_stats()
    for s in range(2):
        act = _actions(cfg, E, rng)
        active = _absent(E, cfg.num_links, rng) if absent else None
        out = _step(env, act, active)
        ref = O.step_batch(cfg, pos, act, active=active, nthreads=8)
        assert ref['status'] == 0
        _compare(out, ref, info)
        if active is not None:
            assert (out['obs'][active == 0][:, 4:] == 0).all() and (out['capacity_mbps'][active == 0] == 0).all()
        assert (env.step_count.cpu().numpy() == s + 1).all() and (out['done'] == 0).all()
    assert env.stats()['env_steps'] == 2 * E
    _to_episode_end(env, act, active, ref)
    env.close()
    return want


def _to_episode_end(env, act, active, ref):
    """The last actions again until the episode ends (envs/d2d_env.py:65,68): done exactly from the EPISODE_LENGTH-th step on,
    the same rewards as the oracle's for those actions, every env-step counted."""
    E, T = env.num_envs, env.episode_length
    s0 = int(env.step_count[0])
    for s in range(s0, T):
        out = _step(env, act, active)
        assert (env.step_count.cpu().numpy() == s + 1).all() and (out['done'] == (1 if s + 1 >= T else 0)).all()
    assert_rel(out['reward'], ref['reward'], RTOL, 'reward at the end of the episode')
    assert env.stats()['env_steps'] == T * E


@pytest.mark.parametrize('info', [True, False])
@pytest.mark.parametrize('ple', [2.0, 3.5])
@pytest.mark.parametrize('shape', list(SHAPES))
def test_instantiation_matches_oracle(monkeypatch, tmp_path, shape, ple, info):
    """Every shape at ple = 2 and 3.5 (the PLE2 template parameter), with and without the info outputs (FULL: exactly the core
    outputs, taken when the link constants are uniform), crowded RBs in every fifth env, two consecutive steps compared with the
    oracle, then on to the end of the episode (done)."""
    _run_cell(monkeypatch, tmp_path, shape, ple=ple, info=info)


# one shape per family (and the dense kernel's SPEC and N = 1024 shapes) for each variant of the link budget / inputs
VARIANT_SHAPES = ['warp_2w', 'dense_2x320', 'dense_4x256_n1024', 'sorting_2', 'sorting_4_n1024', 'general_n1025']


@pytest.mark.parametrize('variant', ['exact', 'cost_hata', 'overrides', 'absent'])
@pytest.mark.parametrize('shape', VARIANT_SHAPES + ['dense_2x320_spec'])
def test_variants_match_oracle(monkeypatch, tmp_path, shape, variant):
    """exact_positions=True on unrounded float64 positions with D2D pairs 5 cm - 1 m apart (the EXACT instantiations);
    CostHataPathLoss (the receiver's folded constant, ple != 2); per-device overrides through a device_config_file (the
    per-link tables instead of the constant bank); ~30 % absent agents and an env with a single agent."""
    for info in (True, False):
        _run_cell(monkeypatch, tmp_path, shape, info=info, exact=variant == 'exact', cost_hata=variant == 'cost_hata',
                  overrides=variant == 'overrides', absent=variant == 'absent')


def test_matrix_reaches_every_instantiation():
    """The (shape, ple, info) cells test_instantiation_matches_oracle is parametrized with run every compiled step-kernel
    instantiation at least once: 3 warp shapes, 7 dense shapes (+ SPEC), 4 sorting shapes and the general-topology kernel, each
    with PLE2 true and false and with FULL (info=False) true and false."""
    import itertools
    params = {}
    for m in test_instantiation_matches_oracle.pytestmark:
        if m.name == 'parametrize':
            params[m.args[0]] = list(m.args[1])
    seen = set()
    for shape, ple, info in itertools.product(params['shape'], params['ple'], params['info']):
        R, C, D, E, knobs, _ = SHAPES[shape]
        kw = dict(num_rbs=R, num_cues=C, num_due_pairs=D)
        if ple != 2.0:
            import gym_d2d_b200 as G
            kw['path_loss_model'] = functools.partial(G.LogDistancePathLoss, ple=ple)
        k = expected_kernel(kw, E, env=knobs)
        seen.add((k['family'], k['lpt'], k['bt'], k['wpb'], k['spec'], k['ple2'], not info and k['uniform']))
    want = {('warp', 0, 0, w, False, p, f) for w in (2, 4, 8) for p in (True, False) for f in (True, False)}
    want |= {('dense', l, b, 0, False, p, f) for l, b in [(1, 256), (2, 256), (3, 256), (4, 256), (1, 320), (2, 320), (3, 320)]
             for p in (True, False) for f in (True, False)}
    want |= {('dense', 2, 320, 0, True, True, f) for f in (True, False)}
    want |= {('sorting', l, 0, 0, False, p, f) for l in (1, 2, 3, 4) for p in (True, False) for f in (True, False)}
    want |= {('general', 0, 0, 0, False, p, f) for p in (True, False) for f in (True, False)}
    assert want <= seen, sorted(want - seen)


def test_past_the_general_kernels_shared_memory_is_refused_at_construction():
    """100 RBs / 800 CUEs / 3200 DUE pairs needs 275 KB of shared memory on the general-topology kernel: d2d_create refuses it
    with D2D_ERR_UNSUPPORTED (D2DUnsupportedError), not the first step.  One link fewer than the largest accepted N still runs
    (general_n3300 above is the largest at 100 RBs)."""
    import gym_d2d_b200 as G
    from gym_d2d_b200 import _lib
    _need_gpu()
    kw = dict(num_rbs=100, num_cues=800, num_due_pairs=3200)
    assert expected_kernel(kw, 4)['family'] == 'unsupported'
    with pytest.raises(_lib.D2DUnsupportedError, match='shared memory'):
        G.VecD2DEnv(4, dict(kw), device='cuda')
    kw = dict(num_rbs=100, num_cues=1101, num_due_pairs=2200)         # N = 3301: 70 bytes over 227 KB
    assert expected_kernel(kw, 4)['family'] == 'unsupported'
    with pytest.raises(_lib.D2DUnsupportedError, match='shared memory'):
        G.VecD2DEnv(4, dict(kw), device='cuda')


# ---- the fp64 pass on the block kernels: links a few hundredths of a dB from 0 dB --------------------------------------------------
def _band_scenario(cfg, E, n_rbs_band, rng, ple, lo, hi, in_band):
    """Random positions and actions, except that RBs 0 .. n_rbs_band - 1 belong to constructed links: DUE pairs alone on their RB
    with the receiver at the distance that gives SNR = SINR = +-target, DUE pairs whose SNR is 6 - 12 dB with one interfering
    pair placed so that SINR = +-target (as in test_band_edge_sweep_of_sinr_and_snr), and up to four CUEs alone on their RB at
    SNR = +-target.  Targets are uniform in [lo, hi]; in every fourth env (env 0 included) in the range in_band, inside the
    band of the fp64 pass and close enough to 0 dB that the pass rewrites the dB values.  Every other link acts on the
    remaining RBs."""
    C, D, R = cfg.num_cues, cfg.num_due_pairs, cfg.num_rbs
    npw_c, npw_d = cfg.cue_max_tx_power_dBm + 1, cfg.due_max_tx_power_dBm - cfg.due_min_tx_power_dBm + 1
    pos = O.random_positions(cfg, E, rng, fp32_exact=False)
    act = np.empty((E, cfg.num_links), np.int32)
    act[:, :C] = rng.integers(n_rbs_band, R, (E, C)) * npw_c + rng.integers(0, npw_c, (E, C))
    act[:, C:] = rng.integers(n_rbs_band, R, (E, D)) * npw_d + rng.integers(0, npw_d, (E, D))
    n_cue = min(C, 4)
    n_pair = n_rbs_band - n_cue
    n_alone = n_pair // 2
    n_ix = n_pair - n_alone
    assert n_alone + 2 * n_ix <= D
    K = 10 * ple * np.log10(cfg.carrier_freq_GHz * 1e9) + 10 * ple * np.log10(4 * np.pi / 299792458.0)
    snr0_due = -6.0 - 3.0 - K + 104.5              # UE Tx (eirp - p) + UE Rx offset - K - UE noise (device.py:12-41 defaults)
    snr0_cue = -6.0 + 17.5 - K + 118.4             # UE Tx + MBS Rx offset - K - MBS noise
    narrow = np.arange(E) % 4 == 0

    def targets(n):
        t = rng.uniform(lo, hi, (E, n))
        t[narrow] = rng.uniform(*in_band, (int(narrow.sum()), n))
        return t * rng.choice([-1.0, 1.0], (E, n))

    def unit(n):
        th = rng.uniform(0, 2 * np.pi, (E, n))
        return np.stack([np.cos(th), np.sin(th)], -1)

    rb = 0
    # CUEs alone on their RB (the receiver is the MBS at the origin)
    p = rng.integers(0, 6, (E, n_cue))
    d = 10 ** ((p + snr0_cue - targets(n_cue)) / (10 * ple))
    pos[:, 1:1 + n_cue] = d[..., None] * unit(n_cue)
    act[:, :n_cue] = (rb + np.arange(n_cue)) * npw_c + p
    rb += n_cue
    # DUE pairs alone on their RB
    dd = np.arange(n_alone)
    p = rng.integers(0, npw_d, (E, n_alone))
    d = 10 ** ((p + snr0_due - targets(n_alone)) / (10 * ple))
    tx = rng.uniform(-50, 50, (E, n_alone, 2))
    pos[:, 1 + C + 2 * dd] = tx
    pos[:, 2 + C + 2 * dd] = tx + d[..., None] * unit(n_alone)
    act[:, C + dd] = (rb + dd) * npw_d + p
    rb += n_alone
    # victim pair + one interfering pair per RB
    v = n_alone + 2 * np.arange(n_ix)
    p = rng.integers(0, npw_d, (E, n_ix))
    pi = rng.integers(0, npw_d, (E, n_ix))
    snr = rng.uniform(6.0, 12.0, (E, n_ix))
    d2 = 10 ** ((p + snr0_due - snr) / (10 * ple))
    tx = rng.uniform(-50, 50, (E, n_ix, 2))
    rx = tx + d2[..., None] * unit(n_ix)
    S = 10 ** ((p - 6.0 - 3.0 - K) / 10) * d2 ** (-ple)                   # received signal, linear mW
    I = S / 10 ** (targets(n_ix) / 10) - 10 ** (-104.5 / 10)              # interference that gives SINR = target
    w = 10 ** ((pi - 6.0 - K) / 10)                                        # interferer EIRP minus the path-loss constant
    itx = rx + ((w / I) ** (1.0 / ple))[..., None] * unit(n_ix)
    pos[:, 1 + C + 2 * v], pos[:, 2 + C + 2 * v] = tx, rx
    pos[:, 1 + C + 2 * (v + 1)], pos[:, 2 + C + 2 * (v + 1)] = itx, itx + np.array([3.0, 4.0])
    act[:, C + v] = (rb + np.arange(n_ix)) * npw_d + p
    act[:, C + v + 1] = (rb + np.arange(n_ix)) * npw_d + pi
    band_links = np.concatenate([np.arange(n_cue), C + dd, C + v])
    return pos.astype(np.float32).astype(np.float64), act, band_links


@pytest.mark.parametrize('ple', [2.0, 3.5])
@pytest.mark.parametrize('shape,n_rbs_band', [('dense_2x256', 20), ('dense_1x320', 24), ('sorting_2', 56), ('general_n2000', 40)])
def test_fp64_pass_at_the_band_edge(monkeypatch, tmp_path, shape, n_rbs_band, ple):
    """SINR and SNR a few hundredths of a dB either side of 0 dB and of the band edge of the fp64 pass (0.0625 dB at ple = 2,
    0.5 dB otherwise) on the dense, sorting and general-topology kernels.  Several band links share a warp of the dense kernel;
    the sorting kernel gets more band links per env than its cooperative queue holds (D2D_BLOCK_RESQ = 32), so the inline
    fallback runs.  The oracle judges every link of every env."""
    kw, cfg, E, rng = _setup(monkeypatch, tmp_path, shape, ple)
    band = 0.0625 if ple == 2.0 else 0.5
    # (the fp64 pass rewrites a SINR / SNR whose linear ratio is within 1/16 of one, |dB| < 0.26; at ple != 2 its band is
    # 0.5 dB, so the envs of in_band sit below 0.26 dB there and the wide range covers the band edge)
    lo, hi, in_band = (0.02, 0.15, (0.02, 0.05)) if ple == 2.0 else (0.3, 0.7, (0.02, 0.25))
    env, want = _make_env(shape, kw, E, info=True)
    pos, act, links = _band_scenario(cfg, E, n_rbs_band, rng, ple, lo, hi, in_band)
    env.set_positions(pos)
    env.reset_stats()
    out = _step(env, act)
    ref = O.step_batch(cfg, pos, act, nthreads=8)
    check_against_oracle(out, ref)
    near = np.minimum(np.abs(ref['sinr_db']), np.abs(ref['snr_db']))
    rs = ref['sinr_db'][:, links]
    # the construction hit what it aimed at: band links inside and outside the band, on both sides of 0 dB
    assert (np.abs(rs) < band).sum() > 20 and (np.abs(rs) > band).sum() > 20 and (rs > 0).sum() > 20 and (rs < 0).sum() > 20
    assert (np.abs(rs) < hi + 0.03).all() and (np.abs(rs) < 0.25).sum() > 20      # some where the pass rewrites the dB values
    inside = (near < band - 1e-3).sum(axis=1)
    if want['family'] == 'sorting':
        assert inside[0] > 32                      # one env queues more links than the cooperative pass takes
    assert env.stats()['rescues'] >= inside.sum() > 0
    env.close()


# ---- many envs per block: the sorting kernel's groups of 256 per-env scalars, the general kernel's loop over envs --------------------
@pytest.mark.parametrize('info', [True, False])
@pytest.mark.parametrize('shape', ['sorting_2', 'sorting_4_n1024', 'dense_4x256_n1024', 'general_n1025'])
def test_block_kernels_step_many_envs_per_block(monkeypatch, tmp_path, shape, info):
    """Two blocks step 700 envs (D2D_B200_GRID=2): the sorting kernel flushes a group of 256 per-env scalars (step counter,
    reward, done) in mid-range and ends on a partial group; crowded RBs (everyone on one RB, or on two), absent agents, two
    consecutive steps compared with the oracle, then on to the end of the episode; step counters, done and the statistics' env
    count checked."""
    kw, cfg, _, rng = _setup(monkeypatch, tmp_path, shape, seed_tag=f'grid2/{info}')
    monkeypatch.setenv('D2D_B200_GRID', '2')
    E = 700
    env, _ = _make_env(shape, kw, E, info)
    assert env.step_geometry()['grid'] == 2
    pos = O.random_positions(cfg, E, rng, fp32_exact=True)
    env.set_positions(pos)
    env.reset_stats()
    npw = _npw(cfg)
    for s in range(2):
        act = O.random_actions(cfg, E, rng)
        one = np.arange(E) % 5 == 0
        act[one] = act[one] % npw                                   # rb = 0 for every link
        two = np.arange(E) % 11 == 3
        act[two] = act[two] % (2 * npw)
        absent = (np.arange(E) % 7 == 0)[:, None] & (rng.random((E, cfg.num_links)) < 0.5)
        active = (~absent).astype(np.uint8)
        out = _step(env, act, active)
        ref = O.step_batch(cfg, pos, act, active=active, nthreads=8)
        _compare(out, ref, info)
        assert (out['capacity_mbps'][absent] == 0).all() and (out['obs'][..., 4][absent] == 0).all()
        assert (env.step_count.cpu().numpy() == s + 1).all() and (out['done'] == 0).all()
    assert env.stats()['env_steps'] == 2 * E
    _to_episode_end(env, act, active, ref)
    env.close()
