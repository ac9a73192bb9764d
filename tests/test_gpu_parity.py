"""GPU tier (-m gpu): the CUDA step path, called through the C ABI (VecD2DEnv / D2DEnv -> libd2d_b200.so),
against the float64 oracle on identical positions and actions, against the committed outputs of the
reference, and through size-independent properties at BASELINE.json's full sizes.

Tolerances (BASELINE.json north_star): rb / tx power bit-exact; SINR_dB, SNR_dB, rate, capacity,
observations and reward within 1e-4 RELATIVE of the float64 reference (tests/_util.RTOL), no absolute
slack - the kernel recomputes near-0 dB SINRs in fp64 for exactly this reason.
"""
import functools
import json
import zlib

import numpy as np
import pytest

from oracle import d2d_oracle as O
from tests._util import RTOL, assert_rel, check_against_oracle

torch = pytest.importorskip('torch')
pytestmark = pytest.mark.gpu


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.fail('the gpu tier needs a CUDA device (no CPU fallback exists)')


def make_vec(E, cfg_kw=None, **kw):
    _need_gpu()
    import gym_d2d_b200 as G
    return G.VecD2DEnv(E, dict(cfg_kw or {}), device='cuda', info=True, **kw)


def run_step(env, positions, actions):
    """positions float64 (E,V,2), actions int32 (E,N) numpy -> dict of numpy outputs via the device API."""
    env.set_positions(positions)
    a = torch.as_tensor(actions, dtype=torch.int32, device='cuda').contiguous()
    obs, reward, done, info = env.step(a)
    torch.cuda.synchronize()
    return dict(obs=obs.cpu().numpy(), reward=reward.cpu().numpy(), done=done.cpu().numpy(),
                capacity_mbps=info['capacity_mbps'].cpu().numpy(), rate_bps=info['rate_bps'].cpu().numpy(),
                rb=info['rb'].cpu().numpy().astype(np.int32), tx_pwr_dbm=info['tx_pwr_dbm'].cpu().numpy().astype(np.int32))


CONFIGS = {
    'default': {},
    'tiny': dict(num_rbs=1, num_cues=1, num_due_pairs=1),
    'small': dict(num_rbs=3, num_cues=4, num_due_pairs=5),
    'cue_only': dict(num_rbs=4, num_cues=9, num_due_pairs=0),
    'due_only': dict(num_rbs=5, num_cues=0, num_due_pairs=12),
    'warp_max': dict(num_rbs=64, num_cues=32, num_due_pairs=32),      # the warp kernel's limits: both lane slots full, 64 RBs
    'dense_64_links': dict(num_rbs=16, num_cues=24, num_due_pairs=40),   # N = 64, but D > 32: the dense kernel (1 x 256)
    'block_min': dict(num_rbs=16, num_cues=25, num_due_pairs=40),     # N = 65: first block-kernel size
    'dense_small': dict(num_rbs=8, num_cues=6, num_due_pairs=30),
    'dense': dict(num_rbs=100, num_cues=100, num_due_pairs=500),
    'one_rb_crowded': dict(num_rbs=1, num_cues=20, num_due_pairs=30),  # every link interferes with every other
    'many_rbs_few_links': dict(num_rbs=100, num_cues=10, num_due_pairs=20),   # R > 64 with N <= 64
    'sorting': dict(num_rbs=600, num_cues=80, num_due_pairs=320),     # R > 512: the sorting block kernel, 2 links per thread
    'general': dict(num_rbs=25, num_cues=225, num_due_pairs=800),     # N = 1025: the general-topology kernel
    'one_power_level': dict(num_rbs=6, num_cues=8, num_due_pairs=8, cue_max_tx_power_dBm=0, due_max_tx_power_dBm=0),
}


@pytest.mark.parametrize('name,E', [('default', 512), ('tiny', 64), ('small', 128), ('cue_only', 64), ('due_only', 64),
                                    ('warp_max', 96), ('dense_64_links', 96), ('block_min', 48), ('dense_small', 64), ('dense', 12),
                                    ('one_rb_crowded', 64), ('many_rbs_few_links', 64), ('one_power_level', 64)])
def test_step_matches_oracle(name, E):
    kw = CONFIGS[name]
    cfg = O.OracleConfig(**kw)
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    env = make_vec(E, kw)
    for s in range(3):
        pos = O.random_positions(cfg, E, rng, fp32_exact=True)
        act = O.random_actions(cfg, E, rng)
        out = run_step(env, pos, act)
        ref = O.step_batch(cfg, pos, act, nthreads=4)
        assert ref['status'] == 0
        check_against_oracle(out, ref)
    env.close()


def test_fp64_positions_are_rounded_once():
    """Arbitrary float64 positions are quantised to the fp32 device state; the result must match the oracle
    evaluated on the same rounded positions, and stay within tolerance of the unrounded ones for ordinary
    geometry (D2D pairs not centimetres apart)."""
    cfg = O.OracleConfig()
    rng = np.random.default_rng(5)
    E = 256
    pos = O.random_positions(cfg, E, rng, fp32_exact=False)
    act = O.random_actions(cfg, E, rng)
    env = make_vec(E)
    out = run_step(env, pos, act)
    ref32 = O.step_batch(cfg, pos.astype(np.float32).astype(np.float64), act, nthreads=4)
    check_against_oracle(out, ref32)
    np.testing.assert_array_equal(env.positions.cpu().numpy(), pos.astype(np.float32) * (np.arange(cfg.num_devices) > 0)[None, :, None])
    env.close()


@pytest.mark.parametrize('name,E', [('default', 2048), ('dense_small', 256), ('block_min', 128)])
def test_exact_positions_mode_matches_unrounded_float64(name, E):
    """exact_positions=True: arbitrary float64 positions (as a device_config_file gives them) - results within
    1e-4 relative of the oracle evaluated on the UNROUNDED positions, including very close D2D pairs."""
    kw = CONFIGS[name]
    cfg = O.OracleConfig(**kw)
    rng = np.random.default_rng(31)
    pos = O.random_positions(cfg, E, rng, fp32_exact=False)
    C = cfg.num_cues
    # make every 7th env's first D2D pair 5 cm .. 1 m apart: worst case for the fp32 rounding of positions
    pos[::7, 2 + C] = pos[::7, 1 + C] + rng.uniform(0.05, 1.0, (len(pos[::7]), 1)) * np.array([0.6, 0.8])
    act = O.random_actions(cfg, E, rng)
    env = make_vec(E, kw, exact_positions=True)
    out = run_step(env, pos, act)
    check_against_oracle(out, O.step_batch(cfg, pos, act, nthreads=4))
    env.close()


@pytest.mark.parametrize('name,kw', [
    ('default_25_25_25', {}), ('default_fp64_positions', {}),
    ('dense_small_8_6_30', dict(num_rbs=8, num_cues=6, num_due_pairs=30)),
    ('dense_100_100_500', dict(num_rbs=100, num_cues=100, num_due_pairs=500)),
    ('tiny_1_1_1', dict(num_rbs=1, num_cues=1, num_due_pairs=1)),
])
def test_reference_fixtures(golden_dir, name, kw):
    """The CUDA path against outputs of the unmodified reference (tests/golden/gen_golden.py)."""
    g = np.load(golden_dir / f'{name}.npz')
    E = g['positions'].shape[0]
    env = make_vec(E, kw, exact_positions=(name == 'default_fp64_positions'))
    for s in range(g['actions'].shape[0]):
        out = run_step(env, g['positions'], g['actions'][s])
        np.testing.assert_array_equal(out['rb'], g['rb'][s])
        np.testing.assert_array_equal(out['tx_pwr_dbm'], g['tx_pwr_dbm'][s])
        assert_rel(out['obs'][..., 4], g['sinr_db'][s], RTOL, 'sinr_db')
        assert_rel(out['obs'][..., 5], g['snr_db'][s], RTOL, 'snr_db')
        assert_rel(out['rate_bps'], g['rate_bps'][s], RTOL, 'rate_bps')
        assert_rel(out['capacity_mbps'], g['capacity_mbps'][s], RTOL, 'capacity_mbps')
        assert_rel(out['reward'], g['reward'][s], RTOL, 'reward')
        # the reference's per-agent layout (envs/obs_fn.py:43-53) for the first and last agent
        pa = env.per_agent_obs().cpu().numpy()
        assert_rel(pa[:, 0], g['agent0_obs'][s], RTOL, 'agent 0 obs')
        assert_rel(pa[:, -1], g['agentlast_obs'][s], RTOL, 'last agent obs')
    env.close()


def test_fixed_scenario_10k_steps(golden_dir):
    """BASELINE config #4: the reference's fixed device_config_file scenario, 10 000 steps of default_rng(0)
    actions, every step compared (rewards + capacity sums of all steps, full outputs every 50th step).
    The 10 000 steps are independent given the positions, so they run as a batch of 10 000 envs."""
    g = np.load(golden_dir / 'fixed_scenario_10k.npz')
    dev = json.loads((golden_dir / 'fixed_device_config.json').read_text())
    cfg = O.OracleConfig()
    pos1 = np.array([dev[i]['position'] for i in cfg.device_ids()])
    acts = g['actions'].astype(np.int32)
    T = acts.shape[0]
    env = make_vec(T, exact_positions=True)     # the file's positions are arbitrary float64
    out = run_step(env, np.broadcast_to(pos1, (T,) + pos1.shape), acts)
    assert_rel(out['reward'], g['reward'], RTOL, 'reward[10k]')
    assert_rel(out['capacity_mbps'].sum(1, dtype=np.float64), g['capsum'], RTOL, 'capsum[10k]')
    every = int(g['every'])
    np.testing.assert_array_equal(out['rb'][::every], g['rb'])
    np.testing.assert_array_equal(out['tx_pwr_dbm'][::every], g['tx_pwr_dbm'])
    assert_rel(out['obs'][::every, :, 4], g['sinr_db'], RTOL, 'sinr_db')
    assert_rel(out['obs'][::every, :, 5], g['snr_db'], RTOL, 'snr_db')
    assert_rel(out['rate_bps'][::every], g['rate_bps'], RTOL, 'rate_bps')
    assert_rel(out['capacity_mbps'][::every], g['capacity_mbps'], RTOL, 'capacity_mbps')
    # and every step against the oracle on the unrounded positions (decode bit-exact on all 500 000 actions)
    p64 = np.broadcast_to(pos1, (T,) + pos1.shape).copy()
    p64[:, 0] = 0
    check_against_oracle(out, O.step_batch(cfg, p64, acts, nthreads=4))
    assert 0 < env.stats()['rescues'] < 0.05 * T * cfg.num_links     # the fp64 path is taken, and stays rare
    env.close()


def test_free_space_equals_log_distance_ple2():
    """FreeSpacePathLoss is defined as LogDistancePathLoss(f, ple=2) (SURVEY 0.1 / path_loss.py:43-51)."""
    import gym_d2d_b200 as G
    kw = CONFIGS['dense_small']
    cfg = O.OracleConfig(**kw)
    rng = np.random.default_rng(9)
    pos, act = O.random_positions(cfg, 64, rng), O.random_actions(cfg, 64, rng)
    a = run_step(make_vec(64, dict(kw, path_loss_model=G.FreeSpacePathLoss)), pos, act)
    b = run_step(make_vec(64, dict(kw, path_loss_model=G.LogDistancePathLoss)), pos, act)
    for k in a:
        np.testing.assert_array_equal(a[k], b[k])
    check_against_oracle(a, O.step_batch(cfg, pos, act))


@pytest.mark.parametrize('name,ple', [('default', 3.5), ('dense_small', 2.7), ('block_min', 4.0)])
def test_general_path_loss_exponent(name, ple):
    """LogDistancePathLoss with ple != 2 (reachable in the reference through functools.partial)."""
    import gym_d2d_b200 as G
    kw = CONFIGS[name]
    cfg = O.OracleConfig(**kw, ple=ple)
    rng = np.random.default_rng(int(ple * 10))
    E = 128
    pos, act = O.random_positions(cfg, E, rng), O.random_actions(cfg, E, rng)
    env = make_vec(E, dict(kw, path_loss_model=functools.partial(G.LogDistancePathLoss, ple=ple)))
    check_against_oracle(run_step(env, pos, act), O.step_batch(cfg, pos, act, nthreads=4))
    env.close()


@pytest.mark.parametrize('name', ['default', 'small', 'block_min'])
def test_absent_agents(name):
    """Appendix B.8: agents missing from the action dict do not transmit (action < 0 in the tensor API)."""
    kw = CONFIGS[name]
    cfg = O.OracleConfig(**kw)
    rng = np.random.default_rng(21)
    E = 128
    pos, act = O.random_positions(cfg, E, rng), O.random_actions(cfg, E, rng)
    active = (rng.random(act.shape) < 0.7).astype(np.uint8)
    active[0] = 0                      # an env with nobody transmitting
    active[0, 0] = 1
    active[1] = 1
    ref = O.step_batch(cfg, pos, act, active=active, nthreads=4)
    env = make_vec(E, kw)
    out = run_step(env, pos, np.where(active > 0, act, -1).astype(np.int32))
    check_against_oracle(out, ref)
    assert (out['obs'][active == 0][:, 4:] == 0).all() and (out['capacity_mbps'][active == 0] == 0).all()
    env.close()


def test_near_zero_db_sinr_is_rescued():
    """Links engineered to sit within +-0.1 dB of 0 dB SINR: a pure 1e-4 relative tolerance on a value that
    crosses zero needs the fp64 rescue path; check it is taken and that it delivers."""
    kw = dict(num_rbs=1, num_cues=1, num_due_pairs=1)
    cfg = O.OracleConfig(**kw)
    E = 4096
    rng = np.random.default_rng(17)
    pos = np.zeros((E, 4, 2))
    pos[:, 1] = [300.0, 0.0]                                   # CUE
    pos[:, 2] = [-200.0, 50.0]                                 # DUE tx
    pos[:, 3, 0] = -200.0 + rng.uniform(5.0, 19.0, E)
    pos[:, 3, 1] = 50.0
    pos = pos.astype(np.float32).astype(np.float64)
    act = np.zeros((E, 2), np.int32)
    act[:, 0] = 23
    act[:, 1] = 10
    # move the CUE along x until the DUE link's SINR is ~0 dB (bisection on the oracle)
    lo, hi = np.full(E, 0.5), np.full(E, 4000.0)
    tx, rx = pos[:, 2], pos[:, 3]
    for _ in range(60):
        mid = 0.5 * (lo + hi)
        pos[:, 1, 0] = rx[:, 0] + mid
        pos[:, 1, 1] = rx[:, 1]
        s = O.step_batch(cfg, pos, act)['sinr_db'][:, 1]
        lo = np.where(s < 0, mid, lo)
        hi = np.where(s < 0, hi, mid)
    pos = pos.astype(np.float32).astype(np.float64)
    ref = O.step_batch(cfg, pos, act)
    assert (np.abs(ref['sinr_db'][:, 1]) < 0.1).mean() > 0.9
    env = make_vec(E, kw)
    env.reset_stats()
    out = run_step(env, pos, act)
    check_against_oracle(out, ref)
    assert env.stats()['rescues'] > 0.9 * E
    env.close()


def test_penalty_branch_and_device_overrides(golden_dir):
    """envs/reward_fn.py:30-41 through a device_config_file with per-device overrides (simulator.py:31),
    driven through the dict API (D2DEnv) so key parsing, file loading and the reward broadcast are covered."""
    import gym_d2d_b200 as G
    _need_gpu()
    doc = json.loads((golden_dir / 'overrides_penalty.json').read_text())
    env = G.make('D2DEnv-v0', env_config=dict(doc['env_config'], device_config_file=golden_dir / 'overrides_device_config.json'))
    env.reset()
    keys = doc['keys']
    seen = set()
    for s, act in enumerate(doc['actions']):
        obs, rewards, done, info = env.step(dict(zip(keys, act)))
        assert list(rewards) == keys and len(set(rewards.values())) == 1
        assert_rel(rewards[keys[0]], doc['reward'][s], RTOL, 'reward')
        seen.add(rewards[keys[0]] == -1.0)
        for i, k in enumerate(keys):
            assert info[k]['rb'] == doc['rb'][s][i] and info[k]['tx_pwr_dbm'] == doc['tx_pwr_dbm'][s][i]
            for f in ['sinr_db', 'snr_db', 'rate_bps', 'capacity_mbps']:
                assert_rel(info[k][f], doc[f][s][i], RTOL, f)
        assert done['__all__'] == (s + 1 >= 10)
    assert seen == {True, False}
    env.close()


def test_dict_api_subset_order_and_layout(golden_dir):
    """Appendix B.8 + envs/obs_fn.py:43-53 through D2DEnv: a subset of agents in caller order."""
    import gym_d2d_b200 as G
    _need_gpu()
    doc = json.loads((golden_dir / 'subset_order.json').read_text())
    env = G.D2DEnv(dict(doc['env_config']))
    first = env.reset()
    assert list(first) == doc['keys_all'] and first[doc['keys_all'][0]].shape == (6 * len(doc['keys_all']),)
    assert first[doc['keys_all'][0]].dtype == np.float64
    env.set_device_positions({id_: p for id_, p in zip(env.device_ids, doc['positions'])})
    keys = [doc['keys_all'][i] for i in doc['order']]
    obs, rewards, done, info = env.step({k: doc['actions_all'][i] for k, i in zip(keys, doc['order'])})
    assert list(obs) == keys
    for i, k in enumerate(keys):
        assert_rel(obs[k], doc['per_agent_obs'][i], RTOL, f'obs[{k}]')
        assert_rel(info[k]['capacity_mbps'], doc['capacity_mbps'][i], RTOL, 'capacity')
        assert_rel(rewards[k], doc['reward'][i], RTOL, 'reward')
    # error behaviour of the reference surface
    with pytest.raises(ValueError, match='Unable to decode action type'):
        env.step({keys[0]: 1.5})
    with pytest.raises(KeyError):
        env.step({'nope:mbs': 1})
    env.close()


def test_appendix_c_through_dict_api(golden_dir):
    import gym_d2d_b200 as G
    _need_gpu()
    doc = json.loads((golden_dir / 'appendix_c.json').read_text())
    env = G.make('D2DEnv-v0', env_config=dict(doc['env_config']))
    env.reset()
    env.set_device_positions(dict(zip(env.device_ids, doc['positions'])))
    obs, rewards, done, info = env.step(dict(zip(doc['keys'], doc['actions'])))
    for i, k in enumerate(doc['keys']):
        assert_rel(obs[k], doc['per_agent_obs'][k], RTOL, k)
        assert info[k]['rb'] == doc['rb'][i] and info[k]['tx_pwr_dbm'] == doc['tx_pwr_dbm'][i]
        assert_rel(rewards[k], doc['reward'], RTOL, 'reward')
    env.close()


def test_save_and_reload_device_config(tmp_path):
    """envs/d2d_env.py:124-134 + envs/env_config.py:32-37 round trip through the CUDA env."""
    import gym_d2d_b200 as G
    _need_gpu()
    env = G.D2DEnv({}, seed=3)
    env.reset()
    f = tmp_path / 'device_config.json'
    env.save_device_config(f)
    doc = json.loads(f.read_text())
    assert list(doc) == env.device_ids and doc['mbs']['position'] == [0.0, 0.0]
    assert doc['cue00']['config']['max_tx_power_dBm'] == 23 and doc['due00']['config']['max_tx_power_dBm'] == 20
    env2 = G.D2DEnv({'device_config_file': f}, seed=99)
    env2.reset()
    assert env2.device_positions() == env.device_positions()
    acts = {k: 7 for k in env.link_keys}
    o1, r1, _, _ = env.step(acts)
    o2, r2, _, _ = env2.step(acts)
    assert r1 == r2 and all((o1[k] == o2[k]).all() for k in o1)
    env.close(); env2.close()


def test_reset_kernel_matches_philox_oracle():
    cfg = O.OracleConfig()
    E = 2048
    env = make_vec(E, seed=1234, global_env_offset=1000)
    env.reset()
    torch.cuda.synchronize()
    got = env.positions.cpu().numpy().astype(np.float64)
    ref = O.reset_positions(cfg, seed=1234, first_global_env=1000, num_envs=E)
    # fp32 sincospi / sqrt vs float64: ~1e-4 m absolute at 500 m; an accept/reject decision of the in-cell
    # re-draw can flip only when a candidate lies within that distance of the cell edge
    close = np.abs(got - ref).max(-1) < 5e-3
    assert close.mean() > 0.9995
    assert (got[:, 0] == 0).all()
    assert ((got ** 2).sum(-1) <= cfg.cell_radius_m ** 2 * (1 + 1e-6)).all()
    tx, rx = got[:, 1 + cfg.num_cues::2], got[:, 2 + cfg.num_cues::2]
    assert (np.sqrt(((tx - rx) ** 2).sum(-1)) <= cfg.d2d_radius_m * (1 + 1e-5)).all()
    # uniform-in-disc: E[r^2] = R^2 / 2 (position.py:24-28)
    r2 = (got[:, 1:1 + cfg.num_cues] ** 2).sum(-1)
    assert abs(r2.mean() / (cfg.cell_radius_m ** 2 / 2) - 1) < 0.02
    # sharding invariance: the same global envs drawn by another "rank"
    env2 = make_vec(256, seed=1234, global_env_offset=1000 + 512)
    env2.reset()
    np.testing.assert_array_equal(env2.positions.cpu().numpy(), env.positions[512:768].cpu().numpy())
    env.close(); env2.close()


def test_episode_counter_done_and_masked_reset():
    E = 64
    env = make_vec(E, CONFIGS['small'])
    obs0 = env.reset()
    assert obs0.shape == (E, 9, 6) and (env.step_count == 0).all()        # the reset step is not counted
    p0 = env.positions.clone()
    for t in range(1, 13):
        _, _, done, _ = env.step(env.sample_actions())
        assert (env.step_count == t).all()
        assert (done == (1 if t >= 10 else 0)).all()                       # envs/d2d_env.py:68, no auto-reset
    assert (env.positions == p0).all()                                     # positions only change on reset
    mask = torch.zeros(E, dtype=torch.uint8, device='cuda')
    mask[::2] = 1
    env.reset(mask=mask)
    assert (env.step_count[::2] == 0).all() and (env.step_count[1::2] == 12).all()
    assert (env.positions[1::2] == p0[1::2]).all() and not (env.positions[::2] == p0[::2]).all()
    env.close()


def test_stats_accumulate_and_match():
    E = 1000
    cfg = O.OracleConfig()
    env = make_vec(E)
    env.reset(seed=5)
    env.reset_stats()
    tot_r = tot_c = tot_r2 = 0.0
    for _ in range(3):
        _, reward, _, info = env.step(env.sample_actions())
        r = reward.double().cpu().numpy()
        tot_r += r.sum(); tot_r2 += (r * r).sum(); tot_c += info['capacity_mbps'].double().sum().item()
    st = env.stats()
    assert st['env_steps'] == 3 * E
    assert st['sum_reward'] == pytest.approx(tot_r, rel=1e-5)
    assert st['sum_capacity_mbps'] == pytest.approx(tot_c, rel=1e-5)
    assert st['sum_reward_sq'] == pytest.approx(tot_r2, rel=1e-5)
    env.close()


def test_host_call_equals_device_call():
    """d2d_step_host (host buffers, copies inside) returns exactly what the device-pointer call computes."""
    cfg = O.OracleConfig()
    E = 300
    rng = np.random.default_rng(2)
    pos, act = O.random_positions(cfg, E, rng), O.random_actions(cfg, E, rng)
    env = make_vec(E)
    dev = run_step(env, pos, act)
    host = env.step_host(act)
    for k in ['obs', 'capacity_mbps', 'reward', 'rate_bps']:
        np.testing.assert_array_equal(host[k], dev[k])
    np.testing.assert_array_equal(host['rb'], dev['rb'])
    assert (host['done'] == 0).all() and (env.step_count == 2).all()
    env.close()


@pytest.mark.parametrize('name', ['default', 'block_min'])
def test_chunked_launch_equals_single_launch(name, monkeypatch):
    """Batches beyond 2^31 / max(6N, 2V) envs are stepped in several launches with offset pointers; force tiny
    chunks (D2D_B200_CHUNK) and require bit-identical results, counters and statistics."""
    kw = CONFIGS[name]
    cfg = O.OracleConfig(**kw)
    E = 1000
    rng = np.random.default_rng(4)
    pos, act = O.random_positions(cfg, E, rng), O.random_actions(cfg, E, rng)
    whole = make_vec(E, kw)
    monkeypatch.setenv('D2D_B200_CHUNK', '300')
    parts = make_vec(E, kw)
    monkeypatch.delenv('D2D_B200_CHUNK')
    for env in (whole, parts):
        env.reset_stats()
    a, b = run_step(whole, pos, act), run_step(parts, pos, act)
    assert parts.launch_count - whole.launch_count == 3          # 4 launches instead of 1
    for k in a:
        if name == 'default' or a[k].dtype.kind in 'iu':
            np.testing.assert_array_equal(a[k], b[k], err_msg=k)
        else:   # block kernel: the order of links inside an RB bin follows the shared-memory atomics, so the fp32
            np.testing.assert_allclose(a[k], b[k], rtol=2e-5, atol=0, err_msg=k)   # interference sum may differ in the last bit
    assert torch.equal(whole.step_count, parts.step_count)
    sa, sb = whole.stats(), parts.stats()
    assert sa['env_steps'] == sb['env_steps'] == E and sa['sum_reward'] == pytest.approx(sb['sum_reward'], rel=1e-6)
    whole.close(); parts.close()


def test_out_of_range_actions_cannot_corrupt_memory():
    """Appendix B.9: the reference decodes out-of-range actions silently.  The tensor API leaves their result
    unspecified but must stay memory-safe and must not disturb other envs (run under compute-sanitizer too)."""
    cfg = O.OracleConfig()
    E = 256
    rng = np.random.default_rng(12)
    pos, act = O.random_positions(cfg, E, rng), O.random_actions(cfg, E, rng)
    bad = act.copy()
    bad[::2, ::7] = 2 ** 31 - 1
    bad[::2, 1::7] = 600 * 50
    env = make_vec(E)
    out = run_step(env, pos, bad)
    ref = O.step_batch(cfg, pos, act, nthreads=4)
    clean = np.arange(1, E, 2)
    assert_rel(out['obs'][clean, :, 4], ref['sinr_db'][clean], RTOL, 'untouched envs')
    assert_rel(out['reward'][clean], ref['reward'][clean], RTOL, 'untouched envs reward')
    env.close()


def test_pipelined_host_steps_equal_synchronous_ones():
    """d2d_step_host_async / _wait with two steps in flight deliver, step for step, what d2d_step_host delivers."""
    cfg = O.OracleConfig()
    E, T = 500, 7
    rng = np.random.default_rng(8)
    pos = O.random_positions(cfg, E, rng)
    acts = [O.random_actions(cfg, E, rng) for _ in range(T)]
    sync_env, pipe_env = make_vec(E), make_vec(E)
    sync_env.set_positions(pos); pipe_env.set_positions(pos)
    want = [{k: v.copy() for k, v in sync_env.step_host(a).items()} for a in acts]
    outs = [pipe_env.alloc_host_outputs(pinned=True), pipe_env.alloc_host_outputs(pinned=True)]
    got = []
    for i, a in enumerate(acts):
        if i >= 2:
            pipe_env.step_host_wait(i & 1)
            got.append({k: v.copy() for k, v in outs[i & 1].items()})
        pipe_env.step_host_async(a, outs[i & 1], i & 1)
    for i in (T - 2, T - 1):
        pipe_env.step_host_wait(i & 1)
        got.append({k: v.copy() for k, v in outs[i & 1].items()})
    for w, g in zip(want, got):
        for k in w:
            np.testing.assert_array_equal(w[k], g[k], err_msg=k)
    assert (got[-1]['done'] == 0).all() and (pipe_env.step_count == T).all()
    sync_env.close(); pipe_env.close()


@pytest.mark.parametrize('E', [100, 4096, 70000])      # the three launch shapes of the warp kernel (2-, 4- and 8-warp blocks)
def test_core_output_fast_path_equals_general_path(E):
    """VecD2DEnv(info=False) passes exactly the core outputs and takes the kernel instantiation that tests no output
    pointer; it must produce bit-identical obs / capacity / reward / done to the general instantiation."""
    import gym_d2d_b200 as G
    _need_gpu()
    cfg = O.OracleConfig()
    rng = np.random.default_rng(E)
    pos, act = O.random_positions(cfg, E, rng), O.random_actions(cfg, E, rng)
    act[::5, ::3] = -1                                   # some absent agents too
    a = torch.as_tensor(act, device='cuda')
    fast, gen = G.VecD2DEnv(E, {}, info=False), G.VecD2DEnv(E, {}, info=True)
    for env in (fast, gen):
        env.set_positions(pos)
        env.step(a)
    torch.cuda.synchronize()
    for name in ('obs', 'capacity_mbps', 'reward', 'done'):
        assert torch.equal(getattr(fast, name), getattr(gen, name)), name
    ref = O.step_batch(cfg, pos, act, active=(act >= 0).astype(np.uint8), nthreads=4)
    assert_rel(fast.obs[..., 4].cpu().numpy(), ref['sinr_db'], RTOL, 'sinr_db')
    assert_rel(fast.capacity_mbps.cpu().numpy(), ref['capacity_mbps'], RTOL, 'capacity')
    assert_rel(fast.reward.cpu().numpy(), ref['reward'], RTOL, 'reward')
    fast.close(); gen.close()


@pytest.mark.parametrize('exact', [False, True])
def test_warp_launch_shapes_bit_identical(monkeypatch, exact):
    """The warp kernel's three launch shapes (2-, 4-, 8-warp blocks; D2D_B200_WPB forces one) differ in where the fp64 pass
    runs - before griddepcontrol.wait with its results kept in registers (2-warp latency shape), or after the env's stores,
    overwriting them - and must produce bit-identical outputs, counters and statistics, each within tolerance of the oracle.
    Crowded RBs (all agents on 3 RBs in a third of the envs) take the all-pairs path and several fp64 links per env."""
    import gym_d2d_b200 as G
    _need_gpu()
    cfg = O.OracleConfig()
    E = 1500
    rng = np.random.default_rng(77)
    pos = O.random_positions(cfg, E, rng, fp32_exact=not exact)
    act = O.random_actions(cfg, E, rng)
    act[::3, :cfg.num_cues] = (act[::3, :cfg.num_cues] % (3 * 24))        # CUE action = rb * 24 + p
    act[::3, cfg.num_cues:] = (act[::3, cfg.num_cues:] % (3 * 21))        # DUE action = rb * 21 + p
    act[::7, ::4] = -1
    a = torch.as_tensor(act, device='cuda')
    got = {}
    for wpb in (2, 4, 8, 102, 104, 108):            # 10x: the same shape on 40 blocks, so every warp steps 5-19 envs
        monkeypatch.setenv('D2D_B200_WPB', str(wpb % 100))
        if wpb > 100:
            monkeypatch.setenv('D2D_B200_GRID', '40')
        env = G.VecD2DEnv(E, {}, info=True, exact_positions=exact)
        assert env.step_geometry()['block'] == 32 * (wpb % 100) and (wpb < 100 or env.step_geometry()['grid'] == 40)
        env.set_positions(pos)
        for _ in range(3):                          # back-to-back launches: the programmatic-dependent-launch path
            env.step(a)
        torch.cuda.synchronize()
        st = env.stats()
        assert st['rescues'] > 0
        got[wpb] = dict(obs=env.obs.clone(), cap=env.capacity_mbps.clone(), reward=env.reward.clone(), done=env.done.clone(),
                        rate=env.rate_bps.clone(), count=env.step_count.clone(), rescues=st['rescues'], cap_sum=st['sum_capacity_mbps'])
        env.close()
        # the same three steps as ONE d2d_step_many launch of this shape
        many = G.VecD2DEnv(E, {}, info=True, exact_positions=exact)
        many.set_positions(pos)
        out = many.step_many(torch.stack([a, a, a]).contiguous())
        torch.cuda.synchronize()
        for k, v in dict(obs='obs', cap='capacity_mbps', reward='reward', done='done', rate='rate_bps').items():
            assert torch.equal(out[v][2], got[wpb][k]), (wpb, 'step_many', k)
        assert torch.equal(many.step_count, got[wpb]['count']) and many.stats()['rescues'] == st['rescues']
        many.close()
    monkeypatch.delenv('D2D_B200_WPB')
    monkeypatch.delenv('D2D_B200_GRID')
    for wpb in (4, 8, 102, 104, 108):
        for k in ('obs', 'cap', 'reward', 'done', 'rate', 'count'):
            assert torch.equal(got[2][k], got[wpb][k]), (wpb, k)
        assert got[2]['rescues'] == got[wpb]['rescues']
    assert (got[2]['count'] == 3).all()
    ref = O.step_batch(cfg, pos, act, active=(act >= 0).astype(np.uint8), nthreads=4)
    assert_rel(got[2]['obs'][..., 4].cpu().numpy(), ref['sinr_db'], RTOL, 'sinr_db')
    assert_rel(got[2]['obs'][..., 5].cpu().numpy(), ref['snr_db'], RTOL, 'snr_db')
    assert_rel(got[2]['cap'].cpu().numpy(), ref['capacity_mbps'], RTOL, 'capacity')
    assert_rel(got[2]['rate'].cpu().numpy(), ref['rate_bps'], RTOL, 'rate')
    assert_rel(got[2]['reward'].cpu().numpy(), ref['reward'], RTOL, 'reward')


def test_step_is_graph_capturable_and_deterministic():
    E = 512
    env = make_vec(E)
    env.reset(seed=11)
    a = env.sample_actions()
    env.step(a)
    torch.cuda.synchronize()
    eager = (env.obs.clone(), env.reward.clone(), env.capacity_mbps.clone())
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        env.step(a)                       # warm-up on the capture stream
        with torch.cuda.graph(g, stream=s):
            env.step(a)
    env.obs.zero_(); env.reward.zero_(); env.capacity_mbps.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(env.obs, eager[0]) and torch.equal(env.reward, eager[1]) and torch.equal(env.capacity_mbps, eager[2])
    env.close()


# ---- BASELINE.json full sizes: size-independent properties + sampled oracle checks ---------------------------
def _properties(env, cfg, actions):
    obs, reward, done, info = env.step(actions)
    torch.cuda.synchronize()
    cap = info['capacity_mbps']
    sinr, snr = obs[..., 4], obs[..., 5]
    assert torch.isfinite(obs).all() and torch.isfinite(cap).all()
    assert (sinr <= snr + 1e-3).all()                                   # interference can only lower SINR
    ok = reward != -1.0
    mean_cap = cap.double().mean(dim=1)
    assert torch.allclose(reward[ok].double(), mean_cap[ok], rtol=2e-5)  # envs/reward_fn.py:42
    C = cfg.num_cues
    pos = env.positions
    assert torch.equal(obs[:, :C, 0:2], pos[:, 1:1 + C])                 # tx of CUE j = device 1+j
    assert torch.equal(obs[:, C:, 0:2], pos[:, 1 + C::2]) and torch.equal(obs[:, C:, 2:4], pos[:, 2 + C::2])
    assert (obs[:, :C, 2:4] == 0).all()                                  # MBS at the origin
    return obs.clone(), reward.clone(), cap.clone()


def test_config2_4096_default_envs_properties():
    """BASELINE configs[1]: 4096 default envs; env-permutation equivariance + idempotence + sampled oracle."""
    cfg = O.OracleConfig()
    E = 4096
    env = make_vec(E)
    env.reset(seed=0)
    a = env.sample_actions()
    obs, reward, cap = _properties(env, cfg, a)
    obs2, reward2, cap2 = _properties(env, cfg, a)
    assert torch.equal(obs, obs2) and torch.equal(reward, reward2)       # stateless given positions + actions
    perm = torch.randperm(E, device='cuda')
    env.positions.copy_(env.positions[perm].clone())
    obs3, reward3, cap3 = _properties(env, cfg, a[perm].contiguous())
    assert torch.equal(obs3, obs[perm]) and torch.equal(reward3, reward[perm]) and torch.equal(cap3, cap[perm])
    idx = torch.arange(0, E, 64, device='cuda')
    ref = O.step_batch(cfg, env.positions[idx].double().cpu().numpy(), a[perm][idx].cpu().numpy(), nthreads=4)
    assert_rel(obs3[idx, :, 4].cpu().numpy(), ref['sinr_db'], RTOL, 'sinr_db')
    assert_rel(cap3[idx].cpu().numpy(), ref['capacity_mbps'], RTOL, 'capacity')
    assert_rel(reward3[idx].cpu().numpy(), ref['reward'], RTOL, 'reward')
    env.close()


def test_config5_slice_131072_default_envs_properties():
    """BASELINE configs[4]: one GPU's slice (131 072 envs) of the 1M-env run.  Every warp steps a contiguous range of 37 envs
    here, so the per-group scalar I/O (groups of 32 + a partial group) is exercised: reward / done / step counters of ALL
    envs are checked against the per-link outputs, sampled envs against the oracle, statistics against the outputs."""
    cfg = O.OracleConfig()
    E = 131072
    env = make_vec(E)
    env.reset(seed=5)
    env.reset_stats()
    a = env.sample_actions()
    obs, reward, cap = _properties(env, cfg, a)                    # counted step 1 (incl. reward == mean capacity for every env)
    assert (env.step_count == 1).all() and (env.done == 0).all()
    for _ in range(9):
        env.step(a)
    torch.cuda.synchronize()
    assert (env.step_count == 10).all() and (env.done == 1).all()        # EPISODE_LENGTH = 10 (envs/d2d_env.py:16,68)
    assert torch.equal(env.reward, reward)                               # same actions, same positions: same reward
    st = env.stats()
    assert st['env_steps'] == 10 * E
    assert st['sum_reward'] == pytest.approx(10 * float(reward.double().sum()), rel=1e-5)
    assert st['sum_capacity_mbps'] == pytest.approx(10 * float(cap.double().sum()), rel=1e-5)
    idx = torch.arange(17, E, 2048, device='cuda')
    ref = O.step_batch(cfg, env.positions[idx].double().cpu().numpy(), a[idx].cpu().numpy(), nthreads=4)
    assert_rel(obs[idx, :, 4].cpu().numpy(), ref['sinr_db'], RTOL, 'sinr_db')
    assert_rel(cap[idx].cpu().numpy(), ref['capacity_mbps'], RTOL, 'capacity')
    assert_rel(reward[idx].cpu().numpy(), ref['reward'], RTOL, 'reward')
    env.close()


def test_config3_dense_65536_free_space_properties():
    """BASELINE configs[2]: 100 RBs / 100 CUEs / 500 DUE pairs, 65 536 envs, FreeSpacePathLoss."""
    import gym_d2d_b200 as G
    kw = dict(CONFIGS['dense'], path_loss_model=G.FreeSpacePathLoss)
    cfg = O.OracleConfig(**CONFIGS['dense'])
    E = 65536
    env = make_vec(E, kw)
    env.reset(seed=3)
    a = env.sample_actions()
    obs, reward, cap = _properties(env, cfg, a)
    idx = torch.arange(0, E, 4096, device='cuda')
    ref = O.step_batch(cfg, env.positions[idx].double().cpu().numpy(), a[idx].cpu().numpy(), nthreads=4)
    assert_rel(obs[idx, :, 4].cpu().numpy(), ref['sinr_db'], RTOL, 'sinr_db')
    assert_rel(obs[idx, :, 5].cpu().numpy(), ref['snr_db'], RTOL, 'snr_db')
    assert_rel(cap[idx].cpu().numpy(), ref['capacity_mbps'], RTOL, 'capacity')
    assert_rel(reward[idx].cpu().numpy(), ref['reward'], RTOL, 'reward')
    env.close()


def test_unsupported_plugins_rejected_on_gpu_box():
    """Construction-time rejection also holds with a device present (no kernel launch needed)."""
    import gym_d2d_b200 as G

    class MyPathLoss(G.LogDistancePathLoss):   # examples/custom_path_loss.py-style subclass
        pass

    class MyReward(G.ShannonRewardFunction):
        pass

    for bad in (dict(path_loss_model=MyPathLoss), dict(reward_fn=MyReward)):
        with pytest.raises(G.UnsupportedPluginError):
            make_vec(4, bad)
    with pytest.raises(TypeError):
        make_vec(4, dict(not_a_key=1))


@pytest.mark.parametrize('name', ['default', 'small', 'one_rb_crowded', 'block_min'])
def test_step_many_equals_consecutive_steps(name):
    """d2d_step_many (T steps of every env in one launch, positions read once) writes, slice by slice, exactly what T
    d2d_step calls write - observations, capacities, rewards, done flags, info, step counters and statistics - and the
    first slices match the float64 oracle."""
    kw = CONFIGS[name]
    cfg = O.OracleConfig(**kw)
    E, T = 333, 13                      # > EPISODE_LENGTH steps: done flips inside the fused launch
    rng = np.random.default_rng(21)
    pos = O.random_positions(cfg, E, rng)
    acts = np.stack([O.random_actions(cfg, E, rng) for _ in range(T)])
    acts[3, ::5, ::3] = -1              # some agents absent in one of the steps
    one, many = make_vec(E, kw), make_vec(E, kw)
    for env in (one, many):
        env.set_positions(pos)
        env.reset_stats()
    a_dev = torch.as_tensor(acts, dtype=torch.int32, device='cuda').contiguous()
    ref = {k: [] for k in ['obs', 'capacity_mbps', 'reward', 'done', 'rate_bps', 'rb', 'tx_pwr_dbm']}
    for t in range(T):
        obs, reward, done, info = one.step(a_dev[t])
        for k, v in dict(obs=obs, reward=reward, done=done, **{k: info[k] for k in ['capacity_mbps', 'rate_bps', 'rb', 'tx_pwr_dbm']}).items():
            ref[k].append(v.clone())
    out = many.step_many(a_dev)
    torch.cuda.synchronize()
    if name != 'block_min':
        assert many.launch_count - one.launch_count == 1 - T      # one launch instead of T
    for k in ref:
        want, got = torch.stack(ref[k]).cpu().numpy(), out[k].cpu().numpy()
        if name == 'block_min' and want.dtype.kind == 'f':   # block kernel: bin order follows the shared-memory atomics
            np.testing.assert_allclose(got, want, rtol=2e-5, atol=0, err_msg=k)
        else:
            np.testing.assert_array_equal(got, want, err_msg=k)
    assert torch.equal(one.step_count, many.step_count) and int(many.step_count[0]) == T
    assert out['done'][8].sum() == 0 and out['done'][9].all()       # EPISODE_LENGTH = 10 (envs/d2d_env.py:16,68)
    sa, sb = one.stats(), many.stats()
    assert sa['env_steps'] == sb['env_steps'] == E * T
    assert sa['sum_reward'] == pytest.approx(sb['sum_reward'], rel=1e-6) and sa['rescues'] == sb['rescues']
    o = O.step_batch(cfg, pos, acts[0], nthreads=4)
    assert_rel(out['obs'][0, :, :, 4].cpu().numpy(), o['sinr_db'], RTOL, 'step_many slice 0 vs oracle')
    one.close(); many.close()


# ---- SURVEY 8(f)-3: the remaining built-in plugins ---------------------------------------------------------------------
def _agent_reward_check(got, want, sinr_ref, thr):
    """Per-agent rewards within RTOL - every agent, also those whose float64 SINR sits right at the decision threshold: links
    within the threshold band take the kernels' fp64 pass, whose stored value falls on the float64 value's side of it
    (d2d_sinr_store, d2d_common.cuh).  Only a float64 SINR within float64 noise of the threshold (1e-11 dB: the kernel's and
    the reference's evaluation orders differ) could still be decided differently."""
    assert not ((np.abs(sinr_ref - thr) < 1e-11) & (sinr_ref != 0.0)).any()      # (absent agents carry sinr = 0)
    err = rel_err_np(got, want)
    assert (err <= RTOL).all(), float(err.max())


def rel_err_np(got, ref):
    from tests._util import rel_err
    return rel_err(got, ref)


@pytest.mark.parametrize('name', ['default', 'small', 'block_min', 'one_rb_crowded'])
@pytest.mark.parametrize('kind', ['shannon', 'cue_sinr_shannon'])
def test_per_agent_reward_functions(name, kind):
    """ShannonRewardFunction / CueSinrShannonRewardFunction (envs/reward_fn.py:47-78) against the oracle's restatement, with
    absent agents; `reward` is the mean over the acting agents and the reward statistics follow it."""
    import gym_d2d_b200 as G
    kw = CONFIGS[name]
    cfg = O.OracleConfig(**kw)
    cls, param = (G.ShannonRewardFunction, -70.0) if kind == 'shannon' else (G.CueSinrShannonRewardFunction, 0.0)
    rng = np.random.default_rng(33)
    E = 200
    pos, act = O.random_positions(cfg, E, rng), O.random_actions(cfg, E, rng)
    active = (rng.random(act.shape) < 0.8).astype(np.uint8)
    active[:, 0] = 1
    ref = O.step_batch(cfg, pos, act, active=active, nthreads=4)
    want = O.agent_rewards(cfg, ref, kind, param, active=active)
    env = make_vec(E, dict(kw, reward_fn=cls))
    env.reset_stats()
    env.set_positions(pos)
    a = torch.as_tensor(np.where(active > 0, act, -1), dtype=torch.int32, device='cuda').contiguous()
    obs, reward, done, info = env.step(a)
    torch.cuda.synchronize()
    got = info['agent_reward'].cpu().numpy()
    assert_rel(obs[..., 4].cpu().numpy(), ref['sinr_db'], RTOL, 'sinr_db')
    _agent_reward_check(got, want, ref['sinr_db'], param)
    assert (got[active == 0] == 0).all()
    mean = (got * active).sum(axis=1) / active.sum(axis=1)
    np.testing.assert_allclose(reward.cpu().numpy(), mean, rtol=2e-6, atol=1e-7)
    assert env.stats()['sum_reward'] == pytest.approx(float(mean.sum()), rel=1e-5)
    if kind == 'cue_sinr_shannon' and name != 'one_rb_crowded':
        assert (want == -1).any() and (want > 0).any()
    env.close()


def test_reward_plugins_match_reference_fixture_gpu(golden_dir):
    """The CUDA path against per-agent rewards of the unmodified reference (tests/golden/reward_plugins.npz), incl. the dict
    API: `env.step(dict)` returns one reward per agent key like envs/d2d_env.py:67."""
    import gym_d2d_b200 as G
    g = np.load(golden_dir / 'reward_plugins.npz')
    kw = dict(num_rbs=4, num_cues=6, num_due_pairs=9)
    steps, E, N = g['actions'].shape
    for kind, cls, thr in [('shannon', G.ShannonRewardFunction, -70.0), ('cue_sinr_shannon', G.CueSinrShannonRewardFunction, 0.0)]:
        env = make_vec(E, dict(kw, reward_fn=cls))
        env.set_positions(g['positions'])
        for s in range(steps):
            _, _, _, info = env.step(torch.as_tensor(g['actions'][s], dtype=torch.int32, device='cuda').contiguous())
            _agent_reward_check(info['agent_reward'].cpu().numpy(), g[f'{kind}_reward'][s], g['sinr_db'][s], thr)
        env.close()
    denv = G.make('D2DEnv-v0', env_config=dict(kw, reward_fn=G.CueSinrShannonRewardFunction))
    denv.reset()
    keys = [str(k) for k in g['keys']]
    ids = denv.device_ids
    denv.set_device_positions({ids[i]: tuple(g['positions'][0, i]) for i in range(len(ids))})
    present = [int(i) for i in g['subset_present']]
    _, rewards, _, _ = denv.step({keys[i]: int(g['actions'][0, 0, i]) for i in present})
    assert list(rewards) == [keys[i] for i in present]
    assert_rel(np.array([rewards[keys[i]] for i in present]), g['subset_cue_sinr_shannon_reward'], RTOL, 'dict-API per-agent rewards')
    denv.close()


@pytest.mark.parametrize('name', ['default', 'small', 'block_min'])
@pytest.mark.parametrize('area', [1, 2])
def test_cost_hata_path_loss(name, area):
    """CostHataPathLoss (path_loss.py:90-123), SUBURBAN and URBAN, against the oracle's restatement of the reference formula."""
    import gym_d2d_b200 as G
    kw = CONFIGS[name]
    cfg = O.OracleConfig(**kw, path_loss_model='cost_hata', area_type=area)
    rng = np.random.default_rng(50 + area)
    E = 128
    pos, act = O.random_positions(cfg, E, rng), O.random_actions(cfg, E, rng)
    model = functools.partial(G.CostHataPathLoss, area_type=G.AreaType(area))
    env = make_vec(E, dict(kw, path_loss_model=model))
    check_against_oracle(run_step(env, pos, act), O.step_batch(cfg, pos, act, nthreads=4))
    env.close()


def test_cost_hata_matches_reference_fixture(golden_dir):
    """The CUDA path against step results of the unmodified reference with path_loss_model=CostHataPathLoss (cost_hata.npz)."""
    import gym_d2d_b200 as G
    g = np.load(golden_dir / 'cost_hata.npz')
    kw = dict(num_rbs=3, num_cues=5, num_due_pairs=7)
    steps, E, N = g['actions'].shape
    for name, model in [('suburban', G.CostHataPathLoss), ('urban', functools.partial(G.CostHataPathLoss, area_type=G.AreaType.URBAN))]:
        env = make_vec(E, dict(kw, path_loss_model=model))
        for s in range(steps):
            out = run_step(env, g['positions'], g['actions'][s])
            assert_rel(out['obs'][..., 4], g[f'{name}_sinr_db'][s], RTOL, f'{name} sinr')
            assert_rel(out['obs'][..., 5], g[f'{name}_snr_db'][s], RTOL, f'{name} snr')
            assert_rel(out['capacity_mbps'], g[f'{name}_capacity_mbps'][s], RTOL, f'{name} capacity')
            assert_rel(out['reward'], g[f'{name}_reward'][s], RTOL, f'{name} reward')
        env.close()


def test_step_many_with_per_agent_rewards():
    """d2d_step_many + a per-agent reward function: the post-pass kernel covers all T x E env-steps of the fused launch."""
    import gym_d2d_b200 as G
    cfg = O.OracleConfig()
    E, T = 64, 5
    rng = np.random.default_rng(8)
    pos = O.random_positions(cfg, E, rng)
    acts = np.stack([O.random_actions(cfg, E, rng) for _ in range(T)])
    env = make_vec(E, dict(reward_fn=G.ShannonRewardFunction))
    env.set_positions(pos)
    out = env.step_many(torch.as_tensor(acts, dtype=torch.int32, device='cuda').contiguous())
    torch.cuda.synchronize()
    for t in range(T):
        ref = O.step_batch(cfg, pos, acts[t], nthreads=4)
        want = O.agent_rewards(cfg, ref, 'shannon', -70.0)
        assert_rel(out['agent_reward'][t].cpu().numpy(), want, RTOL, f'slice {t}')
        np.testing.assert_allclose(out['reward'][t].cpu().numpy(), want.mean(axis=1), rtol=1e-5)
    env.close()


def test_downlink_actions_tensor_api_and_dict_api(golden_dir):
    """'mbs:cueXX' DOWNLINK actions (envs/d2d_env.py:87-89, Appendix B.8): the general-topology kernel against the oracle on
    random scenarios, and against step results of the unmodified reference (tests/golden/downlink.npz) through the dict API
    (the first 'mbs:' key switches the env to the 2C + D link table; uplink / sidelink indices do not move)."""
    import gym_d2d_b200 as G
    kw = dict(num_rbs=4, num_cues=5, num_due_pairs=6)
    cfg = O.OracleConfig(**kw, downlinks=True)
    C, D, N = 5, 6, 16
    rng = np.random.default_rng(71)
    E = 96
    pos = O.random_positions(cfg, E, rng)
    act = O.random_actions(cfg, E, rng)
    act[:, :C] = rng.integers(0, 2, (E, C)) * 24 + rng.integers(0, 24, (E, C))            # uplinks on RB 0-1
    act[:, C + D:] = rng.integers(2, 4, (E, C)) * 47 + rng.integers(0, 47, (E, C))        # downlinks on RB 2-3
    active = (rng.random(act.shape) < 0.8).astype(np.uint8)
    ref = O.step_batch(cfg, pos, act, active=active, nthreads=4)
    env = make_vec(E, kw, downlink=True)
    assert env.num_links == N and env.link_keys[-1] == 'mbs:cue04'
    out = run_step(env, pos, np.where(active > 0, act, -1).astype(np.int32))
    check_against_oracle(out, ref)
    assert out['tx_pwr_dbm'][:, C + D:].max() > 23
    env.close()

    g = np.load(golden_dir / 'downlink.npz')
    keys = [str(k) for k in g['keys']]
    denv = G.make('D2DEnv-v0', env_config=dict(kw))
    denv.reset()
    ids = denv.device_ids
    for s in range(g['actions'].shape[0]):
        for e in range(g['actions'].shape[1]):
            denv.set_device_positions({ids[i]: tuple(g['positions'][e, i]) for i in range(len(ids))})
            present = [i for i in range(N) if g['active'][s, e, i]]
            _, rewards, _, info = denv.step({keys[i]: int(g['actions'][s, e, i]) for i in present})
            assert list(rewards) == [keys[i] for i in present]
            for k in ['sinr_db', 'snr_db', 'rate_bps', 'capacity_mbps']:
                assert_rel(np.array([info[keys[i]][k] for i in present]), g[k][s, e][present], RTOL, f'downlink {k}')
            assert [info[keys[i]]['tx_pwr_dbm'] for i in present] == [int(v) for v in g['tx_pwr_dbm'][s, e][present]]
            assert_rel(np.array([rewards[keys[present[0]]]]), g['reward'][s, e:e + 1], RTOL, 'downlink reward')
    denv.close()


@pytest.mark.parametrize('name', ['default', 'small', 'block_min'])
def test_shadowing_path_loss_matches_oracle_draw_for_draw(name):
    """ShadowingPathLoss (path_loss.py:69-81): the kernel's counter-based draws (global env, victim, source, evaluation kind, step
    call) are restated by the oracle, so results match value for value - on consecutive step calls (fresh draws each) and
    for a shard that starts at a non-zero global env index.  (The distribution is pinned to the reference on the CPU side.)"""
    import gym_d2d_b200 as G
    kw = dict(CONFIGS[name], cell_radius_m=500.0, d2d_radius_m=180.0)       # D2D links on both sides of d0 = 100 m
    rng = np.random.default_rng(91)
    E, first = 96, 1000
    okw = {k: v for k, v in kw.items()}
    cfg = O.OracleConfig(**okw, path_loss_model='shadowing', shadow_chi_dB=3.1, shadow_d0_m=90.0, rng_seed=77, first_global_env=first)
    pos = O.random_positions(cfg, E, rng)
    model = functools.partial(G.ShadowingPathLoss, chi_dB=3.1, d0_m=90.0)
    env = make_vec(E, dict(kw, path_loss_model=model), seed=77, global_env_offset=first)
    prev = None
    for call in range(2):
        act = O.random_actions(cfg, E, rng)
        cfg.rng_step = call
        ref = O.step_batch(cfg, pos, act, nthreads=4)
        out = run_step(env, pos, act)
        check_against_oracle(out, ref)
        if prev is not None:
            assert not np.allclose(prev, out['obs'][..., 5])            # the SNR of far links changes from call to call
        prev = out['obs'][..., 5].copy()
    far = np.linalg.norm(pos[:, 1 + cfg.num_cues::2] - pos[:, 2 + cfg.num_cues::2], axis=-1) > 90.0
    assert far.any() and (~far).any()
    env.close()


@pytest.mark.parametrize('info,kw', [(True, dict(num_rbs=4, num_cues=40, num_due_pairs=60)),         # N = 100: 256 threads x 1 link
                                     (False, dict(num_rbs=4, num_cues=40, num_due_pairs=60)),
                                     (False, dict(num_rbs=6, num_cues=60, num_due_pairs=240)),       # N = 300: 320 threads x 1 link
                                     (True, dict(num_rbs=12, num_cues=100, num_due_pairs=500))])     # N = 600: 320 threads x 2 links
def test_dense_kernel_pipeline_crowded_rbs_and_absent_agents(monkeypatch, info, kw):
    """The binned one-barrier kernel (d2d_step_dense.cuh) where its bookkeeping is hardest: three blocks stepping 300 envs each
    (so consecutive envs overlap inside a block, the counter / bin buffers rotate and a group of 256 per-env scalars is flushed
    mid-range), RBs that hold more links than a bin has slots (everybody on one RB -> the overflow list and its extra
    barrier), absent agents, two consecutive steps (step counters, done).  info=False runs the FULL instantiation."""
    import gym_d2d_b200 as G
    monkeypatch.setenv('D2D_B200_GRID', '3')
    cfg = O.OracleConfig(**kw)
    E = 900 if cfg.num_links <= 300 else 780
    rng = np.random.default_rng(4242)
    pos = O.random_positions(cfg, E, rng, fp32_exact=True)
    env = G.VecD2DEnv(E, dict(kw), device='cuda', info=info)
    assert env.step_geometry()['grid'] == 3
    env.set_positions(pos)
    for s in range(2):
        act = O.random_actions(cfg, E, rng)
        npw = np.where(np.arange(cfg.num_links) < cfg.num_cues, cfg.cue_max_tx_power_dBm + 1,
                       cfg.due_max_tx_power_dBm - cfg.due_min_tx_power_dBm + 1)
        crowded = np.arange(E) % 5 == 0
        act[crowded] = act[crowded] % npw                           # rb = 0 for every link: all N links on one RB
        two = np.arange(E) % 11 == 3
        act[two] = act[two] % (2 * npw)                             # two RBs of ~N/2 links: both overflow
        absent = (np.arange(E) % 7 == 0)[:, None] & (rng.random((E, cfg.num_links)) < 0.5)
        ref = O.step_batch(cfg, pos, act, active=(~absent).astype(np.uint8), nthreads=8)
        obs, reward, done, inf = env.step(torch.as_tensor(np.where(absent, -1, act), dtype=torch.int32, device='cuda').contiguous())
        torch.cuda.synchronize()
        on = ~absent
        assert_rel(obs[..., 4].cpu().numpy()[on], ref['sinr_db'][on], RTOL, 'sinr_db')
        assert_rel(obs[..., 5].cpu().numpy()[on], ref['snr_db'][on], RTOL, 'snr_db')
        assert_rel(inf['capacity_mbps'].cpu().numpy()[on], ref['capacity_mbps'][on], RTOL, 'capacity')
        assert (inf['capacity_mbps'].cpu().numpy()[~on] == 0).all() and (obs[..., 4].cpu().numpy()[~on] == 0).all()
        assert_rel(reward.cpu().numpy(), ref['reward'], RTOL, 'reward')
        assert (env.step_count.cpu().numpy() == s + 1).all() and (done.cpu().numpy() == 0).all()
        if info:
            np.testing.assert_array_equal(inf['rb'].cpu().numpy()[on], ref['rb'][on])
            np.testing.assert_array_equal(inf['tx_pwr_dbm'].cpu().numpy()[on], ref['tx_pwr_dbm'][on])
    st = env.stats()
    assert st['env_steps'] == 2 * E
    env.close()


def test_dense_kernel_fp64_pass_on_a_crowded_rb():
    """The dense kernel's warp-cooperative fp64 pass when the victim's RB holds more records than one per lane (and more than a bin:
    the overflow list): one RB for 70 links, enough envs that some links land within the band around 0 dB; the pure 1e-4
    relative check only passes if they were recomputed."""
    kw = dict(num_rbs=1, num_cues=30, num_due_pairs=40)
    cfg = O.OracleConfig(**kw)
    E = 512
    rng = np.random.default_rng(77)
    env = make_vec(E, kw)
    env.reset_stats()
    near = 0
    for s in range(2):
        pos = O.random_positions(cfg, E, rng, fp32_exact=True)
        act = O.random_actions(cfg, E, rng)
        ref = O.step_batch(cfg, pos, act, nthreads=8)
        out = run_step(env, pos, act)
        check_against_oracle(out, ref)
        near += int((np.minimum(np.abs(ref['sinr_db']), np.abs(ref['snr_db'])) < 0.05).sum())
    assert near > 0 and env.stats()['rescues'] >= near
    env.close()
