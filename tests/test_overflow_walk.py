"""RBs that hold more links than a warp-kernel bin has records (D2D_BIN_CAP = 8), held to the float64 oracle.

The warp step kernel keeps the first 8 links of an RB as records in the RB's bin; every victim walks those records, and the links
ranked 8 and above add their terms in a shuffle pass over just those links.  These envs put exactly 8, 9, 10, 12, 16, 25 or 50
live links on one RB (CUE-only, DUE-only and mixed crowds), or two overflowing RBs in one env, so that victims ranked below and
above the bin's capacity are both present.  Some envs add absent agents whose actions point at the crowded RB, and some put a
DUE link at the SNR band edge (|SNR_dB| < 0.0625 dB) on the crowded RB, where the fp64 pass recomputes it.
"""
import functools

import numpy as np
import pytest

from oracle import d2d_oracle as O
from tests._util import RTOL, assert_rel, check_against_oracle

torch = pytest.importorskip('torch')

CAP = 8
LOADS = (8, 9, 10, 12, 16, 25, 50)
# (load, kind) of one crowded RB, or two crowded RBs in one env
SCENARIOS = [((L, k),) for L in LOADS for k in ('cue', 'due', 'mixed') if L <= (50 if k == 'mixed' else 25)]
SCENARIOS += [((9, 'mixed'), (12, 'mixed')), ((16, 'cue'), (10, 'due')), ((9, 'due'), (9, 'cue'))]
N_ABSENT = 3                 # absent agents on the crowded RB of an env with absent agents


def _npw(cfg):
    return np.where(np.arange(cfg.num_links) < cfg.num_cues, cfg.cue_max_tx_power_dBm + 1,
                    cfg.due_max_tx_power_dBm - cfg.due_min_tx_power_dBm + 1)


def crowd_scenario(cfg, E, rng, exact=False):
    """(positions, actions, active, loads [E][R] of live links per RB, band [(env, link)]).  Env e takes SCENARIOS[e % S]; every
    other round of scenarios adds absent agents (N_ABSENT on the first crowded RB, ~10 % elsewhere), and every third env whose first
    crowd holds a DUE link puts that link's receiver where its SNR is within 0.05 dB of 0 dB.  Every RB that is not crowded holds
    at most 8 live links."""
    C, D, R, N = cfg.num_cues, cfg.num_due_pairs, cfg.num_rbs, cfg.num_links
    npw = _npw(cfg)
    pos = O.random_positions(cfg, E, rng, fp32_exact=not exact)
    act = np.empty((E, N), np.int32)
    active = np.ones((E, N), np.uint8)
    band = []
    K = 10 * cfg.ple * np.log10(cfg.carrier_freq_GHz * 1e9) + 10 * cfg.ple * np.log10(4 * np.pi / 299792458.0)
    snr0_due = -6.0 - 3.0 - K + 104.5              # UE Tx (eirp - p) + UE Rx offset - K - UE noise (device.py:12-41 defaults)
    for e in range(E):
        scen = SCENARIOS[e % len(SCENARIOS)]
        absent = (e // len(SCENARIOS)) % 2 == 1
        rbs = rng.choice(R, len(scen), replace=False)
        rb = np.full(N, -1)
        free_c, free_d = list(rng.permutation(C)), list(rng.permutation(np.arange(C, N)))
        for r, (L, kind) in zip(rbs, scen):
            nc = L if kind == 'cue' else 0 if kind == 'due' else min(L // 2, len(free_c))
            members = [free_c.pop() for _ in range(nc)] + [free_d.pop() for _ in range(L - nc)]
            rb[members] = r
        if absent:
            gone = (free_c + free_d)[:N_ABSENT]
            rb[gone] = rbs[0]
            active[e, gone] = 0
        rest = np.flatnonzero(rb < 0)
        others = np.setdiff1d(np.arange(R), rbs)
        while True:
            rb[rest] = rng.choice(others, rest.size)
            live = active[e] > 0
            if np.bincount(rb[rest][live[rest]], minlength=R)[others].max() <= CAP:
                break
        if absent:
            active[e, rest[rng.random(rest.size) < 0.1]] = 0
        p = rng.integers(0, npw)
        act[e] = rb * npw + p
        due = [j for j in np.flatnonzero(rb == rbs[0]) if j >= C and active[e, j]]
        if due and e % 3 == 0:
            j = due[0]
            target = rng.uniform(0.005, 0.05) * rng.choice([-1.0, 1.0])
            d = 10 ** ((p[j] + cfg.due_min_tx_power_dBm + snr0_due - target) / (10 * cfg.ple))
            th = rng.uniform(0, 2 * np.pi)
            tx = 1 + C + 2 * (j - C)
            pos[e, tx + 1] = pos[e, tx] + d * np.array([np.cos(th), np.sin(th)])
            band.append((e, j))
    if not exact:
        pos = pos.astype(np.float32).astype(np.float64)
    loads = np.stack([np.bincount(np.where(active[e] > 0, act[e] // npw, R), minlength=R + 1)[:R] for e in range(E)])
    return pos, act, active, loads, band


def _cfg(ple=2.0):
    return O.OracleConfig() if ple == 2.0 else O.OracleConfig(ple=ple)


# ---- CPU tier -------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('exact', [False, True])
def test_scenario_has_the_loads_it_claims(exact):
    """Every scenario's crowded RBs hold exactly the claimed live links (absent agents excluded), every other RB at most 8, and the
    float64 oracle decodes the same peer sets: per env and RB, the live links it puts on the RB are the ones the constructor put there."""
    cfg = _cfg()
    E = 2 * len(SCENARIOS) * 3
    pos, act, active, loads, band = crowd_scenario(cfg, E, np.random.default_rng(5), exact)
    for e in range(E):
        scen = SCENARIOS[e % len(SCENARIOS)]
        assert sorted(loads[e][loads[e] > CAP]) == sorted(L for L, _ in scen if L > CAP), (e, scen, loads[e])
        assert sorted(loads[e], reverse=True)[:len(scen)] == sorted((L for L, _ in scen), reverse=True)
    assert (loads.sum(1) == active.sum(1)).all()
    ref = O.step_batch(cfg, pos, act, active=active, nthreads=4)
    assert ref['status'] == 0
    npw = _npw(cfg)
    live = active > 0
    np.testing.assert_array_equal(ref['rb'][live], (act // npw)[live])
    for e in range(E):
        for r in np.flatnonzero(loads[e] > CAP):
            assert ((ref['rb'][e] == r) & live[e]).sum() == loads[e, r]
    # absent agents pointed at a crowded RB, victims of every rank, band-edge DUE links on crowded RBs
    assert (~live & (act // npw == np.argmax(loads, 1)[:, None])).sum() >= N_ABSENT * E // 4
    assert len(band) >= E // 8
    snr = np.array([ref['snr_db'][e, j] for e, j in band])
    assert (np.abs(snr) < 0.0625).all() and (snr > 0).any() and (snr < 0).any()
    assert all(loads[e, act[e, j] // npw[j]] > CAP for e, j in band if loads[e].max() > CAP)


# ---- GPU tier -------------------------------------------------------------------------------------------------------------------
E = 4096


def _make(monkeypatch, knobs, ple, info, exact):
    import gym_d2d_b200 as G
    if not torch.cuda.is_available():
        pytest.fail('the gpu tier needs a CUDA device (no CPU fallback exists)')
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    kw = {} if ple == 2.0 else dict(path_loss_model=functools.partial(G.LogDistancePathLoss, ple=ple))
    env = G.VecD2DEnv(E, kw, device='cuda', info=info, exact_positions=exact)
    for k in knobs:
        monkeypatch.delenv(k)
    return env


def _np(o, info, t=None):
    g = (lambda x: x.cpu().numpy()) if t is None else (lambda x: x[t].cpu().numpy())
    out = dict(obs=g(o['obs']), reward=g(o['reward']), capacity_mbps=g(o['capacity_mbps']))
    if info:
        out.update(rate_bps=g(o['rate_bps']), rb=g(o['rb']).astype(np.int32), tx_pwr_dbm=g(o['tx_pwr_dbm']).astype(np.int32))
    return out


def _compare(out, ref, info):
    assert ref['status'] == 0
    if info:
        check_against_oracle(out, ref)
    else:       # the core outputs only: the FULL instantiations write nothing else
        assert_rel(out['obs'][..., 4], ref['sinr_db'], RTOL, 'sinr_db')
        assert_rel(out['obs'][..., 5], ref['snr_db'], RTOL, 'snr_db')
        assert_rel(out['obs'][..., :4], ref['obs'][..., :4], RTOL, 'obs positions')
        assert_rel(out['capacity_mbps'], ref['capacity_mbps'], RTOL, 'capacity_mbps')
        assert_rel(out['reward'], ref['reward'], RTOL, 'reward')


VARIANTS = {
    'default': ({}, 2.0, False, None),
    'generic_shape': ({'D2D_B200_SPEC': '0'}, 2.0, False, None),
    'ple_3_5': ({}, 3.5, False, None),
    'exact_positions': ({}, 2.0, True, None),
    'wpb_2': ({'D2D_B200_WPB': '2'}, 2.0, False, 2),
    'wpb_4': ({'D2D_B200_WPB': '4'}, 2.0, False, 4),
    'wpb_8': ({'D2D_B200_WPB': '8'}, 2.0, False, 8),
}


@pytest.mark.gpu
@pytest.mark.parametrize('info', [True, False])
@pytest.mark.parametrize('variant', list(VARIANTS))
def test_crowded_rbs_match_oracle(monkeypatch, variant, info):
    """One step of the crowd scenarios on the warp kernel (default shape, the generic shape, ple 3.5, fp64 positions, 2 / 4 / 8
    warps per block; with and without the info outputs) against the float64 oracle."""
    knobs, ple, exact, wpb = VARIANTS[variant]
    env = _make(monkeypatch, knobs, ple, info, exact)
    if wpb is not None:
        assert env.step_geometry()['block'] == 32 * wpb
    cfg = _cfg(ple)
    pos, act, active, _, _ = crowd_scenario(cfg, E, np.random.default_rng(11), exact)
    env.set_positions(pos)
    a = torch.as_tensor(np.where(active > 0, act, -1), dtype=torch.int32, device='cuda').contiguous()
    obs, reward, done, inf = env.step(a)
    torch.cuda.synchronize()
    _compare(_np(dict(obs=obs, reward=reward, **inf), info), O.step_batch(cfg, pos, act, active=active, nthreads=8), info)
    env.close()


@pytest.mark.gpu
def test_crowded_rbs_step_many_matches_oracle(monkeypatch):
    """d2d_step_many over three steps of crowd scenarios with given actions: every slice against the oracle."""
    env = _make(monkeypatch, {}, 2.0, True, False)
    cfg = _cfg()
    rng = np.random.default_rng(12)
    pos, _, _, _, _ = crowd_scenario(cfg, E, rng)
    steps = [crowd_scenario(cfg, E, rng)[1:3] for _ in range(3)]
    env.set_positions(pos)
    acts = torch.as_tensor(np.stack([np.where(m > 0, a, -1) for a, m in steps]), dtype=torch.int32, device='cuda').contiguous()
    o = env.step_many(acts)
    torch.cuda.synchronize()
    for t, (a, m) in enumerate(steps):
        _compare(_np(o, True, t), O.step_batch(cfg, pos, a, active=m, nthreads=8), True)
    env.close()


@pytest.mark.gpu
def test_crowded_rbs_late_wait_chain_is_bit_identical(monkeypatch):
    """A CUDA graph of late-wait steps over a ring of output sets equals eager steps without programmatic dependent launch, bit for
    bit, and each output set holds the oracle's values for its actions."""
    RING = 4
    plain, late = _make(monkeypatch, {'D2D_B200_PDL': '0'}, 2.0, True, False), _make(monkeypatch, {}, 2.0, True, False)
    cfg = _cfg()
    rng = np.random.default_rng(13)
    pos, _, _, _, _ = crowd_scenario(cfg, E, rng)
    steps = [crowd_scenario(cfg, E, rng)[1:3] for _ in range(RING)]
    acts = [torch.as_tensor(np.where(m > 0, a, -1), dtype=torch.int32, device='cuda').contiguous() for a, m in steps]
    outs = {env: [env.alloc_outputs() for _ in range(RING)] for env in (plain, late)}
    for env in (plain, late):
        env.set_positions(pos)
    order = [0, 1, 2, 3, 2, 0, 3, 1]
    graph = late.capture_steps([acts[i] for i in order], [outs[late][i] for i in order], inputs_stable=True)
    names = ('obs', 'capacity_mbps', 'reward', 'done', 'rate_bps', 'rb', 'tx_pwr_dbm')
    for _ in range(3):
        for i in order:
            plain.step(acts[i], out=outs[plain][i])
        graph.replay()
    torch.cuda.synchronize()
    assert (plain.step_count == late.step_count).all()
    for i in range(RING):
        for name in names:
            assert torch.equal(getattr(outs[plain][i], name), getattr(outs[late][i], name)), (i, name)
        o = outs[late][i]
        got = dict(obs=o.obs, reward=o.reward, capacity_mbps=o.capacity_mbps, rate_bps=o.rate_bps, rb=o.rb, tx_pwr_dbm=o.tx_pwr_dbm)
        _compare(_np(got, True), O.step_batch(cfg, pos, steps[i][0], active=steps[i][1], nthreads=8), True)
    for env in (plain, late):
        env.close()
