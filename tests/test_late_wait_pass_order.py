"""Late-wait step chains in which the fp64 pass runs in the env that closes a warp's first group.

In a late-wait launch (D2D_PF_LATE_WAIT) a warp stores its envs' per-link outputs ahead of griddepcontrol.wait, and the fp64
pass that overwrites a flagged link's outputs runs there too - also for the env whose group end carries the wait.  These chains
put a DUE link at the SNR band edge (|SNR_dB| < 0.0625 dB, the band below which the kernel recomputes a link in fp64) into most
envs, so that the last env of most warps runs a pass, and crowd a few envs' CUEs onto one RB (the all-pairs overflow path).
Everything a step writes, the step counters and the rescue / penalty / env-step statistics must be bit-identical to the same
chain with the late wait switched off and to a library without programmatic dependent launch.
"""
import numpy as np
import pytest

from oracle import d2d_oracle as O

E, RING = 4096, 4
CFG = O.OracleConfig()
N_PWR_CUE, N_PWR_DUE = CFG.cue_max_tx_power_dBm + 1, CFG.due_max_tx_power_dBm - CFG.due_min_tx_power_dBm + 1


def band_edge_chain(seed=21):
    """(positions, [RING] actions, flagged env mask, DUE link per env): default EnvConfig, E envs.  A flagged env's DUE pair l
    keeps its power level in every action set (its RB changes) and its receiver sits at the distance that puts its SNR within
    0.05 dB of 0 dB; ~3 % of the envs of each action set have every CUE on RB 0 (more links than a bin holds)."""
    rng = np.random.default_rng(seed)
    pos = O.random_positions(CFG, E, rng, fp32_exact=True)
    acts = [O.random_actions(CFG, E, rng) for _ in range(RING)]
    flagged = rng.random(E) < 0.6
    link = rng.integers(0, CFG.num_due_pairs, E)
    p = rng.integers(0, N_PWR_DUE, E)
    target = rng.uniform(0.005, 0.05, E) * rng.choice([-1.0, 1.0], E)
    # DUE pair link budget (device.py:12-41 defaults, log-distance path loss, ple = 2): SNR_dB = p + snr0 - 20 log10(d)
    K = 20 * np.log10(2.1e9) + 20 * np.log10(4 * np.pi / 299792458.0)
    snr0 = -6.0 - 3.0 - K + 104.5
    d = 10 ** ((p + CFG.due_min_tx_power_dBm + snr0 - target) / 20)
    th = rng.uniform(0, 2 * np.pi, E)
    e = np.nonzero(flagged)[0]
    tx, rx = 1 + CFG.num_cues + 2 * link[e], 2 + CFG.num_cues + 2 * link[e]
    pos[e, rx] = pos[e, tx] + np.stack([d[e] * np.cos(th[e]), d[e] * np.sin(th[e])], -1)
    pos = pos.astype(np.float32).astype(np.float64)
    for a in acts:
        a[e, CFG.num_cues + link[e]] = rng.integers(0, CFG.num_rbs, len(e)) * N_PWR_DUE + p[e]
        crowd = rng.random(E) < 0.03
        a[crowd, :CFG.num_cues] %= N_PWR_CUE                  # RB 0, power level kept
    return pos, acts, flagged, link


def test_band_edge_chain_hits_the_band():
    """The construction does what the GPU test relies on: every flagged env's DUE link is inside the fp64 band (float64 oracle)."""
    pos, acts, flagged, link = band_edge_chain()
    ref = O.step_batch(CFG, pos, acts[0], nthreads=4)
    e = np.nonzero(flagged)[0]
    snr = ref['snr_db'][e, CFG.num_cues + link[e]]
    assert flagged.mean() > 0.5 and (np.abs(snr) < 0.0625).all() and (snr > 0).sum() > 100 and (snr < 0).sum() > 100


@pytest.mark.gpu
@pytest.mark.parametrize('info', [False, True])
@pytest.mark.parametrize('grid', [None, '148'])
def test_late_wait_pass_before_the_wait_is_bit_identical(monkeypatch, grid, info):
    """Graph replays and eager chains over a ring of output sets, on the default late-wait grid and on one block per SM: every
    output, the counters and the rescue / penalty / env-step statistics equal the chains with D2D_B200_LATE_WAIT=0 and with
    D2D_B200_PDL=0, bit for bit."""
    torch = pytest.importorskip('torch')
    import gym_d2d_b200 as G
    if grid:
        monkeypatch.setenv('D2D_B200_LATE_GRID', grid)

    def make(**env):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        v = G.VecD2DEnv(E, {}, device='cuda', info=info)
        for k in env:
            monkeypatch.delenv(k)
        return v

    plain, late, early = make(D2D_B200_PDL='0'), make(), make(D2D_B200_LATE_WAIT='0')
    envs = (plain, late, early)
    pos, acts_np, _, _ = band_edge_chain()
    acts = [torch.as_tensor(a, dtype=torch.int32, device='cuda') for a in acts_np]
    outs = {env: [env.alloc_outputs() for _ in range(RING)] for env in envs}
    names = ('obs', 'capacity_mbps', 'reward', 'done') + (('rate_bps', 'rb', 'tx_pwr_dbm') if info else ())
    for env in envs:
        env.set_positions(pos)
        env.reset_stats()
    order = [0, 1, 2, 3, 1, 0, 3, 2]
    graphs = {env: env.capture_steps([acts[i] for i in order], [outs[env][i] for i in order], inputs_stable=True) for env in (late, early)}
    diff = torch.zeros((), dtype=torch.int64, device='cuda')

    def check():
        d = (plain.step_count != late.step_count).sum() + (plain.step_count != early.step_count).sum()
        for i in range(RING):
            for name in names:
                ref = getattr(outs[plain][i], name)
                d = d + (ref != getattr(outs[late][i], name)).sum() + (ref != getattr(outs[early][i], name)).sum()
        return d

    for it in range(300):
        for i in order:
            plain.step(acts[i], out=outs[plain][i])
        graphs[late].replay()
        graphs[early].replay()
        if it % 10 == 0:
            diff += check()
        if it % 25 == 24:                                       # counters back to 0 (the episode length is 10 steps)
            for env in envs:
                env.set_positions(pos)
    for it in range(20):                                        # eager chains
        for env in envs:
            for k in range(7):
                env.step(acts[(it + k) % RING], out=outs[env][(it + k) % RING], inputs_stable=True)
        diff += check()
    torch.cuda.synchronize()
    assert int(diff.item()) == 0
    sp, sl, se = plain.stats(), late.stats(), early.stats()
    for key in ('env_steps', 'rescues', 'penalties'):
        assert sp[key] == sl[key] == se[key], key
    assert sp['rescues'] > 0.5 * sp['env_steps']                # the chains did run the fp64 pass in most envs
    assert late.stats()['ticket_timeouts'] == 0
    for env in envs:
        env.close()
