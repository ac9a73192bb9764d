"""Next-step auto-reset (D2D_STEP_AUTORESET, VecD2DEnv(autoreset=True)).

An auto-reset step treats each env by its step counter at entry: below episode_length it steps exactly like a plain d2d_step;
at or past it, it is reset as d2d_reset + d2d_sample_actions(step 0) + one uncounted d2d_step would do it, under the key
autoreset_key(base, n) with n the env's episode index after the increment, and returns reward = 0 and done = 0.  The GPU tests
desynchronise the envs by writing random counters 0-12 and compare every auto-reset step bit for bit with that composition run on a
second VecD2DEnv, then hold every row to the float64 oracle with the actions the env actually used.
"""
import functools
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

from oracle import d2d_oracle as O
from tests._util import check_against_oracle, check_reset_distribution

ROOT = Path(__file__).resolve().parent.parent
L = 10                                   # EPISODE_LENGTH (envs/d2d_env.py:16)


# ---- CPU tier -------------------------------------------------------------------------------------------------------------------
_KEY_PROBE = r'''
#include <cstdio>
#include "d2d_common.cuh"
int main() {
    unsigned long long base, n;
    while (std::scanf("%llu %llu", &base, &n) == 2) std::printf("%llu\n", (unsigned long long)d2d_autoreset_key(base, n));
    return 0;
}
'''


def test_autoreset_key_matches_the_library(tmp_path):
    """VecD2DEnv.autoreset_key restates d2d_autoreset_key (d2d_common.cuh): the host side of the real function, compiled with nvcc,
    must give the same 64-bit key over a sweep of bases (0, reset keys, values near 2^64) and episode indices (0 .. 2^32 - 1)."""
    from gym_d2d_b200.vec_env import autoreset_key
    nvcc = shutil.which('nvcc') or ('/usr/local/cuda/bin/nvcc' if Path('/usr/local/cuda/bin/nvcc').exists() else None)
    if nvcc is None:
        pytest.skip('nvcc not found')
    src = tmp_path / 'key_probe.cu'
    src.write_text(_KEY_PROBE)
    exe = tmp_path / 'key_probe'
    subprocess.run([nvcc, '-gencode', 'arch=compute_100a,code=sm_100a', '-std=c++17', '-I', str(ROOT / 'gym_d2d_b200' / 'csrc'),
                    '-o', str(exe), str(src)], check=True, capture_output=True)
    rng = np.random.default_rng(3)
    bases = [0, 1, 1234, 0x9E3779B97F4A7C15, 2 ** 64 - 1, 2 ** 63] + [int(x) for x in rng.integers(0, 2 ** 63, 20, dtype=np.int64) * 2 + 1]
    ns = [0, 1, 2, 3, 10, 255, 256, 65535, 2 ** 31, 2 ** 32 - 1] + [int(x) for x in rng.integers(0, 2 ** 32, 10)]
    cases = [(b, n) for b in bases for n in ns]
    res = subprocess.run([str(exe)], input=''.join(f'{b} {n}\n' for b, n in cases), check=True, capture_output=True, text=True)
    got = [int(x) for x in res.stdout.split()]
    assert got == [autoreset_key(b, n) for b, n in cases]
    for b in bases:                          # one base: a fresh key for every episode index
        assert len({autoreset_key(b, n) for n in ns}) == len(ns)
    # the bases VecD2DEnv.reset() binds (its key through splitmix64 once): the streams of successive full resets share no key, although
    # the reset keys seed + k * 0x9E3779B97F4A7C15 advance by the same constant as n
    for seed in (0, 7, 2 ** 64 - 5):
        keys = [autoreset_key(autoreset_key((seed + k * 0x9E3779B97F4A7C15) % 2 ** 64, 0), n) for k in range(8) for n in range(1, 200)]
        assert len(set(keys)) == len(keys)


# ---- GPU tier -------------------------------------------------------------------------------------------------------------------
def _torch():
    torch = pytest.importorskip('torch')
    if not torch.cuda.is_available():
        pytest.skip('needs a CUDA device')
    return torch


def _vec(E, cfg_kw=None, **kw):
    import gym_d2d_b200 as G
    return G.VecD2DEnv(E, dict(cfg_kw or {}), device='cuda', **kw)


def _snap(env, o=None):
    """Host copies of one step's outputs and of the env's state."""
    torch = _torch()
    torch.cuda.synchronize()
    o = o if o is not None else env._out
    d = dict(obs=o.obs, capacity_mbps=o.capacity_mbps, reward=o.reward, done=o.done, rate_bps=o.rate_bps, rb=o.rb,
             tx_pwr_dbm=o.tx_pwr_dbm, agent_reward=o.agent_reward, positions=env.positions, step_count=env.step_count,
             positions_f64=env.positions_f64)
    return {k: v.cpu().numpy().copy() for k, v in d.items() if v is not None}


def compose(B, base, ep_before, actions):
    """One auto-reset step composed from plain calls on B, whose positions and counters equal the auto-reset env's before its step:
    a counted d2d_step with `actions` for the counted envs; for the reset envs, per distinct episode index n,
    d2d_reset(autoreset_key(base, n), mask) and sample_actions_philox(key, 0), then one uncounted step.  Returns (outputs and state
    as the auto-reset step must leave them, the actions each env used, the episode indices after the step)."""
    torch = _torch()
    from gym_d2d_b200 import _lib
    from gym_d2d_b200.vec_env import autoreset_key
    rst = B.step_count.cpu().numpy() >= L
    B.step(actions)
    counted = _snap(B)
    ep_after = ep_before + rst.astype(np.int64)
    used = actions.clone()
    for n in np.unique(ep_after[rst]):
        m = torch.as_tensor((rst & (ep_after == n)).astype(np.uint8), device='cuda')
        key = autoreset_key(base, int(n))
        _lib.check(B._lib.d2d_reset(B._h, key, B.global_env_offset, m.data_ptr(), B._stream()))
        drawn = B.sample_actions_philox(key, 0)
        used[m.bool()] = drawn[m.bool()]
    B._bind(False)
    try:
        B._launch(used)
    finally:
        B._bind(True)
    reset = _snap(B)
    want = {}
    for k, v in counted.items():
        if k in ('positions', 'positions_f64', 'step_count'):
            want[k] = reset[k]
        else:
            want[k] = np.where(rst.reshape((-1,) + (1,) * (v.ndim - 1)), reset[k], v)
    want['reward'][rst] = 0
    want['done'][rst] = 0
    return want, used.cpu().numpy(), ep_after, rst


def _desync(torch, A, B, rng, exact, ocfg):
    """Same positions in both envs, random counters 0-12 and random episode indices 0-3."""
    E = A.num_envs
    if exact:
        pos = O.random_positions(ocfg, E, rng, fp32_exact=False)
        A.set_positions(pos)
        B.set_positions(pos)
    else:
        B.positions.copy_(A.positions)
    ns = torch.as_tensor(rng.integers(0, 13, E).astype(np.uint8), device='cuda')
    A.step_count.copy_(ns)
    B.step_count.copy_(ns)
    ep = rng.integers(0, 4, E)
    A.episode_index.copy_(torch.as_tensor(ep, dtype=torch.int32, device='cuda'))
    return ep


def _actions(torch, A, rng, absent):
    a = A.sample_actions(torch.Generator(device='cuda').manual_seed(int(rng.integers(1 << 30))))
    if absent:
        a[torch.as_tensor(rng.random(a.shape) < 0.2, device='cuda')] = -1
    return a


def _assert_same(got, want, what):
    for k in want:
        np.testing.assert_array_equal(got[k], want[k], err_msg=f'{what}: {k}')


CROWDED = dict(num_rbs=1, num_cues=20, num_due_pairs=30)
# (name, env_config, oracle config, environment, info, exact_positions, absent agents)
CASES = [
    ('spec', {}, {}, {}, True, False, False),
    ('spec_full', {}, {}, {}, False, False, False),
    ('generic', {}, {}, {'D2D_B200_SPEC': '0'}, True, False, False),
    ('ple35', 'ple35', {'ple': 3.5}, {}, True, False, False),
    ('exact', {}, {}, {}, True, True, False),
    ('exact_full', {}, {}, {}, False, True, False),
    ('absent', {}, {}, {}, True, False, True),
    ('crowded', CROWDED, CROWDED, {}, True, False, True),
    ('crowded_exact', CROWDED, CROWDED, {}, True, True, False),
    ('wpb2', {}, {}, {'D2D_B200_WPB': '2'}, True, False, True),
    ('wpb2_exact_full', {}, {}, {'D2D_B200_WPB': '2'}, False, True, False),
    ('wpb4', {}, {}, {'D2D_B200_WPB': '4'}, True, True, False),
    ('wpb8', {}, {}, {'D2D_B200_WPB': '8'}, True, False, True),
    ('wpb8_exact_full', {}, {}, {'D2D_B200_WPB': '8'}, False, True, False),
    ('grid', {}, {}, {'D2D_B200_GRID': '3'}, True, False, True),
    ('grid_exact', {}, {}, {'D2D_B200_GRID': '3', 'D2D_B200_SPEC': '0'}, True, True, False),
    ('chunk', {}, {}, {'D2D_B200_CHUNK': '700'}, True, False, False),
    ('chunk_full', {}, {}, {'D2D_B200_CHUNK': '700'}, False, False, True),
]


def _rescued_reset_links(got, used, rst, cell_radius=500.0, ple=2.0):
    """Links of reset envs that the fp64 pass certainly recomputed: with a position shadow a live link is recomputed when
    min(|SINR_dB|, |SNR_dB|) < 0.0625 + rescue_c / d_min (d2d_common.cuh: d2d_needs_rescue; rescue_c as d2d_abi.cu folds it), and
    d_min is at most the link's own length, read from its observation row."""
    ulp = 2.0 ** (np.floor(np.log2(max(cell_radius, 1.0))) - 23)
    c = 2.0 * 1e4 * 4.3429448190325 * ple * np.sqrt(2.0) * ulp
    obs = got['obs'].astype(np.float64)
    d = np.hypot(obs[..., 0] - obs[..., 2], obs[..., 1] - obs[..., 3])
    lo = np.minimum(np.abs(obs[..., 4]), np.abs(obs[..., 5]))
    return int((rst[:, None] & (used >= 0) & (lo < 0.0625 + c / d - 1e-3)).sum())


@pytest.mark.gpu
@pytest.mark.parametrize('case', CASES, ids=[c[0] for c in CASES])
def test_autoreset_step_equals_reset_composition(case, monkeypatch):
    """Three auto-reset steps from desynchronised counters, each equal bit for bit to the composition (outputs, counters, episode
    indices, fp32 positions, fp64 shadow), and every row of the last one within 1e-4 of the float64 oracle on the actions it used."""
    torch = _torch()
    import gym_d2d_b200 as G
    name, cfg_kw, okw, envv, info, exact, absent = case
    for k, v in envv.items():
        monkeypatch.setenv(k, v)
    if cfg_kw == 'ple35':
        cfg_kw = dict(path_loss_model=functools.partial(G.LogDistancePathLoss, ple=3.5))
    E = 3000
    A = _vec(E, cfg_kw, seed=7, info=info, exact_positions=exact, autoreset=True)
    B = _vec(E, cfg_kw, seed=7, info=info, exact_positions=exact)
    ocfg = O.OracleConfig(**okw)
    rng = np.random.default_rng(11)
    A.reset(seed=21)
    base = A._ar_base
    ep = _desync(torch, A, B, rng, exact, ocfg)
    rescued = 0
    for t in range(3):
        a = _actions(torch, A, rng, absent)
        want, used, ep, rst = compose(B, base, ep, a)
        A.step(a)
        got = _snap(A)
        _assert_same(got, want, f'{name} step {t}')
        np.testing.assert_array_equal(A.episode_index.cpu().numpy(), ep)
        assert rst.any() and (~rst).any()
        rescued += _rescued_reset_links(got, used, rst)
    if exact:       # the fp64 pass ran on reset envs, whose shadow rows it must not read (they hold the finished episode)
        assert rescued > 0, name
    if info:
        pos = got['positions_f64'] if exact else got['positions'].astype(np.float64)
        ref = O.step_batch(ocfg, pos, used, active=(used >= 0).astype(np.uint8), nthreads=8)
        assert ref['status'] == 0
        ref['reward'] = np.where(rst, 0.0, ref['reward'])
        check_against_oracle(got, ref)
    A.close(); B.close()


@pytest.mark.gpu
def test_autoreset_statistics_count_the_counted_steps_only():
    """stats() of an auto-reset step equal those of the counted envs' plain step: a separate env holding only the counted envs (the
    reset step enters no statistic - no reward, capacity, penalty, rescue or env-step)."""
    torch = _torch()
    E = 4096
    A = _vec(E, seed=3, autoreset=True)
    B = _vec(E, seed=3)
    rng = np.random.default_rng(5)
    A.reset(seed=9)
    _desync(torch, A, B, rng, False, O.OracleConfig())
    B.close()
    cnt = (A.step_count < L).cpu().numpy()
    S = _vec(int(cnt.sum()), seed=3)
    S.positions.copy_(A.positions[torch.as_tensor(cnt, device='cuda')])
    S.step_count.copy_(A.step_count[torch.as_tensor(cnt, device='cuda')])
    a = A.sample_actions(torch.Generator(device='cuda').manual_seed(1))
    A.reset_stats(); S.reset_stats()
    A.step(a)
    S.step(a[torch.as_tensor(cnt, device='cuda')].contiguous())
    got, want = A.stats(), S.stats()
    for k in ('env_steps', 'penalties', 'rescues', 'ticket_timeouts'):
        assert got[k] == want[k], (k, got[k], want[k])
    assert got['env_steps'] == cnt.sum()
    for k in ('sum_reward', 'sum_capacity_mbps', 'sum_reward_sq'):
        assert abs(got[k] - want[k]) <= 1e-5 * abs(want[k]), (k, got[k], want[k])
    A.close(); S.close()


def _mixed_sequence(torch, A, rounds=3, n=6):
    """`rounds` x (n flagged plain steps, n auto-reset steps, n flagged plain steps), every launch with its own actions and output set."""
    g = torch.Generator(device='cuda').manual_seed(17)
    return [(A.sample_actions(g), A.alloc_outputs(), plain) for _ in range(rounds) for plain in (True, False, True) for _ in range(n)]


def _launch_all(A, seq):
    for a, o, plain in seq:
        A._launch(a, o, True, not plain)        # flagged INPUTS_STABLE; the auto-reset steps take the default ordering anyway


def _digest(A, seq):
    """One synchronisation for the whole sequence: a digest of every launch's outputs, and the final state."""
    import hashlib
    torch = _torch()
    torch.cuda.synchronize()
    out = []
    for _, o, _ in seq:
        h = hashlib.sha1()
        for t in (o.obs, o.capacity_mbps, o.reward, o.done):
            h.update(t.cpu().numpy().tobytes())
        out.append(h.hexdigest())
    out.append({k: v.cpu().numpy().tobytes() for k, v in
                dict(positions=A.positions, step_count=A.step_count, episode_index=A.episode_index).items()})
    return out


@pytest.mark.gpu
@pytest.mark.parametrize('E,envv', [(4096, {}), (6144, {'D2D_B200_LATE_WAIT': '0'})], ids=['late_wait', 'tickets'])
def test_autoreset_between_flagged_plain_steps_orders_like_serialised_launches(E, envv, monkeypatch):
    """Three rounds of flagged plain steps (late wait at E = 4096, per-warp tickets at E = 6144 with the late wait off), auto-reset
    steps, flagged plain steps again - 54 launches enqueued with no host synchronisation between them, eagerly and as two replays of
    a CUDA graph, so that consecutive launches overlap.  Every launch's outputs and the final state equal the same sequences with
    programmatic dependent launch switched off.  (An auto-reset step writes the positions of the envs it resets: a plain step that
    read them ahead of its wait would see the previous episode's.)"""
    torch = _torch()
    for k, v in envv.items():
        monkeypatch.setenv(k, v)
    runs = []
    for pdl in ('1', '0'):
        monkeypatch.setenv('D2D_B200_PDL', pdl)
        A = _vec(E, seed=4, autoreset=True)
        A.reset(seed=2)
        A.step_count.copy_(torch.as_tensor(np.random.default_rng(E).integers(0, 13, E).astype(np.uint8), device='cuda'))
        seq = _mixed_sequence(torch, A)
        torch.cuda.synchronize()
        _launch_all(A, seq)
        r = [_digest(A, seq)]
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            with torch.cuda.graph(graph, stream=side):
                _launch_all(A, seq)
        torch.cuda.current_stream().wait_stream(side)
        for _ in range(2):
            graph.replay()
            r.append(_digest(A, seq))
        assert A.stats()['ticket_timeouts'] == 0
        runs.append(r)
        A.close()
    for what, fast, ref in zip(('eager', 'replay 1', 'replay 2'), *runs):
        for i, (x, y) in enumerate(zip(fast, ref)):
            assert x == y, f'{what}: ' + (f'launch {i}' if i < len(fast) - 1 else 'final state')


@pytest.mark.gpu
def test_autoreset_graph_replays_draw_fresh_episodes():
    """A captured graph of 25 auto-reset steps from a fresh reset crosses two episode boundaries.  Two replays draw different
    positions, and each replay equals the same 25 steps run eagerly from the same state."""
    torch = _torch()
    E = 4096
    A = _vec(E, seed=6, autoreset=True)
    A.reset(seed=8)
    g = torch.Generator(device='cuda').manual_seed(3)
    seq = [A.sample_actions(g) for _ in range(25)]
    outs = [A.alloc_outputs() for _ in range(25)]
    state0 = [t.clone() for t in (A.positions, A.step_count, A.episode_index)]
    graph = A.capture_steps(seq, outs)
    replays = []
    for _ in range(2):
        graph.replay()
        replays.append([_snap(A, o) for o in outs] + [{'episode_index': A.episode_index.cpu().numpy()}])
    assert (replays[0][-1]['episode_index'] == 2).all() and (replays[1][-1]['episode_index'] == 4).all()
    assert not np.array_equal(replays[0][-2]['positions'], replays[1][-2]['positions'])
    for dst, src in zip((A.positions, A.step_count, A.episode_index), state0):
        dst.copy_(src)
    for r in replays:
        for a, o in zip(seq, outs):
            A.step(a, out=o)
        eager = [_snap(A, o) for o in outs] + [{'episode_index': A.episode_index.cpu().numpy()}]
        for i, (x, y) in enumerate(zip(eager, r)):
            _assert_same(x, y, f'step {i}')
    A.close()


@pytest.mark.gpu
def test_autoreset_sharded_equals_one_handle(monkeypatch):
    """Two handles with global_env_offset splitting the batch step exactly like one handle over it: the reset draws depend on the
    global env, the key base and the episode index only."""
    torch = _torch()
    monkeypatch.setenv('D2D_B200_WPB', '4')
    E, H = 4096, 2048
    full = _vec(E, seed=5, info=True, autoreset=True)
    parts = [_vec(H, seed=5, info=True, autoreset=True, global_env_offset=k * H) for k in range(2)]
    rng = np.random.default_rng(2)
    ns = torch.as_tensor(rng.integers(0, 13, E).astype(np.uint8), device='cuda')
    ep = torch.as_tensor(rng.integers(0, 4, E).astype(np.int32), device='cuda')
    for env, sl in [(full, slice(0, E))] + [(p, slice(k * H, (k + 1) * H)) for k, p in enumerate(parts)]:
        env.reset(seed=12)
        env.step_count.copy_(ns[sl])
        env.episode_index.copy_(ep[sl])
    for k, p in enumerate(parts):
        p.positions.copy_(full.positions[k * H:(k + 1) * H])
    g = torch.Generator(device='cuda').manual_seed(9)
    for t in range(12):
        a = full.sample_actions(g)
        full.step(a)
        want = _snap(full)
        got = []
        for k, p in enumerate(parts):
            p.step(a[k * H:(k + 1) * H].contiguous())
            got.append(_snap(p))
        _assert_same({k: np.concatenate([x[k] for x in got]) for k in want}, want, f'step {t}')
    for env in [full] + parts:
        env.close()


@pytest.mark.gpu
@pytest.mark.parametrize('kind', ['shannon', 'cue_sinr_shannon'])
def test_autoreset_per_agent_rewards(kind):
    """With a per-agent reward function the rows of reset envs have agent_reward = 0 and reward = 0; every other row equals a plain
    step on the same positions and actions."""
    torch = _torch()
    import gym_d2d_b200 as G
    fn = G.ShannonRewardFunction if kind == 'shannon' else G.CueSinrShannonRewardFunction
    E = 3000
    A = _vec(E, {'reward_fn': fn}, seed=1, autoreset=True)
    B = _vec(E, {'reward_fn': fn}, seed=1)
    rng = np.random.default_rng(8)
    A.reset(seed=4)
    _desync(torch, A, B, rng, False, O.OracleConfig())
    rst = (A.step_count >= L).cpu().numpy()
    a = _actions(torch, A, rng, True)
    A.reset_stats(); B.reset_stats()
    A.step(a)
    B.step(a)
    got, want = _snap(A), _snap(B)
    assert (got['agent_reward'][rst] == 0).all() and (got['reward'][rst] == 0).all()
    np.testing.assert_array_equal(got['agent_reward'][~rst], want['agent_reward'][~rst])
    np.testing.assert_array_equal(got['reward'][~rst], want['reward'][~rst])
    r = want['reward'][~rst].astype(np.float64)
    st = A.stats()
    assert st['env_steps'] == (~rst).sum()
    assert abs(st['sum_reward'] - r.sum()) <= 1e-5 * max(1.0, abs(r.sum()))
    A.close(); B.close()


@pytest.mark.gpu
def test_autoreset_positions_follow_the_reference_distribution(golden_dir):
    """Positions drawn by 100 000 auto-resets pass the same KS checks as d2d_reset against the reference's samplers."""
    torch = _torch()
    fx = np.load(golden_dir / 'reset_distribution.npz')
    E = 100_000
    A = _vec(E, seed=13, autoreset=True)
    A.reset(seed=1)
    A.step_count.fill_(L)
    A.step(A.sample_actions())
    assert (A.step_count == 0).all() and (A.episode_index == 1).all() and (A.done == 0).all() and (A.reward == 0).all()
    check_reset_distribution(A.positions.cpu().numpy(), 25, fx)
    A.close()


@pytest.mark.gpu
def test_autoreset_refusals():
    """autoreset=True raises at construction where the warp kernel does not serve the configuration (dense, downlinks); the flag is
    refused by every step entry point but d2d_step, and without a bound episode index or step counter."""
    import ctypes as C
    _torch()
    import gym_d2d_b200 as G
    from gym_d2d_b200 import _lib
    for cfg_kw, kw in ((dict(num_rbs=100, num_cues=100, num_due_pairs=500), {}), (dict(num_rbs=16, num_cues=24, num_due_pairs=40), {}),
                       ({}, dict(downlink=True)), (dict(path_loss_model=G.ShadowingPathLoss), {})):
        with pytest.raises(_lib.D2DUnsupportedError):
            _vec(64, cfg_kw, autoreset=True, **kw)
    A = _vec(64, autoreset=True)
    A.reset()
    a = A.sample_actions()
    many = A.alloc_many_outputs(2)
    a2 = a.unsqueeze(0).repeat(2, 1, 1).contiguous()
    io = _lib.D2DStepIO(actions=a2.data_ptr(), obs=many['obs'].data_ptr(), capacity_mbps=many['capacity_mbps'].data_ptr(),
                        reward=many['reward'].data_ptr(), done=many['done'].data_ptr(), flags=_lib.STEP_AUTORESET)
    assert A._lib.d2d_step_many(A._h, C.byref(io), 2, A._stream()) == _lib.ERR_UNSUPPORTED
    assert A._lib.d2d_episode(A._h, C.byref(io), 1, 1, 1, 0, A._stream()) == _lib.ERR_UNSUPPORTED
    assert A._lib.d2d_rollout(A._h, C.byref(io), 2, 1, 1, A._stream()) == _lib.ERR_UNSUPPORTED
    B = _vec(64)
    io1 = B._out._io
    io1.actions = a.data_ptr()
    io1.flags = _lib.STEP_AUTORESET
    assert B._lib.d2d_step(B._h, C.byref(io1), B._stream()) == _lib.ERR_STATE          # no episode index bound
    B._bind(False)
    _lib.check(B._lib.d2d_bind_autoreset(B._h, A.episode_index.data_ptr(), 0))
    assert B._lib.d2d_step(B._h, C.byref(io1), B._stream()) == _lib.ERR_STATE          # no step counter bound
    io1.flags = 0
    A.close(); B.close()
