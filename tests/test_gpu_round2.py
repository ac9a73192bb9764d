"""GPU tier (-m gpu), second batch: the episode path (device-side reset, on-device action sampling, d2d_episode), the
per-step observation columns (obs_dyn) and packed host slots, the programmatic-dependent-launch ordering rule, and the
device guard.  Same conventions as test_gpu_parity.py: everything goes through the C ABI; the oracle is the checker.
"""
import numpy as np
import pytest

from oracle import d2d_oracle as O
from tests._util import check_reset_distribution
from tests.test_gpu_parity import CONFIGS, make_vec

torch = pytest.importorskip('torch')
pytestmark = pytest.mark.gpu

# Configurations served by the one-warp-per-env kernel are bit-reproducible from launch to launch.  The block kernels rank a
# link inside its RB bin with shared-memory atomics from several warps, so the ORDER of an interference sum - and with it the
# last ulp of an fp32 result - may differ between two launches on the same inputs (the reference sums in Python-set order,
# actions.py:27-31, which is no more canonical); two launches are then compared to 1e-5 (relative, or absolute dB).
WARP_CONFIGS = {'default', 'small', 'one_rb_crowded', 'dense_small', 'tiny', 'cue_only', 'due_only', 'warp_max'}


def same(a, b, name):
    if name in WARP_CONFIGS:
        return torch.equal(a, b)
    return torch.allclose(a.float(), b.float(), rtol=1e-5, atol=1e-5) if a.is_floating_point() else torch.equal(a, b)


# ---- reset: the distribution of the reference's own sampler (position.py:18-45) -------------------------------------------
def test_reset_distribution_matches_reference_sampler(golden_dir):
    fx = np.load(golden_dir / 'reset_distribution.npz')
    env = make_vec(8192, seed=99)
    env.reset()
    torch.cuda.synchronize()
    check_reset_distribution(env.positions.cpu().numpy(), 25, fx)
    out = env.episode(2)                                   # the fused kernel draws the same way
    torch.cuda.synchronize()
    check_reset_distribution(env.positions.cpu().numpy(), 25, fx)
    assert out['obs'].shape == (3, 8192, 50, 6)
    env.close()


def test_sample_actions_match_oracle_and_are_uniform():
    for name in ('default', 'small', 'block_min'):
        kw = CONFIGS[name]
        cfg = O.OracleConfig(**kw)
        E = 3000
        env = make_vec(E, kw, global_env_offset=77)
        for t in (0, 1, 2, 7):
            got = env.sample_actions_philox(seed=1234, step_index=t).cpu().numpy()
            want = O.sample_actions(cfg, 1234, 77, t, E)
            np.testing.assert_array_equal(got, want)
        a = np.concatenate([env.sample_actions_philox(5, t).cpu().numpy() for t in range(8)])
        nvec = env.action_nvec
        assert (a >= 0).all() and (a < nvec).all()
        # uniform over 0 .. n - 1 (gym.spaces.Discrete.sample): mean (n - 1) / 2, every value's share 1 / n
        assert np.abs(a.mean(0) / ((nvec - 1) / 2) - 1).max() < 0.03
        j = 0
        counts = np.bincount(a[:, j], minlength=int(nvec[j]))
        expect = a.shape[0] / nvec[j]
        assert np.abs(counts - expect).max() < 6 * np.sqrt(expect) + 1
        env.close()


# ---- d2d_episode == d2d_reset + d2d_sample_actions + d2d_step x (T + 1) --------------------------------------------------------
@pytest.mark.parametrize('name', ['default', 'small', 'one_rb_crowded', 'block_min', 'dense_small'])
@pytest.mark.parametrize('given_actions', [False, True])
def test_episode_equals_reset_plus_single_steps(name, given_actions):
    kw = CONFIGS[name]
    E, T = 257, 10
    fused = make_vec(E, kw, seed=31, global_env_offset=5)
    single = make_vec(E, kw, seed=31, global_env_offset=5)
    for ep in range(2):                                     # two consecutive episodes: the key sequence advances alike
        key = (31 + 0x9E3779B97F4A7C15 * ep) & 0xFFFFFFFFFFFFFFFF
        fused.reset_stats(); single.reset_stats()
        acts = None
        if given_actions:
            acts = torch.stack([single.sample_actions() for _ in range(T + 1)]).contiguous()
        out = fused.episode(T, actions=acts, record_actions=True)
        torch.cuda.synchronize()
        # positions: exactly what reset() draws for the same episode key
        single.reset(mask=torch.ones(E, dtype=torch.uint8, device='cuda'))
        assert torch.equal(fused.positions, single.positions)
        assert (fused.step_count == T).all()
        for t in range(T + 1):
            a = acts[t] if given_actions else single.sample_actions_philox(key, t)
            if not given_actions:
                assert torch.equal(out['actions'][t], a)
            if t == 0:                                      # envs/d2d_env.py:50: the reset step is not counted
                single._bind(False)
            obs, reward, done, info = single.step(a)
            single._bind(True)
            torch.cuda.synchronize()
            assert same(out['obs'][t], obs, name), (name, t)
            assert same(out['capacity_mbps'][t], info['capacity_mbps'], name)
            assert same(out['rate_bps'][t], info['rate_bps'], name)
            assert torch.equal(out['rb'][t], info['rb']) and torch.equal(out['tx_pwr_dbm'][t], info['tx_pwr_dbm'])
            assert same(out['reward'][t], reward, name)
            assert (out['done'][t] == (1 if t >= 10 else 0)).all()
        assert (single.step_count == T).all()
        sf, ss = fused.stats(), single.stats()
        assert sf['env_steps'] == ss['env_steps'] == T * E
        assert sf['penalties'] == ss['penalties'] and (sf['rescues'] == ss['rescues'] or name not in WARP_CONFIGS)
        for k in ('sum_reward', 'sum_capacity_mbps', 'sum_reward_sq'):
            assert sf[k] == pytest.approx(ss[k], rel=1e-6)
    # the episode leaves a state d2d_step continues from
    a = single.sample_actions()
    o1 = fused.step(a)[0].clone()
    o2 = single.step(a)[0]
    assert same(o1, o2, name) and (fused.step_count == T + 1).all()
    fused.close(); single.close()


def test_episode_first_step_matches_oracle():
    cfg = O.OracleConfig()
    E = 512
    env = make_vec(E, seed=3)
    out = env.episode(3, record_actions=True)
    torch.cuda.synchronize()
    pos = env.positions.double().cpu().numpy()
    for t in range(4):
        ref = O.step_batch(cfg, pos, out['actions'][t].cpu().numpy(), nthreads=4)
        from tests._util import RTOL, assert_rel
        assert_rel(out['obs'][t, :, :, 4].cpu().numpy(), ref['sinr_db'], RTOL, f'sinr slice {t}')
        assert_rel(out['capacity_mbps'][t].cpu().numpy(), ref['capacity_mbps'], RTOL, f'capacity slice {t}')
        assert_rel(out['reward'][t].cpu().numpy(), ref['reward'], RTOL, f'reward slice {t}')
        np.testing.assert_array_equal(out['rb'][t].cpu().numpy(), ref['rb'])
    env.close()


def test_episode_with_per_agent_rewards():
    import gym_d2d_b200 as G
    E, T = 300, 4
    kw = dict(reward_fn=G.ShannonRewardFunction)
    fused = make_vec(E, dict(kw), seed=8)
    single = make_vec(E, dict(kw), seed=8)
    out = fused.episode(T, record_actions=True)
    single.reset(mask=torch.ones(E, dtype=torch.uint8, device='cuda'))
    single.reset_stats()
    for t in range(T + 1):
        if t == 0:
            single._bind(False)
        obs, reward, done, info = single.step(out['actions'][t].contiguous())
        single._bind(True)
        assert torch.equal(out['agent_reward'][t], info['agent_reward']) and torch.equal(out['reward'][t], reward)
    # the reset step's rewards enter no statistic
    assert fused.stats()['sum_reward'] == pytest.approx(out['reward'][1:].double().sum().item(), rel=1e-5)
    fused.close(); single.close()


# ---- obs_dyn / packed host slots --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('name', ['default', 'small', 'block_min', 'dense_small', 'dense'])
def test_obs_dyn_reassembles_the_full_table_bit_for_bit(name):
    """obs == (positions gathered per link, obs_dyn): BOTH outputs of the SAME launch, through the packed host slots, must
    reassemble bit for bit; the default slot layout (obs_dyn + capacity + reward + done) must equal a full-table host step."""
    kw = CONFIGS[name]
    E = 300 if name != 'dense' else 24
    env = make_vec(E, kw, seed=4)
    env.reset()
    static = env.obs_static()
    both = [env.host_slot_buffers(s, outputs=('obs', 'obs_dyn', 'capacity_mbps', 'reward', 'done')) for s in (0, 1)]
    for i in range(6):
        a = env.sample_actions().cpu().numpy()
        if i % 2:
            a[::3, ::2] = -1                                 # absent agents keep their position columns
        s = both[i & 1]
        s['actions'][...] = a
        env.step_host_async(s['actions'], s, i & 1)
        env.step_host_wait(i & 1)
        np.testing.assert_array_equal(env.assemble_obs(static, s['obs_dyn']), s['obs'])
        assert np.abs(s['obs'][..., 4]).max() > 0
    # the default slot layout against a full-table host step on caller-owned buffers (two launches: see WARP_CONFIGS)
    full = env.alloc_host_outputs(info=True)
    slots = [env.host_slot_buffers(s) for s in (2, 3)]
    assert set(slots[0]) == {'actions', 'actions16', 'obs_dyn', 'capacity_mbps', 'reward', 'done'}      # ('actions16': the same pinned bytes as int16)
    dyn = env.alloc_host_outputs(info=False, dyn=True)
    for i in range(4):
        a = env.sample_actions().cpu().numpy()
        env.step_count.zero_(); env.step_host(a, full)
        env.step_count.zero_()
        s = slots[i & 1]
        env.step_host_async(a, s, 2 + (i & 1))                # actions from the caller's own buffer, outputs into the slot
        env.step_host_wait(2 + (i & 1))
        env.step_count.zero_(); env.step_host(a, dyn)
        for got in (s, dyn):
            if name in WARP_CONFIGS:
                np.testing.assert_array_equal(env.assemble_obs(static, got['obs_dyn']), full['obs'])
                np.testing.assert_array_equal(got['capacity_mbps'], full['capacity_mbps'])
                np.testing.assert_array_equal(got['reward'], full['reward'])
            else:
                np.testing.assert_allclose(env.assemble_obs(static, got['obs_dyn']), full['obs'], rtol=1e-5, atol=1e-5)
                np.testing.assert_allclose(got['capacity_mbps'], full['capacity_mbps'], rtol=1e-5, atol=1e-6)
            np.testing.assert_array_equal(got['done'], full['done'])
    # a positions change shows up in get_positions
    env.reset()
    assert not np.array_equal(env.obs_static(), static)
    env.close()


# ---- the ordering rule of include/d2d_b200.h ----------------------------------------------------------------------------------------
def _policy(env, obs, out):
    """A stand-in policy kernel: the next actions are a function of the current observation (a real data dependency)."""
    x = (obs[..., 4].abs() * 977.0 + obs[..., 5].abs() * 131.0).to(torch.int64)
    out.copy_((x % env._nvec_dev).to(torch.int32))


@pytest.mark.parametrize('E', [256, 4096])
def test_pdl_policy_writes_actions_between_steps(monkeypatch, E):
    """10 000 iterations of {torch kernels write the actions -> step}: the default ordering must give exactly what a library
    without programmatic dependent launch gives, eagerly and from a replayed CUDA graph."""
    iters = 10000
    monkeypatch.setenv('D2D_B200_PDL', '0')
    plain = make_vec(E, seed=21)
    monkeypatch.delenv('D2D_B200_PDL')
    pdl = make_vec(E, seed=21)
    graphed = make_vec(E, seed=21)
    for env in (plain, pdl, graphed):
        env.reset(initial_actions=torch.zeros((E, 50), dtype=torch.int32, device='cuda'))
    acts = {env: torch.zeros((E, 50), dtype=torch.int32, device='cuda') for env in (plain, pdl, graphed)}
    diff = torch.zeros((), dtype=torch.int64, device='cuda')

    def one(env):
        _policy(env, env.obs, acts[env])
        env.step(acts[env])                                   # default: ordered after the policy's writes

    # the graph holds 8 policy + step pairs
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            for _ in range(8):
                one(graphed)
    torch.cuda.current_stream().wait_stream(s)
    for env in (plain, pdl):                                  # the capture did not execute: start all three from one state
        env.step_count.zero_()
    graphed.step_count.zero_()
    for it in range(iters // 8):
        for _ in range(8):
            one(plain); one(pdl)
        g.replay()
        if it % 50 == 0:
            diff += (plain.obs != pdl.obs).sum() + (plain.obs != graphed.obs).sum() + (plain.reward != pdl.reward).sum()
    diff += (plain.obs != pdl.obs).sum() + (plain.obs != graphed.obs).sum() + (acts[plain] != acts[pdl]).sum() + (acts[plain] != acts[graphed]).sum()
    torch.cuda.synchronize()
    assert int(diff.item()) == 0
    assert torch.equal(plain.step_count, pdl.step_count) and torch.equal(plain.step_count, graphed.step_count)
    for env in (plain, pdl, graphed):
        env.close()


def test_pdl_reset_then_step_and_stable_flag(monkeypatch):
    """{reset -> step} x 10 000 and a run of inputs_stable steps: bit-identical to a library without PDL."""
    E = 1024
    monkeypatch.setenv('D2D_B200_PDL', '0')
    plain = make_vec(E, seed=5)
    monkeypatch.delenv('D2D_B200_PDL')
    pdl = make_vec(E, seed=5)
    ring = [pdl.sample_actions() for _ in range(4)]
    all_envs = torch.ones(E, dtype=torch.uint8, device='cuda')
    diff = torch.zeros((), dtype=torch.int64, device='cuda')
    for it in range(10000):
        a = ring[it & 3]
        for env in (plain, pdl):
            env.reset(mask=all_envs)                          # new positions every iteration (same key sequence in both)
            env.step(a, inputs_stable=True)                   # the library must ignore the flag right after a reset
            env.step(ring[(it + 1) & 3], inputs_stable=True)  # honoured here: follows a step, actions long written
        if it % 100 == 0:
            diff += (plain.obs != pdl.obs).sum() + (plain.positions != pdl.positions).sum()
    diff += (plain.obs != pdl.obs).sum() + (plain.reward != pdl.reward).sum()
    torch.cuda.synchronize()
    assert int(diff.item()) == 0
    plain.close(); pdl.close()


def test_episode_then_step_orders_after_the_position_writes(monkeypatch):
    E = 2048
    monkeypatch.setenv('D2D_B200_PDL', '0')
    plain = make_vec(E, seed=6)
    monkeypatch.delenv('D2D_B200_PDL')
    pdl = make_vec(E, seed=6)
    a = pdl.sample_actions()
    diff = torch.zeros((), dtype=torch.int64, device='cuda')
    outs = {env: env.alloc_many_outputs(3) for env in (plain, pdl)}
    for it in range(2000):
        for env in (plain, pdl):
            env.episode(2, out=outs[env])
            env.step(a, inputs_stable=True)                   # reads the positions the episode kernel just wrote
        if it % 50 == 0:
            diff += (plain.obs != pdl.obs).sum() + (outs[plain]['obs'] != outs[pdl]['obs']).sum()
    diff += (plain.obs != pdl.obs).sum()
    torch.cuda.synchronize()
    assert int(diff.item()) == 0
    plain.close(); pdl.close()


# ---- device guard (ADVICE r1): a handle on a device other than the caller's current one -------------------------------------------------
def test_env_on_another_device_than_the_current_one():
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    import gym_d2d_b200 as G
    torch.cuda.set_device(0)
    cfg = O.OracleConfig()
    env1 = G.VecD2DEnv(300, {}, device='cuda:1', info=True, seed=1)
    env0 = G.VecD2DEnv(300, {}, device='cuda:0', info=True, seed=1)
    assert torch.cuda.current_device() == 0
    env1.reset(); env0.reset()
    assert torch.cuda.current_device() == 0
    assert torch.equal(env1.positions.cpu(), env0.positions.cpu())
    a = env0.sample_actions()
    o1 = env1.step(a.to('cuda:1'))[0]
    o0 = env0.step(a)[0]
    assert torch.cuda.current_device() == 0 and o1.device.index == 1
    torch.cuda.synchronize(0); torch.cuda.synchronize(1)
    assert torch.equal(o1.cpu(), o0.cpu())
    ref = O.step_batch(cfg, env1.positions.double().cpu().numpy(), a.cpu().numpy(), nthreads=2)
    from tests._util import RTOL, assert_rel
    assert_rel(o1[..., 4].cpu().numpy(), ref['sinr_db'], RTOL, 'sinr on cuda:1')
    out = env1.episode(3)
    env1.step_host(a.cpu().numpy())
    assert torch.cuda.current_device() == 0
    env1.close(); env0.close()


# ---- ShadowingPathLoss under CUDA graphs: every replay draws fresh values (path_loss.py:75-81) ----------------------------------------------
def test_shadowing_graph_replays_draw_fresh_values():
    import gym_d2d_b200 as G
    E = 64
    kw = dict(num_rbs=3, num_cues=4, num_due_pairs=5, path_loss_model=G.ShadowingPathLoss)
    eager = make_vec(E, dict(kw), seed=9)
    graphed = make_vec(E, dict(kw), seed=9)
    pos = O.random_positions(O.OracleConfig(num_rbs=3, num_cues=4, num_due_pairs=5), E, np.random.default_rng(0))
    eager.set_positions(pos); graphed.set_positions(pos)
    a = eager.sample_actions()
    g = graphed.capture_steps([a])
    seen = []
    for i in range(3):
        want = eager.step(a)[0].clone()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(graphed.obs, want), i              # replay i == the i-th eager call: same counter, same draws
        seen.append(want)
    assert not torch.equal(seen[0], seen[1]) and not torch.equal(seen[1], seen[2])
    eager.close(); graphed.close()


# ---- per-agent rewards with many resource blocks (ADVICE r1: the post-pass asked for 32 B of shared memory per RB) ----------------------------
@pytest.mark.parametrize('kind', ['shannon', 'cue_sinr_shannon'])
def test_per_agent_rewards_with_many_rbs(kind):
    import gym_d2d_b200 as G
    fn, param = (G.ShannonRewardFunction, -70.0) if kind == 'shannon' else (G.CueSinrShannonRewardFunction, 0.0)
    kw = dict(num_rbs=3000, num_cues=6, num_due_pairs=10)
    cfg = O.OracleConfig(**kw)
    E = 40
    env = make_vec(E, dict(kw, reward_fn=fn), seed=2)
    rng = np.random.default_rng(5)
    pos = O.random_positions(cfg, E, rng)
    act = O.random_actions(cfg, E, rng)
    act[:, :] = act[:, :] % (7 * 21)                          # crowd a few RBs so that the CUE-SINR rule has something to do
    env.set_positions(pos)
    obs, reward, done, info = env.step(torch.as_tensor(act, dtype=torch.int32, device='cuda'))
    torch.cuda.synchronize()
    ref = O.step_batch(cfg, pos, act, nthreads=2)
    want = O.agent_rewards(cfg, ref, kind, param)
    from tests.test_gpu_parity import _agent_reward_check
    _agent_reward_check(info['agent_reward'].cpu().numpy(), want, ref['sinr_db'], param)
    env.close()


# ---- per-agent reward thresholds decided in fp64 (VERDICT r1: the threshold neighbourhood used to be exempt) -------------------------
@pytest.mark.parametrize('name', ['default', 'block_min', 'dense_small', 'one_rb_crowded', 'sorting', 'general'])
@pytest.mark.parametrize('kind', ['shannon', 'cue_sinr_shannon'])
def test_reward_threshold_a_hair_from_a_link_sinr(name, kind):
    """The threshold is placed 1e-9 dB above / below the float64 SINR of actual links - far inside fp32's resolution of a dB
    value (4e-6 dB at best) - so only the fp64 pass with threshold-consistent rounding can decide those links like the
    reference (envs/reward_fn.py:55,72).  Every agent is checked, none exempt."""
    import gym_d2d_b200 as G
    from tests._util import RTOL, rel_err
    kw = CONFIGS[name]
    cfg = O.OracleConfig(**kw)
    rng = np.random.default_rng(77)
    E = 96
    pos, act = O.random_positions(cfg, E, rng), O.random_actions(cfg, E, rng)
    ref = O.step_batch(cfg, pos, act, nthreads=4)
    C_ = cfg.num_cues
    cls = G.ShannonRewardFunction if kind == 'shannon' else G.CueSinrShannonRewardFunction
    a = torch.as_tensor(act, dtype=torch.int32, device='cuda')
    flips = 0
    for pick in range(6):
        # a link that matters for the rule: any link for Shannon, a CUE that shares its RB for CueSinrShannon
        e = int(rng.integers(E))
        if kind == 'shannon' or C_ == 0:
            j = int(rng.integers(cfg.num_links))
        else:
            shared = [j for j in range(C_) if (ref['rb'][e] == ref['rb'][e, j]).sum() > 1]
            if not shared:
                continue
            j = int(rng.choice(shared))
        s_star = float(ref['sinr_db'][e, j])
        for eps in (+1e-9, -1e-9):
            thr = s_star + eps
            env = make_vec(E, dict(kw, reward_fn=_with_param(cls, thr)))
            env.set_positions(pos)
            obs, reward, done, info = env.step(a)
            torch.cuda.synchronize()
            want = O.agent_rewards(cfg, ref, kind, thr)
            got = info['agent_reward'].cpu().numpy()
            err = rel_err(got, want)
            assert (err <= RTOL).all(), (name, kind, pick, eps, float(err.max()), np.argwhere(err > RTOL)[:4])
            flips += int((want[e] == -1).sum())
            env.close()
    assert flips > 0                                                   # the -1 branch was exercised at the hair's breadth


def _with_param(cls, value):
    """The plugin surface takes CLASSES (envs/d2d_env.py:27-28 instantiates them without arguments); a threshold other than
    the default is passed the way the reference's users do it: functools.partial over the class."""
    import functools
    import gym_d2d_b200 as G
    return functools.partial(cls, **{'min_sinr' if cls is G.ShannonRewardFunction else 'sinr_threshold_dB': value})


# ---- ADVICE r1: a device_config_file that places a DUE transmitter but not its receiver ------------------------------------------
def test_partial_device_file_redraws_receivers_around_file_transmitters(tmp_path):
    import json
    import gym_d2d_b200 as G
    # transmitters of pairs 0 and 1 pinned near the cell edge / centre; their receivers and everything else left to reset()
    doc = {'due00': {'position': [480.0, 0.0]}, 'due02': {'position': [-3.0, 4.0]}, 'cue00': {'position': [100.0, -50.0]}}
    f = tmp_path / 'partial.json'
    f.write_text(json.dumps(doc))
    env = G.D2DEnv({'device_config_file': f}, seed=3)
    for _ in range(5):
        env.reset()
        pos = env.device_positions()
        assert pos['due00'] == (480.0, 0.0) and pos['due02'] == (-3.0, 4.0) and pos['cue00'] == (100.0, -50.0)
        for tx, rx in (('due00', 'due01'), ('due02', 'due03')):
            d = np.hypot(pos[rx][0] - pos[tx][0], pos[rx][1] - pos[tx][1])
            assert d <= 20.0 and np.hypot(*pos[rx]) <= 500.0, (tx, rx, d)      # simulator.py:70-73, position.py:31-45
        d = np.hypot(pos['due05'][0] - pos['due04'][0], pos['due05'][1] - pos['due04'][1])
        assert d <= 20.0 + 1e-3                                                # untouched pairs keep the device-side draw
    env.close()


@pytest.mark.parametrize('name', ['default', 'small', 'block_min'])
def test_rollout_equals_sampled_single_steps(name):
    """d2d_rollout: T counted steps with on-device sampled actions == d2d_sample_actions + d2d_step, slice for slice."""
    kw = CONFIGS[name]
    E, T = 300, 7
    fused = make_vec(E, kw, seed=12)
    single = make_vec(E, kw, seed=12)
    fused.reset(initial_actions=fused.sample_actions_philox(1, 0)); single.reset(initial_actions=single.sample_actions_philox(1, 0))
    fused.reset_stats(); single.reset_stats()
    out = fused.rollout(T, action_seed=99, first_step_index=3, record_actions=True)
    for t in range(T):
        a = single.sample_actions_philox(99, 3 + t)
        assert torch.equal(out['actions'][t], a)
        obs, reward, done, info = single.step(a)
        assert same(out['obs'][t], obs, name) and same(out['reward'][t], reward, name) and torch.equal(out['done'][t], done)
        assert same(out['capacity_mbps'][t], info['capacity_mbps'], name)
    assert torch.equal(fused.step_count, single.step_count) and (fused.step_count == T).all()
    sf, ss = fused.stats(), single.stats()
    assert sf['env_steps'] == ss['env_steps'] == T * E and sf['penalties'] == ss['penalties']
    assert sf['sum_reward'] == pytest.approx(ss['sum_reward'], rel=1e-6)
    fused.close(); single.close()


# ---- VERDICT r1 weak #3: adversarial sweep of the fp64-pass band edge ------------------------------------------------------------------
@pytest.mark.parametrize('ple', [2.0, 3.5])
def test_band_edge_sweep_of_sinr_and_snr(ple):
    """|SINR_dB| and |SNR_dB| swept densely over 0.05 .. 0.15 dB (ple = 2; 0.4 .. 0.7 dB for ple != 2), both signs - either side of the
    band below which links are recomputed in fp64 (0.0625 dB / 0.5 dB) - on links with and without an interferer.  A pure 1e-4
    relative bound on a dB value is tightest right outside the band; the worst relative error found must leave a 2x margin."""
    import gym_d2d_b200 as G
    kw = dict(num_rbs=1, num_cues=0, num_due_pairs=2, path_loss_model=G.LogDistancePathLoss if ple == 2.0 else
              __import__('functools').partial(G.LogDistancePathLoss, ple=ple))
    okw = dict(num_rbs=1, num_cues=0, num_due_pairs=2, ple=ple)
    cfg = O.OracleConfig(**okw)
    lo, hi = (0.05, 0.15) if ple == 2.0 else (0.4, 0.7)
    E = 40000
    rng = np.random.default_rng(int(ple * 10))
    target = rng.uniform(lo, hi, E) * rng.choice([-1.0, 1.0], E)
    p = rng.integers(0, 21, (E, 2))
    # link budget of a DUE pair (device.py:12-41 defaults): SNR_dB = p + snr0 - 10 ple log10(d)
    K = 10 * ple * np.log10(2.1e9) + 10 * ple * np.log10(4 * np.pi / 299792458.0)
    snr0 = -6.0 - 3.0 - K + 104.5
    pos = np.zeros((E, 5, 2))
    half = E // 2
    # first half: no co-channel interference (the second pair is absent) -> SINR = SNR = target
    d = 10 ** ((p[:, 0] + snr0 - target) / (10 * ple))
    th = rng.uniform(0, 2 * np.pi, E)
    pos[:, 1] = rng.uniform(-50, 50, (E, 2))
    pos[:, 2] = pos[:, 1] + np.stack([d * np.cos(th), d * np.sin(th)], -1)
    # second half: SNR fixed at 6 .. 12 dB, an interferer placed so that SINR = target
    snr = rng.uniform(6.0, 12.0, E)
    d2 = 10 ** ((p[:, 0] + snr0 - snr) / (10 * ple))
    pos[half:, 2] = pos[half:, 1] + np.stack([d2 * np.cos(th), d2 * np.sin(th)], -1)[half:]
    noise = 10 ** (-104.5 / 10)
    S = 10 ** ((p[:, 0] - 6.0 - 3.0 - K) / 10) * d2 ** (-ple)            # received signal, linear mW
    I = S / 10 ** (target / 10) - noise                                    # interference that gives SINR = target
    w = 10 ** ((p[:, 1] - 6.0 - K) / 10)                                   # interferer EIRP minus the path-loss constant
    di = (w / I) ** (1.0 / ple)
    ph = rng.uniform(0, 2 * np.pi, E)
    pos[:, 3] = pos[:, 2] + np.stack([di * np.cos(ph), di * np.sin(ph)], -1)
    pos[:, 4] = pos[:, 3] + np.array([3.0, 4.0])
    pos = pos.astype(np.float32).astype(np.float64)
    act = p.astype(np.int32)                                               # one RB: action = power level
    act[:half, 1] = -1
    active = (act >= 0).astype(np.uint8)
    env = make_vec(E, dict(kw))
    env.set_positions(pos)
    obs, reward, done, info = env.step(torch.as_tensor(act, dtype=torch.int32, device='cuda'))
    torch.cuda.synchronize()
    ref = O.step_batch(cfg, pos, np.where(act >= 0, act, 0), active=active, nthreads=4)
    got_sinr, got_snr = obs[:, 0, 4].double().cpu().numpy(), obs[:, 0, 5].double().cpu().numpy()
    rs, rn = ref['sinr_db'][:, 0], ref['snr_db'][:, 0]
    # the sweep hit what it aimed at: SINR within the swept range, on both sides of the band edge and of zero
    band = 0.0625 if ple == 2.0 else 0.5
    assert (np.abs(rs) < band).sum() > 1000 and (np.abs(rs) > band).sum() > 1000 and (rs > 0).sum() > 1000 and (rs < 0).sum() > 1000
    assert np.abs(np.abs(rs) - np.abs(target)).max() < 0.02
    e_sinr = np.abs(got_sinr - rs) / np.abs(rs)
    e_snr = np.abs(got_snr[:half] - rn[:half]) / np.abs(rn[:half])
    worst = max(e_sinr.max(), e_snr.max())
    print(f'ple={ple}: worst relative error {worst:.3e} (sinr {e_sinr.max():.3e} at {rs[e_sinr.argmax()]:+.4f} dB, '
          f'snr {e_snr.max():.3e} at {rn[:half][e_snr.argmax()]:+.4f} dB); inside the band {e_sinr[np.abs(rs) < band].max():.2e}')
    assert worst < 0.5e-4, worst                                           # a 2x margin to the 1e-4 bound
    env.close()


# ---- per-warp tickets: chains of flagged single-launch steps ---------------------------------------------------------------------------------
@pytest.mark.parametrize('E,grid', [(4096, None), (1000, None), (70000, None), (3000, '7'), (130, '3')])
def test_ticket_chains_bit_identical_to_serialised_launches(monkeypatch, E, grid):
    """Consecutive D2D_STEP_INPUTS_STABLE steps wait per warp for the warp that stepped the same envs one launch earlier
    (d2d_ticket_wait) instead of for the whole previous grid.  Thousands of replays of a 16-step graph that reuses ONE output
    buffer set (so every step overwrites its predecessor's rows and reads its counters), eager chains, chains broken by a reset
    and by a change of stream: all bit-identical to a library without programmatic dependent launch; no ticket ever timed out."""
    if grid:
        monkeypatch.setenv('D2D_B200_GRID', grid)            # few blocks: warps step many envs, some none
    monkeypatch.setenv('D2D_B200_PDL', '0')
    plain = make_vec(E, seed=9)
    monkeypatch.delenv('D2D_B200_PDL')
    chain = make_vec(E, seed=9)
    monkeypatch.setenv('D2D_B200_TICKET', '0')
    noticket = make_vec(E, seed=9)
    monkeypatch.delenv('D2D_B200_TICKET')
    envs = (plain, chain, noticket)
    for env in envs:
        env.reset()
        env.reset_stats()
    ring = [chain.sample_actions() for _ in range(4)]
    seq = [ring[i % 4] for i in range(16)]
    graphs = {env: env.capture_steps(seq, inputs_stable=True) for env in (chain, noticket)}
    diff = torch.zeros((), dtype=torch.int64, device='cuda')
    replays = 400 if E <= 4096 else 60

    def check():
        return ((plain.obs != chain.obs).sum() + (plain.obs != noticket.obs).sum() + (plain.reward != chain.reward).sum() +
                (plain.step_count != chain.step_count).sum() + (plain.capacity_mbps != chain.capacity_mbps).sum())

    for it in range(replays):
        for a in seq:
            plain.step(a)
        graphs[chain].replay(); graphs[noticket].replay()
        if it % 20 == 0:
            diff += check()
    # eager chains, broken in the middle by a masked reset (new positions: the next step must order itself the default way)
    mask = torch.ones(E, dtype=torch.uint8, device='cuda')
    for it in range(40):
        for env in envs:
            for k in range(8):
                env.step(ring[(it + k) % 4], inputs_stable=True)
            env.reset(mask=mask)
            env.step(ring[it % 4], inputs_stable=True)
            env.step(ring[(it + 1) % 4], inputs_stable=True)
        diff += check() + (plain.positions != chain.positions).sum()
    # a chain continued on another stream starts over
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for env in envs:
            for k in range(6):
                env.step(ring[k % 4], inputs_stable=True)
    torch.cuda.current_stream().wait_stream(side)
    diff += check()
    torch.cuda.synchronize()
    assert int(diff.item()) == 0
    sp, sc = plain.stats(), chain.stats()
    assert sc['ticket_timeouts'] == 0 and noticket.stats()['ticket_timeouts'] == 0
    assert sp['env_steps'] == sc['env_steps'] and sp['rescues'] == sc['rescues'] and sp['penalties'] == sc['penalties']
    assert sc['sum_reward'] == pytest.approx(sp['sum_reward'], rel=1e-9)
    for env in envs:
        env.close()


def test_large_batch_fused_launches_use_their_own_shape_and_agree():
    """From 65 536 envs the fused launches (d2d_step_many / d2d_episode / d2d_rollout) run in 8-warp blocks while single steps run
    in 4-warp blocks with per-warp tickets: same results."""
    E, T = 70000, 2
    fused = make_vec(E, seed=41)
    single = make_vec(E, seed=41)
    out = fused.episode(T, record_actions=True)
    single.reset(mask=torch.ones(E, dtype=torch.uint8, device='cuda'))
    assert torch.equal(fused.positions, single.positions)
    for t in range(T + 1):
        if t == 0:
            single._bind(False)
        obs, reward, done, info = single.step(out['actions'][t], inputs_stable=(t > 0))
        single._bind(True)
        assert torch.equal(out['obs'][t], obs) and torch.equal(out['reward'][t], reward) and torch.equal(out['capacity_mbps'][t], info['capacity_mbps'])
    ro = fused.rollout(3, action_seed=5, first_step_index=7, record_actions=True)
    many = single.step_many(ro['actions'].contiguous())
    for k in ('obs', 'reward', 'done', 'capacity_mbps'):
        assert torch.equal(ro[k], many[k]), k
    assert fused.stats()['ticket_timeouts'] == 0 and single.stats()['ticket_timeouts'] == 0
    fused.close(); single.close()


# ---- dense kernel: bulk-copy staging of rows that do not start on 16-byte boundaries -------------------------------------------------------
@pytest.mark.parametrize('kw', [dict(num_rbs=5, num_cues=41, num_due_pairs=60),      # N = 101: action rows rotate through all four alignments, V = 162
                                dict(num_rbs=5, num_cues=40, num_due_pairs=61)])     # N = 101, V = 163: position rows alternate between 0 and 8
def test_dense_staging_of_unaligned_rows(monkeypatch, kw):
    """d2d_step_dense_kernel stages each env's action and position rows with one cp.async.bulk per row for the 16-byte aligned
    interior plus 4-byte cp.asyncs for the words on either side.  Rows of 101 actions / 163 positions start at every possible
    alignment; the action tensor is additionally a view that starts 4 bytes into its allocation and ends exactly at its end
    (nothing beyond the last row may be read: run under compute-sanitizer this is the out-of-bounds check).  Two blocks step
    all envs, so consecutive rows alternate inside one block."""
    from tests._util import RTOL, assert_rel
    monkeypatch.setenv('D2D_B200_GRID', '2')
    cfg = O.OracleConfig(**kw)
    E = 37
    rng = np.random.default_rng(2718)
    pos, act = O.random_positions(cfg, E, rng, fp32_exact=True), O.random_actions(cfg, E, rng)
    env = make_vec(E, kw)
    assert env.step_geometry()['block'] == 256 and env.step_geometry()['smem_bytes'] > 8000      # the dense kernel: bins + staged rows
    env.set_positions(pos)
    flat = torch.empty(E * cfg.num_links + 1, dtype=torch.int32, device='cuda')
    a = flat[1:].view(E, cfg.num_links)
    a.copy_(torch.as_tensor(act, dtype=torch.int32))
    assert a.data_ptr() % 16 == 4 and a.is_contiguous()
    obs, reward, done, info = env.step(a)
    torch.cuda.synchronize()
    ref = O.step_batch(cfg, pos, act, nthreads=4)
    assert_rel(obs[..., 4].cpu().numpy(), ref['sinr_db'], RTOL, 'sinr_db')
    assert_rel(obs[..., 5].cpu().numpy(), ref['snr_db'], RTOL, 'snr_db')
    assert_rel(info['capacity_mbps'].cpu().numpy(), ref['capacity_mbps'], RTOL, 'capacity')
    assert_rel(reward.cpu().numpy(), ref['reward'], RTOL, 'reward')
    np.testing.assert_array_equal(obs[..., :2].cpu().numpy().reshape(E, -1)[:, :2 * cfg.num_cues], pos[:, 1:1 + cfg.num_cues].astype(np.float32).reshape(E, -1))
    env.close()




# ---- late wait: a flagged step whose output buffers its predecessor does not touch stores them ahead of griddepcontrol.wait -----------------
@pytest.mark.parametrize('E,grid', [(4096, None), (1000, None), (148, None), (3000, '7'), (20000, None)])      # (late-wait steps run on 1 / 3 blocks per SM up to 8 288 / 24 568 envs)
def test_late_wait_bit_identical_to_serialised_launches(monkeypatch, E, grid):
    """d2d_step right behind a d2d_step of the same handle, D2D_STEP_INPUTS_STABLE, output buffers disjoint from the predecessor's:
    the per-link outputs go out before the wait, the step counters / reward / done after it (D2D_PF_LATE_WAIT).  Graph replays and
    eager chains over a ring of four output sets - also with the SAME set twice in a row, where the library must fall back to the
    early wait - broken by resets; every buffer of the ring, the counters and the done flags bit-identical to a library without
    programmatic dependent launch and to one with the late wait switched off."""
    if grid:
        monkeypatch.setenv('D2D_B200_GRID', grid)
    monkeypatch.setenv('D2D_B200_PDL', '0')
    plain = make_vec(E, seed=13)
    monkeypatch.delenv('D2D_B200_PDL')
    late = make_vec(E, seed=13)
    monkeypatch.setenv('D2D_B200_LATE_WAIT', '0')
    early = make_vec(E, seed=13)
    monkeypatch.delenv('D2D_B200_LATE_WAIT')
    envs = (plain, late, early)
    for env in envs:
        env.reset()
        env.reset_stats()
    acts = [late.sample_actions() for _ in range(4)]
    outs = {env: [env.alloc_outputs() for _ in range(4)] for env in envs}
    order = [0, 1, 2, 3, 3, 0, 1, 1, 2, 0, 3, 2]               # consecutive steps mostly on different sets, twice on the same one
    graphs = {env: env.capture_steps([acts[i] for i in order], [outs[env][i] for i in order], inputs_stable=True) for env in (late, early)}
    diff = torch.zeros((), dtype=torch.int64, device='cuda')

    def check():
        d = (plain.step_count != late.step_count).sum() + (plain.step_count != early.step_count).sum()
        for i in range(4):
            for name in ('obs', 'capacity_mbps', 'reward', 'done'):
                ref = getattr(outs[plain][i], name)
                d = d + (ref != getattr(outs[late][i], name)).sum() + (ref != getattr(outs[early][i], name)).sum()
        return d

    for it in range(2000 if E <= 4096 else 100):              # E = 4096: 24 000 late-wait steps in 2 000 graph replays
        for i in order:
            plain.step(acts[i], out=outs[plain][i])
        graphs[late].replay(); graphs[early].replay()
        if it % 15 == 0:
            diff += check()
        if it % 40 == 7:                                        # new episodes in between (counters back to 0, new positions)
            for env in envs:
                env.reset()
    mask = torch.ones(E, dtype=torch.uint8, device='cuda')
    for it in range(30):                                        # eager chains
        for env in envs:
            for k in range(9):
                env.step(acts[(it + k) % 4], out=outs[env][(it + k) % 4], inputs_stable=True)
            env.reset(mask=mask)
            env.step(acts[it % 4], out=outs[env][it % 4], inputs_stable=True)
            env.step(acts[(it + 1) % 4], out=outs[env][(it + 1) % 4], inputs_stable=True)
        diff += check() + (plain.positions != late.positions).sum()
    torch.cuda.synchronize()
    assert int(diff.item()) == 0
    sp, sl = plain.stats(), late.stats()
    assert sp['env_steps'] == sl['env_steps'] and sp['rescues'] == sl['rescues'] and sp['penalties'] == sl['penalties']
    # (per-warp fp32 partial sums over the envs a warp steps, then fp64 atomics: a late-wait step runs on fewer, fuller warps than the
    # serialised launch, so the partial sums group differently)
    assert sl['sum_reward'] == pytest.approx(sp['sum_reward'], rel=1e-7)
    for env in envs:
        env.close()


# ---- dense kernel: the instantiation for BASELINE config #3's shape == the generic one ----------------------------------------------------------
@pytest.mark.parametrize('info', [True, False])
def test_dense_spec_instantiation_equals_generic(monkeypatch, info):
    """100 RBs / 100 CUEs / 500 DUE pairs runs on d2d_step_dense_kernel<.., SPEC> (counts, strides and division magics as
    immediates); D2D_B200_SPEC=0 forces the generic instantiation.  Same results (to the last-ulp freedom of two block-kernel
    launches), both within tolerance of the oracle; crowded RBs, absent agents, several envs per block, two steps."""
    import gym_d2d_b200 as G
    from tests._util import RTOL, assert_rel
    kw = CONFIGS['dense']
    cfg = O.OracleConfig(**kw)
    E = 500
    rng = np.random.default_rng(99)
    pos, act = O.random_positions(cfg, E, rng), O.random_actions(cfg, E, rng)
    act[::7, ::3] = -1
    crowd = np.arange(E) % 40 == 3
    act[crowd] = act[crowd] % 21                                       # everybody on RB 0: the overflow list
    a = torch.as_tensor(act, dtype=torch.int32, device='cuda')
    monkeypatch.setenv('D2D_B200_GRID', '30')
    spec = G.VecD2DEnv(E, dict(kw), device='cuda', info=info)
    monkeypatch.setenv('D2D_B200_SPEC', '0')
    generic = G.VecD2DEnv(E, dict(kw), device='cuda', info=info)
    monkeypatch.delenv('D2D_B200_SPEC')
    outs = []
    for env in (spec, generic):
        env.set_positions(pos)
        for _ in range(2):
            obs, reward, done, inf = env.step(a)
        torch.cuda.synchronize()
        outs.append((obs.cpu().numpy(), reward.cpu().numpy(), inf['capacity_mbps'].cpu().numpy(), env.step_count.cpu().numpy()))
    np.testing.assert_allclose(outs[0][0], outs[1][0], rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(outs[0][2], outs[1][2], rtol=1e-5, atol=1e-6)
    np.testing.assert_array_equal(outs[0][3], outs[1][3])
    on = act >= 0
    ref = O.step_batch(cfg, pos, np.where(on, act, 0), active=on.astype(np.uint8), nthreads=4)
    for got in outs:
        assert_rel(got[0][..., 4][on], ref['sinr_db'][on], RTOL, 'sinr_db')
        assert_rel(got[0][..., 5][on], ref['snr_db'][on], RTOL, 'snr_db')
        assert_rel(got[2][on], ref['capacity_mbps'][on], RTOL, 'capacity')
        assert_rel(got[1], ref['reward'], RTOL, 'reward')
    spec.close(); generic.close()


# ---- dict API: cached index tables per set of present agents ----------------------------------------------------------------
def test_dict_api_changing_agent_sets_match_tensor_api():
    """D2DEnv caches its index tables (rows, per-agent observation order, id pairs) per ORDERED set of present agents and builds all
    observations with one gather (envs/obs_fn.py:43-53, envs/d2d_env.py:62-71, 103-116).  Steps with all agents, a shuffled subset, a
    different subset and all agents again (reversed) must each equal the tensor API's step on the same positions and actions -
    row for row, in the caller's key order - and `state` / `actions` must follow the last step only."""
    import gym_d2d_b200 as G
    rng = np.random.default_rng(5)
    vec = make_vec(1, seed=0, exact_positions=True)
    env = G.D2DEnv({}, seed=11)
    env.reset()
    vec.set_positions(env.vec.positions_f64)
    keys_all = list(env.link_keys)
    N = len(keys_all)
    index = {k: i for i, k in enumerate(keys_all)}
    orders = [list(range(N)), list(rng.permutation(N)[:17]), list(rng.permutation(N)[:30]), list(range(N))[::-1], list(rng.permutation(N)[:17])]
    orders.append(orders[1])                                   # a set seen before: served from the cache
    for order in orders:
        keys = [keys_all[i] for i in order]
        acts_row = np.full((1, N), -1, np.int32)
        raw = {}
        for k in keys:
            a = int(rng.integers(0, env.vec.action_nvec[index[k]]))
            raw[k] = a
            acts_row[0, index[k]] = a
        obs, rewards, done, info = env.step(raw)
        t_obs, t_rew, _t_done, t_info = vec.step(torch.as_tensor(acts_row, device='cuda'))
        table = t_obs[0].cpu().numpy().astype(np.float64)
        assert list(obs) == keys and list(info) == keys and list(rewards) == keys
        for pos, k in enumerate(keys):
            rows = [order[pos]] + [j for q, j in enumerate(order) if q != pos]
            np.testing.assert_array_equal(obs[k], table[rows].reshape(-1))
            j = index[k]
            assert info[k]['sinr_db'] == float(table[j, 4]) and info[k]['snr_db'] == float(table[j, 5])
            assert info[k]['capacity_mbps'] == float(t_info['capacity_mbps'][0, j]) and info[k]['rate_bps'] == float(t_info['rate_bps'][0, j])
            assert info[k]['rb'] == int(t_info['rb'][0, j]) and info[k]['tx_pwr_dbm'] == int(t_info['tx_pwr_dbm'][0, j])
            assert rewards[k] == float(t_rew[0])
            assert env.actions[k] == (info[k]['rb'], info[k]['tx_pwr_dbm'])
        assert list(env.state['sinrs_db']) == [tuple(k.split(':')) for k in keys]
    env.close(); vec.close()


# ---- host steps with int16 actions (D2D_STEP_ACTIONS_I16): half the upload, same results --------------------------------------
@pytest.mark.parametrize('E', [1, 333, 4096])
def test_host_steps_with_int16_actions_match_int32(E):
    """d2d_step_host_async with D2D_STEP_ACTIONS_I16: the int16 [E][N] actions are widened on the device (sign-extended: < 0 stays
    'agent absent', envs/d2d_env.py:36-40 spaces fit 15 bits) - every output bit-identical to the int32 upload, through the packed
    pinned slot buffers and through caller-owned arrays, with several steps in flight."""
    rng = np.random.default_rng(E)
    env = make_vec(E, seed=5)
    env.reset()
    N = env.num_links
    acts = [rng.integers(0, 500, size=(E, N), dtype=np.int32) for _ in range(6)]
    for a in acts:
        a[rng.random(a.shape) < 0.1] = -1                      # absent agents
    names = ('obs_dyn', 'capacity_mbps', 'reward', 'done')
    ref = []
    slots = [env.host_slot_buffers(k) for k in range(4)]
    env.step_count.zero_()
    for i, a in enumerate(acts):                                # int32, one step at a time
        slots[0]['actions'][:] = a
        env.step_host_async(slots[0]['actions'], slots[0], 0)
        env.step_host_wait(0)
        ref.append({k: slots[0][k].copy() for k in names})
    env.step_count.zero_()
    got = [None] * len(acts)
    for i, a in enumerate(acts):                                # int16 through the slots' own pinned bytes, four steps in flight
        k = i % 4
        if i >= 4:
            env.step_host_wait(k)
            got[i - 4] = {n: slots[k][n].copy() for n in names}
        slots[k]['actions16'][:] = a.astype(np.int16)
        env.step_host_async(slots[k]['actions16'], slots[k], k)
    for i in range(max(0, len(acts) - 4), len(acts)):
        env.step_host_wait(i % 4)
        got[i] = {n: slots[i % 4][n].copy() for n in names}
    for r, g in zip(ref, got):
        for n in names:
            np.testing.assert_array_equal(r[n], g[n])
    env.step_count.zero_()
    out = env.alloc_host_outputs(pinned=True, info=False, dyn=True)      # caller-owned arrays (per-buffer staging)
    a16 = np.ascontiguousarray(acts[0].astype(np.int16))
    env.step_host_async(a16, out, 1)
    env.step_host_wait(1)
    for n in names:
        np.testing.assert_array_equal(ref[0][n], out[n])
    # the flag belongs to the host entry points: d2d_step (device pointers) refuses it
    import ctypes as C
    from gym_d2d_b200 import _lib
    dev_a = env.sample_actions()
    io = _lib.D2DStepIO(actions=dev_a.data_ptr(), obs=env.alloc_outputs().obs.data_ptr(), flags=_lib.STEP_ACTIONS_I16)
    assert env._lib.d2d_step(env._h, C.byref(io), None) == _lib.ERR_INVALID_ARG
    env.close()
