"""Auto-reset steps against the reset paths they replace: `python profiles/time_autoreset.py [E ...]` (default 4096 131072).

Per batch size, time per COUNTED step of the whole batch (10 per episode) of
  (a) autoreset  - VecD2DEnv(autoreset=True): 11 auto-reset steps per episode (one of them resets every env), actions pre-generated
  (b) reset+10   - reset() (d2d_reset, a torch sampling kernel, the uncounted step) + 10 flagged steps (inputs_stable=True)
  (c) episode    - d2d_episode with actions drawn on the device (one launch per episode), for reference
and a policy loop: us per {two torch kernels that rewrite the actions; step} pair, the step an auto-reset step or today's
default-ordering step (profiles/time_policy_loop.py).  Every arm is a CUDA graph of several episodes (32 pairs for the loop), timed
with CUDA events; the arms alternate, ROUNDS times each, and the median is printed with the spread.  The card's name and power
limit are printed with the numbers.
"""
import statistics
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import torch  # noqa: E402

import gym_d2d_b200 as G  # noqa: E402

EPISODES = 4          # per graph
REPLAYS = 10          # per timed window
ROUNDS = 7


def card():
    try:
        pl = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', str(torch.cuda.current_device())],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:            # the name is still printed; the limit is then unknown
        pl = 'unknown'
    return f'{torch.cuda.get_device_name()}, power limit {pl or "unknown"}'


def capture(fn):
    for _ in range(2):           # warm every shape the graph uses
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    return g


def time_graph(g):
    s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(REPLAYS):
        g.replay()
    t.record()
    torch.cuda.synchronize()
    return s.elapsed_time(t) * 1e3 / REPLAYS        # us per replay


def run(E):
    ar = G.VecD2DEnv(E, {}, device='cuda', seed=0, autoreset=True)
    ar.reset()
    ar.step_count.fill_(10)                         # the graph's first step resets every env: 11 steps = one episode
    plain = G.VecD2DEnv(E, {}, device='cuda', seed=0)
    plain.reset()
    acts = ar.sample_actions()
    outs_ar, outs_pl = [ar.alloc_outputs() for _ in range(2)], [plain.alloc_outputs() for _ in range(2)]
    ep_out = plain.alloc_many_outputs(11)

    def arm_a():
        for i in range(11 * EPISODES):
            ar.step(acts, out=outs_ar[i % 2])

    def arm_b():
        for _ in range(EPISODES):
            plain.reset()
            for i in range(10):
                plain.step(acts, out=outs_pl[i % 2], inputs_stable=True)

    def arm_c():
        for _ in range(EPISODES):
            plain.episode(10, out=ep_out)

    nvec = ar._nvec_dev.to(torch.int32)
    pacts = acts.clone()

    def loop(env, outs):
        def fn():
            for i in range(32):
                pacts.add_(1).remainder_(nvec)      # the "policy": two small torch kernels that rewrite the actions
                env.step(pacts, out=outs[i % 2])
        return fn

    graphs = {'autoreset': capture(arm_a), 'reset+10': capture(arm_b), 'episode': capture(arm_c),
              'loop_autoreset': capture(loop(ar, outs_ar)), 'loop_plain': capture(loop(plain, outs_pl))}
    per = {'autoreset': 10 * EPISODES, 'reset+10': 10 * EPISODES, 'episode': 10 * EPISODES, 'loop_autoreset': 32, 'loop_plain': 32}
    res = {k: [] for k in graphs}
    for _ in range(ROUNDS):
        for k, g in graphs.items():
            res[k].append(time_graph(g) / per[k])
    for k, v in res.items():
        unit = 'us per counted step' if not k.startswith('loop') else 'us per {policy, step} pair'
        print(f'E={E:>6} {k:>15}: {statistics.median(v):8.2f} {unit}  (min {min(v):.2f}, max {max(v):.2f}; '
              f'{statistics.median(v) * 1e3 / E:.3f} ns per env-step)', flush=True)
    for env in (ar, plain):
        env.close()


if __name__ == '__main__':
    assert torch.cuda.is_available(), 'time_autoreset.py measures on the GPU'
    print(card(), flush=True)
    for E in [int(x) for x in sys.argv[1:]] or [4096, 131072]:
        run(E)
