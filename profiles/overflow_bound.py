"""What RBs holding more than D2D_BIN_CAP links cost the headline step chain: `python profiles/overflow_bound.py [E] [rounds]`.

Builds the bench.py headline setup (VecD2DEnv(E, {}), a ring of 32 action / output sets, one CUDA graph of the 32 steps
captured with inputs_stable=True, replays timed with CUDA events behind torch.cuda._sleep) for three action rings and times
them in the same process, alternated over the rounds:
  raw           env.sample_actions(), as bench.py draws them
  no_overflow   the same sets, except that every env with an RB above 8 links has its actions redrawn from the same uniform
                distribution until no RB holds more than 8 (about 0.4 % of the envs)
  one_rb        every link of every env on RB 0 (uniform power levels): the worst case of the overflow path
The gap between raw and no_overflow bounds what any change to the overflow path can gain at the default load.
Prints one line per round and arm, then the median and range per arm, with the card name and power limit read in this run.
"""
import subprocess
import sys
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import torch  # noqa: E402

import gym_d2d_b200 as G  # noqa: E402

E = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
ROUNDS = int(sys.argv[2]) if len(sys.argv) > 2 else 9
RING, REPLAYS, CAP = 32, 64, 8


def card() -> str:
    try:
        return subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as exc:  # noqa: BLE001
        return f'{torch.cuda.get_device_name()} (nvidia-smi: {exc})'


env = G.VecD2DEnv(E, {}, device='cuda', seed=0)
env.reset()
C, R = env.config.num_cues, env.config.num_rbs
npw = np.array([env.num_pwr_actions['cue']] * C + [env.num_pwr_actions['due']] * env.config.num_due_pairs)


def max_load(a: np.ndarray) -> np.ndarray:
    """Per env: the most links any one RB holds (rb = a // n_pwr, envs/d2d_env.py:95)."""
    rb = a // npw
    return np.stack([(rb == r).sum(1) for r in range(R)], 1).max(1)


gen = torch.Generator(device=env.device)
gen.manual_seed(1000)                      # bench.py's generator seed (rank 0)
raw = [env.sample_actions(gen) for _ in range(RING)]
rng = np.random.default_rng(7)
fixed, n_redrawn = [], 0
for a in raw:
    h = a.cpu().numpy().copy()
    over = np.flatnonzero(max_load(h) > CAP)
    n_redrawn += over.size
    for i in over:
        while max_load(h[i:i + 1])[0] > CAP:
            h[i] = np.minimum((rng.random(h.shape[1]) * (R * npw)).astype(np.int32), R * npw - 1)
    fixed.append(torch.from_numpy(h).to(env.device))
one_rb = [torch.from_numpy((rng.random((E, npw.size)) * npw).astype(np.int32)).to(env.device) for _ in range(RING)]
outs = [env.alloc_outputs() for _ in range(RING)]
print(f'E={E}: {n_redrawn / (RING * E):.2%} of the env-steps redrawn for no_overflow; '
      f'raw env-steps with an RB above {CAP}: {np.mean([(max_load(a.cpu().numpy()) > CAP).mean() for a in raw]):.2%}')

graphs = {}
for name, acts in (('raw', raw), ('no_overflow', fixed), ('one_rb', one_rb)):
    for a, o in zip(acts, outs):
        env.step(a, out=o, inputs_stable=True)
    graphs[name] = env.capture_steps(acts, outs, inputs_stable=True)
    graphs[name].replay()
torch.cuda.synchronize()
print(f'geometry {env.step_geometry()}; card: {card()}')

res = {k: [] for k in graphs}
for rnd in range(ROUNDS):
    for name in (graphs if rnd % 2 == 0 else list(graphs)[::-1]):
        g = graphs[name]
        g.replay()                              # warm: the previous arm left other outputs in L2
        torch.cuda.synchronize()
        s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda._sleep(600_000)              # the device is busy while the host enqueues the timed replays
        s.record()
        for _ in range(REPLAYS):
            g.replay()
        t.record()
        torch.cuda.synchronize()
        us = s.elapsed_time(t) * 1e3 / (REPLAYS * RING)
        res[name].append(us)
        print(f'round {rnd}: {name:12s} {us:6.3f} us/step')
print(f'card: {card()}')
med = {k: float(np.median(v)) for k, v in res.items()}
for k, v in res.items():
    print(f'{k:12s} median {med[k]:6.3f} us/step  range {min(v):6.3f} .. {max(v):6.3f}  ({len(v)} rounds of {REPLAYS * RING} steps)')
print(f'no_overflow vs raw: {100 * (1 - med["no_overflow"] / med["raw"]):+.1f} % (positive = no_overflow faster)')
