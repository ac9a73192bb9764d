"""Per-warp timeline of back-to-back step launches: `D2D_B200_LIB=.../_variants/timeline.so python profiles/timeline.py [E]`.

Needs the instrumented build (`nvcc ... -DD2D_TIMELINE`, see profiles/README.md): every warp of d2d_step_warp_kernel stamps
globaltimer + clock64 at entry, clock64 before / after griddepcontrol.wait and at its end, and its SM id.  The script replays
a CUDA graph of 32 step launches (the bench's launch mode), reads the stamps of the last replay and prints, per launch, when
its warps started / reached the wait / were released / ended - relative to the previous launch - i.e. how much of a step
overlaps its predecessor under programmatic dependent launch.  Every warp also counts the envs it stepped, the flagged links it
recomputed in fp64 before / after its wait and the envs that took the overflow pass (an RB above D2D_BIN_CAP links); the script
prints them for the last warp to reach the wait and the last to end, splits the post-wait time by whether a warp ran an fp64 pass
after its wait, and the entry -> wait time by whether it stepped an overflow env.
Numbers from an instrumented build are not bench values.
"""
import ctypes
import sys
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import torch  # noqa: E402

import gym_d2d_b200 as G  # noqa: E402
from gym_d2d_b200 import _lib  # noqa: E402

E = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
SLOTS, WARPS, RING = 64, 4096, 32
env = G.VecD2DEnv(E, {}, device='cuda', seed=0)
env.reset()
acts = [env.sample_actions() for _ in range(RING)]
outs = [env.alloc_outputs() for _ in range(RING)]
lib = _lib.load()
if not hasattr(lib, 'd2d_debug_timeline'):
    raise SystemExit('not an instrumented build: set D2D_B200_LIB to a -DD2D_TIMELINE build of libd2d_b200')
lib.d2d_debug_timeline.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int]
for a, o in zip(acts, outs):
    env.step(a, out=o, inputs_stable=True)
first_slot = env.launch_count % SLOTS          # the graph's nodes keep the slots they were captured with
g = env.capture_steps(acts, outs, inputs_stable=True)      # the bench's launch mode: flagged steps over a ring of output sets
for _ in range(5):
    g.replay()
torch.cuda.synchronize()
s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
s.record()
for _ in range(20):
    g.replay()
t.record()
torch.cuda.synchronize()
print(f'E={E}: {s.elapsed_time(t) * 1e3 / (20 * RING):.2f} us/step (instrumented build)  geom={env.step_geometry()}')

buf = np.zeros((SLOTS, WARPS, 10), dtype=np.uint64)
geom = env.step_geometry()
rc = lib.d2d_debug_timeline(buf.ctypes.data_as(ctypes.c_void_p), buf.nbytes, geom['block'] // 32)      # (one stamp table per warps-per-block shape)
assert rc == 0
nw = min(WARPS, geom['grid'] * geom['block'] // 32)
order = [(first_slot + k) % SLOTS for k in range(RING)]
# a late-wait step runs on fewer blocks than step_geometry reports, and the table keeps older launches' stamps: count the warps of the
# last launch that stamped during the last replay (within 1 ms of the replay's first stamp)
t_cut = int(buf[order[0], 0, 0]) - 1_000_000
nw = int((buf[order[-1], :nw, 0].astype(np.int64) >= t_cut).sum()) or nw
rec = buf[order, :nw].astype(np.int64)              # [launch][warp][g0, c0, c1, c2, c3, smid, n_env, n_pre, n_post, n_ovf]
g0, c0, c1, c2, c3, smid, n_env, n_pre, n_post, n_ovf = (rec[..., i] for i in range(10))
# clock64 is per SM: bring every SM onto the globaltimer axis with one offset per SM (SM clock = 1.965 GHz under load)
GHZ = 1.965
off = np.zeros(256)
for sm in np.unique(smid):
    m = smid == sm
    off[sm] = np.median(g0[m] - c0[m] / GHZ)
to_ns = lambda c: c / GHZ + off[smid]
t0, t1, t2, t3 = to_ns(c0), to_ns(c1), to_ns(c2), to_ns(c3)
print(f'globaltimer granularity ~ {np.min(np.diff(np.unique(g0))):d} ns; SM-offset residual (p95 |g0 - t0|): {np.percentile(np.abs(g0 - t0), 95):.0f} ns')
base = t0[1].min()
print('launch | first start  last start | first at wait  last at wait | first release  last release | first end  last end | '
      'period | pre-wait work (median)  waiting (median)  post-wait (median)   [us, relative to launch 1]')
prev_end = None
for k in range(1, RING):
    f = lambda x: (x.min() - base) / 1e3
    l = lambda x: (x.max() - base) / 1e3
    period = (t3[k].max() - t3[k - 1].max()) / 1e3
    print(f'{k:6d} | {f(t0[k]):8.2f} {l(t0[k]):8.2f} | {f(t1[k]):8.2f} {l(t1[k]):8.2f} | {f(t2[k]):8.2f} {l(t2[k]):8.2f} | '
          f'{f(t3[k]):8.2f} {l(t3[k]):8.2f} | {period:5.2f} | {np.median(t1[k] - t0[k]) / 1e3:5.2f} {np.median(t2[k] - t1[k]) / 1e3:5.2f} '
          f'{np.median(t3[k] - t2[k]) / 1e3:5.2f}')
k = slice(4, RING)
print('means over launches 4..31 [us]:')
print(f'  period (last end -> last end)            {np.mean((t3[k].max(1)[1:] - t3[k].max(1)[:-1])) / 1e3:6.2f}')
print(f'  prev last end -> this first release      {np.mean(t2[5:].min(1) - t3[4:-1].max(1)) / 1e3:6.2f}')
print(f'  prev last end -> this last release       {np.mean(t2[5:].max(1) - t3[4:-1].max(1)) / 1e3:6.2f}')
print(f'  first release -> last end (post-wait)    {np.mean(t3[k].max(1) - t2[k].min(1)) / 1e3:6.2f}')
print(f'  first start -> last start (block launch) {np.mean(t0[k].max(1) - t0[k].min(1)) / 1e3:6.2f}')
print(f'  this first start - prev first start      {np.mean(t0[5:].min(1) - t0[4:-1].min(1)) / 1e3:6.2f}')
print(f'  this first start - prev last end         {np.mean(t0[5:].min(1) - t3[4:-1].max(1)) / 1e3:6.2f}  (negative = overlap)')
print(f'  warps already at the wait when prev ends {np.mean([(t1[j] < t3[j - 1].max()).mean() for j in range(5, RING)]):6.2%}')
print(f'  per-warp: start->wait {np.median(t1[k] - t0[k]) / 1e3:5.2f}  waiting {np.median(t2[k] - t1[k]) / 1e3:5.2f}  release->end {np.median(t3[k] - t2[k]) / 1e3:5.2f}')
print(f'  last release -> last end                 {np.mean(t3[k].max(1) - t2[k].max(1)) / 1e3:6.2f}')

# what the stragglers did: (envs, fp64 links before the wait, fp64 links after it, overflow envs) of the last warp at the wait and
# of the last warp to end; post-wait time (release -> end) of the warps with and without an fp64 pass after their wait
print('launch | last at wait: env pre post ovf | last to end: env pre post ovf | release->end [us] median / max: post-wait pass (n) | none (n)')
attr = lambda k, w: f'{n_env[k, w]:3d} {n_pre[k, w]:3d} {n_post[k, w]:4d} {n_ovf[k, w]:3d}'
for k in range(1, RING):
    wa, we = int(t1[k].argmax()), int(t3[k].argmax())
    post, m = (t3[k] - t2[k]) / 1e3, n_post[k] > 0
    split = lambda x: f'{np.median(x):5.2f} / {x.max():5.2f} ({len(x):4d})' if len(x) else '    -         (   0)'
    print(f'{k:6d} |             {attr(k, wa)} |            {attr(k, we)} | {split(post[m])} | {split(post[~m])}')
k = slice(4, RING)
post, m = (t3[k] - t2[k]) / 1e3, n_post[k] > 0
print(f'launches 4..31: warps with an fp64 pass after the wait {m.mean():.2%} (links before / after the wait per launch: '
      f'{n_pre[k].sum(1).mean():.1f} / {n_post[k].sum(1).mean():.1f}; overflow envs per launch {n_ovf[k].sum(1).mean():.1f})')
print(f'  last warp to end ran a post-wait pass in {np.mean([n_post[j, t3[j].argmax()] > 0 for j in range(4, RING)]):.0%} of launches, '
      f'an overflow env in {np.mean([n_ovf[j, t3[j].argmax()] > 0 for j in range(4, RING)]):.0%}; '
      f'last warp at the wait: overflow env in {np.mean([n_ovf[j, t1[j].argmax()] > 0 for j in range(4, RING)]):.0%}')
if m.any():
    print(f'  release->end with a post-wait pass: median {np.median(post[m]):.2f} us, without: {np.median(post[~m]):.2f} us')
# entry -> wait of the warps that stepped an env with an RB above D2D_BIN_CAP links, against the others
pre, o = (t1[k] - t0[k]) / 1e3, n_ovf[k] > 0
split = lambda x: f'median {np.median(x):5.2f} us  max {x.max():5.2f} us ({x.size} warps)' if x.size else '-'
print(f'  entry->wait with an overflow env: {split(pre[o])}; without: {split(pre[~o])}')
wa = [int(t1[j].argmax()) for j in range(4, RING)]
print(f'  last warp at the wait, launches 4..31: envs {np.mean([n_env[j, w] for j, w in zip(range(4, RING), wa)]):.1f}, '
      f'fp64 links before / after the wait {np.mean([n_pre[j, w] for j, w in zip(range(4, RING), wa)]):.2f} / '
      f'{np.mean([n_post[j, w] for j, w in zip(range(4, RING), wa)]):.2f}, '
      f'overflow env in {np.mean([n_ovf[j, w] > 0 for j, w in zip(range(4, RING), wa)]):.0%}')
np.save(Path(__file__).resolve().parent.parent / 'gpurun_out' / f'timeline_E{E}.npy', rec)
