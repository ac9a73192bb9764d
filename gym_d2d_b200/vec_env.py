"""VecD2DEnv: the batched tensor API over libd2d_b200.so.

E independent default-topology D2D environments live on one GPU (positions, step counters and statistics
resident in HBM as PyTorch tensors); `step(actions)` is ONE fused kernel launch that replaces, for every
env, the reference's D2DEnv.step -> Simulator.step -> LinearObsFunction -> SystemCapacityRewardFunction
chain (envs/d2d_env.py:62-71).  PyTorch is used for device memory, streams and torch.distributed only.
"""
from __future__ import annotations

import ctypes as C
from typing import Any, Dict, Optional, Tuple

import numpy as np
import torch

from . import _lib
from .config import EPISODE_LENGTH, EnvConfig, link_table, to_c_config
from .plugins import (LinearObsFunction, SystemCapacityRewardFunction, resolve_obs_fn, resolve_reward_fn)


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


_M64 = 0xFFFFFFFFFFFFFFFF


def autoreset_key(base: int, n: int) -> int:
    """Philox key of an env's n-th auto-reset under key base `base`: splitmix64(base + n * 0x9E3779B97F4A7C15), the library's
    d2d_autoreset_key (gym_d2d_b200/csrc/d2d_common.cuh)."""
    z = (int(base) + int(n) * 0x9E3779B97F4A7C15) & _M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _M64
    return z ^ (z >> 31)


class StepBuffers:
    """One set of device output tensors of a step (the tensors a d2d_step_io_t points at)."""

    def __init__(self, num_envs: int, num_links: int, device: torch.device, info: bool, agent_reward: bool = False) -> None:
        E, N = num_envs, num_links
        self.agent_reward = torch.zeros((E, N), dtype=torch.float32, device=device) if agent_reward else None
        self.obs = torch.zeros((E, N, 6), dtype=torch.float32, device=device)
        self.capacity_mbps = torch.zeros((E, N), dtype=torch.float32, device=device)
        self.reward = torch.zeros((E,), dtype=torch.float32, device=device)
        self.done = torch.zeros((E,), dtype=torch.uint8, device=device)
        self.rate_bps = torch.zeros((E, N), dtype=torch.float32, device=device) if info else None
        self.rb = torch.zeros((E, N), dtype=torch.int16, device=device) if info else None
        self.tx_pwr_dbm = torch.zeros((E, N), dtype=torch.int16, device=device) if info else None
        # the step descriptor of this set, built once (the tensors above are never reallocated): a step fills in its actions and
        # flags only - ten data_ptr() calls per eager step were a quarter of the host's time per launch
        self._io = _lib.D2DStepIO(obs=self.obs.data_ptr(), capacity_mbps=self.capacity_mbps.data_ptr(), reward=self.reward.data_ptr(),
                                  done=self.done.data_ptr(), rate_bps=_ptr(self.rate_bps), rb=_ptr(self.rb),
                                  tx_pwr_dBm=_ptr(self.tx_pwr_dbm), agent_reward=_ptr(self.agent_reward))

    def nbytes(self) -> int:
        return sum(t.numel() * t.element_size() for t in vars(self).values() if isinstance(t, torch.Tensor))


class VecD2DEnv:
    """Batched GymD2D step path on one B200.

    Parameters
    ----------
    num_envs : number of environments resident on this device (this rank's slice for multi-GPU runs).
    env_config : the reference's env_config dict (same keys/defaults as EnvConfig, plus 'obs_fn' and
        'reward_fn' plugin classes).  Like the reference ctor (envs/d2d_env.py:27-28) the two plugin keys
        are popped from the caller's dict.
    device : CUDA device.
    seed, global_env_offset : Philox key and the global index of local env 0; a sharded batch draws the
        same scenario for a given global env whatever the number of GPUs.
    info : also return rate_bps / rb / tx_pwr_dbm tensors (the reference's info dict, envs/d2d_env.py:106-116).
    downlink : also carry one DOWNLINK link 'mbs:cueXX' per CUE after the canonical links (N = 2C + D; absent unless an
        action >= 0 is given).  Such envs run on the general-topology kernel.
    exact_positions : keep a float64 shadow of positions given through set_positions().  The hot path still
        reads the fp32 state; the shadow is read only by the kernels' rare fp64 recomputation path, so that
        results stay within 1e-4 relative of the reference evaluated on the caller's UNROUNDED float64
        positions (device-config files).  Not needed for positions drawn on the device by reset().
    autoreset : next-step auto-reset (Gymnasium's AutoresetMode.NEXT_STEP) in step() and capture_steps().  An env whose previous
        step returned done = 1 is reset by the next step instead of stepped: its actions in that call are ignored, and its row
        of the results is the first observation of the new episode (new positions, the reset step's obs / capacity / info,
        reward = 0, done = 0, step counter 0).  The reset draws positions and actions on the device under
        autoreset_key(n), n = the env's entry of `episode_index` after the step.  Only configurations served by the warp
        kernel (<= 32 CUEs, <= 32 DUE pairs, <= 64 RBs, no downlinks, no ShadowingPathLoss) support it; others raise here.
    """

    def __init__(self, num_envs: int, env_config: Optional[dict] = None, device: Any = 'cuda', seed: int = 0,
                 global_env_offset: int = 0, info: bool = False, exact_positions: bool = False, downlink: bool = False,
                 autoreset: bool = False) -> None:
        env_config = env_config if env_config is not None else {}
        obs_enum = resolve_obs_fn(env_config.pop('obs_fn', LinearObsFunction))
        reward_enum, min_cap = resolve_reward_fn(env_config.pop('reward_fn', SystemCapacityRewardFunction))
        self.per_agent_reward = reward_enum != _lib.REWARD_SYSTEM_CAPACITY   # envs/reward_fn.py:47-78 reward every agent separately
        self.config = EnvConfig(**env_config)          # unknown key -> TypeError, like the reference dataclass
        self.config.downlinks = bool(downlink)         # also carry the 'mbs:cueXX' DOWNLINK links (envs/d2d_env.py:87-89)
        self.num_envs = int(num_envs)
        if self.num_envs < 1:
            raise ValueError('num_envs must be >= 1')
        self.device = torch.device(device)
        if self.device.type != 'cuda':
            raise _lib.D2DError('gym_d2d_b200 runs on CUDA (sm_100a) only; there is no CPU path')
        if self.device.index is None:
            self.device = torch.device('cuda', torch.cuda.current_device())
        self.seed = int(seed)
        self.global_env_offset = int(global_env_offset)
        self.num_links = self.config.num_links
        self.num_devices = self.config.num_devices
        self.link_keys = self.config.link_keys()
        self.num_pwr_actions = self.config.num_pwr_actions
        npw = self.num_pwr_actions
        # envs/d2d_env.py:36-40: Discrete(num_rbs * n_pwr) per transmitter type
        self.action_nvec = np.array([self.config.num_rbs * npw['cue']] * self.config.num_cues
                                    + [self.config.num_rbs * npw['due']] * self.config.num_due_pairs
                                    + [self.config.num_rbs * npw['mbs']] * (self.config.num_cues if downlink else 0), np.int64)
        self.episode_length = EPISODE_LENGTH
        self.want_info = bool(info)
        self._episode = 0

        self._lib = _lib.load()
        links = link_table(self.config)
        c_links = (_lib.D2DLink * len(links))(*[_lib.D2DLink(**row) for row in links])
        c_cfg = to_c_config(self.config, self.num_envs, self.device.index, obs_enum, reward_enum, min_cap,
                            rng_seed=self.seed, first_global_env=self.global_env_offset)
        handle = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self._lib.d2d_create(C.byref(c_cfg), c_links, C.byref(handle)))
        self._h = handle

        E, N, V = self.num_envs, self.num_links, self.num_devices
        dev = self.device
        self.positions = torch.zeros((E, V, 2), dtype=torch.float32, device=dev)
        self.step_count = torch.zeros((E,), dtype=torch.uint8, device=dev)
        self._stats = torch.zeros((_lib.STATS_REPLICAS, _lib.NUM_STATS), dtype=torch.float64, device=dev)
        self._bind(True)
        self.positions_f64 = torch.zeros((E, V, 2), dtype=torch.float64, device=dev) if exact_positions else None
        if exact_positions:
            _lib.check(self._lib.d2d_bind_positions_f64(self._h, self.positions_f64.data_ptr()))
        # auto-reset: episodes each env has begun since the last full reset() (int32, read as uint32 by the library)
        self.autoreset = bool(autoreset)
        self.episode_index = torch.zeros((E,), dtype=torch.int32, device=dev) if self.autoreset else None
        self._ar_base = autoreset_key(self.seed, 0)      # until the first full reset() (see reset)
        if self.autoreset:
            self._bind_autoreset()
        # default output buffers, reused by every step (clone what you keep, or pass out=alloc_outputs())
        self._out = self.alloc_outputs()
        self.obs, self.capacity_mbps, self.reward, self.done = (self._out.obs, self._out.capacity_mbps,
                                                                self._out.reward, self._out.done)
        self.rate_bps, self.rb, self.tx_pwr_dbm = self._out.rate_bps, self._out.rb, self._out.tx_pwr_dbm
        self._host_io_cache: Dict[tuple, tuple] = {}
        self._nvec_dev = torch.as_tensor(self.action_nvec, device=dev)
        self._nvec_f = self._nvec_dev.to(torch.float32)
        self._nvec_m1 = (self._nvec_dev - 1).to(torch.int32)

    # ---- plumbing -----------------------------------------------------------------------------
    def _bind(self, counted: bool) -> None:
        _lib.check(self._lib.d2d_bind_state(self._h, self.positions.data_ptr(),
                                            self.step_count.data_ptr() if counted else None,
                                            self._stats.data_ptr() if counted else None))

    def _bind_autoreset(self) -> None:
        _lib.check(self._lib.d2d_bind_autoreset(self._h, self.episode_index.data_ptr(), self._ar_base))

    def autoreset_key(self, n: int) -> int:
        """Philox key of an env's n-th auto-reset since the last full reset() (the key d2d_reset / d2d_sample_actions would
        take to draw the same positions and reset actions)."""
        return autoreset_key(self._ar_base, n)

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def alloc_outputs(self) -> StepBuffers:
        """A fresh set of output tensors to pass as step(..., out=...), e.g. one per in-flight step."""
        return StepBuffers(self.num_envs, self.num_links, self.device, self.want_info, self.per_agent_reward)

    def close(self) -> None:
        if getattr(self, '_h', None):
            self._lib.d2d_destroy(self._h)
            self._h = None
            self._host_io_cache.clear()

    def __del__(self) -> None:
        try:
            self.close()
        except Exception:
            pass

    # ---- state --------------------------------------------------------------------------------
    def set_positions(self, positions, first_env: int = 0) -> None:
        """Upload float64 positions [count][V][2] (device order mbs, cues, due tx/rx ...).  Replaces
        Device.set_position (device.py:82-83); device 0 is pinned to the origin (simulator.py:63-64)."""
        if isinstance(positions, torch.Tensor) and positions.is_cuda:
            src = positions.to(torch.float64).contiguous()
            on_dev = 1
            ptr = src.data_ptr()
        else:
            src = np.ascontiguousarray(np.asarray(positions.cpu() if isinstance(positions, torch.Tensor) else positions,
                                                  dtype=np.float64))
            on_dev = 0
            ptr = src.ctypes.data
        if src.ndim != 3 or tuple(src.shape[1:]) != (self.num_devices, 2):
            raise ValueError(f'positions must be [count][{self.num_devices}][2], got {tuple(src.shape)}')
        _lib.check(self._lib.d2d_set_positions(self._h, ptr, on_dev, int(first_env), int(src.shape[0]), self._stream()))

    def get_positions(self, host: bool = True):
        """The bound float32 positions [E][V][2] (d2d_get_positions): a fresh device tensor, or a host ndarray.  With the
        `obs_dyn` output this is the once-per-reset half of the observation table (see obs_static / assemble_obs)."""
        E, V = self.num_envs, self.num_devices
        if host:
            dst = np.empty((E, V, 2), np.float32)
            _lib.check(self._lib.d2d_get_positions(self._h, dst.ctypes.data, 0, 0, E, self._stream()))
            return dst
        dst = torch.empty((E, V, 2), dtype=torch.float32, device=self.device)
        _lib.check(self._lib.d2d_get_positions(self._h, dst.data_ptr(), 1, 0, E, self._stream()))
        return dst

    def obs_static(self, positions=None) -> np.ndarray:
        """Columns 0-3 of the observation table, float32 [E][N][4] = (tx_x, tx_y, rx_x, rx_y) per link (envs/obs_fn.py:55-61),
        from a host copy of the positions: they change only on reset() / set_positions()."""
        pos = self.get_positions() if positions is None else np.asarray(positions, np.float32)
        C_, D = self.config.num_cues, self.config.num_due_pairs
        tx = np.concatenate([1 + np.arange(C_), 1 + C_ + 2 * np.arange(D)] + ([np.zeros(C_, np.int64)] if self.config.downlinks else []))
        rx = np.concatenate([np.zeros(C_, np.int64), 2 + C_ + 2 * np.arange(D)] + ([1 + np.arange(C_)] if self.config.downlinks else []))
        return np.concatenate([pos[:, tx], pos[:, rx]], axis=-1)

    @staticmethod
    def assemble_obs(obs_static: np.ndarray, obs_dyn: np.ndarray) -> np.ndarray:
        """The full [E][N][6] table from its once-per-reset and per-step halves (bit-identical to the `obs` output)."""
        return np.concatenate([obs_static, obs_dyn], axis=-1)

    def sample_actions_philox(self, seed: int, step_index: int = 0, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Discrete(n).sample() for every agent on the device (d2d_sample_actions): counter-based, a function of
        (seed, global env, link, step_index) only - the draws d2d_episode makes internally for that step."""
        a = out if out is not None else torch.empty((self.num_envs, self.num_links), dtype=torch.int32, device=self.device)
        _lib.check(self._lib.d2d_sample_actions(self._h, a.data_ptr(), int(seed) & 0xFFFFFFFFFFFFFFFF, int(step_index), self._stream()))
        return a

    def sample_actions(self, generator: Optional[torch.Generator] = None) -> torch.Tensor:
        """Uniform draw from the reference's Discrete action spaces (envs/d2d_env.py:36-40, :54-60)."""
        u = torch.rand((self.num_envs, self.num_links), device=self.device, generator=generator)
        a = torch.minimum((u * self._nvec_f).to(torch.int32), self._nvec_m1)
        if self.config.downlinks:      # reset() draws uplink and sidelink actions only (envs/d2d_env.py:54-60)
            a[:, self.config.num_cues + self.config.num_due_pairs:] = -1
        return a

    def reset(self, seed: Optional[int] = None, mask: Optional[torch.Tensor] = None,
              initial_actions: Optional[torch.Tensor] = None) -> Optional[torch.Tensor]:
        """Re-draw device positions on the GPU and zero the step counters (Simulator.reset, simulator.py:61-75;
        `num_steps = 0`, envs/d2d_env.py:46).  With mask=None this follows D2DEnv.reset (envs/d2d_env.py:45-52):
        one uncounted step with random actions produces the initial observation table, which is returned.
        With a uint8/bool mask [E] only the flagged envs are re-drawn and nothing is returned.
        With autoreset, a full reset also zeroes episode_index and makes this reset's key the base of the auto-reset keys;
        reset(mask) leaves both alone (zeroing an env's index would make it repeat its own draws)."""
        if seed is not None:
            self.seed = int(seed)
            self._episode = 0
        # a fresh Philox key per reset call so successive episodes differ (the reference re-draws from `random`)
        key = (self.seed + 0x9E3779B97F4A7C15 * self._episode) & 0xFFFFFFFFFFFFFFFF
        self._episode += 1
        m = None
        if mask is not None:
            m = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            if m.shape != (self.num_envs,):
                raise ValueError('mask must have shape [num_envs]')
        _lib.check(self._lib.d2d_reset(self._h, key, self.global_env_offset, _ptr(m), self._stream()))
        if mask is not None:
            return None
        if self.autoreset:
            self.episode_index.zero_()
            # the base is this reset's key passed through splitmix64 once: reset keys advance by the same constant as the episode
            # index inside autoreset_key, so with the raw key the next reset's stream would replay this one's shifted by an episode
            self._ar_base = autoreset_key(key, 0)
            self._bind_autoreset()
        actions = initial_actions if initial_actions is not None else self.sample_actions()
        self._bind(False)            # the reset step is not counted (simulator.step is called directly, :50)
        try:
            self._launch(actions)
        finally:
            self._bind(True)
        return self.obs

    # ---- the hot path --------------------------------------------------------------------------
    def _launch(self, actions: torch.Tensor, out: Optional[StepBuffers] = None, inputs_stable: bool = False,
                autoreset: bool = False) -> None:
        if actions.dtype != torch.int32 or not actions.is_cuda or not actions.is_contiguous():
            raise ValueError('actions must be a contiguous int32 CUDA tensor [num_envs][num_links]')
        if tuple(actions.shape) != (self.num_envs, self.num_links):
            raise ValueError(f'actions must have shape {(self.num_envs, self.num_links)}, got {tuple(actions.shape)}')
        io = (out if out is not None else self._out)._io
        io.actions = actions.data_ptr()
        io.flags = (_lib.STEP_INPUTS_STABLE if inputs_stable else 0) | (_lib.STEP_AUTORESET if autoreset else 0)
        _lib.check(self._lib.d2d_step(self._h, C.byref(io), self._stream()))

    def step(self, actions: torch.Tensor, validate: bool = False, out: Optional[StepBuffers] = None,
             inputs_stable: bool = False) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, Dict[str, torch.Tensor]]:
        """One env.step for all E envs: a single fused kernel launch on the current stream, no host sync.

        inputs_stable=True is the D2D_STEP_INPUTS_STABLE promise of include/d2d_b200.h ("Ordering rule"): `actions` (and the
        positions) were written before the PREVIOUS step call on this stream - pre-generated action buffers - so the kernel may
        read them while its predecessor is still running.  The default orders the step after everything earlier in the stream,
        which is what a loop whose policy writes the actions between steps needs.

        With autoreset=True (constructor), envs whose previous step returned done are reset by this call instead: their actions
        are ignored and their row is the first observation of the new episode (reward 0, done 0).  Such a step is always ordered
        the default way, whatever inputs_stable says.

        actions: int32 [E][N]; < 0 marks an agent absent this step (Appendix B.8).  Returns the preallocated
        (obs [E][N][6], reward [E], done [E] uint8, info) tensors, overwritten by the next call.
        validate=True checks the action range on the device first (costs a host sync); out-of-range actions
        are otherwise the caller's responsibility (the reference accepts them silently, Appendix B.9)."""
        if validate and bool((actions >= self._nvec_dev.to(actions.dtype)).any()):
            raise ValueError('action out of range for its Discrete space')
        self._launch(actions, out, inputs_stable, self.autoreset)
        o = out if out is not None else self._out
        info = {'capacity_mbps': o.capacity_mbps}
        if o.agent_reward is not None:
            info['agent_reward'] = o.agent_reward      # [E][N]; `reward` is then its mean over the acting agents
        if self.want_info:
            info.update(rate_bps=o.rate_bps, rb=o.rb, tx_pwr_dbm=o.tx_pwr_dbm,
                        sinr_db=o.obs[..., 4], snr_db=o.obs[..., 5])
        return o.obs, o.reward, o.done, info

    def step_many(self, actions: torch.Tensor, out: Optional[Dict[str, torch.Tensor]] = None,
                  inputs_stable: bool = False) -> Dict[str, torch.Tensor]:
        """T consecutive env.step calls in ONE kernel launch (d2d_step_many): the reference's agent loop
        (examples/simple_env.py:20-33) when the actions of every step are known up front.

        actions: int32 [T][E][N].  Returns {'obs': [T][E][N][6], 'capacity_mbps': [T][E][N], 'reward': [T][E],
        'done': [T][E] uint8 (+ 'rate_bps', 'rb', 'tx_pwr_dbm' with info=True)}; slice t is exactly what the t-th step()
        call would have returned.  Pass `out` (from alloc_many_outputs) to reuse buffers."""
        if actions.dtype != torch.int32 or not actions.is_cuda or not actions.is_contiguous() or actions.dim() != 3:
            raise ValueError('actions must be a contiguous int32 CUDA tensor [T][num_envs][num_links]')
        T = int(actions.shape[0])
        if tuple(actions.shape[1:]) != (self.num_envs, self.num_links) or T < 1:
            raise ValueError(f'actions must have shape (T, {self.num_envs}, {self.num_links}), got {tuple(actions.shape)}')
        o = out if out is not None else self.alloc_many_outputs(T)
        if int(o['obs'].shape[0]) != T:
            raise ValueError('out was allocated for a different number of steps')
        io = _lib.D2DStepIO(actions=actions.data_ptr(), obs=o['obs'].data_ptr(), capacity_mbps=o['capacity_mbps'].data_ptr(),
                            reward=o['reward'].data_ptr(), done=o['done'].data_ptr(), rate_bps=_ptr(o.get('rate_bps')),
                            rb=_ptr(o.get('rb')), tx_pwr_dBm=_ptr(o.get('tx_pwr_dbm')), agent_reward=_ptr(o.get('agent_reward')),
                            flags=_lib.STEP_INPUTS_STABLE if inputs_stable else 0)
        _lib.check(self._lib.d2d_step_many(self._h, C.byref(io), T, self._stream()))
        return o

    def episode(self, num_steps: int = EPISODE_LENGTH, actions: Optional[torch.Tensor] = None,
                out: Optional[Dict[str, torch.Tensor]] = None, reset_seed: Optional[int] = None,
                action_seed: Optional[int] = None, record_actions: bool = False) -> Dict[str, torch.Tensor]:
        """One whole episode in ONE launch (d2d_episode): D2DEnv.reset (envs/d2d_env.py:45-52: new positions, num_steps = 0,
        one uncounted step with sampled actions) and `num_steps` counted steps.  Every output has a leading
        [num_steps + 1] dimension; slice 0 is the reset step's observation, slice t the t-th counted step.

        actions=None samples every step's actions on the device (Discrete.sample, envs/d2d_env.py:54-60; keyed by
        action_seed - default: this episode's reset key) - the kernel then reads no global memory but its constants;
        otherwise actions is int32 [num_steps + 1][E][N].  reset_seed=None continues the env's own episode key sequence,
        exactly like reset().  record_actions adds 'actions' (what was drawn) to the result."""
        T1 = int(num_steps) + 1
        if reset_seed is None:
            reset_seed = (self.seed + 0x9E3779B97F4A7C15 * self._episode) & 0xFFFFFFFFFFFFFFFF
            self._episode += 1
        if action_seed is None:
            action_seed = reset_seed
        draw = actions is None
        if not draw:
            if actions.dtype != torch.int32 or not actions.is_cuda or not actions.is_contiguous() or \
                    tuple(actions.shape) != (T1, self.num_envs, self.num_links):
                raise ValueError(f'actions must be a contiguous int32 CUDA tensor of shape {(T1, self.num_envs, self.num_links)}')
        o = out if out is not None else self.alloc_many_outputs(T1)
        if int(o['obs'].shape[0]) != T1:
            raise ValueError('out was allocated for a different number of steps')
        if record_actions and 'actions' not in o:
            o['actions'] = torch.empty((T1, self.num_envs, self.num_links), dtype=torch.int32, device=self.device)
        io = _lib.D2DStepIO(actions=_ptr(actions), obs=o['obs'].data_ptr(), capacity_mbps=o['capacity_mbps'].data_ptr(),
                            reward=o['reward'].data_ptr(), done=o['done'].data_ptr(), rate_bps=_ptr(o.get('rate_bps')),
                            rb=_ptr(o.get('rb')), tx_pwr_dBm=_ptr(o.get('tx_pwr_dbm')), agent_reward=_ptr(o.get('agent_reward')),
                            actions_out=_ptr(o.get('actions')) if draw else None)
        _lib.check(self._lib.d2d_episode(self._h, C.byref(io), int(num_steps), int(reset_seed) & 0xFFFFFFFFFFFFFFFF,
                                         int(action_seed) & 0xFFFFFFFFFFFFFFFF, _lib.EPISODE_DRAW_ACTIONS if draw else 0,
                                         self._stream()))
        return o

    def rollout(self, num_steps: int, action_seed: int, first_step_index: int = 1,
                out: Optional[Dict[str, torch.Tensor]] = None, record_actions: bool = False,
                inputs_stable: bool = False) -> Dict[str, torch.Tensor]:
        """`num_steps` counted steps from the current state in ONE launch with actions sampled on the device (d2d_rollout): the
        random-policy agent loop without any action buffer.  Slice t equals sample_actions_philox(action_seed,
        first_step_index + t) + step()."""
        T = int(num_steps)
        o = out if out is not None else self.alloc_many_outputs(T)
        if int(o['obs'].shape[0]) != T:
            raise ValueError('out was allocated for a different number of steps')
        if record_actions and 'actions' not in o:
            o['actions'] = torch.empty((T, self.num_envs, self.num_links), dtype=torch.int32, device=self.device)
        io = _lib.D2DStepIO(obs=o['obs'].data_ptr(), capacity_mbps=o['capacity_mbps'].data_ptr(),
                            reward=o['reward'].data_ptr(), done=o['done'].data_ptr(), rate_bps=_ptr(o.get('rate_bps')),
                            rb=_ptr(o.get('rb')), tx_pwr_dBm=_ptr(o.get('tx_pwr_dbm')), agent_reward=_ptr(o.get('agent_reward')),
                            actions_out=_ptr(o.get('actions')), flags=_lib.STEP_INPUTS_STABLE if inputs_stable else 0)
        _lib.check(self._lib.d2d_rollout(self._h, C.byref(io), T, int(action_seed) & 0xFFFFFFFFFFFFFFFF, int(first_step_index),
                                         self._stream()))
        return o

    def bind_stats(self, stats: torch.Tensor) -> None:
        """Accumulate the episode statistics into another float64 [STATS_REPLICAS][NUM_STATS] device tensor from now on (e.g.
        one of two buffers alternated per episode, so that a side stream can reduce the finished episode's sums)."""
        if stats.dtype != torch.float64 or tuple(stats.shape) != (_lib.STATS_REPLICAS, _lib.NUM_STATS) or not stats.is_cuda:
            raise ValueError('stats must be a float64 CUDA tensor [STATS_REPLICAS][NUM_STATS]')
        self._stats = stats
        self._bind(True)

    def alloc_many_outputs(self, T: int) -> Dict[str, torch.Tensor]:
        E, N, dev = self.num_envs, self.num_links, self.device
        o = {'obs': torch.empty((T, E, N, 6), dtype=torch.float32, device=dev),
             'capacity_mbps': torch.empty((T, E, N), dtype=torch.float32, device=dev),
             'reward': torch.empty((T, E), dtype=torch.float32, device=dev),
             'done': torch.empty((T, E), dtype=torch.uint8, device=dev)}
        if self.per_agent_reward:
            o['agent_reward'] = torch.empty((T, E, N), dtype=torch.float32, device=dev)
        if self.want_info:
            o.update(rate_bps=torch.empty((T, E, N), dtype=torch.float32, device=dev),
                     rb=torch.empty((T, E, N), dtype=torch.int16, device=dev),
                     tx_pwr_dbm=torch.empty((T, E, N), dtype=torch.int16, device=dev))
        return o

    def capture_steps(self, actions_seq, outs_seq=None, inputs_stable: bool = False) -> 'torch.cuda.CUDAGraph':
        """Capture len(actions_seq) consecutive steps (step i reads actions_seq[i], writes outs_seq[i] or the
        default buffers) into one CUDA graph: replay() then costs one launch for the whole sequence.
        inputs_stable: the action buffers are filled before every replay() and not rewritten during it (see step()); the
        first step of the graph is always ordered after whatever precedes the replay.  With ShadowingPathLoss the step-call
        counter lives on the device, so every replay draws fresh shadowing values like the reference (path_loss.py:75-81).
        With autoreset the steps auto-reset finished envs like step(); episode_index lives on the device, so every replay draws
        fresh positions (the key base is the one of the last full reset() before the capture)."""
        outs_seq = outs_seq if outs_seq is not None else [None] * len(actions_seq)
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            with torch.cuda.graph(graph, stream=side):
                for a, o in zip(actions_seq, outs_seq):
                    self._launch(a, o, inputs_stable, self.autoreset)
        torch.cuda.current_stream(self.device).wait_stream(side)
        return graph

    def _host_io(self, actions: np.ndarray, out: Dict[str, np.ndarray]) -> '_lib.D2DStepIO':
        # a pipelined host loop passes the same few (actions, outputs) pairs over and over: their descriptor is built once
        # (ten `.ctypes.data` lookups cost more host time than the call they feed).  The cache holds the arrays, so an id
        # cannot be recycled for another object while its entry lives; a dict whose set of outputs changed misses by length.
        key = (id(actions), id(out), len(out))
        hit = self._host_io_cache.get(key)
        if hit is not None and hit[1] is actions and hit[2] is out and all(a is b for a, b in zip(out.values(), hit[3])):
            return hit[0]
        io = self._build_host_io(actions, out)
        if len(self._host_io_cache) >= 64:
            self._host_io_cache.clear()
        self._host_io_cache[key] = (io, actions, out, tuple(out.values()))
        return io

    def _build_host_io(self, actions: np.ndarray, out: Dict[str, np.ndarray]) -> '_lib.D2DStepIO':
        if actions.dtype not in (np.int32, np.int16) or not actions.flags['C_CONTIGUOUS'] or actions.shape != (self.num_envs, self.num_links):
            raise ValueError(f'actions must be a C-contiguous int32 (or int16) array of shape {(self.num_envs, self.num_links)}')
        return _lib.D2DStepIO(flags=_lib.STEP_ACTIONS_I16 if actions.dtype == np.int16 else 0,   # int16: half the upload (D2D_STEP_ACTIONS_I16)
                              actions=actions.ctypes.data, obs=out['obs'].ctypes.data if 'obs' in out else None,
                              capacity_mbps=out['capacity_mbps'].ctypes.data if 'capacity_mbps' in out else None,
                              reward=out['reward'].ctypes.data if 'reward' in out else None,
                              done=out['done'].ctypes.data if 'done' in out else None,
                              rate_bps=out['rate_bps'].ctypes.data if 'rate_bps' in out else None,
                              rb=out['rb'].ctypes.data if 'rb' in out else None,
                              tx_pwr_dBm=out['tx_pwr_dbm'].ctypes.data if 'tx_pwr_dbm' in out else None,
                              agent_reward=out['agent_reward'].ctypes.data if 'agent_reward' in out else None,
                              obs_dyn=out['obs_dyn'].ctypes.data if 'obs_dyn' in out else None)

    def step_host(self, actions: np.ndarray, out: Optional[Dict[str, np.ndarray]] = None) -> Dict[str, np.ndarray]:
        """End-to-end host call (d2d_step_host): host int32 actions in, host arrays out, copies included.
        This is the entry the reference's CPU-side loop would bind (INTEGRATION.md)."""
        a = np.ascontiguousarray(actions, dtype=np.int32)
        if out is None:
            out = self.alloc_host_outputs()
        io = self._host_io(a, out)
        _lib.check(self._lib.d2d_step_host(self._h, C.byref(io), self._stream()))
        return out

    def step_host_async(self, actions: np.ndarray, out: Dict[str, np.ndarray], slot: int) -> None:
        """Pipelined host step (d2d_step_host_async): enqueue upload -> kernel -> download for `slot` (0 or 1) and
        return at once; the arrays must stay alive (and should be pinned) until step_host_wait(slot)."""
        io = self._host_io(actions, out)
        _lib.check(self._lib.d2d_step_host_async(self._h, C.byref(io), int(slot), self._stream()))

    def step_host_wait(self, slot: int) -> None:
        _lib.check(self._lib.d2d_step_host_wait(self._h, int(slot)))

    _HOST_FIELDS = (('obs', _lib.OUT_OBS, 6, np.float32), ('obs_dyn', _lib.OUT_OBS_DYN, 2, np.float32),
                    ('capacity_mbps', _lib.OUT_CAPACITY, 1, np.float32), ('reward', _lib.OUT_REWARD, 0, np.float32),
                    ('done', _lib.OUT_DONE, 0, np.uint8), ('rate_bps', _lib.OUT_RATE, 1, np.float32), ('rb', _lib.OUT_RB, 1, np.int16),
                    ('tx_pwr_dbm', _lib.OUT_TX_PWR, 1, np.int16), ('agent_reward', _lib.OUT_AGENT_REWARD, 1, np.float32))

    def host_slot_buffers(self, slot: int, outputs=('obs_dyn', 'capacity_mbps', 'reward', 'done')) -> Dict[str, np.ndarray]:
        """Library-owned PINNED host buffers of pipeline slot 0 / 1 (d2d_host_slot_buffers) as numpy views: 'actions' (write
        the step's int32 [E][N] actions here) plus the requested outputs.  Passing the returned dict to
        step_host_async(out['actions'], out, slot) moves each direction with ONE copy.  The default outputs are the per-step
        part of a step's results - 12 N + 5 bytes per env-step instead of 28 N + 5 with the full observation table, whose
        position columns only change on reset (get_positions / obs_static / assemble_obs)."""
        E, N = self.num_envs, self.num_links
        mask = 0
        for name, bit, _w, _dt in self._HOST_FIELDS:
            if name in outputs:
                mask |= bit
        unknown = set(outputs) - {f[0] for f in self._HOST_FIELDS}
        if unknown:
            raise ValueError(f'unknown outputs {sorted(unknown)}')
        io = _lib.D2DStepIO()
        _lib.check(self._lib.d2d_host_slot_buffers(self._h, int(slot), mask, C.byref(io)))

        def view(ptr, shape, dtype):
            n = int(np.prod(shape)) * np.dtype(dtype).itemsize
            return np.frombuffer((C.c_char * n).from_address(ptr), dtype=dtype).reshape(shape)

        out = {'actions': view(io.actions, (E, N), np.int32), 'actions16': view(io.actions, (E, N), np.int16)}    # (the same pinned bytes)
        ptrs = {'obs': io.obs, 'obs_dyn': io.obs_dyn, 'capacity_mbps': io.capacity_mbps, 'reward': io.reward, 'done': io.done,
                'rate_bps': io.rate_bps, 'rb': io.rb, 'tx_pwr_dbm': io.tx_pwr_dBm, 'agent_reward': io.agent_reward}
        for name, _bit, width, dt in self._HOST_FIELDS:
            if name in outputs:
                out[name] = view(ptrs[name], (E, N, width) if width > 1 else (E, N) if width == 1 else (E,), dt)
        return out

    def alloc_host_outputs(self, pinned: bool = False, info: bool = True, dyn: bool = False) -> Dict[str, np.ndarray]:
        """Caller-owned host arrays for step_host*: the full observation table, or with dyn=True its per-step columns only."""
        E, N = self.num_envs, self.num_links
        spec = {'capacity_mbps': ((E, N), torch.float32),
                'reward': ((E,), torch.float32), 'done': ((E,), torch.uint8)}
        spec['obs_dyn' if dyn else 'obs'] = ((E, N, 2), torch.float32) if dyn else ((E, N, 6), torch.float32)
        if self.per_agent_reward:
            spec['agent_reward'] = ((E, N), torch.float32)
        if info:
            spec.update({'rate_bps': ((E, N), torch.float32), 'rb': ((E, N), torch.int16),
                         'tx_pwr_dbm': ((E, N), torch.int16)})
        # the ndarrays keep their (optionally pinned) torch storage alive
        return {k: torch.zeros(s, dtype=d, pin_memory=pinned).numpy() for k, (s, d) in spec.items()}

    def per_agent_obs(self, obs: Optional[torch.Tensor] = None, num_envs: Optional[int] = None) -> torch.Tensor:
        """Materialise the reference's per-agent layout (envs/obs_fn.py:43-53): [E][N][6N].  O(N^2) bytes."""
        obs = self.obs if obs is None else obs
        n = self.num_envs if num_envs is None else int(num_envs)
        out = torch.empty((n, self.num_links, 6 * self.num_links), dtype=torch.float32, device=self.device)
        _lib.check(self._lib.d2d_per_agent_obs(self._h, obs.data_ptr(), out.data_ptr(), n, self._stream()))
        return out

    # ---- statistics ------------------------------------------------------------------------------
    def stats_tensor(self) -> torch.Tensor:
        """float64 [NUM_STATS] device tensor (summed over the atomics replicas) - what dist.all_reduce_stats sums."""
        return self._stats.sum(dim=0)

    def stats(self) -> Dict[str, float]:
        v = self.stats_tensor().cpu().tolist()
        return dict(zip(_lib.STAT_NAMES, v))

    def reset_stats(self) -> None:
        _lib.check(self._lib.d2d_stats_reset(self._h, self._stream()))

    @property
    def launch_count(self) -> int:
        return int(self._lib.d2d_launch_count(self._h))

    def step_geometry(self) -> Dict[str, int]:
        g, b, s, e = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32()
        _lib.check(self._lib.d2d_step_geometry(self._h, C.byref(g), C.byref(b), C.byref(s), C.byref(e)))
        return dict(grid=g.value, block=b.value, smem_bytes=s.value, envs_per_block=e.value)
