"""Host-side mirror of the reference's SnakeEnv interface over libsnk.so.

`SnakeBatch`  N environments resident on one GPU; step()/reset() take and return CUDA tensors
              (the fast path; one kernel launch per step on the current torch stream).
`SnakeEnv`    drop-in for `gym.make('Snake-v1', **kw)` (marlenv/envs/snake_env.py:31): one
              environment, NumPy observation without batch dimension, list rewards / dones, dict info,
              same constructor kwargs, same exceptions.

PyTorch is used for device memory and streams only; every rule of the game runs in the CUDA library.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import SnkConfig, SnkStateView, SnkStepExtra, check, lib
from .spaces import Box, Discrete

DEFAULT_REWARD_DICT = {'fruit': 10.0, 'kill': 0.0, 'lose': -0.5, 'win': 0.0, 'time': -0.001}   # snake_env.py:46-52
ACTION_ANGLE_DICT = {0: 0.0, 1: np.pi / 2.0, 2: -np.pi / 2.0}                                   # snake_env.py:40-44
DEFAULT_ACTION_DICT = {'noop': 0, 'left': 1, 'right': 2, 'down': 3, 'up': 4}                    # snake_env.py:32-38
DEFAULT_MAX_EPISODE_STEPS = 1e4                                                                 # snake_env.py:56


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


class SnakeBatch:
    """A shard of `num_envs` Snake-v1 environments on one GPU."""

    def __init__(self, num_envs, height=20, width=20, num_snakes=4, snake_length=3, vision_range=None,
                 frame_stack=1, observer='snake', reward_dict=None, num_fruits=None,
                 max_episode_steps=DEFAULT_MAX_EPISODE_STEPS, device=0, seed=0, rng='philox',
                 auto_reset=True, env_id_offset=0, done_mode='all', wall_map=None, wall_maps=None, map_ids=None,
                 global_state=False, **ignored):
        """wall_map: one custom wall layout for every env.  wall_maps: a pool of layouts of one shape (a list of arrays or
        map paths, or an [M, H, W] array; 1 <= M <= 256); each env starts every episode on the map its `next_maps`
        entry names at that reset (see next_maps / current_maps).  map_ids: initial next_maps (M ids), default
        (env_id_offset + e) % M.  global_state: keep `global_state` current (see there)."""
        reward_dict = DEFAULT_REWARD_DICT if reward_dict is None else reward_dict
        self.wall_map = None
        self.wall_maps = None
        if wall_map is not None and wall_maps is not None:
            raise ValueError('give either wall_map (one layout) or wall_maps (a pool of layouts), not both')
        if wall_map is not None:                      # custom wall layout: the map decides the grid shape
            from .grid_util import as_wall_plane
            self.wall_map = as_wall_plane(wall_map)
            height, width = self.wall_map.shape
        if wall_maps is not None:                     # wall-map pool: the maps decide the grid shape
            from .grid_util import as_wall_plane
            maps = [wall_maps] if isinstance(wall_maps, (str, bytes)) or hasattr(wall_maps, '__fspath__') else wall_maps
            if isinstance(maps, np.ndarray) and maps.ndim == 3 or isinstance(maps, torch.Tensor) and maps.dim() == 3:
                maps = list(np.asarray(maps.cpu() if isinstance(maps, torch.Tensor) else maps))
            planes = [as_wall_plane(m) for m in maps]
            if not 1 <= len(planes) <= _lib.SNK_MAX_MAPS:
                raise ValueError(f'wall_maps must hold 1..{_lib.SNK_MAX_MAPS} layouts, got {len(planes)}')
            if len({p.shape for p in planes}) != 1:
                raise ValueError(f'every map of wall_maps must have one shape, got {sorted({p.shape for p in planes})}')
            self.wall_maps = np.ascontiguousarray(np.stack(planes))
            height, width = self.wall_maps.shape[1:]
        elif map_ids is not None:
            raise ValueError('map_ids needs wall_maps')
        if reward_dict.keys() != DEFAULT_REWARD_DICT.keys():                      # snake_env.py:77-80
            raise KeyError(f'reward dict keys must correspond to {DEFAULT_REWARD_DICT.keys()}')
        if observer not in ('snake', 'human'):
            raise ValueError("observer must be 'snake' (three relative actions) or 'human' (five absolute)")
        self.observer = observer
        self.action_dict = ACTION_ANGLE_DICT if observer == 'snake' else DEFAULT_ACTION_DICT   # snake_env.py:101-104
        if rng not in ('philox', 'replay'):
            raise ValueError("rng must be 'philox' or 'replay'")
        if not torch.cuda.is_available():
            raise RuntimeError('SnakeBatch needs a CUDA device: the step path has no CPU fallback')
        self.device = torch.device('cuda', device if isinstance(device, int) else torch.device(device).index or 0)
        self.num_envs, self.num_snakes = int(num_envs), int(num_snakes)
        self.grid_shape = (int(height), int(width))
        self.snake_length = int(snake_length)
        self.vision_range = vision_range
        self.frame_stack = int(frame_stack)
        self.reward_dict = dict(reward_dict)
        self.num_fruits = int(round(num_snakes * 0.8)) if num_fruits is None else int(num_fruits)
        self.max_episode_steps = max_episode_steps
        self.auto_reset = bool(auto_reset)
        self.rng = rng

        cfg = SnkConfig(abi_version=_lib.SNK_ABI_VERSION, device=self.device.index, num_envs=self.num_envs,
                        height=height, width=width, num_snakes=num_snakes, snake_length=snake_length,
                        vision_range=int(vision_range or 0), frame_stack=frame_stack,
                        num_fruits=self.num_fruits, auto_reset=int(self.auto_reset),
                        done_mode={'all': 0, 'any': 1}[done_mode],
                        rng_mode=_lib.SNK_RNG_REPLAY if rng == 'replay' else _lib.SNK_RNG_PHILOX,
                        observer=1 if observer == 'human' else 0,
                        seed=int(seed), env_id_offset=int(env_id_offset),
                        max_episode_steps=float(max_episode_steps),
                        reward_fruit=float(reward_dict['fruit']), reward_kill=float(reward_dict['kill']),
                        reward_lose=float(reward_dict['lose']), reward_win=float(reward_dict['win']),
                        reward_time=float(reward_dict['time']))
        self._h = C.c_void_p()
        with torch.cuda.device(self.device):
            if self.wall_maps is not None:
                ids = None
                if map_ids is not None:
                    ids = np.asarray(map_ids.cpu() if isinstance(map_ids, torch.Tensor) else map_ids).reshape(-1)
                    if ids.size != self.num_envs or ids.min(initial=0) < 0 or ids.max(initial=0) >= len(self.wall_maps):
                        raise ValueError(f'map_ids must hold one id in 0..{len(self.wall_maps) - 1} per environment')
                    ids = np.ascontiguousarray(ids, dtype=np.uint8)
                check(lib.snk_create_maps(C.byref(cfg), len(self.wall_maps), self.wall_maps.ctypes.data_as(C.c_void_p),
                                          ids.ctypes.data_as(C.c_void_p) if ids is not None else None,
                                          C.byref(self._h)))
            elif self.wall_map is None:
                check(lib.snk_create(C.byref(cfg), C.byref(self._h)))
            else:
                check(lib.snk_create_map(C.byref(cfg), self.wall_map.ctypes.data_as(C.c_void_p), C.byref(self._h)))
        shape = (C.c_int32 * 4)()
        check(lib.snk_obs_shape(self._h, C.byref(shape)))
        self.obs_shape = tuple(shape)                                  # (ns, oh, ow, 8*fs)
        self.obs_ch = self.obs_shape[-1]
        self.bits_shape = self.obs_shape[:-1] + (self.obs_shape[-1] // 8,)   # channel-bit form: one byte per cell and frame
        self._bits = None
        N, ns, dev = self.num_envs, self.num_snakes, self.device
        self._obs_block = _ObsBlock(dev.index, N * int(np.prod(self.obs_shape)))
        self._obs = torch.as_tensor(self._obs_block, device=dev).view((N,) + self.obs_shape)
        self._rew = torch.empty((N, ns), dtype=torch.float64, device=dev)
        self._done = torch.empty((N, ns), dtype=torch.uint8, device=dev)
        self._fin = torch.zeros((N,), dtype=torch.uint8, device=dev)
        self._rank = torch.zeros((N, ns), dtype=torch.int32, device=dev)
        self._ep_scores = torch.zeros((N, ns), dtype=torch.float64, device=dev)
        self._ep_steps = torch.zeros((N, ns), dtype=torch.int32, device=dev)
        self._ep_fruits = torch.zeros((N, ns), dtype=torch.int32, device=dev)
        self._ep_kills = torch.zeros((N, ns), dtype=torch.int32, device=dev)
        self._extra = SnkStepExtra(self._fin.data_ptr(), self._rank.data_ptr(), self._ep_scores.data_ptr(),
                                   self._ep_steps.data_ptr(), self._ep_fruits.data_ptr(),
                                   self._ep_kills.data_ptr())
        self.observation_space = Box(0, 1, (N,) + self.obs_shape, np.uint8)
        self.action_space = Discrete(len(self.action_dict))
        # Every call that steps, resets, restores or replays the shard bumps `_mutations`; rollout.collect keeps its
        # (alive, episode age) cache only while the counter still has the value it stored.  `_obs_stale` is None while
        # self._obs holds the current observation of every env, else the name of the call that left it behind.
        self._mutations = 0
        self._obs_stale = 'construction (no reset yet)'
        self._rollout_alive = self._rollout_age = self._rollout_mark = None
        self.num_maps = int(lib.snk_num_maps(self._h))
        self.next_maps = self.current_maps = None
        if self.num_maps:
            nxt, cur = C.c_void_p(), C.c_void_p()
            check(lib.snk_map_ids_dev(self._h, C.byref(nxt), C.byref(cur)))
            # views of the handle's own uint8 [N] id arrays, valid until close().  next_maps[e]: the map env e's next
            # reset starts from (rewrite it freely, e.g. next_maps.random_(0, num_maps) after every step);
            # current_maps[e]: the map of env e's current episode, set from next_maps by every reset
            self.next_maps = _tensor_from_ptr(nxt.value, N, torch.uint8, dev)
            self.current_maps = _tensor_from_ptr(cur.value, N, torch.uint8, dev)
        # global state for centralized critics: uint8 [N, H, W], every env's grid as cell codes (type + 10 * owner, the
        # reference's SnakeEnv.grid) as the current observation was encoded from it -- after an auto-reset the new
        # episode's grid.  The step kernel writes it beside the observation (snk_step_grid); like next_maps it is the
        # batch's own buffer, overwritten by the next call.  None unless global_state=True.
        self.global_state = None
        if global_state:
            H, W = self.grid_shape
            self._gs_block = _ObsBlock(dev.index, N * H * W)     # mostly zero bytes: compressible, as the observation
            self.global_state = torch.as_tensor(self._gs_block, device=dev).view(N, H, W)

    @property
    def obs_compressed(self):
        """True when the observation buffer is compressible device memory (snk_alloc_obs): the device supports
        generic compression and granted it.  Values and layout are the same either way."""
        return self._obs_block.compressed

    # ---- lifecycle ---------------------------------------------------------------------------------
    def close(self):
        if getattr(self, '_h', None) is not None and self._h.value:
            lib.snk_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _mutated(self, obs_stale):
        """Bookkeeping after a call that changed the shard: obs_stale None = self._obs is now current for every env,
        False = whatever it was before (still current if it was), else the name of the call that outdated it."""
        self._mutations += 1
        if obs_stale is not False:
            self._obs_stale = obs_stale

    # ---- hot path ----------------------------------------------------------------------------------
    def _bits_buffer(self):
        if self._bits is None:
            self._bits = torch.zeros((self.num_envs,) + self.bits_shape, dtype=torch.uint8, device=self.device)
        return self._bits

    def reset(self, mask=None, copy=False, bits=False):
        """SnakeEnv.reset for all envs (or those with mask != 0). Returns uint8 [N, ns, oh, ow, 8*fs], or with
        bits=True the channel-bit form uint8 [N, ns, oh, ow, fs] (see step_bits)."""
        if mask is not None:
            if mask.numel() != self.num_envs:
                raise ValueError('mask must have one entry per environment')
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        with torch.cuda.device(self.device):
            out = self._bits_buffer() if bits else self._obs
            check(lib.snk_reset_grid(self._h, _ptr(mask), None if bits else _ptr(out), _ptr(out) if bits else None,
                                     _ptr(self.global_state), self._stream()))
        # a masked reset rewrites the observation of the selected envs only: the others keep theirs
        self._mutated('reset(bits=True)' if bits else (None if mask is None else False))
        return out.clone() if copy else out

    def step_bits(self, actions, copy=False, want_info=True):
        """As step(), but the observation comes as channel bits: uint8 [N, ns, oh, ow, fs], one byte per window cell
        and frame, bit c = channel c (np.packbits(obs.reshape(..., fs, 8), -1, bitorder='little')).  The encode
        writes them directly -- no NHWC block, an eighth of the observation traffic; `unpack_obs` widens them."""
        return self._step(actions, copy, want_info, bits=True)

    def step(self, actions, copy=False, want_obs=True, want_info=True):
        """actions: uint8 CUDA tensor [N, ns] in {0,1,2} (observer 'snake') or {0..4} ('human').  Returns (obs, rewards f64, dones bool, info)
        where info holds per-env `finished` and, for finished envs, the terminal `rank` / `episode_*`
        arrays the reference puts in its info dict (snake_env.py:396-410).  The returned tensors are
        the batch's own buffers, overwritten by the next call unless copy=True."""
        return self._step(actions, copy, want_info, want_obs=want_obs)

    def _step(self, actions, copy, want_info, bits=False, want_obs=True):
        """Body of step (observation, or none) and step_bits (channel bits)."""
        if actions.dtype != torch.uint8 or actions.device != self.device or not actions.is_contiguous() \
                or actions.numel() != self.num_envs * self.num_snakes:
            raise ValueError('actions must be a contiguous uint8 CUDA tensor of shape [num_envs, num_snakes]')
        out = self._bits_buffer() if bits else self._obs if want_obs else None
        check(lib.snk_step_grid(self._h, _ptr(actions), None if bits else _ptr(out), _ptr(out) if bits else None,
                                _ptr(self.global_state), _ptr(self._rew), _ptr(self._done),
                                C.byref(self._extra) if want_info else None, self._stream()))
        self._mutated('step_bits' if bits else None if want_obs else 'step(want_obs=False)')
        info = {}
        if want_info:
            info = dict(finished=self._fin.view(torch.bool), rank=self._rank, episode_scores=self._ep_scores,
                        episode_steps=self._ep_steps, episode_fruits=self._ep_fruits,
                        episode_kills=self._ep_kills)
        res = (out, self._rew, self._done.view(torch.bool), info)
        if copy:
            res = (None if out is None else out.clone(), res[1].clone(), res[2].clone(),
                   {k: v.clone() for k, v in info.items()})
        return res

    def step_many(self, actions, obs=None, rewards=None, dones=None, bits=None, finished=None, global_state=None):
        """T steps in one call (snk_step_many) for open-loop action streams.  actions: uint8 CUDA [T, N, ns].
        rewards f64 / dones uint8 [T, N, ns] are allocated when not given.  obs (uint8) / bits / global_state (uint8
        [.., N, H, W]): a [T, N, ...] tensor receives every step's block, an [N, ...] tensor only the last step's; None
        skips that output.  finished: optional uint8 [T, N].  Returns (obs, rewards, dones, bits).  Bit-identical to T
        calls of step().  A batch created with global_state=True keeps its `global_state` current either way."""
        N, ns = self.num_envs, self.num_snakes
        if actions.dtype != torch.uint8 or actions.device != self.device or not actions.is_contiguous() \
                or actions.dim() != 3 or tuple(actions.shape[1:]) != (N, ns):
            raise ValueError('actions must be a contiguous uint8 CUDA tensor of shape [T, num_envs, num_snakes]')
        T = actions.shape[0]
        if rewards is None:
            rewards = torch.empty((T, N, ns), dtype=torch.float64, device=self.device)
        if dones is None:
            dones = torch.empty((T, N, ns), dtype=torch.uint8, device=self.device)
        for name, buf, dtype in (('rewards', rewards, torch.float64), ('dones', dones, torch.uint8)):
            if buf.dtype != dtype or buf.device != self.device or not buf.is_contiguous() \
                    or tuple(buf.shape) != (T, N, ns):
                raise ValueError(f'{name} must be a contiguous {str(dtype)[6:]} CUDA tensor of shape '
                                 '[T, num_envs, num_snakes]')
        every = None
        for name, buf, shape in (('obs', obs, self.obs_shape), ('bits', bits, self.bits_shape),
                                 ('global_state', global_state, self.grid_shape)):
            if buf is None:
                continue
            if buf.dtype != torch.uint8 or buf.device != self.device or not buf.is_contiguous():
                raise ValueError(f'{name} must be a contiguous uint8 CUDA tensor')
            if tuple(buf.shape) == (T, N) + shape and (T > 1 or buf.dim() == len(shape) + 2):
                e = True
            elif tuple(buf.shape) == (N,) + shape:
                e = False
            else:
                raise ValueError(f'{name} must have shape [T, N, ...] (every step) or [N, ...] (last step only)')
            if every is not None and every != e:
                raise ValueError('obs, bits and global_state must all hold every step or all hold the last step only')
            every = e
        extra = None
        if finished is not None:
            if tuple(finished.shape) != (T, N) or finished.dtype != torch.uint8 or finished.device != self.device \
                    or not finished.is_contiguous():
                raise ValueError('finished must be a contiguous uint8 CUDA tensor of shape [T, N]')
            extra = SnkStepExtra(finished.data_ptr(), 0, 0, 0, 0, 0)
        grid = global_state
        if grid is None and self.global_state is not None and not every:
            grid = self.global_state                        # the last step's rows straight into the batch's buffer
        check(lib.snk_step_many_grid(self._h, T, _ptr(actions), _ptr(obs), _ptr(bits), _ptr(grid), int(bool(every)),
                                     _ptr(rewards), _ptr(dones), C.byref(extra) if extra is not None else None,
                                     self._stream()))
        if self.global_state is not None and grid is not self.global_state:
            if grid is not None:
                self.global_state.copy_(grid[-1] if every else grid)
            else:                                           # obs / bits of every step, no caller grid: rebuild it
                self._refresh_global_state()
        self._mutated('step_many')
        return obs, rewards, dones, bits

    def step_host(self, actions, obs, rewards, dones):
        """Reference-shaped call on HOST buffers (pinned NumPy/torch CPU arrays): copies actions in,
        steps, copies obs/rewards/dones out, synchronises.  `obs` may be None."""
        check(lib.snk_step_host(self._h, C.c_void_p(actions.data_ptr()),
                                C.c_void_p(obs.data_ptr()) if obs is not None else C.c_void_p(0),
                                C.c_void_p(rewards.data_ptr()), C.c_void_p(dones.data_ptr())))
        self._refresh_global_state()
        self._mutated('step_host')

    def step_host_info(self, actions, obs, rewards, dones, finished=None, rank=None, episode_scores=None,
                       episode_steps=None, episode_fruits=None, episode_kills=None):
        """step_host plus the terminal info arrays of step() (snk_step_host_info), each into a HOST buffer of the same
        shape (finished uint8 [N], rank / episode_steps / _fruits / _kills int32 [N, ns], episode_scores float64
        [N, ns]); any of them may be None.  Entries of envs that did not finish are unspecified."""
        def hp(x):
            return x.data_ptr() if x is not None else None
        xh = SnkStepExtra(hp(finished), hp(rank), hp(episode_scores), hp(episode_steps), hp(episode_fruits),
                          hp(episode_kills))
        check(lib.snk_step_host_info(self._h, C.c_void_p(actions.data_ptr()),
                                     C.c_void_p(obs.data_ptr()) if obs is not None else C.c_void_p(0),
                                     C.c_void_p(rewards.data_ptr()), C.c_void_p(dones.data_ptr()), C.byref(xh)))
        self._refresh_global_state()
        self._mutated('step_host_info')

    def step_host_bits(self, actions, bits, rewards, dones):
        """As step_host, but `bits` (uint8, obs shape with the last dimension divided by 8) receives channel
        bits -- one byte per (cell, frame) -- and nothing is widened on the host."""
        check(lib.snk_step_host_bits(self._h, C.c_void_p(actions.data_ptr()), C.c_void_p(bits.data_ptr()),
                                     C.c_void_p(rewards.data_ptr()), C.c_void_p(dones.data_ptr())))
        self._refresh_global_state()
        self._mutated('step_host_bits')

    def reset_host(self, obs):
        check(lib.snk_reset_host(self._h, C.c_void_p(obs.data_ptr()) if obs is not None else C.c_void_p(0)))
        self._refresh_global_state()
        self._mutated('reset_host')

    def set_host_transport(self, mode, threads=0):
        """How step_host / reset_host move the observation block over PCIe: 'raw' (one D2H of the NHWC
        bytes) or 'packed' (channel bits on the link, widened by `threads` host threads; 0 = all cores)."""
        check(lib.snk_set_host_transport(self._h, {'raw': _lib.SNK_XFER_RAW, 'packed': _lib.SNK_XFER_PACKED}[mode],
                                         int(threads)))

    def host_transport(self):
        mode, threads = C.c_int(0), C.c_int(0)
        check(lib.snk_get_host_transport(self._h, C.byref(mode), C.byref(threads)))
        return ('raw', 'packed')[mode.value], threads.value

    def pack_obs(self, obs=None, out=None):
        """Channel-bit form of an observation tensor (uint8 0/1, last dim a multiple of 8): one byte per
        (cell, frame), bit c = channel c.  8x smaller for device replay buffers; `unpack_obs` inverts it."""
        obs = self._obs if obs is None else obs
        if obs.dtype != torch.uint8 or not obs.is_cuda or not obs.is_contiguous() or obs.shape[-1] % 8:
            raise ValueError('obs must be a contiguous uint8 CUDA tensor whose last dimension is a multiple of 8')
        shape = (*obs.shape[:-1], obs.shape[-1] // 8)
        if out is None:
            out = torch.empty(shape, dtype=torch.uint8, device=obs.device)
        check(lib.snk_pack_obs(self._h, _ptr(obs), _ptr(out), obs.numel(), self._stream()))
        return out

    # ---- parity / checkpoint interface ---------------------------------------------------------------
    def _refresh_global_state(self):
        """After a call that changes the state without writing `global_state` (set_state, load_checkpoint, the
        host-buffer calls): one snk_get_state launch that fills only the grid."""
        if self.global_state is not None:
            view = SnkStateView(grid=self.global_state.data_ptr())
            check(lib.snk_get_state(self._h, C.byref(view), self._stream()))

    def get_state(self, max_cells=None):
        N, ns, dev = self.num_envs, self.num_snakes, self.device
        H, W = self.grid_shape
        i32 = dict(dtype=torch.int32, device=dev)
        u8 = dict(dtype=torch.uint8, device=dev)
        st = dict(grid=torch.empty((N, H * W), **u8), head=torch.empty((N, ns), **i32),
                  tail=torch.empty((N, ns), **i32), length=torch.empty((N, ns), **i32),
                  dir=torch.empty((N, ns), **u8), alive=torch.empty((N, ns), **u8),
                  alive_counter=torch.empty((N,), **i32), episode_length=torch.empty((N,), **i32))
        if max_cells:
            st['cells'] = torch.empty((N, ns, max_cells), **i32)
        view = SnkStateView(**{k: v.data_ptr() for k, v in st.items()}, max_cells=int(max_cells or 0))
        check(lib.snk_get_state(self._h, C.byref(view), self._stream()))
        st['grid'] = st['grid'].view(N, H, W)
        if self.num_maps:
            st['map'] = self.current_maps.clone()           # the wall map of each env's current episode
        return st

    def set_state(self, grid, alive, dir, length, cells, alive_counter, episode_length=None):
        """Force a state (scenario tests / restore). cells: int32 [N, ns, L] head-first flat cell indices."""
        N, ns, dev = self.num_envs, self.num_snakes, self.device

        def t(x, dtype, shape):
            return torch.as_tensor(np.ascontiguousarray(x), dtype=dtype).reshape(shape).to(dev).contiguous()
        cells = t(cells, torch.int32, (N, ns, -1))
        H, W = self.grid_shape
        length_h = np.asarray(length).reshape(N, ns)
        if cells.shape[-1] < 2 or int(length_h.max(initial=0)) > cells.shape[-1] or int(length_h.min(initial=0)) < 0:
            raise ValueError('length must be within 0..cells.shape[-1] (and cells hold at least two columns)')
        if int(cells.min()) < 0 or int(cells.max()) >= H * W:
            raise ValueError('cells must be flat indices into the H x W grid (pad unused entries with 0)')
        if episode_length is None:
            episode_length = np.zeros(N, dtype=np.int32)
        keep = dict(grid=t(grid, torch.uint8, (N, -1)), alive=t(alive, torch.uint8, (N, ns)),
                    dir=t(dir, torch.uint8, (N, ns)), length=t(length, torch.int32, (N, ns)), cells=cells,
                    alive_counter=t(alive_counter, torch.int32, (N,)),
                    episode_length=t(episode_length, torch.int32, (N,)))
        view = SnkStateView(**{k: v.data_ptr() for k, v in keep.items()}, max_cells=cells.shape[-1])
        check(lib.snk_set_state(self._h, C.byref(view), _ptr(self._obs), self._stream()))
        self._refresh_global_state()
        torch.cuda.current_stream(self.device).synchronize()      # `keep` must outlive the kernels
        self._mutated(None)
        return self._obs

    def save_checkpoint(self):
        """Exact state of the shard as a NumPy byte array (records, frame histories, statistics); a batch
        created with the same arguments continues bit for bit after load_checkpoint()."""
        n = int(lib.snk_checkpoint_bytes(self._h))
        blob = np.empty(n, dtype=np.uint8)
        check(lib.snk_checkpoint_save(self._h, blob.ctypes.data_as(C.c_void_p), n))
        return blob

    def load_checkpoint(self, blob):
        blob = np.ascontiguousarray(blob, dtype=np.uint8)
        check(lib.snk_checkpoint_load(self._h, blob.ctypes.data_as(C.c_void_p), blob.size))
        self._refresh_global_state()
        self._mutated('load_checkpoint')

    # ---- per-env snapshot / restore on the device (snk_snapshot / snk_restore) --------------------------------------
    @property
    def snapshot_bytes(self):
        """Bytes of one snapshot slot: a row of the tensors snapshot() returns and restore() takes."""
        return int(lib.snk_snapshot_bytes(self._h))

    def _ids(self, x, name):
        if not isinstance(x, torch.Tensor) or x.device != self.device or x.dim() != 1 \
                or x.dtype.is_floating_point or x.dtype.is_complex or x.dtype == torch.bool:
            raise ValueError(f'{name} must be a 1-d integer CUDA tensor on the batch device')
        return x.to(torch.int32).contiguous()

    def _slots(self, x, name, rows=None):
        if not isinstance(x, torch.Tensor) or x.dtype != torch.uint8 or x.device != self.device or x.dim() != 2 \
                or not x.is_contiguous() or x.data_ptr() % 16 or x.shape[0] < 1 \
                or x.shape[1] != self.snapshot_bytes or (rows is not None and x.shape[0] != rows):
            want = f'[{rows if rows is not None else "K"}, {self.snapshot_bytes}]'
            raise ValueError(f'{name} must be a contiguous, 16-byte aligned uint8 CUDA tensor of shape {want} '
                             '(rows of snapshot_bytes)')
        return x

    def snapshot(self, env_ids=None, out=None):
        """The exact state of envs env_ids (an integer CUDA tensor, duplicates allowed; None = all envs) as uint8 [K,
        snapshot_bytes] on the device: record, frame history and wall map of each env, byte for byte.  `out` may be a
        preallocated tensor of that shape.  Rows restore into this batch or any batch of the same configuration (see
        restore); ids outside [0, N) raise a device error (raise_on_device_errors) and give rows nothing accepts."""
        if env_ids is not None:
            env_ids = self._ids(env_ids, 'env_ids')
        K = self.num_envs if env_ids is None else env_ids.numel()
        if not 1 <= K <= self.num_envs:
            raise ValueError(f'snapshot takes 1..{self.num_envs} env ids, got {K}')
        if out is None:
            out = torch.empty((K, self.snapshot_bytes), dtype=torch.uint8, device=self.device)
        self._slots(out, 'out', K)
        check(lib.snk_snapshot(self._h, _ptr(env_ids), K, _ptr(out), self._stream()))
        return out

    def restore(self, snapshots, src=None, *, env_ids=None, slots=None, copy=False, bits=False):
        """Put envs back into snapshotted states.  Either src (integer CUDA [N]: env e takes row src[e] of snapshots,
        -1 keeps it) or env_ids (integer CUDA [K]) with slots (row of each, default 0..K-1; ids outside [0, N) are
        skipped).  One row may go to any number of envs.  The restored episode continues exactly -- statistics,
        frame stack, replay cursor and Philox event count included -- with draws keyed by the destination env's id, so
        a row restored into another env continues that env's own stream (snk.h).  Writes the restored envs' rows of
        the observation buffer (the channel-bit buffer with bits=True) and of global_state, and returns that buffer."""
        snapshots = self._slots(snapshots, 'snapshots')
        N = self.num_envs
        if src is not None:
            if env_ids is not None or slots is not None:
                raise ValueError('give either src or env_ids (and slots), not both')
            src = self._ids(src, 'src')
            if src.numel() != N:
                raise ValueError('src must have one entry per environment')
        else:
            if env_ids is None:
                raise ValueError('restore needs src or env_ids')
            env_ids = self._ids(env_ids, 'env_ids')
            slots = torch.arange(env_ids.numel(), dtype=torch.int32, device=self.device) if slots is None \
                else self._ids(slots, 'slots')
            if slots.numel() != env_ids.numel():
                raise ValueError('slots must have one entry per env id')
            # built on the device without a synchronisation: ids outside [0, N) land in a spare last entry
            ids = torch.where((env_ids >= 0) & (env_ids < N), env_ids, N).long()
            src = torch.full((N + 1,), -1, dtype=torch.int32, device=self.device)
            src.index_put_((ids,), slots)
            src = src[:N]
        with torch.cuda.device(self.device):
            out = self._bits_buffer() if bits else self._obs
            check(lib.snk_restore(self._h, _ptr(src), snapshots.shape[0], _ptr(snapshots), None if bits else _ptr(out),
                                  _ptr(out) if bits else None, _ptr(self.global_state), self._stream()))
        # as a masked reset: only the restored envs' observation rows are rewritten
        self._mutated('restore(bits=True)' if bits else False)
        return out.clone() if copy else out

    def set_replay(self, draws_per_env):
        """draws_per_env: sequence of N int arrays -- recorded draw outputs in consumption order."""
        assert len(draws_per_env) == self.num_envs
        off = np.zeros(self.num_envs + 1, dtype=np.int64)
        off[1:] = np.cumsum([len(d) for d in draws_per_env])
        flat = np.concatenate([np.asarray(d, dtype=np.int32).reshape(-1) for d in draws_per_env]) \
            if off[-1] else np.zeros(1, dtype=np.int32)
        flat = np.ascontiguousarray(flat, dtype=np.int32)
        check(lib.snk_set_replay(self._h, flat.ctypes.data_as(C.c_void_p), off.ctypes.data_as(C.c_void_p)))

    def replay_cursors(self):
        out = np.zeros(self.num_envs, dtype=np.int32)
        check(lib.snk_replay_cursors(self._h, out.ctypes.data_as(C.c_void_p)))
        return out

    def device_errors(self, clear=False):
        bits = C.c_uint32(0)
        check(lib.snk_device_errors(self._h, C.byref(bits), int(clear)))
        return bits.value

    def raise_on_device_errors(self):
        bits = self.device_errors(clear=True)
        if bits & 1:
            raise KeyError('action outside {0, 1, 2}')                 # the reference's KeyError (:606)
        if bits:
            raise _lib.SnkError('; '.join(m for b, m in _lib.DEV_ERRORS.items() if bits & b))

    # ---- rollout statistics --------------------------------------------------------------------------
    def stats(self, clear=False):
        out = np.zeros(8, dtype=np.float64)
        check(lib.snk_stats(self._h, out.ctypes.data_as(C.c_void_p), int(clear)))
        return dict(zip(_lib.STAT_NAMES[:7], out[:7]))

    def stats_tensor(self):
        """The device-resident statistics vector (8 doubles) as a torch tensor sharing memory, ready
        for an in-place torch.distributed.all_reduce at the end of a rollout."""
        p = C.c_void_p()
        check(lib.snk_stats_dev(self._h, C.byref(p)))
        return _tensor_from_ptr(p.value, 8, torch.float64, self.device)

    def algorithmic_bytes_per_env_step(self):
        return int(lib.snk_algorithmic_bytes_per_env_step(self._h))


class _ObsBlock:
    """Owner of one observation buffer from snk_alloc_obs: `nbytes` of uint8 device memory, compressible where the
    device grants it.  torch.as_tensor(owner) keeps the owner alive for as long as any tensor views the memory, so
    an observation returned by a batch stays valid after the batch is closed or gone; only __del__ frees it."""

    def __init__(self, device, nbytes):
        ptr, comp = C.c_void_p(), C.c_int(0)
        check(lib.snk_alloc_obs(int(device), int(nbytes), C.byref(ptr), C.byref(comp)))
        self.ptr, self.compressed = ptr, bool(comp.value)
        self.__cuda_array_interface__ = dict(shape=(int(nbytes),), typestr='|u1', data=(ptr.value, False), version=2)

    def __del__(self):
        try:
            if self.ptr.value:
                lib.snk_free_obs(self.ptr)
                self.ptr = C.c_void_p()
        except Exception:
            pass


def _tensor_from_ptr(ptr, n, dtype, device):
    class _Holder:
        pass
    h = _Holder()
    itemsize = torch.empty((), dtype=dtype).element_size()
    typestr = '|u1' if dtype == torch.uint8 else {8: '<f8', 4: '<f4'}[itemsize]
    h.__cuda_array_interface__ = dict(shape=(n,), typestr=typestr, data=(ptr, False), version=2)
    return torch.as_tensor(h, device=device)


class _HostStepper:
    """The host buffers of a batch's host-buffer calls: one C-ABI call per step (snk_step_host_info: actions in, step,
    observation / rewards / dones / terminal info out, one synchronisation) or per reset (snk_reset_host).  `pinned`
    page-locks the buffers, which lets the large transfers of a big batch run asynchronously."""

    def __init__(self, batch, pinned=False):
        N, ns = batch.num_envs, batch.num_snakes

        def host(shape, dtype):
            a = np.zeros(shape, dtype=dtype)
            return torch.from_numpy(a).pin_memory().numpy() if pinned else a
        self.act = host((N, ns), np.uint8)
        self.obs = host((N,) + batch.obs_shape, np.uint8)
        self.rew, self.done = host((N, ns), np.float64), host((N, ns), np.uint8)
        self.fin, self.rank = host((N,), np.uint8), host((N, ns), np.int32)
        self.scores, self.counts = host((N, ns), np.float64), host((3, N, ns), np.int32)
        self._xh = SnkStepExtra(self.fin.ctypes.data, self.rank.ctypes.data, self.scores.ctypes.data,
                                self.counts[0].ctypes.data, self.counts[1].ctypes.data, self.counts[2].ctypes.data)
        # the buffers never move: their addresses (and the handle) are converted for ctypes once, not on every step
        act, obs, rew, done = (x.ctypes.data_as(C.c_void_p) for x in (self.act, self.obs, self.rew, self.done))
        self._step_args = (batch._h, act, obs, rew, done, C.byref(self._xh))
        self._reset_args = (batch._h, obs)

    def reset(self):
        check(lib.snk_reset_host(*self._reset_args))

    def step(self):
        check(lib.snk_step_host_info(*self._step_args))

    def info(self, e):
        """The reference's terminal info dict of env e (snake_env.py:396-410); valid where fin[e] is set."""
        return dict(rank=[int(r) for r in self.rank[e]], episode_scores=self.scores[e].copy(),
                    episode_steps=self.counts[0, e].astype(np.float64),
                    episode_fruits=self.counts[1, e].astype(np.float64),
                    episode_kills=self.counts[2, e].astype(np.float64))


class SnakeEnv:
    """Drop-in for the reference's SnakeEnv (one environment, host-side return types).

    reset() -> np.uint8 [ns, oh, ow, 8*fs]; step(actions) -> (obs, list[float], list[bool], dict).
    Unknown kwargs are ignored as the reference does (snake_env.py:68-69); `reward_func` is accepted as
    an alias of `reward_dict` (README spelling)."""

    default_reward_dict = DEFAULT_REWARD_DICT
    default_action_dict = DEFAULT_ACTION_DICT
    action_angle_dict = ACTION_ANGLE_DICT
    reward_keys = DEFAULT_REWARD_DICT.keys()
    metadata = {}
    _done_mode = 'all'

    def __init__(self, height=20, width=20, num_snakes=4, snake_length=3, vision_range=None, frame_stack=1,
                 observer='snake', *args, **kwargs):
        if 'reward_dict' not in kwargs and isinstance(kwargs.get('reward_func'), dict):
            kwargs['reward_dict'] = kwargs.pop('reward_func')
        reward_dict = kwargs.pop('reward_dict', DEFAULT_REWARD_DICT)
        self._batch = SnakeBatch(1, height=height, width=width, num_snakes=num_snakes,
                                 snake_length=snake_length, vision_range=vision_range, frame_stack=frame_stack,
                                 observer=observer, reward_dict=reward_dict,
                                 num_fruits=kwargs.pop('num_fruits', None),
                                 max_episode_steps=kwargs.pop('max_episode_steps', DEFAULT_MAX_EPISODE_STEPS),
                                 device=kwargs.pop('device', 0), seed=kwargs.pop('seed', 0),
                                 rng=kwargs.pop('rng', 'philox'), auto_reset=False, done_mode=self._done_mode,
                                 wall_map=kwargs.pop('wall_map', None))
        b = self._batch
        self.reward_dict = b.reward_dict
        self.max_episode_steps = b.max_episode_steps
        self.num_snakes, self.num_fruits = b.num_snakes, b.num_fruits
        self.grid_shape, self.snake_length = b.grid_shape, b.snake_length
        self.vision_range, self.frame_stack, self.observer = vision_range, b.frame_stack, observer
        self.low, self.high, self.image_obs = 0, 1, False
        self.action_dict = b.action_dict
        self.obs_ch = b.obs_ch
        self.action_space = Discrete(len(self.action_dict) * self.num_snakes)             # snake_env.py:107-109
        self.observation_space = Box(self.low, self.high, b.obs_shape, np.uint8)          # snake_env.py:115-129
        self._host = _HostStepper(b)

    @property
    def unwrapped(self):
        return self

    def seed(self, seed=42):
        """As in the reference (snake_env.py:161-163) this has no effect on the game: there it only creates
        `self.np_random`, which nothing reads -- spawns and fruits draw from the module-global NumPy generator.  The
        stream of this environment is fixed by the constructor's `seed=` (Philox key) or by `set_replay`."""
        return [seed]

    def close(self):
        self._batch.close()

    def reset(self):
        self._host.reset()
        self.frame_buffer = []                                                            # snake_env.py:151
        return self._host.obs[0].copy()

    def _alive_now(self):
        return self._batch.get_state()['alive'][0].cpu().numpy().astype(bool)

    def step(self, actions):
        if isinstance(actions, int):
            actions = [actions]
        assert len(actions) == self.num_snakes                                            # snake_env.py:313
        hs, alive = self._host, None
        for i, ac in enumerate(actions):
            if isinstance(ac, np.ndarray):
                ac = ac.item()
            if self.observer == 'human':              # unknown actions keep the direction (:610-632)
                hs.act[0, i] = int(ac) if ac in (0, 1, 2, 3, 4) else 0
                continue
            if ac not in self.action_dict:            # the reference looks the action up only for live snakes
                alive = self._alive_now() if alive is None else alive
                if alive[i]:
                    raise KeyError(ac)                                                    # snake_env.py:606
                ac = 0
            hs.act[0, i] = int(ac)
        hs.step()
        info = hs.info(0) if hs.fin[0] else {}
        return (hs.obs[0].copy(), hs.rew[0].tolist(), hs.done[0].astype(bool).tolist(), info)

    @property
    def grid(self):
        """The H x W cell-code grid as the reference keeps it (np.int64)."""
        return self._batch.get_state()['grid'][0].cpu().numpy().astype(np.int64)

    @property
    def alive_snakes(self):
        return int(self._batch.get_state()['alive_counter'][0])

    def render(self, mode='ascii'):
        if mode == 'ascii':
            sym = {0: '.', 1: '#', 2: 'o', 3: 'H', 4: 'b', 5: 't'}
            print('\n'.join(''.join(sym[int(v) % 10] for v in row) for row in self.grid))
        elif mode == 'rgb_array':
            from .render import rgb_from_grid
            return rgb_from_grid(self.grid)
        elif mode == 'gif':                       # append a frame; save_gif() writes them out (snake_env.py:283-288)
            from .render import image_from_grid
            self.frame_buffer.append(image_from_grid(self.grid))

    def save_gif(self, fp=None):
        """Write the frames collected by render('gif') as an animated GIF (snake_env.py:419-436): to `fp`
        (path or file object), or to ./tmp/<timestamp>.gif.  Returns fp."""
        import datetime
        import os
        import warnings
        if fp is None:
            save_dir = os.path.join(os.getcwd(), 'tmp')
            os.makedirs(save_dir, exist_ok=True)
            fp = os.path.join(save_dir, '{}.gif'.format(datetime.datetime.now().strftime('%Y%m%d%H%M%S')))
        if not getattr(self, 'frame_buffer', None):
            warnings.warn("You must call render('gif') first. No images to save.")
        else:
            self.frame_buffer[0].save(fp, save_all=True, append_images=self.frame_buffer[1:], format='GIF', loop=0)
        return fp

    def render_fancy(self, cell_size=40, save_path=None):
        """RGB frame of the current state, pixel for pixel the reference's drawing (snake_env.py:165-263; see
        render.py).  The state -- grid, per-snake body cells, headings -- is exported from the device."""
        from .render import render_fancy
        longest = max(int(self._batch.get_state()['length'].max()), 2)
        st = self._batch.get_state(max_cells=longest)
        img = render_fancy(st['grid'][0].cpu().numpy(), st['cells'][0].cpu().numpy(), st['alive'][0].cpu().numpy(),
                           st['dir'][0].cpu().numpy(), cell_size)
        if save_path:
            from PIL import Image
            Image.fromarray(img).save(save_path)
            print(f"Saved fancy render to {save_path}")
        return img


class CoopSnakeEnv(SnakeEnv):
    """SnakeCoop-v1: the episode ends as soon as any snake is done (coop_snake_env.py:14-22)."""
    _done_mode = 'any'
