"""Every built instance of the step kernel, launched on purpose and checked against the Python oracle.

libsnk.so builds snk_tile_kernel<ns, W, oh, ow, fs, coop, enc, variant> for a few specialised shapes and a generic set
per encode flavour, and which instance a call runs depends on the shape, the tile mode, the handle (wall-map pool, global
state, the uncapped-register threshold) and the call (bits, several steps, where the output lies).  Here a recipe table,
generated from those rules, names for every instance the batch, the knobs and the call that select it.  A CPU test holds
the table against the instances cuobjdump lists, so a new instance without a recipe fails before any GPU run.  On the
GPU a launch witness (torch.profiler's CUDA activity) records the kernels each call launched, every call must launch
exactly its instance, and every output the instance writes is compared with the oracle (oracle/snake_oracle.py with
PhiloxDraws) -- not with HostSim, which compiles the kernels' own rule source, and not with another variant."""
import copy
import ctypes as C
import itertools
import re
import shutil
import subprocess
from contextlib import contextmanager

import numpy as np
import pytest

from oracle.snake_oracle import OracleSnakeEnv
from test_gpu_entry_point_sequences import OracleShard, packbits

ENC_LEGACY, ENC_REG, ENC_DIRECT, ENC_PAD = 0, 1, 2, 3          # snk_kernels.h
GENERIC = (0, 0, 0, 0, 0)                                       # ns, W, oh, ow, fs of the generic instances
VARIANTS = (0, 1, 2, 3, 4, 5, 6, 8, 10, 12, 14)
MAX_STEPS = 7                                                   # episodes end inside the runs and inside step_many
OFFSETS = (0, 1000, 2 ** 32 - 5)                                # the last one straddles the Philox counter's high word

# name: SnakeBatch kwargs, specialisation (ns, W, oh, ow, fs) or GENERIC, encode flavour, tile modes it is built for,
# number of envs.  The generic shapes miss every SNK_TRY of launch_tile_kernel.  N is ragged for every tile shape used
# here: not a multiple of the envs of a warp-private CTA (4 warps of 32 / group(ns) envs) nor of a cooperative tile.
SHAPES = {
    'cfg5': (dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5), (4, 20, 11, 11, 1), ENC_REG,
             (0, 1), 70),
    'cfg2': (dict(height=20, width=20, num_snakes=4, snake_length=3), (4, 20, 20, 20, 1), ENC_DIRECT, (0, 1), 70),
    'cfg3': (dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5, frame_stack=4), (4, 20, 11, 11, 4),
             ENC_LEGACY, (1,), 70),
    'cfg4': (dict(height=64, width=64, num_snakes=16, snake_length=5, vision_range=7), (16, 64, 15, 15, 1), ENC_PAD,
             (1,), 5),
    'reg': (dict(height=13, width=11, num_snakes=3, snake_length=3, vision_range=3), GENERIC, ENC_REG, (0, 1), 70),
    'direct': (dict(height=12, width=14, num_snakes=2, snake_length=3), GENERIC, ENC_DIRECT, (0, 1), 70),
    'pad': (dict(height=32, width=32, num_snakes=8, snake_length=3, vision_range=6), GENERIC, ENC_PAD, (1,), 7),
    # ten snakes: one {as-other, as-own} LUT pair (encode_lut_dual), which only the legacy encode reads; W = 13 keeps the
    # cooperative tiles off the padded-plane encode
    'legacy': (dict(height=15, width=13, num_snakes=10, snake_length=3, vision_range=2), GENERIC, ENC_LEGACY, (0, 1), 37),
}


def tile_group(ns):
    return 1 if ns <= 1 else 2 if ns <= 2 else 4 if ns <= 4 else 8 if ns <= 8 else 16 if ns <= 16 else 32


def built_variants(spec, coop):
    """The variants launch_instance can select for a set of instances: the uncapped copy (3) exists warp-private only,
    and a specialised frame stack has no several-steps-per-launch variants (2, 6): step_many launches once per step."""
    fs = spec[4]
    return [v for v in VARIANTS if not (coop and v == 3) and not (fs > 1 and v in (2, 6))]


def reset_variant(var):
    """What a reset or the encode of a restore runs on the recipe's handle: it never takes several steps."""
    return {2: 0, 6: 4}.get(var, var)


def make_recipes():
    recipes = {}
    for name, (kw, spec, enc, modes, N) in SHAPES.items():
        for coop in modes:
            for var in built_variants(spec, coop):
                key = spec + (coop, enc, var)
                v = var & 3
                fs = kw.get('frame_stack', 1)
                if v == 0:
                    calls = ['step']
                elif v == 1:
                    calls = ['step_bits']
                elif v == 3:
                    calls = ['step_plain']              # a plain torch buffer: the step keeps the uncapped instance
                elif var & 8 and fs > 1:
                    calls = ['step_bits']               # frame stacks: step_many is T single steps (variant 8)
                elif var & 8:
                    calls = ['step_bits', 'many_every', 'step_bits', 'many_last']
                else:
                    calls = ['many_every', 'many_last']
                knobs = {'SNK_COOP': str(coop), 'SNK_TILE_ENVS': str(32 // tile_group(kw['num_snakes'])) if coop else None,
                         'SNK_BIGREG_TILES': '1' if var == 3 else None}
                idx = len(recipes)
                recipes[key] = dict(
                    id=f"{name}-{'coop' if coop else 'warp'}-v{var}", shape=name, kw=dict(kw, max_episode_steps=MAX_STEPS),
                    N=N, coop=coop, var=var, pool=bool(var & 4), grid=bool(var & 8), knobs=knobs, calls=calls,
                    bits=var in (1, 5, 10, 14), seed=idx + 1, offset=OFFSETS[idx % len(OFFSETS)],
                    # REG warp-private: once more with the observation 8 bytes off a 16-byte boundary (no vec16, no
                    # viewer-pair encode); only the variants that write the NHWC block
                    unaligned=enc == ENC_REG and not coop and var not in (1, 5),
                    reset_key=spec + (coop, enc, reset_variant(var)))
    return recipes


RECIPES = make_recipes()

# the kernels other than snk_tile_kernel, by the name the witness gives them, and the test that launches each
OTHER_KERNELS = {
    'init_records': 'test_gpu_other_kernels_match_oracle',
    'get_state': 'test_gpu_instance_matches_oracle',
    'set_state': 'test_gpu_other_kernels_match_oracle',
    'pack_obs': 'test_gpu_other_kernels_match_oracle',
    'snapshot<u32>': 'test_gpu_instance_matches_oracle',
    'restore<u32>': 'test_gpu_instance_matches_oracle',
    'emit_stacked': 'test_gpu_instance_matches_oracle',          # the restores of the frame-stack (cfg3) recipes
}
EXEMPT = {
    'snapshot<u64>': 'only a launch of more than about 2^32 16-byte units of slots selects it: tens of GB of snapshots',
    'restore<u64>': 'only a launch of more than about 2^32 16-byte units of slots selects it: tens of GB of snapshots',
}


# ---------------------------------------------------------------------------------------------------- CPU part
def library_kernels():
    """(tile-kernel keys, names of the other kernels) of the in-tree libsnk.so, from cuobjdump."""
    if not shutil.which('cuobjdump'):
        pytest.skip('cuobjdump not on PATH')
    from test_abi_cpu import _tile_kernels
    import marl_snake_b200 as m
    out = subprocess.run(['cuobjdump', '-res-usage', m.LIB_PATH], capture_output=True, text=True, timeout=300).stdout
    others = set()
    for name, targ in re.findall(r'Function _ZN3snk\d+snk_([a-z_]+)_kernel(I[jm]E)?E', out):
        others.add(name + {'': '', 'IjE': '<u32>', 'ImE': '<u64>'}[targ])
    return set(_tile_kernels()), others


def test_every_instance_has_a_recipe():
    tiles, others = library_kernels()
    missing = sorted(tiles - set(RECIPES))
    extra = sorted(set(RECIPES) - tiles)
    assert not missing, f'instances of libsnk.so without a recipe: {missing}'
    assert not extra, f'recipes for instances libsnk.so does not contain: {extra}'
    for key, r in RECIPES.items():
        assert r['reset_key'] in tiles, (r['id'], r['reset_key'])
    assert not set(OTHER_KERNELS) & set(EXEMPT)
    assert others == set(OTHER_KERNELS) | set(EXEMPT), (sorted(others ^ (set(OTHER_KERNELS) | set(EXEMPT))))


def test_recipes_are_ragged_and_reach_every_rule():
    for key, r in RECIPES.items():
        N, ns = r['N'], r['kw']['num_snakes']
        epw = 32 // tile_group(ns)
        per_cta = epw if r['coop'] else 4 * epw
        assert N % per_cta, (r['id'], N, per_cta)
        if r['coop'] and r['kw'].get('frame_stack', 1) == 1:
            assert N % epw                              # the tiles of step_many (SNK_MANY_TILE_ENVS) too
    assert {r['offset'] for r in RECIPES.values()} == set(OFFSETS)
    assert any(r['unaligned'] for r in RECIPES.values())
    assert {tuple(r['calls']) for r in RECIPES.values() if r['var'] in (10, 14) and r['kw'].get('frame_stack', 1) == 1} \
        == {('step_bits', 'many_every', 'step_bits', 'many_last')}


# ---------------------------------------------------------------------------------------------------- the witness
def parse_kernel(name):
    """('tile', key) or ('other', name) for a demangled libsnk kernel name, None for anything else."""
    m = re.search(r'snk_tile_kernel<([^<>]*)>', name)
    if m:
        args = [a.strip().replace('(bool)', '') for a in m.group(1).split(',')]
        return 'tile', tuple({'false': 0, 'true': 1}[a] if a in ('false', 'true') else int(a) for a in args)
    m = re.search(r'snk_([a-z_]+)_kernel(?:<([a-z ]+)>)?', name)
    if m:
        targ = m.group(2)
        suffix = '' if targ is None else '<u32>' if targ.strip() == 'unsigned int' else '<u64>'
        return 'other', m.group(1) + suffix
    return None


class Launches:
    def __init__(self):
        self.tiles, self.others, self.all = [], [], []

    def expect(self, tiles, others=(), what=''):
        assert self.tiles == list(tiles) and sorted(self.others) == sorted(others), \
            (what, 'launched', self.tiles, self.others, 'expected', list(tiles), list(others), 'CUDA activity', self.all)


@contextmanager
def witness():
    """Records the kernels launched inside the block (CUPTI through torch.profiler).  A profile without any CUDA
    activity fails the test, and every expectation names at least one libsnk kernel: a record the profiler drops can
    only fail a check, never pass one.

    Use it early in a process: on a B200, once test_gpu_parity's tile-mode tests had run in the same process, later
    sessions recorded only synchronous copies and none of the kernels launched inside them.  A test that runs after
    other GPU work witnesses its launches in a fresh process (see witnessed_tiles)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    rec = Launches()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        yield rec
        torch.cuda.synchronize()
    evs = sorted((e for e in prof.events() if str(e.device_type).endswith('CUDA')), key=lambda e: e.time_range.start)
    if not evs:
        pytest.fail('torch.profiler recorded no CUDA activity, so no launch can be witnessed (is CUPTI available?)')
    for e in evs:
        rec.all.append(e.name)
        p = parse_kernel(e.name)
        if p is not None:
            (rec.tiles if p[0] == 'tile' else rec.others).append(p[1])


def witnessed_tiles(code, timeout=600):
    """Runs `code` in a fresh Python process with this one's environment and sys.path; `code` prints one JSON line,
    e.g. the tile keys a witness recorded.  Returns what it printed, parsed."""
    import json
    import os
    import sys
    prelude = f'import sys\nsys.path[:0] = {[p for p in sys.path if p and os.path.isdir(p)]!r}\n'
    out = subprocess.run([sys.executable, '-c', prelude + code], capture_output=True, text=True, timeout=timeout)
    assert out.returncode == 0, out.stderr[-4000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


# ---------------------------------------------------------------------------------------------------- the model
class PoolOracleEnv(OracleSnakeEnv):
    """An oracle env of a wall-map pool: every reset starts on the map pool_next names (test_gpu_map_pool's model)."""

    def reset(self):
        self.pool_cur[self.pool_e] = self.pool_next[self.pool_e]
        self.wall_map = self.pool_walls[self.pool_cur[self.pool_e]]
        return super().reset()


class PoolShard(OracleShard):
    def __init__(self, N, kw, seed, env_id_offset, maps):
        super().__init__(N, kw, seed, env_id_offset)
        self.walls = (np.asarray(maps) != 0).astype(np.int64)
        self.next = np.array([(env_id_offset + e) % len(maps) for e in range(N)], np.int64)
        self.cur = self.next.copy()
        kw = dict(kw)
        kw.pop('done_mode', None)
        self.envs = []
        for e in range(N):
            env = PoolOracleEnv(draws=self.draws[e], wall_map=self.walls[self.cur[e]], **kw)
            env.pool_walls, env.pool_next, env.pool_cur, env.pool_e = self.walls, self.next, self.cur, e
            self.envs.append(env)


def pool_maps(H, W, M=3):
    """The walled box and M - 1 boxes with a few walls inside (deterministic per shape)."""
    rng = np.random.RandomState(H * 1000 + W)
    maps = []
    for m in range(M):
        b = np.ones((H, W), np.uint8)
        b[1:-1, 1:-1] = rng.rand(H - 2, W - 2) < (0.03 if m else 0.0)
        maps.append(b)
    return np.stack(maps)


# ---------------------------------------------------------------------------------------------------- GPU driver
class Driver:
    """One SnakeBatch built as a recipe says, its oracle model, and the calls of the recipe, every one witnessed and
    compared with the model."""

    def __init__(self, r):
        import torch
        from marl_snake_b200 import SnakeBatch
        self.torch, self.r = torch, r
        kw, N = r['kw'], r['N']
        extra = {}
        if r['pool']:
            self.maps = pool_maps(kw['height'], kw['width'])
            extra['wall_maps'] = self.maps
            self.model = PoolShard(N, kw, r['seed'], r['offset'], self.maps)
        else:
            self.model = OracleShard(N, kw, r['seed'], r['offset'])
        self.b = SnakeBatch(N, seed=r['seed'], env_id_offset=r['offset'], global_state=r['grid'], **kw, **extra)
        self.N, self.ns = N, self.b.num_snakes
        self.key = next(k for k, v in RECIPES.items() if v is r)
        self.rng = np.random.RandomState(r['seed'])
        self.gen = torch.Generator(device=self.b.device)
        self.gen.manual_seed(r['seed'])
        self.T = itertools.cycle([3, 5, 4])
        self.state_witnessed = False

    # -- comparisons
    def check_step(self, tag, want, rew, done, fin, info=None):
        mo, mr, md, mf, mi = want
        assert np.array_equal(rew, mr), ('rewards', tag)
        assert np.array_equal(np.asarray(done).astype(bool), md), ('dones', tag)
        assert np.array_equal(np.asarray(fin).astype(bool), mf), ('finished', tag)
        for k, v in (info or {}).items():
            assert np.array_equal(np.asarray(v)[mf], mi[k][mf]), (k, tag)

    def check_grid(self, tag, got, model=None):
        model = model or self.model
        assert np.array_equal(np.asarray(got), np.stack([e.grid for e in model.envs])), ('global state', tag)

    def check_state(self, tag):
        if not self.state_witnessed:
            with witness() as w:
                st = self.b.get_state()
            w.expect([], ['get_state'], ('get_state', tag))
            self.state_witnessed = True
        else:
            st = self.b.get_state()
        ex = self.model.export()
        for k in ('grid', 'alive', 'length', 'alive_counter', 'episode_length'):
            assert np.array_equal(st[k].cpu().numpy(), ex[k]), (k, tag)
        if self.r['pool']:
            assert np.array_equal(self.b.current_maps.cpu().numpy(), self.model.cur), ('current_maps', tag)

    def info_np(self, info):
        return {k: info[k].cpu().numpy() for k in ('rank', 'episode_scores', 'episode_steps', 'episode_fruits',
                                                     'episode_kills')}

    def actions(self, T=None):
        shape = (self.N, self.ns) if T is None else (T, self.N, self.ns)
        a = self.rng.randint(0, 3, size=shape).astype(np.uint8)
        return a, self.torch.as_tensor(a).cuda()

    def draw_next_maps(self):
        if self.r['pool']:
            self.b.next_maps.random_(0, len(self.maps), generator=self.gen)
            self.model.next[:] = self.b.next_maps.cpu().numpy()

    # -- calls
    def reset(self):
        torch, b = self.torch, self.b
        want = self.model.reset()
        with witness() as w:
            out = b.reset(bits=self.r['bits'])
        w.expect([self.r['reset_key']], (), 'reset')
        got = out.cpu().numpy()
        assert np.array_equal(got, packbits(want) if self.r['bits'] else want), 'reset'
        if self.r['grid']:
            self.check_grid('reset', b.global_state.cpu().numpy())
        self.check_state('reset')

    def abi_step(self, tag, obs_offset=0):
        """One step through the C ABI (snk_step_grid) into plain torch buffers, the observation obs_offset bytes into
        its allocation."""
        torch, b, N, ns = self.torch, self.b, self.N, self.ns
        from marl_snake_b200._lib import SnkStepExtra, check, lib
        dev = b.device
        env_bytes = int(np.prod(b.obs_shape))
        raw = torch.full((N * env_bytes + 16,), 0xAB, dtype=torch.uint8, device=dev)
        obs = raw[obs_offset:obs_offset + N * env_bytes].view((N,) + b.obs_shape)
        assert obs.data_ptr() % 16 == obs_offset % 16
        grid = torch.full((N,) + b.grid_shape, 0xAB, dtype=torch.uint8, device=dev) if self.r['grid'] else None
        rew = torch.full((N, ns), 7.0, dtype=torch.float64, device=dev)
        done = torch.full((N, ns), 7, dtype=torch.uint8, device=dev)
        fin = torch.full((N,), 7, dtype=torch.uint8, device=dev)
        info = dict(rank=torch.zeros((N, ns), dtype=torch.int32, device=dev),
                    episode_scores=torch.zeros((N, ns), dtype=torch.float64, device=dev),
                    episode_steps=torch.zeros((N, ns), dtype=torch.int32, device=dev),
                    episode_fruits=torch.zeros((N, ns), dtype=torch.int32, device=dev),
                    episode_kills=torch.zeros((N, ns), dtype=torch.int32, device=dev))
        x = SnkStepExtra(fin.data_ptr(), *(info[k].data_ptr() for k in ('rank', 'episode_scores', 'episode_steps',
                                                                          'episode_fruits', 'episode_kills')))
        self.draw_next_maps()
        a, da = self.actions()
        want = self.model.step(a)
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)  # noqa: E731
        with witness() as w:
            check(lib.snk_step_grid(b._h, ptr(da), ptr(obs), None, ptr(grid), ptr(rew), ptr(done), C.byref(x),
                                    b._stream()))
        w.expect([self.key], (), tag)
        self.check_step(tag, want, rew.cpu().numpy(), done.cpu().numpy(), fin.cpu().numpy(), self.info_np(info))
        assert np.array_equal(obs.cpu().numpy(), want[0]), ('obs', tag)
        assert (raw[:obs_offset] == 0xAB).all() and (raw[obs_offset + N * env_bytes:] == 0xAB).all(), ('outside', tag)
        if grid is not None:
            self.check_grid(tag, grid.cpu().numpy())

    def step(self, tag, kind):
        b = self.b
        self.draw_next_maps()
        a, da = self.actions()
        want = self.model.step(a)
        with witness() as w:
            out, rew, done, info = (b.step_bits if kind == 'step_bits' else b.step)(da)
        w.expect([self.key], (), tag)
        self.check_step(tag, want, rew.cpu().numpy(), done.cpu().numpy(), info['finished'].cpu().numpy(),
                        self.info_np(info))
        got = out.cpu().numpy()
        assert np.array_equal(got, packbits(want[0]) if kind == 'step_bits' else want[0]), ('obs', tag)
        if self.r['grid']:
            self.check_grid(tag, b.global_state.cpu().numpy())

    def step_many(self, tag, every, obs_offset=0):
        torch, b, N = self.torch, self.b, self.N
        dev = b.device
        T = next(self.T)
        lead = (T, N) if every else (N,)
        env_bytes = int(np.prod(b.obs_shape))
        n_obs = int(np.prod(lead)) * env_bytes
        raw = torch.full((n_obs + 16,), 0xAB, dtype=torch.uint8, device=dev)
        obs = raw[obs_offset:obs_offset + n_obs].view(lead + b.obs_shape)
        bits = torch.full(lead + b.bits_shape, 0xAB, dtype=torch.uint8, device=dev)
        grid = torch.full((T, N) + b.grid_shape, 0xAB, dtype=torch.uint8, device=dev) if self.r['grid'] and every \
            else None
        fin = torch.full((T, N), 7, dtype=torch.uint8, device=dev)
        self.draw_next_maps()
        a, da = self.actions(T)
        wants, grids = [], []
        for t in range(T):
            wants.append(self.model.step(a[t]))
            grids.append(np.stack([e.grid for e in self.model.envs]))
        with witness() as w:
            o, r, d, bt = b.step_many(da, obs=obs, bits=bits, finished=fin, global_state=grid)
        w.expect([self.key], (), tag)
        r, d, f = r.cpu().numpy(), d.cpu().numpy(), fin.cpu().numpy()
        o, bt = o.cpu().numpy(), bt.cpu().numpy()
        for t in range(T):
            self.check_step(tag + (t,), wants[t], r[t], d[t], f[t])
        if every:
            g = grid.cpu().numpy() if grid is not None else None
            for t in range(T):
                assert np.array_equal(o[t], wants[t][0]), ('step_many obs', tag, t)
                assert np.array_equal(bt[t], packbits(wants[t][0])), ('step_many bits', tag, t)
                if g is not None:
                    assert np.array_equal(g[t], grids[t]), ('step_many global state', tag, t)
        else:
            assert np.array_equal(o, wants[-1][0]), ('step_many last obs', tag)
            assert np.array_equal(bt, packbits(wants[-1][0])), ('step_many last bits', tag)
        assert (raw[:obs_offset] == 0xAB).all() and (raw[obs_offset + n_obs:] == 0xAB).all(), ('outside', tag)
        if self.r['grid']:
            self.check_grid(tag, b.global_state.cpu().numpy())
        return wants

    def call(self, kind, tag):
        if kind in ('step', 'step_bits'):
            self.step(tag, kind)
        elif kind == 'step_plain':
            self.abi_step(tag)
        else:
            self.step_many(tag, every=kind == 'many_every')
        self.check_state(tag)

    def restore(self, snap, saved):
        """Every env from the snapshot taken earlier, into outputs filled with a byte no observation holds."""
        torch, b, r = self.torch, self.b, self.r
        fs = r['kw'].get('frame_stack', 1)
        buf = b._bits_buffer() if r['bits'] else b._obs
        buf.fill_(0xAB)
        if r['grid']:
            b.global_state.fill_(0xAB)
        src = torch.arange(self.N, dtype=torch.int32, device=b.device)
        with witness() as w:
            out = b.restore(snap, src, bits=r['bits'])
        if fs == 1:      # MODE_ENCODE through the handle's own instance
            w.expect([r['reset_key']], ['restore<u32>'], 'restore')
        else:            # the frame history widened as it stands
            w.expect([], ['restore<u32>', 'emit_stacked'], 'restore')
        self.model = saved
        want = saved.obs()
        assert np.array_equal(out.cpu().numpy(), packbits(want) if r['bits'] else want), 'restore output'
        if r['grid']:
            self.check_grid('restore', b.global_state.cpu().numpy())
        self.check_state('restore')

    def run(self):
        r = self.r
        self.reset()
        calls = r['calls']
        n = 8 if r['N'] > 10 else 6
        snap = saved = None
        for j in range(n):
            if j == n // 2:
                with witness() as w:
                    snap = self.b.snapshot()
                w.expect([], ['snapshot<u32>'], 'snapshot')
                saved = copy.deepcopy(self.model)
            self.call(calls[j % len(calls)], (r['id'], j, calls[j % len(calls)]))
        self.restore(snap, saved)
        for j in range(2):                                      # the restored episodes continue
            self.call(calls[j % len(calls)], (r['id'], 'restored', j))
        if r['unaligned']:
            if r['var'] & 3 == 2:
                self.step_many((r['id'], '+8'), every=True, obs_offset=8)
            else:
                self.abi_step((r['id'], '+8'), obs_offset=8)
            self.check_state((r['id'], '+8'))
        assert self.b.device_errors() == 0


def set_knobs(monkeypatch, knobs):
    import os
    for k in [k for k in os.environ if k.startswith('SNK_') and k != 'SNK_LIB_PATH']:
        monkeypatch.delenv(k)
    for k, v in knobs.items():
        if v is not None:
            monkeypatch.setenv(k, v)


@pytest.mark.gpu
@pytest.mark.parametrize('key', list(RECIPES), ids=[r['id'] for r in RECIPES.values()])
def test_gpu_instance_matches_oracle(monkeypatch, key):
    r = RECIPES[key]
    set_knobs(monkeypatch, r['knobs'])
    d = Driver(r)
    try:
        d.run()
    finally:
        d.b.close()


@pytest.mark.gpu
def test_gpu_other_kernels_match_oracle(monkeypatch):
    """init_records (the constructor), set_state (with the encode it launches) and pack_obs, witnessed and compared
    with the oracle; pack_obs on a block whose 16-byte units are not a multiple of four (its tail loop)."""
    import torch
    from marl_snake_b200 import SnakeBatch
    set_knobs(monkeypatch, {})
    kw = dict(height=13, width=11, num_snakes=3, snake_length=3, vision_range=3, max_episode_steps=MAX_STEPS)
    N, seed, off = 33, 77, 2 ** 32 - 5
    with witness() as w:
        b = SnakeBatch(N, seed=seed, env_id_offset=off, **kw)
    w.expect([], ['init_records'], 'constructor')
    model = OracleShard(N, kw, seed, off)
    key = (0, 0, 0, 0, 0, 1, ENC_REG, 0)                     # the default: cooperative tiles at this size
    with witness() as w:
        out = b.reset()
    w.expect([key], (), 'reset')
    assert np.array_equal(out.cpu().numpy(), model.reset())
    rng = np.random.RandomState(seed)
    for t in range(6):
        a = rng.randint(0, 3, size=(N, 3)).astype(np.uint8)
        want = model.step(a)
        o, rew, done, info = b.step(torch.as_tensor(a).cuda())
        assert np.array_equal(o.cpu().numpy(), want[0]) and np.array_equal(rew.cpu().numpy(), want[1]), t
    n_units = b._obs.numel() // 8
    assert n_units % 4
    with witness() as w:
        bits = b.pack_obs()
    w.expect([], ['pack_obs'], 'pack_obs')
    assert np.array_equal(bits.cpu().numpy(), packbits(want[0]))
    st = b.get_state(max_cells=max(2, int(b.get_state()['length'].max())))
    args = [st[k].cpu().numpy() for k in ('grid', 'alive', 'dir', 'length')] + [st['cells'].clamp(min=0).cpu().numpy()] \
        + [st[k].cpu().numpy() for k in ('alive_counter', 'episode_length')]
    want = model.set_state_roundtrip()
    b._obs.fill_(0xAB)
    with witness() as w:
        got = b.set_state(*args)
    w.expect([key], ['set_state'], 'set_state')
    assert np.array_equal(got.cpu().numpy(), want)
    for t in range(4):                                           # the episodes continue from the forced state
        a = rng.randint(0, 3, size=(N, 3)).astype(np.uint8)
        want = model.step(a)
        o, rew, done, info = b.step(torch.as_tensor(a).cuda())
        assert np.array_equal(o.cpu().numpy(), want[0]) and np.array_equal(rew.cpu().numpy(), want[1]), t
        assert np.array_equal(info['finished'].cpu().numpy(), want[3]), t
    assert b.device_errors() == 0
    b.close()


# ---------------------------------------------------------------------------------------------------- defaults
# (shape, N, output, expected (coop, variant)).  create_impl: cooperative tiles below 148 * 40 tiles of 8 envs (47 352
# envs and fewer), the uncapped instance from 24 576 warp-private tiles of 8 envs (196 601 envs and more) -- unless the
# step writes into a compressible block (step_impl), where the capped one is faster.
THRESHOLDS = [
    ('cfg5', 47352, 'batch', (1, 0)), ('cfg5', 47353, 'batch', (0, 0)),
    ('cfg2', 47352, 'batch', (1, 0)), ('cfg2', 47353, 'batch', (0, 0)),
    ('cfg5', 196600, 'plain', (0, 0)), ('cfg5', 196601, 'plain', (0, 3)), ('cfg5', 196601, 'batch', (0, 0)),
]


@pytest.mark.gpu
@pytest.mark.parametrize('shape,N,out,want', THRESHOLDS, ids=[f'{s}-{n}-{o}' for s, n, o, _ in THRESHOLDS])
def test_gpu_default_selection_at_thresholds(monkeypatch, shape, N, out, want):
    """No knobs: the instance a default batch runs on either side of each threshold, and the first CTA's and the last
    two CTAs' envs (the ragged tail) against the oracle, one model per range with its env_id_offset."""
    import torch
    from marl_snake_b200 import SnakeBatch
    from marl_snake_b200._lib import check, lib
    set_knobs(monkeypatch, {})
    kw, spec, enc, _, _ = SHAPES[shape]
    kw = dict(kw, max_episode_steps=4)
    seed, off = 3, 2 ** 32 - 40
    b = SnakeBatch(N, seed=seed, env_id_offset=off, **kw)
    coop, var = want
    if out == 'batch' and var == 0 and N > 196600 and not b.obs_compressed:
        var = 3                              # the device granted no compressible memory: a plain block after all
    env_bytes = int(np.prod(b.obs_shape))
    per_cta = 32                                              # four warps of 8 envs
    if coop:                                                  # one tile, shrunk to a 64 KB observation block
        per_cta = 8
        while per_cta * env_bytes > 64 * 1024:
            per_cta //= 2
    last = (N + per_cta - 1) // per_cta
    ranges = [(0, per_cta), ((last - 2) * per_cta, N)]
    models = [OracleShard(hi - lo, kw, seed, off + lo) for lo, hi in ranges]
    reset_var = 3 if (not coop and N > 196600) else 0         # a reset keeps the uncapped instance wherever it writes
    with witness() as w:
        o = b.reset()
    w.expect([spec + (coop, enc, reset_var)], (), 'reset')
    for (lo, hi), m in zip(ranges, models):
        assert np.array_equal(o[lo:hi].cpu().numpy(), m.reset()), ('reset', lo)
    dev = b.device
    ns = b.num_snakes
    plain = torch.empty((N,) + b.obs_shape, dtype=torch.uint8, device=dev) if out == 'plain' else None
    rew = torch.empty((N, ns), dtype=torch.float64, device=dev)
    done = torch.empty((N, ns), dtype=torch.uint8, device=dev)
    rng = np.random.RandomState(seed)
    for t in range(6):
        a = rng.randint(0, 3, size=(N, ns)).astype(np.uint8)
        da = torch.as_tensor(a).cuda()
        with witness() as w:
            if plain is None:
                o, r, d, _ = b.step(da, want_info=False)
            else:
                check(lib.snk_step(b._h, C.c_void_p(da.data_ptr()), C.c_void_p(plain.data_ptr()),
                                   C.c_void_p(rew.data_ptr()), C.c_void_p(done.data_ptr()), None, b._stream()))
                o, r, d = plain, rew, done
        w.expect([spec + (coop, enc, var)], (), ('step', t))
        for (lo, hi), m in zip(ranges, models):
            mo, mr, md, _, _ = m.step(a[lo:hi])
            assert np.array_equal(r[lo:hi].cpu().numpy(), mr), ('rewards', t, lo)
            assert np.array_equal(d[lo:hi].cpu().numpy().astype(bool), md), ('dones', t, lo)
            assert np.array_equal(o[lo:hi].cpu().numpy(), mo), ('obs', t, lo)
    assert b.device_errors() == 0
    b.close()
