"""Global state output (snk_reset_grid / snk_step_grid / snk_step_many_grid, SnakeBatch(global_state=True)): the step
kernel writes every env's grid, as cell codes, beside the observation.  Checked against the reference's recorded
grids (golden rollouts and scenarios), against the oracle in Philox mode, against get_state() at full size, and for
leaving every other output byte for byte as it was."""
import ctypes as C

import numpy as np
import pytest
import torch

from golden_util import ROLLOUTS, Rollout, load_map_spawn_tables, load_scenarios
from gpu_backend import GpuBackend
from parity_util import check_rollout_replay, check_scenario

pytestmark = pytest.mark.gpu

CFG5 = dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5)
CFG3 = dict(CFG5, frame_stack=4)
CFG4 = dict(height=64, width=64, num_snakes=16, snake_length=5, vision_range=7,
            reward_dict={'fruit': 10.0, 'kill': 1.0, 'lose': -1.0, 'win': 0.1, 'time': -0.001})


class FusedGridBackend(GpuBackend):
    """GpuBackend whose grid() is the step kernel's global-state output instead of a get_state launch."""

    def __init__(self, num_envs, kw, **a):
        super().__init__(num_envs, dict(kw, global_state=True), **a)

    def grid(self):
        _, counter, cursor = super().grid()
        return self.b.global_state.cpu().numpy().reshape(self.N, -1), counter, cursor


# how the record layout, the tile mode and the store path are forced (the library picks them per handle otherwise)
KNOBS = ['SNK_COMPACT=0,SNK_COOP=1', 'SNK_COMPACT=1,SNK_COOP=1', 'SNK_COMPACT=0,SNK_COOP=0', 'SNK_COMPACT=1,SNK_COOP=0',
         'SNK_TMA=0', 'SNK_NO_DIG=1', 'SNK_TMA=0,SNK_COMPACT=1,SNK_COOP=0']


def set_knobs(monkeypatch, knob):
    for kv in knob.split(','):
        k, v = kv.split('=')
        monkeypatch.setenv(k, v)


@pytest.mark.parametrize('knob', KNOBS)
@pytest.mark.parametrize('name', ROLLOUTS)
def test_rollout_replay_grid_equals_reference(monkeypatch, name, knob):
    set_knobs(monkeypatch, knob)
    g = Rollout(name)
    be = FusedGridBackend(g.num_envs, g.kwargs, rng_mode=1, auto_reset=1, done_mode=g.done_mode)
    check_rollout_replay(be, g)
    assert be.errors() == 0
    be.close()


@pytest.mark.parametrize('knob', KNOBS)
@pytest.mark.parametrize('sc', load_scenarios(), ids=lambda s: s.name)
def test_scenario_grid_equals_reference(monkeypatch, sc, knob):
    set_knobs(monkeypatch, knob)
    kw = dict(height=sc.H, width=sc.W, num_snakes=sc.num_snakes, snake_length=2, **sc.kwargs)
    be = FusedGridBackend(1, kw, rng_mode=1, auto_reset=0)
    check_scenario(be, sc)
    assert be.errors() == 0
    be.close()


def check_philox(kw, N, steps, seed, done_mode='all', **extra):
    """The global state after the reset and after every step (auto-resets included) against the oracle's env.grid."""
    from marl_snake_b200 import SnakeBatch
    from oracle.snake_oracle import CoopOracleSnakeEnv, OracleSnakeEnv, PhiloxDraws
    cls = CoopOracleSnakeEnv if done_mode == 'any' else OracleSnakeEnv
    b = SnakeBatch(N, seed=seed, done_mode=done_mode, global_state=True, **kw, **extra)
    draws = [PhiloxDraws(seed, e) for e in range(N)]
    envs = [cls(draws=d, **kw, **({'wall_map': extra['wall_map']} if 'wall_map' in extra else {})) for d in draws]
    for d in draws:
        d.tick()
    want = np.stack([e.reset() for e in envs])
    assert np.array_equal(b.reset().cpu().numpy(), want)
    assert np.array_equal(b.global_state.cpu().numpy(), np.stack([e.grid for e in envs])), 'reset'
    rng = np.random.RandomState(seed)
    n_act = 5 if kw.get('observer') == 'human' else 3
    resets = 0
    for t in range(steps):
        acts = rng.randint(0, n_act, size=(N, b.num_snakes)).astype(np.uint8)
        obs, rew, done, _ = b.step(torch.as_tensor(acts).cuda())
        obs = obs.cpu().numpy()
        for e, env in enumerate(envs):
            draws[e].tick()
            o, r, dn, inf = env.step([int(a) for a in acts[e]])
            if all(dn):
                o = env.reset()
                resets += 1
            assert np.array_equal(obs[e], o), (t, e)
        assert np.array_equal(b.global_state.cpu().numpy(), np.stack([e.grid for e in envs])), t
    assert resets > 0
    assert b.device_errors() == 0
    b.close()


@pytest.mark.parametrize('kw,N,extra', [
    (CFG5, 37, {}),                                                                 # cfg1 shape
    (dict(height=20, width=20, num_snakes=4, snake_length=3), 21, {}),               # full-grid observation
    (CFG3, 19, {}),                                                                 # frame_stack 4
    (dict(height=14, width=11, num_snakes=4, snake_length=3, vision_range=3, observer='human'), 23, {}),
    (dict(height=16, width=16, num_snakes=8, snake_length=3, vision_range=3), 13, {}),   # 8 snakes: direction plane
    (dict(CFG5, max_episode_steps=15), 17, dict(done_mode='any')),
    (dict(height=10, width=14, num_snakes=3, snake_length=3, vision_range=2, max_episode_steps=20), 29, {}),  # H*W = 140
], ids=['cfg1', 'full_grid', 'fs4', 'human', 'ns8_plane', 'done_any', 'rect_10x14'])
def test_philox_grid_matches_oracle(kw, N, extra):
    check_philox(dict(kw, max_episode_steps=kw.get('max_episode_steps', 25)), N, 60, seed=71, **extra)


def test_philox_grid_matches_oracle_asset_map():
    walls = np.asarray(load_map_spawn_tables()['12x12'][0] != 0, dtype=np.uint8)
    kw = dict(height=12, width=12, num_snakes=3, snake_length=3, vision_range=3, max_episode_steps=12)
    check_philox(kw, 15, 50, seed=5, wall_map=walls)


def full_state_args(b, max_cells):
    st = b.get_state(max_cells=max_cells)
    args = [st[k].cpu().numpy() for k in ('grid', 'alive', 'dir', 'length', 'cells', 'alive_counter')]
    args[4] = np.maximum(args[4], 0)
    return args


def assert_grid_is_state(b, what):
    assert torch.equal(b.global_state, b.get_state()['grid']), what


@pytest.mark.parametrize('kw,N', [(CFG5, 1 << 20), (CFG3, 65536), (CFG4, 16384)], ids=['cfg5', 'cfg3', 'cfg4'])
def test_full_size_grid_equals_get_state(kw, N):
    from marl_snake_b200 import SnakeBatch
    b = SnakeBatch(N, seed=3, max_episode_steps=15, global_state=True, **kw)
    b.reset()
    assert_grid_is_state(b, 'reset')
    g = torch.Generator(device='cuda').manual_seed(1)
    ns = b.num_snakes
    finished = 0
    for t in range(20):
        a = torch.randint(0, 3, (N, ns), dtype=torch.uint8, device='cuda', generator=g)
        _, _, _, info = b.step(a)
        finished += int(info['finished'].sum())
        assert_grid_is_state(b, ('step', t))
    assert finished > 0                                   # steps with auto-resets
    mask = torch.zeros(N, dtype=torch.uint8, device='cuda')
    mask[::7] = 1
    b.reset(mask=mask)
    assert_grid_is_state(b, 'masked reset')
    args = full_state_args(b, max(int(b.get_state()['length'].max()), 2))
    b.step(torch.randint(0, 3, (N, ns), dtype=torch.uint8, device='cuda', generator=g))
    b.set_state(*args)
    assert np.array_equal(b.global_state.cpu().numpy(), args[0])
    assert_grid_is_state(b, 'set_state')
    assert b.device_errors() == 0
    b.close()


@pytest.mark.parametrize('kw,N', [(CFG5, 1 << 20), (CFG3, 65536)], ids=['cfg5', 'cfg3'])
def test_other_outputs_are_unchanged(kw, N):
    from marl_snake_b200 import SnakeBatch
    a = SnakeBatch(N, seed=12, max_episode_steps=12, global_state=True, **kw)
    b = SnakeBatch(N, seed=12, max_episode_steps=12, **kw)
    assert b.global_state is None
    assert torch.equal(a.reset(), b.reset())
    g = torch.Generator(device='cuda').manual_seed(7)
    for t in range(16):
        act = torch.randint(0, 3, (N, 4), dtype=torch.uint8, device='cuda', generator=g)
        oa, ra, da, ia = a.step(act)
        ob, rb, db, ib = b.step(act)
        assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(da, db), t
        for k in ia:
            assert torch.equal(ia[k], ib[k]), (k, t)
    assert torch.equal(a.global_state, b.get_state()['grid'])
    assert a.device_errors() == 0 and b.device_errors() == 0


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


@pytest.mark.parametrize('knob', ['', 'SNK_COMPACT=0,SNK_COOP=0', 'SNK_COMPACT=1,SNK_COOP=1', 'SNK_TMA=0'])
@pytest.mark.parametrize('fs', [1, 2])
def test_every_combination_of_outputs(monkeypatch, knob, fs):
    """grid only, obs + grid, bits + grid and obs + bits + grid through the C ABI, against a twin batch's step()."""
    from marl_snake_b200 import SnakeBatch
    from marl_snake_b200._lib import check, lib
    if knob:
        set_knobs(monkeypatch, knob)
    N, ns = 1500, 4
    kw = dict(CFG5, frame_stack=fs, max_episode_steps=9, seed=4)
    a, b = SnakeBatch(N, **kw), SnakeBatch(N, **kw)
    H, W = a.grid_shape
    obs = torch.empty((N,) + a.obs_shape, dtype=torch.uint8, device='cuda')
    bits = torch.empty((N,) + a.bits_shape, dtype=torch.uint8, device='cuda')
    grid = torch.empty((N, H, W), dtype=torch.uint8, device='cuda')
    rew = torch.empty((N, ns), dtype=torch.float64, device='cuda')
    done = torch.empty((N, ns), dtype=torch.uint8, device='cuda')
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    combos = [(False, False), (True, False), (False, True), (True, True)]
    for k, (want_obs, want_bits) in enumerate(combos):
        grid.fill_(0xEE)
        check(lib.snk_reset_grid(a._h, None, _p(obs if want_obs else None), _p(bits if want_bits else None), _p(grid), s))
        want = b.reset(copy=True)
        assert torch.equal(grid, a.get_state()['grid']), ('reset', k)
        if want_obs:
            assert torch.equal(obs, want), ('reset obs', k)
        if want_bits:
            assert torch.equal(bits, b.pack_obs(want)), ('reset bits', k)
    g = torch.Generator(device='cuda').manual_seed(2)
    for t in range(24):
        want_obs, want_bits = combos[t % 4]
        act = torch.randint(0, 3, (N, ns), dtype=torch.uint8, device='cuda', generator=g)
        grid.fill_(0xEE)
        check(lib.snk_step_grid(a._h, _p(act), _p(obs if want_obs else None), _p(bits if want_bits else None), _p(grid),
                                _p(rew), _p(done), None, s))
        o, r, d, _ = b.step(act)
        assert torch.equal(rew, r) and torch.equal(done.bool(), d), t
        assert torch.equal(grid, b.get_state()['grid']), t
        if want_obs:
            assert torch.equal(obs, o), t
        if want_bits:
            assert torch.equal(bits, b.pack_obs(o)), t
    assert a.device_errors() == 0 and b.device_errors() == 0


@pytest.mark.parametrize('kw', [CFG5, dict(height=10, width=14, num_snakes=3, snake_length=3, vision_range=2)],
                         ids=['cfg5', 'rect_10x14'])
@pytest.mark.parametrize('offset', [1, 4, 8])
def test_unaligned_caller_buffer(kw, offset):
    from marl_snake_b200 import SnakeBatch
    from marl_snake_b200._lib import check, lib
    N = 3000
    b = SnakeBatch(N, seed=6, max_episode_steps=10, **kw)
    ns, (H, W) = b.num_snakes, b.grid_shape
    raw = torch.full((N * H * W + 64,), 0xEE, dtype=torch.uint8, device='cuda')
    grid = raw[offset:offset + N * H * W]
    assert grid.data_ptr() % 16 == offset % 16
    rew = torch.empty((N, ns), dtype=torch.float64, device='cuda')
    done = torch.empty((N, ns), dtype=torch.uint8, device='cuda')
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    check(lib.snk_reset_grid(b._h, None, None, None, _p(grid), s))
    assert torch.equal(grid.view(N, H, W), b.get_state()['grid'])
    g = torch.Generator(device='cuda').manual_seed(offset)
    for t in range(15):
        act = torch.randint(0, 3, (N, ns), dtype=torch.uint8, device='cuda', generator=g)
        check(lib.snk_step_grid(b._h, _p(act), _p(b._obs), None, _p(grid), _p(rew), _p(done), None, s))
        assert torch.equal(grid.view(N, H, W), b.get_state()['grid']), t
    assert bool((raw[:offset] == 0xEE).all()) and bool((raw[offset + N * H * W:] == 0xEE).all())   # nothing outside
    assert b.device_errors() == 0


@pytest.mark.parametrize('knob', ['', 'SNK_COMPACT=0,SNK_COOP=1', 'SNK_COMPACT=1,SNK_COOP=1', 'SNK_TMA=0'])
@pytest.mark.parametrize('fs', [1, 4])
def test_step_many_equals_single_steps(monkeypatch, knob, fs):
    """Every-step and last-only grid output of step_many against T single steps: one launch at frame_stack 1, T
    launches at frame_stack 4.  The batch's own global_state follows either way."""
    from marl_snake_b200 import SnakeBatch
    if knob:
        set_knobs(monkeypatch, knob)
    N, T = 700, 13
    kw = dict(CFG5, frame_stack=fs, max_episode_steps=5, seed=9, global_state=True)
    a, b, c = SnakeBatch(N, **kw), SnakeBatch(N, **kw), SnakeBatch(N, **kw)
    H, W = a.grid_shape
    for x in (a, b, c):
        x.reset()
    acts = torch.randint(0, 3, (T, N, 4), dtype=torch.uint8, device='cuda',
                         generator=torch.Generator(device='cuda').manual_seed(3))
    every = torch.empty((T, N, H, W), dtype=torch.uint8, device='cuda')
    obs = torch.empty((T, N) + a.obs_shape, dtype=torch.uint8, device='cuda')
    _, rew, done, _ = a.step_many(acts, obs=obs, global_state=every)
    last = torch.empty((N, H, W), dtype=torch.uint8, device='cuda')
    _, rew_c, _, _ = c.step_many(acts, global_state=last)
    for t in range(T):
        o, r, d, _ = b.step(acts[t])
        assert torch.equal(every[t], b.global_state), t
        assert torch.equal(obs[t], o) and torch.equal(rew[t], r) and torch.equal(done[t], d.to(torch.uint8)), t
    assert torch.equal(last, b.global_state) and torch.equal(rew_c, rew)
    assert torch.equal(a.global_state, b.global_state) and torch.equal(c.global_state, b.global_state)
    # no caller tensor: the last step's rows go straight to the batch's buffer
    more = torch.randint(0, 3, (T, N, 4), dtype=torch.uint8, device='cuda', generator=torch.Generator(device='cuda').manual_seed(4))
    a.step_many(more)
    for t in range(T):
        b.step(more[t])
    assert torch.equal(a.global_state, b.global_state)
    assert_grid_is_state(a, 'step_many without outputs')
    for x in (a, b, c):
        assert x.device_errors() == 0


@pytest.mark.parametrize('compact', ['0', '1'])
def test_wall_map_pool_rows_carry_the_current_maps_walls(monkeypatch, compact):
    from marl_snake_b200 import SnakeBatch
    from test_gpu_map_pool import maps20
    monkeypatch.setenv('SNK_COMPACT', compact)
    maps, N = maps20(), 96
    b = SnakeBatch(N, wall_maps=maps, seed=2, max_episode_steps=6, global_state=True, **CFG5)
    lay = torch.as_tensor(maps).cuda()
    b.reset()
    gen = torch.Generator(device='cuda').manual_seed(8)
    switched = 0
    for t in range(30):
        before = b.current_maps.clone()
        b.next_maps.random_(0, len(maps), generator=gen)
        b.step(torch.randint(0, 3, (N, 4), dtype=torch.uint8, device='cuda', generator=gen))
        switched += int((b.current_maps != before).sum())
        walls = (b.global_state % 10 == 1).to(torch.uint8)
        assert torch.equal(walls, lay[b.current_maps.long()]), t
        assert_grid_is_state(b, t)
    assert switched > 0
    assert b.device_errors() == 0


def test_graph_replay_and_stale_calls():
    from marl_snake_b200 import GraphedSteps, SnakeBatch
    N, T = 4096, 8
    kw = dict(CFG5, seed=5, max_episode_steps=7, global_state=True)
    a, b = SnakeBatch(N, **kw), SnakeBatch(N, **kw)
    a.reset(); b.reset()
    acts = torch.randint(0, 3, (T, N, 4), dtype=torch.uint8, device='cuda',
                         generator=torch.Generator(device='cuda').manual_seed(1))
    gs = GraphedSteps(a, acts)
    for rep in range(2):
        gs.replay()
        for t in range(T):
            b.step(acts[t], want_info=False)
        torch.cuda.synchronize()
        assert torch.equal(a.global_state, b.global_state), rep
        assert_grid_is_state(a, ('graph', rep))
    # calls that do not write the buffer themselves leave it current all the same
    blob = b.save_checkpoint()
    b.step(acts[0])
    b.load_checkpoint(blob)
    assert torch.equal(b.global_state, a.global_state)
    assert_grid_is_state(b, 'load_checkpoint')
    obs = torch.empty((N,) + b.obs_shape, dtype=torch.uint8).pin_memory()
    rew = torch.empty((N, 4), dtype=torch.float64).pin_memory()
    done = torch.empty((N, 4), dtype=torch.uint8).pin_memory()
    b.step_host(acts[1].cpu(), obs, rew, done)
    a.step(acts[1])
    assert torch.equal(b.global_state, a.global_state)
    assert_grid_is_state(b, 'step_host')
    b.reset_host(obs)
    assert_grid_is_state(b, 'reset_host')
    assert a.device_errors() == 0 and b.device_errors() == 0
