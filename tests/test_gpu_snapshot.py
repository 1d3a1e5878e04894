"""Per-env snapshot / restore on the device (snk_snapshot / snk_restore, SnakeBatch.snapshot / restore): a rewind
continues bit for bit, a partial restore touches only the restored envs' rows, one slot fans out to every env and then
follows the oracle started from the source's state on each destination's own Philox stream, slots move between handles
of one configuration and are refused by others, and the calls behave in CUDA graphs and beside the host-buffer calls."""
import copy
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

CFG5 = dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5, max_episode_steps=12)
CFG4 = dict(height=64, width=64, num_snakes=16, snake_length=5, vision_range=7, max_episode_steps=12,
            reward_dict={'fruit': 10.0, 'kill': 1.0, 'lose': -1.0, 'win': 0.1, 'time': -0.001})


def pool_maps():
    m = np.zeros((3, 20, 20), np.uint8)
    m[:, 0, :] = m[:, -1, :] = m[:, :, 0] = m[:, :, -1] = 1
    m[1, 5:15, 10] = 1
    m[2, 10, 3:17] = 1
    return m


# name: (SnakeBatch kwargs, num_envs, forced knobs)
SHAPES = {
    'cfg5_warp_private': (CFG5, 70, 'SNK_COOP=0'),                                  # compact records, warp-private tiles
    'coop_full_dig': (CFG5, 37, 'SNK_COOP=1,SNK_COMPACT=0'),                        # full records, directions in the grid
    'coop_full_plane': (CFG5, 37, 'SNK_COOP=1,SNK_COMPACT=0,SNK_NO_DIG=1'),         # full records, direction plane
    'fs4': (dict(CFG5, frame_stack=4), 19, ''),
    'enc_pad': (CFG4, 5, ''),
    'full_grid': (dict(CFG5, vision_range=None), 21, ''),
    'human': (dict(height=14, width=11, num_snakes=4, snake_length=3, vision_range=3, observer='human',
                   max_episode_steps=12), 23, ''),
    'done_any': (dict(CFG5, done_mode='any'), 17, ''),
    'pool': (dict(CFG5, wall_maps=pool_maps()), 29, ''),
}
TILE_KNOBS = ['', 'SNK_COOP=0', 'SNK_COOP=1', 'SNK_TMA=0']


def set_knobs(monkeypatch, *knobs):
    for knob in knobs:
        for kv in filter(None, knob.split(',')):
            k, v = kv.split('=')
            monkeypatch.setenv(k, v)


def make(name, monkeypatch, knob='', **extra):
    kw, N, forced = SHAPES[name]
    set_knobs(monkeypatch, forced, knob)
    from marl_snake_b200 import SnakeBatch
    return SnakeBatch(N, global_state=True, **dict(kw, **extra))


def plan(b, steps, seed=5):
    """Actions and next_maps for every step (next_maps rewritten before each step when the batch has a pool)."""
    g = torch.Generator(device=b.device).manual_seed(seed)
    n_act = 5 if b.observer == 'human' else 3
    acts = torch.randint(0, n_act, (steps, b.num_envs, b.num_snakes), dtype=torch.uint8, device=b.device, generator=g)
    maps = torch.randint(0, max(b.num_maps, 1), (steps, b.num_envs), dtype=torch.uint8, device=b.device, generator=g)
    return acts, maps


def state(b):
    st = b.get_state(max_cells=8)
    return {k: v.clone() for k, v in st.items()}


def run(b, acts, maps, t0, T):
    """T steps from step t0: every output, the info arrays, the global state and get_state after each."""
    out = []
    for t in range(t0, t0 + T):
        if b.num_maps:
            b.next_maps.copy_(maps[t])
        obs, rew, done, info = b.step(acts[t], copy=True)
        fin = info['finished']
        # terminal info of envs that did not finish is unspecified (whatever an earlier step left there)
        info = {k: v if k == 'finished' else v * fin.view(-1, *([1] * (v.dim() - 1))).to(v.dtype) for k, v in info.items()}
        out.append(dict(obs=obs, bits=b.pack_obs(obs), rew=rew, done=done, grid=b.global_state.clone(),
                        **{'info_' + k: v for k, v in info.items()}, **{'st_' + k: v for k, v in state(b).items()}))
    return out


def assert_same(a, b, what):
    for t, (x, y) in enumerate(zip(a, b)):
        for k in x:
            assert torch.equal(x[k], y[k]), (what, t, k)


def rewind(b, k=7, T=14):
    acts, maps = plan(b, k + T)
    b.reset()
    at_k = run(b, acts, maps, 0, k)[-1]
    snap = b.snapshot()
    first = run(b, acts, maps, k, T)
    src = torch.arange(b.num_envs, dtype=torch.int32, device=b.device)
    obs = b.restore(snap, src, copy=True)
    assert torch.equal(obs, at_k['obs']) and torch.equal(b.global_state, at_k['grid'])
    assert torch.equal(b.restore(snap, src, bits=True), at_k['bits'])
    assert torch.equal(b.global_state, at_k['grid'])
    for key, v in state(b).items():
        assert torch.equal(v, at_k['st_' + key]), key
    assert_same(first, run(b, acts, maps, k, T), 'second run')
    assert b.device_errors() == 0


@pytest.mark.parametrize('knob', TILE_KNOBS, ids=['default', 'warp_private', 'coop', 'no_tma'])
@pytest.mark.parametrize('name', SHAPES)
def test_rewind_is_exact(monkeypatch, name, knob):
    b = make(name, monkeypatch, knob, seed=11)
    rewind(b)
    b.close()


@pytest.mark.parametrize('knob', TILE_KNOBS, ids=['default', 'warp_private', 'coop', 'no_tma'])
@pytest.mark.parametrize('name', ['cfg5_warp_private', 'fs4', 'full_grid'])
def test_rewind_is_exact_in_replay_mode(monkeypatch, name, knob):
    """The replay cursor is part of the record: after the rewind the same recorded draws are replayed again."""
    from oracle.snake_oracle import NumpyGlobalDraws, OracleSnakeEnv, RecordingDraws
    b = make(name, monkeypatch, knob, rng='replay')
    kw = {k: v for k, v in SHAPES[name][0].items()}
    steps = 7 + 14
    acts, _ = plan(b, steps)
    a = acts.cpu().numpy()
    np.random.seed(3)
    draws = [RecordingDraws(NumpyGlobalDraws()) for _ in range(b.num_envs)]
    for e, d in enumerate(draws):
        env = OracleSnakeEnv(draws=d, **kw)
        env.reset()
        for t in range(steps):
            if all(env.step([int(x) for x in a[t, e]])[2]):
                env.reset()
    b.set_replay([d.log for d in draws])
    rewind(b)
    assert np.array_equal(b.replay_cursors(), [len(d.log) for d in draws])
    b.close()


@pytest.mark.parametrize('name', SHAPES)
def test_partial_restore_touches_only_the_restored_rows(monkeypatch, name):
    b = make(name, monkeypatch, seed=2)
    N = b.num_envs
    acts, maps = plan(b, 12)
    b.reset()
    at_k = run(b, acts, maps, 0, 5)[-1]
    snap = b.snapshot()
    run(b, acts, maps, 5, 7)
    before = state(b)
    grid_before = b.global_state.clone()
    ids = torch.randperm(N, device=b.device)[:N // 3 + 1]
    sel = torch.zeros(N, dtype=torch.bool, device=b.device)
    sel[ids] = True
    for bits in (False, True):
        buf = b._bits_buffer() if bits else b._obs
        buf.fill_(0xAB)
        b.global_state.fill_(0xCD)
        out = b.restore(snap, env_ids=ids, slots=ids, bits=bits)
        want = at_k['bits'] if bits else at_k['obs']
        assert torch.equal(out[sel], want[sel]), bits
        assert bool((out[~sel] == 0xAB).all()), bits
        assert torch.equal(b.global_state[sel], at_k['grid'][sel])
        others = b.global_state[~sel]
        kept = (others == 0xCD).flatten(1).all(1) | (others == grid_before[~sel]).flatten(1).all(1)
        assert bool(kept.all())
        for key, v in state(b).items():
            assert torch.equal(v[sel], at_k['st_' + key][sel]), key
            assert torch.equal(v[~sel], before[key][~sel]), key
    assert b.device_errors() == 0
    b.close()


@pytest.mark.parametrize('name', ['cfg5_warp_private', 'coop_full_dig', 'fs4', 'human', 'done_any', 'full_grid'])
def test_fan_out_follows_the_oracle_on_each_destination_stream(monkeypatch, name):
    """One slot into every env: each env's state is the source's, and its next steps are the oracle's started from a
    deep copy of the source on the destination's own Philox stream at the source's event count.  The episode statistics
    carry over: terminal info counts the steps before the snapshot."""
    from oracle.snake_oracle import CoopOracleSnakeEnv, OracleSnakeEnv, PhiloxDraws
    seed, off = 17, 40
    b = make(name, monkeypatch, seed=seed, env_id_offset=off)
    kw = dict(SHAPES[name][0])
    cls = CoopOracleSnakeEnv if kw.pop('done_mode', 'all') == 'any' else OracleSnakeEnv
    N, k, T = b.num_envs, 6, 16
    draws = [PhiloxDraws(seed, off + e) for e in range(N)]
    envs = [cls(draws=d, **kw) for d in draws]
    for d in draws:
        d.tick()
    for env in envs:
        env.reset()
    b.reset()
    acts, _ = plan(b, k + T)
    a = acts.cpu().numpy()
    for t in range(k):
        b.step(acts[t])
        for e, env in enumerate(envs):
            draws[e].tick()
            if all(env.step([int(x) for x in a[t, e]])[2]):
                env.reset()
    src_state = state(b)
    s = int(src_state['episode_length'].argmax())          # the longest episode: its statistics have the most to carry
    snap = b.snapshot(torch.tensor([s], device=b.device))
    obs = b.restore(snap, torch.zeros(N, dtype=torch.int32, device=b.device))
    assert bool((obs == obs[s]).all()) and bool((b.global_state == b.global_state[s]).all())
    for key, v in state(b).items():
        assert bool((v == src_state[key][s]).all()), key
    clones = []
    for e in range(N):
        env = copy.deepcopy(envs[s])
        env.draws = PhiloxDraws(seed, off + e)
        env.draws.event = draws[s].event
        clones.append(env)
    carried = False
    for t in range(k, k + T):
        obs, rew, done, info = b.step(acts[t])
        obs, rew, done = obs.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy()
        fin = info['finished'].cpu().numpy()
        for e, env in enumerate(clones):
            env.draws.tick()
            o, r, dn, inf = env.step([int(x) for x in a[t, e]])
            assert bool(fin[e]) == bool(inf), (t, e)
            if inf:
                assert np.array_equal(info['episode_steps'][e].cpu().numpy(), inf['episode_steps']), (t, e)
                assert np.array_equal(info['episode_scores'][e].cpu().numpy(), inf['episode_scores']), (t, e)
                assert np.array_equal(info['episode_fruits'][e].cpu().numpy(), inf['episode_fruits']), (t, e)
                assert np.array_equal(info['episode_kills'][e].cpu().numpy(), inf['episode_kills']), (t, e)
                assert list(info['rank'][e].cpu().numpy()) == inf['rank'], (t, e)
                carried |= int(max(inf['episode_steps'])) > t - k + 1
            if all(dn):
                o = env.reset()
            assert np.array_equal(obs[e], o) and np.array_equal(rew[e], np.asarray(r)) \
                and np.array_equal(done[e], np.asarray(dn)), (t, e)
    assert carried, 'no episode ended with steps from before the snapshot'
    assert b.device_errors() == 0
    b.close()


def test_slots_move_between_handles_of_one_configuration(monkeypatch):
    from marl_snake_b200 import SnakeBatch
    from marl_snake_b200._lib import check, lib
    a = SnakeBatch(256, seed=1, global_state=True, **CFG5)
    acts, maps = plan(a, 9)
    a.reset()
    run(a, acts, maps, 0, 9)
    want_obs, want_grid, want = a._obs.clone(), a.global_state.clone(), state(a)
    snap = a.snapshot()
    b = SnakeBatch(100, seed=2, env_id_offset=1000, auto_reset=False, global_state=True,
                   reward_dict={'fruit': 1.0, 'kill': 2.0, 'lose': -3.0, 'win': 4.0, 'time': 0.0}, **CFG5)
    b.reset()
    obs = b.restore(snap, torch.arange(100, dtype=torch.int32, device=b.device) + 50)
    assert torch.equal(obs, want_obs[50:150]) and torch.equal(b.global_state, want_grid[50:150])
    for key, v in state(b).items():
        assert torch.equal(v, want[key][50:150]), key
    assert b.device_errors() == 0

    walls = np.zeros((20, 20), np.uint8)
    walls[0, :] = walls[-1, :] = walls[:, 0] = walls[:, -1] = 1
    walls[10, 5] = 1
    others = [dict(CFG5, vision_range=4),                 # another observation window
              dict(CFG5, wall_map=walls),                 # another wall layout
              dict(CFG5, max_episode_steps=70000)]        # 32-bit episode counters
    # (64 and 256 envs of this shape run cooperative tiles, whose default is the full record layout)
    for kw, knob in [(o, '') for o in others] + [(CFG5, 'SNK_COMPACT=1')]:
        monkeypatch.delenv('SNK_COMPACT', raising=False)
        set_knobs(monkeypatch, knob)
        c = SnakeBatch(64, seed=3, global_state=True, **kw)
        c.reset()
        run(c, acts[:, :64], maps[:, :64], 0, 3)
        src = torch.arange(64, dtype=torch.int32, device=c.device)
        if c.snapshot_bytes != a.snapshot_bytes:
            with pytest.raises(ValueError, match='rows of snapshot_bytes'):
                c.restore(snap, src)
        # the library itself refuses the slots, whatever their row width: a buffer of this handle's slot size, filled
        # with the other handle's slots
        buf = torch.zeros((64, c.snapshot_bytes), dtype=torch.uint8, device=c.device)
        n = min(buf.numel(), snap.numel())
        buf.view(-1)[:n] = snap.view(-1)[:n]
        before = state(c)
        c._obs.fill_(0xAB)
        c.global_state.fill_(0xCD)
        check(lib.snk_restore(c._h, C.c_void_p(src.data_ptr()), 64, C.c_void_p(buf.data_ptr()), C.c_void_p(c._obs.data_ptr()),
                              None, C.c_void_p(c.global_state.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        assert c.device_errors(clear=True) == 256, (kw, knob)
        assert bool((c._obs == 0xAB).all()) and bool(((c.global_state == 0xCD) | (c.global_state == before['grid'])).all())
        for key, v in state(c).items():
            assert torch.equal(v, before[key]), (kw, knob, key)
        c.close()
    a.close()
    b.close()


def test_error_paths(monkeypatch):
    from marl_snake_b200 import SnakeBatch
    from marl_snake_b200._lib import SnkError, lib
    b = SnakeBatch(16, seed=4, global_state=True, **CFG5)
    slot = torch.zeros((17, b.snapshot_bytes + 16), dtype=torch.uint8, device=b.device)
    p = slot.data_ptr()
    src = torch.full((16,), -1, dtype=torch.int32, device=b.device)
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.snk_snapshot(b._h, None, 1, C.c_void_p(p), s) == -4          # before the first reset
    assert lib.snk_restore(b._h, C.c_void_p(src.data_ptr()), 1, C.c_void_p(p), None, None, None, s) == -4
    acts, maps = plan(b, 4)
    b.reset()
    run(b, acts, maps, 0, 4)
    assert lib.snk_snapshot(b._h, None, 1, C.c_void_p(p + 8), s) == -1      # misaligned
    assert lib.snk_snapshot(b._h, None, 0, C.c_void_p(p), s) == -1
    assert lib.snk_snapshot(b._h, None, 17, C.c_void_p(p), s) == -1
    assert lib.snk_restore(b._h, C.c_void_p(src.data_ptr()), 0, C.c_void_p(p), None, None, None, s) == -1
    assert lib.snk_restore(b._h, C.c_void_p(src.data_ptr()), 1, C.c_void_p(p + 8), None, None, None, s) == -1
    snap = b.snapshot()
    before, obs_before, grid_before = state(b), b._obs.clone(), b.global_state.clone()
    for bad in (16, 99, -2):
        src.fill_(-1)
        src[3] = bad
        b.restore(snap, src)
        with pytest.raises(SnkError, match='snapshot'):
            b.raise_on_device_errors()
    bad_ids = b.snapshot(torch.tensor([2, 16], device=b.device))          # id 16 is outside [0, N)
    assert b.device_errors(clear=True) == 256
    b.restore(bad_ids, env_ids=torch.tensor([5], device=b.device), slots=torch.tensor([1], device=b.device))
    assert b.device_errors(clear=True) == 256
    assert torch.equal(b._obs, obs_before) and torch.equal(b.global_state, grid_before)
    for key, v in state(b).items():
        assert torch.equal(v, before[key]), key
    b.restore(bad_ids, env_ids=torch.tensor([5], device=b.device), slots=torch.tensor([0], device=b.device))
    assert b.device_errors() == 0
    assert torch.equal(b._obs[5], obs_before[2])
    b.close()


def test_graph_host_calls_and_statistics(monkeypatch):
    from marl_snake_b200 import SnakeBatch
    from marl_snake_b200._lib import lib
    b = SnakeBatch(48, seed=6, global_state=True, **CFG5)
    acts, maps = plan(b, 12)
    b.reset()
    run(b, acts, maps, 0, 8)
    snap = b.snapshot()
    src = torch.arange(48, dtype=torch.int32, device=b.device).flip(0).contiguous()
    run(b, acts, maps, 8, 3)
    stats = b.stats()
    b.restore(snap, src)
    b.snapshot(out=torch.empty_like(snap))
    torch.cuda.synchronize()
    assert b.stats() == stats                             # no step was executed
    obs, rew, done, _ = b.step(acts[11], copy=True)
    eager = (obs, rew, done, b.global_state.clone())

    # the same two calls replayed from a CUDA graph
    run(b, acts, maps, 8, 2)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            b.restore(snap, src)
            b.step(acts[11], want_info=False)
    g.replay()
    lib.snk_note_stream(b._h, C.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert torch.equal(b._obs, eager[0]) and torch.equal(b._rew, eager[1]) and torch.equal(b._done.view(torch.bool), eager[2])
    assert torch.equal(b.global_state, eager[3])

    # a host-buffer step after a restore sees the restored state
    b.restore(snap, src)
    o = np.zeros((48,) + b.obs_shape, np.uint8)
    r = np.zeros((48, 4), np.float64)
    d = np.zeros((48, 4), np.uint8)
    b.step_host(torch.from_numpy(acts[11].cpu().numpy()), torch.from_numpy(o), torch.from_numpy(r), torch.from_numpy(d))
    assert np.array_equal(o, eager[0].cpu().numpy()) and np.array_equal(r, eager[1].cpu().numpy())
    assert np.array_equal(d.astype(bool), eager[2].cpu().numpy())
    assert b.device_errors() == 0
    b.close()
