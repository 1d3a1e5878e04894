"""Wall-map pools (snk_create_maps / SnakeBatch(wall_maps=...)): every env starts each episode on the map its
`next_maps` entry names at that reset.  Checked against the Python oracle, which switches layout by setting
OracleSnakeEnv.wall_map before reset(), in Philox and replay mode, in both tile modes and both record layouts, and
against single-map handles where a pool must not make a difference."""
import numpy as np
import pytest
import torch

from golden_util import load_map_spawn_tables

pytestmark = pytest.mark.gpu


def box(h, w):
    b = np.ones((h, w), dtype=np.uint8)
    b[1:-1, 1:-1] = 0
    return b


def maps20():
    """Five 20x20 layouts with different spawn counts: the reference's cross asset map, the walled box, and three more."""
    cross = np.asarray(load_map_spawn_tables()['20x20_cross'][0] != 0, dtype=np.uint8)
    b = box(20, 20)
    block = b.copy()
    block[7:13, 7:13] = 1
    bars = b.copy()
    bars[5, 2:15] = 1
    bars[14, 5:18] = 1
    rooms = b.copy()
    rooms[10, 1:19] = 1
    rooms[10, 4] = rooms[10, 15] = 0
    rooms[1:19, 10] = 1
    rooms[5, 10] = rooms[15, 10] = 0
    return np.stack([cross, b, block, bars, rooms])


def spawn_counts(maps, k):
    from oracle.snake_oracle import spawn_candidates
    return [len(spawn_candidates(m.shape[0], m.shape[1], k, m)) for m in maps]


def oracle_envs(kw, maps, ids, draws, done_mode):
    from oracle.snake_oracle import CoopOracleSnakeEnv, OracleSnakeEnv
    cls = CoopOracleSnakeEnv if done_mode == 'any' else OracleSnakeEnv
    return [cls(draws=d, wall_map=maps[m], **kw) for d, m in zip(draws, ids)]


def oracle_reset(env, maps, m):
    env.wall_map = (np.asarray(maps[m]) != 0).astype(np.int64)
    return env.reset()


def make_batch(monkeypatch, N, maps, kw, compact=None, coop=None, **extra):
    from marl_snake_b200 import SnakeBatch
    if compact is not None:
        monkeypatch.setenv('SNK_COMPACT', str(compact))
    if coop is not None:
        monkeypatch.setenv('SNK_COOP', str(coop))
    b = SnakeBatch(N, wall_maps=maps, **kw, **extra)
    monkeypatch.delenv('SNK_COMPACT', raising=False)
    monkeypatch.delenv('SNK_COOP', raising=False)
    return b


def walls_of(grid):
    return (np.asarray(grid) % 10 == 1).astype(np.uint8)


def check_philox_pool(monkeypatch, kw, maps, N, steps, seed, compact=None, coop=None, done_mode='all', env_id_offset=0):
    """Philox mode: next_maps is rewritten from torch before every step; the oracle resets on the same map ids."""
    from oracle.snake_oracle import PhiloxDraws
    M = len(maps)
    b = make_batch(monkeypatch, N, maps, kw, compact, coop, seed=seed, done_mode=done_mode, env_id_offset=env_id_offset)
    assert b.num_maps == M
    ids0 = (env_id_offset + np.arange(N)) % M
    assert np.array_equal(b.next_maps.cpu().numpy(), ids0)
    draws = [PhiloxDraws(seed, env_id_offset + e) for e in range(N)]
    envs = oracle_envs(kw, maps, ids0, draws, done_mode)
    for d in draws:
        d.tick()
    want = np.stack([oracle_reset(env, maps, m) for env, m in zip(envs, ids0)])
    assert np.array_equal(b.reset().cpu().numpy(), want)
    cur = ids0.copy()
    assert np.array_equal(b.current_maps.cpu().numpy(), cur)
    gen = torch.Generator(device=b.device)
    gen.manual_seed(seed)
    rng = np.random.RandomState(seed)
    n_actions = 5 if kw.get('observer') == 'human' else 3
    switches = 0
    for t in range(steps):
        b.next_maps.random_(0, M, generator=gen)
        nxt = b.next_maps.cpu().numpy()
        acts = rng.randint(0, n_actions, size=(N, b.num_snakes)).astype(np.uint8)
        obs, rew, done, info = b.step(torch.as_tensor(acts).cuda())
        obs, rew, done = obs.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy()
        fin = info['finished'].cpu().numpy()
        for e, env in enumerate(envs):
            draws[e].tick()
            o, r, dn, inf = env.step([int(a) for a in acts[e]])
            if all(dn):
                switches += int(cur[e] != nxt[e])
                cur[e] = nxt[e]
                o = oracle_reset(env, maps, cur[e])
            tag = (t, e)
            assert np.array_equal(rew[e], np.asarray(r)), ('rew', tag)
            assert np.array_equal(done[e], np.asarray(dn)), ('done', tag)
            assert np.array_equal(obs[e], o), ('obs', tag)
            assert bool(fin[e]) == bool(inf), ('finished', tag)
            if inf:
                assert np.array_equal(info['rank'][e].cpu().numpy(), inf['rank']), ('rank', tag)
                assert np.array_equal(info['episode_scores'][e].cpu().numpy(), inf['episode_scores']), ('scores', tag)
        st = b.get_state()
        assert np.array_equal(st['grid'].cpu().numpy(), np.stack([env.grid for env in envs])), ('grid', t)
        assert np.array_equal(st['map'].cpu().numpy(), cur), ('current_maps', t)
    assert switches > 0
    assert b.device_errors() == 0
    b.close()


KW = dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5, max_episode_steps=9)


def test_pool_maps_have_different_spawn_counts():
    counts = spawn_counts(maps20(), 3)
    assert len(set(counts)) == len(counts), counts


@pytest.mark.parametrize('compact', [0, 1])
@pytest.mark.parametrize('coop', [0, 1])
def test_philox_pool_matches_oracle(monkeypatch, compact, coop):
    check_philox_pool(monkeypatch, KW, maps20(), 16, 40, seed=5 + 2 * compact + coop, compact=compact, coop=coop)


@pytest.mark.parametrize('kw,extra', [
    (dict(KW, frame_stack=2), {}),
    (KW, dict(done_mode='any')),
    (dict(KW, num_snakes=8, vision_range=3), dict(compact=0)),
    (dict(KW, num_snakes=8, vision_range=3), dict(compact=1)),
    (dict(KW, vision_range=None, observer='human'), {}),
], ids=['fs2', 'coop_done', 'ns8_plane', 'ns8_compact', 'full_grid_human'])
def test_philox_pool_matches_oracle_more_shapes(monkeypatch, kw, extra):
    check_philox_pool(monkeypatch, kw, maps20(), 12, 36, seed=17, **extra)


def test_philox_pool_asset_map_12x12(monkeypatch):
    walls = np.asarray(load_map_spawn_tables()['12x12'][0] != 0, dtype=np.uint8)
    alt = box(12, 12)
    alt[6, 3:9] = 1
    kw = dict(height=12, width=12, num_snakes=3, snake_length=3, vision_range=3, max_episode_steps=7)
    check_philox_pool(monkeypatch, kw, np.stack([walls, box(12, 12), alt]), 10, 40, seed=3)


def test_replay_pool_matches_oracle_logs(monkeypatch):
    from marl_snake_b200 import SnakeBatch
    from oracle.snake_oracle import NumpyGlobalDraws, RecordingDraws
    maps, N, steps = maps20(), 8, 40
    M = len(maps)
    np.random.seed(123)
    plan = np.random.RandomState(9)
    next_seq = plan.randint(0, M, size=(steps + 1, N)).astype(np.uint8)
    acts = plan.randint(0, 3, size=(steps, N, 4)).astype(np.uint8)
    draws = [RecordingDraws(NumpyGlobalDraws()) for _ in range(N)]
    envs = oracle_envs(KW, maps, next_seq[0], draws, 'all')
    ref_obs, ref_rew, ref_done, ref_map = [], [], [], []
    ref_obs.append(np.stack([oracle_reset(env, maps, m) for env, m in zip(envs, next_seq[0])]))
    cur = next_seq[0].copy()
    for t in range(steps):
        o_t, r_t, d_t = [], [], []
        for e, env in enumerate(envs):
            o, r, dn, _ = env.step([int(a) for a in acts[t, e]])
            if all(dn):
                cur[e] = next_seq[t + 1, e]
                o = oracle_reset(env, maps, cur[e])
            o_t.append(o); r_t.append(r); d_t.append(dn)
        ref_obs.append(np.stack(o_t)); ref_rew.append(np.asarray(r_t)); ref_done.append(np.asarray(d_t))
        ref_map.append(cur.copy())
    b = SnakeBatch(N, wall_maps=maps, map_ids=next_seq[0], rng='replay', **KW)
    b.set_replay([d.log for d in draws])
    assert np.array_equal(b.reset().cpu().numpy(), ref_obs[0])
    for t in range(steps):
        b.next_maps.copy_(torch.as_tensor(next_seq[t + 1]).cuda())
        obs, rew, done, _ = b.step(torch.as_tensor(acts[t]).cuda())
        assert np.array_equal(rew.cpu().numpy(), ref_rew[t]), t
        assert np.array_equal(done.cpu().numpy(), ref_done[t]), t
        assert np.array_equal(obs.cpu().numpy(), ref_obs[t + 1]), t
        assert np.array_equal(b.current_maps.cpu().numpy(), ref_map[t]), t
    assert np.array_equal(b.replay_cursors(), [len(d.log) for d in draws])
    assert b.device_errors() == 0


def test_replayed_spawn_index_is_checked_against_the_map_table():
    from marl_snake_b200 import SnakeBatch
    from oracle.snake_oracle import NumpyGlobalDraws, OracleSnakeEnv, RecordingDraws
    maps = maps20()
    counts = spawn_counts(maps, 3)
    small, big = int(np.argmin(counts)), int(np.argmax(counts))
    for seed in range(200):                       # a reset on the big map whose poses lie past the small map's table
        np.random.seed(seed)
        rec = RecordingDraws(NumpyGlobalDraws())
        env = OracleSnakeEnv(draws=rec, wall_map=maps[big], **KW)
        want = env.reset()
        if max(rec.log[:4]) >= counts[small]:
            break
    assert max(rec.log[:4]) >= counts[small]
    ok = SnakeBatch(2, wall_maps=maps, map_ids=[big, big], rng='replay', **KW)
    ok.set_replay([rec.log, rec.log])
    assert np.array_equal(ok.reset().cpu().numpy(), np.stack([want, want]))
    assert ok.device_errors() == 0
    bad = SnakeBatch(2, wall_maps=maps, map_ids=[small, small], rng='replay', **KW)
    bad.set_replay([rec.log, rec.log])
    bad.reset()
    assert bad.device_errors() & 4


def rollout(b, steps, seed, M, rewrite=True, ids_fn=None):
    """Steps a batch with seeded actions, rewriting next_maps every step; returns every output as host arrays."""
    gen = torch.Generator(device=b.device)
    gen.manual_seed(seed)
    rng = np.random.RandomState(seed)
    out = [b.reset().cpu().numpy()]
    for t in range(steps):
        if rewrite:
            if ids_fn is None:
                b.next_maps.random_(0, M, generator=gen)
            else:
                b.next_maps.copy_(ids_fn(t))
        acts = torch.as_tensor(rng.randint(0, 3, size=(b.num_envs, b.num_snakes)).astype(np.uint8)).cuda()
        obs, rew, done, info = b.step(acts)
        st = b.get_state()
        out += [obs.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy(), info['finished'].cpu().numpy(),
                st['grid'].cpu().numpy()]
    return out


def assert_same(a, b):
    assert len(a) == len(b)
    for k, (x, y) in enumerate(zip(a, b)):
        assert np.array_equal(x, y), k


@pytest.mark.parametrize('compact', [0, 1])
def test_pool_of_copies_equals_single_map_handle(monkeypatch, compact):
    from marl_snake_b200 import SnakeBatch
    cross = maps20()[0]
    monkeypatch.setenv('SNK_COMPACT', str(compact))
    ref = SnakeBatch(24, wall_map=cross, seed=8, **KW)
    pool = SnakeBatch(24, wall_maps=np.stack([cross] * 7), seed=8, **KW)
    one = SnakeBatch(24, wall_maps=[cross], seed=8, **KW)
    want = rollout(ref, 50, 4, 1, rewrite=False)
    assert_same(rollout(pool, 50, 4, 7), want)
    assert_same(rollout(one, 50, 4, 1), want)
    assert np.array_equal(one.current_maps.cpu().numpy(), np.zeros(24))
    for x in (ref, pool, one):
        assert x.device_errors() == 0


def test_two_shards_equal_one_run():
    from marl_snake_b200 import SnakeBatch
    maps, N = maps20(), 16
    seq = np.random.RandomState(2).randint(0, len(maps), size=(40, N)).astype(np.uint8)
    whole = SnakeBatch(N, wall_maps=maps, seed=21, **KW)
    lo = SnakeBatch(N // 2, wall_maps=maps, seed=21, env_id_offset=0, **KW)
    hi = SnakeBatch(N // 2, wall_maps=maps, seed=21, env_id_offset=N // 2, **KW)
    assert np.array_equal(hi.next_maps.cpu().numpy(), (N // 2 + np.arange(N // 2)) % len(maps))
    rng = np.random.RandomState(0)
    outs = [x.reset().cpu().numpy() for x in (whole, lo, hi)]
    assert np.array_equal(outs[0], np.concatenate(outs[1:]))
    for t in range(40):
        whole.next_maps.copy_(torch.as_tensor(seq[t]).cuda())
        lo.next_maps.copy_(torch.as_tensor(seq[t, :N // 2]).cuda())
        hi.next_maps.copy_(torch.as_tensor(seq[t, N // 2:]).cuda())
        a = rng.randint(0, 3, size=(N, 4)).astype(np.uint8)
        r = [x.step(torch.as_tensor(aa).cuda(), copy=True) for x, aa in ((whole, a), (lo, a[:N // 2]), (hi, a[N // 2:]))]
        for k in range(3):
            assert np.array_equal(r[0][k].cpu().numpy(), np.concatenate([r[1][k].cpu().numpy(), r[2][k].cpu().numpy()])), (t, k)
        assert np.array_equal(whole.current_maps.cpu().numpy(),
                              np.concatenate([lo.current_maps.cpu().numpy(), hi.current_maps.cpu().numpy()]))


def test_masked_and_explicit_reset_pick_up_next_map():
    from marl_snake_b200 import SnakeBatch
    maps, N = maps20(), 10
    b = SnakeBatch(N, wall_maps=maps, seed=1, **KW)
    b.reset()
    b.next_maps.copy_(torch.full((N,), 3, dtype=torch.uint8))
    mask = torch.zeros(N, dtype=torch.uint8)
    mask[[1, 4, 7]] = 1
    before = b.current_maps.cpu().numpy().copy()
    b.reset(mask=mask.cuda())
    want = before.copy()
    want[[1, 4, 7]] = 3
    assert np.array_equal(b.current_maps.cpu().numpy(), want)
    grid = b.get_state()['grid'].cpu().numpy()
    for e in range(N):
        assert np.array_equal(walls_of(grid[e]), maps[want[e]]), e
    b.next_maps.copy_(torch.full((N,), 2, dtype=torch.uint8))
    b.reset()
    assert np.array_equal(b.current_maps.cpu().numpy(), np.full(N, 2))
    b.next_maps.fill_(4)
    obs = np.empty((N,) + b.obs_shape, dtype=np.uint8)
    b.reset_host(torch.from_numpy(obs))
    assert np.array_equal(b.current_maps.cpu().numpy(), np.full(N, 4))
    assert np.array_equal(walls_of(b.get_state()['grid'].cpu().numpy()[0]), maps[4])
    assert b.device_errors() == 0


@pytest.mark.parametrize('compact', [0, 1])
def test_set_state_starts_an_episode_on_next_map(monkeypatch, compact):
    from marl_snake_b200 import SnakeBatch
    maps, N = maps20(), 4
    monkeypatch.setenv('SNK_COMPACT', str(compact))
    b = SnakeBatch(N, wall_maps=maps, map_ids=[0, 0, 0, 0], seed=2, **KW)
    b.reset()
    st = b.get_state(max_cells=8)
    args = [st[k].cpu().numpy() for k in ('grid', 'alive', 'dir', 'length', 'cells', 'alive_counter')]
    args[4] = np.maximum(args[4], 0)                  # set_state wants unused cell entries padded with 0, not -1
    b.next_maps.fill_(0)
    b.current_maps.fill_(1)
    obs = b.set_state(*args).cpu().numpy()
    assert b.device_errors(clear=True) == 0
    assert np.array_equal(b.current_maps.cpu().numpy(), np.zeros(N))
    c = SnakeBatch(N, wall_map=maps[0], seed=2, **KW)
    c.reset()
    assert np.array_equal(c.set_state(*args).cpu().numpy(), obs)
    # the cross map's walls are not map 2's: refused through the sticky state bit
    b.next_maps.fill_(2)
    b.set_state(*args)
    assert b.device_errors(clear=True) & 64
    assert np.array_equal(b.current_maps.cpu().numpy(), np.full(N, 2))


def test_checkpoint_resumes_with_map_ids_and_refuses_another_pool():
    from marl_snake_b200 import SnakeBatch
    from marl_snake_b200._lib import SnkError
    maps, N = maps20(), 12
    a = SnakeBatch(N, wall_maps=maps, seed=6, **KW)
    rng = np.random.RandomState(1)
    a.reset()
    for _ in range(7):
        a.step(torch.as_tensor(rng.randint(0, 3, size=(N, 4)).astype(np.uint8)).cuda())
    a.next_maps.copy_(torch.as_tensor(rng.randint(0, len(maps), size=N).astype(np.uint8)).cuda())
    blob = a.save_checkpoint()
    b = SnakeBatch(N, wall_maps=maps, seed=6, **KW)
    b.load_checkpoint(blob)
    assert np.array_equal(b.next_maps.cpu().numpy(), a.next_maps.cpu().numpy())
    assert np.array_equal(b.current_maps.cpu().numpy(), a.current_maps.cpu().numpy())
    seq = rng.randint(0, len(maps), size=(30, N)).astype(np.uint8)
    for t in range(30):
        acts = torch.as_tensor(rng.randint(0, 3, size=(N, 4)).astype(np.uint8)).cuda()
        outs = []
        for x in (a, b):
            obs, rew, done, info = x.step(acts, copy=True)
            outs.append((obs.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy(), x.current_maps.cpu().numpy()))
            x.next_maps.copy_(torch.as_tensor(seq[t]).cuda())
        for u, v in zip(*outs):
            assert np.array_equal(u, v), t
    other = SnakeBatch(N, wall_maps=maps[::-1].copy(), seed=6, **KW)
    with pytest.raises(SnkError, match='different wall-map pool'):
        other.load_checkpoint(blob)
    single = SnakeBatch(N, wall_map=maps[0], seed=6, **KW)
    with pytest.raises(SnkError):
        single.load_checkpoint(blob)
    with pytest.raises(SnkError):
        a.load_checkpoint(single.save_checkpoint())


@pytest.mark.parametrize('compact', [0, 1])
def test_step_many_with_map_switches_equals_single_steps(monkeypatch, compact):
    from marl_snake_b200 import SnakeBatch
    maps, N, T = maps20(), 64, 23
    kw = dict(KW, max_episode_steps=5)
    monkeypatch.setenv('SNK_COMPACT', str(compact))
    a = SnakeBatch(N, wall_maps=maps, seed=4, **kw)
    b = SnakeBatch(N, wall_maps=maps, seed=4, **kw)
    ids = torch.as_tensor(np.random.RandomState(3).randint(0, len(maps), size=N).astype(np.uint8)).cuda()
    a.reset(); b.reset()
    a.next_maps.copy_(ids); b.next_maps.copy_(ids)
    acts = torch.as_tensor(np.random.RandomState(5).randint(0, 3, size=(T, N, 4)).astype(np.uint8)).cuda()
    obs = torch.empty((T, N) + a.obs_shape, dtype=torch.uint8, device=a.device)
    _, rew, done, _ = a.step_many(acts, obs=obs)
    for t in range(T):
        o, r, d, _ = b.step(acts[t])
        assert torch.equal(o, obs[t]) and torch.equal(r, rew[t]) and torch.equal(d.to(torch.uint8), done[t]), t
    assert torch.equal(a.current_maps, b.current_maps)
    assert torch.equal(a.current_maps, ids)            # every env reset at least once on its next map
    assert torch.equal(a.get_state()['grid'], b.get_state()['grid'])
    assert a.device_errors() == 0 and b.device_errors() == 0


def test_out_of_range_map_id_reads_as_map_zero(monkeypatch):
    from marl_snake_b200 import SnakeBatch
    maps, N = maps20(), 8
    monkeypatch.setenv('SNK_COMPACT', '1')            # compact records: tiles paint their grids from current_maps
    b = SnakeBatch(N, wall_maps=maps, map_ids=[1] * N, seed=3, **KW)
    b.reset()
    b.next_maps[3] = 200
    b.next_maps[5] = len(maps)
    b.reset()
    assert b.device_errors(clear=True) & 128
    cur = b.current_maps.cpu().numpy()
    assert cur[3] == 0 and cur[5] == 0 and (np.delete(cur, [3, 5]) == 1).all()
    grid = b.get_state()['grid'].cpu().numpy()
    assert np.array_equal(walls_of(grid[3]), maps[0]) and np.array_equal(walls_of(grid[5]), maps[0])
    # a bad id the caller writes into current_maps is caught where the tile paints the grid
    b.current_maps[2] = 77
    b.step(torch.zeros((N, 4), dtype=torch.uint8, device=b.device))
    assert b.device_errors(clear=True) & 128
    # the reset's tile load still reads env 2's bad id before the reset replaces it with next_maps; after it all is well
    b.next_maps.fill_(2)
    b.reset()
    b.device_errors(clear=True)
    b.step(torch.zeros((N, 4), dtype=torch.uint8, device=b.device))
    assert b.device_errors() == 0
    assert (b.current_maps.cpu().numpy() == 2).all()


def test_full_size_pool_rerandomised_every_step():
    from marl_snake_b200 import SnakeBatch
    from oracle.snake_oracle import OracleSnakeEnv, PhiloxDraws
    N, M, steps, seed = 1 << 20, 16, 100, 31
    kw = dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5)
    base = maps20()
    rng = np.random.RandomState(4)
    maps = []
    for k in range(M):                                  # sixteen layouts: the five above with extra wall blocks
        m = base[k % len(base)].copy()
        if k >= len(base):
            r, c = rng.randint(2, 16, size=2)
            m[r:r + 2, c:c + 3] = 1
        maps.append(m)
    maps = np.stack(maps)
    b = SnakeBatch(N, wall_maps=maps, seed=seed, max_episode_steps=12, **kw)
    watch = np.r_[0:8, N - 8:N]
    draws = [PhiloxDraws(seed, int(e)) for e in watch]
    ids0 = watch % M
    envs = [OracleSnakeEnv(draws=d, wall_map=maps[m], max_episode_steps=12, **kw) for d, m in zip(draws, ids0)]
    for d in draws:
        d.tick()
    want = np.stack([oracle_reset(env, maps, m) for env, m in zip(envs, ids0)])
    widx = torch.as_tensor(watch).cuda()
    obs = b.reset()
    assert np.array_equal(obs[widx].cpu().numpy(), want)
    gen = torch.Generator(device=b.device)
    gen.manual_seed(seed)
    cur = ids0.copy()
    for t in range(steps):
        b.next_maps.random_(0, M, generator=gen)
        nxt = b.next_maps[widx].cpu().numpy()
        acts = torch.randint(0, 3, (N, 4), dtype=torch.uint8, device=b.device, generator=gen)
        obs, rew, done, _ = b.step(acts)
        a_w = acts[widx].cpu().numpy()
        o_w, r_w, d_w = obs[widx].cpu().numpy(), rew[widx].cpu().numpy(), done[widx].cpu().numpy()
        for k, env in enumerate(envs):
            draws[k].tick()
            o, r, dn, _ = env.step([int(a) for a in a_w[k]])
            if all(dn):
                cur[k] = nxt[k]
                o = oracle_reset(env, maps, cur[k])
            assert np.array_equal(r_w[k], np.asarray(r)) and np.array_equal(d_w[k], np.asarray(dn)), (t, k)
            assert np.array_equal(o_w[k], o), (t, k)
    assert np.array_equal(b.current_maps[widx].cpu().numpy(), cur)
    assert b.device_errors() == 0
    st = b.get_state()
    grid = st['grid']
    lay = torch.as_tensor(maps).cuda()[st['map'].long()]
    assert torch.equal((grid % 10 == 1).to(torch.uint8), lay)
    assert np.array_equal(grid[widx].cpu().numpy(), np.stack([env.grid for env in envs]))
    assert len(torch.unique(st['map'])) == M


def test_collect_runs_on_a_pool_batch():
    from marl_snake_b200 import DeviceReplayBuffer, SnakeBatch, collect
    from test_gpu_rollout import ExactNet, reference_style_loop
    maps, N = maps20(), 6
    kw = dict(KW, vision_range=3, max_episode_steps=15)
    a = SnakeBatch(N, wall_maps=maps, seed=12, **kw)
    b = SnakeBatch(N, wall_maps=maps, seed=12, **kw)
    ns, oh, ow, ch = a.obs_shape
    net = ExactNet(ch, oh, ow).cuda()
    want = reference_style_loop(a, net, 60, 10, -1.0, 40)
    buf = DeviceReplayBuffer(len(want) + 100, b.obs_shape[1:], b.device)
    n = int(collect(b, net, 60, buf, epsilon=0.0, early_death=(10, -1.0), max_steps=40))
    assert n == len(want) == buf.size
    assert np.array_equal(buf.obs[:n].cpu().numpy(), np.stack([t[0] for t in want]))
    assert np.array_equal(buf.next_obs[:n].cpu().numpy(), np.stack([t[3] for t in want]))
    assert torch.equal(a.current_maps, b.current_maps)
    assert a.device_errors() == 0 and b.device_errors() == 0
