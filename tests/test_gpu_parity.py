"""GPU parity tests proper: the CUDA path, called through the C ABI (libsnk.so), against the golden
vectors recorded from the reference and against the oracle.  Integer / byte data and the float64
rewards must match exactly (rewards are fixed-order sums of the configured constants)."""
import numpy as np
import pytest
import torch

from golden_util import ROLLOUTS, Rollout, load_scenarios
from gpu_backend import GpuBackend
from parity_util import check_against_oracle_philox, check_rollout_replay, check_scenario

pytestmark = pytest.mark.gpu

# Record layout in HBM: '1' = compact (no grid; rebuilt in shared memory from walls + fruit slots + bodies), '0' = the
# whole working record.  By default the library picks per handle (compact for warp-private tiles, frame stacks and
# large grids), so tests that mean to cover a layout force it.
both_layouts = pytest.mark.parametrize('compact', ['0', '1'])


@both_layouts
@pytest.mark.parametrize('name', ROLLOUTS)
def test_gpu_rollout_replay(monkeypatch, name, compact):
    monkeypatch.setenv('SNK_COMPACT', compact)
    g = Rollout(name)
    be = GpuBackend(g.num_envs, g.kwargs, rng_mode=1, auto_reset=1, done_mode=g.done_mode)
    check_rollout_replay(be, g)
    assert be.errors() == 0
    be.close()


@both_layouts
@pytest.mark.parametrize('sc', load_scenarios(), ids=lambda s: s.name)
def test_gpu_scenarios(monkeypatch, sc, compact):
    monkeypatch.setenv('SNK_COMPACT', compact)
    kw = dict(height=sc.H, width=sc.W, num_snakes=sc.num_snakes, snake_length=2, **sc.kwargs)
    be = GpuBackend(1, kw, rng_mode=1, auto_reset=0)
    check_scenario(be, sc)
    assert be.errors() == 0
    be.close()


@pytest.mark.parametrize('kw,num_envs,steps', [
    (dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5), 67, 150),
    (dict(height=20, width=20, num_snakes=4, snake_length=3), 33, 80),
    (dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5, frame_stack=4), 40, 120),
    (dict(height=9, width=12, num_snakes=3, snake_length=4, vision_range=2, frame_stack=3,
          max_episode_steps=30), 35, 100),
    (dict(height=16, width=16, num_snakes=7, snake_length=4, vision_range=7,
          reward_dict={'fruit': 10.0, 'kill': 1.0, 'lose': -1.0, 'win': 0.1, 'time': -0.001}), 9, 80),
    (dict(height=10, width=10, num_snakes=1, snake_length=3, num_fruits=4), 21, 100),
    (dict(height=14, width=11, num_snakes=4, snake_length=3, vision_range=3, observer='human'), 37, 120),
])
def test_gpu_philox_matches_oracle(kw, num_envs, steps):
    be = check_against_oracle_philox(GpuBackend, kw, num_envs=num_envs, steps=steps, seed=0xC0FFEE1234,
                                     env_id_offset=3)
    assert be.errors() == 0
    be.close()


def test_gpu_matches_hostsim_large():
    """Same rule source on both sides; checks the kernel's tiling / warp-cooperative paths at a size the
    Python oracle cannot reach quickly: 4099 envs (ragged last tile) x 300 steps, Philox mode."""
    from hostsim_util import HostSim
    kw = dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5)
    N = 4099
    hs = HostSim(N, kw, rng_mode=0, auto_reset=1, seed=77)
    be = GpuBackend(N, kw, rng_mode=0, auto_reset=1, seed=77)
    assert np.array_equal(hs.reset(), be.reset())
    rng = np.random.RandomState(1)
    for t in range(300):
        a = rng.randint(0, 3, size=(N, 4)).astype(np.uint8)
        o1, r1, d1, i1 = hs.step(a)
        o2, r2, d2, i2 = be.step(a)
        assert np.array_equal(r1, r2) and np.array_equal(d1, d2.astype(np.uint8)), t
        assert np.array_equal(o1, o2), t
        assert np.array_equal(i1['finished'], i2['finished'].astype(np.uint8)), t
    assert np.array_equal(hs.grid()[0], be.grid()[0])
    assert be.errors() == 0


def test_gpu_shard_invariance():
    """Streams are keyed by global env id: two shards reproduce the single-batch run (multi-GPU rule)."""
    kw = dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5)
    whole = GpuBackend(64, kw, rng_mode=0, seed=9)
    lo = GpuBackend(24, kw, rng_mode=0, seed=9, env_id_offset=0)
    hi = GpuBackend(40, kw, rng_mode=0, seed=9, env_id_offset=24)
    assert np.array_equal(whole.reset(), np.concatenate([lo.reset(), hi.reset()]))
    rng = np.random.RandomState(4)
    for t in range(120):
        a = rng.randint(0, 3, size=(64, 4)).astype(np.uint8)
        o, r, d, _ = whole.step(a)
        o1, r1, d1, _ = lo.step(a[:24])
        o2, r2, d2, _ = hi.step(a[24:])
        assert np.array_equal(o, np.concatenate([o1, o2])) and np.array_equal(r, np.concatenate([r1, r2]))


@pytest.mark.parametrize('N', [131072, 1048576])
def test_gpu_invariants_full_size(N):
    """BASELINE cfg5 at its full size (1,048,576 envs, warp-private tiles) and one 8-GPU shard of it (131,072
    envs, cooperative tiles): size-independent properties after 64 steps."""
    from marl_snake_b200 import SnakeBatch
    ns = 4
    b = SnakeBatch(N, num_snakes=ns, vision_range=5, seed=1)
    b.reset()
    g = torch.Generator(device='cuda').manual_seed(0)
    for _ in range(64):
        a = torch.randint(0, 3, (N, ns), dtype=torch.uint8, device='cuda', generator=g)
        obs, rew, done, info = b.step(a)
    st = b.get_state(max_cells=16)
    grid = st['grid'].reshape(N, -1).long()
    kind, owner = grid % 10, grid // 10
    alive = st['alive'].bool()
    # exactly one HEAD and one TAIL cell per live snake, none for dead ones
    for i in range(ns):
        heads = ((kind == 3) & (owner == i)).sum(1)
        tails = ((kind == 5) & (owner == i)).sum(1)
        assert torch.equal(heads, alive[:, i].long()) and torch.equal(tails, alive[:, i].long())
        cells = ((kind >= 3) & (owner == i)).sum(1)
        assert torch.equal(cells, st['length'][:, i].long())
    # head cell of every live snake holds its HEAD code; the observation centre shows it on channel 5
    idx = st['head'].clamp(min=0).long()
    code = torch.gather(grid, 1, idx)
    want = 3 + 10 * torch.arange(ns, device='cuda')[None, :]
    assert torch.equal(code[alive], want.expand(N, ns)[alive])
    centre = obs[:, :, 5, 5, 5].bool()
    assert torch.equal(centre, alive)
    # walls intact, observation is 0/1, dones mirror alive
    border = torch.zeros(20, 20, dtype=torch.bool, device='cuda')
    border[0] = border[-1] = True
    border[:, 0] = border[:, -1] = True
    assert bool((grid.view(N, 20, 20)[:, border] == 1).all())
    assert int(obs.max()) == 1
    live_env = ~info['finished']            # envs reset this step return the terminal dones (A1)
    assert torch.equal(done[live_env], ~alive[live_env])
    assert b.device_errors() == 0


def test_gpu_full_size_prefix_matches_rule_source():
    """The first 2,500 and the last 1,500 environments of a 1,048,576-env batch (BASELINE cfg5, the bench's
    own configuration) against the host build of the rule source stepping only those environments: Philox
    streams are keyed by global env id, so every output of those environments must be bit-identical."""
    from hostsim_util import HostSim
    from marl_snake_b200 import SnakeBatch
    N, ns, head, tail = 1 << 20, 4, 2500, 1500
    kw = dict(height=20, width=20, num_snakes=ns, snake_length=3, vision_range=5)
    b = SnakeBatch(N, seed=9, **kw)
    lo = HostSim(head, kw, rng_mode=0, auto_reset=1, seed=9)
    hi = HostSim(tail, kw, rng_mode=0, auto_reset=1, seed=9, env_id_offset=N - tail)
    obs = b.reset()
    assert np.array_equal(obs[:head].cpu().numpy(), lo.reset()) and np.array_equal(obs[N - tail:].cpu().numpy(), hi.reset())
    g = torch.Generator(device='cuda').manual_seed(4)
    for t in range(40):
        a = torch.randint(0, 3, (N, ns), dtype=torch.uint8, device='cuda', generator=g)
        obs, rew, done, info = b.step(a)
        for sim, sl in ((lo, slice(0, head)), (hi, slice(N - tail, N))):
            o, r, d, i = sim.step(a[sl].cpu().numpy())
            assert np.array_equal(obs[sl].cpu().numpy(), o), t
            assert np.array_equal(rew[sl].cpu().numpy(), r) and np.array_equal(done[sl].cpu().numpy(), d.astype(bool)), t
            assert np.array_equal(info['finished'][sl].cpu().numpy(), i['finished'].astype(bool)), t
    assert b.device_errors() == 0


def test_dropin_api():
    """make_snake / SnakeEnv return contract of the reference (wrappers.py:203-223, snake_env.py:159,414)."""
    from marl_snake_b200 import make, make_snake
    env, o_s, a_s, props = make_snake(num_envs=1, num_snakes=4, height=20, width=20, snake_length=3,
                                      vision_range=5)
    assert o_s is None and a_s is None
    assert props == {'action_info': {'action_n': 3}, 'num_envs': 1, 'num_snakes': 4}
    obs = env.reset()
    assert isinstance(obs, np.ndarray) and obs.shape == (4, 11, 11, 8) and obs.dtype == np.uint8
    assert env.observation_space.shape == (4, 11, 11, 8) and env.action_space.n == 3
    obs, rews, dones, info = env.step([env.action_space.sample() for _ in range(4)])
    assert isinstance(rews, list) and isinstance(rews[0], float) and isinstance(dones[0], bool)
    assert isinstance(info, dict)
    with pytest.raises(AssertionError):
        env.step([0])
    with pytest.raises(KeyError):
        env.step([0, 1, 2, 5])
    with pytest.raises(KeyError):
        make('Snake-v1', reward_dict={'fruit': 1.0})
    single, _, _, _ = make_snake(num_envs=1, num_snakes=1, num_fruits=4)
    o = single.reset()
    assert o.shape == (20, 20, 8)
    o, r, d, i = single.step(1)
    assert isinstance(r, float) and isinstance(d, bool) and i == {}
    venv, _, _, props = make_snake(num_envs=16, num_snakes=4, vision_range=5)
    o = venv.reset()
    assert o.shape == (16, 4, 11, 11, 8)
    o, r, d, infos = venv.step(np.zeros((16, 4), dtype=np.int64))
    assert r.shape == (16, 4) and d.shape == (16, 4) and len(infos) == 16


def test_vector_env_numpy_equals_torch_output():
    """make_snake(num_envs > 1): the host-array mode (snk_step_host_info, pinned buffers) and the CUDA-tensor
    mode step the same trajectories; infos carry the terminal dict of finished envs (wrappers.py:138-146)."""
    from marl_snake_b200 import make_snake
    kw = dict(num_snakes=3, height=10, width=10, vision_range=3, max_episode_steps=9, seed=5)
    a_env, _, _, _ = make_snake(num_envs=40, **kw)
    b_env, _, _, _ = make_snake(num_envs=40, output='torch', **kw)
    assert np.array_equal(a_env.reset(), b_env.reset().cpu().numpy())
    rng = np.random.RandomState(1)
    ended = 0
    for t in range(30):
        act = rng.randint(0, 3, size=(40, 3))
        o1, r1, d1, infos = a_env.step(act)
        o2, r2, d2, info2 = b_env.step(act)
        assert np.array_equal(o1, o2.cpu().numpy()) and np.array_equal(r1, r2.cpu().numpy())
        assert d1.dtype == np.bool_ and np.array_equal(d1, d2.cpu().numpy())
        fin = info2['finished'].cpu().numpy()
        for e in range(40):
            assert bool(infos[e]) == bool(fin[e])
            if fin[e]:
                ended += 1
                assert infos[e]['rank'] == [int(x) for x in info2['rank'][e].cpu().numpy()]
                assert np.array_equal(infos[e]['episode_scores'], info2['episode_scores'][e].cpu().numpy())
    assert ended >= 80
    with pytest.raises(KeyError):
        a_env.step(np.full((40, 3), 3))
    a_env.close(); b_env.close()


def test_dropin_human_observer():
    """observer='human': five absolute actions, Discrete(5*ns) on the env, Discrete(5) behind the wrapper
    (snake_env.py:101-109, wrappers.py:111), unknown actions are no-ops instead of KeyError (:610-632)."""
    from marl_snake_b200 import make, make_snake
    raw = make('Snake-v1', num_snakes=2, observer='human', vision_range=3, seed=4)
    assert raw.action_space.n == 10 and raw.action_dict == {'noop': 0, 'left': 1, 'right': 2, 'down': 3, 'up': 4}
    raw.reset()
    raw.step([9, 4])                                                  # no KeyError on this path
    env, _, _, props = make_snake(num_envs=1, num_snakes=2, observer='human', vision_range=3)
    assert props['action_info'] == {'action_n': 5} and env.action_space.n == 5
    venv, _, _, props = make_snake(num_envs=8, num_snakes=2, observer='human', vision_range=3)
    assert props['action_info'] == {'action_n': 5}
    venv.reset()
    o, r, d, _ = venv.step(np.full((8, 2), 4))
    assert o.shape == (8, 2, 7, 7, 8)
    with pytest.raises(ValueError):
        make('Snake-v1', observer='bird')


def test_gpu_generic_kernel_instance(monkeypatch):
    """The BASELINE shapes run specialised template instances; the unspecialised instance must agree."""
    from hostsim_util import HostSim
    monkeypatch.setenv('SNK_FORCE_GENERIC', '1')
    for kw in (dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5),
               dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5, frame_stack=4),
               dict(height=20, width=20, num_snakes=4, snake_length=3)):
        N = 301
        hs = HostSim(N, kw, rng_mode=0, auto_reset=1, seed=5)
        be = GpuBackend(N, kw, rng_mode=0, auto_reset=1, seed=5)
        assert np.array_equal(hs.reset(), be.reset())
        rng = np.random.RandomState(2)
        for t in range(150):
            a = rng.randint(0, 3, size=(N, 4)).astype(np.uint8)
            o1, r1, d1, _ = hs.step(a)
            o2, r2, d2, _ = be.step(a)
            assert np.array_equal(o1, o2) and np.array_equal(r1, r2) and np.array_equal(d1, d2.astype(np.uint8)), t
        be.close()


@pytest.mark.parametrize('kw,N', [
    (dict(height=20, width=20, num_snakes=4, snake_length=3), 1000),                                  # cfg2 shape
    (dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5, frame_stack=4), 1000),   # cfg3 shape
    (dict(height=64, width=64, num_snakes=16, snake_length=5, vision_range=7,
          reward_dict={'fruit': 10.0, 'kill': 1.0, 'lose': -1.0, 'win': 0.1, 'time': -0.001}), 70),   # cfg4 shape
    (dict(height=12, width=17, num_snakes=5, snake_length=3, vision_range=3), 257),                   # generic, odd window
    (dict(height=8, width=8, num_snakes=1, snake_length=2, vision_range=1, frame_stack=3), 129),
])
def test_gpu_matches_hostsim_shapes(kw, N):
    """BASELINE config shapes (specialised instances) and odd generic shapes against the host build of
    the same rule source, Philox mode, with info outputs."""
    from hostsim_util import HostSim
    ns = kw['num_snakes']
    hs = HostSim(N, kw, rng_mode=0, auto_reset=1, seed=11)
    be = GpuBackend(N, kw, rng_mode=0, auto_reset=1, seed=11)
    assert np.array_equal(hs.reset(), be.reset())
    rng = np.random.RandomState(3)
    for t in range(120):
        a = rng.randint(0, 3, size=(N, ns)).astype(np.uint8)
        o1, r1, d1, i1 = hs.step(a)
        o2, r2, d2, i2 = be.step(a)
        assert np.array_equal(r1, r2) and np.array_equal(d1, d2.astype(np.uint8)), t
        assert np.array_equal(o1, o2), t
        fin = i1['finished'].astype(bool)
        assert np.array_equal(fin, i2['finished'])
        for k in ('rank', 'episode_scores', 'episode_steps', 'episode_fruits', 'episode_kills'):
            assert np.array_equal(i1[k][fin], i2[k][fin]), (k, t)
    assert np.array_equal(hs.grid()[0], be.grid()[0])
    assert be.errors() == 0
    be.close()


def test_gpu_rollout_stats():
    """Device-side rollout statistics equal the sums of the per-step terminal info."""
    from marl_snake_b200 import SnakeBatch
    N, ns = 3000, 4
    b = SnakeBatch(N, num_snakes=ns, vision_range=5, seed=3)
    b.reset()
    g = torch.Generator(device='cuda').manual_seed(1)
    eps = ret = fruits = kills = 0.0
    for _ in range(200):
        a = torch.randint(0, 3, (N, ns), dtype=torch.uint8, device='cuda', generator=g)
        _, _, _, info = b.step(a)
        fin = info['finished']
        eps += float(fin.sum())
        ret += float(info['episode_scores'][fin].sum())
        fruits += float(info['episode_fruits'][fin].sum())
        kills += float(info['episode_kills'][fin].sum())
    st = b.stats()
    assert st['episodes'] == eps and eps > 1000
    assert st['fruits_sum'] == fruits and st['kills_sum'] == kills
    assert abs(st['return_sum'] - ret) < 1e-6 * max(1.0, abs(ret))
    assert st['env_steps'] == 200 * N
    t = b.stats_tensor()
    assert float(t[0]) == eps


@both_layouts
@pytest.mark.parametrize('coop', ['0', '1', '1-small'])
@pytest.mark.parametrize('kw,N', [
    (dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5), 2051),
    (dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5, frame_stack=4), 515),
    (dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5, frame_stack=3), 260),
    (dict(height=64, width=64, num_snakes=16, snake_length=5, vision_range=7), 37),
    (dict(height=24, width=24, num_snakes=9, snake_length=3, vision_range=9), 50),     # window > 16: no table
    (dict(height=12, width=12, num_snakes=2, snake_length=3), 300),
    (dict(height=30, width=30, num_snakes=20, snake_length=3, vision_range=4), 21),   # one env per warp, dual LUT
    (dict(height=26, width=26, num_snakes=25, snake_length=2, num_fruits=30), 9),       # max snakes, full-grid obs
    (dict(height=9, width=9, num_snakes=1, snake_length=3, vision_range=2), 700),      # 32 envs per warp
    # 32 fruits and 12 snakes: head-on meetings on fruit cells push the fruit count past num_fruits (C3) -- more than
    # 32 fruit slots in a compact record
    (dict(height=24, width=34, num_snakes=12, snake_length=3, vision_range=4, num_fruits=32, max_episode_steps=12), 130),
])
def test_gpu_tile_modes(monkeypatch, coop, kw, N, compact):
    """Both tile modes (warp-private tiles / CTA-cooperative tile; '1-small' = one environment per
    cooperative tile with 64 threads) against the host build of the rule source; by default the mode and the
    tile size are chosen from the batch size, so each is forced here."""
    from hostsim_util import HostSim
    monkeypatch.setenv('SNK_COOP', coop[0])
    monkeypatch.setenv('SNK_COMPACT', compact)
    if coop == '1-small':
        monkeypatch.setenv('SNK_THREADS', '64')
        monkeypatch.setenv('SNK_TILE_ENVS', '1')
    ns = kw['num_snakes']
    hs = HostSim(N, kw, rng_mode=0, auto_reset=1, seed=21)
    be = GpuBackend(N, kw, rng_mode=0, auto_reset=1, seed=21)
    assert np.array_equal(hs.reset(), be.reset())
    rng = np.random.RandomState(5)
    for t in range(100):
        a = rng.randint(0, 3, size=(N, ns)).astype(np.uint8)
        o1, r1, d1, i1 = hs.step(a)
        o2, r2, d2, i2 = be.step(a)
        assert np.array_equal(r1, r2) and np.array_equal(d1, d2.astype(np.uint8)), t
        assert np.array_equal(o1, o2), t
        assert np.array_equal(i1['finished'].astype(bool), i2['finished']), t
    assert np.array_equal(hs.grid()[0], be.grid()[0])
    assert be.errors() == 0
    be.close()


@pytest.mark.parametrize('knob', ['SNK_TMA=0', 'SNK_ENC_LEGACY=1', 'SNK_NO_TABLE=1', 'SNK_TMA=0,SNK_COOP=0', 'SNK_NO_DIG=1',
                                  'SNK_NO_DIG=1,SNK_COOP=0', 'SNK_NO_COMPACT=1', 'SNK_COMPACT=0,SNK_COOP=0',
                                  'SNK_COMPACT=1,SNK_COOP=1', 'SNK_COMPACT=1,SNK_TMA=0', 'SNK_COMPACT=1,SNK_TMA=0,SNK_COOP=0',
                                  'SNK_COMPACT=0,SNK_TMA=0', 'SNK_COMPACT=1,SNK_ENC_LEGACY=1', 'SNK_BIGREG_TILES=1,SNK_COOP=0',
                                  'SNK_L2_KEEP=1', 'SNK_L2_KEEP=0', 'SNK_L2_KEEP=1,SNK_COOP=0'])
@pytest.mark.parametrize('kw,N', [
    (dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5), 1500),
    (dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5, frame_stack=4), 300),
    (dict(height=14, width=12, num_snakes=3, snake_length=3), 200),
])
def test_gpu_alternative_code_paths(monkeypatch, knob, kw, N):
    """The A/B switches of INTEGRATION.md section 6 select real code paths (plain loads / stores instead of
    TMA bulk copies, the table-driven or index-arithmetic encode instead of the register / direct ones);
    each must give the same bytes as the default."""
    from hostsim_util import HostSim
    for kv in knob.split(','):
        k, v = kv.split('=')
        monkeypatch.setenv(k, v)
    ns = kw['num_snakes']
    # the uncapped instance: a step into the batch's own (compressible) block runs the capped one, so step into a
    # plain buffer, and check through the launch witness (in a fresh process, where the profiler records reliably)
    # that the steps run the warp-private variant 3
    bigreg = 'SNK_BIGREG_TILES' in knob
    if bigreg:
        from test_gpu_instances import witnessed_tiles
        tiles = witnessed_tiles(f"""
import json, numpy as np
from gpu_backend import GpuBackend
from test_gpu_instances import witness
be = GpuBackend({N}, {kw!r}, rng_mode=0, auto_reset=1, seed=8, plain_obs=True)
be.reset()
rng = np.random.RandomState(4)
tiles = []
for t in range(2):
    be.step(rng.randint(0, 3, size=({N}, {kw['num_snakes']})).astype(np.uint8), around=witness)
    tiles.append(be.around_value.tiles)
print(json.dumps(tiles))
""")
        assert len(tiles) == 2 and all(len(w) == 1 and w[0][5] == 0 and w[0][7] == 3 for w in tiles), tiles
    hs = HostSim(N, kw, rng_mode=0, auto_reset=1, seed=8)
    be = GpuBackend(N, kw, rng_mode=0, auto_reset=1, seed=8, plain_obs=bigreg)
    assert np.array_equal(hs.reset(), be.reset())
    rng = np.random.RandomState(4)
    for t in range(60):
        a = rng.randint(0, 3, size=(N, ns)).astype(np.uint8)
        o1, r1, d1, _ = hs.step(a)
        o2, r2, d2, _ = be.step(a)
        assert np.array_equal(r1, r2) and np.array_equal(d1, d2.astype(np.uint8)), t
        assert np.array_equal(o1, o2), t
    assert np.array_equal(hs.grid()[0], be.grid()[0])
    assert be.errors() == 0
    be.close()


@pytest.mark.parametrize('kw,N,steps', [
    (dict(height=80, width=90, num_snakes=2, snake_length=3, vision_range=3, num_fruits=20), 6, 60),
    (dict(height=200, width=201, num_snakes=4, snake_length=4, vision_range=6, num_fruits=32), 3, 40),
    (dict(height=255, width=257, num_snakes=3, snake_length=2, vision_range=2, num_fruits=9,
          max_episode_steps=7), 2, 30),                                  # the largest grid the ABI accepts
])
def test_gpu_large_grids(kw, N, steps):
    """Grids of thousands of cells: the fruit rank-select walks several 32-word groups per lane range, resets
    repaint the walls row by row, and the tile shrinks to what fits in shared memory (one record is up to
    80 KB).  Against the host build of the rule source, Philox mode, step cap forcing resets."""
    from hostsim_util import HostSim
    ns = kw['num_snakes']
    hs = HostSim(N, kw, rng_mode=0, auto_reset=1, seed=77)
    be = GpuBackend(N, kw, rng_mode=0, auto_reset=1, seed=77)
    assert np.array_equal(hs.reset(), be.reset())
    assert np.array_equal(hs.grid()[0], be.grid()[0])
    rng = np.random.RandomState(3)
    for t in range(steps):
        a = rng.randint(0, 3, size=(N, ns)).astype(np.uint8)
        o1, r1, d1, i1 = hs.step(a)
        o2, r2, d2, i2 = be.step(a)
        assert np.array_equal(r1, r2) and np.array_equal(d1, d2.astype(np.uint8)), t
        assert np.array_equal(o1, o2), t
        assert np.array_equal(hs.grid()[0], be.grid()[0]), t
    assert be.errors() == 0
    be.close()


def _fuzz_configs(n, seed):
    rng = np.random.RandomState(seed)
    out = []
    while len(out) < n:
        H, W = int(rng.randint(6, 41)), int(rng.randint(6, 41))
        ns, K = int(rng.randint(1, 13)), int(rng.randint(2, 7))
        if ns * K * 6 > (H - 2) * (W - 2):
            continue                                          # keep spawn rejection sampling cheap
        V = [None, 1, 2, 3, 4, 5, 6, 8][rng.randint(0, 8)]
        kw = dict(height=H, width=W, num_snakes=ns, snake_length=K, vision_range=V,
                  frame_stack=int([1, 1, 1, 2, 3, 4, 5][rng.randint(0, 7)]),
                  num_fruits=int(rng.randint(0, min(32, (H - 2) * (W - 2) // 4) + 1)),
                  max_episode_steps=int([10000, 10000, 12, 5][rng.randint(0, 4)]),
                  observer=['snake', 'snake', 'human'][rng.randint(0, 3)],
                  reward_dict={'fruit': float(rng.randint(1, 9)), 'kill': 0.25 * rng.randint(0, 9), 'lose': -0.125 * rng.randint(0, 9),
                               'win': 0.5 * rng.randint(0, 5), 'time': -0.001 * rng.randint(0, 5)})
        out.append((kw, int(rng.randint(0, 2)), int([1, 7, 40, 130][rng.randint(0, 4)])))
    return out


FUZZ_CASES = int(__import__('os').environ.get('SNK_FUZZ_CASES', 48))      # soak runs: SNK_FUZZ_CASES=400 SNK_FUZZ_SEED=7
FUZZ_SEED = int(__import__('os').environ.get('SNK_FUZZ_SEED', 20240611))


@pytest.mark.parametrize('case', range(FUZZ_CASES))
def test_gpu_fuzz_shapes(monkeypatch, case):
    """Seeded random shapes (grid 6..40, 1..12 snakes, length 2..6, vision None..8, frame_stack 1..5, fruit
    counts 0..32, step caps, both done rules and observers, odd batch sizes) against the host build of the rule
    source in Philox mode: every output of every step bit-exact."""
    from hostsim_util import HostSim
    kw, done_mode, N = _fuzz_configs(FUZZ_CASES, FUZZ_SEED)[case]
    monkeypatch.setenv('SNK_COMPACT', str(case & 1))         # both record layouts ...
    if case & 2:
        monkeypatch.setenv('SNK_COOP', '0')                  # ... and warp-private tiles for half of the cases
    ns = kw['num_snakes']
    hs = HostSim(N, kw, rng_mode=0, auto_reset=1, seed=1000 + case, done_mode=done_mode)
    be = GpuBackend(N, kw, rng_mode=0, auto_reset=1, seed=1000 + case, done_mode=done_mode)
    assert np.array_equal(hs.reset(), be.reset()), kw
    rng = np.random.RandomState(case)
    n_act = 5 if kw['observer'] == 'human' else 3
    for t in range(50):
        a = rng.randint(0, n_act, size=(N, ns)).astype(np.uint8)
        o1, r1, d1, i1 = hs.step(a)
        o2, r2, d2, i2 = be.step(a)
        assert np.array_equal(r1, r2) and np.array_equal(d1, d2.astype(np.uint8)), (t, kw)
        assert np.array_equal(o1, o2), (t, kw)
        f = i1['finished'].astype(bool)
        assert np.array_equal(f, i2['finished']), (t, kw)
        for k in ('rank', 'episode_scores', 'episode_steps', 'episode_fruits', 'episode_kills'):
            assert np.array_equal(i1[k][f], i2[k][f]), (k, t, kw)
        assert np.array_equal(hs.grid()[0], be.grid()[0]), (t, kw)
    assert hs.errors() == 0 and be.errors() == 0
    hs.close(); be.close()


def test_render_export_and_gui_wrapper():
    """N3: one environment's state exported to the host renderers (render_fancy / rgb_array / RenderGUI)."""
    from marl_snake_b200 import RenderGUI, make_snake
    env, _, _, _ = make_snake(num_envs=1, num_snakes=4, vision_range=5)
    env = RenderGUI(env)
    env.reset()
    env.step([0, 1, 2, 0])
    frame = env.render()
    assert frame.shape == (20 * 30, 20 * 30, 3) and frame.dtype == np.uint8 and frame.max() > 0
    rgb = env.unwrapped.render('rgb_array')
    assert rgb.shape == (20, 20, 3)
    env.close()


def test_gif_rendering_like_the_reference_tests(tmp_path, monkeypatch):
    """marlenv/tests/test_snake.py:85-111: 100 random steps with render('gif'), then save_gif() to the default
    ./tmp/<timestamp>.gif and to a file object."""
    import io
    import os
    from PIL import Image
    from marl_snake_b200 import make
    monkeypatch.chdir(tmp_path)
    env = make('Snake-v1', num_snakes=1, num_fruits=4, disable_env_checker=True,
               reward_dict={'fruit': 1.0, 'kill': 0.0, 'lose': -10.0, 'win': 0.0, 'time': 0.0})
    env.reset()
    with pytest.warns(UserWarning):
        env.save_gif(io.BytesIO())                       # nothing rendered yet
    for _ in range(100):                                   # the reference's rollout keeps stepping a finished env too
        env.render('gif')
        env.step(int(np.random.randint(3)))
    path = env.save_gif()
    assert os.path.exists(path) and os.path.dirname(path) == os.path.join(str(tmp_path), 'tmp')
    gif = Image.open(path)
    gif.seek(1)
    assert gif.size == (300, 300)
    with io.BytesIO() as f:
        env.save_gif(f)
        assert f.tell() > 0


def test_device_rollout_with_q_network():
    """N1: epsilon-greedy from the device observation + device replay buffer, no host sync per step."""
    from marl_snake_b200 import DeviceReplayBuffer, SnakeBatch, collect
    torch.manual_seed(0)
    N, ns = 512, 4
    b = SnakeBatch(N, num_snakes=ns, vision_range=5, seed=4)
    net = torch.nn.Sequential(torch.nn.Conv2d(8, 16, 3, padding=1), torch.nn.ReLU(), torch.nn.Flatten(),
                              torch.nn.Linear(16 * 11 * 11, 3)).cuda()
    buf = DeviceReplayBuffer(50000, b.obs_shape[1:], b.device)
    n = int(collect(b, net, 40, buf, epsilon=0.2))
    assert 0 < n <= 40 * N * ns and buf.size == min(n, 50000)
    o, a, r, o2, d = buf.sample(256)
    assert o.shape == (256, 11, 11, 8) and o.dtype == torch.uint8 and int(a.max()) <= 2
    assert bool((o[:, 5, 5, 5] == 1).all())          # every stored state belongs to a live snake: own head at the centre
    assert b.device_errors() == 0


def test_packed_replay_buffer_and_graphed_steps():
    """N1 plumbing: a replay buffer that stores channel bits (packed by the library, an eighth of the memory)
    returns the same transitions as the unpacked one; T steps captured in a CUDA graph equal T eager steps."""
    from marl_snake_b200 import DeviceReplayBuffer, GraphedSteps, SnakeBatch, unpack_obs
    N, ns, T = 300, 4, 12
    kw = dict(num_snakes=ns, vision_range=5, frame_stack=2, seed=6)
    b = SnakeBatch(N, **kw)
    plain = DeviceReplayBuffer(5000, b.obs_shape[1:], b.device)
    packed = DeviceReplayBuffer(5000, b.obs_shape[1:], b.device, pack=b)
    assert packed.obs.numel() * 8 == plain.obs.numel()
    g = torch.Generator(device='cuda').manual_seed(3)
    obs = b.reset().clone()
    for t in range(6):
        act = torch.randint(0, 3, (N, ns), dtype=torch.uint8, device='cuda', generator=g)
        nxt, rew, done, _ = b.step(act, copy=True)
        flat = lambda x: x.reshape(N * ns, *x.shape[2:])  # noqa: E731
        for buf in (plain, packed):
            buf.push(flat(obs), act.reshape(-1), rew.reshape(-1), flat(nxt), done.reshape(-1))
        obs = nxt
    assert torch.equal(unpack_obs(packed.obs[:packed.size]), plain.obs[:plain.size])
    s1 = plain.sample(64, generator=torch.Generator(device='cuda').manual_seed(1))
    s2 = packed.sample(64, generator=torch.Generator(device='cuda').manual_seed(1))
    assert all(torch.equal(x, y) for x, y in zip(s1, s2))

    eager, graphed = SnakeBatch(N, **kw), SnakeBatch(N, **kw)
    eager.reset(); graphed.reset()
    actions = torch.randint(0, 3, (T, N, ns), dtype=torch.uint8, device='cuda', generator=g)
    gs = GraphedSteps(graphed, actions)                     # capture runs nothing
    for rep in range(2):
        want_r, want_d = [], []
        for t in range(T):
            o, r, d, _ = eager.step(actions[t], copy=True)
            want_r.append(r); want_d.append(d)
        got_o, got_r, got_d = gs.replay()
        torch.cuda.synchronize()
        assert torch.equal(got_o, o) and torch.equal(got_r, torch.stack(want_r)) and torch.equal(got_d, torch.stack(want_d))
        actions.copy_(torch.randint(0, 3, (T, N, ns), dtype=torch.uint8, device='cuda', generator=g))


def test_gpu_stepping_a_finished_env_matches_oracle():
    """Without auto-reset the reference keeps accepting steps after the episode ended (SURVEY E1, probe g3):
    dead snakes return 0 / True, a capped episode keeps moving its live snakes, and the terminal info dict is
    emitted again on every such step with the statistics accumulated since the previous emission."""
    from oracle.snake_oracle import OracleSnakeEnv, PhiloxDraws
    kw = dict(height=9, width=9, num_snakes=3, snake_length=3, vision_range=2, max_episode_steps=6)
    N, seed = 6, 77
    be = GpuBackend(N, kw, rng_mode=0, auto_reset=0, seed=seed)
    draws = [PhiloxDraws(seed, e) for e in range(N)]
    envs = [OracleSnakeEnv(draws=draws[e], **kw) for e in range(N)]
    for dr in draws:
        dr.tick()
    assert np.array_equal(be.reset(), np.stack([e.reset() for e in envs]))
    rng = np.random.RandomState(3)
    emitted = 0
    for t in range(25):
        acts = rng.randint(0, 3, size=(N, 3)).astype(np.uint8)
        obs, rew, done, info = be.step(acts)
        for e, env in enumerate(envs):
            draws[e].tick()
            o, r, d, inf = env.step([int(a) for a in acts[e]])
            assert np.array_equal(obs[e], o) and np.array_equal(rew[e], np.asarray(r)), (t, e)
            assert np.array_equal(done[e].astype(bool), np.asarray(d)), (t, e)
            assert bool(info['finished'][e]) == bool(inf), (t, e)
            if inf:
                emitted += 1
                assert list(info['rank'][e]) == list(inf['rank'])
                assert np.array_equal(info['episode_scores'][e], inf['episode_scores'])
                assert np.array_equal(info['episode_steps'][e], inf['episode_steps'])
        assert np.array_equal(be.grid()[0].reshape(N, 9, 9), np.stack([e.grid for e in envs])), t
    assert emitted >= N * 15                               # every step from the cap on emits info again
    assert be.errors() == 0
    be.close()


def test_gpu_long_spawn_pose_matches_oracle():
    """snake_length 6 on a 7x9 grid: bent spawn poses and the head-boxed pruning of the DFS table."""
    kw = dict(height=7, width=9, num_snakes=2, snake_length=6, vision_range=2, num_fruits=3)
    be = check_against_oracle_philox(GpuBackend, kw, num_envs=40, steps=60, seed=99)
    assert be.errors() == 0
    be.close()


@pytest.mark.parametrize('fs', [1, 3])
def test_gpu_masked_reset(fs):
    """snk_reset with a mask: only the selected envs restart (and get a fresh observation)."""
    from marl_snake_b200 import SnakeBatch
    N, ns = 257, 3
    b = SnakeBatch(N, num_snakes=ns, vision_range=3, frame_stack=fs, seed=8, auto_reset=False)
    b.reset()
    g = torch.Generator(device='cuda').manual_seed(2)
    for _ in range(25):
        obs, _, _, _ = b.step(torch.randint(0, 3, (N, ns), dtype=torch.uint8, device='cuda', generator=g))
    before = {k: v.clone() for k, v in b.get_state(max_cells=12).items()}
    obs_before = obs.clone()
    mask = torch.zeros(N, dtype=torch.uint8, device='cuda')
    mask[::3] = 1
    sel = mask.bool()
    obs_after = b.reset(mask=mask).clone()
    after = b.get_state(max_cells=12)
    for k in before:
        assert torch.equal(before[k][~sel], after[k][~sel]), k           # untouched envs keep their state
    assert torch.equal(obs_after[~sel], obs_before[~sel])                # ... and their observation buffer
    assert bool(after['alive'][sel].all()) and int(after['episode_length'][sel].abs().sum()) == 0
    assert bool((after['alive_counter'][sel] == ns).all()) and bool((after['length'][sel] == 3).all())
    if fs > 1:                                                           # every frame of a reset env is the first frame
        o = obs_after[sel]
        assert torch.equal(o[..., :8], o[..., 8:16]) and torch.equal(o[..., :8], o[..., 16:24])
    assert b.device_errors() == 0


@pytest.mark.parametrize('fs', [1, 4])
def test_gpu_step_without_obs_keeps_history(fs):
    """want_obs=False steps (obs pointer NULL) must leave state and frame history exactly as if rendered."""
    from marl_snake_b200 import SnakeBatch
    N, ns = 300, 4
    kw = dict(num_snakes=ns, vision_range=5, frame_stack=fs, seed=12)
    a, b = SnakeBatch(N, **kw), SnakeBatch(N, **kw)
    a.reset(); b.reset()
    g = torch.Generator(device='cuda').manual_seed(3)
    for t in range(60):
        act = torch.randint(0, 3, (N, ns), dtype=torch.uint8, device='cuda', generator=g)
        oa, ra, da, _ = a.step(act)
        ob, rb, db, _ = b.step(act, want_obs=(t % 5 == 4))
        assert torch.equal(ra, rb) and torch.equal(da, db)
        if t % 5 == 4:
            assert torch.equal(oa, ob), t


def test_gpu_host_buffer_entry_points():
    """snk_reset_host / snk_step_host (host pointers, copies inside) against the device-pointer path."""
    from marl_snake_b200 import SnakeBatch
    N, ns = 129, 4
    kw = dict(num_snakes=ns, vision_range=5, seed=31)
    dev, host = SnakeBatch(N, **kw), SnakeBatch(N, **kw)
    h_obs = torch.empty((N,) + host.obs_shape, dtype=torch.uint8).pin_memory()
    h_rew = torch.empty((N, ns), dtype=torch.float64).pin_memory()
    h_done = torch.empty((N, ns), dtype=torch.uint8).pin_memory()
    host.reset_host(h_obs)
    assert torch.equal(dev.reset().cpu(), h_obs)
    g = torch.Generator().manual_seed(5)
    for _ in range(30):
        act = torch.randint(0, 3, (N, ns), dtype=torch.uint8, generator=g)
        host.step_host(act, h_obs, h_rew, h_done)
        o, r, d, _ = dev.step(act.cuda())
        assert torch.equal(o.cpu(), h_obs) and torch.equal(r.cpu(), h_rew) and torch.equal(d.cpu(), h_done.bool())


@pytest.mark.parametrize('kw,N', [
    (dict(num_snakes=4, vision_range=5), 1237),                       # odd window: 8-byte aligned viewers only
    (dict(num_snakes=3, vision_range=2, frame_stack=3), 811),
    (dict(num_snakes=4), 300),                                        # full-grid observation
    (dict(num_snakes=1, vision_range=3), 5),                          # a few hundred bytes
])
def test_gpu_packed_host_transport_equals_raw(kw, N):
    """snk_step_host / snk_reset_host deliver the same bytes whether the observation block crosses PCIe as
    NHWC bytes or as channel bits widened by the host pool (any thread count, pageable or pinned)."""
    from marl_snake_b200 import SnakeBatch
    ns = kw['num_snakes']
    raw, packed, dev = SnakeBatch(N, seed=3, **kw), SnakeBatch(N, seed=3, **kw), SnakeBatch(N, seed=3, **kw)
    raw.set_host_transport('raw')
    packed.set_host_transport('packed', threads=3)
    assert raw.host_transport()[0] == 'raw' and packed.host_transport() == ('packed', 3)
    bufs = []
    for pin in (True, False):
        o = torch.empty((N,) + raw.obs_shape, dtype=torch.uint8)
        r, d = torch.empty((N, ns), dtype=torch.float64), torch.empty((N, ns), dtype=torch.uint8)
        bufs.append(tuple(t.pin_memory() if pin else t for t in (o, r, d)))
    (o1, r1, d1), (o2, r2, d2) = bufs
    raw.reset_host(o1); packed.reset_host(o2)
    assert torch.equal(o1, o2) and torch.equal(dev.reset().cpu(), o2)
    g = torch.Generator().manual_seed(11)
    for t in range(25):
        if t == 12:
            packed.set_host_transport('packed', threads=0)            # pool rebuilt with one thread per core
        act = torch.randint(0, 3, (N, ns), dtype=torch.uint8, generator=g)
        raw.step_host(act, o1, r1, d1); packed.step_host(act, o2, r2, d2)
        o, r, d, _ = dev.step(act.cuda())
        assert torch.equal(o1, o2) and torch.equal(r1, r2) and torch.equal(d1, d2), t
        assert torch.equal(o.cpu(), o2) and torch.equal(r.cpu(), r2)


def test_gpu_step_host_bits():
    """snk_step_host_bits delivers np.packbits(obs, little) of what snk_step_host delivers."""
    from marl_snake_b200 import SnakeBatch
    N, ns = 333, 4
    kw = dict(num_snakes=ns, vision_range=5, frame_stack=2, seed=21)
    a, b = SnakeBatch(N, **kw), SnakeBatch(N, **kw)
    a.reset(); b.reset()
    obs = torch.empty((N,) + a.obs_shape, dtype=torch.uint8).pin_memory()
    bits = torch.empty((N,) + a.obs_shape[:-1] + (a.obs_shape[-1] // 8,), dtype=torch.uint8).pin_memory()
    r1, r2 = (torch.empty((N, ns), dtype=torch.float64).pin_memory() for _ in range(2))
    d1, d2 = (torch.empty((N, ns), dtype=torch.uint8).pin_memory() for _ in range(2))
    g = torch.Generator().manual_seed(2)
    for t in range(12):
        act = torch.randint(0, 3, (N, ns), dtype=torch.uint8, generator=g)
        a.step_host(act, obs, r1, d1)
        b.step_host_bits(act, bits, r2, d2)
        assert torch.equal(r1, r2) and torch.equal(d1, d2)
        want = np.packbits(obs.numpy().reshape(-1, 8), axis=1, bitorder='little').reshape(bits.shape)
        assert np.array_equal(bits.numpy(), want), t


def test_gpu_pack_obs_roundtrip():
    """snk_pack_obs (device) and snk_widen_bits_host (host) are inverse; the packed form is np.packbits."""
    import ctypes as C
    import marl_snake_b200 as m
    b = m.SnakeBatch(77, num_snakes=4, vision_range=5, frame_stack=2, seed=8)
    obs = b.reset()
    for t in range(5):
        obs, *_ = b.step(torch.randint(0, 3, (77, 4), dtype=torch.uint8, device='cuda'))
    bits = b.pack_obs()
    assert bits.shape == (*obs.shape[:-1], obs.shape[-1] // 8)
    want = np.packbits(obs.cpu().numpy().reshape(-1, 8), axis=1, bitorder='little').reshape(bits.shape)
    assert np.array_equal(bits.cpu().numpy(), want)
    back = np.empty(obs.numel(), dtype=np.uint8)
    src = np.ascontiguousarray(bits.cpu().numpy())
    assert m.lib.snk_widen_bits_host(src.ctypes.data_as(C.c_void_p), back.ctypes.data_as(C.c_void_p), src.size, 2) == 0
    assert np.array_equal(back.reshape(obs.shape), obs.cpu().numpy())
    with pytest.raises(ValueError):
        b.pack_obs(obs[..., :4])


@pytest.mark.parametrize('N', [3, 700])
def test_gpu_step_host_info_matches_device_path(N):
    """snk_step_host_info: host buffers incl. the terminal info arrays (one output block for a few
    environments, separate copies for many) against the device-pointer call."""
    import ctypes as C
    from marl_snake_b200 import SnakeBatch
    from marl_snake_b200._lib import SnkStepExtra, check, lib
    ns = 3
    kw = dict(num_snakes=ns, height=9, width=11, vision_range=2, frame_stack=2, max_episode_steps=6, seed=13)
    dev, host = SnakeBatch(N, **kw), SnakeBatch(N, **kw)
    obs = np.empty((N,) + host.obs_shape, np.uint8)
    rew, done = np.empty((N, ns), np.float64), np.empty((N, ns), np.uint8)
    fin, rank = np.zeros(N, np.uint8), np.zeros((N, ns), np.int32)
    sc, cnt = np.zeros((N, ns), np.float64), np.zeros((3, N, ns), np.int32)
    xh = SnkStepExtra(fin.ctypes.data, rank.ctypes.data, sc.ctypes.data, cnt[0].ctypes.data, cnt[1].ctypes.data,
                      cnt[2].ctypes.data)
    p = lambda x: x.ctypes.data_as(C.c_void_p)  # noqa: E731
    check(lib.snk_reset_host(host._h, p(obs)))
    assert np.array_equal(dev.reset().cpu().numpy(), obs)
    rng = np.random.RandomState(2)
    seen = 0
    for t in range(20):
        a = rng.randint(0, 3, size=(N, ns)).astype(np.uint8)
        check(lib.snk_step_host_info(host._h, p(a), p(obs), p(rew), p(done), C.byref(xh)))
        o, r, d, info = dev.step(torch.as_tensor(a).cuda())
        assert np.array_equal(o.cpu().numpy(), obs) and np.array_equal(r.cpu().numpy(), rew)
        assert np.array_equal(d.cpu().numpy(), done.astype(bool))
        f = info['finished'].cpu().numpy()
        assert np.array_equal(f, fin.astype(bool))
        seen += int(f.sum())
        assert np.array_equal(info['rank'].cpu().numpy()[f], rank[f])
        assert np.array_equal(info['episode_scores'].cpu().numpy()[f], sc[f])
        for k, name in enumerate(('episode_steps', 'episode_fruits', 'episode_kills')):
            assert np.array_equal(info[name].cpu().numpy()[f], cnt[k][f])
    assert seen >= N * 2                                   # the step cap ended every env at least twice


@both_layouts
@pytest.mark.parametrize('kw', [dict(num_snakes=4, vision_range=5), dict(num_snakes=3, vision_range=3, frame_stack=4),
                                dict(num_snakes=9, height=16, width=16, vision_range=2, max_episode_steps=15)])
def test_gpu_exact_checkpoint_resume(monkeypatch, kw, compact):
    """snk_checkpoint_save / _load: a second batch continues bit for bit -- grid, frame history, episode
    statistics, Philox position and rollout statistics included."""
    from marl_snake_b200 import SnakeBatch, SnkError
    monkeypatch.setenv('SNK_COMPACT', compact)
    N, ns = 700, kw['num_snakes']
    a, b = SnakeBatch(N, seed=44, **kw), SnakeBatch(N, seed=44, **kw)
    a.reset()
    g = torch.Generator(device='cuda').manual_seed(1)
    for _ in range(25):
        a.step(torch.randint(0, 3, (N, ns), dtype=torch.uint8, device='cuda', generator=g))
    blob = a.save_checkpoint()
    b.load_checkpoint(blob)
    for t in range(40):
        act = torch.randint(0, 3, (N, ns), dtype=torch.uint8, device='cuda', generator=g)
        oa, ra, da, ia = a.step(act)
        ob, rb, db, ib = b.step(act)
        assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(da, db), t
        fin = ia['finished']
        assert torch.equal(fin, ib['finished']), t
        for k in ia:                              # terminal arrays are only defined for finished envs
            assert torch.equal(ia[k][fin], ib[k][fin]), (k, t)
    sa, sb = a.stats(), b.stats()
    for k in sa:                                  # counters are exact; the return sum is a float64 atomicAdd
        if k == 'return_sum':                     # reduction whose order differs from launch to launch
            assert abs(sa[k] - sb[k]) <= 1e-9 * max(1.0, abs(sa[k])), k
        else:
            assert sa[k] == sb[k], k
    other = SnakeBatch(N + 1, seed=44, **kw)
    with pytest.raises(SnkError):
        other.load_checkpoint(blob)
    monkeypatch.setenv('SNK_COMPACT', '1' if compact == '0' else '0')      # the other record layout: refused as well
    other = SnakeBatch(N, seed=44, **kw)
    with pytest.raises(SnkError):
        other.load_checkpoint(blob)


@both_layouts
def test_gpu_state_roundtrip(monkeypatch, compact):
    """get_state -> set_state on a second batch reproduces the trajectory (checkpoint / restore)."""
    from marl_snake_b200 import SnakeBatch
    monkeypatch.setenv('SNK_COMPACT', compact)
    N, ns = 200, 4
    kw = dict(num_snakes=ns, vision_range=5, seed=17)
    a, b = SnakeBatch(N, **kw), SnakeBatch(N, seed=999, num_snakes=ns, vision_range=5)
    a.reset(); b.reset()
    g = torch.Generator(device='cuda').manual_seed(9)
    for _ in range(40):
        a.step(torch.randint(0, 3, (N, ns), dtype=torch.uint8, device='cuda', generator=g))
    st = a.get_state(max_cells=64)
    obs_b = b.set_state(st['grid'].cpu().numpy(), st['alive'].cpu().numpy(), st['dir'].cpu().numpy(),
                        st['length'].cpu().numpy(), st['cells'].clamp(min=0).cpu().numpy(),
                        st['alive_counter'].cpu().numpy(), st['episode_length'].cpu().numpy())
    st2 = b.get_state(max_cells=64)
    for k in ('grid', 'head', 'tail', 'length', 'alive', 'alive_counter', 'episode_length', 'cells'):
        assert torch.equal(st[k], st2[k]), k
    # same next step; envs that drew randomness this step (fruit respawn, reset) differ by design (other seed)
    act = torch.randint(0, 3, (N, ns), dtype=torch.uint8, device='cuda', generator=g)
    oa, ra, da, ia = a.step(act)
    ob, rb, db, ib = b.step(act)
    assert torch.equal(ra, rb) and torch.equal(da, db) and torch.equal(ia['finished'], ib['finished'])
    quiet = (~ia['finished']) & (a.get_state()['grid'] == b.get_state()['grid']).all(2).all(1)
    assert int(quiet.sum()) > N // 2
    assert torch.equal(oa[quiet], ob[quiet])
    assert b.device_errors() == 0
    # A compact record stores fruit cells and bodies only: a grid that is anything but walls + fruits + the given bodies
    # cannot be represented and raises the sticky SNK_DEV_STATE bit (the full layout takes the grid as it is).
    grid = st['grid'].cpu().numpy().copy()
    stray = np.argwhere(grid[0] == 0)[0]
    grid[0][tuple(stray)] = 4                                  # a BODY cell of snake 0 that no body accounts for
    b.set_state(grid, st['alive'].cpu().numpy(), st['dir'].cpu().numpy(), st['length'].cpu().numpy(),
                st['cells'].clamp(min=0).cpu().numpy(), st['alive_counter'].cpu().numpy(), st['episode_length'].cpu().numpy())
    assert b.device_errors(clear=True) == (64 if compact == '1' else 0)


BITS_CASES = [
    (dict(num_snakes=4, vision_range=5), 1237, {}),                                   # register encode, warp-private
    (dict(num_snakes=4, vision_range=5), 700, {'SNK_COOP': '1'}),                     # register encode, cooperative
    (dict(num_snakes=4), 300, {}),                                                    # full-grid (direct) encode
    (dict(num_snakes=3, vision_range=2, frame_stack=3), 811, {}),                     # stacked
    (dict(num_snakes=4, vision_range=5, frame_stack=4), 130, {'SNK_COOP': '0'}),      # cfg3 shape warp-private: generic
    (dict(height=64, width=64, num_snakes=16, snake_length=5, vision_range=7), 40, {}),          # padded-plane encode, dual LUT
    (dict(height=64, width=64, num_snakes=16, snake_length=5, vision_range=7), 40, {'SNK_ENC_NOPAD': '1'}),   # table encode, dual LUT, generic
    (dict(height=24, width=24, num_snakes=9, snake_length=3, vision_range=9), 50, {}),            # window > 16: index arithmetic
    (dict(height=32, width=32, num_snakes=8, snake_length=4, vision_range=6), 90, {'SNK_COOP': '1'}),   # padded plane, per-viewer LUT
    (dict(num_snakes=4, vision_range=5), 400, {'SNK_ENC_LEGACY': '1'}),               # table encode, per-viewer LUT, generic
    (dict(height=13, width=11, num_snakes=2, vision_range=3), 77, {'SNK_FORCE_GENERIC': '1'}),
]


@pytest.mark.parametrize('kw,N,env', BITS_CASES)
def test_gpu_step_bits_equals_packbits_of_obs(monkeypatch, kw, N, env):
    """snk_step_bits / snk_reset_bits (channel bits written by the encode itself, no NHWC block) deliver exactly
    np.packbits of what snk_step / snk_reset deliver, for every encode flavour and tile mode."""
    from marl_snake_b200 import SnakeBatch, unpack_obs
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    ns = kw['num_snakes']
    a, b = SnakeBatch(N, seed=19, max_episode_steps=25, **kw), SnakeBatch(N, seed=19, max_episode_steps=25, **kw)
    o = a.reset()
    bits = b.reset(bits=True)
    assert bits.shape == (N,) + a.obs_shape[:-1] + (a.obs_shape[-1] // 8,)
    want = np.packbits(o.cpu().numpy().reshape(-1, 8), axis=1, bitorder='little').reshape(bits.shape)
    assert np.array_equal(bits.cpu().numpy(), want)
    g = torch.Generator(device='cuda').manual_seed(2)
    for t in range(40):
        act = torch.randint(0, 3, (N, ns), dtype=torch.uint8, device='cuda', generator=g)
        o, r1, d1, i1 = a.step(act)
        bits, r2, d2, i2 = b.step_bits(act)
        assert torch.equal(r1, r2) and torch.equal(d1, d2) and torch.equal(i1['finished'], i2['finished']), t
        assert torch.equal(unpack_obs(bits), o), t
    assert a.device_errors() == 0 and b.device_errors() == 0


def test_gpu_mixed_stream_ordering():
    """ADVICE r01: device-pointer calls on the caller's stream followed by host-buffer calls (the handle's own
    stream) and back, with no synchronisation in between, see each other's results."""
    from marl_snake_b200 import SnakeBatch
    N, ns = 20000, 4
    kw = dict(num_snakes=ns, vision_range=5, seed=3)
    a, b = SnakeBatch(N, **kw), SnakeBatch(N, **kw)
    h_obs = torch.empty((N,) + a.obs_shape, dtype=torch.uint8).pin_memory()
    h_rew = torch.empty((N, ns), dtype=torch.float64).pin_memory()
    h_done = torch.empty((N, ns), dtype=torch.uint8).pin_memory()
    side = torch.cuda.Stream()
    g = torch.Generator().manual_seed(1)
    acts = [torch.randint(0, 3, (N, ns), dtype=torch.uint8, generator=g) for _ in range(12)]
    dacts = [x.cuda() for x in acts]
    torch.cuda.synchronize()
    b.reset()
    for t in range(12):
        b.step(dacts[t])
    want = b._obs.cpu()
    with torch.cuda.stream(side):                 # device-pointer calls on a non-default stream, no sync after them
        a.reset()
        for t in range(5):
            a.step(dacts[t])
    a.step_host(acts[5], h_obs, h_rew, h_done)    # must wait for the five steps queued on `side`
    with torch.cuda.stream(side):
        for t in range(6, 11):
            a.step(dacts[t])
    a.step_host(acts[11], h_obs, h_rew, h_done)
    assert torch.equal(h_obs, want)
    assert a.stats()['env_steps'] == 12 * N        # counted on the device


def test_gpu_calls_leave_current_device_alone():
    """ADVICE r01: entry points restore the calling thread's current CUDA device."""
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    from marl_snake_b200 import SnakeBatch
    b = SnakeBatch(64, num_snakes=2, vision_range=2, device=1)
    torch.cuda.set_device(0)
    b.reset()
    b.step(torch.zeros((64, 2), dtype=torch.uint8, device='cuda:1'))
    b.stats()
    assert torch.cuda.current_device() == 0


@pytest.mark.parametrize('kw,N,T,env', [
    (dict(num_snakes=4), 4096, 24, {}),                                             # BASELINE cfg2: full-grid, cooperative tiles
    (dict(num_snakes=4, vision_range=5), 3001, 17, {'SNK_COOP': '0'}),             # warp-private tiles, ragged batch
    (dict(num_snakes=4, vision_range=5), 1500, 9, {'SNK_COOP': '1'}),
    (dict(height=64, width=64, num_snakes=16, snake_length=5, vision_range=7), 33, 12, {}),    # padded-plane encode
    (dict(height=12, width=14, num_snakes=3, vision_range=2, max_episode_steps=7), 257, 30, {}),   # resets inside the launch
    (dict(num_snakes=3, vision_range=3, frame_stack=3), 200, 8, {}),                # frame_stack > 1: T launches
])
def test_gpu_step_many_equals_single_steps(monkeypatch, kw, N, T, env):
    """snk_step_many (records resident in shared memory for T steps) is bit-identical to T calls of snk_step:
    every step's observation, rewards, dones, finished flags, the final state and the statistics."""
    from marl_snake_b200 import SnakeBatch, unpack_obs
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    ns = kw['num_snakes']
    a, b, c = (SnakeBatch(N, seed=41, **kw) for _ in range(3))
    for x in (a, b, c):
        x.reset()
    g = torch.Generator(device='cuda').manual_seed(7)
    for rep in range(2):
        acts = torch.randint(0, 3, (T, N, ns), dtype=torch.uint8, device='cuda', generator=g)
        obs_all = torch.empty((T, N) + a.obs_shape, dtype=torch.uint8, device='cuda')
        fin_all = torch.empty((T, N), dtype=torch.uint8, device='cuda')
        _, rew, done, _ = b.step_many(acts, obs=obs_all, finished=fin_all)
        last_bits = torch.empty((N,) + a.bits_shape, dtype=torch.uint8, device='cuda')
        _, rew_c, done_c, _ = c.step_many(acts, bits=last_bits)                  # last step only, as channel bits
        for t in range(T):
            o, r, d, info = a.step(acts[t])
            assert torch.equal(obs_all[t], o), (rep, t)
            assert torch.equal(rew[t], r) and torch.equal(done[t].bool(), d), (rep, t)
            assert torch.equal(fin_all[t].bool(), info['finished']), (rep, t)
        assert torch.equal(rew_c, rew) and torch.equal(done_c, done)
        assert torch.equal(unpack_obs(last_bits), o)
    sa, sb = a.get_state(max_cells=12), b.get_state(max_cells=12)
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
    st_a, st_b = a.stats(), b.stats()
    assert st_a['env_steps'] == st_b['env_steps'] == 2 * T * N and st_a['episodes'] == st_b['episodes']
    assert a.device_errors() == 0 and b.device_errors() == 0 and c.device_errors() == 0
