"""Seeded programs that switch between every entry point on ONE batch, checked after every operation against a model
built from the Python oracle (oracle/snake_oracle.py with PhiloxDraws).

The per-entry-point tests compare each call with a twin batch driven by plain step() calls.  Here a single batch goes
through step / step_bits / step_many / the host-buffer calls / every reset flavour / set_state / checkpoint swaps /
CUDA-graph replays / rollout.collect in random order, and each call must both return what the model returns and leave
the batch in a state the next call continues correctly.  The CPU part checks the program generator and pins the
model's event-tick and set_state rules against the host build of the kernel's rule source (HostSim)."""
import numpy as np
import pytest

from oracle.snake_oracle import CoopOracleSnakeEnv, OracleSnakeEnv, PhiloxDraws

CFG4_REW = {'fruit': 10.0, 'kill': 1.0, 'lose': -1.0, 'win': 0.1, 'time': -0.001}
STAT_KEYS = ('episodes', 'return_sum', 'episode_steps_sum', 'fruits_sum', 'kills_sum', 'deaths', 'env_steps')
SMALL_BLOCK_LIMIT = 64 * 1024      # snk_step_host_info: one mapped output block up to this size, device mirrors above


def _cross_map():
    from test_wall_maps import cross_map
    return cross_map()


# name, N, SnakeBatch kwargs, environment knobs (None = unset), seed, env_id_offset
CASES = [
    ('cfg5_20x20', 96, dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5, max_episode_steps=40),
     {'SNK_COOP': None, 'SNK_COMPACT': None}, 5, 0),
    ('warp_private_compact', 70, dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5,
                                      max_episode_steps=40), {'SNK_COOP': '0', 'SNK_COMPACT': '1'}, 6, 0),
    ('stacked_fs4', 48, dict(height=20, width=20, num_snakes=4, vision_range=5, frame_stack=4),
     {'SNK_COOP': '1', 'SNK_COMPACT': '0'}, 7, 0),
    ('human_9x12', 33, dict(height=9, width=12, num_snakes=3, snake_length=4, vision_range=2, frame_stack=3,
                            max_episode_steps=12, observer='human'), {'SNK_COOP': None, 'SNK_COMPACT': None}, 8, 0),
    ('full_grid_small_host', 5, dict(height=12, width=12, num_snakes=2), {'SNK_COOP': None, 'SNK_COMPACT': None}, 9, 0),
    ('cfg4_64x64', 6, dict(height=64, width=64, num_snakes=16, snake_length=5, vision_range=7, reward_dict=CFG4_REW),
     {'SNK_COOP': None, 'SNK_COMPACT': None}, 10, 0),
    ('wall_map_coop', 40, dict(wall_map='cross', num_snakes=4, vision_range=4, done_mode='any'),
     {'SNK_COOP': None, 'SNK_COMPACT': '1'}, 11, 0),
    ('one_snake_offset', 130, dict(height=10, width=10, num_snakes=1, num_fruits=4),
     {'SNK_COOP': '0', 'SNK_COMPACT': None}, 0x9E3779B97F4A7C15, 1000),
]

KINDS = ('step', 'step_bits', 'step_many', 'step_host', 'step_host_bits', 'step_host_info', 'reset', 'reset_host',
         'state', 'checkpoint', 'graph', 'collect')
HOST_KINDS = ('step_host', 'step_host_bits', 'step_host_info', 'reset_host')


def resolve(kw):
    kw = dict(kw)
    if kw.get('wall_map') == 'cross':
        kw['wall_map'] = _cross_map()
        kw['height'], kw['width'] = kw['wall_map'].shape
    return kw


def obs_shape(kw):
    kw = resolve(kw)
    vr = kw.get('vision_range') or 0
    oh, ow = (2 * vr + 1,) * 2 if vr else (kw.get('height', 20), kw.get('width', 20))
    return kw['num_snakes'], oh, ow, 8 * kw.get('frame_stack', 1)


def small_layout_total(N, kw):
    """small_layout() of snk_api.cu: the single output block of snk_step_host_info for a few environments."""
    up = lambda x: (x + 15) & ~15  # noqa: E731
    ns = kw['num_snakes']
    nn = N * ns
    env_bytes = int(np.prod(obs_shape(kw)))
    return up(nn) + up(N * env_bytes) + up(nn * 8) + up(nn) + up(N) + up(nn * 4) + up(nn * 8) + up(3 * nn * 4)


# ---------------------------------------------------------------------------------------------------- the model
class OracleShard:
    """N oracle environments stepped the way the kernel steps a shard: every step ticks each env's Philox event once
    (an env that finishes is auto-reset with the same event), reset() ticks every env, reset(mask) only the selected
    ones, set_state keeps the event, zeroes the episode statistics and restarts the frame history from the current
    frame.  Accumulates the rollout statistics of snk_stats."""

    def __init__(self, N, kw, seed, env_id_offset=0):
        kw = resolve(kw)
        self.done_mode = kw.pop('done_mode', 'all')
        cls = CoopOracleSnakeEnv if self.done_mode == 'any' else OracleSnakeEnv
        self.draws = [PhiloxDraws(seed, env_id_offset + e) for e in range(N)]
        self.envs = [cls(draws=self.draws[e], **kw) for e in range(N)]
        self.N, self.ns = N, kw['num_snakes']
        self.stats = dict.fromkeys(STAT_KEYS, 0.0)

    def obs(self):
        return np.stack([e._stacked() for e in self.envs])

    def reset(self, mask=None):
        for e, env in enumerate(self.envs):
            if mask is None or mask[e]:
                self.draws[e].tick()
                env.reset()
        return self.obs()

    def step(self, actions):
        N, ns = self.N, self.ns
        rew = np.zeros((N, ns)); done = np.zeros((N, ns), bool); fin = np.zeros(N, bool)
        info = dict(rank=np.zeros((N, ns), np.int64), episode_scores=np.zeros((N, ns)),
                    episode_steps=np.zeros((N, ns)), episode_fruits=np.zeros((N, ns)), episode_kills=np.zeros((N, ns)))
        st = self.stats
        for e, env in enumerate(self.envs):
            self.draws[e].tick()
            was = np.asarray(env.alive, bool)
            _, r, d, inf = env.step([int(a) for a in actions[e]])
            st['deaths'] += float(np.sum(was & ~np.asarray(env.alive, bool)))      # step_group's newly_dead
            rew[e], done[e] = r, d
            if inf:
                fin[e] = True
                for k in info:
                    info[k][e] = inf[k]
                st['episodes'] += 1
                st['return_sum'] += float(np.sum(inf['episode_scores']))
                st['episode_steps_sum'] += env.episode_length
                st['fruits_sum'] += float(np.sum(inf['episode_fruits']))
                st['kills_sum'] += float(np.sum(inf['episode_kills']))
                env.reset()                                                         # same event as the step
        st['env_steps'] += N
        return self.obs(), rew, done, fin, info

    def state_args(self):
        """Arguments of set_state that reproduce the current state (cells from the oracle's bodies)."""
        ex = [e.export_state() for e in self.envs]
        L = max(2, max(len(b) for e in self.envs for b in e.body))
        W = self.envs[0].grid_shape[1]
        cells = np.zeros((self.N, self.ns, L), np.int32)
        for q, env in enumerate(self.envs):
            for i, b in enumerate(env.body):
                for k, (r, c) in enumerate(b):
                    cells[q, i, k] = r * W + c
        return dict(grid=np.stack([x['grid'] for x in ex]), alive=np.stack([x['alive'] for x in ex]),
                    dir=np.stack([x['dir'] for x in ex]).astype(np.uint8), length=np.stack([x['length'] for x in ex]),
                    cells=cells, alive_counter=np.array([x['alive_counter'] for x in ex], np.int32),
                    episode_length=np.array([x['episode_length'] for x in ex], np.int32))

    def import_state(self, a):
        for q, env in enumerate(self.envs):
            env.import_state(a['grid'][q], a['alive'][q], a['dir'][q], a['length'][q], a['cells'][q],
                             a['alive_counter'][q], a['episode_length'][q])
        return self.obs()

    def set_state_roundtrip(self):
        return self.import_state(self.state_args())

    def export(self):
        ex = [e.export_state() for e in self.envs]
        return {k: np.stack([np.asarray(x[k]) for x in ex]) for k in ('grid', 'alive', 'length', 'alive_counter',
                                                                    'episode_length')}


# ---------------------------------------------------------------------------------------------------- programs
def obs_valid_after(op, valid):
    """Whether the batch's own observation buffer holds the current observation of every env after `op`."""
    k = op['kind']
    if k == 'step':
        return op['want_obs']
    if k == 'reset':
        if op['bits']:
            return False
        return True if not op['masked'] else valid
    if k in ('state', 'graph'):
        return True
    if k == 'collect':
        return valid
    return False


def make_program(seed, n_actions=3):
    rng = np.random.RandomState(seed % (1 << 32))
    weights = dict(step=5, step_bits=2, step_many=3, step_host=2, step_host_bits=1, step_host_info=2, reset=2,
                   reset_host=1, state=1, checkpoint=1, graph=2, collect=3)
    kinds = list(weights)
    p = np.array([weights[k] for k in kinds], float)
    seq = list(rng.choice(kinds, size=rng.randint(150, 251), p=p / p.sum()))
    for k in KINDS:                                           # every kind at least twice
        while seq.count(k) < 2:
            seq.insert(rng.randint(0, len(seq) + 1), k)

    def params(k):
        op = dict(kind=str(k), seed=int(rng.randint(1 << 30)))
        if k == 'step':
            op.update(want_obs=bool(rng.rand() < 0.75), want_info=bool(rng.rand() < 0.7), side=bool(rng.rand() < 0.5))
        elif k == 'step_many':
            op.update(T=int(rng.choice([1, 2, 5])), obs=str(rng.choice(['every', 'last', 'none'])),
                      bits=str(rng.choice(['every', 'last', 'none'])), finished=bool(rng.rand() < 0.5))
            if 'every' in (op['obs'], op['bits']) and 'last' in (op['obs'], op['bits']):
                op['bits'] = op['obs']                        # the library takes both per step or both last-step only
        elif k in HOST_KINDS:
            op.update(xfer=str(rng.choice(['raw', 'packed'])))
        elif k == 'reset':
            op.update(masked=bool(rng.rand() < 0.5), bits=bool(rng.rand() < 0.4))
        elif k == 'collect':
            op.update(steps=int(rng.randint(1, 6)), packed=bool(rng.rand() < 0.5), threshold=int(rng.randint(2, 15)),
                      penalty=float(rng.choice([-1.0, -0.25])), max_steps=int(rng.randint(4, 40)))
        return op

    prog = [params(k) for k in seq]
    # collect must run on a current observation at least twice and meet an outdated one at least once
    while True:
        valid, ok, stale = True, [], []
        for j, op in enumerate(prog):
            if op['kind'] == 'collect':
                (ok if valid else stale).append(j)
            valid = obs_valid_after(op, valid)
        if len(ok) >= 2 and stale:
            return prog
        cols = ok + stale
        j = cols[rng.randint(len(cols))]
        if len(ok) < 2:
            prog.insert(j, dict(kind='reset', seed=int(rng.randint(1 << 30)), masked=False, bits=False))
        else:
            prog.insert(j, dict(kind='step_bits', seed=int(rng.randint(1 << 30))))


# ---------------------------------------------------------------------------------------------------- CPU part
@pytest.mark.parametrize('case', CASES, ids=[c[0] for c in CASES])
def test_program_generator_covers_every_entry_point(case):
    name, N, kw, env, seed, off = case
    prog = make_program(seed)
    assert 150 <= len(prog) <= 300
    for k in KINDS:
        assert sum(op['kind'] == k for op in prog) >= 2, k
    sm = [op for op in prog if op['kind'] == 'step_many']
    assert {op['T'] for op in sm} and all(op['T'] in (1, 2, 5) for op in sm)
    assert any(op['kind'] == 'step' and op['side'] for op in prog)
    resets = [(op['masked'], op['bits']) for op in prog if op['kind'] == 'reset']
    assert len(resets) >= 2
    valid, seen = True, set()
    for op in prog:
        if op['kind'] == 'collect':
            seen.add(valid)
        valid = obs_valid_after(op, valid)
    assert seen == {True, False}


def test_cases_cover_both_host_paths():
    """snk_step_host_info keeps a few environments in one mapped block and copies through device mirrors above
    64 KB: the cases must reach both sides of that threshold."""
    sizes = {c[0]: small_layout_total(c[1], c[2]) for c in CASES}
    assert any(s <= SMALL_BLOCK_LIMIT for s in sizes.values()), sizes
    assert any(s > SMALL_BLOCK_LIMIT for s in sizes.values()), sizes
    assert sizes['full_grid_small_host'] <= SMALL_BLOCK_LIMIT < sizes['cfg5_20x20']


@pytest.mark.parametrize('case', [c for c in CASES if c[0] in ('cfg5_20x20', 'human_9x12', 'wall_map_coop',
                                                                    'one_snake_offset', 'stacked_fs4')],
                         ids=lambda c: c[0])
def test_model_matches_hostsim(case):
    """The model's event ticks and set_state rule against the kernel's rule source compiled for the host, on programs
    made of the calls HostSim has: step, full reset and a set_state round trip."""
    from hostsim_util import HostSim
    name, N, kw, env, seed, off = case
    N = min(N, 24)
    rk = resolve(kw)
    done_mode = rk.pop('done_mode', 'all')
    hs = HostSim(N, rk, rng_mode=0, seed=seed, env_id_offset=off, done_mode={'all': 0, 'any': 1}[done_mode])
    model = OracleShard(N, kw, seed, off)
    n_actions = 5 if rk.get('observer') == 'human' else 3
    rng = np.random.RandomState(seed & 0xFFFF)
    assert np.array_equal(hs.reset(), model.reset())
    H, W = model.envs[0].grid_shape
    for t in range(120):
        u = rng.rand()
        if u < 0.05:
            assert np.array_equal(hs.reset(), model.reset()), t
        elif u < 0.12:
            a = model.state_args()
            want = model.import_state(a)
            got = hs.set_state(a['grid'], a['alive'], a['dir'], a['length'], a['cells'], a['alive_counter'],
                               a['episode_length'])
            assert np.array_equal(got, want), t
        else:
            acts = rng.randint(0, n_actions, size=(N, model.ns)).astype(np.uint8)
            obs, rew, done, info = hs.step(acts)
            mo, mr, md, mf, mi = model.step(acts)
            assert np.array_equal(rew, mr) and np.array_equal(done.astype(bool), md), t
            assert np.array_equal(info['finished'].astype(bool), mf), t
            assert np.array_equal(obs, mo), t
            for k in mi:
                assert np.array_equal(info[k][mf], mi[k][mf]), (k, t)
        grid, counter, _ = hs.grid()
        ex = model.export()
        assert np.array_equal(grid.reshape(N, H, W), ex['grid']), t
        assert np.array_equal(counter, ex['alive_counter']), t
    assert hs.errors() == 0
    hs.close()


# ---------------------------------------------------------------------------------------------------- GPU part
def make_net(ch, oh, ow, n_actions):
    import torch
    from test_gpu_rollout import ExactNet
    net = ExactNet(ch, oh, ow)
    if n_actions != 3:
        g = torch.Generator().manual_seed(1)
        net.head = torch.nn.Linear(4 * oh * ow, n_actions, bias=False)
        with torch.no_grad():
            net.head.weight.copy_(torch.randint(-2, 3, net.head.weight.shape, generator=g).float())
    return net.cuda()


def packbits(obs):
    return np.packbits(obs.reshape(-1, 8), axis=1, bitorder='little').reshape(*obs.shape[:-1], obs.shape[-1] // 8)


class Runner:
    """Drives one SnakeBatch and the model through a program, comparing after every operation."""

    def __init__(self, N, kw, seed, off):
        import torch
        from marl_snake_b200 import DeviceReplayBuffer, SnakeBatch
        self.torch = torch
        self.N, self.seed, self.off = N, seed, off
        rk = resolve(kw)
        self.bkw = dict(rk, seed=seed, env_id_offset=off)
        self.b = SnakeBatch(N, **self.bkw)
        self.model = OracleShard(N, kw, seed, off)
        self.ns = self.model.ns
        self.n_actions = 5 if rk.get('observer') == 'human' else 3
        self.H, self.W = self.model.envs[0].grid_shape
        ns_, oh, ow, ch = self.b.obs_shape
        self.net = make_net(ch, oh, ow, self.n_actions)
        cap = N * self.ns * 5
        self.bufs = {False: DeviceReplayBuffer(cap, self.b.obs_shape[1:], self.b.device),
                     True: DeviceReplayBuffer(cap, self.b.obs_shape[1:], self.b.device, pack=self.b)}
        pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory()  # noqa: E731
        nn = (N, self.ns)
        self.h = dict(act=pin(nn, torch.uint8), obs=pin((N,) + self.b.obs_shape, torch.uint8),
                      bits=pin((N,) + self.b.bits_shape, torch.uint8), rew=pin(nn, torch.float64),
                      done=pin(nn, torch.uint8), fin=pin((N,), torch.uint8), rank=pin(nn, torch.int32),
                      scores=pin(nn, torch.float64), steps=pin(nn, torch.int32), fruits=pin(nn, torch.int32),
                      kills=pin(nn, torch.int32))
        self.side = torch.cuda.Stream()
        self.gs = None
        self.pending = None               # a step issued on the side stream whose outputs are checked after the next op
        self.counts = dict(collect_ran=0, collect_refused=0)

    # -- helpers
    def actions(self, seed, T=None):
        rng = np.random.RandomState(seed)
        shape = (self.N, self.ns) if T is None else (T, self.N, self.ns)
        return rng.randint(0, self.n_actions, size=shape).astype(np.uint8)

    def check_step_outputs(self, tag, want, rew, done, obs=None, fin=None, info=None):
        mo, mr, md, mf, mi = want
        assert np.array_equal(rew, mr), ('rewards', tag)
        assert np.array_equal(np.asarray(done).astype(bool), md), ('dones', tag)
        if obs is not None:
            assert np.array_equal(obs, mo), ('obs', tag)
        if fin is not None:
            assert np.array_equal(np.asarray(fin).astype(bool), mf), ('finished', tag)
        if info is not None:
            for k, v in info.items():
                assert np.array_equal(np.asarray(v)[mf], mi[k][mf]), (k, tag)

    def check_state(self, tag):
        st = self.b.get_state()
        ex = self.model.export()
        got = {k: v.cpu().numpy() for k, v in st.items()}
        assert np.array_equal(got['grid'], ex['grid']), ('grid', tag)
        for k in ('alive', 'length', 'alive_counter', 'episode_length'):
            assert np.array_equal(got[k], ex[k]), (k, tag)

    def info_np(self, info):
        return {k: info[k].cpu().numpy() for k in ('rank', 'episode_scores', 'episode_steps', 'episode_fruits',
                                                     'episode_kills')}

    def flush_pending(self):
        if self.pending is None:
            return
        tag, want, outs = self.pending
        self.pending = None
        self.torch.cuda.synchronize()
        o, r, d, info = outs
        self.check_step_outputs(tag, want, r.cpu().numpy(), d.cpu().numpy(),
                                None if o is None else o.cpu().numpy(),
                                info['finished'].cpu().numpy() if info else None, self.info_np(info) if info else None)

    # -- operations
    def op_step(self, op, tag):
        torch = self.torch
        a = self.actions(op['seed'])
        da = torch.as_tensor(a).cuda()
        want = self.model.step(a)
        if op['side']:
            self.flush_pending()
            self.side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(self.side):
                outs = self.b.step(da, copy=True, want_obs=op['want_obs'], want_info=op['want_info'])
            self.pending = (tag, want, outs)
            self._keep = da                                   # the side stream still reads it
            return False                                      # state is checked after the next op
        o, r, d, info = self.b.step(da, want_obs=op['want_obs'], want_info=op['want_info'])
        self.check_step_outputs(tag, want, r.cpu().numpy(), d.cpu().numpy(),
                                None if o is None else o.cpu().numpy(),
                                info['finished'].cpu().numpy() if info else None, self.info_np(info) if info else None)
        return True

    def op_step_bits(self, op, tag):
        a = self.actions(op['seed'])
        want = self.model.step(a)
        bits, r, d, info = self.b.step_bits(self.torch.as_tensor(a).cuda())
        assert np.array_equal(bits.cpu().numpy(), packbits(want[0])), ('bits', tag)
        self.check_step_outputs(tag, want, r.cpu().numpy(), d.cpu().numpy(), None,
                                info['finished'].cpu().numpy(), self.info_np(info))
        return True

    def op_step_many(self, op, tag):
        torch = self.torch
        T, N = op['T'], self.N
        a = self.actions(op['seed'], T)
        wants = [self.model.step(a[t]) for t in range(T)]
        dev = self.b.device

        def buf(mode, shape):
            if mode == 'none':
                return None
            return torch.full(((T, N) if mode == 'every' else (N,)) + shape, 0xAB, dtype=torch.uint8, device=dev)
        obs, bits = buf(op['obs'], self.b.obs_shape), buf(op['bits'], self.b.bits_shape)
        fin = torch.full((T, N), 7, dtype=torch.uint8, device=dev) if op['finished'] else None
        o, r, d, bt = self.b.step_many(torch.as_tensor(a).cuda(), obs=obs, rewards=None, dones=None, bits=bits,
                                       finished=fin)
        r, d = r.cpu().numpy(), d.cpu().numpy()
        for t in range(T):
            self.check_step_outputs(tag + (t,), wants[t], r[t], d[t], None,
                                    None if fin is None else fin[t].cpu().numpy())
        for mode, x, conv in ((op['obs'], o, lambda v: v), (op['bits'], bt, packbits)):
            if mode == 'every':
                x = x.cpu().numpy()
                for t in range(T):
                    assert np.array_equal(x[t], conv(wants[t][0])), ('step_many block', mode, tag, t)
            elif mode == 'last':
                assert np.array_equal(x.cpu().numpy(), conv(wants[-1][0])), ('step_many last block', tag)
        return True

    def op_host(self, op, tag):
        b, h, k = self.b, self.h, op['kind']
        b.set_host_transport(op['xfer'])
        if k == 'reset_host':
            want = self.model.reset()
            b.reset_host(h['obs'])
            assert np.array_equal(h['obs'].numpy(), want), ('reset_host obs', tag)
            return True
        a = self.actions(op['seed'])
        h['act'].copy_(self.torch.as_tensor(a))
        want = self.model.step(a)
        if k == 'step_host':
            b.step_host(h['act'], h['obs'], h['rew'], h['done'])
            self.check_step_outputs(tag, want, h['rew'].numpy(), h['done'].numpy(), h['obs'].numpy())
        elif k == 'step_host_bits':
            b.step_host_bits(h['act'], h['bits'], h['rew'], h['done'])
            self.check_step_outputs(tag, want, h['rew'].numpy(), h['done'].numpy())
            assert np.array_equal(h['bits'].numpy(), packbits(want[0])), ('host bits', tag)
        else:
            b.step_host_info(h['act'], h['obs'], h['rew'], h['done'], finished=h['fin'], rank=h['rank'],
                             episode_scores=h['scores'], episode_steps=h['steps'], episode_fruits=h['fruits'],
                             episode_kills=h['kills'])
            info = dict(rank=h['rank'].numpy(), episode_scores=h['scores'].numpy(), episode_steps=h['steps'].numpy(),
                        episode_fruits=h['fruits'].numpy(), episode_kills=h['kills'].numpy())
            self.check_step_outputs(tag, want, h['rew'].numpy(), h['done'].numpy(), h['obs'].numpy(),
                                    h['fin'].numpy(), info)
        return True

    def op_reset(self, op, tag):
        torch, b = self.torch, self.b
        mask = None
        if op['masked']:
            mask = np.random.RandomState(op['seed']).rand(self.N) < 0.35
        want = self.model.reset(mask)
        prev = (b._bits_buffer() if op['bits'] else b._obs).clone()
        out = b.reset(mask=None if mask is None else torch.as_tensor(mask.astype(np.uint8)).cuda(), bits=op['bits'])
        out, prev = out.cpu().numpy(), prev.cpu().numpy()
        if op['bits']:
            want = packbits(want)
        sel = np.ones(self.N, bool) if mask is None else mask
        assert np.array_equal(out[sel], want[sel]), ('reset selected', tag)
        assert np.array_equal(out[~sel], prev[~sel]), ('reset keeps the others', tag)
        return True

    def op_state(self, op, tag):
        b = self.b
        longest = max(2, int(b.get_state()['length'].max()))
        st = b.get_state(max_cells=longest)
        want = self.model.set_state_roundtrip()
        got = b.set_state(st['grid'].cpu().numpy(), st['alive'].cpu().numpy(), st['dir'].cpu().numpy(),
                          st['length'].cpu().numpy(), st['cells'].clamp(min=0).cpu().numpy(),
                          st['alive_counter'].cpu().numpy(), st['episode_length'].cpu().numpy())
        assert np.array_equal(got.cpu().numpy(), want), ('set_state obs', tag)
        return True

    def op_checkpoint(self, op, tag):
        from marl_snake_b200 import SnakeBatch
        blob = self.b.save_checkpoint()
        nb = SnakeBatch(self.N, **self.bkw)
        nb.load_checkpoint(blob)
        self.b.close()
        self.b, self.gs = nb, None
        self.bufs[True].pack = nb
        return True

    def op_graph(self, op, tag):
        torch = self.torch
        from marl_snake_b200 import GraphedSteps
        if self.gs is None:
            self.gs_actions = torch.zeros((3, self.N, self.ns), dtype=torch.uint8, device=self.b.device)
            self.gs = GraphedSteps(self.b, self.gs_actions)
        a = self.actions(op['seed'], 3)
        self.gs_actions.copy_(torch.as_tensor(a))
        wants = [self.model.step(a[t]) for t in range(3)]
        o, r, d = self.gs.replay()
        r, d = r.cpu().numpy(), d.cpu().numpy()
        for t in range(3):
            self.check_step_outputs(tag + (t,), wants[t], r[t], d[t])
        assert np.array_equal(o.cpu().numpy(), wants[-1][0]), ('graph obs', tag)
        return True

    def op_collect(self, op, tag, valid):
        torch = self.torch
        from marl_snake_b200 import collect
        buf = self.bufs[op['packed']]
        if not valid:
            before = self.b._mutations
            with pytest.raises(ValueError, match=r'reset\(\) or step\(\)'):
                collect(self.b, self.net, op['steps'], buf, epsilon=0.0,
                        early_death=(op['threshold'], op['penalty']), max_steps=op['max_steps'])
            assert self.b._mutations == before
            self.counts['collect_refused'] += 1
            return True
        # the model runs the same loop on its own observations
        m = self.model
        N, ns = self.N, self.ns
        exp = []
        for _ in range(op['steps']):
            obs = m.obs()
            x = torch.as_tensor(obs.reshape(N * ns, *obs.shape[2:])).cuda().permute(0, 3, 1, 2).float()
            acts = self.net(x).float().argmax(dim=1).to(torch.uint8).cpu().numpy().reshape(N, ns)
            alive = np.stack([np.asarray(e.alive, bool) for e in m.envs])
            age = np.array([e.episode_length for e in m.envs])
            acts = np.where(alive, acts, 0).astype(np.uint8)
            nobs, rew, done, fin, _ = m.step(acts)
            rew = rew + (done & (age < op['threshold'])[:, None]) * op['penalty']
            for e in range(N):
                for i in range(ns):
                    if alive[e, i]:
                        exp.append((obs[e, i], acts[e, i], np.float32(rew[e, i]), nobs[e, i], done[e, i]))
            cut = np.array([env.episode_length >= op['max_steps'] for env in m.envs])
            if cut.any():
                m.reset(cut)
        pos0 = buf.pos
        n = int(collect(self.b, self.net, op['steps'], buf, epsilon=0.0,
                        early_death=(op['threshold'], op['penalty']), max_steps=op['max_steps']))
        assert n == len(exp), ('collect count', tag, n, len(exp))
        self.counts['collect_ran'] += 1
        if n == 0:
            return True
        idx = torch.as_tensor((pos0 + np.arange(n)) % buf.capacity).cuda()
        from marl_snake_b200 import unpack_obs
        got_o, got_no = buf.obs[idx], buf.next_obs[idx]
        if buf.pack is not None:
            got_o, got_no = unpack_obs(got_o), unpack_obs(got_no)
        assert np.array_equal(got_o.cpu().numpy(), np.stack([t[0] for t in exp])), ('collect obs', tag)
        assert np.array_equal(got_no.cpu().numpy(), np.stack([t[3] for t in exp])), ('collect next_obs', tag)
        assert np.array_equal(buf.action[idx].cpu().numpy(), np.array([t[1] for t in exp], np.uint8)), ('action', tag)
        assert np.array_equal(buf.reward[idx].cpu().numpy(), np.array([t[2] for t in exp], np.float32)), ('rew', tag)
        assert np.array_equal(buf.done[idx].cpu().numpy(), np.array([t[4] for t in exp], bool)), ('done', tag)
        return True

    def run(self, prog, name):
        torch = self.torch
        self.model.reset()
        o = self.b.reset()
        assert np.array_equal(o.cpu().numpy(), self.model.obs())
        valid = True
        for j, op in enumerate(prog):
            tag = (name, j, op['kind'])
            k = op['kind']
            if self.pending is not None and k not in HOST_KINDS:
                torch.cuda.current_stream().wait_stream(self.side)   # the caller orders device-pointer calls
            if k in HOST_KINDS:
                checked = self.op_host(op, tag)
            elif k == 'collect':
                checked = self.op_collect(op, tag, valid)
            else:
                checked = getattr(self, 'op_' + k)(op, tag)
            if checked:
                self.flush_pending()
                self.check_state(tag)
            valid = obs_valid_after(op, valid)
        self.flush_pending()
        self.check_state((name, 'end'))
        got, want = self.b.stats(), self.model.stats
        for k in STAT_KEYS:
            if k == 'return_sum':                  # float64 atomicAdd reduction, order differs from launch to launch
                assert abs(got[k] - want[k]) <= 1e-9 * max(1.0, abs(want[k])), (k, got[k], want[k])
            else:
                assert got[k] == want[k], (k, got[k], want[k])
        assert self.b.device_errors() == 0
        assert self.counts['collect_ran'] >= 2 and self.counts['collect_refused'] >= 1


def set_knobs(monkeypatch, env):
    for k, v in env.items():
        if v is None:
            monkeypatch.delenv(k, raising=False)
        else:
            monkeypatch.setenv(k, v)


@pytest.mark.gpu
@pytest.mark.parametrize('case', CASES, ids=[c[0] for c in CASES])
def test_gpu_entry_point_sequence_matches_oracle(monkeypatch, case):
    name, N, kw, env, seed, off = case
    set_knobs(monkeypatch, env)
    r = Runner(N, kw, seed, off)
    try:
        r.run(make_program(seed, r.n_actions), name)
    finally:
        r.b.close()


@pytest.mark.gpu
def test_gpu_host_call_after_graph_replay_waits_for_it():
    """GraphedSteps.replay() launches captured kernels the library never sees; a host-buffer call right after it
    (no synchronisation) must still run after them.  Compared with a twin batch stepped eagerly."""
    import torch
    from marl_snake_b200 import GraphedSteps, SnakeBatch
    N, ns, T = 20000, 4, 8
    kw = dict(num_snakes=ns, vision_range=5, seed=23)
    a, b = SnakeBatch(N, **kw), SnakeBatch(N, **kw)
    h_obs = torch.empty((N,) + a.obs_shape, dtype=torch.uint8).pin_memory()
    h_rew = torch.empty((N, ns), dtype=torch.float64).pin_memory()
    h_done = torch.empty((N, ns), dtype=torch.uint8).pin_memory()
    h_fin = torch.empty((N,), dtype=torch.uint8).pin_memory()
    g = torch.Generator().manual_seed(4)
    a.reset(); b.reset()
    acts = torch.empty((T, N, ns), dtype=torch.uint8, device='cuda')
    gs = GraphedSteps(a, acts)
    for call in ('step_host', 'step_host_info', 'reset_host'):
        new = torch.randint(0, 3, (T, N, ns), dtype=torch.uint8, generator=g)
        host_act = torch.randint(0, 3, (N, ns), dtype=torch.uint8, generator=g).pin_memory()
        acts.copy_(new.cuda())
        torch.cuda.synchronize()
        for t in range(T):
            b.step(acts[t])
        gs.replay()                                            # no synchronisation before the host-buffer call
        if call == 'step_host':
            a.step_host(host_act, h_obs, h_rew, h_done)
            o, r, d, _ = b.step(host_act.cuda())
        elif call == 'step_host_info':
            a.step_host_info(host_act, h_obs, h_rew, h_done, finished=h_fin)
            o, r, d, info = b.step(host_act.cuda())
            assert torch.equal(h_fin.cuda().bool(), info['finished'])
        else:
            a.reset_host(h_obs)
            o = b.reset()
            r = d = None
        assert torch.equal(h_obs, o.cpu()), call
        if r is not None:
            assert torch.equal(h_rew, r.cpu()) and torch.equal(h_done, d.cpu().to(torch.uint8)), call
    assert a.stats()['env_steps'] == b.stats()['env_steps'] == 2 * (T + 1) * N + T * N
    assert a.device_errors() == 0


@pytest.mark.gpu
def test_gpu_step_many_rejects_bad_output_buffers():
    """step_many refuses rewards / dones / finished of the wrong dtype, shape, layout or device with ValueError
    before anything is launched: the next call continues the trajectory as if nothing happened.  Every bad buffer
    here is large enough to hold what the library would write into it."""
    import torch
    N, kw, seed = 40, dict(height=12, width=12, num_snakes=3, vision_range=3, max_episode_steps=15), 31
    r = Runner(N, kw, seed, 0)
    b, m, T, ns = r.b, r.model, 5, 3
    m.reset(); b.reset()
    dev = b.device
    rng = np.random.RandomState(0)
    good_r = torch.empty((T, N, ns), dtype=torch.float64, device=dev)
    good_d = torch.empty((T, N, ns), dtype=torch.uint8, device=dev)
    bad = [
        dict(rewards=torch.empty((T, N, ns, 2), dtype=torch.float32, device=dev)),                 # float32
        dict(rewards=torch.empty((T, N, ns * 2), dtype=torch.float64, device=dev)[..., ::2]),      # strided view
        dict(rewards=torch.empty((T * N * ns,), dtype=torch.float64, device=dev)),                 # wrong shape
        dict(dones=torch.empty((T, N, ns), dtype=torch.bool, device=dev)),                         # bool
        dict(dones=torch.empty((T, N, ns), dtype=torch.int32, device=dev)),                        # int32
        dict(dones=torch.empty((T, N, ns * 2), dtype=torch.uint8, device=dev)[..., ::2]),          # strided view
        dict(finished=torch.empty((T, N), dtype=torch.uint8).pin_memory()),                        # host memory
        dict(finished=torch.empty((T, N), dtype=torch.int32, device=dev)),                         # int32
    ]
    for j, extra in enumerate(bad):
        a = rng.randint(0, 3, size=(T, N, ns)).astype(np.uint8)
        args = dict(rewards=good_r, dones=good_d)
        args.update(extra)
        with pytest.raises(ValueError):
            b.step_many(torch.as_tensor(a).cuda(), **args)
        a = rng.randint(0, 3, size=(N, ns)).astype(np.uint8)       # the trajectory goes on unchanged
        want = m.step(a)
        o, rw, d, info = b.step(torch.as_tensor(a).cuda())
        r.check_step_outputs(('bad step_many', j), want, rw.cpu().numpy(), d.cpu().numpy(), o.cpu().numpy(),
                             info['finished'].cpu().numpy())
        r.check_state(('bad step_many', j))
    assert b.device_errors() == 0
    b.close()
