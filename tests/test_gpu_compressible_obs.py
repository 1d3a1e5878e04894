"""The observation buffer of SnakeBatch in compressible device memory (snk_alloc_obs): same bytes as a plain
cudaMalloc buffer from every call that writes it, a returned observation outlives its batch, graph replays and
host-buffer calls keep working, and the block lands on the batch's device."""
import ctypes as C
import gc

import numpy as np
import pytest
import torch

from marl_snake_b200 import GraphedSteps, SnakeBatch

pytestmark = pytest.mark.gpu

CFG5 = dict(height=20, width=20, num_snakes=4, snake_length=3, vision_range=5, frame_stack=1)
CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED = 107
CU_POINTER_ATTRIBUTE_DEVICE_ORDINAL = 9


def _libcuda():
    cu = C.CDLL('libcuda.so.1')
    assert cu.cuInit(0) == 0
    return cu


def _device_supports_compression(device):
    v = C.c_int(0)
    assert _libcuda().cuDeviceGetAttribute(C.byref(v), CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, device) == 0
    return bool(v.value)


def _cross_map(n=16):
    m = np.zeros((n, n), dtype=np.uint8)
    m[0, :] = m[-1, :] = m[:, 0] = m[:, -1] = 1
    m[n // 2, 3:n - 3] = 1
    m[3:n - 3, n // 2] = 1
    return m


def _pair(num_envs, **kw):
    """Two batches from the same seed: `comp` keeps its snk_alloc_obs buffer, `plain` gets a torch.empty one."""
    comp = SnakeBatch(num_envs, seed=11, **kw)
    plain = SnakeBatch(num_envs, seed=11, **kw)
    plain._obs = torch.empty_like(plain._obs)
    return comp, plain


def test_obs_compressed_follows_the_device():
    b = SnakeBatch(64, **CFG5)
    assert b.obs_compressed == _device_supports_compression(b.device.index)
    with pytest.raises(AttributeError):
        b.obs_compressed = False
    b.close()


@pytest.mark.parametrize('num_envs,kw', [
    (1 << 20, CFG5),
    (3000, dict(CFG5, frame_stack=4)),
    (2000, dict(wall_map=_cross_map(), num_snakes=4, vision_range=4, done_mode='any')),
], ids=['cfg5_full', 'frame_stack4', 'wall_map'])
def test_step_reset_set_state_are_byte_equal_to_a_plain_buffer(num_envs, kw):
    comp, plain = _pair(num_envs, **kw)
    assert torch.equal(comp.reset(), plain.reset())
    g = torch.Generator(device='cuda').manual_seed(3)
    for t in range(40):
        a = torch.randint(0, 3, (num_envs, comp.num_snakes), dtype=torch.uint8, device='cuda', generator=g)
        oc, rc, dc, ic = comp.step(a)
        op, rp, dp, ip = plain.step(a)
        assert torch.equal(oc, op) and torch.equal(rc, rp) and torch.equal(dc, dp), f'step {t}'
        assert torch.equal(ic['finished'], ip['finished'])
    mask = (torch.arange(num_envs, device='cuda') % 3 == 0).to(torch.uint8)
    assert torch.equal(comp.reset(mask), plain.reset(mask))
    st = comp.get_state(max_cells=max(2, int(comp.get_state()['length'].max())))
    args = [st[k].cpu().numpy() for k in ('grid', 'alive', 'dir', 'length', 'cells', 'alive_counter', 'episode_length')]
    cells, length = args[4], args[3]
    cells[np.arange(cells.shape[-1]) >= length[..., None]] = 0          # entries past a body are unspecified
    assert torch.equal(comp.set_state(*args), plain.set_state(*args))
    assert comp.device_errors() == 0 and plain.device_errors() == 0
    comp.close()
    plain.close()


def test_obs_stays_readable_after_close():
    b = SnakeBatch(4096, seed=5, **CFG5)
    obs = b.reset()
    a = torch.zeros((4096, 4), dtype=torch.uint8, device='cuda')
    obs, _, _, _ = b.step(a)
    want = obs.clone()
    b.close()
    del b
    gc.collect()
    torch.cuda.synchronize()
    assert torch.equal(obs, want)
    assert int(obs.view(-1, 8).sum(1).max()) == 1


def test_graph_replay_writes_into_the_compressible_buffer():
    N, T = 8192, 6
    comp, plain = _pair(N, **CFG5)
    comp.reset()
    plain.reset()
    acts = torch.randint(0, 3, (T, N, 4), dtype=torch.uint8, device='cuda',
                         generator=torch.Generator(device='cuda').manual_seed(9))
    graphed = GraphedSteps(comp, acts)
    obs, rew, _ = graphed.replay()
    assert obs.data_ptr() == comp._obs.data_ptr()
    for t in range(T):
        op, rp, _, _ = plain.step(acts[t], want_info=False)
        assert torch.equal(rew[t], rp)
    assert torch.equal(obs, op)
    comp.close()
    plain.close()


@pytest.mark.parametrize('transport', ['raw', 'packed'])
def test_step_host_with_both_transports(transport):
    N = 20000
    host, dev = SnakeBatch(N, seed=8, **CFG5), SnakeBatch(N, seed=8, **CFG5)
    host.set_host_transport(transport, threads=2)
    h_obs = torch.empty((N,) + host.obs_shape, dtype=torch.uint8).pin_memory()
    h_rew = torch.empty((N, 4), dtype=torch.float64).pin_memory()
    h_done = torch.empty((N, 4), dtype=torch.uint8).pin_memory()
    host.reset_host(h_obs)
    assert torch.equal(h_obs, dev.reset().cpu())
    g = torch.Generator().manual_seed(2)
    for t in range(10):
        a = torch.randint(0, 3, (N, 4), dtype=torch.uint8, generator=g).pin_memory()
        host.step_host(a, h_obs, h_rew, h_done)
        o, r, d, _ = dev.step(a.cuda(), want_info=False)
        assert torch.equal(h_obs, o.cpu()) and torch.equal(h_rew, r.cpu()) and torch.equal(h_done.bool(), d.cpu())
    host.close()
    dev.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_buffer_lands_on_the_batch_device():
    b = SnakeBatch(4096, device=1, seed=1, **CFG5)
    assert b._obs.device == torch.device('cuda', 1)
    ordinal = C.c_int(-1)
    assert _libcuda().cuPointerGetAttribute(C.byref(ordinal), CU_POINTER_ATTRIBUTE_DEVICE_ORDINAL,
                                            C.c_uint64(b._obs.data_ptr())) == 0
    assert ordinal.value == 1
    assert b.obs_compressed == _device_supports_compression(1)
    with torch.cuda.device(1):
        ref = SnakeBatch(4096, device=1, seed=1, **CFG5)
        ref._obs = torch.empty_like(ref._obs)
        assert torch.equal(b.reset(), ref.reset())
        ref.close()
    b.close()
