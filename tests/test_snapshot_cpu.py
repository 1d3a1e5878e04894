"""CPU-side checks of per-env snapshot / restore (snk_snapshot_bytes / snk_snapshot / snk_restore): the calls are exported
through the C ABI and refuse a null handle, SnakeBatch checks its arguments before it calls the library, and the three
new kernels are in libsnk.so within a register and stack budget."""
import ctypes as C
import re
import shutil
import subprocess

import pytest
import torch

SNAPSHOT_CALLS = ('snk_snapshot_bytes', 'snk_snapshot', 'snk_restore')


def test_snapshot_calls_are_exported():
    import marl_snake_b200 as m
    from marl_snake_b200._lib import PROTOTYPES
    for name in SNAPSHOT_CALLS:
        assert name in PROTOTYPES and hasattr(m.lib, name), name


def test_snapshot_error_bit_is_named():
    from marl_snake_b200._lib import DEV_ERRORS
    assert 256 in DEV_ERRORS and 'snapshot' in DEV_ERRORS[256]


def test_snapshot_calls_refuse_a_null_handle():
    import marl_snake_b200 as m
    buf = (C.c_uint8 * 64)()
    p = C.cast(buf, C.c_void_p)
    assert m.lib.snk_snapshot_bytes(None) == 0
    assert m.lib.snk_snapshot(None, None, 1, p, None) == -1
    assert 'null argument' in m.lib.snk_last_error().decode()
    assert m.lib.snk_restore(None, p, 1, p, None, None, None, None) == -1
    assert 'null argument' in m.lib.snk_last_error().decode()


def fake_batch(N=6, slot=272):
    """A SnakeBatch shell on the CPU with just what the argument checks of snapshot / restore read (they run before any
    library call, so no handle is needed)."""
    from marl_snake_b200 import SnakeBatch

    class Shell(SnakeBatch):
        snapshot_bytes = slot                                 # the real property asks the library
    b = object.__new__(Shell)
    b.num_envs, b.num_snakes, b.device = N, 2, torch.device('cpu')
    b._h = C.c_void_p()
    return b


@pytest.fixture
def batch():
    return fake_batch()


def test_snapshot_checks_env_ids(batch):
    with pytest.raises(ValueError, match='integer CUDA tensor'):
        batch.snapshot(torch.zeros(3, dtype=torch.float32))
    with pytest.raises(ValueError, match='integer CUDA tensor'):
        batch.snapshot(torch.zeros((2, 2), dtype=torch.int64))
    with pytest.raises(ValueError, match='integer CUDA tensor'):
        batch.snapshot([0, 1])
    with pytest.raises(ValueError, match='env ids'):
        batch.snapshot(torch.zeros(7, dtype=torch.int64))
    with pytest.raises(ValueError, match=r'shape \[2, 272\]'):
        batch.snapshot(torch.zeros(2, dtype=torch.int64), out=torch.zeros((3, 272), dtype=torch.uint8))


@pytest.mark.parametrize('bad', [
    torch.zeros((2, 256), dtype=torch.uint8),                 # row width is not snapshot_bytes
    torch.zeros((2, 272), dtype=torch.int8),                  # dtype
    torch.zeros(544, dtype=torch.uint8),                      # flat
    torch.zeros((0, 272), dtype=torch.uint8),                 # no slot
    torch.zeros((272, 2), dtype=torch.uint8).t(),             # not contiguous
    torch.zeros(2 * 272 + 8, dtype=torch.uint8)[8:].view(2, 272),   # misaligned
], ids=['width', 'dtype', 'flat', 'empty', 'strided', 'misaligned'])
def test_restore_checks_the_snapshot_tensor(batch, bad):
    with pytest.raises(ValueError, match='snapshots must be'):
        batch.restore(bad, torch.full((6,), -1, dtype=torch.int32))


def test_restore_checks_its_index_arguments(batch):
    snaps = torch.zeros((2, 272), dtype=torch.uint8)
    with pytest.raises(ValueError, match='needs src or env_ids'):
        batch.restore(snaps)
    with pytest.raises(ValueError, match='not both'):
        batch.restore(snaps, torch.full((6,), -1, dtype=torch.int32), env_ids=torch.zeros(1, dtype=torch.int32))
    with pytest.raises(ValueError, match='one entry per environment'):
        batch.restore(snaps, torch.full((5,), -1, dtype=torch.int32))
    with pytest.raises(ValueError, match='integer CUDA tensor'):
        batch.restore(snaps, torch.full((6,), -1.0))
    with pytest.raises(ValueError, match='one entry per env id'):
        batch.restore(snaps, env_ids=torch.arange(3), slots=torch.zeros(2, dtype=torch.int64))


def test_snapshot_kernels_keep_their_register_budget():
    """The copy kernels are bandwidth bound: they need few registers and no stack, and the emit kernel of frame stacks
    runs one warp per env without spilling."""
    if not shutil.which('cuobjdump'):
        pytest.skip('cuobjdump not on PATH')
    import marl_snake_b200 as m
    out = subprocess.run(['cuobjdump', '-res-usage', m.LIB_PATH], capture_output=True, text=True, timeout=300).stdout
    found = {name: (int(reg), int(stack)) for name, reg, stack in
             re.findall(r'Function (\S*(?:snk_snapshot_kernel|snk_restore_kernel|snk_emit_stacked_kernel)\S*):\s*\n'
                        r'\s*REG:(\d+) STACK:(\d+)', out)}
    for kernel, count, max_reg in (('snk_snapshot_kernel', 2, 32), ('snk_restore_kernel', 2, 32),
                                   ('snk_emit_stacked_kernel', 1, 64)):
        hits = [v for k, v in found.items() if kernel in k]
        assert len(hits) == count, (kernel, found)
        for reg, stack in hits:
            assert reg <= max_reg and stack == 0, (kernel, reg, stack)
