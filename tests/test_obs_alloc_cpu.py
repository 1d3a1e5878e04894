"""CPU-side checks of the observation allocator (snk_alloc_obs / snk_free_obs): exported through the C ABI, and
libsnk.so reaches the driver API through the runtime, so loading it needs no libcuda."""
import ctypes as C
import os
import shutil
import subprocess

import pytest


def test_alloc_exports_are_in_the_abi():
    import marl_snake_b200 as m
    from marl_snake_b200._lib import PROTOTYPES
    for name in ('snk_alloc_obs', 'snk_free_obs'):
        assert name in PROTOTYPES and hasattr(m.lib, name)


@pytest.mark.skipif(shutil.which('readelf') is None, reason='needs readelf')
def test_library_does_not_link_libcuda():
    import marl_snake_b200 as m
    dyn = subprocess.run(['readelf', '-d', m.LIB_PATH], capture_output=True, text=True, check=True).stdout
    needed = [ln for ln in dyn.splitlines() if '(NEEDED)' in ln]
    assert needed and not [ln for ln in needed if 'libcuda.so' in ln], needed
    assert os.path.exists(m.LIB_PATH)


def test_alloc_rejects_bad_arguments_and_foreign_pointers():
    import marl_snake_b200 as m
    p, comp = C.c_void_p(), C.c_int(0)
    assert m.lib.snk_alloc_obs(0, 0, C.byref(p), C.byref(comp)) == -1            # zero size
    assert m.lib.snk_alloc_obs(0, 1024, None, C.byref(comp)) == -1
    assert m.lib.snk_free_obs(None) == 0
    x = C.create_string_buffer(64)
    assert m.lib.snk_free_obs(C.cast(x, C.c_void_p)) == -1                          # not from snk_alloc_obs
    assert b'snk_alloc_obs' in m.lib.snk_last_error()
