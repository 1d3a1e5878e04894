import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _ensure_native_builds():
    """The suite needs libsnk.so (and, for the host simulation, g++): build what is missing so that a fresh
    checkout can run `pytest` directly.  On the GPU box the built files travel with the snapshot."""
    import shutil
    import subprocess
    lib = os.path.join(ROOT, 'marl-snake_b200', 'libsnk.so')
    if not os.path.exists(lib) and shutil.which('nvcc'):
        subprocess.check_call(['make', '-s', '-C', os.path.join(ROOT, 'marl-snake_b200', 'csrc')],
                              stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)


def pytest_configure(config):
    _ensure_native_builds()
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    config.addinivalue_line("markers", "needs_reference: needs the original MARL-Snake project: its checkout at "
                                       "SNK_REFERENCE_DIR or BASELINE.json's reference_path, or its install in oracle/_ref")


def pytest_collection_modifyitems(config, items):
    from oracle.cpu_runner import reference_search_path
    have_ref = reference_search_path() is not None
    try:
        import torch
        have_gpu = torch.cuda.is_available()
    except Exception:
        have_gpu = False
    for item in items:
        if 'needs_reference' in item.keywords and not have_ref:
            item.add_marker(pytest.mark.skip(reason='original MARL-Snake not found (SNK_REFERENCE_DIR / BASELINE.json reference_path / oracle/_ref)'))
        if 'gpu' in item.keywords and not have_gpu:
            item.add_marker(pytest.mark.skip(reason='no CUDA device'))
