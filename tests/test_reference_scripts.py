"""The reference's own caller scripts, unmodified, executed against this repo's import shim (SURVEY 8b / north_star:
"drops in for test_env.py / train_dqn.py / train_ga.py").  Each scenario runs in a subprocess (tests/ref_script_driver.py)
so the `marlenv` module name resolves to exactly one implementation.  The same scenarios run on the CPU against the
unmodified reference package first: that proves the harness (shortened configs, `neat` / cv2-window stand-ins) on the
code the scripts were written for."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRIVER = os.path.join(ROOT, 'tests', 'ref_script_driver.py')
SCRIPTS = os.path.join(ROOT, 'oracle', '_ref', 'scripts')
needs_scripts = pytest.mark.skipif(not os.path.exists(os.path.join(SCRIPTS, 'train_dqn.py')),
                                   reason='oracle/_ref/scripts absent (make -C oracle ref needs the original checkout)')
SCENARIOS = ['test_env', 'train_dqn', 'train_ga']


def run(backend, scenario, work):
    env = dict(os.environ)
    env.pop('PYTHONPATH', None)
    p = subprocess.run([sys.executable, DRIVER, backend, scenario, str(work)], cwd=str(work), env=env,
                       capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-4000:]
    return json.loads(p.stdout.strip().splitlines()[-1])


@needs_scripts
@pytest.mark.parametrize('scenario', SCENARIOS)
def test_harness_on_the_unmodified_reference(scenario, tmp_path):
    out = run('reference', scenario, tmp_path)
    assert out['env_module'].startswith(os.path.join(ROOT, 'oracle', '_ref'))


@pytest.mark.gpu
@needs_scripts
@pytest.mark.parametrize('scenario', SCENARIOS)
def test_reference_scripts_run_on_the_cuda_path(scenario, tmp_path):
    out = run('ours', scenario, tmp_path)
    lib_name = os.path.basename(os.environ.get('SNK_LIB_PATH', 'libsnk.so'))      # e.g. libsnk_dbg.so, the debug-checks build
    assert any(s.endswith(lib_name) for s in out['native_so']), out
    if scenario == 'test_env':
        assert out['gui_calls'].get('imshow', 0) == out['steps']       # one window frame per env step (RenderGUI)
    if scenario == 'train_dqn':
        assert out['updates'] > 20 and out['video'] > 0
