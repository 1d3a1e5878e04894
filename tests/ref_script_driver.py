"""Runs ONE of the reference's own caller scripts, unmodified, against an environment backend (TEST INFRASTRUCTURE).

    python tests/ref_script_driver.py <backend> <scenario> <workdir>

backend   'ours'       repo root first on sys.path: `from marlenv.marlenv.wrappers import make_snake, RenderGUI`
                       (test_env.py:1, train_dqn.py:22, train_ga.py:25) resolves to this repo's import shim, i.e. the
                       CUDA step path behind the C ABI.  Needs a GPU.
          'reference'  the unmodified reference package from oracle/_ref behind oracle/gym_stub.  CPU only; this leg
                       exists so that the harness itself (stubs, shortened configs) is proven on the reference first.
scenario  'test_env'   the original's test_env.py as __main__: make_snake -> RenderGUI -> reset -> render/step until
                       all(done) -> close
          'train_dqn'  train_dqn.Trainer(config).train() for a few short episodes including update_model(),
                       target-net sync and checkpoint save/delete (train_dqn.py:187-199, 228-381), then
                       DQN_Evaluator.evaluate with render=True (RenderGUI + mp4 writer, :582-676)
          'train_ga'   train_ga.run_neat's environment loop: make_snake as :263-274, FeatureExtractor on the DQN
                       checkpoint written by the train_dqn scenario, eval_genomes (:224-258) on two genomes

The scripts are read from oracle/_ref/scripts/ (copied there, git-ignored, by `make -C oracle ref` from the
original's checkout).  Third-party packages that are absent from the image (`neat`; cv2 windows on a headless box)
are replaced by inert stand-ins -- none of them touches the environment.
Prints one JSON line with what happened; exit code 0 = the script ran to completion.
"""
import importlib.util
import json
import os
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SCRIPTS = os.path.join(ROOT, 'oracle', '_ref', 'scripts')


def select_backend(backend):
    for p in list(sys.path):
        if os.path.abspath(p or '.') in (ROOT, HERE, SCRIPTS):
            sys.path.remove(p)
    if backend == 'ours':
        sys.path.insert(0, ROOT)
        from marlenv.marlenv.wrappers import make_snake
        import marl_snake_b200
        assert make_snake is marl_snake_b200.make_snake
        return marl_snake_b200.LIB_PATH
    ref = os.path.join(ROOT, 'oracle', '_ref')
    sys.path.insert(0, os.path.join(ROOT, 'oracle', 'gym_stub'))
    sys.path.insert(0, ref)
    import marlenv
    import marlenv.wrappers
    assert marlenv.__file__.startswith(ref), marlenv.__file__
    # the scripts spell the package `marlenv.marlenv` (they are run from the reference checkout's root)
    sys.modules['marlenv.marlenv'] = marlenv
    sys.modules['marlenv.marlenv.wrappers'] = marlenv.wrappers
    marlenv.marlenv = marlenv
    return marlenv.__file__


def install_stand_ins(counters):
    """`neat` (not in the image) and cv2's window calls (headless box)."""
    if importlib.util.find_spec('neat') is None:
        neat = types.ModuleType('neat')

        class LinearNet:
            def __init__(self, genome):
                self.bias = getattr(genome, 'bias', 0.0)

            def activate(self, x):
                s = float(sum(x[:8])) + self.bias
                return [s, -s, 0.5 * s + 0.01]

        class FeedForwardNetwork:
            @staticmethod
            def create(genome, config):
                return LinearNet(genome)

        neat.nn = types.SimpleNamespace(FeedForwardNetwork=FeedForwardNetwork)
        for name in ('DefaultGenome', 'DefaultReproduction', 'DefaultSpeciesSet', 'DefaultStagnation', 'Config',
                     'Population', 'StdOutReporter'):
            setattr(neat, name, type(name, (), {}))
        sys.modules['neat'] = neat
    try:
        import cv2
    except ImportError:
        return

    def count(name):
        def f(*a, **k):
            counters[name] = counters.get(name, 0) + 1
            return 0
        return f
    for name in ('namedWindow', 'resizeWindow', 'imshow', 'waitKey', 'destroyWindow', 'destroyAllWindows'):
        setattr(cv2, name, count(name))


def load_script(name):
    path = os.path.join(SCRIPTS, name + '.py')
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def scenario_test_env(out):
    import runpy
    import time
    import builtins
    time.sleep = lambda s: None
    steps = {'n': 0}
    real_print = builtins.print

    def quiet_print(*a, **k):
        if a and a[0] == 'obs = ':
            steps['n'] += 1
            assert a[1].shape == (4, 11, 11, 8) and a[1].dtype.name == 'uint8', (a[1].shape, a[1].dtype)
            return
        real_print(*a, **k)
    builtins.print = quiet_print
    try:
        runpy.run_path(os.path.join(SCRIPTS, 'test_env.py'), run_name='__main__')
    finally:
        builtins.print = real_print
    out['steps'] = steps['n']
    assert steps['n'] >= 1


def short_dqn_config(m, work):
    cfg = m.Config()
    cfg.NUM_EPISODES, cfg.MAX_STEPS_PER_EPISODE = 10, 60
    cfg.HEIGHT = cfg.WIDTH = 12                 # the Q-net's first dense layer is h*w*64 x 256
    cfg.BATCH_SIZE, cfg.MIN_BUFFER_SIZE, cfg.BUFFER_SIZE = 32, 64, 4000
    cfg.TARGET_UPDATE_FREQ, cfg.SAVE_FREQ, cfg.KEEP_LAST_N, cfg.SAVE_BEST_ONLY = 2, 2, 2, True
    cfg.SAVE_DIR, cfg.LOG_DIR = os.path.join(work, 'checkpoints'), os.path.join(work, 'runs_dqn')
    cfg.RESUME_FROM = None
    return cfg


def scenario_train_dqn(out, work):
    m = load_script('train_dqn')
    cfg = short_dqn_config(m, work)
    trainer = m.Trainer(cfg)
    losses = []
    real_update = trainer.update_model

    def counting_update():
        loss = real_update()
        if loss is not None:
            losses.append(loss)
        return loss
    trainer.update_model = counting_update
    trainer.train()
    out['updates'], out['buffer'] = len(losses), len(trainer.memory)
    out['checkpoints'] = sorted(os.listdir(cfg.SAVE_DIR))
    assert len(losses) > 20 and all(l == l for l in losses), 'update_model never ran'
    assert 'shared_model_final.pth' in out['checkpoints']
    # a second trainer resumes from a numbered checkpoint (load_checkpoint, :359-371) and runs one more episode
    cfg2 = short_dqn_config(m, work)
    cfg2.RESUME_FROM, cfg2.NUM_EPISODES = 10, 11
    m.Trainer(cfg2).train()
    # evaluation mode with the GUI wrapper and the mp4 writer
    os.chdir(work)
    ev = m.DQN_Evaluator(config=cfg, model_class=m.DQN, checkpoint_tag='final')
    reward, timelife = ev.evaluate(num_episodes=1, render=True)
    out['eval'] = [float(reward), float(timelife)]
    out['video'] = os.path.getsize(os.path.join(work, f'snake_eval_{cfg.HEIGHT}x{cfg.WIDTH}.mp4'))
    assert timelife >= 1 and out['video'] > 0


def scenario_train_ga(out, work):
    os.chdir(work)
    dqn = load_script('train_dqn')
    cfg = short_dqn_config(dqn, work)
    ckpt = os.path.join(cfg.SAVE_DIR, 'shared_model_final.pth')
    if not os.path.exists(ckpt):                # standalone run: a random-weight checkpoint of the right shape
        import torch
        os.makedirs(cfg.SAVE_DIR, exist_ok=True)
        net = dqn.DQN((4, cfg.HEIGHT, cfg.WIDTH, 8), 3)
        torch.save({'policy_net': net.state_dict()}, ckpt)
    m = load_script('train_ga')
    m.HEIGHT, m.WIDTH = cfg.HEIGHT, cfg.WIDTH
    m.RESULT_FILENAME = os.path.join(work, 'hybrid_neat_best.pkl')
    m.env, _, _, props = m.make_snake(                                   # as run_neat, train_ga.py:263-274
        num_envs=1, num_snakes=m.NUM_SNAKES, height=m.HEIGHT, width=m.WIDTH, snake_length=m.SNAKE_LENGTH,
        reward_dict={'fruit': +10.0, 'kill': +0.0, 'lose': -20.0, 'win': +0.0, 'time': -0.03})
    m.extractor = m.FeatureExtractor(ckpt, m.env.observation_space.shape)
    genomes = [(i, types.SimpleNamespace(bias=0.1 * i, fitness=None)) for i in range(2)]
    m.eval_genomes(genomes, config=None)
    out['fitness'] = [g.fitness for _, g in genomes]
    assert all(isinstance(f, float) and f == f for f in out['fitness'])
    assert os.path.exists(m.RESULT_FILENAME)
    m.env.close()


def main():
    backend, scenario, work = sys.argv[1:4]
    os.makedirs(work, exist_ok=True)
    import numpy as np
    import random
    counters = {}
    out = {'backend': backend, 'scenario': scenario}
    out['env_module'] = select_backend(backend)
    install_stand_ins(counters)
    np.random.seed(7)
    random.seed(7)
    if scenario == 'test_env':
        scenario_test_env(out)
    elif scenario == 'train_dqn':
        scenario_train_dqn(out, work)
    elif scenario == 'train_ga':
        scenario_train_ga(out, work)
    else:
        raise SystemExit('unknown scenario ' + scenario)
    out['gui_calls'] = counters
    if backend == 'ours':
        loaded = [l.split()[-1] for l in open('/proc/self/maps') if 'libsnk' in l]
        out['native_so'] = sorted(set(loaded))
        assert out['native_so'], 'libsnk.so is not loaded: the scripts did not run on the CUDA path'
    print(json.dumps(out))


if __name__ == '__main__':
    main()
