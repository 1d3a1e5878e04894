"""make_snake and the agent wrappers, same names and return contract as the reference's
marlenv/wrappers.py (make_snake :203-223, SingleAgent :84-105, SingleMultiAgent :107-124).

The reference vectorises with one OS process per environment (gym AsyncVectorEnv, :211-212); here
`num_envs > 1` is one `SnakeBatch` on the GPU with the reference worker's auto-reset rule (:138-146).
"""
import numpy as np
import torch

from .env import SnakeBatch, _HostStepper
from .registration import make
from .spaces import Box, Discrete


class _Wrapper:
    def __init__(self, env):
        self.env = env
        self.action_space = env.action_space
        self.observation_space = env.observation_space

    def __getattr__(self, name):
        if name.startswith('_'):
            raise AttributeError(name)
        return getattr(self.env, name)

    @property
    def unwrapped(self):
        return self.env.unwrapped

    def reset(self, **kwargs):
        return self.env.reset(**kwargs)

    def step(self, action, **kwargs):
        return self.env.step(action, **kwargs)

    def close(self):
        return self.env.close()


def _obs_hw(env):
    vr = getattr(env, 'vision_range', None)
    return (vr * 2 + 1, vr * 2 + 1) if vr else tuple(env.grid_shape)


class SingleAgent(_Wrapper):
    """num_snakes == 1: squeeze the snake axis (wrappers.py:84-105)."""

    def __init__(self, env):
        super().__init__(env)
        assert env.num_snakes == 1, "Number of player must be one"
        self.action_space = Discrete(len(env.action_dict))
        self.observation_space = Box(0, 255, (*_obs_hw(env), env.obs_ch), np.uint8)

    def reset(self, **kwargs):
        return self.env.reset(**kwargs)[0]

    def step(self, action, **kwargs):
        obs, rews, dones, infos = self.env.step([action], **kwargs)
        return obs[0], rews[0], dones[0], {}


class SingleMultiAgent(_Wrapper):
    """num_snakes > 1: per-snake Discrete(3) action space, obs [ns, h, w, c] (wrappers.py:107-124)."""

    def __init__(self, env):
        super().__init__(env)
        self.action_space = Discrete(len(env.action_dict))
        self.observation_space = Box(0, 255, (env.num_snakes, *_obs_hw(env), getattr(env, 'obs_ch', 3)), np.uint8)


class RenderGUI(_Wrapper):
    """The reference's window / video wrapper (wrappers.py:20-82): render() draws the env's `render_fancy`
    frame in a cv2 window and optionally appends it to an mp4.  Needs cv2 and a display; without them
    render() still returns the RGB frame."""

    def __init__(self, env, window_name="Snake AI", save_video=False, video_path="output.mp4", fps=20):
        super().__init__(env)
        self.window_name, self.render_size = window_name, 30
        self.save_video, self.video_path, self.fps = save_video, video_path, fps
        self.window_initialized, self.video_writer = False, None

    def render(self):
        img_rgb = self.env.render_fancy(cell_size=self.render_size)
        try:
            import cv2
        except ImportError:
            return img_rgb
        img_bgr = cv2.cvtColor(img_rgb, cv2.COLOR_RGB2BGR)
        try:
            if not self.window_initialized:
                cv2.namedWindow(self.window_name, cv2.WINDOW_NORMAL)
                cv2.resizeWindow(self.window_name, img_bgr.shape[1], img_bgr.shape[0])
                self.window_initialized = True
            cv2.imshow(self.window_name, img_bgr)
            cv2.waitKey(1)
        except cv2.error:
            pass                                   # headless box
        if self.save_video:
            if self.video_writer is None:
                h, w, _ = img_bgr.shape
                self.video_writer = cv2.VideoWriter(self.video_path, cv2.VideoWriter_fourcc(*"mp4v"), self.fps, (w, h))
            self.video_writer.write(img_bgr)
        return img_rgb

    def close(self):
        if self.video_writer is not None:
            self.video_writer.release()
        if self.window_initialized:
            try:
                import cv2
                cv2.destroyWindow(self.window_name)
            except Exception:                      # noqa: BLE001  (headless box / cv2 gone)
                pass
        super().close()


class VectorSnakeEnv:
    """`num_envs` environments stepped by one kernel launch.  By default returns host arrays shaped like
    gym's vector API (obs [N, ns, h, w, c], rewards [N, ns], dones [N, ns], tuple of info dicts) through the
    host-buffer C-ABI call (`snk_step_host_info`: pinned buffers, packed PCIe transport for large batches);
    `copy=False` hands out the env's own buffers instead of copies (gym's `AsyncVectorEnv(copy=...)`).
    `output='torch'` returns the batch's CUDA tensors and a dict of info tensors instead."""

    def __init__(self, num_envs, num_snakes, output='numpy', copy=True, **kwargs):
        self.batch = SnakeBatch(num_envs, num_snakes=num_snakes, auto_reset=True, **kwargs)
        self.num_envs, self.num_snakes, self.output, self.copy = num_envs, num_snakes, output, copy
        b = self.batch
        self.action_dict = b.action_dict
        self.vision_range, self.obs_ch, self.grid_shape = b.vision_range, b.obs_ch, b.grid_shape
        single = b.obs_shape if num_snakes > 1 else b.obs_shape[1:]
        self.single_observation_space = Box(0, 255, single, np.uint8)
        self.observation_space = Box(0, 255, (num_envs, *single), np.uint8)
        self.single_action_space = self.action_space = Discrete(len(self.action_dict))
        self._act = torch.zeros((num_envs, num_snakes), dtype=torch.uint8, device=b.device)
        if output != 'torch':
            self._host = _HostStepper(b, pinned=True)

    def _squeeze(self, x):
        return x[:, 0] if self.num_snakes == 1 else x

    def _out(self, x):
        x = self._squeeze(x)
        return x.copy() if self.copy else x

    def reset(self):
        if self.output == 'torch':
            return self._squeeze(self.batch.reset())
        self._host.reset()
        return self._out(self._host.obs)

    def step(self, actions):
        if self.output == 'torch':
            if isinstance(actions, torch.Tensor) and actions.is_cuda:
                self._act.copy_(actions.reshape(self.num_envs, self.num_snakes))
            else:
                self._act.copy_(torch.as_tensor(np.asarray(actions, dtype=np.uint8).reshape(self.num_envs, self.num_snakes)))
            obs, rew, done, info = self.batch.step(self._act)
            return self._squeeze(obs), self._squeeze(rew), self._squeeze(done), info
        if isinstance(actions, torch.Tensor):
            actions = actions.cpu().numpy()
        a = np.asarray(actions).reshape(self.num_envs, self.num_snakes)
        if self.batch.observer == 'snake' and ((a < 0) | (a > 2)).any():
            # the reference looks an action up only for live snakes (snake_env.py:321, 606)
            alive = self.batch.get_state()['alive'].cpu().numpy().astype(bool)
            bad = ((a < 0) | (a > 2)) & alive
            if bad.any():
                raise KeyError(int(a[bad][0]))
            a = np.where((a < 0) | (a > 2), 0, a)
        elif self.batch.observer == 'human':
            a = np.where((a < 0) | (a > 4), 0, a)
        hs = self._host
        hs.act[...] = a
        hs.step()
        infos = [{} for _ in range(self.num_envs)]
        if self.num_snakes > 1 and hs.fin.any():
            for e in np.nonzero(hs.fin)[0]:
                infos[e] = hs.info(e)
        return self._out(hs.obs), self._out(hs.rew), self._out(hs.done.view(np.bool_)), tuple(infos)

    def close(self):
        self.batch.close()


def make_snake(num_envs=1, num_snakes=4, env_id="Snake-v1", **kwargs):
    """Same signature and 4-tuple return as the reference (wrappers.py:203-223):
    (env, None, None, {'action_info': {'action_n': 3}, 'num_envs', 'num_snakes'})."""
    if num_envs > 1:
        coop = env_id.lower() == 'snakecoop-v1'
        env = VectorSnakeEnv(num_envs, num_snakes, done_mode='any' if coop else 'all', **kwargs)
        action_n = env.action_space.n
    else:
        wrapper = SingleMultiAgent if num_snakes > 1 else SingleAgent
        for k in ('output', 'copy'):
            kwargs.pop(k, None)
        env = wrapper(make(env_id, num_snakes=num_snakes, **kwargs))
        action_n = env.action_space.n
    properties = {'action_info': {'action_n': action_n}, 'num_envs': num_envs, 'num_snakes': num_snakes}
    return env, None, None, properties
