"""A device-resident stand-in for the emulator side of MultiEnv, for measuring the path with synthetic inputs
(SURVEY 2 #11: "replaced by a synthetic batched env for measurement"): raw 210x160x3 frame pairs, rewards and
terminal flags come from pre-generated device buffers; each step runs the K-PRE kernel to produce the stacked
S x S x k observations (84 x 84 x 4 by default) exactly as FrameskipWrapper -> PreprocessFrameWrapper ->
FrameStackWrapper -> _AutoResetWrapper would (a2c_acktr.py:175-215 wrapper order, frameskip max over the last two
frames)."""
import torch

from ... import spaces
from .wrappers import BatchedAtariPreprocessor, check_frame_shape
import numpy as np


class DeviceAtariMultiEnv:
    device_resident = True

    def __init__(self, num_envs, num_actions=4, pool_frames=64, terminal_prob=0.01, seed=0, device=None, size=84,
                 num_stacked_frames=4):
        size, num_stacked_frames = check_frame_shape(size, num_stacked_frames)
        self.num_envs = num_envs
        self.device = torch.device("cuda") if device is None else torch.device(device)
        self.observation_space = spaces.Box(low=0, high=255, shape=(size, size, num_stacked_frames), dtype=np.uint8)
        self.action_space = spaces.Discrete(num_actions)
        g = torch.Generator(device="cpu").manual_seed(seed)
        # a pool of raw frames per environment, cycled through (synthetic emulator output)
        self.pool = torch.randint(0, 256, (pool_frames, num_envs, 210, 160, 3), dtype=torch.uint8, generator=g).to(self.device)
        self.rewards = torch.randint(-1, 2, (pool_frames, num_envs), generator=g).float().to(self.device)
        self.terminals = (torch.rand((pool_frames, num_envs), generator=g) < terminal_prob).to(torch.uint8).to(self.device)
        self.pre = BatchedAtariPreprocessor(num_envs, self.device, num_stacked_frames=num_stacked_frames, size=size)
        self.t = 0

    def rollout_repeats(self, num_steps):
        """True when every rollout of `num_steps` steps reads the same pool entries (frames are indexed by 2t + 1 .. 2t + 3,
        rewards / terminals by t, all modulo pool_frames): such a rollout can be replayed as one CUDA graph
        (agents.MultiEnvAgent) with exactly the results of stepping one by one."""
        return num_steps % self.pool.shape[0] == 0 and self.t % num_steps == 0

    envs = property(lambda self: [self] * self.num_envs)

    def reset(self):
        self.t = 0
        return self.pre.reset(self.pool[0]).clone()

    def step_device(self, actions):
        """actions: int32 [E] on the device (ignored by the synthetic dynamics).  Returns device tensors
        (observations uint8 [E,S,S,k], rewards f32 [E], terminals uint8 [E])."""
        n = self.pool.shape[0]
        i = (2 * self.t + 1) % n
        j = (2 * self.t + 2) % n
        k = (2 * self.t + 3) % n
        term = self.terminals[self.t % n]
        obs = self.pre.step(self.pool[i], self.pool[j], term, reset_raw=self.pool[k], keep_terminal_view=True)
        rew = self.rewards[self.t % n]
        self.t += 1
        return obs, rew, term

    def step(self, actions):
        obs, rew, term = self.step_device(None)
        return list(obs.cpu().numpy()), rew.cpu().tolist(), term.bool().cpu().tolist(), [{} for _ in range(self.num_envs)]

    def close(self):
        pass
