"""The array-processing subset of actorcritic/envs/atari/wrappers.py, batched over environments and run by the
K-PRE kernel (preprocess.cu): 2-frame max (wrappers.py:64-65), RGB->gray + 84x84 INTER_AREA resize (:30-33), frame
stack push / zero-on-terminal / reset-to-4-copies (:224-235) in the order MultiEnv's auto-reset imposes
(multi_env.py:127-132).  Bit-exact with the reference's cv2 + NumPy path (tests/test_gpu_preprocess.py).

`BatchedAtariPreprocessor` is the batched form; the per-environment classes keep the reference's names and call
the same kernel with one environment.

Every class takes an output size S in [4, 128] (square frames, `size=84` by default) and, where it stacks, a depth k in
[1, 16] (4 by default): 84 x 84 x 4 runs K-PRE, every other pair the S x S kernel (acx_preprocess_stack_sq_u8), with the
same semantics and the same bit-exactness against cv2 at that size."""
import numpy as np
import torch

from ... import ops
from ... import spaces


MIN_SIZE, MAX_SIZE = 4, 128           # CNNModel's image sizes
MIN_FRAMES, MAX_FRAMES = 1, 16        # CNNModel's channel counts


def check_frame_shape(size=84, num_stacked_frames=4):
    """Validate an output size S and a stack depth k; returns them as ints."""
    if isinstance(size, bool) or not isinstance(size, (int, np.integer)) or not MIN_SIZE <= size <= MAX_SIZE:
        raise ValueError("size must be an integer in [%d, %d], got %r" % (MIN_SIZE, MAX_SIZE, size))
    if (isinstance(num_stacked_frames, bool) or not isinstance(num_stacked_frames, (int, np.integer))
            or not MIN_FRAMES <= num_stacked_frames <= MAX_FRAMES):
        raise ValueError("num_stacked_frames must be an integer in [%d, %d], got %r"
                         % (MIN_FRAMES, MAX_FRAMES, num_stacked_frames))
    return int(size), int(num_stacked_frames)


class BatchedAtariPreprocessor:
    """Frame stacks uint8 [E, S, S, k] of E environments on the device."""

    def __init__(self, num_envs, device=None, num_stacked_frames=4, size=84):
        self.size, self.num_stacked_frames = check_frame_shape(size, num_stacked_frames)
        self.kpre = (self.size, self.num_stacked_frames) == (84, 4)      # the specialised kernel
        self.num_envs = num_envs
        self.device = torch.device("cuda") if device is None else torch.device(device)
        self.stacks = torch.zeros((num_envs, self.size, self.size, self.num_stacked_frames), dtype=torch.uint8,
                                  device=self.device)
        self.stack_bytes = self.size * self.size * self.num_stacked_frames
        self.prev_terminal = torch.zeros(num_envs, dtype=torch.uint8, device=self.device)

    def reset(self, raw_frames):
        """MultiEnv.reset: stack = k copies of preprocess(frame) (wrappers.py:232-235)."""
        if self.kpre:
            ops.preprocess_reset(raw_frames, out=self.stacks, out_env_stride=28224)
        else:
            ops.preprocess_reset_sq(raw_frames, self.size, self.num_stacked_frames, out=self.stacks,
                                    out_env_stride=self.stack_bytes)
        self.prev_terminal.zero_()
        return self.stacks

    def step(self, raw_a, raw_b, terminal, reset_raw=None, out=None, out_env_stride=None, keep_terminal_view=False):
        """One MultiEnv.step: raw_a/raw_b = the last two emulator frames of each frameskip window, `terminal` = this
        step's terminal flags; environments whose PREVIOUS step was terminal are first reset from reset_raw.
        `out` may be a slice [:, t] of a batch-major rollout buffer."""
        reset_mask = self.prev_terminal if reset_raw is not None else None
        step = ops.preprocess_stack if self.kpre else ops.preprocess_stack_sq
        step(raw_a, raw_b, self.stacks, terminal=terminal, reset_mask=reset_mask, reset_raw=reset_raw, out=self.stacks,
             out_env_stride=self.stack_bytes)
        if out is not None:
            out.copy_(self.stacks)
        if terminal is None:
            self.prev_terminal = torch.zeros_like(self.prev_terminal)
        else:       # keep_terminal_view: the caller guarantees that `terminal` is not overwritten before the next step
            self.prev_terminal = terminal if keep_terminal_view else terminal.clone()
        return self.stacks


class AtariPreprocessFrameWrapper:
    """wrappers.py:16-33 for one environment: observation(frame) -> uint8 [S,S,1] (S = `size`, 84 by default)."""

    def __init__(self, env, size=84):
        self.size, _ = check_frame_shape(size)
        self.env = env
        self.observation_space = spaces.Box(low=0, high=255, shape=(self.size, self.size, 1), dtype=np.uint8)
        self.action_space = getattr(env, "action_space", None)

    def observation(self, frame):
        raw = torch.from_numpy(np.ascontiguousarray(frame, dtype=np.uint8)[None]).cuda()
        if self.size == 84:
            return ops.preprocess_reset(raw)[0, :, :, 3:4].cpu().numpy()
        return ops.preprocess_reset_sq(raw, self.size, 1)[0].cpu().numpy()

    def reset(self, **kwargs):
        return self.observation(self.env.reset(**kwargs))

    def step(self, action):
        observation, reward, terminal, info = self.env.step(action)
        return self.observation(observation), reward, terminal, info


class AtariFrameskipWrapper:
    """wrappers.py:36-70 for one environment: repeats the action `frameskip` times, sums the rewards, stops at a terminal
    step, and returns the byte-wise max of the last two frames (acx_frame_max_u8) - or the only frame when the first
    sub-step was terminal."""

    def __init__(self, env, frameskip):
        self.env = env
        self._frameskip = frameskip
        self.action_space = getattr(env, "action_space", None)
        self.observation_space = getattr(env, "observation_space", None)

    def step(self, action):
        older = newest = None            # only the last two frames of the window matter
        reward_sum, done, info = 0.0, False, None
        for _ in range(self._frameskip):
            frame, reward, done, info = self.env.step(action)
            older, newest = newest, frame
            reward_sum += reward
            if done:
                break
        if older is None:                # the first sub-step ended the episode: a one-frame window (wrappers.py:66-67)
            return newest, reward_sum, done, info
        pair = torch.from_numpy(np.ascontiguousarray(np.stack([older, newest]), dtype=np.uint8)).cuda()
        return ops.frame_max(pair[0], pair[1]).cpu().numpy(), reward_sum, done, info

    def reset(self, **kwargs):
        return self.env.reset(**kwargs)


class FrameStackWrapper:
    """wrappers.py:201-235 for one environment that already yields [S,S,1] frames (host arrays, S in [4, 128], read from
    the environment's observation space, 84 without one); the stack of k = num_stacked_frames in [1, 16] lives on the
    device and is pushed by acx_framestack_push_u8 (84 x 84 x 4) or acx_framestack_push_sq_u8."""

    def __init__(self, env, num_stacked_frames):
        shape = getattr(getattr(env, "observation_space", None), "shape", None)
        size = int(shape[0]) if shape is not None and len(shape) == 3 else 84
        if shape is not None and len(shape) == 3 and (shape[0] != shape[1] or shape[2] != 1):
            raise ValueError("FrameStackWrapper stacks square one-channel frames [S, S, 1], got %s" % (tuple(shape),))
        self.size, self.num_stacked_frames = check_frame_shape(size, num_stacked_frames)
        self.env = env
        self.action_space = getattr(env, "action_space", None)
        self.observation_space = spaces.Box(low=0, high=255, shape=(self.size, self.size, self.num_stacked_frames),
                                            dtype=np.uint8)
        self._stack = torch.zeros((1, self.size, self.size, self.num_stacked_frames), dtype=torch.uint8, device="cuda")

    def _push(self, frame, mode):
        f = torch.from_numpy(np.ascontiguousarray(frame, np.uint8).reshape(1, self.size, self.size)).cuda()
        m = torch.tensor([mode], dtype=torch.uint8, device="cuda")
        push = ops.framestack_push if (self.size, self.num_stacked_frames) == (84, 4) else ops.framestack_push_sq
        push(f, self._stack, mode=m, out=self._stack)
        return self._stack[0].cpu().numpy()

    def step(self, action):
        frame, reward, terminal, info = self.env.step(action)
        return self._push(frame, 1 if terminal else 0), reward, terminal, info       # wrappers.py:226-229

    def reset(self, **kwargs):
        return self._push(self.env.reset(**kwargs), 2)                                 # wrappers.py:234


class EpisodeInfoWrapper:
    """wrappers.py:263-323: accumulates the rewards of an episode and, on its terminal step, reports them as
    info['episode']['total_reward'] (host-side bookkeeping; stacks on any environment, also on those a RawFrameMultiEnv
    hosts)."""

    def __init__(self, env):
        self.env = env
        self.action_space = getattr(env, "action_space", None)
        self.observation_space = getattr(env, "observation_space", None)
        self.total_reward = 0.0

    def step(self, action):
        observation, reward, terminal, info = self.env.step(action)
        self.total_reward += reward
        if terminal:
            info = dict(info) if info is not None else {}
            info["episode"] = {"total_reward": self.total_reward}
            self.total_reward = 0.0
        return observation, reward, terminal, info

    def reset(self, **kwargs):
        self.total_reward = 0.0
        return self.env.reset(**kwargs)

    @staticmethod
    def get_episode_rewards_from_info_batch(infos):
        """Batch-major [environment][step] infos (as `Agent.interact` returns them) -> float32 array of the same shape
        with the episode reward where an episode ended and NaN elsewhere (wrappers.py:296-323); the caller takes
        `np.nanmean` of it for the 'episode_reward' summary (a2c_acktr.py:112-114)."""
        environments = len(infos)
        steps = len(infos[0]) if environments else 0
        rewards = np.full((environments, steps), np.nan, np.float32)
        for e, row in enumerate(infos):
            for t, info in enumerate(row):
                episode = info.get("episode") if info else None
                if episode is not None:
                    rewards[e, t] = episode["total_reward"]
        return rewards
