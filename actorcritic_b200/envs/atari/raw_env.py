"""RawFrameMultiEnv - the step BEFORE the accelerated path (SURVEY 8(f) f2): hosts emulator-like environments that
yield RAW 210x160x3 RGB frames and hands the frame work to the K-PRE kernel.

In the reference every environment runs the whole wrapper chain on the CPU - `AtariFrameskipWrapper` (repeat the action,
max of the last two frames, wrappers.py:52-67), `AtariPreprocessFrameWrapper` (cv2 gray + resize, :30-33),
`FrameStackWrapper` (:224-235) under `MultiEnv`'s auto-reset (multi_env.py:127-132) - and ships the processed stack to
the learner process.  Here the environments only run the emulator part of that chain (action repeat, reward sum, early
exit on terminal, auto-reset): each step leaves the last two raw frames of every environment in PINNED host buffers, one
asynchronous copy moves them to the GPU, and one K-PRE launch does max + gray + resize + stack push for all of them.
Observations are uint8 [E, S, S, k]: `size` S in [4, 128] (84 by default) and `num_stacked_frames` k in [1, 16] (4 by
default); 84 x 84 x 4 runs K-PRE, any other pair its S x S form.
Observations stay on the device (`device_resident`), so `MultiEnvAgent.interact` feeds them to acting and to the train
step without another copy.

The environments need the gym surface the reference uses: `reset() -> frame`, `step(action) -> (frame, reward, terminal,
info)`, `action_space`, optionally `close()`.

Wrapper order.  In the reference the frameskip sits BELOW the game-logic wrappers (a2c_acktr.py:190-208: NoopReset ->
Frameskip -> Preprocess -> EpisodeInfo -> EpisodicLife -> FireReset -> ClipReward): rewards are clipped AFTER the 4-frame
sum, and the FIRE / life logic sees agent steps, not emulator frames.  Here the frameskip is applied by this class, so
wrappers stacked on the hosted environments sit below it and see single emulator frames: only wrappers that are indifferent
to that may go there (AtariNoopResetWrapper, a2c_acktr.py:190).  What must act on agent steps is given to this class
instead: `clip_rewards=True` clips the summed reward to [-1, 1] (AtariClipRewardWrapper, wrappers.py:73-86), and
`step_hook(env_index, reward, terminal, info) -> (reward, terminal, info)` runs after every agent step (the place for
episodic-life / episode-info logic).  The game-logic wrappers themselves are Python and out of scope (SURVEY 8(f) f2).
"""
import concurrent.futures

import numpy as np
import torch

from ... import spaces
from .wrappers import BatchedAtariPreprocessor, check_frame_shape

RAW_SHAPE = (210, 160, 3)


class RawFrameMultiEnv:
    device_resident = True

    def __init__(self, envs, frameskip=4, device=None, num_threads=None, clip_rewards=False, step_hook=None, size=84,
                 num_stacked_frames=4):
        size, num_stacked_frames = check_frame_shape(size, num_stacked_frames)
        if len(envs) == 0:
            raise ValueError("at least one environment is required")
        if not torch.cuda.is_available():
            from ... import _lib
            raise _lib.AcxError("RawFrameMultiEnv needs a CUDA device (the frame work runs in libacx's K-PRE kernel); there is "
                                "no CPU fallback")
        if frameskip < 1:
            raise ValueError("frameskip must be >= 1")
        self._envs = list(envs)
        self.num_envs = len(self._envs)
        self.frameskip = int(frameskip)
        self.clip_rewards = bool(clip_rewards)
        self.step_hook = step_hook
        self.device = torch.device("cuda") if device is None else torch.device(device)
        self.observation_space = spaces.Box(low=0, high=255, shape=(size, size, num_stacked_frames), dtype=np.uint8)
        self.action_space = self._envs[0].action_space
        self._executor = concurrent.futures.ThreadPoolExecutor(num_threads or min(32, self.num_envs))
        e = self.num_envs
        pin = lambda *shape, dtype=torch.uint8: torch.empty(shape, dtype=dtype).pin_memory()
        # host staging (pinned): frames [3] = (second-to-last, last, reset frame) of the current step
        self._h_frames = pin(3, e, *RAW_SHAPE)
        self._h_flags = pin(2, e)                       # [0] terminal of this step, [1] reset-before-this-step mask
        self._h_rewards = pin(e, dtype=torch.float32)
        self._np_frames = self._h_frames.numpy()
        self._np_flags = self._h_flags.numpy()
        self._np_rewards = self._h_rewards.numpy()
        self._d_frames = torch.empty((3, e) + RAW_SHAPE, dtype=torch.uint8, device=self.device)
        self._d_flags = torch.empty((2, e), dtype=torch.uint8, device=self.device)
        self._d_rewards = torch.empty(e, dtype=torch.float32, device=self.device)
        self._terminated = [False] * e                  # _AutoResetWrapper._terminated (multi_env.py:124,131)
        self._staged = torch.cuda.Event()
        self.pre = BatchedAtariPreprocessor(e, self.device, num_stacked_frames=num_stacked_frames, size=size)
        self.last_infos = [{} for _ in range(e)]
        self._closed = False

    envs = property(lambda self: self._envs)

    # ------------------------------------------------------------------ host side (one thread per environment)
    def _reset_one(self, i):
        frame = self._envs[i].reset()
        self._np_frames[0, i] = frame
        self._terminated[i] = False

    def _step_one(self, i, action):
        env = self._envs[i]
        did_reset = self._terminated[i]
        if did_reset:                                   # multi_env.py:128-129: reset first, its observation is discarded
            self._np_frames[2, i] = env.reset()         # ... but it seeds the frame stack (wrappers.py:232-235)
        self._np_flags[1, i] = 1 if did_reset else 0
        total_reward, terminal, info = 0.0, False, None
        prev = last = None
        for _ in range(self.frameskip):                 # wrappers.py:52-62
            frame, reward, terminal, info = env.step(action)
            prev, last = last, frame
            total_reward += reward
            if terminal:
                break
        # wrappers.py:64-67: max of the last two frames, or the only frame when the first sub-step was terminal
        self._np_frames[0, i] = last if prev is None else prev
        self._np_frames[1, i] = last
        if self.clip_rewards:                           # wrappers.py:85-86, applied to the agent step's reward like the reference
            total_reward = float(np.clip(total_reward, -1.0, 1.0))
        if self.step_hook is not None:
            total_reward, terminal, info = self.step_hook(i, total_reward, terminal, info)
        self._np_rewards[i] = total_reward
        self._np_flags[0, i] = 1 if terminal else 0
        self._terminated[i] = bool(terminal)
        self.last_infos[i] = info if info is not None else {}

    def _wait_staging_free(self):
        # the previous step's asynchronous host-to-device copies must have read the pinned buffers
        self._staged.synchronize()

    # ------------------------------------------------------------------ MultiEnv surface
    def reset(self):
        """MultiEnv.reset (multi_env.py:49-57): uint8 [E,S,S,k] on the device, k copies of the first frame."""
        self._wait_staging_free()
        list(self._executor.map(self._reset_one, range(self.num_envs)))
        self._d_frames[0].copy_(self._h_frames[0], non_blocking=True)
        self._staged.record()
        return self.pre.reset(self._d_frames[0])

    def step_device(self, actions):
        """actions: int tensor [E] (device or host) or a list.  Returns device tensors (observations uint8 [E,S,S,k],
        rewards float32 [E], terminals uint8 [E]); `last_infos` holds the environments' info dicts."""
        if isinstance(actions, torch.Tensor):
            actions = actions.cpu().tolist()            # the emulators need the actions on the host: one small sync
        if len(actions) != self.num_envs:
            raise ValueError("expected %d actions, got %d" % (self.num_envs, len(actions)))
        self._wait_staging_free()
        list(self._executor.map(self._step_one, range(self.num_envs), actions))
        # the reset frames (slot 2) only travel when some environment was reset before this step
        slots = 3 if self._np_flags[1].any() else 2
        self._d_frames[:slots].copy_(self._h_frames[:slots], non_blocking=True)
        self._d_flags.copy_(self._h_flags, non_blocking=True)
        self._d_rewards.copy_(self._h_rewards, non_blocking=True)
        self._staged.record()
        self.pre.prev_terminal = self._d_flags[1]       # environments that were reset before this step
        obs = self.pre.step(self._d_frames[0], self._d_frames[1], self._d_flags[0], reset_raw=self._d_frames[2])
        return obs, self._d_rewards.clone(), self._d_flags[0].clone()

    def step(self, actions):
        """MultiEnv.step (multi_env.py:59-81) with host lists, for callers that are not device aware."""
        obs, rew, term = self.step_device(actions)
        return list(obs.cpu().numpy()), rew.cpu().tolist(), term.bool().cpu().tolist(), list(self.last_infos)

    def close(self):
        if self._closed:
            return
        self._closed = True
        for env in self._envs:
            if hasattr(env, "close"):
                env.close()
        self._executor.shutdown()
