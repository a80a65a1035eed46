"""K-PRE at any square size S and stack depth k (csrc/preprocess.cu `preprocess_sq_kernel`, `framestack_sq_kernel`;
acx_preprocess_stack_sq_u8 / acx_preprocess_reset_sq_u8 / acx_framestack_push_sq_u8) byte for byte against the oracle
(oracle/preprocess_sq.py `batched_stack_step_sq`), and its resize against cv2."""
import numpy as np
import pytest
import torch

import synth
from oracle import preprocess_sq as PS

pytestmark = pytest.mark.gpu

SIZES = [4, 5, 10, 11, 16, 42, 64, 84, 96, 127, 128]      # 5 and 10 take cv2's integer-scale path
DEPTHS = [1, 2, 3, 4, 8, 16]
POOL = synth.raw_frames(11, 24, "mixed")


def _raw(rng, e_count):
    return POOL[rng.integers(0, len(POOL), e_count)]


def _run_sequence(size, k, e_count, seed, flags=True, stride_buffer=False):
    """3k + 5 steps of acx_preprocess_stack_sq_u8 from an acx_preprocess_reset_sq_u8 start, with random terminals and
    reset masks (or NULL flag pointers), single-frame windows (raw_a is raw_b) on every third step, in place or into the
    step slices of a [E, T, S, S, k] buffer; every step compared with the oracle."""
    from actorcritic_b200 import ops
    rng = np.random.default_rng(seed)
    steps = 3 * k + 5
    first = _raw(rng, e_count)
    stacks = ops.preprocess_reset_sq(torch.from_numpy(first).cuda(), size, k)
    want = np.repeat(PS.preprocess_frame_sq(first, size), k, axis=-1)
    assert tuple(stacks.shape) == (e_count, size, size, k)
    assert np.array_equal(stacks.cpu().numpy(), want), "reset"
    buf = torch.zeros((e_count, steps, size, size, k), dtype=torch.uint8, device="cuda") if stride_buffer else None
    for t in range(steps):
        a = _raw(rng, e_count)
        b = a if t % 3 == 2 else _raw(rng, e_count)
        reset_raw = _raw(rng, e_count)
        term = (rng.random(e_count) < 0.25) if flags else np.zeros(e_count, bool)
        mask = (rng.random(e_count) < 0.25) if flags else None
        da = torch.from_numpy(a).cuda()
        db = da if b is a else torch.from_numpy(b).cuda()
        kw = {}
        if flags:
            kw = dict(terminal=torch.from_numpy(term.astype(np.uint8)).cuda(),
                      reset_mask=torch.from_numpy(mask.astype(np.uint8)).cuda(), reset_raw=torch.from_numpy(reset_raw).cuda())
        want = PS.batched_stack_step_sq(want, a, b, term, mask, reset_raw if flags else None, size)
        if stride_buffer:
            ops.preprocess_stack_sq(da, db, stacks, out=buf[:, t], **kw)
            stacks = buf[:, t].contiguous()
        else:
            ops.preprocess_stack_sq(da, db, stacks, out=stacks, **kw)                  # in place
        assert np.array_equal(stacks.cpu().numpy(), want), "S=%d k=%d E=%d step %d" % (size, k, e_count, t)


@pytest.mark.parametrize("k", DEPTHS)
@pytest.mark.parametrize("size", SIZES)
def test_stack_step_matches_the_oracle(size, k):
    _run_sequence(size, k, 7, seed=size * 100 + k)


@pytest.mark.parametrize("size, k", [(4, 16), (11, 3), (64, 2), (84, 4), (128, 1), (127, 8)])
@pytest.mark.parametrize("e_count", [1, 300])
@pytest.mark.parametrize("flags", [True, False], ids=["flags", "null_flags"])
def test_batch_sizes_flag_pointers_and_strided_output(size, k, e_count, flags):
    _run_sequence(size, k, e_count, seed=size + k + e_count, flags=flags, stride_buffer=e_count == 300)


@pytest.mark.parametrize("size", SIZES)
def test_resize_matches_cv2(size):
    cv2 = pytest.importorskip("cv2")
    from actorcritic_b200 import ops
    raw = synth.raw_frames(size, 8, "mixed")
    raw[4] = 255                                                     # saturated frames: cv2's rounding at the top
    raw[5] = np.random.default_rng(size).integers(250, 256, raw[5].shape, dtype=np.uint8)
    got = ops.preprocess_reset_sq(torch.from_numpy(raw).cuda(), size, 1).cpu().numpy()[..., 0]
    for i, f in enumerate(raw):
        g = cv2.cvtColor(f, cv2.COLOR_RGB2GRAY)
        assert np.array_equal(got[i], cv2.resize(g, (size, size), interpolation=cv2.INTER_AREA)), "frame %d" % i


def test_the_new_kernel_at_84_by_4_produces_k_pre_bytes():
    from actorcritic_b200 import ops
    rng = np.random.default_rng(5)
    e_count = 300
    a, b, r = (torch.from_numpy(_raw(rng, e_count)).cuda() for _ in range(3))
    stacks = torch.from_numpy(rng.integers(0, 256, (e_count, 84, 84, 4), dtype=np.uint8)).cuda()
    term = torch.from_numpy((rng.random(e_count) < 0.3).astype(np.uint8)).cuda()
    mask = torch.from_numpy((rng.random(e_count) < 0.3).astype(np.uint8)).cuda()
    for kw in (dict(), dict(terminal=term, reset_mask=mask, reset_raw=r)):
        assert torch.equal(ops.preprocess_stack_sq(a, b, stacks, **kw), ops.preprocess_stack(a, b, stacks, **kw))
    assert torch.equal(ops.preprocess_reset_sq(a, 84, 4), ops.preprocess_reset(a))


@pytest.mark.parametrize("size, k", [(84, 4), (84, 2), (64, 1), (13, 16), (128, 3)])
def test_framestack_push_in_all_three_modes(size, k):
    from actorcritic_b200 import ops
    rng = np.random.default_rng(size * k)
    e_count = 6
    stacks = rng.integers(0, 256, (e_count, size, size, k), dtype=np.uint8)
    frames = rng.integers(0, 256, (e_count, size, size), dtype=np.uint8)
    mode = np.array([0, 1, 2, 0, 2, 1], np.uint8)
    want = np.roll(stacks, -1, axis=-1)
    want[mode == 1] = 0
    want[..., -1] = frames
    want[mode == 2] = np.repeat(frames[mode == 2][..., None], k, axis=-1)
    d_stacks = torch.from_numpy(stacks).cuda()
    got = ops.framestack_push_sq(torch.from_numpy(frames).cuda(), d_stacks, mode=torch.from_numpy(mode).cuda())
    assert np.array_equal(got.cpu().numpy(), want)
    # NULL mode = push everywhere; in place
    want0 = np.roll(stacks, -1, axis=-1)
    want0[..., -1] = frames
    ops.framestack_push_sq(torch.from_numpy(frames).cuda(), d_stacks, out=d_stacks)
    assert np.array_equal(d_stacks.cpu().numpy(), want0)


class _Scripted:
    def __init__(self, frames, terminals, observation_space=None):
        self.frames, self.terminals, self.i = frames, terminals, 0
        self.action_space = None
        if observation_space is not None:
            self.observation_space = observation_space

    def reset(self):
        self.i += 1
        return self.frames[self.i - 1]

    def step(self, action):
        self.i += 1
        return self.frames[self.i - 1], 1.0, self.terminals[self.i - 1], {}


@pytest.mark.parametrize("size, k", [(64, 2), (36, 1), (84, 8), (84, 4), (96, 16)])
def test_preprocess_and_frame_stack_wrappers(size, k):
    """AtariPreprocessFrameWrapper(size) -> FrameStackWrapper(k) for one environment against the oracle's FrameStackSq."""
    from actorcritic_b200.envs.atari import wrappers as W
    rng = np.random.default_rng(size + k)
    n = 3 * k + 6
    raw = [POOL[i] for i in rng.integers(0, len(POOL), n)]
    term = [bool(x) for x in rng.random(n) < 0.2]
    pre = W.AtariPreprocessFrameWrapper(_Scripted(raw, term), size=size)
    assert pre.observation_space.shape == (size, size, 1)
    fs = W.FrameStackWrapper(pre, k)
    assert fs.observation_space.shape == (size, size, k)
    ref = PS.FrameStackSq((size, size, 1), k)
    assert np.array_equal(fs.reset(), ref.reset(PS.preprocess_frame_sq(raw[0], size)))
    for i in range(1, n):
        obs, _, terminal, _ = fs.step(0)
        assert terminal == term[i]
        assert np.array_equal(obs, ref.step(PS.preprocess_frame_sq(raw[i], size), term[i])), "step %d" % i


@pytest.mark.parametrize("size, k", [(3, 4), (129, 4), (64, 0), (64, 17)])
def test_the_c_entry_points_reject_shapes_out_of_range(size, k):
    from actorcritic_b200 import _lib
    lib = _lib.load()
    raw = torch.zeros((1, 210, 160, 3), dtype=torch.uint8, device="cuda")
    out = torch.zeros(1 << 20, dtype=torch.uint8, device="cuda")
    p = lambda t: t.data_ptr()
    assert lib.acx_preprocess_stack_sq_u8(p(raw), p(raw), None, None, None, p(out), p(out), 1 << 20, 1, size, k, None) != 0
    assert b"size" in lib.acx_last_error() or b"num_frames" in lib.acx_last_error()
    assert lib.acx_preprocess_reset_sq_u8(p(raw), p(out), 1 << 20, 1, size, k, None) != 0
    assert lib.acx_framestack_push_sq_u8(p(out), None, p(out), p(out), 1, size, k, None) != 0
