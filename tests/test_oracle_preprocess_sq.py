"""The S x S, k-frame preprocessing oracle (oracle/preprocess_sq.py `resize_area`, `FrameStackSq`, `batched_stack_step_sq`)
against the real cv2 and against the reference's FrameStackWrapper lines, and the construction limits of the classes
that produce such frames (S in [4, 128], k in [1, 16])."""
import numpy as np
import pytest

import synth
from oracle import preprocess as P
from oracle import preprocess_sq as PS


def _gray_frames(seed):
    """8+ uint8 [210, 160] images: four random kinds, constant, vertical and horizontal ramps, a checkerboard."""
    rng = np.random.default_rng(seed)
    out = list(P.rgb_to_gray(synth.raw_frames(seed, 4, "mixed")))
    out.append(np.full((210, 160), rng.integers(0, 256), np.uint8))
    out.append(np.repeat((np.arange(210) * 255 // 209).astype(np.uint8)[:, None], 160, axis=1))
    out.append(np.repeat((np.arange(160) * 255 // 159).astype(np.uint8)[None, :], 210, axis=0))
    yy, xx = np.mgrid[:210, :160]
    out.append(np.where((yy // 3 + xx // 5) % 2 == 0, 255, 7).astype(np.uint8))
    out.append(rng.integers(250, 256, (210, 160), dtype=np.uint8))          # near saturation
    return np.stack(out)


@pytest.mark.parametrize("sizes", [range(4, 46), range(46, 88), range(88, 129)], ids=["4-45", "46-87", "88-128"])
def test_resize_area_bit_exact_against_cv2(sizes):
    cv2 = pytest.importorskip("cv2")
    frames = _gray_frames(3)
    assert len(frames) >= 8
    for s in sizes:
        got = PS.resize_area(frames, s)
        for i, g in enumerate(frames):
            want = cv2.resize(g, (s, s), interpolation=cv2.INTER_AREA)
            assert np.array_equal(got[i], want), "size %d frame %d" % (s, i)


def test_area_tables_pack_area_tab():
    for ssize, dsize in ((160, 84), (210, 84), (160, 11), (210, 11), (210, 128)):
        off, src, w = PS.area_tables(ssize, dsize)
        tab = P.area_tab(ssize, dsize)
        assert off[0] == 0 and off[-1] == len(tab) == len(src) == len(w)
        for d in range(dsize):
            row = [(s, a) for dd, s, a in tab if dd == d]
            assert list(src[off[d]:off[d + 1]]) == [s for s, _ in row]
            assert list(w[off[d]:off[d + 1]]) == [a for _, a in row]
    # the widest tables any size needs: 16 horizontal and 20 vertical taps at S = 11 (K-PRE's are 3 / 3)
    assert np.diff(PS.area_tables(160, 11)[0]).max() == 16 and np.diff(PS.area_tables(210, 11)[0]).max() == 20
    assert np.diff(PS.area_tables(160, 84)[0]).max() == 3 and np.diff(PS.area_tables(210, 84)[0]).max() == 3


def test_preprocess_frame_sq_at_84_is_preprocess_frame():
    raw = synth.raw_frames(4, 4, "mixed")
    assert np.array_equal(PS.preprocess_frame_sq(raw, 84), P.preprocess_frame(raw))


class RefFrameStack:
    """The array lines of the reference's FrameStackWrapper (wrappers.py:224-235), written out once more."""

    def __init__(self, k):
        self.k = k
        self.frames = None

    def reset(self, observation):
        self.frames = np.repeat(observation, self.k, axis=-1)
        return self.frames

    def step(self, observation, terminal):
        self.frames = np.roll(self.frames, shift=-1, axis=-1)
        if terminal:
            self.frames.fill(0)
        self.frames[..., -1:] = observation
        return self.frames


@pytest.mark.parametrize("k", [1, 2, 3, 4, 8, 16])
def test_frame_stack_sq_matches_the_reference_lines(k):
    rng = np.random.default_rng(k)
    ours, ref = PS.FrameStackSq((9, 9, 1), k), RefFrameStack(k)
    f = rng.integers(0, 256, (9, 9, 1), dtype=np.uint8)
    assert np.array_equal(ours.reset(f), ref.reset(f))
    for _ in range(50):
        f = rng.integers(0, 256, (9, 9, 1), dtype=np.uint8)
        if rng.random() < 0.1:
            assert np.array_equal(ours.reset(f), ref.reset(f))
        else:
            term = bool(rng.random() < 0.2)
            assert np.array_equal(ours.step(f, term), ref.step(f, term))


@pytest.mark.parametrize("k", [1, 2, 3, 4, 8, 16])
def test_batched_stack_step_sq_matches_per_environment_auto_reset(k):
    """MultiEnv's order per environment (multi_env.py:127-132): reset first when the previous step was terminal (the
    stack becomes k copies of that frame), then push max(a, b) with zero-on-terminal."""
    size, e_count, steps = 10, 3, 50
    rng = np.random.default_rng(100 + k)
    pre = lambda raw: PS.preprocess_frame_sq(raw, size)
    first = synth.raw_frames(k, e_count, "mixed")
    stacks = np.stack([np.repeat(pre(f), k, axis=-1) for f in first])
    refs = [RefFrameStack(k) for _ in range(e_count)]
    for e in range(e_count):
        refs[e].reset(pre(first[e]))
    prev_term = np.zeros(e_count, bool)
    for t in range(steps):
        raw = synth.raw_frames(1000 * k + t, 3 * e_count, "mixed")
        a, b, reset_raw = raw[:e_count], raw[e_count:2 * e_count], raw[2 * e_count:]
        term = rng.random(e_count) < 0.25
        stacks = PS.batched_stack_step_sq(stacks, a, b, term, prev_term, reset_raw, size)
        for e in range(e_count):
            if prev_term[e]:
                refs[e].reset(pre(reset_raw[e]))
            refs[e].step(pre(np.maximum(a[e], b[e])), term[e])
        assert np.array_equal(stacks, np.stack([r.frames for r in refs])), "step %d" % t
        prev_term = term


def test_batched_stack_step_sq_at_84_by_4_is_batched_stack_step():
    rng = np.random.default_rng(7)
    raw = synth.raw_frames(8, 12, "mixed")
    a, b, reset_raw = raw[:4], raw[4:8], raw[8:]
    stacks = rng.integers(0, 256, (4, 84, 84, 4), dtype=np.uint8)
    term = np.array([0, 1, 0, 1], bool)
    mask = np.array([1, 0, 0, 1], bool)
    assert np.array_equal(PS.batched_stack_step_sq(stacks, a, b, term, mask, reset_raw, 84),
                          P.batched_stack_step(stacks, a, b, term, mask, reset_raw))
    assert np.array_equal(PS.batched_stack_step_sq(stacks, a, b, term, size=84), P.batched_stack_step(stacks, a, b, term))


BAD_SHAPES = [(3, 4), (129, 4), (0, 1), (84.0, 4), (64, 0), (64, 17), (64, 2.0), (True, 4)]


@pytest.mark.parametrize("size, k", BAD_SHAPES)
def test_construction_rejects_sizes_and_depths_out_of_range(size, k):
    from actorcritic_b200.envs.atari import wrappers as W
    from actorcritic_b200.envs.atari.device_env import DeviceAtariMultiEnv
    from actorcritic_b200.envs.atari.raw_env import RawFrameMultiEnv
    with pytest.raises(ValueError):
        W.BatchedAtariPreprocessor(2, num_stacked_frames=k, size=size)
    with pytest.raises(ValueError):
        RawFrameMultiEnv([object()], size=size, num_stacked_frames=k)
    with pytest.raises(ValueError):
        DeviceAtariMultiEnv(2, size=size, num_stacked_frames=k)
    if not 4 <= size <= 128 or isinstance(size, (bool, float)):
        with pytest.raises(ValueError):
            W.AtariPreprocessFrameWrapper(object(), size=size)


@pytest.mark.parametrize("k", [0, 17, 2.0])
def test_frame_stack_wrapper_rejects_depths_out_of_range(k):
    from actorcritic_b200.envs.atari import wrappers as W
    with pytest.raises(ValueError):
        W.FrameStackWrapper(object(), k)


@pytest.mark.parametrize("shape", [(200, 200, 1), (3, 3, 1), (64, 32, 1), (64, 64, 3)])
def test_frame_stack_wrapper_rejects_frames_it_cannot_stack(shape):
    from actorcritic_b200 import spaces
    from actorcritic_b200.envs.atari import wrappers as W

    class Env:
        observation_space = spaces.Box(low=0, high=255, shape=shape, dtype=np.uint8)

    with pytest.raises(ValueError):
        W.FrameStackWrapper(Env(), 2)
