"""Oracle for Atari frame preprocessing and frame stacking at any square output size S and stack depth k (uint8,
bit-exact): AtariPreprocessFrameWrapper with another resolution and FrameStackWrapper(env, k), in MultiEnv's auto-reset
order.  It builds on oracle/preprocess.py (gray conversion, OpenCV's area tables), which stays the 84x84x4 restatement
K-PRE is pinned to.  tests/test_oracle_preprocess_sq.py pins it bit-for-bit against the real cv2 at every S in [4, 128].
"""
import numpy as np

from .preprocess import RAW_H, RAW_W, area_tab, rgb_to_gray


def area_tables(ssize, dsize):
    """`area_tab` packed CSR-style: (offsets int32 [dsize + 1], src int32 [taps], weights float32 [taps]); the taps of
    output d are src / weights[offsets[d]:offsets[d + 1]], in table order.  These are the arrays the S x S kernel reads."""
    tab = area_tab(ssize, dsize)
    counts = np.bincount([d for d, _, _ in tab], minlength=dsize)
    offsets = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    src = np.array([s for _, s, _ in tab], np.int32)
    w = np.array([a for _, _, a in tab], np.float32)
    return offsets, src, w


def area_fast_factors(size):
    """(x, y) integer scale factors when cv2.resize takes its integer-scale INTER_AREA path (resizeAreaFast_) for
    210x160 -> size x size, else None.  OpenCV takes it when |1 / (size / src) - round(...)| < DBL_EPSILON on both axes:
    sizes 5 (32 x 42 blocks) and 10 (16 x 21)."""
    fx, fy = 1.0 / (size / RAW_W), 1.0 / (size / RAW_H)
    ix, iy = round(fx), round(fy)
    eps = np.finfo(np.float64).eps
    return (ix, iy) if abs(fx - ix) < eps and abs(fy - iy) < eps else None


def resize_area(gray, size):
    """cv2.resize(gray, (size, size), interpolation=cv2.INTER_AREA) for 210x160 uint8 images [..., 210, 160]: the
    horizontal pass per source row (buf[dx] = buf[dx] + S[sx] * w from 0, table order), then the vertical pass (first
    term assigned, the rest added, table order); fp32 with separate roundings, round half to even, clamp.  At the sizes
    of `area_fast_factors` cv2 instead rounds float(integer block sum) * (1.f / block area)."""
    gray = np.asarray(gray)
    assert gray.dtype == np.uint8 and gray.shape[-2:] == (RAW_H, RAW_W)
    lead = gray.shape[:-2]
    fast = area_fast_factors(size)
    if fast is not None:
        ix, iy = fast
        sums = gray.reshape((-1, size, iy, size, ix)).astype(np.int64).sum(axis=(2, 4))
        out = sums.astype(np.float32) * np.float32(1.0 / (ix * iy))
        return np.clip(np.rint(out), 0, 255).astype(np.uint8).reshape(lead + (size, size))
    src = gray.reshape((-1, RAW_H, RAW_W)).astype(np.float32)
    xo, xs, xw = area_tables(RAW_W, size)
    yo, ys, yw = area_tables(RAW_H, size)
    buf = np.zeros((src.shape[0], RAW_H, size), np.float32)
    for d in range(size):
        for t in range(xo[d], xo[d + 1]):
            buf[:, :, d] = buf[:, :, d] + src[:, :, xs[t]] * xw[t]
    out = np.empty((src.shape[0], size, size), np.float32)
    for d in range(size):
        acc = buf[:, ys[yo[d]], :] * yw[yo[d]]
        for t in range(yo[d] + 1, yo[d + 1]):
            acc = acc + buf[:, ys[t], :] * yw[t]
        out[:, d, :] = acc
    return np.clip(np.rint(out), 0, 255).astype(np.uint8).reshape(lead + (size, size))


def preprocess_frame_sq(rgb, size):
    """AtariPreprocessFrameWrapper.observation at size x size: [..., 210, 160, 3] u8 -> [..., size, size, 1] u8."""
    return resize_area(rgb_to_gray(rgb), size)[..., None]


class FrameStackSq:
    """FrameStackWrapper (wrappers.py:201-235) for one environment whose frames have any shape [..., 1]."""

    def __init__(self, frame_shape, num_stacked_frames):
        self.k = num_stacked_frames
        self.stack = np.zeros(tuple(frame_shape[:-1]) + (num_stacked_frames,), np.uint8)

    def step(self, frame, terminal):
        self.stack = np.roll(self.stack, shift=-1, axis=-1)
        if terminal:
            self.stack.fill(0)
        self.stack[..., -1:] = frame
        return self.stack

    def reset(self, frame):
        self.stack = np.repeat(frame, self.k, axis=-1)
        return self.stack


def batched_stack_step_sq(stacks, raw_a, raw_b, terminal, reset_mask=None, reset_raw=None, size=84):
    """`batched_stack_step` for stacks uint8 [E, size, size, k] of any size and depth k."""
    stacks = np.array(stacks, copy=True)
    k = stacks.shape[-1]
    assert stacks.shape[1:3] == (size, size)
    if reset_mask is not None:
        for e in range(stacks.shape[0]):
            if reset_mask[e]:
                stacks[e] = np.repeat(preprocess_frame_sq(reset_raw[e], size), k, axis=-1)
    frames = resize_area(rgb_to_gray(np.maximum(raw_a, raw_b)), size)
    stacks = np.roll(stacks, -1, axis=-1)
    stacks[np.asarray(terminal, bool)] = 0
    stacks[..., -1] = frames
    return stacks
