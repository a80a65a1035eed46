"""Thin torch-tensor wrappers over the C ABI (device memory and streams come from torch; every
computation is a libacx kernel).  Used by the API layer and by the parity tests."""
import ctypes

import torch

from . import _lib


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


def _need_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise _lib.AcxError("libacx operates on CUDA tensors only (no CPU fallback)")


def preprocess_stack(raw_a, raw_b, stack_in, terminal=None, reset_mask=None, reset_raw=None, out=None,
                     out_env_stride=None):
    """K-PRE (include/acx.h acx_preprocess_stack_u8).  raw_*: uint8 [E,210,160,3]; stack_in uint8 [E,84,84,4].
    `out` may be a slice of a batch-major rollout buffer; out_env_stride is then its env stride in bytes."""
    _need_cuda(raw_a, raw_b, stack_in)
    e = raw_a.shape[0]
    assert raw_a.dtype == torch.uint8 and tuple(raw_a.shape[1:]) == (210, 160, 3) and raw_a.is_contiguous()
    assert raw_b.shape == raw_a.shape and raw_b.is_contiguous() and stack_in.is_contiguous()
    if out is None:
        out = torch.empty((e, 84, 84, 4), dtype=torch.uint8, device=raw_a.device)
        out_env_stride = 28224
    elif out_env_stride is None:
        out_env_stride = out.stride(0)
    for t in (terminal, reset_mask):
        assert t is None or (t.dtype == torch.uint8 and t.is_contiguous())
    _lib.check(_lib.load().acx_preprocess_stack_u8(_ptr(raw_a), _ptr(raw_b), _ptr(terminal), _ptr(reset_mask),
                                                   _ptr(reset_raw), _ptr(stack_in), _ptr(out),
                                                   ctypes.c_size_t(out_env_stride), e, _stream()))
    return out


def preprocess_reset(raw, out=None, out_env_stride=None):
    _need_cuda(raw)
    e = raw.shape[0]
    if out is None:
        out = torch.empty((e, 84, 84, 4), dtype=torch.uint8, device=raw.device)
        out_env_stride = 28224
    elif out_env_stride is None:
        out_env_stride = out.stride(0)
    _lib.check(_lib.load().acx_preprocess_reset_u8(_ptr(raw), _ptr(out), ctypes.c_size_t(out_env_stride), e, _stream()))
    return out


def frame_max(a, b):
    """acx_frame_max_u8: byte-wise max of two uint8 CUDA tensors of the same shape (wrappers.py:64-65)."""
    _need_cuda(a, b)
    assert a.dtype == torch.uint8 and b.dtype == torch.uint8 and a.shape == b.shape and a.is_contiguous() and b.is_contiguous()
    out = torch.empty_like(a)
    _lib.check(_lib.load().acx_frame_max_u8(_ptr(a), _ptr(b), _ptr(out), ctypes.c_size_t(a.numel()), _stream()))
    return out


def framestack_push(frames, stack_in, mode=None, out=None):
    """acx_framestack_push_u8: frames uint8 [E,84,84(,1)], stacks uint8 [E,84,84,4]; mode uint8 [E]: 0 push, 1 push after
    a terminal step, 2 reset (wrappers.py:224-235)."""
    _need_cuda(frames, stack_in)
    e = stack_in.shape[0]
    assert frames.dtype == torch.uint8 and frames.is_contiguous() and frames.numel() == e * 84 * 84
    assert stack_in.dtype == torch.uint8 and stack_in.is_contiguous() and tuple(stack_in.shape[1:]) == (84, 84, 4)
    assert mode is None or (mode.dtype == torch.uint8 and mode.is_contiguous() and mode.numel() == e)
    if out is None:
        out = torch.empty_like(stack_in)
    _lib.check(_lib.load().acx_framestack_push_u8(_ptr(frames), _ptr(mode), _ptr(stack_in), _ptr(out), e, _stream()))
    return out


def preprocess_stack_sq(raw_a, raw_b, stack_in, terminal=None, reset_mask=None, reset_raw=None, out=None,
                        out_env_stride=None):
    """K-PRE at any square size and stack depth (acx_preprocess_stack_sq_u8): the size S and depth k are read from
    stack_in uint8 [E,S,S,k]; raw_*: uint8 [E,210,160,3].  `out` may be a slice of a batch-major rollout buffer
    [E,T,S,S,k]; out_env_stride is then its env stride in bytes."""
    _need_cuda(raw_a, raw_b, stack_in)
    e = raw_a.shape[0]
    assert raw_a.dtype == torch.uint8 and tuple(raw_a.shape[1:]) == (210, 160, 3) and raw_a.is_contiguous()
    assert raw_b.shape == raw_a.shape and raw_b.is_contiguous()
    assert stack_in.dtype == torch.uint8 and stack_in.dim() == 4 and stack_in.shape[0] == e and stack_in.is_contiguous()
    size, k = stack_in.shape[1], stack_in.shape[3]
    assert stack_in.shape[2] == size
    if out is None:
        out = torch.empty_like(stack_in)
        out_env_stride = size * size * k
    elif out_env_stride is None:
        out_env_stride = out.stride(0)
    for t in (terminal, reset_mask):
        assert t is None or (t.dtype == torch.uint8 and t.is_contiguous())
    assert reset_raw is None or (reset_raw.shape == raw_a.shape and reset_raw.is_contiguous())
    _lib.check(_lib.load().acx_preprocess_stack_sq_u8(_ptr(raw_a), _ptr(raw_b), _ptr(terminal), _ptr(reset_mask),
                                                      _ptr(reset_raw), _ptr(stack_in), _ptr(out),
                                                      ctypes.c_size_t(out_env_stride), e, size, k, _stream()))
    return out


def preprocess_reset_sq(raw, size, num_frames, out=None, out_env_stride=None):
    """acx_preprocess_reset_sq_u8: stacks uint8 [E,size,size,num_frames] = num_frames copies of preprocess(raw)."""
    _need_cuda(raw)
    e = raw.shape[0]
    assert raw.dtype == torch.uint8 and tuple(raw.shape[1:]) == (210, 160, 3) and raw.is_contiguous()
    if out is None:
        out = torch.empty((e, size, size, num_frames), dtype=torch.uint8, device=raw.device)
        out_env_stride = size * size * num_frames
    elif out_env_stride is None:
        out_env_stride = out.stride(0)
    _lib.check(_lib.load().acx_preprocess_reset_sq_u8(_ptr(raw), _ptr(out), ctypes.c_size_t(out_env_stride), e, size,
                                                      num_frames, _stream()))
    return out


def framestack_push_sq(frames, stack_in, mode=None, out=None):
    """acx_framestack_push_sq_u8: frames uint8 [E,S,S(,1)], stacks uint8 [E,S,S,k]; mode uint8 [E]: 0 push, 1 push after a
    terminal step, 2 reset (k copies)."""
    _need_cuda(frames, stack_in)
    assert stack_in.dtype == torch.uint8 and stack_in.dim() == 4 and stack_in.is_contiguous()
    e, size, k = stack_in.shape[0], stack_in.shape[1], stack_in.shape[3]
    assert stack_in.shape[2] == size
    assert frames.dtype == torch.uint8 and frames.is_contiguous() and frames.numel() == e * size * size
    assert mode is None or (mode.dtype == torch.uint8 and mode.is_contiguous() and mode.numel() == e)
    if out is None:
        out = torch.empty_like(stack_in)
    assert out.shape == stack_in.shape and out.is_contiguous()
    _lib.check(_lib.load().acx_framestack_push_sq_u8(_ptr(frames), _ptr(mode), _ptr(stack_in), _ptr(out), e, size, k,
                                                     _stream()))
    return out


def returns_adv(rewards, terminals, values, bootstrap_values, gamma):
    """K-RET.  rewards f32 [E,T], terminals uint8/bool [E,T], values f32 [E,T], bootstrap f32 [E]."""
    _need_cuda(rewards, terminals, values, bootstrap_values)
    e, t = rewards.shape
    term = terminals.to(torch.uint8).contiguous()
    targets = torch.empty((e, t), dtype=torch.float32, device=rewards.device)
    adv = torch.empty_like(targets)
    _lib.check(_lib.load().acx_returns_adv(_ptr(rewards.contiguous()), _ptr(term), _ptr(values.contiguous()),
                                           _ptr(bootstrap_values.contiguous()), float(gamma), e, t,
                                           _ptr(targets), _ptr(adv), _stream()))
    return targets, adv


def pad8(n):
    return (n + 7) // 8 * 8


def split_planes(x, num_planes, scale=1.0):
    """fp32 [rows, cols] -> list of bf16 planes [rows, pad8(cols)] with x*scale ~= sum(planes)."""
    _need_cuda(x)
    x = x.contiguous().float()
    rows, cols = x.shape
    ld = pad8(cols)
    planes = [torch.empty((rows, ld), dtype=torch.bfloat16, device=x.device) for _ in range(num_planes)]
    arr = (ctypes.c_void_p * num_planes)(*[p.data_ptr() for p in planes])
    _lib.check(_lib.load().acx_split_planes(_ptr(x), x.stride(0), rows, cols, float(scale), arr, num_planes, ld, _stream()))
    return planes


def gather_view(planes, dim, stride_bytes, gx, gy, samples, chunks):
    """acx_gather_t (include/acx.h): a patch operand read in place.  `chunks` = per 64-column chunk the coordinates
    (c0, c1, c2, c3) added to (0, x, 0, y, sample) of the 5-D view `dim` / `stride_bytes` (innermost first)."""
    g = _lib.Gather()
    for i, p in enumerate(planes):
        g.planes[i] = p.data_ptr()
    g.num_planes = len(planes)
    for i in range(5):
        g.dim[i] = dim[i]
    for i in range(4):
        g.stride_bytes[i] = stride_bytes[i]
    g.gx, g.gy, g.samples, g.num_chunks = gx, gy, samples, len(chunks)
    for q, (c0, c1, c2, c3) in enumerate(chunks):
        g.c0[q], g.c1[q], g.c2[q], g.c3[q] = c0, c1, c2, c3
    return g


def nature_cnn_gather(planes, layer, samples):
    """The in-place patch operand of a Nature-CNN conv layer (csrc/learner.cu:setup_gather): layer "conv1" on the row-pair
    observation copy [S,42,84,2,4], "conv2" on act1 planes [S,20,20,32], "conv3" on act2 planes [S,9,9,64]."""
    if layer == "conv2":
        px = 32 * 2
        return gather_view(planes, (64, 10, 4, 9, samples), (2 * px, 20 * px, 40 * px, 400 * px), 9, 9, samples,
                           [(0, h, kh, 0) for kh in range(4) for h in range(2)])
    if layer == "conv3":
        px = 64 * 2
        return gather_view(planes, (64, 9, 1, 9, samples), (px, px, 9 * px, 81 * px), 7, 7, samples,
                           [(0, kw, 0, kh) for kh in range(3) for kw in range(3)])
    prow = 84 * 8 * 2
    return gather_view(planes, (64, 20, 4, 20, samples), (64, prow, 2 * prow, 42 * prow), 20, 20, samples,
                       [(0, 0, j, 0) for j in range(4)])


def obs_pairs(obs):
    """uint8 [S, 84, 84, 4] -> the row-pair interleaved bf16 copy [S, 42, 84, 2, 4] (acx_obs_pairs_bf16)."""
    assert obs.dtype == torch.uint8 and obs.is_contiguous() and tuple(obs.shape[1:]) == (84, 84, 4)
    out = torch.empty((obs.shape[0], 42, 84, 2, 4), dtype=torch.bfloat16, device=obs.device)
    _lib.check(_lib.load().acx_obs_pairs_bf16(obs.data_ptr(), out.data_ptr(), obs.shape[0], _stream()))
    return out


def conv1_pairs_forward(pairs_copy, w, bias, pairs=None, out_planes=2, w_planes=3, alpha=1.0 / 255.0):
    """relu(alpha * conv1(obs, w) + bias) from the row-pair copy (acx_conv1_pairs_forward); w fp32 [256, 32] with rows (kh, kw, c).
    Returns bf16 planes [S * 400, 32]."""
    lib = _lib.load()
    samples = pairs_copy.shape[0]
    f = torch.arange(256, device=w.device)
    kh, kw, c = f // 32, (f // 4) % 8, f % 4
    col = (kh // 2) * 64 + kw * 8 + (kh % 2) * 4 + c
    wt = torch.empty((32, 256), dtype=torch.float32, device=w.device)
    wt[:, col] = w.t().float()
    wp = split_planes(wt, w_planes)
    outs = [torch.zeros((samples * 400, 32), dtype=torch.bfloat16, device=w.device) for _ in range(out_planes)]
    if pairs is None:
        pairs = [(0, j) for j in range(min(w_planes, 2))]
    pa = (ctypes.c_int * len(pairs))(*[p[0] for p in pairs])
    pb = (ctypes.c_int * len(pairs))(*[p[1] for p in pairs])
    ws, os_ = _planes_struct(wp, 32, 256), _planes_struct(outs, samples * 400, 32)
    _lib.check(lib.acx_conv1_pairs_forward(pairs_copy.data_ptr(), ctypes.byref(ws), samples, bias.data_ptr(), ctypes.c_float(alpha),
                                           ctypes.byref(os_), len(pairs), pa, pb, _stream()))
    return outs


def _planes_struct(planes, rows, cols):
    s = _lib.Planes()
    for i, p in enumerate(planes):
        s.planes[i] = p.data_ptr()
    s.num_planes = len(planes)
    s.rows, s.cols, s.ld = rows, cols, planes[0].stride(0)
    return s


PAIRS = {1: [(0, 0)], 3: [(0, 0), (0, 1), (1, 0)], 6: [(0, 0), (0, 1), (1, 0), (0, 2), (2, 0), (1, 1)]}


def gemm(a_planes, b_planes, m, n, k, trans=False, pairs=None, alpha=1.0, bias=None, relu=False, symmetric=False,
         out_planes=0, want_f32=True, mask=None, mask_rows=0, splits=0, impl=0, a_gather=None, b_gather=None, perm_m=0,
         perm_n=0):
    """C[m,n] = alpha * sum_pairs op(A_i) op(B_j) (+bias) via acx_gemm.
    trans=False: A planes stored [m,k], B planes stored [n,k];  trans=True: A stored [k,m], B stored [k,n]."""
    lib = _lib.load()
    if a_gather is not None:
        # operands read in place from NHWC tensors (acx_gather_t, include/acx.h); `a_planes` / `b_planes` only keep the tensors alive
        assert trans and pairs is not None
        dev = a_planes[0].device
        g = _lib.Gemm()
        g.a.num_planes, g.b.num_planes = a_gather.num_planes, (b_gather or a_gather).num_planes
        g.a_gather = ctypes.pointer(a_gather)
        if b_gather is not None:
            g.b_gather = ctypes.pointer(b_gather)
        g.perm_m, g.perm_n = perm_m, perm_n
        g.trans_a = g.trans_b = 1
        g.m, g.n, g.k = m, n, k
        g.num_pairs = len(pairs)
        for i, (pa, pb) in enumerate(pairs):
            g.pair_a[i], g.pair_b[i] = pa, pb
        g.alpha = alpha
        g.symmetric = int(symmetric)
        c = torch.empty((m, n), dtype=torch.float32, device=dev)
        g.c, g.ldc = c.data_ptr(), n
        g.splits = splits
        ws_bytes = lib.acx_gemm_workspace_bytes(ctypes.byref(g))
        ws = torch.zeros(max(ws_bytes, 4) // 4, dtype=torch.float32, device=dev)
        g.workspace, g.workspace_bytes = ws.data_ptr(), ws_bytes
        _lib.check(lib.acx_gemm(ctypes.byref(g), impl, _stream()))
        return c, []
    dev = b_planes[0].device
    if pairs is None:
        pairs = PAIRS[{1: 1, 2: 3, 3: 6}[min(len(a_planes), len(b_planes))]]
    g = _lib.Gemm()
    if trans:
        g.a = _planes_struct(a_planes, k, m)
        g.b = _planes_struct(b_planes, k, n)
    else:
        g.a = _planes_struct(a_planes, m, k)
        g.b = _planes_struct(b_planes, n, k)
    g.trans_a = g.trans_b = 1 if trans else 0
    g.m, g.n, g.k = m, n, k
    g.num_pairs = len(pairs)
    for i, (pa, pb) in enumerate(pairs):
        g.pair_a[i], g.pair_b[i] = pa, pb
    g.alpha = alpha
    g.bias = bias.data_ptr() if bias is not None else None
    g.relu = int(relu)
    g.symmetric = int(symmetric)
    c = None
    if want_f32:
        c = torch.empty((m, n), dtype=torch.float32, device=dev)
        g.c, g.ldc = c.data_ptr(), n
    cps = []
    if out_planes:
        ld = pad8(n)
        cps = [torch.zeros((m, ld), dtype=torch.bfloat16, device=dev) for _ in range(out_planes)]
        for i, p in enumerate(cps):
            g.c_planes[i] = p.data_ptr()
        g.c_num_planes, g.ldc_planes = out_planes, ld
    if mask is not None:
        g.mask_plane, g.mask_ld, g.mask_rows = mask.data_ptr(), mask.stride(0), mask_rows or mask.shape[0]
    g.splits = splits
    ws_bytes = lib.acx_gemm_workspace_bytes(ctypes.byref(g))
    ws = None
    if ws_bytes:
        ws = torch.zeros(ws_bytes // 4, dtype=torch.float32, device=dev)   # the counter head must be zero (acx.h)
        g.workspace, g.workspace_bytes = ws.data_ptr(), ws_bytes
    _lib.check(lib.acx_gemm(ctypes.byref(g), impl, _stream()))
    return c, cps


def _tensor_planes(planes, rows, cols):
    s = _lib.Planes()
    for i, p in enumerate(planes):
        s.planes[i] = p.data_ptr()
    s.num_planes = len(planes)
    s.rows, s.cols, s.ld = rows, cols, cols
    return s


def conv(x_planes, w_planes, geom, samples, dgrad=False, bias=None, relu=False, mask=None, mask_samples=0, pairs=None,
         out_planes=3, outs=None):
    """acx_conv: implicit-GEMM conv forward (x planes [samples,hw_in,hw_in,c_in], w = W^T planes [c_out, k*k*c_in]) or
    gather-form input gradient (x = output-gradient planes [samples,hw_out,hw_out,c_out], w = conv_dgrad_weights planes).
    geom = (hw_in, c_in, k, stride, hw_out, c_out).  Returns the list of bf16 output planes."""
    lib = _lib.load()
    hw_in, c_in, k, stride, hw_out, c_out = geom
    dev = x_planes[0].device
    c = _lib.Conv()
    c.dgrad, c.samples = int(dgrad), samples
    c.hw_in, c.c_in, c.k, c.stride, c.hw_out, c.c_out = geom
    if dgrad:
        c.x = _tensor_planes(x_planes, samples * hw_out * hw_out, c_out)
        out_shape = (samples, hw_in, hw_in, c_in)
    else:
        c.x = _tensor_planes(x_planes, samples * hw_in * hw_in, c_in)
        out_shape = (samples, hw_out, hw_out, c_out)
    c.w = _planes_struct(w_planes, w_planes[0].shape[0], w_planes[0].shape[1])
    if outs is None:
        outs = [torch.zeros(out_shape, dtype=torch.bfloat16, device=dev) for _ in range(out_planes)]
    c.out = _tensor_planes(outs, out_shape[0] * out_shape[1] * out_shape[2], out_shape[3])
    c.bias = bias.data_ptr() if bias is not None else None
    c.relu = int(relu)
    if mask is not None:
        c.mask_plane, c.mask_samples = mask.data_ptr(), mask_samples or mask.shape[0]
    if pairs is None:
        pairs = PAIRS[{1: 1, 2: 3, 3: 6}[min(len(x_planes), len(w_planes))]]
    c.num_pairs = len(pairs)
    for i, (pa, pb) in enumerate(pairs):
        c.pair_a[i], c.pair_b[i] = pa, pb
    if not lib.acx_conv_supported(ctypes.byref(c)):
        raise _lib.AcxError("acx_conv: unsupported geometry %r (dgrad=%s)" % (geom, dgrad))
    _lib.check(lib.acx_conv(ctypes.byref(c), _stream()))
    return outs


def conv_dgrad_weights(w, geom):
    """fp32 HWIO weights [k*k*c_in, c_out] -> 3 bf16 planes [stride^2*c_in, pad8((k/stride)^2*c_out)] (acx_conv_dgrad_weights)."""
    hw_in, c_in, k, stride, hw_out, c_out = geom
    m = k // stride
    rows, ld = stride * stride * c_in, pad8(m * m * c_out)
    planes = [torch.empty((rows, ld), dtype=torch.bfloat16, device=w.device) for _ in range(3)]
    arr = (ctypes.c_void_p * 3)(*[p.data_ptr() for p in planes])
    _lib.check(_lib.load().acx_conv_dgrad_weights(_ptr(w.contiguous().float()), hw_in, c_in, k, stride, hw_out, c_out, arr, ld,
                                                  _stream()))
    return planes


def sample_actions(logits, uniform=None, seed=0, step=0, greedy=False):
    """acx_sample_actions: DistributionPolicy.sample / mode (policies.py:86-87) on device logits [rows, A] -> int32 [rows]."""
    _need_cuda(logits, uniform)
    logits = logits.contiguous().float()
    rows, num_actions = logits.shape
    actions = torch.empty(rows, dtype=torch.int32, device=logits.device)
    _lib.check(_lib.load().acx_sample_actions(_ptr(logits), _ptr(uniform), ctypes.c_uint64(seed), ctypes.c_uint64(step), rows,
                                              num_actions, int(bool(greedy)), _ptr(actions), _stream()))
    return actions


def clip_rmsprop_step(params, ms, grads, lr, decay=0.9, epsilon=1e-10, clip_norm=3.4e38):
    """acx_clip_rmsprop_step on flat fp32 CUDA vectors, in place; returns the gradient's global norm (device scalar)."""
    _need_cuda(params, ms, grads)
    scratch = torch.empty(297, dtype=torch.float32, device=params.device)
    _lib.check(_lib.load().acx_clip_rmsprop_step(_ptr(params), _ptr(ms), _ptr(grads), ctypes.c_size_t(params.numel()), float(lr),
                                                 float(decay), float(epsilon), float(clip_norm), _ptr(scratch),
                                                 ctypes.c_void_p(scratch.data_ptr() + 296 * 4), _stream()))
    return scratch[296]


def clip_momentum_step(params, accum, grads, lr, momentum=0.9, clip_norm=3.4e38):
    """acx_clip_momentum_step on flat fp32 CUDA vectors, in place; returns the gradient's global norm (device scalar)."""
    _need_cuda(params, accum, grads)
    scratch = torch.empty(297, dtype=torch.float32, device=params.device)
    _lib.check(_lib.load().acx_clip_momentum_step(_ptr(params), _ptr(accum), _ptr(grads), ctypes.c_size_t(params.numel()),
                                                  float(lr), float(momentum), float(clip_norm), _ptr(scratch),
                                                  ctypes.c_void_p(scratch.data_ptr() + 296 * 4), _stream()))
    return scratch[296]


def kfac_invert(a_sums, g_sums, tnorm=None, shared_heads=False, damping=0.01, debias=1.0, path=0, side_stream=False):
    """acx_debug_kfac_invert: one K-FAC inverse refresh of the blocks the learners would build, on host fp32 running sums.
    a_sums: one [d, d] input factor per block (one fewer with shared_heads: the last two blocks share the last one);
    g_sums: one [C, C] output factor per block; tnorm: T~ per block (default 1).  path 0 = the learners' refresh,
    1 = the resident kernel only, 2 = the fp64 chain only.  Returns None when path 1 does not fit, else a dict with
    inv_a / inv_g (fp32 [n, n] per block), planes_a / planes_g (uint16 bf16 bits [3, n, pad8(n)] per block),
    damp (fp32 [num_blocks, 2]: damp_A, damp_G) and path (0 = resident kernel ran, 1 = fp64 chain)."""
    import numpy as np
    a_sums = [np.ascontiguousarray(a, dtype=np.float32) for a in a_sums]
    g_sums = [np.ascontiguousarray(g, dtype=np.float32) for g in g_sums]
    nb = len(g_sums)
    assert len(a_sums) == (nb - 1 if shared_heads else nb)
    dims_a = [a_sums[min(i, len(a_sums) - 1)].shape[0] for i in range(nb)]
    dims_g = [g.shape[0] for g in g_sums]
    tnorm = [1] * nb if tnorm is None else list(tnorm)
    sums = np.concatenate([s.ravel() for s in a_sums + g_sums])
    dims = dims_a + dims_g
    inv = np.empty(sum(n * n for n in dims), np.float32)
    planes = np.empty(sum(3 * n * pad8(n) for n in dims), np.uint16)
    damp = np.empty(2 * nb, np.float32)
    ran = ctypes.c_int(-1)

    def ints(v):
        return (ctypes.c_int * nb)(*[int(x) for x in v])
    st = _lib.load().acx_debug_kfac_invert(nb, ints([d - 1 for d in dims_a]), ints(dims_g), ints(tnorm), int(bool(shared_heads)),
                                           float(damping), float(debias), sums.ctypes.data, int(path), int(bool(side_stream)),
                                           inv.ctypes.data, planes.ctypes.data, damp.ctypes.data, ctypes.byref(ran))
    if st == -1 and path == 1:
        return None
    _lib.check(st)
    out = dict(inv_a=[], inv_g=[], planes_a=[], planes_g=[], damp=damp.reshape(nb, 2), path=ran.value)
    io = po = 0
    for j, n in enumerate(dims):
        kind = "a" if j < nb else "g"
        out["inv_" + kind].append(inv[io:io + n * n].reshape(n, n))
        out["planes_" + kind].append(planes[po:po + 3 * n * pad8(n)].reshape(3, n, pad8(n)))
        io += n * n
        po += 3 * n * pad8(n)
    return out
