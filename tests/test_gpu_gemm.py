"""acx_gemm (csrc/gemm.cu) through the C ABI against fp64 products of the same bf16 planes: both operand layouts,
split-K with the reduction inside the kernel (one group, two levels, the SYRK panel), symmetric results with mirrored
tiles, every epilogue option on the reduced path, ragged shapes, run-to-run bit reproducibility, and the workspace
contract of include/acx.h (arrival counters zero on entry, left zero).  The operations these GEMMs stand for:
nn.py:110 (conv as patch GEMM), nn.py:48-52 (fully connected), tf.gradients of both (objectives.py:79) and kfac's
factor statistics (SURVEY A.5)."""
import ctypes
import os

import pytest
import torch

pytestmark = pytest.mark.gpu


def _ops():
    from actorcritic_b200 import _lib, ops
    return _lib, ops


def _ref(a_pl, b_pl, pairs, trans, m, n, k):
    acc = None
    for pa, pb in pairs:
        a = a_pl[pa].double()
        b = b_pl[pb].double()
        t = (a[:k, :m].t() @ b[:k, :n]) if trans else (a[:m, :k] @ b[:n, :k].t())
        acc = t if acc is None else acc + t
    return acc


def _operands(ops, m, n, k, trans, nplanes, symmetric, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    xa = torch.randn((k, m) if trans else (m, k), device="cuda", generator=g)
    a_pl = ops.split_planes(xa, nplanes)
    if symmetric:
        return a_pl, a_pl
    xb = torch.randn((k, n) if trans else (n, k), device="cuda", generator=g)
    return a_pl, ops.split_planes(xb, nplanes)


CASES = [
    # name, m, n, k, trans, planes, splits, symmetric
    ("k_major_direct", 256, 128, 256, False, 1, 1, False),
    ("k_major_one_group", 300, 200, 4096, False, 2, 6, False),
    ("k_major_two_levels", 128, 64, 16384, False, 2, 37, False),
    ("k_major_ragged", 333, 203, 1111, False, 2, 3, False),
    ("mn_major_auto", 512, 64, 20000, True, 2, 0, False),          # conv2 weight gradient shape: deep automatic split
    ("mn_major_two_levels", 256, 32, 40000, True, 2, 73, False),   # conv1 weight gradient shape
    ("syrk_tiles", 512, 512, 5184, True, 2, 0, True),              # conv2 input factor shape (10 upper tiles)
    ("syrk_ragged", 577, 577, 1000, True, 2, 0, True),
    ("syrk_panel", 256, 256, 30000, True, 1, 0, True),             # conv1 input factor: panel mode, two-level reduction
    ("syrk_narrow", 32, 32, 50000, True, 2, 0, True),              # conv output factor: one tile, maximal split
    ("syrk_single_split", 1569, 1569, 64, True, 2, 1, True),       # splits = 1: every CTA is its own last arrival
]


@pytest.fixture(params=[0, 1, 2], ids=["finalize_launch", "fused_where_cheap", "fused_always"])
def reduce_mode(request):
    """Where split-K partials are summed (acx.h: acx_debug_set_fuse_reduce).  Each case restores the library default
    (ACX_GEMM_FUSE_REDUCE, else 0 = finalize launches), so the test files that run after this one see the mode users get."""
    _lib, _ = _ops()
    _lib.load().acx_debug_set_fuse_reduce(request.param)
    yield request.param
    _lib.load().acx_debug_set_fuse_reduce(int(os.environ.get("ACX_GEMM_FUSE_REDUCE", "0")))


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_gemm_matches_fp64_and_is_reproducible(case, reduce_mode):
    _lib, ops = _ops()
    name, m, n, k, trans, nplanes, splits, symmetric = case
    a_pl, b_pl = _operands(ops, m, n, k, trans, nplanes, symmetric, seed=len(name) + m + k)
    pairs = ops.PAIRS[{1: 1, 2: 3, 3: 6}[nplanes]]
    want = _ref(a_pl, b_pl, pairs, trans, m, n, k)
    c1, _ = ops.gemm(a_pl, b_pl, m, n, k, trans=trans, pairs=pairs, splits=splits, symmetric=symmetric)
    c2, _ = ops.gemm(a_pl, b_pl, m, n, k, trans=trans, pairs=pairs, splits=splits, symmetric=symmetric)
    torch.cuda.synchronize()
    assert _lib.load().acx_debug_tc_error() == 0
    scale = float(want.abs().max())
    assert float((c1.double() - want).abs().max()) <= 5e-5 * scale, name
    assert torch.equal(c1, c2), "split-K reduction must not depend on the arrival order"
    if symmetric:
        assert torch.equal(c1, c1.t()) or float((c1 - c1.t()).abs().max()) <= 1e-6 * scale   # mirrored blocks are exact copies
        iu = torch.triu_indices(m, m, offset=32, device="cuda")   # beyond the diagonal 32-blocks the mirror is bit-exact
        assert torch.equal(c1[iu[0], iu[1]], c1[iu[1], iu[0]])


def test_reduced_path_applies_every_epilogue_option(reduce_mode):
    _lib, ops = _ops()
    m, n, k = 200, 134, 8192
    a_pl, b_pl = _operands(ops, m, n, k, False, 2, False, seed=5)
    pairs = ops.PAIRS[3]
    g = torch.Generator(device="cuda").manual_seed(9)
    bias = torch.randn(n, device="cuda", generator=g)
    mask = (torch.rand((50, 136), device="cuda", generator=g) > 0.4).to(torch.bfloat16)[:, :n]   # row stride 136
    want = 0.5 * _ref(a_pl, b_pl, pairs, False, m, n, k) + bias.double()[None, :]
    want = want.clamp_min(0) * (mask.double() > 0).repeat(4, 1)
    for splits in (1, 3, 5, 20):
        c, planes = ops.gemm(a_pl, b_pl, m, n, k, pairs=pairs, alpha=0.5, bias=bias, relu=True, mask=mask, mask_rows=50,
                             out_planes=3, splits=splits)
        torch.cuda.synchronize()
        scale = float(want.abs().max())
        assert float((c.double() - want).abs().max()) <= 5e-5 * scale, splits
        rebuilt = sum(p.double() for p in planes)[:, :n]
        assert float((rebuilt - c.double()).abs().max()) <= 2e-7 * scale, splits   # three bf16 planes carry the fp32 value
        assert not bool(sum(p.float().abs() for p in planes)[:, n:].any()), "padding columns of the planes stay zero"


def test_workspace_counters_are_left_zero_and_reusable(reduce_mode):
    """include/acx.h: the head of the workspace holds arrival counters - zero on entry, zero on exit."""
    _lib, ops = _ops()
    lib = _lib.load()
    m, n, k = 256, 64, 32768
    a_pl, b_pl = _operands(ops, m, n, k, True, 2, False, seed=3)
    pairs = ops.PAIRS[3]
    want = _ref(a_pl, b_pl, pairs, True, m, n, k)
    g = _lib.Gemm()
    g.a = ops._planes_struct(a_pl, k, m)
    g.b = ops._planes_struct(b_pl, k, n)
    g.trans_a = g.trans_b = 1
    g.m, g.n, g.k = m, n, k
    g.num_pairs = len(pairs)
    for i, (pa, pb) in enumerate(pairs):
        g.pair_a[i], g.pair_b[i] = pa, pb
    g.alpha = 1.0
    c = torch.empty((m, n), dtype=torch.float32, device="cuda")
    g.c, g.ldc = c.data_ptr(), n
    g.splits = 0 if reduce_mode == 2 else 4
    nbytes = lib.acx_gemm_workspace_bytes(ctypes.byref(g))
    assert nbytes > 16384
    ws = torch.zeros(nbytes // 4, dtype=torch.float32, device="cuda")
    ws[4096:] = float("nan")   # the partial-sum area may hold anything
    g.workspace, g.workspace_bytes = ws.data_ptr(), nbytes
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    for _ in range(3):   # reused without clearing
        c.fill_(float("nan"))
        _lib.check(lib.acx_gemm(ctypes.byref(g), 0, stream))
        torch.cuda.synchronize()
        assert not bool(ws[:4096].view(torch.int32).any()), "counters must be left zero"
        assert float((c.double() - want).abs().max()) <= 5e-5 * float(want.abs().max())
