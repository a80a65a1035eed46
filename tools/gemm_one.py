"""Run one GEMM shape a few times (for ncu --set full).  usage: gemm_one.py name  (see SHAPES)."""
import sys, os
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from actorcritic_b200 import ops

SHAPES = {  # name: (m, n, k, trans, sym, planes, out_planes)
    "fwd_conv1": (268800, 32, 256, False, False, 3, 3),
    "fwd_conv2": (54432, 64, 512, False, False, 3, 3),
    "dgrad_conv2": (103680, 512, 64, False, False, 3, 0),
    "wgrad_conv1": (256, 32, 256000, True, False, 3, 0),
    "syrk_conv1": (256, 256, 256000, True, True, 1, 0),
    "syrk_conv2": (512, 512, 51840, True, True, 2, 0),
    "fc4": (672, 512, 1568, False, False, 3, 3),
}
name = sys.argv[1]
if name == "syrk_conv2_gather":   # the default path: A2 = P2^T P2 read in place from act1 planes [640, 20, 20, 32] (acx_gather_t)
    import ctypes
    from actorcritic_b200 import _lib
    lib = _lib.load()
    iters = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    xp = ops.split_planes(torch.rand((640 * 400, 32), device="cuda"), 2)
    ga = ops.nature_cnn_gather(xp, "conv2", 640)
    lib.acx_gemm_enable_timing(1)
    durs = []
    for _ in range(max(iters, 5)):
        ops.gemm(xp, xp, 512, 512, 51840, trans=True, symmetric=True, pairs=ops.PAIRS[3], alpha=1.0 / 51840, a_gather=ga)
        ms = ctypes.c_float(0)
        _lib.check(lib.acx_gemm_last_ms(ctypes.byref(ms)))
        durs.append(ms.value)
    print(name, "kernel-only us (library events):", " ".join("%.1f" % (1e3 * d) for d in durs))
    sys.exit(0)
iters = int(sys.argv[2]) if len(sys.argv) > 2 else 3
m, n, k, trans, sym, npl, outp = SHAPES[name]
x = torch.randn((k, m) if trans else (m, k), device="cuda")
a_pl = ops.split_planes(x, npl if name not in ("fwd_conv1", "wgrad_conv1") else 1)
b_pl = a_pl if sym else ops.split_planes(torch.randn((k, n) if trans else (n, k), device="cuda"), npl)
pairs = None
if name in ("fwd_conv1", "wgrad_conv1"):
    pairs = [(0, 0), (0, 1), (0, 2)]
bias = torch.randn(n, device="cuda") if outp else None
for _ in range(iters):
    ops.gemm(a_pl, b_pl, m, n, k, trans=trans, symmetric=sym, out_planes=outp, want_f32=outp == 0, pairs=pairs, bias=bias, relu=bool(outp))
torch.cuda.synchronize()
import ctypes
from actorcritic_b200 import _lib
lib = _lib.load()
lib.acx_gemm_enable_timing(1)
durs = []
for _ in range(max(iters, 5)):
    ops.gemm(a_pl, b_pl, m, n, k, trans=trans, symmetric=sym, out_planes=outp, want_f32=outp == 0, pairs=pairs, bias=bias, relu=bool(outp))
    ms = ctypes.c_float(0)
    _lib.check(lib.acx_gemm_last_ms(ctypes.byref(ms)))
    durs.append(ms.value)
lib.acx_gemm_enable_timing(0)
print(name, "kernel-only us (library events):", " ".join("%.1f" % (1e3 * d) for d in durs))
if os.environ.get("ACX_GEMM_TRACE"):
    arr = (ctypes.c_longlong * 12)()
    lib.acx_debug_gemm_trace(arr)
    t = list(arr)
    print("  CTA 0 MMA warp: %d cycles, %d k-blocks (%.0f cycles each); waiting for operands %.0f%%, for an accumulator %.0f%%"
          % (t[0], t[3], t[0] / max(t[3], 1), 100.0 * t[1] / max(t[0], 1), 100.0 * t[2] / max(t[0], 1)))
sys.exit(0)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(iters):
    ops.gemm(a_pl, b_pl, m, n, k, trans=trans, symmetric=sym, out_planes=outp, want_f32=outp == 0, pairs=pairs, bias=bias, relu=bool(outp))
e1.record()
torch.cuda.synchronize()
print(name, "ms", e0.elapsed_time(e1) / iters)
