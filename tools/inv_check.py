"""python tools/inv_check.py [c3]: runs 4 refreshing updates (invert_every = 1) and prints a digest of the inverses (equal
digests across two builds mean bit-identical inverses), their error against numpy fp64, the inverse-stage time and which
refresh path ran, read from the launch count: the resident fp32 kernel is one launch, its fallback for factors whose tiles do
not fit the SMs (conv3 > 64) is the fp64 chain of about three launches per 32-row pivot step.  With ACX_INV_TRACE=1|2 it
also prints the per-step clock64 breakdown of the resident kernel."""
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import synth  # noqa: E402
from actorcritic_b200 import engine as eng  # noqa: E402
from actorcritic_b200 import _lib  # noqa: E402

c3 = int(sys.argv[1]) if len(sys.argv) > 1 else 32
envs, steps = (32, 20) if c3 == 32 else (8, 5)
cfg = eng.EngineConfig(num_envs=envs, num_steps=steps, conv3_filters=c3, num_cold_updates=0, invert_every=1)
e = eng.Engine(cfg)
e.set_params(eng.orthogonal_init(4, c3, seed=0))
b = synth.rollout(1, envs, steps, 4, obs_kind="uniform")
y, eps = synth.fisher_samples(2, envs * steps)
fl, fe = torch.from_numpy(y).cuda(), torch.from_numpy(eps).cuda()
for u in range(4):
    e.update(b, fl, fe, fetch=False)
torch.cuda.synchronize()
inv = e.buffer("inverses").cpu().numpy()
print("c3", c3, "tc_error", _lib.load().acx_debug_tc_error(),
      "finite", bool(np.isfinite(inv).all()), "digest", hashlib.sha1(inv.tobytes()).hexdigest()[:16],
      "params", hashlib.sha1(e.get_params_flat().tobytes()).hexdigest()[:16])
# accuracy of every stored inverse against numpy fp64 on the engine's own running sums and dampings
damp = e.buffer("dampings").cpu().numpy().astype(np.float64)
ncov = e.get_state()["num_cov_updates"]
debias = 1.0 / (1.0 - 0.99 ** ncov)
worst = {}
for li, layer in enumerate(eng.LAYERS):
    fac = "heads" if layer.startswith("fc_p") or layer.startswith("fc_b") else layer
    for which, name, d in (("A", fac, damp[2 * li]), ("G", layer, damp[2 * li + 1])):
        sm = e.factor("sums", which, name).cpu().numpy().astype(np.float64)
        m = 0.5 * (sm + sm.T) * debias + d * np.eye(sm.shape[0])
        want = np.linalg.inv(m)
        got = e.factor("inv", which, layer).cpu().numpy().astype(np.float64)
        worst["%s/%s" % (which, layer)] = float(np.linalg.norm(got - want) / np.linalg.norm(want))
        if which == "A" and layer == "fc4":
            err = np.abs(got - want)
            blk = err[: (err.shape[0] // 32) * 32, : (err.shape[0] // 32) * 32].reshape(err.shape[0] // 32, 32, -1, 32).max(axis=(1, 3))
            top = np.dstack(np.unravel_index(np.argsort(blk.ravel())[::-1][:12], blk.shape))[0]
            print("fc4 A: max |err| %.3e at %s, |want| max %.3e; worst 32-blocks (row, col, err):" % (
                err.max(), np.unravel_index(err.argmax(), err.shape), np.abs(want).max()),
                [(int(r), int(c), "%.1e" % blk[r, c]) for r, c in top])
            print("   error by block row:", ["%.0e" % v for v in blk.max(axis=1)])
            print("   edge rows/cols err:", "%.2e" % err[-1, :].max(), "%.2e" % err[:, -1].max(), "diag err max %.2e" % np.abs(np.diag(got - want)).max(),
                  "asym %.2e" % np.abs(got - got.T).max())
print("inverse rel err vs fp64:", {k: "%.1e" % v for k, v in worst.items()})
e.set_profiling(True)
ts = []
launches0 = _lib.launch_count()
for u in range(6):
    e.update(b, fl, fe, fetch=False)
    torch.cuda.synchronize()
    ts.append(e.stage_ms()["inverse"])
e.set_profiling(False)
launches = (_lib.launch_count() - launches0) / 6
n_fc4 = 49 * c3 + 1
path = "fp64 chain" if launches > 3 * (n_fc4 // 32) else "resident fp32"
print("inverse stage ms per refresh (serial, eager):", ["%.3f" % t for t in ts])
print("launches per refreshing update %.0f: %s refresh" % (launches, path))
# graph-replayed whole update with refresh
ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
with torch.cuda.stream(e.stream):
    for u in range(3):
        e.update(b, fl, fe, fetch=False)
    ev0.record()
    for u in range(10):
        e.update(b, fl, fe, fetch=False)
    ev1.record()
torch.cuda.synchronize()
print("ms per refreshing update (graphs): %.3f" % (ev0.elapsed_time(ev1) / 10), "tc_error", _lib.load().acx_debug_tc_error())

if os.environ.get("ACX_INV_TRACE"):
    import ctypes
    buf = (ctypes.c_longlong * 1024)()
    _lib.load().acx_debug_inv_trace(buf, 1024)
    t = np.array(list(buf), np.int64).reshape(128, 8)
    steps = (int(49 * c3 / 32) + 1 + 31) // 32 if False else None
    print("step: panels | bar1 | update | bar2 | total (cycles)   || cta0: look-ahead")
    for p in range(0, 100):
        r = t[p]
        if r[4] == 0:
            break
        if p < 6 or p % 8 == 0 or p > 44:
            print(p, r[1] - r[0], r[2] - r[1], r[3] - r[2], r[4] - r[3], r[4] - r[0], "||", r[6] - r[5],
                  "| first tile: staged +%d, updated +%d, published +%d" % (r[5] - r[2], r[6] - r[5], r[7] - r[6])
                  if os.environ.get("ACX_INV_TRACE") == "2" else "")
    valid = t[(t[:, 4] > 0)]
    tot = valid[:, 4] - valid[:, 0]
    print("sum cycles", int(tot.sum()), "panels", int((valid[:, 1] - valid[:, 0]).sum()), "bar1", int((valid[:, 2] - valid[:, 1]).sum()),
          "update", int((valid[:, 3] - valid[:, 2]).sum()), "bar2", int((valid[:, 4] - valid[:, 3]).sum()), "lookahead", int((valid[:, 6] - valid[:, 5]).sum()))
