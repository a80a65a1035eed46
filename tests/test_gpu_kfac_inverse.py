"""The K-FAC inverse refresh on its own (include/acx.h acx_debug_kfac_invert): KfacBlocks::invert as the learners run it -
the resident fp32 kernel (csrc/kfac_inv.cu) or, when its tiles do not fit, the fp64 chain (csrc/kfac.cu) - and each of the
two forced, against the fp64 reference oracle.kfac.damped_inverse computed with the kernel's own fp32 damping and debias
factor (which separates damping errors from inverse errors).

Per job:
  dampings   within 2 ulp of the fp64 pi formula (oracle.kfac.pi_dampings);
  chain      relative Frobenius error <= 1e-7 + 1e-15 n kappa: fp32 output rounding plus an fp64 Gauss-Jordan term;
  resident   relative Frobenius error <= 16 x that of scipy's fp32 Cholesky inverse of the same matrix, plus 2e-6 (fp32
             Gauss-Jordan without pivoting against a backward-stable fp32 inverse), up to RESIDENT_KAPPA_LIMIT;
  structure  finite and bit-symmetric (both finish stages write the two halves from one value); diagonal in
             (0, (1 + 1e-3) / lambda_min(M)] with lambda_min(M) >= damping (M >= lambda_min I  =>  M^-1 <= I / lambda_min);
             the bf16 planes bit-equal to a torch restatement of split3 (round to nearest bf16, three times), padding zero;
  determinism two runs give the same bits; the chain the same bits with and without its side stream;
  error flags acx_debug_tc_error() == 0 after every call.
Sizes cover the tile edges of both paths (32-row pivot blocks, 64 x 64 tiles), the job sets of every learner geometry the
other tests run, the largest factor the resident kernel holds on this device and the next tile row, condition numbers 1e1 ..
1e7, and the factors of a trained network.  Every line starting with "kfac-inv" is a measurement (pytest -s shows them)."""
import functools
import json

import numpy as np
import pytest
import scipy.linalg
import torch

from oracle import kfac as K

from actorcritic_b200 import _lib
from actorcritic_b200 import engine as eng
from actorcritic_b200 import ops

pytestmark = pytest.mark.gpu

DEBIAS3 = 1.0 / (1.0 - 0.99 ** 3)   # zero-debias factor after three covariance updates
# The resident kernel's accuracy bound is asserted up to this condition number of a damped factor, at least ten times the
# largest one measured on the factors of a trained network (test_factors_of_a_trained_network; DESIGN.md section 4).  Beyond
# it the fp32 Gauss-Jordan without pivoting loses accuracy much faster than a Cholesky inverse (measured on a B200 at 1e7 with
# a rank-64 factor of 513: relative error 4 - 200 against 6e-2); there only the structure is checked.
RESIDENT_KAPPA_LIMIT = 1e6
# The resident bound is twice the one derived from the arithmetic (8 x Cholesky + 1e-6): the test factors are strongly graded
# (column scales over 14 octaves), which an fp32 Cholesky inverse does not feel (it is invariant under diagonal scaling) and
# Gauss-Jordan does; measured on a B200 the kernel reached 1.9 x the derived bound (n = 1569, full rank, kappa 1e4:
# 3.6e-6 against a Cholesky error of 1.3e-7), at every kappa from 10 on, so the excess grows with n, not with kappa.
RESIDENT_FACTOR, RESIDENT_FLOOR = 16.0, 2e-6


def record(kind, **kw):
    print("kfac-inv", json.dumps(dict(kind=kind, **kw), default=float))


class Case:
    """A set of K-FAC blocks with their running sums: a[f] input factors, g[i] output factors (float64 tensors holding fp32
    values), T~ per block, shared heads; `spectra` maps id(sum) -> (lambda_min, lambda_max) of sym(sum) where known."""

    def __init__(self, a, g, tnorm=None, shared=False, damping=0.01, debias=1.0, spectra=None):
        self.a, self.g, self.shared, self.damping, self.debias = a, g, shared, damping, debias
        self.tnorm = tnorm or [1] * len(g)
        self.spectra = spectra or {}

    def a_of(self, i):
        return self.a[min(i, len(self.a) - 1)]

    def extremes(self, s):
        if id(s) not in self.spectra:
            lam = torch.linalg.eigvalsh(0.5 * (s + s.T))
            self.spectra[id(s)] = (float(lam[0]), float(lam[-1]))
        return self.spectra[id(s)]


def run(case, path, side=False):
    r = ops.kfac_invert([a.numpy() for a in case.a], [g.numpy() for g in case.g], case.tnorm, case.shared, case.damping,
                        case.debias, path, side)
    assert _lib.load().acx_debug_tc_error() == 0
    return r


def split3_bits(x):
    """split3 (csrc/common.cuh) restated: three round-to-nearest bf16 planes of the fp32 values, as uint16 bits."""
    r = torch.from_numpy(np.ascontiguousarray(x))
    out = []
    for _ in range(3):
        p = r.to(torch.bfloat16)
        out.append(p.view(torch.int16).numpy().view(np.uint16))
        r = r - p.float()
    return out


def chol32_error(m, want):
    """Relative error of scipy's fp32 Cholesky inverse; None when the fp32 matrix is not positive definite to LAPACK."""
    try:
        c = scipy.linalg.cho_factor(m.astype(np.float32), lower=True)
    except np.linalg.LinAlgError:
        return None
    got = scipy.linalg.cho_solve(c, np.eye(m.shape[0], dtype=np.float32))
    return float(np.linalg.norm(got.astype(np.float64) - want) / np.linalg.norm(want))


def check(case, r, tag, resident_kappa_limit=None):
    """Every per-job assertion of the module docstring for one refresh result; returns the worst ratio of error to bound."""
    limit = RESIDENT_KAPPA_LIMIT if resident_kappa_limit is None else resident_kappa_limit
    nb = len(case.g)
    debias = float(np.float32(case.debias))
    worst = 0.0
    for i in range(nb):
        lam = float(np.float32(np.float32(case.damping) / np.float32(case.tnorm[i])))
        want_da, want_dg = K.pi_dampings(case.a_of(i), case.g[i], lam)
        for which, s, want_d, d32, inv, planes in (
                ("A", case.a_of(i), want_da, r["damp"][i, 0], r["inv_a"][i], r["planes_a"][i] if "planes_a" in r else None),
                ("G", case.g[i], want_dg, r["damp"][i, 1], r["inv_g"][i], r["planes_g"][i] if "planes_g" in r else None)):
            n = s.shape[0]
            job = "%s %s%d n=%d" % (tag, which, i, n)
            assert abs(float(d32) - want_d) <= 2 * float(np.spacing(np.float32(want_d))), (job, float(d32), want_d)
            d = float(d32)
            want = K.damped_inverse(s, debias, d).numpy()
            lo, hi = case.extremes(s)
            lam_min = debias * lo + d
            kappa = (debias * hi + d) / lam_min
            got = inv.astype(np.float64)
            err = float(np.linalg.norm(got - want) / np.linalg.norm(want)) if np.isfinite(got).all() else float("inf")
            if r["path"] == 1:
                bound = 1e-7 + 1e-15 * n * kappa
                ref = None
            else:
                m = 0.5 * (s + s.T).numpy() * debias + d * np.eye(n)
                ref = chol32_error(m, want)
                bound = RESIDENT_FACTOR * ref + RESIDENT_FLOOR if ref is not None else float("inf")
                assert ref is not None or kappa > limit, (job, "fp32 Cholesky failed", kappa)
            record("job", job=job, path=("resident", "chain")[r["path"]], kappa=kappa, err=err, bound=bound, chol32=ref,
                   ratio=err / bound)
            # structure (both finish stages): bit-symmetric, planes from the stored fp32 values, zero padding
            assert np.array_equal(inv.view(np.uint32), inv.T.view(np.uint32)), job
            if planes is not None and np.isfinite(inv).all():
                for q, p in enumerate(split3_bits(inv)):
                    assert np.array_equal(planes[q][:, :n], p), (job, q)
                assert not planes[:, :, n:].any(), job
            if r["path"] == 0 and kappa > limit:
                continue
            worst = max(worst, err / bound)
            assert np.isfinite(inv).all(), job
            diag = np.diag(got)
            assert (diag > 0).all() and diag.max() <= (1 + 1e-3) / min(d, lam_min), (job, diag.max() * d)
            assert err <= bound, (job, err, bound, kappa)
    return worst


def same_bits(r0, r1):
    for k in ("inv_a", "inv_g", "planes_a", "planes_g"):
        for x, y in zip(r0[k], r1[k]):
            if not np.array_equal(x.view(np.uint8), y.view(np.uint8)):
                return False
    return np.array_equal(r0["damp"].view(np.uint32), r1["damp"].view(np.uint32))


def both_paths(case, tag, want_path=None):
    """The learners' refresh, the resident kernel (when it fits) and the chain (with and without its side stream) on one
    case: each meets the bounds, runs are deterministic and the learners' refresh is bit-identical to the path it took."""
    r0 = run(case, 0)
    assert same_bits(r0, run(case, 0)), tag
    if want_path is not None:
        assert r0["path"] == {"resident": 0, "chain": 1}[want_path], (tag, r0["path"])
    r1 = run(case, 1)
    assert (r1 is None) == (r0["path"] == 1), tag
    r2 = run(case, 2)
    assert same_bits(r2, run(case, 2, side=True)), tag
    assert same_bits(r0, r1 if r0["path"] == 0 else r2), tag
    if r1 is not None:
        check(case, r1, tag + " resident")
    check(case, r2, tag + " chain")


# ------------------------------------------------------------------------------------------------ factor sets
@functools.lru_cache(maxsize=None)
def gram(n, rows, seed):
    return K.gram_factor(n, rows, seed)


def small_g(c, seed):
    return K.spectrum_factor(np.geomspace(1.0, 1e-2, c) * (1.0 + 0.1 * seed), seed)


def blocks_case(ks, cs, tnorm=None, shared=True, seed=0, **kw):
    """Input factors: Gram matrices of 64 scaled integer rows with the homogeneous column (rank-deficient beyond 64);
    output factors: Gram matrices of 64 rows without it."""
    nfac = len(ks) - 1 if shared else len(ks)
    spectra = {}
    a = []
    for f in range(nfac):
        s, lo, hi = gram(ks[f] + 1, 64, seed + f)
        spectra[id(s)] = (lo, hi)
        a.append(s)
    g = []
    for i, c in enumerate(cs):
        s, lo, hi = K.gram_factor(c, 64, seed + 100 + i, homogeneous=False, scale_octaves=4)
        spectra[id(s)] = (lo, hi)
        g.append(s)
    return Case(a, g, tnorm, shared, spectra=spectra, **kw)


def atari_case(c3, num_actions=4):
    return blocks_case([256, 512, 576, 49 * c3, 512, 512], [32, 64, c3, 512, num_actions, 1], [400, 81, 49, 1, 1, 1])


def mlp_case(obs_dim, hidden_sizes, num_actions, **_):
    shapes = eng.mlp_param_shapes(obs_dim, hidden_sizes, num_actions)
    layers = eng.mlp_layers(len(hidden_sizes))
    return blocks_case([shapes[l + "/weights"][0] for l in layers], [shapes[l + "/weights"][1] for l in layers])


def cnn_case(obs_hw, obs_channels, conv_layers, hidden_sizes, num_actions, **_):
    shapes = eng.cnn_param_shapes(obs_hw, obs_channels, conv_layers, hidden_sizes, num_actions)
    layers = eng.cnn_layers(len(conv_layers), len(hidden_sizes))
    geo = eng.cnn_conv_geometry(obs_hw, obs_channels, conv_layers)
    tnorm = [g[5] * g[5] for g in geo] + [1] * (len(layers) - len(geo))
    ks = [int(np.prod(shapes[l + "/weights"][:-1])) for l in layers]
    return blocks_case(ks, [shapes[l + "/weights"][-1] for l in layers], tnorm)


# ------------------------------------------------------------------------------------------------ sizes
SWEEP = [1, 2, 3, 8, 31, 32, 33, 63, 64, 65, 95, 96, 97, 127, 128, 129, 257, 511, 513, 1025, 1569]


@pytest.mark.parametrize("path", [1, 2], ids=["resident", "chain"])
@pytest.mark.parametrize("n", SWEEP)
def test_single_block_sizes(n, path):
    """One block: an n x n input factor (64 scaled rows with the homogeneous column, one-ulp antisymmetric part) and a
    3 x 3 output factor, at every tile edge of both paths; two runs give the same bits."""
    s, lo, hi = gram(n, 64, n)
    a = K.with_antisymmetric_ulp(s)
    assert not torch.equal(a, a.T) or n == 1
    g = small_g(3, n)
    case = Case([a], [g], spectra={id(a): (lo, hi)})
    r = run(case, path)
    assert r is not None and r["path"] == path - 1
    assert same_bits(r, run(case, path)), n
    check(case, r, "n=%d" % n)


def test_zero_factor_damps_with_pi_one():
    """An all-zero output factor: pi falls back to 1, both inverses are the plain damped inverses."""
    s, lo, hi = gram(65, 64, 7)
    z = K.zero_factor(5)
    case = Case([s], [z], spectra={id(s): (lo, hi), id(z): (0.0, 0.0)})
    for path in (1, 2):
        r = run(case, path)
        assert r["damp"][0, 0] == r["damp"][0, 1] == np.float32(np.sqrt(np.float64(np.float32(0.01))))
        check(case, r, "zero G path %d" % path)


# ------------------------------------------------------------------------------------------------ job mixes
def _mixes():
    from test_gpu_cnn import SIZES as CNN_SIZES
    from test_gpu_mlp import LARGE, SMALL
    out = {"atari_c3_32": (lambda: atari_case(32), "resident"), "atari_c3_64": (lambda: atari_case(64), "resident"),
           "atari_c3_96": (lambda: atari_case(96), "chain"),
           "mlp_small": (lambda: mlp_case(**SMALL), "resident"), "mlp_large": (lambda: mlp_case(**LARGE), "resident"),
           "six_equal_blocks": (lambda: blocks_case([63] * 6, [64] * 6), "resident"),
           "large_a_1x1_g": (lambda: blocks_case([1024], [1], shared=False), "resident")}
    for name, (shape, want) in CNN_SIZES.items():
        out["cnn_" + name] = (functools.partial(cnn_case, **shape), "chain" if want == "fp64 chain" else "resident")
    return out


MIXES = _mixes()


@pytest.mark.parametrize("mix", list(MIXES))
def test_job_mixes(mix):
    """The job sets of the Atari learner (conv3 = 32, 64: resident; 96: chain), the fully connected and convolutional test
    geometries, six equal blocks and one large input factor with 1 x 1 output factors, through all three paths."""
    make, want = MIXES[mix]
    both_paths(make(), mix, want)


def test_shared_head_factor_with_two_dampings():
    """The two heads read one input factor; output factors of different scale give them different pi and so different
    dampings: two different inverses of one sum, each the correct one."""
    case = blocks_case([64, 32, 32], [32, 5, 1])
    case.g[2] = case.g[2] * 64.0
    for path in (1, 2):
        r = run(case, path)
        assert r["damp"][1, 0] != r["damp"][2, 0]
        assert not np.array_equal(r["inv_a"][1], r["inv_a"][2])
        check(case, r, "shared heads path %d" % path)
    both_paths(case, "shared heads", "resident")


def test_where_the_resident_kernel_stops_fitting():
    """The largest single-block input factor (whole 64-row tiles) the resident kernel accepts on this device, and one row
    more: on both sides the learners' refresh is bit-identical to the path it takes, and both paths meet the bounds."""
    def fits(tiles):
        n = 64 * tiles
        r = ops.kfac_invert([np.eye(n, dtype=np.float32)], [np.ones((1, 1), np.float32)], path=1)
        return r is not None

    lo, hi = 1, 96
    assert fits(lo) and not fits(hi)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if fits(mid) else (lo, mid)
    n_fit = 64 * lo
    name = torch.cuda.get_device_name()
    record("resident_limit", device=name, largest=n_fit)
    for n, want in ((n_fit, "resident"), (n_fit + 1, "chain")):
        s, a_lo, a_hi = gram(n, 64, n)
        g = K.spectrum_factor([1.0], 0)
        case = Case([s], [g], spectra={id(s): (a_lo, a_hi)})
        both_paths(case, "n=%d" % n, want)


# ------------------------------------------------------------------------------------------------ conditioning
@pytest.mark.parametrize("debias", [1.0, DEBIAS3], ids=["debias1", "debias3"])
@pytest.mark.parametrize("rows", [64, 2048], ids=["rank64", "full_rank"])
@pytest.mark.parametrize("n", [513, 1569])
@pytest.mark.parametrize("kappa", [1e1, 1e3, 1e4, 1e5, 1e6, 1e7])
def test_conditioning(kappa, n, rows, debias):
    """One block whose damped input factor has condition number kappa (the damping chosen through the fp64 pi formula):
    the chain at every kappa, the resident kernel up to RESIDENT_KAPPA_LIMIT (beyond it its error is recorded)."""
    s, lo, hi = gram(n, rows, 11)
    g = small_g(4, 1)
    damping = K.damping_for_kappa(s, g, kappa, debias, lam_min=lo, lam_max=hi)
    case = Case([s], [g], damping=damping, debias=debias, spectra={id(s): (lo, hi)})
    tag = "kappa=%.0e n=%d rows=%d debias=%.3f" % (kappa, n, rows, debias)
    _, a_hi = case.extremes(s)
    r2 = run(case, 2)
    d = float(r2["damp"][0, 0])
    got_kappa = (float(np.float32(debias)) * a_hi + d) / (float(np.float32(debias)) * lo + d)
    assert abs(got_kappa / kappa - 1) < 1e-3, (tag, got_kappa)
    check(case, r2, tag + " chain")
    r1 = run(case, 1)
    worst = check(case, r1, tag + " resident")
    record("conditioning", case=tag, resident_worst_ratio=worst)


# ------------------------------------------------------------------------------------------------ a trained network
def test_factors_of_a_trained_network():
    """ACKTR with invert_every = 1 on the contextual bandit of test_gpu_mlp (reward 1 when the action is the argmax of the
    first four context features): every 50 updates the engine's stored inverses are checked against the fp64 reference of
    its own running sums, dampings and debias factor, and the condition number of every damped factor is recorded."""
    cfg = eng.MLPEngineConfig(num_envs=64, num_steps=1, obs_dim=8, hidden_sizes=(64, 64), num_actions=4, num_cold_updates=5,
                              invert_every=1, seed=1)
    e = eng.MLPEngine(cfg)
    from test_gpu_mlp import params_for
    e.set_params(params_for(cfg, 1))
    rng = np.random.default_rng(2)
    kappas, hits = [], 0
    for u in range(1, 401):
        ctx = rng.uniform(-1, 1, (64, 1, 8)).astype(np.float32)
        acts = e.act(torch.from_numpy(ctx[:, 0]).cuda()).cpu().numpy().astype(np.uint8)
        rew = (acts == ctx[:, 0, :4].argmax(1)).astype(np.float32)
        hits += int(rew.sum()) if u > 300 else 0
        e.update(dict(observations=ctx, bootstrap_observations=ctx[:, 0], actions=acts.reshape(64, 1),
                      rewards=rew.reshape(64, 1), terminals=np.ones((64, 1), bool)), fetch=False)
        if u % 50:
            continue
        torch.cuda.synchronize()
        assert _lib.load().acx_debug_tc_error() == 0
        debias = float(e.buffer("sched", torch.float32)[5])
        damp = e.buffer("dampings", torch.float32).cpu().numpy()
        a_sums, g_sums, inv_a, inv_g = [], [], [], []
        for i, layer in enumerate(e.layers):
            fac = "heads" if layer in ("fc_policy", "fc_baseline") else layer
            if fac not in ("heads",) or layer == "fc_policy":
                a_sums.append(e.factor("sums", "A", fac).cpu().double())
            g_sums.append(e.factor("sums", "G", layer).cpu().double())
            inv_a.append(e.factor("inv", "A", layer).cpu().numpy())
            inv_g.append(e.factor("inv", "G", layer).cpu().numpy())
        case = Case(a_sums, g_sums, shared=True, damping=cfg.damping, debias=debias)
        for i, layer in enumerate(e.layers):
            for which, s, d in (("A", case.a_of(i), float(damp[2 * i])), ("G", case.g[i], float(damp[2 * i + 1]))):
                lo, hi = case.extremes(s)
                kappas.append((u, which + "/" + layer, (debias * hi + d) / (debias * lo + d)))
                record("trained_kappa", update=u, factor=which + "/" + layer, kappa=kappas[-1][2])
        stored = dict(inv_a=inv_a, inv_g=inv_g, damp=damp.reshape(-1, 2), path=0)
        check(case, stored, "trained u=%d" % u, resident_kappa_limit=float("inf"))
    record("trained_kappa_max", kappa=max(k for _, _, k in kappas), accuracy_last_100=hits / (100 * 64))
    assert max(k for _, _, k in kappas) * 10 <= RESIDENT_KAPPA_LIMIT
