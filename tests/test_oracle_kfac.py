"""G5 on the CPU: self-checks that pin the K-FAC oracle (oracle/kfac.py, oracle/learner.py).

tensorflow/kfac is not available (oracle/kfac.py header), so the arithmetic is pinned three ways:
  * the schedule against tests/golden/schedule.npz, which make_golden.py records by running the REFERENCE'S OWN class
    ColdStartPeriodicInvUpdateKfacOpt.apply_gradients (kfac_utils.py:38-53) on a recording KfacOptimizer skeleton;
  * exact identities of the published algorithm: the Kronecker identity vec(A^-1 V G^-1) = (G (x) A)^-1 vec(V), the
    definitions of the factors as averaged outer products with the homogeneous coordinate, pi-damping, zero-debias,
    KL clip, momentum;
  * hypothesis-driven rollout shapes, terminal patterns and Fisher samples through the whole oracle `compute`;
  * the unpinned choices of SURVEY A.7 (U1 num_locations, U3 cov_init / zero_debias / inv_init) as explicit parameters.
It also holds the evidence for the ReLU-branch synchronisation the GPU parity tests use (DESIGN.md section 2).
"""
import math
import os

import numpy as np
import pytest
import torch
from hypothesis import HealthCheck, given, settings
from hypothesis import strategies as st

import synth
from oracle import kfac as K
from oracle import learner as OL
from oracle import network as onet
from oracle import returns as R


# ------------------------------------------------------------------------------------------------ schedule (a17)
def _golden_schedule(golden_dir):
    return np.load(os.path.join(golden_dir, "schedule.npz"))


@pytest.mark.parametrize("tag", ["reference", "short", "odd"])
def test_schedule_events_match_the_reference_class(golden_dir, tag):
    g = _golden_schedule(golden_dir)
    num_cold, every = (int(v) for v in g[tag + "_config"])
    for gs_before, cold, cov, inv, apply_, gs_after in g[tag]:
        plan = K.schedule_events(int(gs_before), num_cold, every)
        assert (int(plan["cold"]), int(plan["cov"]), int(plan["inv"]), int(plan["kfac_apply"]), plan["gs_after"]) == (
            cold, cov, inv, apply_, gs_after), (tag, gs_before)


def test_reference_schedule_landmarks(golden_dir):
    """What the reference class does with its own constants (30 cold updates, invert every 10; SURVEY 3.4 / D.2)."""
    rows = _golden_schedule(golden_dir)["reference"]
    cold_rows = rows[rows[:, 1] == 1]
    assert len(cold_rows) == 15 and list(cold_rows[:, 0]) == list(range(0, 30, 2))      # cold steps count twice
    assert (rows[:, 4] == 1).all()                                                        # K-FAC apply always runs
    first_cov = rows[rows[:, 2] == 1][0]
    assert first_cov[0] == 30
    inv_rows = rows[rows[:, 3] == 1]
    assert list(inv_rows[:, 0]) == [40, 50, 60, 70][: len(inv_rows)]                      # first refresh starts at gs 40


def test_oracle_learner_follows_the_golden_schedule(golden_dir):
    g = _golden_schedule(golden_dir)
    num_cold, every = (int(v) for v in g["short_config"])
    cfg = K.KfacConfig(num_cold_updates=num_cold, invert_every=every)
    params = onet.perturbed_params(4, 32, 0)
    o = OL.OracleLearner(params, 4, 32, acktr=True, cfg=cfg)
    batch = synth.rollout(3, 1, 2, 4, obs_kind="sparse")
    y_hat, eps = synth.fisher_samples(4, 2)
    ncov = 0
    for gs_before, cold, cov, inv, _, gs_after in g["short"][:8]:
        assert o.global_step == gs_before
        before = {k: v.clone() for k, v in o.kfac.inv_a.items()}
        info = o.update(batch, y_hat, eps)
        ncov += int(cov)
        assert o.global_step == gs_after and o.kfac.num_cov_updates == ncov
        assert bool(info.get("inverted", False)) == bool(inv)
        changed = any(not torch.equal(before[k], o.kfac.inv_a[k]) for k in before)
        assert changed == bool(inv)
        assert ("grad_norm" in info) == bool(cold)


# ------------------------------------------------------------------------------------------------ identities
def _state_after_updates(num_updates, e=1, t=3, c3=32, cfg=None, seed=0):
    cfg = cfg or K.KfacConfig(num_cold_updates=0, invert_every=1)
    o = OL.OracleLearner(onet.perturbed_params(4, c3, seed), 4, c3, acktr=True, cfg=cfg)
    info = None
    for u in range(num_updates):
        batch = synth.rollout(20 + u, e, t, 4, obs_kind="sparse")
        y_hat, eps = synth.fisher_samples(30 + u, e * t)
        info = o.update(batch, y_hat, eps)
    return o, info


def test_kronecker_identity_of_the_preconditioner():
    """U = A^-1 V G^-1  <=>  (G (x) A) vec(U) = vec(V) with column-major vec, for the DAMPED factors the oracle inverts
    (SURVEY A.5 'Precondition'); checked on the two head blocks (513 x 4 and 513 x 1), where the Kronecker matrix is
    small enough to form."""
    o, info = _state_after_updates(2)
    for layer in ("fc_policy", "fc_baseline"):
        damp_a, damp_g = o.kfac.dampings(layer)
        a = o.kfac.cov_a("heads") + damp_a * torch.eye(513, dtype=torch.float64)
        g = o.kfac.cov_g(layer)
        g = g + damp_g * torch.eye(g.shape[0], dtype=torch.float64)
        v = info["grads"][layer]
        u = info["precon"][layer] * o.cfg.locations(layer)
        kron = torch.kron(g.contiguous(), a.contiguous())                      # (G (x) A), acts on column-major vec
        lhs = kron @ u.T.reshape(-1)                                         # vec(U) column-major = U^T flattened row-major
        assert float((lhs - v.T.reshape(-1)).norm() / v.norm()) < 1e-9
        # and the stored inverses are the inverses of exactly those damped matrices
        assert float((o.kfac.inv_a[layer] @ a - torch.eye(513, dtype=torch.float64)).abs().max()) < 1e-8
        assert float((o.kfac.inv_g[layer] @ g - torch.eye(g.shape[0], dtype=torch.float64)).abs().max()) < 1e-8


def test_pi_damping_definition():
    o, _ = _state_after_updates(1)
    for layer in onet.LAYERS:
        damp_a, damp_g = o.kfac.dampings(layer)
        lam = o.cfg.damping / o.cfg.locations(layer)
        assert math.isclose(damp_a * damp_g, lam, rel_tol=1e-12)                # pi cancels in the product
        a, g = o.kfac.cov_a(K.A_FACTOR_OF[layer]), o.kfac.cov_g(layer)
        pi = math.sqrt((float(torch.trace(a)) / a.shape[0]) / (float(torch.trace(g)) / g.shape[0]))
        assert math.isclose(damp_a / damp_g, pi * pi, rel_tol=1e-10)


@pytest.mark.parametrize("mode", ["true", "input_div_stride"])
def test_num_locations_modes(mode):
    cfg = K.KfacConfig(num_locations_mode=mode)
    want = {"true": (400, 81, 49), "input_div_stride": (441, 100, 81)}[mode]
    assert tuple(cfg.locations(n) for n in ("conv1", "conv2", "conv3")) == want
    assert all(cfg.locations(n) == 1 for n in ("fc4", "fc_policy", "fc_baseline"))


def test_zero_debias_makes_the_first_average_exact():
    """S_1 = 0.01 C_1 and the debiased value S_1 / (1 - 0.99) is C_1; after n updates with a constant contribution the
    debiased value is that contribution (SURVEY A.5 'EMA')."""
    params = onet.to_torch(onet.perturbed_params(4, 32, 0))
    st_ = K.KfacState(params, K.KfacConfig())
    rng = np.random.default_rng(0)
    new_a = {k: torch.as_tensor(rng.standard_normal(v.shape)) for k, v in st_.sum_a.items()}
    new_g = {k: torch.as_tensor(rng.standard_normal(v.shape)) for k, v in st_.sum_g.items()}
    for n in range(1, 4):
        st_.update_covs(new_a, new_g)
        assert float((st_.cov_a("conv2") - new_a["conv2"]).abs().max()) < 1e-12
        assert float((st_.cov_g("fc4") - new_g["fc4"]).abs().max()) < 1e-12
        assert float((st_.sum_a["conv2"] - (1 - 0.99 ** n) * new_a["conv2"]).abs().max()) < 1e-12


def test_cov_init_and_debias_knobs():
    """U3: identity-initialised covariances without zero-debias (older tf.contrib.kfac)."""
    params = onet.to_torch(onet.perturbed_params(4, 32, 0))
    st_ = K.KfacState(params, K.KfacConfig(cov_init="identity", zero_debias=False))
    assert torch.equal(st_.sum_a["conv1"], torch.eye(257, dtype=torch.float64))
    c = {k: torch.full(v.shape, 2.0, dtype=torch.float64) for k, v in st_.sum_a.items()}
    g = {k: torch.full(v.shape, 3.0, dtype=torch.float64) for k, v in st_.sum_g.items()}
    st_.update_covs(c, g)
    want = 0.99 * torch.eye(257, dtype=torch.float64) + 0.01 * 2.0
    assert float((st_.cov_a("conv1") - want).abs().max()) < 1e-15       # no debias factor applied
    st2 = K.KfacState(params, K.KfacConfig(zero_debias=False))
    st2.update_covs(c, g)
    assert float((st2.cov_a("conv1") - 0.02).abs().max()) < 1e-15


def test_inv_init_identity_takes_kfac_steps_from_the_start():
    """U3: with identity-initialised inverses the always-run K-FAC apply (kfac_utils.py:52-53) is a real step before the
    first refresh (U = V / T~, KL-clipped); with kfac 0.1's zero initialisation it is an exact no-op."""
    batch = synth.rollout(3, 1, 2, 4, obs_kind="sparse")
    y_hat, eps = synth.fisher_samples(4, 2)
    moved = {}
    for init in ("zero", "identity"):
        cfg = K.KfacConfig(num_cold_updates=0, invert_every=100, inv_init=init)
        o = OL.OracleLearner(onet.perturbed_params(4, 32, 0), 4, 32, acktr=True, cfg=cfg)
        before = onet.join_vmat("conv2", o.params).clone()
        info = o.update(batch, y_hat, eps)
        moved[init] = float((onet.join_vmat("conv2", o.params) - before).abs().max())
        if init == "identity":
            for layer in onet.LAYERS:
                assert torch.allclose(info["precon"][layer], info["grads"][layer] / cfg.locations(layer), rtol=0, atol=1e-15)
            s = sum(float((info["grads"][l] * info["precon"][l]).sum()) for l in onet.LAYERS)
            assert math.isclose(info["fisher_norm"], s, rel_tol=1e-12)
            assert math.isclose(info["clip_coeff"], min(1.0, math.sqrt(1e-4 / (info["lr"] ** 2 * s))), rel_tol=1e-12)
    assert moved["zero"] == 0.0 and moved["identity"] > 0.0


def test_kl_clip_and_momentum_recurrence():
    o, info = _state_after_updates(2)
    lr, c, s = info["lr"], info["clip_coeff"], info["fisher_norm"]
    assert 0.0 < c <= 1.0
    assert lr * lr * c * c * s <= 1e-4 * (1 + 1e-9)                        # the clipped step satisfies the KL constraint
    # one more update: v <- 0.9 v + c U ; theta <- theta - lr v
    v_before = {k: v.clone() for k, v in o.kfac.velocity.items()}
    p_before = {l: onet.join_vmat(l, o.params).clone() for l in onet.LAYERS}
    batch = synth.rollout(50, 1, 3, 4, obs_kind="sparse")
    y_hat, eps = synth.fisher_samples(51, 3)
    info = o.update(batch, y_hat, eps)
    for l in onet.LAYERS:
        v = 0.9 * v_before[l] + info["clip_coeff"] * info["precon"][l]
        assert torch.allclose(o.kfac.velocity[l], v, rtol=0, atol=1e-15)
        assert torch.allclose(onet.join_vmat(l, o.params), p_before[l] - info["lr"] * v, rtol=0, atol=1e-14)


# ------------------------------------------------------------------------------------------------ hypothesis
@settings(max_examples=12, deadline=None, suppress_health_check=[HealthCheck.too_slow])
@given(e=st.integers(1, 3), t=st.integers(1, 4), seed=st.integers(0, 2 ** 16), c3=st.sampled_from([32, 64]),
       term=st.sampled_from(["random", "none", "all", "first", "last"]))
def test_factors_are_averaged_outer_products(e, t, seed, c3, term):
    """Whatever the rollout shape and terminal pattern: every factor the oracle's `compute` returns is the definition of
    SURVEY A.5 evaluated independently (conv patches through torch's own unfold, reordered), symmetric, with the
    homogeneous corner 1 and border = mean input; the head output factors follow from the injected Fisher samples; the
    targets equal the reference's matrix form (objectives.py:178-214)."""
    n = e * t
    batch = synth.rollout(seed, e, t, 4, obs_kind="sparse" if seed % 2 else "uniform")
    if term != "random":
        tm = np.zeros((e, t), bool)
        if term == "all":
            tm[:] = True
        elif term == "first":
            tm[:, 0] = True
        elif term == "last":
            tm[:, -1] = True
        batch["terminals"] = tm
    params = onet.perturbed_params(4, c3, seed % 5)
    o = OL.OracleLearner(params, 4, c3, acktr=True)
    logits_seed = onet.forward(o.params, batch["observations"].reshape((n,) + batch["observations"].shape[2:]))["logits"]
    y_hat, eps = synth.fisher_samples(seed + 1, n, logits=logits_seed.numpy())
    info = o.compute(batch, y_hat, eps, need_fisher=True)
    # targets: recursion == the reference's matrix form, whatever the terminal pattern (the reference builds its discount
    # factors through float32 products, objectives.py:188-196,209-211: ~1e-7 relative)
    want = R.targets_matrix_form(batch["rewards"], batch["terminals"], info["bootstrap_values"].numpy(), o.gamma, np.float64)
    np.testing.assert_allclose(info["targets"].numpy().reshape(e, t), want, rtol=0, atol=2e-6)
    # conv input factors from torch's own unfold ((cin, kh, kw) feature order -> (kh, kw, cin))
    x = torch.as_tensor(batch["observations"].reshape(n, 84, 84, 4)).double() / 255.0
    acts = {"conv1": x, "conv2": info["fwd"]["conv1"]["act"].reshape(n, 20, 20, 32),
            "conv3": info["fwd"]["conv2"]["act"].reshape(n, 9, 9, 64)}
    for name, inp in acts.items():
        k, s, cin, _, hw = onet.CONV_GEOM[name]
        cols = torch.nn.functional.unfold(inp.permute(0, 3, 1, 2), k, stride=s)            # [n, cin*k*k, hw*hw]
        cols = cols.reshape(n, cin, k, k, hw * hw).permute(0, 4, 2, 3, 1).reshape(n * hw * hw, k * k * cin)
        ph = torch.cat([cols, torch.ones(cols.shape[0], 1, dtype=torch.float64)], 1)
        a = ph.T @ ph / cols.shape[0]
        got = info["new_a"][name]
        assert float((got - a).abs().max()) <= 1e-12 * max(1.0, float(a.abs().max()))
        assert torch.equal(got, got.T) and float(got[-1, -1]) == 1.0
        assert torch.allclose(got[:-1, -1], cols.mean(0), rtol=0, atol=1e-13)
    flat = info["fwd"]["conv3"]["act"].reshape(n, 49 * c3)
    assert info["new_a"]["fc4"].shape == (49 * c3 + 1,) * 2
    assert torch.allclose(info["new_a"]["fc4"][:-1, :-1], flat.T @ flat / n, rtol=0, atol=1e-12)
    # output factors of the heads from the injected samples: d/dz = p - onehot(y), d/dV = -eps
    p = torch.softmax(info["fwd"]["logits"], -1)
    gz = p - torch.nn.functional.one_hot(torch.as_tensor(y_hat).long(), 4).double()
    assert torch.allclose(info["new_g"]["fc_policy"], gz.T @ gz / n, rtol=0, atol=1e-14)
    assert abs(float(info["new_g"]["fc_baseline"]) - float(np.mean(eps.astype(np.float64) ** 2))) < 1e-12
    for g in info["new_g"].values():
        assert torch.equal(g, g.T) and float(torch.linalg.eigvalsh(g).min()) > -1e-12


@settings(max_examples=40, deadline=None)
@given(rows=st.integers(1, 30), d=st.integers(1, 9), seed=st.integers(0, 2 ** 16))
def test_input_and_output_factor_properties(rows, d, seed):
    x = torch.as_tensor(np.random.default_rng(seed).standard_normal((rows, d)))
    a, g = K.input_factor(x), K.output_factor(x)
    outer = sum(torch.outer(torch.cat([r, torch.ones(1, dtype=r.dtype)]), torch.cat([r, torch.ones(1, dtype=r.dtype)])) for r in x) / rows
    assert torch.allclose(a, outer, rtol=0, atol=1e-12) and torch.equal(a, a.T)
    assert torch.allclose(a[:-1, :-1], g, rtol=0, atol=1e-12)
    assert float(torch.linalg.eigvalsh(a).min()) > -1e-10


# ------------------------------------------------------------------------------------------------ ReLU branches
def test_one_relu_unit_within_rounding_of_zero_moves_a_conv_gradient_by_1e_4():
    """Evidence for the mask synchronisation of the GPU parity tests (tests/learner_checks.py, DESIGN.md section 2).

    The same oracle evaluated in float32 (the reference's arithmetic class) against float64, both with their OWN ReLU
    branches, at BASELINE.json's size (32 x 20, iid-uniform observations = the adversarial input): the arithmetic error
    of every gradient is ~3e-7, but as soon as ONE of the ~12 M ReLU units has a pre-activation so close to zero that the
    two precisions disagree on its sign, the conv gradients upstream of it differ by 1e-5 .. 1e-3 of their norm - a
    thousand times the arithmetic error - because the true-loss gradient is a cancelling sum over 51 840 .. 256 000
    rows.  With the float64 side differentiating at the float32 side's masks the difference is back at ~3e-7.  Any
    finite-precision implementation (the reference's fp32 TensorFlow kernels included) sits on one side or the other of
    such units; the engine's 2^-17 products put 3 - 15 units there (profiles/r1_precision.md)."""
    params = onet.perturbed_params(4, 32, 1)
    found = None
    clean_checked = False
    for seed in range(7, 19):
        batch = synth.rollout(seed, 32, 20, 4, obs_kind="uniform")
        o64 = OL.OracleLearner(params, 4, 32, acktr=False, dtype=torch.float64)
        o32 = OL.OracleLearner(params, 4, 32, acktr=False, dtype=torch.float32)
        i64 = o64.compute(batch, need_fisher=False)
        i32 = o32.compute(batch, need_fisher=False)
        masks32 = {n: i32["fwd"][n]["pre"] > 0 for n in ("conv1", "conv2", "conv3", "fc4")}
        flips, worst = 0, 0.0
        for n, m in masks32.items():
            pre = i64["fwd"][n]["pre"]
            d = m != (pre > 0)
            if int(d.sum()):
                flips += int(d.sum())
                worst = max(worst, float(pre[d].abs().max()) / float(pre.pow(2).mean().sqrt()))

        def rel(a, b):
            return float((a.double() - b).norm() / b.norm())
        own = {l: rel(i32["grads"][l], i64["grads"][l]) for l in onet.LAYERS}
        if flips == 0:
            assert max(own.values()) < 5e-6, (seed, own)           # pure arithmetic error
            clean_checked = True
            continue
        synced = o64.compute(batch, need_fisher=False, masks=masks32)
        sync = {l: rel(i32["grads"][l], synced["grads"][l]) for l in onet.LAYERS}
        found = (seed, flips, worst, own, sync)
        if clean_checked:
            break
    assert found is not None, "no near-zero ReLU unit in 12 seeded batches"
    seed, flips, worst, own, sync = found
    assert worst < 1e-5                                            # the disagreeing units ARE within rounding of zero
    assert max(sync.values()) < 5e-6, sync                         # arithmetic error once the branches agree
    assert own["conv1"] > 20 * sync["conv1"] and own["conv1"] > 1e-5, (flips, own, sync)


# ------------------------------------------------------------------------------------------------ inverse-refresh reference
def test_kfac_state_inverses_are_the_shared_reference():
    """KfacState.dampings / update_inverses go through pi_dampings / damped_inverse, and give exactly what the inline formulas
    gave before: pi from the traces of the debiased factors, (S debias + damp I)^-1 of the (symmetric) running sums."""
    o, _ = _state_after_updates(2)
    st_ = o.kfac
    debias = st_._debias()
    assert debias != 1.0
    st_.update_inverses()
    for layer in onet.LAYERS:
        a, g = st_.cov_a(K.A_FACTOR_OF[layer]), st_.cov_g(layer)
        lam = st_.cfg.damping / st_.cfg.locations(layer)
        tr_a, tr_g = float(torch.trace(a)) / a.shape[0], float(torch.trace(g)) / g.shape[0]
        pi = math.sqrt(tr_a / tr_g)
        assert st_.dampings(layer) == (pi * math.sqrt(lam), math.sqrt(lam) / pi)
        want_a = torch.linalg.inv(a + pi * math.sqrt(lam) * torch.eye(a.shape[0], dtype=torch.float64))
        want_g = torch.linalg.inv(g + math.sqrt(lam) / pi * torch.eye(g.shape[0], dtype=torch.float64))
        assert torch.equal(st_.inv_a[layer], want_a) and torch.equal(st_.inv_g[layer], want_g)


def test_pi_dampings_edge_cases():
    a, g = torch.eye(3, dtype=torch.float64) * 4.0, torch.eye(2, dtype=torch.float64)
    assert K.pi_dampings(a, g, 0.01) == pytest.approx((0.2, 0.05), rel=1e-15)
    assert K.pi_dampings(a * 7.0, g * 7.0, 0.01) == K.pi_dampings(a, g, 0.01)     # a common scale cancels
    assert K.pi_dampings(a, K.zero_factor(2), 0.01) == (0.1, 0.1)                  # zero trace: pi = 1
    assert K.pi_dampings(K.zero_factor(3), g, 0.25) == (0.5, 0.5)


def test_damped_inverse_symmetrises():
    s, _, _ = K.gram_factor(40, 16, 3)
    a = K.with_antisymmetric_ulp(s)
    assert not torch.equal(a, a.T) and torch.equal(a.float().double(), a)
    assert float((a - s).abs().max()) <= float(s.abs().max()) * 2.0 ** -23
    assert float((0.5 * (a + a.T) - s).abs().max()) <= float(s.abs().max()) * 2.0 ** -24
    inv = K.damped_inverse(a, 2.0, 0.5)
    m = 2.0 * 0.5 * (a + a.T) + 0.5 * torch.eye(40, dtype=torch.float64)
    assert torch.equal(inv, inv.T) or float((inv - inv.T).abs().max()) < 1e-14
    assert float((inv @ m - torch.eye(40, dtype=torch.float64)).abs().max()) < 1e-12


@pytest.mark.parametrize("n, rows", [(1, 64), (33, 64), (513, 64), (65, 128)])
def test_gram_factor_is_exact_with_the_stated_spectrum(n, rows):
    s, lo, hi = K.gram_factor(n, rows, n)
    assert torch.equal(s, s.T) and torch.equal(s, s.float().double())
    assert float(s[-1, -1]) == 1.0                                              # homogeneous corner
    lam = torch.linalg.eigvalsh(s)
    assert abs(float(lam[-1]) - hi) <= 1e-12 * hi
    assert abs(float(lam[0]) - lo) <= 1e-12 * hi
    assert int((lam > 1e-10 * hi).sum()) == min(n, rows)


def test_spectrum_factor_has_the_prescribed_spectrum():
    want = np.geomspace(1.0, 1e-3, 50)
    s = K.spectrum_factor(want, 4)
    assert torch.equal(s, s.T) and torch.equal(s, s.float().double())
    got = torch.linalg.eigvalsh(s).numpy()[::-1]
    assert np.abs(got - want).max() <= 1e-6


@pytest.mark.parametrize("kappa", [1e1, 1e4, 1e7])
@pytest.mark.parametrize("n, rows", [(513, 64), (513, 2048), (1569, 64), (1569, 2048)])
@pytest.mark.parametrize("debias", [1.0, 1.0 / (1.0 - 0.99 ** 3)])
def test_damping_for_kappa_reaches_the_target(kappa, n, rows, debias):
    """The damping the conditioning tests use puts the damped input factor at the target condition number, through the fp64
    pi formula and the fp32 lambda the learners store (damping / T~ in fp32)."""
    s, lo, hi = K.gram_factor(n, rows, 11)
    g = K.spectrum_factor([1.0, 0.5, 0.25, 0.125], 1)
    damping = K.damping_for_kappa(s, g, kappa, debias, tnorm=4, lam_min=lo, lam_max=hi)
    lam = float(np.float32(np.float32(damping) / np.float32(4)))
    d = float(np.float32(K.pi_dampings(s, g, lam)[0]))
    assert abs((debias * hi + d) / (debias * lo + d) / kappa - 1) < 1e-5
    if n == 513:   # the spectrum the shortcut used, against the full eigendecomposition
        lam_m = torch.linalg.eigvalsh(debias * s + d * torch.eye(n, dtype=torch.float64))
        assert abs(float(lam_m[-1] / lam_m[0]) / kappa - 1) < 1e-4
