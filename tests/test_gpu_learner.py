"""G4/G5 on the GPU: the learner engine (libacx through the C ABI) against the fp64 oracle on identical seeded
inputs, weights and injected Fisher samples.

Tolerances (north_star): factors and preconditioned updates <= 1e-3; here every compared quantity must meet
1e-3 in the norm-relative sense ||X-Y||_F / ||Y||_F, and the default (parity-grade) precision is additionally
held to 2e-4 so that regressions show up long before the contract is at risk.  uint8/int quantities (actions)
are compared exactly."""
import numpy as np
import pytest
import torch

import learner_checks as LC
import synth
from oracle import network as onet

pytestmark = pytest.mark.gpu

TOL = 1e-3          # the contract
TOL_DEFAULT = 2e-4  # what precision 0 is held to


def _engine_mod():
    from actorcritic_b200 import engine
    return engine


def _compute(precision, e_count, t_count, c3, obs_kind, mode="true", **kw):
    eng = _engine_mod()
    cfg = eng.EngineConfig(num_envs=e_count, num_steps=t_count, conv3_filters=c3, precision=precision,
                           num_locations_mode=mode, **kw)
    e, o = LC.make_pair(cfg, seed=1)
    e.set_state(30, 0, False)
    o.global_step = 30
    n = e_count * t_count
    batch = synth.rollout(7, e_count, t_count, 4, obs_kind=obs_kind)
    y_hat, eps = synth.fisher_samples(9, n)
    e.load_batch(batch["observations"], batch["bootstrap_observations"], batch["actions"], batch["rewards"],
                 batch["terminals"])
    e.phase1(torch.from_numpy(y_hat).cuda(), torch.from_numpy(eps).cuda())
    torch.cuda.synchronize()
    # The oracle takes its ReLU derivatives at the engine's masks, and the units where that is not the oracle's own
    # branch must have an fp64 pre-activation within rounding of zero (<= 1e-4 of the layer's rms, at most 1e-3 of the
    # units): a unit that close to zero takes either branch in any finite-precision implementation, and because the
    # true-loss gradients are cancelling sums a single such unit moves a conv gradient by 1e-3 .. 1e-2 of its norm.
    masks = LC.engine_relu_masks(e)
    info = o.compute(batch, y_hat, eps, need_fisher=True, masks=masks)
    for name, (count, frac, worst) in LC.mask_disagreement(masks, info["fwd"]).items():
        assert worst <= 1e-4 and frac <= 1e-3, ("ReLU branch disagreement", name, count, frac, worst)
    return LC.compare_compute(e, info, cfg, True)


@pytest.mark.parametrize("e_count,t_count,c3", [(4, 5, 32), (3, 7, 64), (16, 5, 64)])
def test_phase1_matches_oracle(e_count, t_count, c3):
    errs = _compute(0, e_count, t_count, c3, "sparse")
    bad = {k: v for k, v in errs.items() if not v["rel"] <= TOL_DEFAULT}
    assert not bad, bad


@pytest.mark.parametrize("kw", [dict(conv_impl=1), dict(num_lanes=1), dict(conv_impl=1, num_lanes=1), dict(use_graphs=False)])
def test_phase1_alternative_routes_match_oracle(kw):
    """the im2col + GEMM + col2im route (conv_impl=1, also what an unsupported conv3 width uses) and the strictly serial
    schedule (num_lanes=1) must give the same results as the default implicit-GEMM / three-lane update."""
    errs = _compute(0, 4, 5, 32, "sparse", **kw)
    bad = {k: v for k, v in errs.items() if not v["rel"] <= TOL_DEFAULT}
    assert not bad, bad


def test_phase1_conv3_width_without_implicit_gemm_support():
    errs = _compute(0, 3, 4, 48, "sparse")
    bad = {k: v for k, v in errs.items() if not v["rel"] <= TOL_DEFAULT}
    assert not bad, bad


def test_phase1_uniform_random_observations():
    """iid-uniform observations are the adversarial input for parity: sums of ~256 terms of magnitude ~0.5 cancel to
    O(1) pre-activations, so more units sit within rounding of zero than for Atari-like frames.  With the ReLU branches
    synchronised (see _compute) every quantity meets the tight bound here too."""
    errs = _compute(0, 4, 5, 32, "uniform")
    bad = {k: v for k, v in errs.items() if not v["rel"] <= TOL_DEFAULT}
    assert not bad, bad


@pytest.mark.parametrize("kind", ["sparse", "uniform"])
def test_phase1_headline_size(kind):
    """BASELINE.json's size (32 environments x 20 steps, conv3 = 32): ~12 M ReLU units, of which a handful have an fp64
    pre-activation within 1e-5 rms of zero (measured: 3 - 15 units); everything is held to the parity bound."""
    errs = _compute(0, 32, 20, 32, kind)
    bad = {k: v for k, v in errs.items() if not v["rel"] <= TOL_DEFAULT}
    assert not bad, bad


def test_phase1_three_plane_preset_is_not_more_accurate():
    """preset 5 (3 planes, 6 plane pairs in forward / backward - the former default) against the default (2 planes, 3
    pairs): both sit on the fp32 accumulation floor."""
    a = _compute(0, 8, 5, 32, "sparse")
    b = _compute(5, 8, 5, 32, "sparse")
    assert all(v["rel"] <= TOL_DEFAULT for v in a.values()) and all(v["rel"] <= TOL_DEFAULT for v in b.values())


def test_phase1_fast_precision_within_contract():
    errs = _compute(1, 8, 5, 32, "sparse")
    bad = {k: v for k, v in errs.items() if not v["rel"] <= TOL}
    assert not bad, bad


def test_returns_bitexact_inside_engine():
    """targets inside the engine = the fp32 reverse recursion on the engine's own values (K-RET, bit-exact)."""
    eng = _engine_mod()
    from oracle import returns as R
    cfg = eng.EngineConfig(num_envs=6, num_steps=9)
    e, _ = LC.make_pair(cfg, seed=2)
    batch = synth.rollout(11, 6, 9, 4, terminal_prob=0.2)
    e.load_batch(batch["observations"], batch["bootstrap_observations"], batch["actions"], batch["rewards"], batch["terminals"])
    e.phase1()
    torch.cuda.synchronize()
    vals = e.values.cpu().numpy()
    want = R.targets_recursive(batch["rewards"], batch["terminals"], vals[54:], np.float32(0.99), np.float32)
    assert np.array_equal(e.buffer("targets").cpu().numpy().reshape(6, 9), want)
    assert np.array_equal(e.buffer("advantages").cpu().numpy().reshape(6, 9), want - vals[:54].reshape(6, 9))


def _check_schedule(records, tol):
    for rec in records:
        assert rec["gs_after"] == rec["oracle_gs_after"], rec
        assert rec["params_rel"] <= 1e-5, rec   # parameters after the update (fp32 storage: ~1e-7 floor)
        for key in ("precon", "inv_A", "inv_G", "sums_A", "sums_G"):
            for name, err in rec.get(key, {}).items():
                assert err <= tol, (rec["update"], key, name, err)
        for key in ("policy_loss", "baseline_loss", "mean_entropy", "clip_coeff", "fisher_norm", "grad_norm"):
            if key in rec and rec[key][0] is not None:
                got, want = rec[key]
                assert abs(got - want) <= tol * max(1.0, abs(want)), (rec["update"], key, got, want)


def test_acktr_schedule_matches_oracle_update_by_update():
    """ColdStartPeriodicInvUpdateKfacOpt as coded (kfac_utils.py:38-53): cold steps count twice, covariances
    start after the cold phase, inverses every `invert_every`; each update is compared from identical state."""
    eng = _engine_mod()
    cfg = eng.EngineConfig(num_envs=4, num_steps=5, conv3_filters=32, num_cold_updates=4, invert_every=2)
    records = LC.run_schedule(cfg, 9, obs_kind="sparse")
    assert [r["gs_after"] for r in records] == [2, 4, 5, 6, 7, 8, 9, 10, 11]
    assert any("inv_A" in r for r in records) and any("precon" in r for r in records)
    _check_schedule(records, TOL_DEFAULT)


def test_acktr_reference_schedule_constants():
    """The reference's own constants (30 cold, invert every 10): the first inverse refresh happens in the update
    that starts at gs 39 (gs reaches 40), nothing moves between gs 30 and 39."""
    eng = _engine_mod()
    cfg = eng.EngineConfig(num_envs=2, num_steps=3)
    e, o = LC.make_pair(cfg, seed=3)
    batch = synth.rollout(5, 2, 3, 4, obs_kind="sparse")
    gs_trace, valid_trace = [], []
    for _ in range(27):
        e.update(batch, fetch=False)
        gs_trace.append(e.global_step)
        valid_trace.append(e.get_state()["inverses_valid"])
    assert gs_trace[:15] == list(range(2, 32, 2))
    assert gs_trace[15:] == list(range(31, 43))
    assert valid_trace.index(True) == gs_trace.index(41)   # refresh when gs == 40 inside that update
    assert e.get_state()["num_cov_updates"] == 12


def test_acktr_input_div_stride_locations():
    eng = _engine_mod()
    cfg = eng.EngineConfig(num_envs=4, num_steps=5, num_cold_updates=2, invert_every=1, num_locations_mode="input_div_stride")
    _check_schedule(LC.run_schedule(cfg, 4, obs_kind="sparse"), TOL_DEFAULT)


def test_a2c_rmsprop_matches_oracle():
    eng = _engine_mod()
    cfg = eng.EngineConfig.a2c(num_envs=16, num_steps=5)
    records = LC.run_schedule(cfg, 3, obs_kind="sparse")
    assert [r["gs_after"] for r in records] == [1, 2, 3]
    _check_schedule(records, TOL_DEFAULT)
    for rec in records:
        assert rec["step_rel"] <= 1e-2      # the step itself (fp32 parameters: ~1e-8 * |theta| / |step| noise floor)


def test_act_indexing_exact_given_logits_and_noise():
    """sample_actions / select_max_actions (model.py:135-169): given the engine's own logits and the injected
    uniforms, the action indices are exact (inverse-CDF on softmax / argmax)."""
    eng = _engine_mod()
    cfg = eng.EngineConfig(num_envs=32, num_steps=4)
    e, o = LC.make_pair(cfg, seed=4)
    obs = torch.from_numpy(synth.rollout(21, 32, 1, 4, obs_kind="sparse")["bootstrap_observations"]).cuda()
    u = torch.from_numpy(np.random.default_rng(0).random(32).astype(np.float32)).cuda()
    actions, logits, values = e.act(obs, uniform=u, want_logits=True)
    greedy = e.act(obs, greedy=True)
    torch.cuda.synchronize()
    z = logits.cpu().numpy().astype(np.float32)
    assert np.array_equal(greedy.cpu().numpy(), z.argmax(1))
    fwd = onet.forward(o.params, obs.cpu().numpy())
    assert LC.rel_err(z, fwd["logits"].numpy()) <= TOL_DEFAULT
    assert LC.rel_err(values.cpu().numpy(), fwd["value"].numpy()) <= TOL_DEFAULT
    mx = z.max(1, keepdims=True)
    ex = np.exp(z - mx, dtype=np.float32)
    p = ex / ex.sum(1, keepdims=True, dtype=np.float32)
    want = np.minimum((np.cumsum(p, 1, dtype=np.float32) <= u.cpu().numpy()[:, None]).sum(1), 3)
    got = actions.cpu().numpy()
    # the device evaluates expf/cumsum in fp32 too; allow disagreement only where u sits within 1e-6 of a CDF edge
    edge = np.abs(np.cumsum(p, 1) - u.cpu().numpy()[:, None]).min(1) < 1e-6
    assert np.array_equal(got[~edge], want[~edge])
    assert ((got >= 0) & (got < 4)).all()


def test_philox_fisher_sampling_statistics():
    """Without injected samples the Fisher labels come from the on-device Philox stream: G_policy must be close to
    E[(p - e_y)(p - e_y)^T] = diag(p) - p p^T averaged over rows, and G_value close to 1."""
    eng = _engine_mod()
    cfg = eng.EngineConfig(num_envs=64, num_steps=20, seed=123)
    e, o = LC.make_pair(cfg, seed=5)
    e.set_state(30, 0, False)
    batch = synth.rollout(31, 64, 20, 4, obs_kind="sparse")
    e.load_batch(batch["observations"], batch["bootstrap_observations"], batch["actions"], batch["rewards"], batch["terminals"])
    e.phase1()
    torch.cuda.synchronize()
    p = torch.softmax(e.logits[:1280].double().cpu(), -1)
    want = (torch.diag_embed(p) - p[:, :, None] * p[:, None, :]).mean(0).numpy()
    got = e.factor("stats", "G", "fc_policy").cpu().numpy()
    assert np.abs(got - want).max() < 0.05
    assert abs(float(e.factor("stats", "G", "fc_baseline").cpu()) - 1.0) < 0.15


def test_async_scalar_fetch_matches_the_synchronous_one():
    eng = _engine_mod()
    cfg = eng.EngineConfig(num_envs=4, num_steps=5, conv3_filters=32, num_cold_updates=2, invert_every=1)
    e, _ = LC.make_pair(cfg, seed=2)
    batch = synth.rollout(11, 4, 5, 4, obs_kind="sparse")
    handles = [e.update(batch, fetch="async") for _ in range(3)]     # three updates enqueued before the first read
    sync = e.fetch_scalars()
    vals = [h.result() for h in handles]
    assert vals[-1] == sync
    assert all(np.isfinite(v["policy_loss"]) for v in vals) and vals[0] != vals[-1]


def test_state_dict_roundtrip_resumes_identically():
    eng = _engine_mod()
    cfg = eng.EngineConfig(num_envs=4, num_steps=5, num_cold_updates=2, invert_every=1)
    e1, _ = LC.make_pair(cfg, seed=6)
    batches = [synth.rollout(40 + i, 4, 5, 4, obs_kind="sparse") for i in range(5)]
    y, eps = synth.fisher_samples(1, 20)
    fl, fe = torch.from_numpy(y).cuda(), torch.from_numpy(eps).cuda()
    for b in batches[:3]:
        e1.update(b, fl, fe, fetch=False)
    sd = e1.state_dict()
    e2 = eng.Engine(cfg)
    e2.load_state_dict(sd)
    for b in batches[3:]:
        e1.update(b, fl, fe, fetch=False)
        e2.update(b, fl, fe, fetch=False)
    assert e1.global_step == e2.global_step
    assert np.array_equal(e1.get_params_flat(), e2.get_params_flat())


def test_data_parallel_equivalence_single_device():
    """G6 without NCCL: two shards of E/2 environments (world_size 2 engines), buckets summed by hand, must take
    the same step as one engine over all E environments."""
    eng = _engine_mod()
    kw = dict(num_steps=5, num_cold_updates=2, invert_every=1, lr_decay_steps=1000.0)
    full = eng.Engine(eng.EngineConfig(num_envs=8, **kw))
    halves = [eng.Engine(eng.EngineConfig(num_envs=4, world_size=2, **kw)) for _ in range(2)]
    params = onet.perturbed_params(4, 32, 7)
    for e in [full] + halves:
        e.set_params(params)
    for u in range(4):
        batch = synth.rollout(60 + u, 8, 5, 4, obs_kind="sparse")
        y, eps = synth.fisher_samples(70 + u, 40)
        full.update(batch, torch.from_numpy(y).cuda(), torch.from_numpy(eps).cuda(), fetch=False)
        for r, e in enumerate(halves):
            sl = slice(4 * r, 4 * r + 4)
            e.load_batch(*(batch[k][sl] for k in ("observations", "bootstrap_observations", "actions", "rewards", "terminals")))
            yy = torch.from_numpy(y.reshape(8, 5)[sl].reshape(-1).copy()).cuda()
            ee = torch.from_numpy(eps.reshape(8, 5)[sl].reshape(-1).copy()).cuda()
            e.phase1(yy, ee)
        total = halves[0].bucket + halves[1].bucket
        for e in halves:
            e.bucket.copy_(total)
            e.phase2()
        torch.cuda.synchronize()
        assert np.array_equal(halves[0].get_params_flat(), halves[1].get_params_flat())
        assert LC.rel_err(halves[0].get_params_flat(), full.get_params_flat()) <= 1e-6
    assert LC.rel_err(halves[0].buffer("factor_sums").cpu().numpy(), full.buffer("factor_sums").cpu().numpy()) <= 1e-5


# ------------------------------------------------------------------------------------------------ BASELINE sizes, end to end
def _refreshing_update(cfg, obs_kind):
    """Two updates from global_step 0 with no cold phase and invert_every = 1: the first accumulates covariances (the
    K-FAC apply is the exact no-op of zero-initialised inverses), the second runs the WHOLE path - forward, backward,
    Fisher backward, 11 factor statistics, EMA, pi-damping, all 12 inverses, preconditioning, KL clip, momentum, apply -
    and is compared quantity by quantity from identical state."""
    records = LC.run_schedule(cfg, 2, obs_kind=obs_kind)
    last = records[-1]
    assert [r["gs_after"] for r in records] == [1, 2]
    for key in ("sums_A", "sums_G", "inv_A", "inv_G", "precon", "clip_coeff", "fisher_norm"):
        assert key in last, key
    return records


@pytest.mark.parametrize("kind", ["sparse", "uniform"])
def test_full_update_with_inverse_refresh_headline_size(kind):
    """BASELINE.json configs[2] (32 envs x 20 steps, conv3 = 32): factor sums, all inverses (1569^2 for fc4), the
    preconditioned update of every block, the KL-clip coefficient, <V,U> and the parameter step against the fp64 oracle:
    contract 1e-3, default precision held to 2e-4."""
    eng = _engine_mod()
    cfg = eng.EngineConfig(num_envs=32, num_steps=20, conv3_filters=32, num_cold_updates=0, invert_every=1)
    records = _refreshing_update(cfg, kind)
    _check_schedule(records, TOL_DEFAULT)
    assert records[-1]["step_rel"] <= TOL_DEFAULT, records[-1]["step_rel"]
    assert 0.0 < records[-1]["clip_coeff"][0] <= 1.0


def test_full_update_with_inverse_refresh_conv3_64():
    """The class default conv3 = 64 (envs/atari/model.py:45): the 3137 x 3137 input factor of fc4 that north_star names
    is accumulated, inverted and used by the fc4 preconditioning GEMMs."""
    eng = _engine_mod()
    cfg = eng.EngineConfig(num_envs=8, num_steps=5, conv3_filters=64, num_cold_updates=0, invert_every=1)
    records = _refreshing_update(cfg, "sparse")
    assert records[-1]["inv_A"]["fc4"] <= TOL_DEFAULT
    _check_schedule(records, TOL_DEFAULT)
    assert records[-1]["step_rel"] <= TOL_DEFAULT, records[-1]["step_rel"]


@pytest.mark.parametrize("tag", ["reference", "short", "odd"])
def test_engine_schedule_matches_the_reference_class(golden_dir, tag):
    """a17 against tests/golden/schedule.npz (recorded from kfac_utils.ColdStartPeriodicInvUpdateKfacOpt itself): per
    update, whether the covariances are updated, whether the inverses are refreshed, and how global_step moves."""
    import ctypes
    import os
    eng = _engine_mod()
    g = np.load(os.path.join(golden_dir, "schedule.npz"))
    num_cold, every = (int(v) for v in g[tag + "_config"])
    cfg = eng.EngineConfig(num_envs=2, num_steps=3, num_cold_updates=num_cold, invert_every=every)
    e, _ = LC.make_pair(cfg, seed=3)
    batch = synth.rollout(5, 2, 3, 4, obs_kind="sparse")
    ncov = 0
    for gs_before, cold, cov, inv, _, gs_after in g[tag][:45]:
        assert e.global_step == gs_before
        has_factors, will_invert = ctypes.c_int(0), ctypes.c_int(0)
        e.lib.acx_learner_update_plan(e._h, ctypes.byref(has_factors), ctypes.byref(will_invert))
        assert (has_factors.value, will_invert.value) == (cov, inv), (tag, gs_before)
        inv_before = e.buffer("inverses").clone()
        e.update(batch, fetch=False)
        torch.cuda.synchronize()
        ncov += int(cov)
        assert e.global_step == gs_after
        assert e.get_state()["num_cov_updates"] == ncov
        assert (not torch.equal(inv_before, e.buffer("inverses"))) == bool(inv), (tag, gs_before)


@pytest.mark.parametrize("kw", [dict(inv_init="identity"), dict(cov_init="identity"), dict(zero_debias=False),
                                dict(cov_init="identity", inv_init="identity", zero_debias=False)])
def test_acktr_init_conventions(kw):
    """SURVEY A.7-U3 knobs (older tf.contrib.kfac conventions), engine against oracle update by update: identity inverses
    make the always-run K-FAC apply a real step in the cold phase and before the first refresh."""
    eng = _engine_mod()
    cfg = eng.EngineConfig(num_envs=4, num_steps=5, num_cold_updates=2, invert_every=2, **kw)
    records = LC.run_schedule(cfg, 5, obs_kind="sparse")
    _check_schedule(records, TOL_DEFAULT)
    if kw.get("inv_init") == "identity":
        assert all("precon" in r for r in records)          # K-FAC steps from the very first update
        assert records[0]["step_rel"] <= TOL_DEFAULT
    else:
        assert "precon" not in records[0]


# ------------------------------------------------------------------------------------------------ NCCL, 2 ranks
def _nccl_worker(rank, world, port, out_dir):
    import os
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for p in (root, os.path.join(root, "tests"), os.path.join(root, "tests", "golden")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torch.distributed as dist
    from actorcritic_b200 import engine as eng
    from actorcritic_b200 import parallel
    torch.cuda.set_device(rank)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        kw = dict(num_steps=5, num_cold_updates=2, invert_every=2, lr_decay_steps=1000.0)
        params = onet.perturbed_params(4, 32, 7)
        results = {}
        # split exchange (default) and the single all-reduce, each with the exchange inside phase 2 over NVLink peer memory
        # (csrc/peer.cu, default) and with NCCL between the phases
        # ("2" = the general two-shot route of the peer kernel, which two ranks would not take by themselves)
        for split, peer in (("1", "1"), ("0", "1"), ("1", "0"), ("0", "0"), ("1", "2")):
            os.environ["ACX_DP_SPLIT"] = split
            os.environ["ACX_PEER"] = "0" if peer == "0" else "1"
            os.environ["ACX_PEER_TWO_SHOT"] = "1" if peer == "2" else "0"
            e = eng.Engine(eng.EngineConfig(num_envs=8 // world, world_size=world, **kw))
            e.set_params(params)
            for u in range(7):
                batch = parallel.shard_batch(synth.rollout(60 + u, 8, 5, 4, obs_kind="sparse"), rank, world)
                y, eps = synth.fisher_samples(70 + u, 40)
                lo, hi = parallel.shard_range(8, rank, world)
                yy = torch.from_numpy(y.reshape(8, 5)[lo:hi].reshape(-1).copy()).cuda()
                ee = torch.from_numpy(eps.reshape(8, 5)[lo:hi].reshape(-1).copy()).cuda()
                e.update(batch, yy, ee, fetch=False)
            torch.cuda.synchronize()
            assert bool(getattr(e, "_peer_state", False)) == (peer != "0"), "the peer exchange must be what ran"
            from actorcritic_b200 import _lib
            assert _lib.load().acx_peer_error() == 0
            results[split + peer] = dict(params=e.get_params_flat().copy(), sums=e.buffer("factor_sums").cpu().numpy().copy(),
                                         inv=e.buffer("inverses").cpu().numpy().copy(), gs=e.global_step)
        np.savez(os.path.join(out_dir, "rank%d.npz" % rank),
                 **{"%s_%s" % (k, s): v for s, r in results.items() for k, v in r.items()})
    finally:
        dist.destroy_process_group()


def test_nccl_two_ranks_split_exchange_equals_single_device(tmp_path):
    """G6 over NCCL: 2 ranks x 4 environments through Engine.update (the split exchange: [G | grads | scalars] on the
    engine's stream, the input-factor prefix on a second communicator under phase 2) against one engine over all 8
    environments; the split exchange must be bit-identical to the single all-reduce and both ranks identical."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 CUDA devices")
    import socket
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_nccl_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = (np.load(str(tmp_path / ("rank%d.npz" % r))) for r in (0, 1))
    for key in ("params", "sums", "inv"):
        for mode in ("11", "01", "10", "00", "12"):
            assert np.array_equal(r0[key + "_" + mode], r1[key + "_" + mode]), (key, mode)     # ranks never diverge
            # split exchange == single all-reduce, peer-memory exchange == NCCL (two ranks: one commutative addition)
            assert np.array_equal(r0[key + "_11"], r0[key + "_" + mode]), (key, mode)
    eng = _engine_mod()
    full = eng.Engine(eng.EngineConfig(num_envs=8, num_steps=5, num_cold_updates=2, invert_every=2, lr_decay_steps=1000.0))
    full.set_params(onet.perturbed_params(4, 32, 7))
    for u in range(7):
        batch = synth.rollout(60 + u, 8, 5, 4, obs_kind="sparse")
        y, eps = synth.fisher_samples(70 + u, 40)
        full.update(batch, torch.from_numpy(y).cuda(), torch.from_numpy(eps).cuda(), fetch=False)
    torch.cuda.synchronize()
    assert full.global_step == int(r0["gs_11"])
    assert LC.rel_err(r0["sums_11"], full.buffer("factor_sums").cpu().numpy()) <= 1e-5
    # seven free-running K-FAC updates (lr 0.25): the 2-rank sum order differs from the single-device one by fp32 rounding
    assert LC.rel_err(r0["params_11"], full.get_params_flat()) <= 1e-4
