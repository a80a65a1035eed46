"""The convolutional learner (csrc/mlp.cu `acx_cnn_*`, CNNEngine, CNNModel) on the GPU against the fp64 oracle
(oracle/cnn.py): per-update parity on uint8 and float32 images of several geometries (padded first-layer patches, a col2im
row wider than one CTA, a kernel-1 layer, a stride that does not divide its input), on both inverse-refresh paths, the ACKTR
schedule and A2C; a cross-check against AtariModel's learner at the Nature geometry; determinism, resume, acting, the
reference loop and learning on a visual bandit.  Every parity check uses seeded inputs and injected Fisher samples."""
import numpy as np
import pytest
import torch

import synth
from learner_checks import rel_err
from oracle import cnn as OC
from oracle import kfac as K
from oracle import learner as OL
from oracle import mlp as OM

from actorcritic_b200 import _lib
from actorcritic_b200 import engine as eng

pytestmark = pytest.mark.gpu

U8_36 = dict(obs_hw=36, obs_channels=4, obs_u8=True, conv_layers=((16, 8, 4), (32, 3, 1)), hidden_sizes=(64,), num_actions=4,
             num_envs=8, num_steps=5)
F32_10 = dict(obs_hw=10, obs_channels=7, obs_u8=False, conv_layers=((16, 3, 1),), hidden_sizes=(128,), num_actions=6,
              num_envs=16, num_steps=5)
# conv2 reads a 31 x 31 x 64 input: one col2im row is 496 threads (two CTAs); (31 - 5) / 3 leaves a remainder
U8_64 = dict(obs_hw=64, obs_channels=3, obs_u8=True, conv_layers=((64, 4, 2), (32, 5, 3)), hidden_sizes=(64,), num_actions=5,
             num_envs=4, num_steps=5)
# a kernel-1 conv3, and input factors of 2049 (conv2) and 3137 (fc4): more tiles than the SMs' shared memory holds, so
# the inverse refresh takes the fp64 chain
WIDE = dict(obs_hw=22, obs_channels=16, obs_u8=True, conv_layers=((128, 4, 2), (128, 4, 1), (64, 1, 1)), hidden_sizes=(1024,),
            num_actions=3, num_envs=4, num_steps=5)
SIZES = {"u8_36x36x4": (U8_36, "resident"), "f32_10x10x7": (F32_10, "resident"), "u8_64x64x3": (U8_64, "resident"),
         "u8_22x22x16_k1": (WIDE, "fp64 chain")}


def params_for(cfg, seed=0):
    """Orthogonal weights with non-zero biases and a policy gain of 0.5, so that every gradient term is exercised."""
    from actorcritic_b200 import nn
    rng = np.random.default_rng(seed)
    shapes = eng.cnn_param_shapes(cfg.obs_hw, cfg.obs_channels, cfg.conv_layers, cfg.hidden_sizes, cfg.num_actions)
    p = {}
    for layer in eng.cnn_layers(len(cfg.conv_layers), len(cfg.hidden_sizes)):
        shape = shapes[layer + "/weights"]
        gain = {"fc_policy": 0.5, "fc_baseline": 1.0}.get(layer, 2 ** 0.5)
        if len(shape) == 4:
            w, _ = nn.conv2d_params(shape[2], shape[3], shape[0], rng=rng, gain=gain)
        else:
            w, _ = nn.fully_connected_params(*shape, rng=rng, gain=gain)
        p[layer + "/weights"] = w
        p[layer + "/bias"] = (0.05 * rng.standard_normal(shapes[layer + "/bias"])).astype(np.float32)
    return p


def images(rng, shape, u8):
    if u8:   # sparse bright pixels over a dark background, as game frames
        return (rng.integers(0, 256, shape) * (rng.random(shape) < 0.3)).astype(np.uint8)
    return rng.standard_normal(shape).astype(np.float32)


def rollout(seed, cfg):
    rng = np.random.default_rng(seed)
    e, t = cfg.num_envs, cfg.num_steps
    img = (cfg.obs_hw, cfg.obs_hw, cfg.obs_channels)
    return dict(observations=images(rng, (e, t) + img, cfg.obs_u8), bootstrap_observations=images(rng, (e,) + img, cfg.obs_u8),
                actions=rng.integers(0, cfg.num_actions, (e, t)).astype(np.uint8),
                rewards=rng.standard_normal((e, t)).astype(np.float32), terminals=rng.random((e, t)) < 0.1)


def oracle_for(cfg, params):
    n = cfg.num_envs * cfg.num_steps
    decay = cfg.lr_decay_steps or 1e7 / n
    if cfg.acktr:
        ocfg = K.KfacConfig(learning_rate_start=cfg.lr_start, learning_rate_end=cfg.lr_end, decay_steps=decay,
                            cov_ema_decay=cfg.cov_ema_decay, damping=cfg.damping, momentum=cfg.momentum,
                            norm_constraint=cfg.norm_constraint, invert_every=cfg.invert_every,
                            num_cold_updates=cfg.num_cold_updates, cold_learning_rate=cfg.cold_lr,
                            cold_momentum=cfg.cold_momentum, clip_norm=cfg.clip_norm)
    else:
        ocfg = OL.A2CConfig(learning_rate_start=cfg.lr_start, learning_rate_end=cfg.lr_end, decay_steps=decay,
                            rms_decay=cfg.rms_decay, rms_epsilon=cfg.rms_epsilon, clip_norm=cfg.clip_norm)
    return OC.CNNOracle(params, cfg.obs_hw, cfg.obs_channels, cfg.conv_layers, len(cfg.hidden_sizes), obs_u8=cfg.obs_u8,
                        acktr=cfg.acktr, cfg=ocfg, gamma=cfg.gamma, beta=cfg.entropy_beta, value_weight=cfg.value_loss_weight)


def sync(e, o):
    """The oracle's complete learner state into the engine (single-update parity from identical state)."""
    for layer in o.layers:
        e.layer_matrix("params", layer).copy_(OM.vmat(o.params, layer).float())
        if o.acktr:
            e.layer_matrix("velocity", layer).copy_(o.velocity[layer].float())
            e.layer_matrix("accum", layer).copy_(o.cold_accum[layer].float())
            e.factor("sums", "G", layer).copy_(o.sum_g[layer].float())
            e.factor("inv", "A", layer).copy_(o.inv_a[layer].float())
            e.factor("inv", "G", layer).copy_(o.inv_g[layer].float())
        else:
            e.layer_matrix("accum", layer).copy_(o.rms[layer].float())
    valid = False
    if o.acktr:
        for f, s in o.sum_a.items():
            e.factor("sums", "A", f).copy_(s.float())
        valid = any(float(v.abs().max()) > 0 for v in o.inv_a.values())
    e.set_state(o.global_step, o.num_cov_updates if o.acktr else 0, valid)
    e.refresh_derived()


def engine_masks(e, trunk):
    """The ReLU masks the engine's backward applies (hi plane of each activation > 0), train rows [N * T, C]."""
    n = e.rows
    out = {}
    for name in trunk:
        c = e._layer_cols(name)
        hi = e.buffer("act_hi/" + name, torch.bfloat16).view(e.rows + e.num_envs, -1, c)[:n]
        out[name] = (hi.float() > 0).reshape(-1, c).cpu()
    return out


def run_parity(cfg, num_updates, seed=0):
    params = params_for(cfg, seed)
    e = eng.CNNEngine(cfg)
    e.set_params(params)
    o = oracle_for(cfg, params)
    n = cfg.num_envs * cfg.num_steps
    recs = []
    for u in range(num_updates):
        batch = rollout(100 + u + 1000 * seed, cfg)
        y_hat, eps = synth.fisher_samples(500 + u, n, num_actions=cfg.num_actions)
        if u > 0:
            sync(e, o)
        before = o.flat_params()
        gs = e.global_step
        launches = _lib.launch_count()
        scal = e.update(batch, torch.from_numpy(y_hat).cuda() if cfg.acktr else None,
                        torch.from_numpy(eps).cuda() if cfg.acktr else None)
        launches = _lib.launch_count() - launches
        masks = engine_masks(e, o.hidden)
        info = o.update(batch, y_hat, eps, masks=masks) if cfg.acktr else o.update(batch, masks=masks)
        for name, m in masks.items():   # units on the other ReLU branch than the fp64 oracle: within rounding of zero
            pre = info["fwd"]["pre"][name]
            diff = m.reshape(pre.shape) != (pre > 0)
            if diff.any():
                assert float(pre[diff].abs().max()) <= 1e-4 * float(pre.pow(2).mean().sqrt()), (u, name)
        torch.cuda.synchronize()
        rec = dict(update=u, gs=(gs, e.global_step, o.global_step), state=e.get_state(), launches=launches,
                   inverted=bool(info.get("inverted")))
        err = {}
        err["logits"] = rel_err(e.logits[:n].cpu().numpy(), info["fwd"]["logits"].numpy())
        err["values"] = rel_err(e.values[:n].cpu().numpy(), info["fwd"]["value"].numpy())
        err["bootstrap_values"] = rel_err(e.values[n:].cpu().numpy(), info["bootstrap_values"].numpy())
        losses = info["losses"]
        err["losses"] = rel_err([scal[k] for k in ("policy_loss", "baseline_loss", "mean_entropy", "loss")],
                                [float(losses[k]) for k in ("policy_loss", "baseline_loss", "mean_entropy", "loss")])
        for layer in o.layers:
            err["grad/" + layer] = rel_err(e.layer_matrix("grads", layer).cpu().numpy(), info["grads"][layer].numpy())
        if "new_a" in info:
            for f, a in info["new_a"].items():
                err["A/" + f] = rel_err(e.factor("stats", "A", f).cpu().numpy(), a.numpy())
            for layer, g in info["new_g"].items():
                err["G/" + layer] = rel_err(e.factor("stats", "G", layer).cpu().numpy(), g.numpy())
        rec["fwd"] = err
        tight = {}
        if info.get("inverted"):
            for layer in o.layers:
                tight["invA/" + layer] = rel_err(e.factor("inv", "A", layer).cpu().numpy(), o.inv_a[layer].numpy())
                tight["invG/" + layer] = rel_err(e.factor("inv", "G", layer).cpu().numpy(), o.inv_g[layer].numpy())
        if cfg.acktr and e.get_state()["inverses_valid"]:
            for layer in o.layers:
                tight["precon/" + layer] = rel_err(e.layer_matrix("precon", layer).cpu().numpy(), info["precon"][layer].numpy())
            tight["clip_coeff"] = abs(scal["clip_coeff"] - info["clip_coeff"]) / abs(info["clip_coeff"])
        after = e.get_params_flat().astype(np.float64)
        rec["params_rel"] = rel_err(after, o.flat_params())
        step = rel_err(after - before, o.flat_params() - before)
        if cfg.acktr and e.get_state()["inverses_valid"] and gs >= cfg.num_cold_updates:
            tight["step"] = step            # a K-FAC step
        else:
            rec["small_step"] = step        # cold / RMSProp steps: fp32 parameters leave a ~1e-8 |theta| / |step| floor
        rec["tight"] = tight
        recs.append(rec)
    return e, o, recs


def check(recs, fwd_tol=2e-4, tight_tol=1e-3):
    worst = {}
    for rec in recs:
        for k, v in rec["fwd"].items():
            assert v <= fwd_tol, (rec["update"], k, v)
            worst[k] = max(worst.get(k, 0.0), v)
        for k, v in rec["tight"].items():
            assert v <= tight_tol, (rec["update"], k, v)
            worst[k] = max(worst.get(k, 0.0), v)
        assert rec["params_rel"] <= 1e-5, (rec["update"], rec["params_rel"])
        worst["params"] = max(worst.get("params", 0.0), rec["params_rel"])
        if "small_step" in rec:
            assert rec["small_step"] <= 1e-2, (rec["update"], rec["small_step"])
            worst["small_step"] = max(worst.get("small_step", 0.0), rec["small_step"])
    print("measured maxima:", {k: "%.1e" % v for k, v in sorted(worst.items())})
    return worst


def inverse_path(recs):
    """The refresh path, from the launches a refreshing K-FAC update adds to a non-refreshing one: the resident kernel is
    one launch, the fp64 chain about three per 32-row pivot step of the largest factor."""
    inv = [r["launches"] for r in recs if r["inverted"]]
    plain = [r["launches"] for r in recs if not r["inverted"] and r["state"]["inverses_valid"] and r["gs"][0] > 2]
    added = inv[-1] - plain[-1]
    return ("fp64 chain" if added > 50 else "resident"), added


@pytest.mark.parametrize("size", list(SIZES), ids=list(SIZES))
def test_acktr_schedule_parity(size):
    """num_cold_updates=2, invert_every=2, 8 updates: cold steps, covariance-only steps, refreshes and K-FAC steps."""
    shape, want_path = SIZES[size]
    cfg = eng.CNNEngineConfig(num_cold_updates=2, invert_every=2, seed=3, **shape)
    e, o, recs = run_parity(cfg, 8)
    for rec in recs:
        gs, gs_after, ogs = rec["gs"]
        assert gs_after == ogs == K.schedule_events(gs, 2, 2)["gs_after"], rec["gs"]
    assert any("invA/conv1" in r["tight"] for r in recs) and any("precon/conv1" in r["tight"] for r in recs)
    assert recs[-1]["state"]["num_cov_updates"] == o.num_cov_updates
    path, added = inverse_path(recs)
    print("inverse refresh path: %s (%d launches added by the refresh)" % (path, added))
    assert path == want_path, (path, added)
    check(recs)


@pytest.mark.parametrize("size", ["u8_36x36x4", "f32_10x10x7"])
def test_a2c_parity(size):
    """ClipGlobalNorm(RMSProp) over 5 updates."""
    cfg = eng.CNNEngineConfig(acktr=False, lr_start=7e-4, lr_end=7e-5, seed=4, **SIZES[size][0])
    e, o, recs = run_parity(cfg, 5)
    assert [r["gs"][1] for r in recs] == [1, 2, 3, 4, 5]
    check(recs)


def test_matches_the_atari_learner_at_the_nature_geometry():
    """84x84x4 uint8, conv (32,8,4), (64,4,2), (32,3,1), fc 512 on 4 x 5: one cold update, then one covariance + refresh +
    K-FAC update, from the same parameters and Fisher samples in CNNEngine and AtariModel's engine.Engine.  Logits,
    gradients, factors and parameters agree within 5e-4.  The preconditioned blocks agree within 2e-3: each learner keeps
    them within 1e-3 of the fp64 oracle, and the inverses amplify the rounding differences of the two learners' factors
    (measured on B200: 1.1e-3 for fc_baseline)."""
    from oracle import network as onet
    shape = dict(num_envs=4, num_steps=5, num_actions=4, num_cold_updates=1, invert_every=1, seed=2)
    atari = eng.Engine(eng.EngineConfig(conv3_filters=32, **shape))
    cnn = eng.CNNEngine(eng.CNNEngineConfig(obs_hw=84, obs_channels=4, obs_u8=True,
                                            conv_layers=((32, 8, 4), (64, 4, 2), (32, 3, 1)), hidden_sizes=(512,), **shape))
    params = onet.perturbed_params(4, 32, seed=1)
    atari.set_params(params)
    cnn.set_params(params)
    assert cnn.layers == onet.LAYERS
    n = 20
    worst = {}
    for u in range(2):
        batch = synth.rollout(40 + u, 4, 5, 4, obs_kind="uniform")
        y, eps = synth.fisher_samples(60 + u, n, num_actions=4)
        fl, fe = torch.from_numpy(y).cuda(), torch.from_numpy(eps).cuda()
        atari.update(batch, fl, fe, fetch=False)
        cnn.update(batch, fl, fe, fetch=False)
        torch.cuda.synchronize()
        got = {"logits": (cnn.logits[:n], atari.logits[:n]), "values": (cnn.values, atari.values),
               "params": (cnn.buffer("params"), atari.buffer("params"))}
        for layer in onet.LAYERS:
            got["grad/" + layer] = (cnn.layer_matrix("grads", layer), atari.layer_matrix("grads", layer))
        if u == 1:
            for f in K.A_FACTORS:
                got["A/" + f] = (cnn.factor("stats", "A", f), atari.factor("stats", "A", f))
            for layer in onet.LAYERS:
                got["G/" + layer] = (cnn.factor("stats", "G", layer), atari.factor("stats", "G", layer))
                got["precon/" + layer] = (cnn.layer_matrix("precon", layer), atari.layer_matrix("precon", layer))
        for k, (a, b) in got.items():
            err = rel_err(a.cpu().numpy(), b.cpu().numpy())
            worst[k] = max(worst.get(k, 0.0), err)
            assert err <= (2e-3 if k.startswith("precon/") else 5e-4), (u, k, err)
    assert cnn.get_state() == atari.get_state() and cnn.get_state()["inverses_valid"]
    print("CNNEngine vs Engine maxima:", {k: "%.1e" % v for k, v in sorted(worst.items())})


def _run_free(cfg, updates, seed=7, sd=None, start=0):
    e = eng.CNNEngine(cfg)
    e.set_params(params_for(cfg, seed))
    if sd is not None:
        e.load_state_dict(sd)
    n = cfg.num_envs * cfg.num_steps
    for u in range(start, start + updates):
        y, eps = synth.fisher_samples(900 + u, n, num_actions=cfg.num_actions)
        e.update(rollout(700 + u, cfg), torch.from_numpy(y).cuda(), torch.from_numpy(eps).cuda(), fetch=False)
    torch.cuda.synchronize()
    return e


@pytest.mark.parametrize("size", ["u8_64x64x3", "f32_10x10x7"])
def test_graphs_and_runs_are_bit_identical(size):
    base = dict(SIZES[size][0], num_cold_updates=1, invert_every=2, seed=5)
    a = _run_free(eng.CNNEngineConfig(**base), 7)
    b = _run_free(eng.CNNEngineConfig(**base), 7)
    c = _run_free(eng.CNNEngineConfig(use_graphs=False, **base), 7)
    pa, pb, pc = a.get_params_flat(), b.get_params_flat(), c.get_params_flat()
    assert np.array_equal(pa, pb) and np.array_equal(pa, pc)
    for name in ("factor_sums", "inverses", "velocity"):
        assert torch.equal(a.buffer(name).cpu(), c.buffer(name).cpu()), name


def test_resume_in_another_batch_shape():
    """state_dict after k updates, passed through an engine of another batch shape, continues bit-identically."""
    base = {k: v for k, v in U8_36.items() if k not in ("num_envs", "num_steps")}
    base.update(num_cold_updates=1, invert_every=2, seed=5)
    shape, other = dict(num_envs=8, num_steps=5), dict(num_envs=4, num_steps=3)
    straight = _run_free(eng.CNNEngineConfig(**base, **shape), 7)
    first = _run_free(eng.CNNEngineConfig(**base, **shape), 4)
    middle = eng.CNNEngine(eng.CNNEngineConfig(**base, **other))
    middle.load_state_dict(first.state_dict())
    assert middle.get_state() == first.get_state()
    resumed = _run_free(eng.CNNEngineConfig(**base, **shape), 3, sd=middle.state_dict(), start=4)
    assert np.array_equal(resumed.get_params_flat(), straight.get_params_flat())
    for name in ("factor_sums", "inverses", "velocity", "accum"):
        assert torch.equal(resumed.buffer(name).cpu(), straight.buffer(name).cpu()), name


@pytest.mark.parametrize("size", ["u8_36x36x4", "f32_10x10x7"])
def test_acting_greedy_and_inverse_cdf(size):
    """acx_cnn_act against the oracle's forward and against acx_sample_actions on the same logits."""
    from actorcritic_b200 import ops
    cfg = eng.CNNEngineConfig(acktr=False, **SIZES[size][0])
    e = eng.CNNEngine(cfg)
    e.set_params(params_for(cfg, 1))
    rows = 30
    obs = torch.from_numpy(images(np.random.default_rng(0), (rows, cfg.obs_hw, cfg.obs_hw, cfg.obs_channels), cfg.obs_u8))
    greedy, logits, values = e.act(obs.cuda(), greedy=True, want_logits=True)
    z = logits.cpu().numpy()
    assert np.array_equal(greedy.cpu().numpy(), z.argmax(1))
    o = oracle_for(cfg, params_for(cfg, 1))
    want = o._forward(obs.numpy())
    assert rel_err(z, want["logits"].numpy()) <= 1e-4 and rel_err(values.cpu().numpy(), want["value"].numpy()) <= 1e-4
    u = torch.rand(rows, generator=torch.Generator().manual_seed(1)).cuda()
    sampled = e.act(obs.cuda(), uniform=u, greedy=False, want_logits=True)
    ref = ops.sample_actions(sampled[1], uniform=u)
    assert torch.equal(sampled[0], ref)
    assert torch.equal(ops.sample_actions(logits, greedy=True), greedy)


class ImageBanditEnv:
    """Seeded visual contextual bandit: a 12x12x1 uint8 image, dark but for a bright 2x2 patch at a random place in one of
    its four quadrants; reward 1 when the action is that quadrant; every step terminal."""

    def __init__(self, seed):
        self.rng = np.random.default_rng(seed)
        self.obs, self.quadrant = None, 0

    @staticmethod
    def draw(rng, count):
        q = rng.integers(0, 4, count)
        img = np.zeros((count, 12, 12, 1), np.uint8)
        ys = (q // 2) * 6 + rng.integers(0, 5, count)
        xs = (q % 2) * 6 + rng.integers(0, 5, count)
        for i in range(count):
            img[i, ys[i]:ys[i] + 2, xs[i]:xs[i] + 2, 0] = 255
        return img, q

    def reset(self):
        img, q = self.draw(self.rng, 1)
        self.obs, self.quadrant = img[0], int(q[0])
        return self.obs

    def step(self, action):
        r = float(int(action) == self.quadrant)
        return self.reset(), r, True, {}


def _setup(acktr, num_envs, num_steps, seed=0):
    import actorcritic_b200 as ac
    from actorcritic_b200 import kfac, nn, objectives, spaces
    from actorcritic_b200.cnn import CNNModel
    from actorcritic_b200.kfac_utils import ColdStartPeriodicInvUpdateKfacOpt
    model = CNNModel(spaces.Box(low=0, high=255, shape=(12, 12, 1), dtype=np.uint8), spaces.Discrete(4),
                     conv_layers=((16, 3, 1), (16, 3, 2)), hidden_sizes=(64,), random_seed=seed)
    objective = objectives.A2CObjective(model, discount_factor=0.99, entropy_regularization_strength=0.01)
    global_step = ac.GlobalStep()
    max_step = 1e7 / (num_envs * num_steps)
    if acktr:
        lr = nn.linear_decay(0.25, 0.025, global_step, max_step)
        lc = kfac.LayerCollection()
        model.register_layers(lc)
        model.register_predictive_distributions(lc)
        cold = nn.ClipGlobalNormOptimizer(nn.MomentumOptimizer(learning_rate=0.0003, momentum=0.9), clip_norm=0.5)
        optimizer = ColdStartPeriodicInvUpdateKfacOpt(num_cold_updates=5, cold_optimizer=cold, invert_every=5,
                                                      learning_rate=lr, cov_ema_decay=0.99, damping=0.01, layer_collection=lc,
                                                      momentum=0.9, norm_constraint=0.0001)
    else:
        lr = nn.linear_decay(0.0007, 0.00007, global_step, max_step)
        optimizer = nn.ClipGlobalNormOptimizer(nn.RMSPropOptimizer(learning_rate=lr), clip_norm=0.5)
    optimize_op = objective.optimize_shared(optimizer, baseline_loss_weight=0.5, global_step=global_step)
    return ac, model, objective, global_step, optimize_op


@pytest.mark.parametrize("acktr", [True, False], ids=["acktr", "a2c"])
def test_reference_loop_with_multi_env_agent(acktr):
    """a2c_acktr.py:117-126 with CNNModel: MultiEnvAgent on host image environments, Session.run([summary, global_step,
    optimize_op]) for both optimizers."""
    from actorcritic_b200 import agents, multi_env, summary
    summary.reset_default_collection()
    ac, model, objective, global_step, optimize_op = _setup(acktr, 4, 5)
    with summary.name_scope("model"):
        summary.scalar("policy_loss", objective.policy_loss)
    summary_op = summary.merge_all()
    env = multi_env.MultiEnv([ImageBanditEnv(s) for s in range(4)])
    agent = agents.MultiEnvAgent(env, model, num_steps=5)
    with ac.Session() as session:
        for _ in range(3):
            obs, act, rew, term, nxt, _ = agent.interact(session)
            out = session.run([summary_op, global_step, optimize_op],
                              feed_dict={model.observations_placeholder: obs, model.bootstrap_observations_placeholder: nxt,
                                         model.actions_placeholder: act, model.rewards_placeholder: rew,
                                         model.terminals_placeholder: term})
            assert out[0] is not None
        assert int(out[1]) in (2, 3, 4, 5, 6) and model.engine.is_learner
    v = model.get_variables()
    assert all(np.isfinite(a).all() for a in v.values())


def _learn(acktr, updates, num_envs=64, held_out=128):
    """Train on the visual bandit through Session.run (one step per episode); greedy accuracy on held-out images."""
    ac, model, objective, global_step, optimize_op = _setup(acktr, num_envs, 1, seed=1)
    rng = np.random.default_rng(2)
    with ac.Session() as session:
        for _ in range(updates):
            img, q = ImageBanditEnv.draw(rng, num_envs)
            ctx = img.reshape(num_envs, 1, 12, 12, 1)
            acts = np.asarray(model.sample_actions(ctx, session), np.uint8).reshape(num_envs, 1)
            rew = (acts[:, 0] == q).astype(np.float32).reshape(num_envs, 1)
            session.run(optimize_op, feed_dict={model.observations_placeholder: ctx,
                                                model.bootstrap_observations_placeholder: ctx[:, 0],
                                                model.actions_placeholder: acts, model.rewards_placeholder: rew,
                                                model.terminals_placeholder: np.ones((num_envs, 1), bool)})
        img, q = ImageBanditEnv.draw(np.random.default_rng(99), held_out)
        greedy = np.asarray(model.select_max_actions(img.reshape(held_out, 1, 12, 12, 1), session)).reshape(-1)
    return float((greedy == q).mean())


@pytest.mark.parametrize("acktr, updates", [(True, 600), (False, 1200)], ids=["acktr", "a2c"])
def test_learns_visual_bandit(acktr, updates):
    acc = _learn(acktr, updates)
    print("greedy accuracy on held-out images (%s, %d updates): %.3f" % ("ACKTR" if acktr else "A2C", updates, acc))
    assert acc >= 0.9
