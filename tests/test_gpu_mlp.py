"""The fully connected learner (csrc/mlp.cu, MLPEngine, MLPModel) on the GPU against the fp64 oracle (oracle/mlp.py):
per-update parity at two sizes, the ACKTR schedule, A2C, determinism, resume, acting, the reference loop and learning on a
contextual bandit.  Every parity check uses seeded inputs and injected Fisher samples."""
import numpy as np
import pytest
import torch

import synth
from learner_checks import rel_err
from oracle import kfac as K
from oracle import learner as OL
from oracle import mlp as OM

from actorcritic_b200 import engine as eng

pytestmark = pytest.mark.gpu

SMALL = dict(obs_dim=17, hidden_sizes=(64, 40), num_actions=5, num_envs=8, num_steps=5)
LARGE = dict(obs_dim=128, hidden_sizes=(256, 256), num_actions=8, num_envs=256, num_steps=20)


def params_for(cfg, seed=0):
    """Orthogonal weights (nn.fully_connected_params) with non-zero biases and a policy gain of 0.5, so that every
    gradient term is exercised."""
    from actorcritic_b200 import nn
    rng = np.random.default_rng(seed)
    shapes = eng.mlp_param_shapes(cfg.obs_dim, cfg.hidden_sizes, cfg.num_actions)
    p = {}
    for layer in eng.mlp_layers(len(cfg.hidden_sizes)):
        gain = {"fc_policy": 0.5, "fc_baseline": 1.0}.get(layer, 2 ** 0.5)
        w, _ = nn.fully_connected_params(*shapes[layer + "/weights"], rng=rng, gain=gain)
        p[layer + "/weights"] = w
        p[layer + "/bias"] = (0.05 * rng.standard_normal(shapes[layer + "/bias"])).astype(np.float32)
    return p


def rollout(seed, cfg):
    rng = np.random.default_rng(seed)
    e, t, d = cfg.num_envs, cfg.num_steps, cfg.obs_dim
    return dict(observations=rng.standard_normal((e, t, d)).astype(np.float32),
                bootstrap_observations=rng.standard_normal((e, d)).astype(np.float32),
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
    return OM.MLPOracle(params, len(cfg.hidden_sizes), acktr=cfg.acktr, cfg=ocfg, gamma=cfg.gamma, beta=cfg.entropy_beta,
                        value_weight=cfg.value_loss_weight)


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


def engine_masks(e, hidden):
    n = e.rows
    return {name: (e.buffer("act_hi/" + name, torch.bfloat16).view(-1, e._layer_cols(name))[:n].float() > 0).cpu()
            for name in hidden}


def run_parity(cfg, num_updates, seed=0, resync=True):
    params = params_for(cfg, seed)
    e = eng.MLPEngine(cfg)
    e.set_params(params)
    o = oracle_for(cfg, params)
    n = cfg.num_envs * cfg.num_steps
    recs = []
    for u in range(num_updates):
        batch = rollout(100 + u + 1000 * seed, cfg)
        y_hat, eps = synth.fisher_samples(500 + u, n, num_actions=cfg.num_actions)
        if resync and u > 0:
            sync(e, o)
        before = o.flat_params()
        gs = e.global_step
        scal = e.update(batch, torch.from_numpy(y_hat).cuda() if cfg.acktr else None,
                        torch.from_numpy(eps).cuda() if cfg.acktr else None)
        masks = engine_masks(e, o.hidden)
        info = o.update(batch, y_hat, eps, masks=masks) if cfg.acktr else o.update(batch, masks=masks)
        for name, m in masks.items():   # units on the other ReLU branch than the fp64 oracle: within rounding of zero
            pre = info["fwd"]["pre"][name]
            diff = m.reshape(pre.shape) != (pre > 0)
            if diff.any():
                assert float(pre[diff].abs().max()) <= 1e-4 * float(pre.pow(2).mean().sqrt()), (u, name)
        torch.cuda.synchronize()
        rec = dict(update=u, gs=(gs, e.global_step, o.global_step), state=e.get_state())
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
            tight["step"] = step            # a K-FAC step (lr 0.25 scale)
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


@pytest.mark.parametrize("size", [SMALL, LARGE], ids=["small", "large"])
def test_acktr_schedule_parity(size):
    """num_cold_updates=2, invert_every=2, 8 updates: cold steps, covariance-only steps, refreshes and K-FAC steps."""
    cfg = eng.MLPEngineConfig(num_cold_updates=2, invert_every=2, seed=3, **size)
    e, o, recs = run_parity(cfg, 8)
    for rec in recs:
        gs, gs_after, ogs = rec["gs"]
        ev = K.schedule_events(gs, 2, 2)
        assert gs_after == ogs == ev["gs_after"], rec["gs"]
    assert any("invA/fc1" in r["tight"] for r in recs) and any("precon/fc1" in r["tight"] for r in recs)
    assert recs[-1]["state"]["num_cov_updates"] == o.num_cov_updates
    check(recs)


@pytest.mark.parametrize("size", [SMALL, LARGE], ids=["small", "large"])
def test_a2c_parity(size):
    """ClipGlobalNorm(RMSProp) over 5 updates."""
    cfg = eng.MLPEngineConfig(acktr=False, lr_start=7e-4, lr_end=7e-5, seed=4, **size)
    e, o, recs = run_parity(cfg, 5)
    assert [r["gs"][1] for r in recs] == [1, 2, 3, 4, 5]
    check(recs)


def _run_free(cfg, updates, seed=7, sd=None, start=0):
    e = eng.MLPEngine(cfg)
    e.set_params(params_for(cfg, seed))
    if sd is not None:
        e.load_state_dict(sd)
    n = cfg.num_envs * cfg.num_steps
    for u in range(start, start + updates):
        y, eps = synth.fisher_samples(900 + u, n, num_actions=cfg.num_actions)
        e.update(rollout(700 + u, cfg), torch.from_numpy(y).cuda(), torch.from_numpy(eps).cuda(), fetch=False)
    torch.cuda.synchronize()
    return e


def test_graphs_and_runs_are_bit_identical():
    base = dict(num_cold_updates=1, invert_every=2, seed=5, **SMALL)
    a = _run_free(eng.MLPEngineConfig(**base), 7)
    b = _run_free(eng.MLPEngineConfig(**base), 7)
    c = _run_free(eng.MLPEngineConfig(use_graphs=False, **base), 7)
    pa, pb, pc = a.get_params_flat(), b.get_params_flat(), c.get_params_flat()
    assert np.array_equal(pa, pb) and np.array_equal(pa, pc)
    for name in ("factor_sums", "inverses", "velocity"):
        assert torch.equal(a.buffer(name).cpu(), c.buffer(name).cpu()), name


def test_resume_in_another_batch_shape():
    """state_dict after k updates, passed through an engine of another batch shape, continues bit-identically: the
    learner state does not depend on the batch shape."""
    base = dict(obs_dim=17, hidden_sizes=(64, 40), num_actions=5, num_cold_updates=1, invert_every=2, seed=5)
    shape, other = dict(num_envs=8, num_steps=5), dict(num_envs=4, num_steps=3)
    straight = _run_free(eng.MLPEngineConfig(**base, **shape), 7)
    first = _run_free(eng.MLPEngineConfig(**base, **shape), 4)
    middle = eng.MLPEngine(eng.MLPEngineConfig(**base, **other))
    middle.load_state_dict(first.state_dict())
    assert middle.get_state() == first.get_state()
    resumed = _run_free(eng.MLPEngineConfig(**base, **shape), 3, sd=middle.state_dict(), start=4)
    assert np.array_equal(resumed.get_params_flat(), straight.get_params_flat())
    for name in ("factor_sums", "inverses", "velocity", "accum"):
        assert torch.equal(resumed.buffer(name).cpu(), straight.buffer(name).cpu()), name


def test_acting_greedy_and_inverse_cdf():
    cfg = eng.MLPEngineConfig(acktr=False, **SMALL)
    e = eng.MLPEngine(cfg)
    e.set_params(params_for(cfg, 1))
    rows = 30
    obs = torch.randn(rows, cfg.obs_dim, generator=torch.Generator().manual_seed(0)).cuda()
    greedy, logits, values = e.act(obs, greedy=True, want_logits=True)
    z = logits.cpu().numpy()
    assert np.array_equal(greedy.cpu().numpy(), z.argmax(1))
    want = OM.forward({k: torch.tensor(v, dtype=torch.float64) for k, v in params_for(cfg, 1).items()}, obs.cpu().numpy(),
                      ("fc1", "fc2"))
    assert rel_err(z, want["logits"].numpy()) <= 1e-4 and rel_err(values.cpu().numpy(), want["value"].numpy()) <= 1e-4
    u = torch.rand(rows, generator=torch.Generator().manual_seed(1)).cuda()
    sampled = e.act(obs, uniform=u, greedy=False).cpu().numpy()
    zz = torch.from_numpy(z)
    p = torch.exp(zz - zz.max(1, keepdim=True).values)
    p = p / p.sum(1, keepdim=True)
    cum = torch.cumsum(p, 1).numpy()
    uu = u.cpu().numpy()
    want_pick = np.array([min(int(np.searchsorted(cum[r], uu[r], side="right")), cfg.num_actions - 1) for r in range(rows)])
    # the kernel accumulates exp(z - max) / sum in fp32 in the same order; compare away from CDF ties
    gap = np.abs(cum - uu[:, None]).min(1)
    assert np.array_equal(sampled[gap > 1e-5], want_pick[gap > 1e-5])


class BanditEnv:
    """Seeded contextual bandit: observation = a random context in [-1, 1]^D, reward 1 when the action equals
    argmax(obs[:n]), every step terminal (a new context follows)."""

    def __init__(self, dim, num_actions, seed):
        self.dim, self.n = dim, num_actions
        self.rng = np.random.default_rng(seed)
        self.obs = None

    def reset(self):
        self.obs = self.rng.uniform(-1, 1, self.dim).astype(np.float32)
        return self.obs

    def step(self, action):
        r = float(int(action) == int(np.argmax(self.obs[: self.n])))
        return self.reset(), r, True, {}


def _setup(acktr, dim, num_actions, num_envs, num_steps, seed=0):
    import actorcritic_b200 as ac
    from actorcritic_b200 import kfac, nn, objectives, spaces
    from actorcritic_b200.kfac_utils import ColdStartPeriodicInvUpdateKfacOpt
    from actorcritic_b200.mlp import MLPModel
    model = MLPModel(spaces.Box(low=-1, high=1, shape=(dim,), dtype=np.float32), spaces.Discrete(num_actions),
                     hidden_sizes=(64, 64), random_seed=seed)
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
    """a2c_acktr.py:117-126 with MLPModel: MultiEnvAgent on host vector environments, Session.run([summary, global_step,
    optimize_op]) for both optimizers."""
    from actorcritic_b200 import agents, multi_env, summary
    summary.reset_default_collection()
    ac, model, objective, global_step, optimize_op = _setup(acktr, 6, 3, 4, 5)
    with summary.name_scope("model"):
        summary.scalar("policy_loss", objective.policy_loss)
    summary_op = summary.merge_all()
    env = multi_env.MultiEnv([BanditEnv(6, 3, s) for s in range(4)])
    agent = agents.MultiEnvAgent(env, model, num_steps=5)
    with ac.Session() as session:
        for it in range(3):
            obs, act, rew, term, nxt, _ = agent.interact(session)
            out = session.run([summary_op, global_step, optimize_op],
                              feed_dict={model.observations_placeholder: obs, model.bootstrap_observations_placeholder: nxt,
                                         model.actions_placeholder: act, model.rewards_placeholder: rew,
                                         model.terminals_placeholder: term})
            assert out[0] is not None
        assert int(out[1]) in (2, 3, 4, 5, 6) and model.engine.is_learner
    v = model.get_variables()
    assert all(np.isfinite(a).all() for a in v.values())


def _learn(acktr, updates, num_envs=64, dim=8, n=4, held_out=128):
    """Train on the bandit through Session.run (one step per episode); greedy accuracy on held-out contexts (at most
    the N + E rows of the learner)."""
    ac, model, objective, global_step, optimize_op = _setup(acktr, dim, n, num_envs, 1, seed=1)
    rng = np.random.default_rng(2)
    with ac.Session() as session:
        for _ in range(updates):
            ctx = rng.uniform(-1, 1, (num_envs, 1, dim)).astype(np.float32)
            acts = np.asarray(model.sample_actions(ctx, session), np.uint8).reshape(num_envs, 1)
            rew = (acts[:, 0] == ctx[:, 0, :n].argmax(1)).astype(np.float32).reshape(num_envs, 1)
            session.run(optimize_op, feed_dict={model.observations_placeholder: ctx,
                                                model.bootstrap_observations_placeholder: ctx[:, 0],
                                                model.actions_placeholder: acts, model.rewards_placeholder: rew,
                                                model.terminals_placeholder: np.ones((num_envs, 1), bool)})
        test = np.random.default_rng(99).uniform(-1, 1, (held_out, 1, dim)).astype(np.float32)
        greedy = np.asarray(model.select_max_actions(test, session)).reshape(-1)
    return float((greedy == test[:, 0, :n].argmax(1)).mean())


# measured on B200 with 64 held-out contexts: ACKTR 0.92 / 0.91 / 0.95 after 100 / 200 / 400 updates, A2C 0.56 / 0.73 / 0.91
# (chance 0.25); the counts below leave both well past the bar
@pytest.mark.parametrize("acktr, updates", [(True, 600), (False, 1200)], ids=["acktr", "a2c"])
def test_learns_contextual_bandit(acktr, updates):
    acc = _learn(acktr, updates)
    print("greedy accuracy on held-out contexts (%s, %d updates): %.3f" % ("ACKTR" if acktr else "A2C", updates, acc))
    assert acc >= 0.9
