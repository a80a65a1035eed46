"""Shared machinery of the GPU parity tests for the learner engine: runs the CUDA engine and the fp64
oracle on the same seeded inputs and reports, per quantity, the norm-relative and guarded element-wise
errors (SURVEY 7, hard part 3: ||X-Y||_F / ||Y||_F and |x-y| <= tol * max(|y|, 1e-3 * max|Y|))."""
import numpy as np
import torch

import synth
from oracle import kfac as K
from oracle import learner as OL
from oracle import network as onet

from actorcritic_b200 import _lib
from actorcritic_b200 import engine as eng


def rel_err(got, want):
    got = np.asarray(got, np.float64)
    want = np.asarray(want, np.float64)
    denom = np.linalg.norm(want)
    return float(np.linalg.norm(got - want) / denom) if denom > 0 else float(np.linalg.norm(got))


def elem_err(got, want):
    """max over elements of |x-y| / max(|y|, 1e-3 * max|Y|)."""
    got = np.asarray(got, np.float64)
    want = np.asarray(want, np.float64)
    floor = 1e-3 * float(np.abs(want).max()) if want.size else 0.0
    if floor == 0.0:
        return float(np.abs(got).max()) if got.size else 0.0
    return float((np.abs(got - want) / np.maximum(np.abs(want), floor)).max())


def oracle_config(cfg):
    if not cfg.acktr:
        return OL.A2CConfig(learning_rate_start=cfg.lr_start, learning_rate_end=cfg.lr_end,
                            decay_steps=cfg.lr_decay_steps or 1e7 / (cfg.num_envs * cfg.num_steps),
                            rms_decay=cfg.rms_decay, rms_epsilon=cfg.rms_epsilon, clip_norm=cfg.clip_norm)
    return K.KfacConfig(learning_rate_start=cfg.lr_start, learning_rate_end=cfg.lr_end,
                        decay_steps=cfg.lr_decay_steps or 1e7 / (cfg.num_envs * cfg.num_steps),
                        cov_ema_decay=cfg.cov_ema_decay, damping=cfg.damping, momentum=cfg.momentum,
                        norm_constraint=cfg.norm_constraint, invert_every=cfg.invert_every,
                        num_cold_updates=cfg.num_cold_updates, cold_learning_rate=cfg.cold_lr,
                        cold_momentum=cfg.cold_momentum, clip_norm=cfg.clip_norm,
                        num_locations_mode=cfg.num_locations_mode, zero_debias=cfg.zero_debias, cov_init=cfg.cov_init,
                        inv_init=cfg.inv_init)


def make_pair(cfg, seed=0):
    """(engine, oracle learner) with identical perturbed-orthogonal weights."""
    params = onet.perturbed_params(cfg.num_actions, cfg.conv3_filters, seed)
    e = eng.Engine(cfg)
    e.set_params(params)
    o = OL.OracleLearner(params, cfg.num_actions, cfg.conv3_filters, acktr=cfg.acktr, cfg=oracle_config(cfg),
                         gamma=cfg.gamma, beta=cfg.entropy_beta, value_weight=cfg.value_loss_weight, dtype=torch.float64)
    return e, o


def engine_relu_masks(e):
    """The ReLU masks the engine's backward pass applies: hi plane of each forward activation > 0, train rows only
    ({layer: bool [rows_l, C_l]} in the oracle's row order)."""
    n, c3 = e.rows, e.config.conv3_filters
    geom = {"conv1": (400, 32), "conv2": (81, 64), "conv3": (49, c3), "fc4": (1, 512)}
    masks = {}
    for name, (locs, ch) in geom.items():
        hi = e.buffer("act_hi/" + name, torch.bfloat16).view(-1, ch)[: n * locs]
        masks[name] = (hi.float() > 0).cpu()
    return masks


def mask_disagreement(masks, fwd):
    """Units where the engine's ReLU branch differs from the fp64 oracle's: {layer: (count, fraction, largest
    |pre-activation| among them relative to the layer's rms pre-activation)}."""
    out = {}
    for name, m in masks.items():
        pre = fwd[name]["pre"].detach()
        diff = m.reshape(pre.shape) != (pre > 0)
        cnt = int(diff.sum())
        rms = float(pre.pow(2).mean().sqrt())
        worst = float(pre[diff].abs().max()) / rms if cnt else 0.0
        out[name] = (cnt, cnt / pre.numel(), worst)
    return out


def oracle_flat_params(o):
    return np.concatenate([onet.join_vmat(name, o.params).detach().numpy().ravel() for name in onet.LAYERS])


def sync_engine_to_oracle(e, o):
    """Copy the oracle's complete learner state into the engine, so that one update can be compared from
    identical state (trajectories of a K-FAC learner with lr 0.25 diverge chaotically otherwise)."""
    cfg = e.config
    for layer in onet.LAYERS:
        e.layer_matrix("params", layer).copy_(onet.join_vmat(layer, o.params).detach().float())
        if cfg.acktr:
            e.layer_matrix("velocity", layer).copy_(o.kfac.velocity[layer].float())
            e.layer_matrix("accum", layer).copy_(o.cold_accum[layer].float())
            e.factor("sums", "G", layer).copy_(o.kfac.sum_g[layer].float())
            e.factor("inv", "A", layer).copy_(o.kfac.inv_a[layer].float())
            e.factor("inv", "G", layer).copy_(o.kfac.inv_g[layer].float())
        else:
            e.layer_matrix("accum", layer).copy_(o.rms[layer].float())
    inv_valid = False
    if cfg.acktr:
        for f in K.A_FACTORS:
            e.factor("sums", "A", f).copy_(o.kfac.sum_a[f].float())
        inv_valid = any(float(v.abs().max()) > 0 for v in o.kfac.inv_a.values())
    e.set_state(o.global_step, o.kfac.num_cov_updates if cfg.acktr else 0, inv_valid)
    e.refresh_derived()


def compare_compute(e, info, cfg, fisher):
    """Errors of everything phase 1 produces against the oracle's `compute` result."""
    torch.cuda.synchronize()
    n = cfg.num_envs * cfg.num_steps
    out = {}

    def put(name, got, want):
        out[name] = dict(rel=rel_err(got, want), elem=elem_err(got, want))

    put("logits", e.logits[:n].cpu().numpy(), info["fwd"]["logits"].detach().numpy())
    put("values", e.values[:n].cpu().numpy(), info["fwd"]["value"].detach().numpy())
    put("bootstrap_values", e.values[n:].cpu().numpy(), info["bootstrap_values"].detach().numpy())
    put("targets", e.buffer("targets").cpu().numpy(), info["targets"].detach().numpy())
    b = e.bucket[-4:].cpu().numpy()
    losses = info["losses"]
    put("scalars", b, np.array([float(losses["policy_loss"]), float(losses["baseline_loss"]),
                                float(losses["mean_entropy"]), float(losses["loss"])]))
    for layer in onet.LAYERS:
        put("grad/" + layer, e.layer_matrix("grads", layer).cpu().numpy(), info["grads"][layer].detach().numpy())
    if fisher:
        for f in K.A_FACTORS:
            put("A/" + f, e.factor("stats", "A", f).cpu().numpy(), info["new_a"][f].detach().numpy())
        for layer in onet.LAYERS:
            put("G/" + layer, e.factor("stats", "G", layer).cpu().numpy(), info["new_g"][layer].detach().numpy())
    return out


def run_schedule(cfg, num_updates, seed=0, obs_kind="uniform", collect=None, resync=True):
    """Drive engine and oracle through `num_updates` updates from global_step 0 with identical batches and
    injected Fisher samples; returns a list of per-update error records.  With resync the engine is reset to
    the oracle's state before every update (single-update parity); without, the two run freely."""
    e, o = make_pair(cfg, seed)
    n = cfg.num_envs * cfg.num_steps
    records = []
    for u in range(num_updates):
        batch = synth.rollout(100 + seed * 1000 + u, cfg.num_envs, cfg.num_steps, cfg.num_actions, obs_kind=obs_kind)
        y_hat, eps = synth.fisher_samples(500 + u, n, num_actions=cfg.num_actions)
        fl = torch.from_numpy(y_hat).cuda()
        fe = torch.from_numpy(eps).cuda()
        if resync and u > 0:
            sync_engine_to_oracle(e, o)
        gs_before = e.global_step
        assert gs_before == o.global_step
        params_before = oracle_flat_params(o)
        launches_before = _lib.launch_count()
        scal = e.update(batch, fl if cfg.acktr else None, fe if cfg.acktr else None)
        launches = _lib.launch_count() - launches_before
        # the oracle differentiates its ReLUs at the engine's masks (the forward activations of this update are still in
        # the arena), and the units where that differs from its own branch must be within rounding of zero
        masks = engine_relu_masks(e)
        info = o.update(batch, y_hat, eps, masks=masks) if cfg.acktr else o.update(batch, masks=masks)
        for name, (count, frac, worst) in mask_disagreement(masks, info["fwd"]).items():
            assert worst <= 1e-4 and frac <= 1e-3, ("ReLU branch disagreement", u, name, count, frac, worst)
        torch.cuda.synchronize()
        rec = dict(update=u, gs_before=gs_before, gs_after=e.global_step, oracle_gs_after=o.global_step, launches=launches,
                   params_rel=rel_err(e.get_params_flat(), oracle_flat_params(o)),
                   step_rel=rel_err(e.get_params_flat().astype(np.float64) - params_before,
                                    oracle_flat_params(o) - params_before),
                   policy_loss=[scal["policy_loss"], float(info["losses"]["policy_loss"])],
                   baseline_loss=[scal["baseline_loss"], float(info["losses"]["baseline_loss"])],
                   mean_entropy=[scal["mean_entropy"], float(info["losses"]["mean_entropy"])])
        if (cfg.acktr and "clip_coeff" in info and (o.kfac.num_cov_updates > 0 or cfg.inv_init == "identity")
                and e.get_state()["inverses_valid"]):
            rec["clip_coeff"] = [scal["clip_coeff"], float(info["clip_coeff"])]
            rec["fisher_norm"] = [scal["fisher_norm"], float(info["fisher_norm"])]
            rec["precon"] = {layer: rel_err(e.layer_matrix("precon", layer).cpu().numpy(), info["precon"][layer].numpy())
                             for layer in onet.LAYERS}
            if info.get("inverted"):
                rec["inv_A"] = {layer: rel_err(e.factor("inv", "A", layer).cpu().numpy(), o.kfac.inv_a[layer].numpy())
                                for layer in onet.LAYERS}
                rec["inv_G"] = {layer: rel_err(e.factor("inv", "G", layer).cpu().numpy(), o.kfac.inv_g[layer].numpy())
                                for layer in onet.LAYERS}
        if cfg.acktr and o.kfac.num_cov_updates > 0:
            rec["sums_A"] = {f: rel_err(e.factor("sums", "A", f).cpu().numpy(), o.kfac.sum_a[f].numpy()) for f in K.A_FACTORS}
            rec["sums_G"] = {layer: rel_err(e.factor("sums", "G", layer).cpu().numpy(), o.kfac.sum_g[layer].numpy())
                             for layer in onet.LAYERS}
        if "grad_norm" in info:
            rec["grad_norm"] = [scal["grad_norm"], float(info["grad_norm"])]
        rec["lr"] = [scal["learning_rate"], float(info["lr"])]
        records.append(rec)
        if collect is not None:
            collect(e, o, rec)
    return records
