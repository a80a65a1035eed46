"""Oracle for the fully connected learner (actorcritic_b200.mlp.MLPModel, csrc/mlp.cu): torch-CPU, dtype selectable
(float64 for parity, float32 on all host threads as the CPU baseline of tools/mlp_bench.py).

The same update as oracle/learner.py for an arbitrary stack of fully connected ReLU layers fc1 .. fcL plus the heads
fc_policy / fc_baseline reading the last hidden layer: forward, n-step targets, the A2C loss and its gradients, the
Fisher-sample output gradients, the input / output factors of every fully connected block (the heads share one input
factor), EMA with zero-debias, pi-damping, inverses, preconditioning with T~ = 1, KL clip, momentum, and the cold
momentum / A2C RMSProp steps, on the schedule of kfac_utils.py:38-53 (oracle.kfac.schedule_events).
"""
import math

import numpy as np
import torch

from . import kfac as K
from . import network as net


def layer_names(num_hidden):
    return tuple("fc%d" % (i + 1) for i in range(num_hidden)) + ("fc_policy", "fc_baseline")


def factor_of(layer):
    """Input factor of a block: its own, the two heads share "heads"."""
    return "heads" if layer in ("fc_policy", "fc_baseline") else layer


def vmat(params, layer):
    """[K+1, C]: weights [in, out] then the bias row."""
    return torch.cat([params[layer + "/weights"], params[layer + "/bias"].reshape(1, -1)], 0)


def set_vmat(params, layer, v):
    params[layer + "/weights"], params[layer + "/bias"] = v[:-1].clone(), v[-1].clone()


def forward(params, obs, hidden):
    """obs [R, D] -> dict(inputs {layer: x}, pre {hidden layer: pre-activation}, logits [R, A], value [R])."""
    x = torch.as_tensor(np.asarray(obs)).to(params[hidden[0] + "/weights"].dtype)
    inputs, pre = {}, {}
    for name in hidden:
        inputs[name] = x
        pre[name] = x @ params[name + "/weights"] + params[name + "/bias"]
        x = torch.relu(pre[name])
    inputs["fc_policy"] = inputs["fc_baseline"] = x
    logits = x @ params["fc_policy/weights"] + params["fc_policy/bias"]
    value = (x @ params["fc_baseline/weights"] + params["fc_baseline/bias"])[:, 0]
    return dict(inputs=inputs, pre=pre, logits=logits, value=value)


def backward(params, fwd, dlogits, dvalue, hidden, masks=None):
    """Hand-derived backward for output gradients (dlogits [R, A], dvalue [R]) -> (grads {layer: [K+1, C]},
    pre-activation gradients {layer: [R, C]}).  masks: {hidden layer: bool [R, C]} replacing `pre > 0` (the parity tests
    pass the engine's, see network.backward)."""
    grads, g = {}, {}
    x = fwd["inputs"]["fc_policy"]
    g["fc_policy"], g["fc_baseline"] = dlogits, dvalue[:, None]
    for name in ("fc_policy", "fc_baseline"):
        grads[name] = torch.cat([x.T @ g[name], g[name].sum(0, keepdim=True)], 0)
    d = dlogits @ params["fc_policy/weights"].T + g["fc_baseline"] @ params["fc_baseline/weights"].T
    for name in reversed(hidden):
        pre = fwd["pre"][name]
        mask = (pre > 0) if masks is None or name not in masks else torch.as_tensor(masks[name]).reshape(pre.shape)
        gl = d * mask
        g[name] = gl
        grads[name] = torch.cat([fwd["inputs"][name].T @ gl, gl.sum(0, keepdim=True)], 0)
        d = gl @ params[name + "/weights"].T
    return grads, g


def batch_factors(fwd, fisher_pre_grads, layers):
    """New covariance contributions of one batch (train rows): A per input factor, G per block."""
    a = {factor_of(l): K.input_factor(fwd["inputs"][l]) for l in layers}
    g = {l: K.output_factor(fisher_pre_grads[l]) for l in layers}
    return a, g


class MLPOracle:
    """One learner (ACKTR with a kfac.KfacConfig, or A2C with a learner.A2CConfig) on a fully connected model."""

    def __init__(self, params, num_hidden, acktr=True, cfg=None, gamma=0.99, beta=0.01, value_weight=0.5,
                 dtype=torch.float64):
        self.dtype = dtype
        self.hidden = layer_names(num_hidden)[:num_hidden]
        self.layers = layer_names(num_hidden)
        self.params = {k: torch.tensor(np.asarray(v), dtype=dtype) for k, v in params.items()}
        self.acktr, self.cfg = acktr, cfg
        self.gamma, self.beta, self.value_weight = float(np.float32(gamma)), beta, value_weight   # gamma as the fp32 the engine gets
        self.global_step = 0
        zeros = {l: torch.zeros_like(vmat(self.params, l)) for l in self.layers}
        if acktr:
            dims_a = {factor_of(l): self.params[l + "/weights"].shape[0] + 1 for l in self.layers}
            self.sum_a = {f: torch.zeros((d, d), dtype=dtype) for f, d in dims_a.items()}
            self.sum_g = {l: torch.zeros((v.shape[1], v.shape[1]), dtype=dtype) for l, v in zeros.items()}
            self.inv_a = {l: torch.zeros_like(self.sum_a[factor_of(l)]) for l in self.layers}
            self.inv_g = {l: torch.zeros_like(self.sum_g[l]) for l in self.layers}
            self.num_cov_updates = 0
            self.velocity = dict(zeros)
            self.cold_accum = {l: v.clone() for l, v in zeros.items()}
        else:
            self.rms = {l: torch.ones_like(v) for l, v in zeros.items()}

    # ------------------------------------------------------------------ gradient side
    def compute(self, batch, y_hat=None, eps=None, need_fisher=True, masks=None):
        obs = np.asarray(batch["observations"])
        e_count, t_count = obs.shape[:2]
        n = e_count * t_count
        fwd = forward(self.params, obs.reshape(n, -1), self.hidden)
        boot = forward(self.params, np.asarray(batch["bootstrap_observations"]).reshape(e_count, -1), self.hidden)
        targets = net.targets_torch(batch["rewards"], batch["terminals"], boot["value"], self.gamma).reshape(n)
        actions = np.asarray(batch["actions"]).reshape(n)
        losses = net.a2c_loss(fwd["logits"], fwd["value"], actions, targets, self.beta, self.value_weight)
        dz, dv = net.output_grads(fwd["logits"], fwd["value"], actions, targets, self.beta, self.value_weight)
        grads, pre_grads = backward(self.params, fwd, dz, dv, self.hidden, masks)
        out = dict(fwd=fwd, bootstrap_values=boot["value"], targets=targets, losses=losses, grads=grads, pre_grads=pre_grads)
        if need_fisher:
            fz, fv = net.fisher_output_grads(fwd["logits"], fwd["value"], y_hat, eps)
            _, fisher_pre = backward(self.params, fwd, fz, fv, self.hidden, masks)
            out["new_a"], out["new_g"] = batch_factors(fwd, fisher_pre, self.layers)
        return out

    # ------------------------------------------------------------------ K-FAC
    def _debias(self):
        return 1.0 if self.num_cov_updates == 0 else 1.0 / (1.0 - self.cfg.cov_ema_decay ** self.num_cov_updates)

    def update_covs(self, new_a, new_g):
        d = self.cfg.cov_ema_decay
        for k in self.sum_a:
            self.sum_a[k] = d * self.sum_a[k] + (1 - d) * new_a[k]
        for k in self.sum_g:
            self.sum_g[k] = d * self.sum_g[k] + (1 - d) * new_g[k]
        self.num_cov_updates += 1

    def update_inverses(self):
        """pi-damped inverses (damping / T~ with T~ = 1 for fully connected blocks)."""
        for l in self.layers:
            a = self.sum_a[factor_of(l)] * self._debias()
            g = self.sum_g[l] * self._debias()
            tr_a, tr_g = float(torch.trace(a)) / a.shape[0], float(torch.trace(g)) / g.shape[0]
            pi = math.sqrt(tr_a / tr_g) if tr_a > 0 and tr_g > 0 else 1.0
            root = math.sqrt(self.cfg.damping)
            self.inv_a[l] = torch.linalg.inv(a + pi * root * torch.eye(a.shape[0], dtype=self.dtype))
            self.inv_g[l] = torch.linalg.inv(g + root / pi * torch.eye(g.shape[0], dtype=self.dtype))

    def precondition(self, grads):
        return {l: self.inv_a[l] @ grads[l] @ self.inv_g[l] for l in self.layers}

    def learning_rate(self):
        c = self.cfg
        return K.linear_decay(c.learning_rate_start, c.learning_rate_end, self.global_step, c.decay_steps)

    # ------------------------------------------------------------------ one update
    def update(self, batch, y_hat=None, eps=None, masks=None):
        if not self.acktr:
            return self._update_a2c(batch, masks)
        cfg = self.cfg
        plan = K.schedule_events(self.global_step, cfg.num_cold_updates, cfg.invert_every)
        info = self.compute(batch, y_hat, eps, need_fisher=not plan["cold"], masks=masks)
        grads = info["grads"]
        lr = self.learning_rate()
        if plan["cold"]:                                             # kfac_utils.py:42-43
            clipped, norm = K.clip_by_global_norm(grads, cfg.clip_norm)
            for l in self.layers:
                self.cold_accum[l] = cfg.cold_momentum * self.cold_accum[l] + clipped[l]
                set_vmat(self.params, l, vmat(self.params, l) - cfg.cold_learning_rate * self.cold_accum[l])
            self.global_step += 1
            info["grad_norm"] = norm
        else:                                                        # :44
            self.update_covs(info["new_a"], info["new_g"])
        if plan["inv"]:                                              # :47-50
            self.update_inverses()
            info["inverted"] = True
        # :52-53 always: precondition with the stored inverses, KL clip, momentum, apply
        precon = self.precondition(grads)
        s = sum(float((grads[l] * precon[l]).sum()) for l in self.layers)
        coeff = 1.0 if s <= 0.0 else min(1.0, math.sqrt(cfg.norm_constraint / (lr * lr * s)))
        for l in self.layers:
            self.velocity[l] = cfg.momentum * self.velocity[l] + coeff * precon[l]
            set_vmat(self.params, l, vmat(self.params, l) - lr * self.velocity[l])
        self.global_step += 1
        assert self.global_step == plan["gs_after"]
        info.update(clip_coeff=coeff, fisher_norm=s, precon=precon, lr=lr)
        return info

    def _update_a2c(self, batch, masks=None):
        cfg = self.cfg
        info = self.compute(batch, need_fisher=False, masks=masks)
        lr = self.learning_rate()
        clipped, norm = K.clip_by_global_norm(info["grads"], cfg.clip_norm)
        for l in self.layers:
            g = clipped[l]
            self.rms[l] = cfg.rms_decay * self.rms[l] + (1 - cfg.rms_decay) * g * g
            set_vmat(self.params, l, vmat(self.params, l) - lr * g / torch.sqrt(self.rms[l] + cfg.rms_epsilon))
        self.global_step += 1
        info.update(grad_norm=norm, lr=lr)
        return info

    def flat_params(self):
        return np.concatenate([vmat(self.params, l).detach().numpy().ravel() for l in self.layers])
