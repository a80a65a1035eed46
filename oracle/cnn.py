"""Oracle for the convolutional learner (actorcritic_b200.cnn.CNNModel, csrc/mlp.cu `acx_cnn_*`): torch-CPU, dtype
selectable (float64 for parity, float32 on all host threads as the CPU baseline of tools/cnn_bench.py).

The model is conv1 .. convK (VALID, ReLU; HWIO kernels) on square NHWC images, the (h, w, c) flatten, fc(K+1) .. fc(K+L)
(ReLU) and the heads fc_policy / fc_baseline on the last hidden layer.  Convolutions are explicit im2col + matmul
(oracle.network.im2col / col2im, patch order (kh, kw, c_in)), so that the patch matrices the K-FAC input factors need fall
out.  The optimizer side is oracle.mlp.MLPOracle with the true VALID location count T = oh * ow of each conv block
(damping / T, preconditioned block / T; oracle.kfac TRUE_LOCATIONS at the Nature geometry).  Parameters: conv kernels HWIO
in and [k*k*c_in, filters] (the [K+1, C] block layout) inside the learner; forward / backward accept either.
"""

import numpy as np
import torch

from . import kfac as K
from . import mlp as OM
from . import network as net


def layer_names(num_conv, num_hidden):
    return (tuple("conv%d" % (i + 1) for i in range(num_conv))
            + tuple("fc%d" % (num_conv + i + 1) for i in range(num_hidden)) + ("fc_policy", "fc_baseline"))


def conv_geometry(obs_hw, obs_channels, conv_layers):
    """[(hw_in, c_in, filters, kernel, stride, hw_out)] per conv layer."""
    out, hw, c = [], int(obs_hw), int(obs_channels)
    for f, k, s in conv_layers:
        o = (hw - int(k)) // int(s) + 1
        out.append((hw, c, int(f), int(k), int(s), o))
        hw, c = o, int(f)
    return out


def forward(params, obs, geo, trunk, obs_u8):
    """obs [R, H, H, C] (uint8: scaled by 1/255) -> dict(inputs {layer: patches or x}, pre {trunk layer: pre-activation
    [R * T, C]}, logits, value, rows)."""
    dtype = params[trunk[0] + "/weights"].dtype
    x = torch.as_tensor(np.asarray(obs)).to(dtype)
    if obs_u8:
        x = x / 255.0
    r = x.shape[0]
    inputs, pre = {}, {}
    a = x
    for name, (_, c, f, k, s, _) in zip(trunk, geo):
        p, oh, ow = net.im2col(a, k, s)
        inputs[name] = p
        pre[name] = p @ params[name + "/weights"].reshape(k * k * c, f) + params[name + "/bias"]
        a = torch.relu(pre[name]).reshape(r, oh, ow, f)
    a = a.reshape(r, -1)                                              # nn.flatten: (h, w, c)
    for name in trunk[len(geo):]:
        inputs[name] = a
        pre[name] = a @ params[name + "/weights"] + params[name + "/bias"]
        a = torch.relu(pre[name])
    inputs["fc_policy"] = inputs["fc_baseline"] = a
    logits = a @ params["fc_policy/weights"] + params["fc_policy/bias"]
    value = (a @ params["fc_baseline/weights"] + params["fc_baseline/bias"])[:, 0]
    return dict(inputs=inputs, pre=pre, logits=logits, value=value, rows=r)


def backward(params, fwd, dlogits, dvalue, geo, trunk, masks=None):
    """Hand-derived backward -> (grads {layer: [K+1, C]}, pre-activation gradients {trunk layer: [R * T, C]}).  masks:
    {trunk layer: bool, any shape of R * T * C elements} replacing `pre > 0` (the engine's, as oracle.network.backward)."""
    grads, g = {}, {}
    x = fwd["inputs"]["fc_policy"]
    g["fc_policy"], g["fc_baseline"] = dlogits, dvalue[:, None]
    for name in ("fc_policy", "fc_baseline"):
        grads[name] = torch.cat([x.T @ g[name], g[name].sum(0, keepdim=True)], 0)
    d = dlogits @ params["fc_policy/weights"].T + g["fc_baseline"] @ params["fc_baseline/weights"].T
    r = fwd["rows"]
    for i in reversed(range(len(trunk))):
        name = trunk[i]
        pre = fwd["pre"][name]
        mask = (pre > 0) if masks is None or name not in masks else torch.as_tensor(masks[name]).reshape(pre.shape)
        gl = d.reshape(pre.shape) * mask
        g[name] = gl
        grads[name] = torch.cat([fwd["inputs"][name].T @ gl, gl.sum(0, keepdim=True)], 0)
        if i == 0:
            break
        w = params[name + "/weights"]
        d = gl @ w.reshape(-1, w.shape[-1]).T
        if i < len(geo):                                             # conv: patch gradients -> input gradient
            hw, c, _, k, s, _ = geo[i]
            d = net.col2im(d, r, hw, hw, c, k, s).reshape(r * hw * hw, c)
    return grads, g


class CNNOracle(OM.MLPOracle):
    """One learner (ACKTR or A2C, as MLPOracle) on a convolutional model.

    MLPOracle's optimizer steps (cold momentum, EMA, KL clip, momentum, RMSProp, the schedule) are used as they are.  It
    keeps conv kernels as [k*k*c_in, filters] matrices (the [K+1, C] block layout), and this class adds the convolutional
    forward / backward, the factors over every output location and the location counts T of the conv blocks (damping
    lambda / T, preconditioned block / T)."""

    def __init__(self, params, obs_hw, obs_channels, conv_layers, num_hidden, obs_u8=True, **kw):
        self.geo = conv_geometry(obs_hw, obs_channels, conv_layers)
        self.obs_shape = (int(obs_hw), int(obs_hw), int(obs_channels))
        self.obs_u8 = bool(obs_u8)
        names = layer_names(len(self.geo), num_hidden)
        trunk = len(names) - 2
        # MLPOracle names the blocks of a trunk fc1 ..: build its state from the same parameters under those names, then
        # give every per-block entry the model's own name
        to_mlp = dict(zip(names, OM.layer_names(trunk)))
        flat = {}
        for key, v in params.items():
            layer, kind = key.split("/")
            v = np.asarray(v)
            flat[to_mlp[layer] + "/" + kind] = v.reshape(-1, v.shape[-1]) if kind == "weights" else v
        super().__init__(flat, trunk, **kw)
        back = {m: n for n, m in to_mlp.items()}
        self.params = {back[k.split("/")[0]] + "/" + k.split("/")[1]: v for k, v in self.params.items()}
        for attr in ("sum_a", "sum_g", "inv_a", "inv_g", "velocity", "cold_accum", "rms"):
            if hasattr(self, attr):
                setattr(self, attr, {back.get(k, k): v for k, v in getattr(self, attr).items()})
        self.layers, self.hidden = names, names[:trunk]
        self.locations = {l: 1 for l in names}
        self.locations.update({names[i]: g[5] * g[5] for i, g in enumerate(self.geo)})

    def _forward(self, obs_rows):
        return forward(self.params, obs_rows, self.geo, self.hidden, self.obs_u8)

    def _backward(self, fwd, dlogits, dvalue, masks):
        return backward(self.params, fwd, dlogits, dvalue, self.geo, self.hidden, masks)

    def compute(self, batch, y_hat=None, eps=None, need_fisher=True, masks=None):
        """MLPOracle.compute on image rows: forward, targets, loss, gradients and (need_fisher) the batch factors."""
        obs = np.asarray(batch["observations"])
        e_count, t_count = obs.shape[:2]
        n = e_count * t_count
        fwd = self._forward(obs.reshape((n,) + self.obs_shape))
        boot = self._forward(np.asarray(batch["bootstrap_observations"]).reshape((e_count,) + self.obs_shape))
        targets = net.targets_torch(batch["rewards"], batch["terminals"], boot["value"], self.gamma).reshape(n)
        actions = np.asarray(batch["actions"]).reshape(n)
        losses = net.a2c_loss(fwd["logits"], fwd["value"], actions, targets, self.beta, self.value_weight)
        dz, dv = net.output_grads(fwd["logits"], fwd["value"], actions, targets, self.beta, self.value_weight)
        grads, pre_grads = self._backward(fwd, dz, dv, masks)
        out = dict(fwd=fwd, bootstrap_values=boot["value"], targets=targets, losses=losses, grads=grads, pre_grads=pre_grads)
        if need_fisher:
            fz, fv = net.fisher_output_grads(fwd["logits"], fwd["value"], y_hat, eps)
            _, fisher_pre = self._backward(fwd, fz, fv, masks)
            out["new_a"], out["new_g"] = OM.batch_factors(fwd, fisher_pre, self.layers)
        return out

    def update_inverses(self):
        """pi-damped inverses with damping lambda / T (oracle.kfac.KfacState.dampings)."""
        for l in self.layers:
            sa, sg, debias = self.sum_a[OM.factor_of(l)], self.sum_g[l], self._debias()
            damp_a, damp_g = K.pi_dampings(sa * debias, sg * debias, self.cfg.damping / self.locations[l])
            self.inv_a[l] = K.damped_inverse(sa, debias, damp_a)
            self.inv_g[l] = K.damped_inverse(sg, debias, damp_g)

    def precondition(self, grads):
        """U = A^-1 V G^-1 / T with the stored inverses."""
        return {l: u / self.locations[l] for l, u in super().precondition(grads).items()}
