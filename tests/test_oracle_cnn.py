"""oracle/cnn.py on the CPU: the hand-written backward against torch autograd through torch.nn.functional.conv2d, the
K-FAC factors against patches built independently with unfold, and the Nature geometry against oracle/network.py +
oracle/kfac.py."""
import numpy as np
import pytest
import torch

import synth
from oracle import cnn as OC
from oracle import kfac as K
from oracle import learner as OL
from oracle import network as net

GEOMETRIES = {
    "u8_36x36x4": (36, 4, True, ((16, 8, 4), (32, 3, 1)), (64,)),
    "f32_10x10x7": (10, 7, False, ((16, 3, 1),), (128,)),
    "u8_31_stride3": (31, 3, True, ((16, 4, 2), (8, 5, 3), (8, 1, 1)), (32,)),
}


def _params(hw, c, conv, hidden, num_actions, seed=0):
    rng = np.random.default_rng(seed)
    geo = OC.conv_geometry(hw, c, conv)
    names = OC.layer_names(len(conv), len(hidden))
    p = {}
    for name, (_, cin, f, k, _, _) in zip(names, geo):
        p[name + "/weights"] = rng.standard_normal((k, k, cin, f)) / np.sqrt(k * k * cin)
        p[name + "/bias"] = 0.05 * rng.standard_normal(f)
    ins = [geo[-1][5] ** 2 * geo[-1][2]] + list(hidden)
    outs = list(hidden) + [num_actions, 1]
    ins.append(ins[-1])
    for name, k, c_out in zip(names[len(conv):], ins, outs):
        p[name + "/weights"] = rng.standard_normal((k, c_out)) / np.sqrt(k)
        p[name + "/bias"] = 0.05 * rng.standard_normal(c_out)
    return p


def _obs(rng, shape, u8):
    return rng.integers(0, 256, shape).astype(np.uint8) if u8 else rng.standard_normal(shape).astype(np.float32)


@pytest.mark.parametrize("name", list(GEOMETRIES))
def test_backward_matches_autograd_through_conv2d(name):
    hw, c, u8, conv, hidden = GEOMETRIES[name]
    params = {k: torch.tensor(v, dtype=torch.float64) for k, v in _params(hw, c, conv, hidden, 5).items()}
    geo = OC.conv_geometry(hw, c, conv)
    trunk = OC.layer_names(len(conv), len(hidden))[:-2]
    rng = np.random.default_rng(1)
    obs = _obs(rng, (6, hw, hw, c), u8)
    fwd = OC.forward(params, obs, geo, trunk, u8)
    dz = torch.tensor(rng.standard_normal((6, 5)))
    dv = torch.tensor(rng.standard_normal(6))
    grads, _ = OC.backward(params, fwd, dz, dv, geo, trunk)
    # autograd: NCHW conv2d with OIHW kernels from the HWIO variables
    leaves = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    x = torch.tensor(np.asarray(obs), dtype=torch.float64)
    x = (x / 255.0 if u8 else x).permute(0, 3, 1, 2)
    for i, (_, _, _, _, s, _) in enumerate(geo):
        w = leaves[trunk[i] + "/weights"].permute(3, 2, 0, 1)
        x = torch.relu(torch.nn.functional.conv2d(x, w, leaves[trunk[i] + "/bias"], stride=s))
    x = x.permute(0, 2, 3, 1).reshape(6, -1)
    for layer in trunk[len(geo):]:
        x = torch.relu(x @ leaves[layer + "/weights"] + leaves[layer + "/bias"])
    logits = x @ leaves["fc_policy/weights"] + leaves["fc_policy/bias"]
    value = (x @ leaves["fc_baseline/weights"] + leaves["fc_baseline/bias"])[:, 0]
    torch.testing.assert_close(logits, fwd["logits"], rtol=1e-12, atol=1e-12)
    ((logits * dz).sum() + (value * dv).sum()).backward()
    for layer in OC.layer_names(len(conv), len(hidden)):
        w, b = leaves[layer + "/weights"].grad, leaves[layer + "/bias"].grad
        want = torch.cat([w.reshape(-1, w.shape[-1]), b.reshape(1, -1)], 0)
        torch.testing.assert_close(grads[layer], want, rtol=1e-10, atol=1e-12)


@pytest.mark.parametrize("name", list(GEOMETRIES))
def test_factors_match_unfold_patches(name):
    hw, c, u8, conv, hidden = GEOMETRIES[name]
    params = _params(hw, c, conv, hidden, 4)
    cfg = K.KfacConfig(num_cold_updates=0, invert_every=1)
    o = OC.CNNOracle(params, hw, c, conv, len(hidden), obs_u8=u8, cfg=cfg)
    rng = np.random.default_rng(2)
    e, t = 3, 2
    batch = dict(observations=_obs(rng, (e, t, hw, hw, c), u8), bootstrap_observations=_obs(rng, (e, hw, hw, c), u8),
                 actions=rng.integers(0, 4, (e, t)), rewards=rng.standard_normal((e, t)), terminals=rng.random((e, t)) < 0.2)
    y, eps = synth.fisher_samples(3, e * t, num_actions=4)
    info = o.compute(batch, y, eps)
    x = torch.tensor(np.asarray(batch["observations"]).reshape(e * t, hw, hw, c), dtype=torch.float64)
    x = (x / 255.0 if u8 else x).permute(0, 3, 1, 2)
    for i, (_, cin, f, k, s, oh) in enumerate(o.geo):
        name_i = o.layers[i]
        cols = torch.nn.functional.unfold(x, k, stride=s)                   # [n, c*k*k, L], order (c, kh, kw)
        cols = cols.reshape(e * t, cin, k, k, oh * oh).permute(0, 4, 2, 3, 1).reshape(e * t * oh * oh, k * k * cin)
        torch.testing.assert_close(info["new_a"][name_i], K.input_factor(cols), rtol=1e-10, atol=1e-12)
        assert info["new_g"][name_i].shape == (f, f)
        assert o.locations[name_i] == oh * oh
        pre = info["fwd"]["pre"][name_i]
        x = torch.relu(pre).reshape(e * t, oh, oh, f).permute(0, 3, 1, 2)
    fisher_g = o._backward(info["fwd"], *net.fisher_output_grads(info["fwd"]["logits"], info["fwd"]["value"], y, eps),
                           None)[1]
    for layer in o.layers[:len(o.geo)]:
        g = fisher_g[layer]
        torch.testing.assert_close(info["new_g"][layer], g.T @ g / g.shape[0], rtol=1e-10, atol=1e-14)


def test_nature_geometry_reproduces_the_atari_oracle():
    """84x84x4 uint8, conv (32,8,4),(64,4,2),(32,3,1), fc4 512: three ACKTR updates (cold, covariance, refresh + K-FAC) of
    CNNOracle and oracle.learner.OracleLearner agree to fp64 rounding."""
    params = net.perturbed_params(4, 32, seed=0)
    cfg = K.KfacConfig(num_cold_updates=1, invert_every=1, decay_steps=1e7 / 20)
    a = OL.OracleLearner(params, 4, 32, acktr=True, cfg=cfg, dtype=torch.float64)
    b = OC.CNNOracle(params, 84, 4, ((32, 8, 4), (64, 4, 2), (32, 3, 1)), 1, obs_u8=True, acktr=True, cfg=cfg)
    assert b.layers == net.LAYERS and b.locations == K.TRUE_LOCATIONS
    for u in range(3):
        batch = synth.rollout(10 + u, 4, 5, 4, obs_kind="uniform")
        y, eps = synth.fisher_samples(20 + u, 20, num_actions=4)
        ia = a.update(batch, y, eps)
        ib = b.update(batch, y, eps)
        torch.testing.assert_close(ib["fwd"]["logits"], ia["fwd"]["logits"], rtol=1e-12, atol=1e-14)
        for layer in net.LAYERS:
            torch.testing.assert_close(ib["grads"][layer], ia["grads"][layer], rtol=1e-10, atol=1e-14)
        if "new_a" in ib:
            for f in K.A_FACTORS:
                torch.testing.assert_close(ib["new_a"][f], ia["new_a"][f], rtol=1e-10, atol=1e-14)
        np.testing.assert_allclose(b.flat_params(), np.concatenate(
            [net.join_vmat(layer, a.params).detach().numpy().ravel() for layer in net.LAYERS]), rtol=1e-10, atol=1e-13)
    assert b.global_step == a.global_step
