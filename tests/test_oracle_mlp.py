"""The fully connected oracle (oracle/mlp.py) against independent derivations: the Kronecker identity behind K-FAC
preconditioning of fc blocks, torch autograd and finite differences of the A2C loss."""
import numpy as np
import torch

from oracle import kfac as K
from oracle import mlp as OM
from oracle import network as net


def _params(d, hidden, a, seed=0):
    rng = np.random.default_rng(seed)
    dims = [d] + list(hidden)
    p = {}
    for name, k, c in zip(OM.layer_names(len(hidden)), dims + [dims[-1]], list(hidden) + [a, 1]):
        p[name + "/weights"] = rng.standard_normal((k, c)) / np.sqrt(k)
        p[name + "/bias"] = 0.1 * rng.standard_normal(c)
    return {k: torch.tensor(v, dtype=torch.float64) for k, v in p.items()}


def _batch(e, t, d, a, seed=0):
    rng = np.random.default_rng(seed)
    return dict(observations=rng.standard_normal((e, t, d)), bootstrap_observations=rng.standard_normal((e, d)),
                actions=rng.integers(0, a, (e, t)), rewards=rng.standard_normal((e, t)),
                terminals=rng.random((e, t)) < 0.2)


def test_kronecker_identity_for_fc_blocks():
    """(G (x) A) vec(U) = vec(A U G) for every fc block of the oracle: the preconditioned block A^-1 V G^-1 solves the
    Kronecker-factored system with the factors the oracle builds."""
    hidden = (16, 8)
    params = _params(5, hidden, 3)
    o = OM.MLPOracle({k: v.numpy() for k, v in params.items()}, len(hidden), cfg=K.KfacConfig(damping=0.01))
    b = _batch(3, 4, 5, 3)
    y = np.random.default_rng(1).integers(0, 3, 12)
    eps = np.random.default_rng(2).standard_normal(12)
    info = o.compute(b, y, eps)
    o.update_covs(info["new_a"], info["new_g"])
    o.update_inverses()
    precon = o.precondition(info["grads"])
    for layer in o.layers:
        a = torch.linalg.inv(o.inv_a[layer])
        g = torch.linalg.inv(o.inv_g[layer])
        u = precon[layer]
        lhs = torch.kron(g, a) @ u.T.reshape(-1)            # column-major vec
        rhs = info["grads"][layer].T.reshape(-1)
        assert torch.allclose(lhs, rhs, rtol=1e-9, atol=1e-10), layer
        assert a.shape[0] == u.shape[0] and g.shape[0] == u.shape[1]


def test_gradients_against_autograd_and_finite_differences():
    hidden = (16, 8)
    params = _params(7, hidden, 4, seed=3)
    b = _batch(2, 5, 7, 4, seed=4)
    o = OM.MLPOracle({k: v.numpy() for k, v in params.items()}, len(hidden), acktr=False)
    info = o.compute(b, need_fisher=False)
    targets = info["targets"].detach()
    n = 10
    obs = b["observations"].reshape(n, 7)
    actions = b["actions"].reshape(n)

    adv0 = (targets - info["fwd"]["value"]).detach()

    def loss_of(p):     # objectives.py:128-154 with the advantage held at its value (tf.stop_gradient)
        fwd = OM.forward(p, obs, o.hidden)
        logp_all = torch.log_softmax(fwd["logits"], -1)
        logp = logp_all[torch.arange(n), torch.as_tensor(actions).long()]
        entropy = -(logp_all.exp() * logp_all).sum(-1).mean()
        return -((adv0 * logp).mean() + 0.01 * entropy) + 0.5 * ((targets - fwd["value"]) ** 2 / 2).mean()

    leaf = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    fwd = OM.forward(leaf, obs, o.hidden)
    net.a2c_loss(fwd["logits"], fwd["value"], actions, targets)["loss"].backward()
    for layer in o.layers:
        want = torch.cat([leaf[layer + "/weights"].grad, leaf[layer + "/bias"].grad.reshape(1, -1)], 0)
        assert torch.allclose(info["grads"][layer], want, rtol=1e-10, atol=1e-12), layer
    # central differences on a few entries of every variable
    rng = np.random.default_rng(5)
    for key in params:
        flat = params[key].reshape(-1)
        for idx in rng.choice(flat.numel(), size=min(3, flat.numel()), replace=False):
            h = 1e-6
            plus = {k: v.clone() for k, v in params.items()}
            minus = {k: v.clone() for k, v in params.items()}
            plus[key].reshape(-1)[idx] += h
            minus[key].reshape(-1)[idx] -= h
            fd = (float(loss_of(plus)) - float(loss_of(minus))) / (2 * h)
            layer, kind = key.split("/")
            g = info["grads"][layer]
            got = float(g[-1].reshape(-1)[idx]) if kind == "bias" else float(g[:-1].reshape(-1)[idx])
            assert abs(got - fd) <= 1e-6 * max(1.0, abs(fd)), (key, idx, got, fd)


def test_factors_are_the_fc_block_statistics():
    hidden = (8,)
    params = _params(4, hidden, 2, seed=6)
    o = OM.MLPOracle({k: v.numpy() for k, v in params.items()}, 1, cfg=K.KfacConfig())
    b = _batch(2, 3, 4, 2, seed=7)
    info = o.compute(b, np.zeros(6, np.int64), np.zeros(6))
    x = torch.as_tensor(b["observations"].reshape(6, 4))
    xh = torch.cat([x, torch.ones(6, 1, dtype=x.dtype)], 1)
    assert torch.allclose(info["new_a"]["fc1"], xh.T @ xh / 6)
    assert set(info["new_a"]) == {"fc1", "heads"} and set(info["new_g"]) == set(o.layers)
    assert info["new_g"]["fc_baseline"].shape == (1, 1)
