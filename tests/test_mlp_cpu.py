"""MLPModel on the CPU: construction checks, variables, K-FAC registration (no device needed)."""
import numpy as np
import pytest

from actorcritic_b200 import kfac, spaces
from actorcritic_b200.mlp import MLPModel


def _box(shape, dtype=np.float32):
    return spaces.Box(low=0, high=1, shape=shape, dtype=dtype)


@pytest.mark.parametrize("obs_space, act_space, hidden, error", [
    (_box((8,), np.uint8), spaces.Discrete(4), (64,), TypeError),          # not float32
    (spaces.Discrete(3), spaces.Discrete(4), (64,), TypeError),            # not a Box
    (_box((8,)), _box((2,)), (64,), TypeError),                            # continuous actions
    (_box((2049,)), spaces.Discrete(4), (64,), ValueError),
    (_box((8,)), spaces.Discrete(32), (64,), ValueError),
    (_box((8,)), spaces.Discrete(4), (), ValueError),
    (_box((8,)), spaces.Discrete(4), (8, 8, 8, 8, 8), ValueError),
    (_box((8,)), spaces.Discrete(4), (60,), ValueError),
    (_box((8,)), spaces.Discrete(4), (1032,), ValueError),
])
def test_construction_errors(obs_space, act_space, hidden, error):
    with pytest.raises(error):
        MLPModel(obs_space, act_space, hidden_sizes=hidden)


def test_variables_shapes_and_gains():
    model = MLPModel(_box((3, 4)), spaces.Discrete(5), hidden_sizes=(64, 32, 16), random_seed=1)
    v = model.get_variables()
    assert list(v) == ["fc1/weights", "fc1/bias", "fc2/weights", "fc2/bias", "fc3/weights", "fc3/bias",
                       "fc_policy/weights", "fc_policy/bias", "fc_baseline/weights", "fc_baseline/bias"]
    shapes = {k: a.shape for k, a in v.items()}
    assert shapes["fc1/weights"] == (12, 64) and shapes["fc2/weights"] == (64, 32) and shapes["fc3/weights"] == (32, 16)
    assert shapes["fc_policy/weights"] == (16, 5) and shapes["fc_baseline/weights"] == (16, 1)
    for k, a in v.items():
        assert a.dtype == np.float32
        if k.endswith("/bias"):
            assert not a.any()
    # orthogonal with gain g: the smaller Gram matrix of W / g is the identity
    for layer, gain in (("fc1", 2 ** 0.5), ("fc2", 2 ** 0.5), ("fc3", 2 ** 0.5), ("fc_policy", 0.01), ("fc_baseline", 1.0)):
        w = v[layer + "/weights"].astype(np.float64) / gain
        gram = w.T @ w if w.shape[0] >= w.shape[1] else w @ w.T
        np.testing.assert_allclose(gram, np.eye(gram.shape[0]), atol=1e-5)
    again = MLPModel(_box((3, 4)), spaces.Discrete(5), hidden_sizes=(64, 32, 16), random_seed=1).get_variables()
    assert all(np.array_equal(again[k], v[k]) for k in v)
    assert model.observations_placeholder.shape == (None, None, 3, 4)


def test_set_variables_checks_shapes():
    model = MLPModel(_box((6,)), spaces.Discrete(2), hidden_sizes=(8,), random_seed=0)
    v = model.get_variables()
    v["fc1/weights"] = v["fc1/weights"] + 1.0
    model.set_variables(v)
    assert np.array_equal(model.get_variables()["fc1/weights"], v["fc1/weights"])
    v["fc_policy/weights"] = np.zeros((8, 3), np.float32)
    with pytest.raises(ValueError):
        model.set_variables(v)


@pytest.mark.parametrize("hidden", [(64,), (64, 40), (32, 32, 32, 32)])
def test_register_layers_and_factor_counts(hidden):
    model = MLPModel(_box((17,)), spaces.Discrete(5), hidden_sizes=hidden)
    lc = kfac.LayerCollection()
    model.register_layers(lc)
    model.register_predictive_distributions(lc)
    assert not lc.conv2d and len(lc.fully_connected) == len(hidden) + 2
    names = [rec["params"][0].split("/")[0] for rec in lc.fully_connected]
    assert names == ["fc%d" % (i + 1) for i in range(len(hidden))] + ["fc_policy", "fc_baseline"]
    heads = lc.fully_connected[-2:]
    assert heads[0]["inputs"] is heads[1]["inputs"]
    assert len(lc.input_factor_groups()) == len(hidden) + 1
    opt = kfac.KfacOptimizer(learning_rate=0.25, layer_collection=lc)
    cov, inv = opt.make_vars_and_create_op_thunks()
    assert len(cov) == len(inv) == (len(hidden) + 1) + (len(hidden) + 2)
    assert len(lc.categorical) == 1 and len(lc.normal) == 1
