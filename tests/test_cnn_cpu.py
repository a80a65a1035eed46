"""CNNModel on the CPU: construction limits, variables and initial gains, K-FAC registration (no device needed)."""
import numpy as np
import pytest

from actorcritic_b200 import engine as eng
from actorcritic_b200 import kfac, spaces
from actorcritic_b200.cnn import CNNModel


def _img(hw=36, c=4, dtype=np.uint8, shape=None):
    return spaces.Box(low=0, high=255 if dtype == np.uint8 else 1, shape=shape or (hw, hw, c), dtype=dtype)


@pytest.mark.parametrize("obs_space, act_space, kw, error, message", [
    (spaces.Discrete(3), spaces.Discrete(4), {}, TypeError, "Box observation space"),
    (_img(dtype=np.float64), spaces.Discrete(4), {}, TypeError, "uint8 or float32"),
    (_img(), _img(shape=(2,), dtype=np.float32), {}, TypeError, "Unsupported space"),
    (_img(shape=(36, 30, 4)), spaces.Discrete(4), {}, ValueError, "square images"),
    (_img(shape=(36 * 36 * 4,)), spaces.Discrete(4), {}, ValueError, "square images"),
    (_img(hw=3), spaces.Discrete(4), dict(conv_layers=((8, 1, 1),)), ValueError, "image size H"),
    (_img(hw=129), spaces.Discrete(4), dict(conv_layers=((8, 8, 4),)), ValueError, "image size H"),
    (_img(c=17), spaces.Discrete(4), dict(conv_layers=((8, 3, 1),)), ValueError, "image channels C"),
    (_img(), spaces.Discrete(32), {}, ValueError, "1 to 31 actions"),
    (_img(), spaces.Discrete(4), dict(conv_layers=()), ValueError, "1 to 3 layers"),
    (_img(), spaces.Discrete(4), dict(conv_layers=((8, 3, 1),) * 4, hidden_sizes=(64,)), ValueError, "1 to 3 layers"),
    (_img(), spaces.Discrete(4), dict(conv_layers=((8, 3, 1), (8, 3, 1)), hidden_sizes=(64, 64, 64)), ValueError,
     "at most 4 conv and fully connected"),
    (_img(), spaces.Discrete(4), dict(conv_layers=((12, 8, 4),)), ValueError, "filters must be a multiple of 8"),
    (_img(), spaces.Discrete(4), dict(conv_layers=((136, 8, 4),)), ValueError, "filters must be a multiple of 8"),
    (_img(), spaces.Discrete(4), dict(conv_layers=((16, 9, 4),)), ValueError, "kernel must be in"),
    (_img(), spaces.Discrete(4), dict(conv_layers=((16, 0, 1),)), ValueError, "kernel must be in"),
    (_img(), spaces.Discrete(4), dict(conv_layers=((16, 3, 4),)), ValueError, "stride must be in"),
    (_img(), spaces.Discrete(4), dict(conv_layers=((16, 8, 5),)), ValueError, "stride must be in"),
    (_img(hw=8), spaces.Discrete(4), dict(conv_layers=((16, 4, 2), (16, 4, 1))), ValueError, "does not fit"),
    (_img(c=16), spaces.Discrete(4), dict(conv_layers=((128, 2, 2), (32, 5, 1))), ValueError, "conv2: input factor"),
    (_img(hw=64, c=3), spaces.Discrete(4), dict(conv_layers=((32, 8, 4), (64, 3, 1))), ValueError, "fc3: input factor"),
    (_img(), spaces.Discrete(4), dict(hidden_sizes=()), ValueError, "hidden_sizes"),
    (_img(), spaces.Discrete(4), dict(hidden_sizes=(60,)), ValueError, "hidden_sizes"),
    (_img(), spaces.Discrete(4), dict(hidden_sizes=(1032,)), ValueError, "hidden_sizes"),
    (_img(), spaces.Discrete(4), dict(conv_layers=((16, 8),)), ValueError, "conv_layers"),
])
def test_construction_errors(obs_space, act_space, kw, error, message):
    with pytest.raises(error, match=message):
        CNNModel(obs_space, act_space, **kw)


def test_limits_at_their_edges_are_accepted():
    CNNModel(_img(hw=4, c=1), spaces.Discrete(1), conv_layers=((8, 4, 4),), hidden_sizes=(8,))
    CNNModel(_img(hw=128, c=16, dtype=np.float32), spaces.Discrete(31), conv_layers=((128, 8, 4), (8, 4, 4)),
             hidden_sizes=(1024, 8))
    # 84x84x4 with conv3 = 64: the fc4 input factor 3137 is the largest allowed
    CNNModel(_img(hw=84), spaces.Discrete(6))


def test_variables_shapes_and_gains():
    model = CNNModel(_img(hw=36), spaces.Discrete(5), conv_layers=((16, 8, 4), (32, 3, 1)), hidden_sizes=(64, 32),
                     random_seed=1)
    v = model.get_variables()
    assert list(v) == ["conv1/weights", "conv1/bias", "conv2/weights", "conv2/bias", "fc3/weights", "fc3/bias",
                       "fc4/weights", "fc4/bias", "fc_policy/weights", "fc_policy/bias", "fc_baseline/weights",
                       "fc_baseline/bias"]
    shapes = {k: a.shape for k, a in v.items()}
    assert shapes["conv1/weights"] == (8, 8, 4, 16) and shapes["conv2/weights"] == (3, 3, 16, 32)
    assert shapes["fc3/weights"] == (6 * 6 * 32, 64) and shapes["fc4/weights"] == (64, 32)
    assert shapes["fc_policy/weights"] == (32, 5) and shapes["fc_baseline/weights"] == (32, 1)
    for k, a in v.items():
        assert a.dtype == np.float32
        if k.endswith("/bias"):
            assert not a.any()
    for layer, gain in (("conv1", 2 ** 0.5), ("conv2", 2 ** 0.5), ("fc3", 2 ** 0.5), ("fc4", 2 ** 0.5),
                        ("fc_policy", 0.01), ("fc_baseline", 1.0)):
        w = v[layer + "/weights"].astype(np.float64)
        w = w.reshape(-1, w.shape[-1]) / gain
        gram = w.T @ w if w.shape[0] >= w.shape[1] else w @ w.T
        np.testing.assert_allclose(gram, np.eye(gram.shape[0]), atol=1e-5)
    again = CNNModel(_img(hw=36), spaces.Discrete(5), conv_layers=((16, 8, 4), (32, 3, 1)), hidden_sizes=(64, 32),
                     random_seed=1).get_variables()
    assert all(np.array_equal(again[k], v[k]) for k in v)
    assert model.observations_placeholder.shape == (None, None, 36, 36, 4)
    assert model.obs_u8 and not CNNModel(_img(dtype=np.float32), spaces.Discrete(2)).obs_u8


def test_set_variables_checks_shapes():
    model = CNNModel(_img(hw=10, c=7, dtype=np.float32), spaces.Discrete(6), conv_layers=((16, 3, 1),), hidden_sizes=(128,))
    v = model.get_variables()
    v["conv1/weights"] = v["conv1/weights"] + 1.0
    model.set_variables(v)
    assert np.array_equal(model.get_variables()["conv1/weights"], v["conv1/weights"])
    v["conv1/weights"] = np.zeros((3, 3, 8, 16), np.float32)
    with pytest.raises(ValueError):
        model.set_variables(v)


@pytest.mark.parametrize("conv, hidden", [(((8, 8, 4),), (128,)), (((32, 8, 4), (64, 4, 2), (64, 3, 1)), (256,)),
                                          (((16, 4, 4), (16, 3, 2)), (64, 32))])
def test_register_layers(conv, hidden):
    model = CNNModel(_img(hw=64, c=3), spaces.Discrete(5), conv_layers=conv, hidden_sizes=hidden)
    lc = kfac.LayerCollection()
    model.register_layers(lc)
    model.register_predictive_distributions(lc)
    assert [rec["params"][0].split("/")[0] for rec in lc.conv2d] == ["conv%d" % (i + 1) for i in range(len(conv))]
    assert [rec["strides"] for rec in lc.conv2d] == [[1, s, s, 1] for _, _, s in conv]
    assert all(rec["padding"] == "VALID" for rec in lc.conv2d)
    names = [rec["params"][0].split("/")[0] for rec in lc.fully_connected]
    assert names == ["fc%d" % (len(conv) + i + 1) for i in range(len(hidden))] + ["fc_policy", "fc_baseline"]
    heads = lc.fully_connected[-2:]
    assert heads[0]["inputs"] is heads[1]["inputs"]
    assert len(lc.input_factor_groups()) == len(conv) + len(hidden) + 1
    assert len(lc.categorical) == 1 and len(lc.normal) == 1


def test_engine_config_and_shapes():
    cfg = eng.CNNEngineConfig(obs_hw=10, obs_channels=7, obs_u8=False, conv_layers=((16, 3, 1),), hidden_sizes=(128,),
                              num_actions=6)
    c = cfg.to_c()
    assert (c.mlp.obs_dim, c.mlp.num_hidden, c.mlp.hidden[0], c.num_conv, c.obs_u8) == (700, 1, 128, 1, 0)
    assert (c.filters[0], c.kernel[0], c.stride[0]) == (16, 3, 1)
    shapes = eng.cnn_param_shapes(10, 7, ((16, 3, 1),), (128,), 6)
    assert shapes["conv1/weights"] == (3, 3, 7, 16) and shapes["fc2/weights"] == (8 * 8 * 16, 128)
    assert eng.cnn_layers(1, 1) == ("conv1", "fc2", "fc_policy", "fc_baseline")
