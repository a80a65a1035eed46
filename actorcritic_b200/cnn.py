"""CNNModel - a convolutional actor-critic for square image observations (`Box` [H, H, C], uint8 or float32) of any size
and `Discrete` actions: MinAtar-style grids, Procgen-style frames, Atari at another resolution or frame stack.

    conv1 .. convK  VALID conv2d (HWIO kernel, stride s) + bias, ReLU      (nn.py:88-110)
    flatten         (h, w, c)                                              (nn.py:125-126)
    fc(K+1) ..      x @ W + b, ReLU                                        (nn.py:37-52)
    fc_policy       [H_L, n] logits      fc_baseline [H_L, 1] value, both reading the last hidden layer

uint8 observations are scaled by 1/255 (envs/atari/model.py:93), float32 ones are used as given.  Variables are
{conv<i>, fc<j>, fc_policy, fc_baseline}/{weights, bias}, the layer numbers continuing from the conv layers to the fully
connected ones as the reference numbers conv3 -> fc4; orthogonal weights with gains sqrt(2) (trunk), 0.01 (policy), 1.0
(value), zero biases.  Training and acting are MLPModel's: the train step runs in libacx's fully connected learner with a
convolutional trunk (acx_cnn_create, then the acx_mlp_* calls), one conv K-FAC block per conv layer.

The default layers are the Nature-CNN's (AtariModel's trunk with conv3 = 64).  Limits, checked at construction: H in
[4, 128], C in [1, 16]; 1 to 3 conv layers with filters a multiple of 8 in [8, 128], kernel in [1, 8], stride in
[1, min(kernel, 4)], every output at least 1 x 1; 1 to 4 hidden widths as MLPModel; at most 4 conv and fully connected
layers in all; every input factor (kernel^2 * input channels + 1 for a conv layer, the flattened conv output + 1 for the
first fully connected layer) at most 3137 wide.
"""
import numpy as np

from . import engine as eng
from . import nn
from . import spaces
from .mlp import MLPModel

MAX_FACTOR_DIM = 3137      # the largest input factor the learners invert (AtariModel's fc4 with conv3 = 64)


class CNNModel(MLPModel):
    _ENGINE = eng.CNNEngine

    def __init__(self, observation_space, action_space, conv_layers=((32, 8, 4), (64, 4, 2), (64, 3, 1)),
                 hidden_sizes=(512,), random_seed=None, name=None):
        try:
            self.conv_layers = tuple((int(f), int(k), int(s)) for f, k, s in conv_layers)
        except (TypeError, ValueError):
            raise ValueError("conv_layers: (filters, kernel, stride) per layer, got %r" % (conv_layers,)) from None
        super().__init__(observation_space, action_space, hidden_sizes=hidden_sizes, random_seed=random_seed, name=name)

    # ------------------------------------------------------------------ MLPModel hooks
    def _check_observation_space(self, observation_space):
        if not spaces.is_box(observation_space):
            raise TypeError("CNNModel needs a Box observation space, got %r" % (observation_space,))
        dtype = np.dtype(observation_space.low.dtype)
        if dtype not in (np.dtype(np.uint8), np.dtype(np.float32)):
            raise TypeError("CNNModel observations must be uint8 or float32, got %s" % dtype)
        shape = tuple(int(d) for d in observation_space.shape)
        if len(shape) != 3 or shape[0] != shape[1]:
            raise ValueError("CNNModel observations must be square images [H, H, C], got shape %s" % (shape,))
        if not 4 <= shape[0] <= 128:
            raise ValueError("image size H must be in [4, 128], got %d" % shape[0])
        if not 1 <= shape[2] <= 16:
            raise ValueError("image channels C must be in [1, 16], got %d" % shape[2])
        self.obs_shape = shape
        self.obs_dim = int(np.prod(shape))
        self.obs_u8 = dtype == np.dtype(np.uint8)
        self._engine_obs_shape = shape
        self._obs_dtype = dtype.type

    def _check_trunk(self):
        conv = self.conv_layers
        if not 1 <= len(conv) <= 3:
            raise ValueError("conv_layers: 1 to 3 layers, got %d" % len(conv))
        if len(conv) + len(self.hidden_sizes) > 4:
            raise ValueError("at most 4 conv and fully connected layers in all, got %d + %d"
                             % (len(conv), len(self.hidden_sizes)))
        hw, c = self.obs_shape[0], self.obs_shape[2]
        for i, (f, k, s) in enumerate(conv):
            name = "conv%d" % (i + 1)
            if f < 8 or f > 128 or f % 8:
                raise ValueError("%s: filters must be a multiple of 8 in [8, 128], got %d" % (name, f))
            if not 1 <= k <= 8:
                raise ValueError("%s: kernel must be in [1, 8], got %d" % (name, k))
            if not 1 <= s <= min(k, 4):
                raise ValueError("%s: stride must be in [1, min(kernel, 4)] = [1, %d], got %d" % (name, min(k, 4), s))
            if k > hw:
                raise ValueError("%s: kernel %d does not fit its %dx%d input (output below 1x1)" % (name, k, hw, hw))
            if k * k * c + 1 > MAX_FACTOR_DIM:
                raise ValueError("%s: input factor kernel^2 * channels + 1 = %d exceeds %d"
                                 % (name, k * k * c + 1, MAX_FACTOR_DIM))
            hw, c = (hw - k) // s + 1, f
        if hw * hw * c + 1 > MAX_FACTOR_DIM:
            raise ValueError("fc%d: input factor (flattened conv output %dx%dx%d) + 1 = %d exceeds %d"
                             % (len(conv) + 1, hw, hw, c, hw * hw * c + 1, MAX_FACTOR_DIM))

    def _layer_names(self):
        return eng.cnn_layers(len(self.conv_layers), len(self.hidden_sizes))

    def _initial_params(self, rng):
        shapes = eng.cnn_param_shapes(self.obs_shape[0], self.obs_shape[2], self.conv_layers, self.hidden_sizes,
                                      self.num_actions)
        gains = {"fc_policy": 0.01, "fc_baseline": 1.0}
        params = {}
        for layer in self.layers:
            shape = shapes[layer + "/weights"]
            gain = gains.get(layer, 2.0 ** 0.5)
            if len(shape) == 4:
                w, b = nn.conv2d_params(shape[2], shape[3], shape[0], rng=rng, gain=gain)
            else:
                w, b = nn.fully_connected_params(*shape, rng=rng, gain=gain)
            params[layer + "/weights"], params[layer + "/bias"] = w, b
        return params

    def _engine_config(self, **kw):
        return eng.CNNEngineConfig(obs_hw=self.obs_shape[0], obs_channels=self.obs_shape[2], obs_u8=self.obs_u8,
                                   conv_layers=self.conv_layers, hidden_sizes=self.hidden_sizes, **kw)

    # ------------------------------------------------------------------ K-FAC registration
    def register_layers(self, layer_collection):
        """One conv2d block per conv layer (VALID, envs/atari/model.py:227-237), one fully connected block per fully
        connected layer; the two heads share one inputs tensor and so one input factor."""
        for (_, _, s), name in zip(self.conv_layers, self.layers):
            inputs, outputs = self._layer_tokens[name]
            layer_collection.register_conv2d(params=(name + "/weights", name + "/bias"), strides=[1, s, s, 1],
                                             padding="VALID", inputs=inputs, outputs=outputs)
        for name in self.layers[len(self.conv_layers):]:
            inputs, outputs = self._layer_tokens[name]
            layer_collection.register_fully_connected(params=(name + "/weights", name + "/bias"), inputs=inputs,
                                                      outputs=outputs)
