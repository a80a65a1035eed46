"""MLPModel - a fully connected actor-critic for vector (`Box`) observations and `Discrete` actions, the counterpart of
envs/atari/model.py for the models most users build first.

    fc1 .. fcL  x @ W + b, ReLU      (nn.py:37-52; observations flattened row-major)
    fc_policy   [H_L, n] logits      fc_baseline [H_L, 1] value, both reading the last hidden layer

Variables are named {fc1 .. fcL, fc_policy, fc_baseline}/{weights, bias} in nn.fully_connected_params' layout (weights
[in, out]); orthogonal weights with gains sqrt(2) (hidden), 0.01 (policy), 1.0 (value), zero biases, as AtariModel.  The
train step runs in libacx's fully connected learner (acx_mlp_*), created on the first train step, when the
[environments, steps] batch shape is known; `A2CObjective(model).optimize_shared(...)` with nn.ClipGlobalNormOptimizer
(RMSProp) or kfac.KfacOptimizer / kfac_utils.ColdStartPeriodicInvUpdateKfacOpt drives it through `Session.run` as for
AtariModel.
"""
import numpy as np
import torch

from . import engine as eng
from . import nn
from . import spaces
from .baselines import StateValueFunction
from .model import ActorCriticModel
from .policies import SoftmaxPolicy
from .session import Fetch

MAX_OBS_DIM = 2048


class MLPModel(ActorCriticModel):
    def __init__(self, observation_space, action_space, hidden_sizes=(64, 64), random_seed=None, name=None):
        super().__init__(observation_space, action_space)
        if not spaces.is_box(observation_space) or np.dtype(observation_space.low.dtype) != np.float32:
            raise TypeError("MLPModel needs a float32 Box observation space, got %r" % (observation_space,))
        if not spaces.is_discrete(action_space):
            raise TypeError("Unsupported space")
        self.obs_shape = tuple(int(d) for d in observation_space.shape)
        self.obs_dim = int(np.prod(self.obs_shape))
        if not 1 <= self.obs_dim <= MAX_OBS_DIM:
            raise ValueError("observations must have 1 to %d features, got %d" % (MAX_OBS_DIM, self.obs_dim))
        self.num_actions = int(action_space.n)
        if not 1 <= self.num_actions <= 31:
            raise ValueError("MLPModel supports 1 to 31 actions, got %d" % self.num_actions)
        self.hidden_sizes = tuple(int(h) for h in hidden_sizes)
        if not 1 <= len(self.hidden_sizes) <= 4 or any(h < 8 or h > 1024 or h % 8 for h in self.hidden_sizes):
            raise ValueError("hidden_sizes: 1 to 4 widths, each a multiple of 8 in [8, 1024], got %s" % (hidden_sizes,))
        self.random_seed = random_seed
        self.layers = eng.mlp_layers(len(self.hidden_sizes))
        shapes = eng.mlp_param_shapes(self.obs_dim, self.hidden_sizes, self.num_actions)
        rng = np.random.default_rng(random_seed)
        gains = {"fc_policy": 0.01, "fc_baseline": 1.0}
        self._params = {}
        for layer in self.layers:
            w, b = nn.fully_connected_params(*shapes[layer + "/weights"], rng=rng, gain=gains.get(layer, 2.0 ** 0.5))
            self._params[layer + "/weights"], self._params[layer + "/bias"] = w, b
        self._policy = SoftmaxPolicy(self, self.num_actions)
        self._baseline = StateValueFunction(self)
        self._bootstrap_values = Fetch("bootstrap_values", self, "bootstrap_values")
        self._engine = None
        self._engine_key = None
        self._layer_tokens = {n: (Fetch("inputs", self, n + "/inputs"), Fetch("outputs", self, n + "/outputs"))
                              for n in self.layers}
        # the two heads are registered with the SAME inputs tensor (as envs/atari/model.py:243,246) -> one shared factor
        self._layer_tokens["fc_baseline"] = (self._layer_tokens["fc_policy"][0], self._layer_tokens["fc_baseline"][1])
        self.engine_options = {}     # extra MLPEngineConfig fields (seed, use_graphs ...)

    # ------------------------------------------------------------------ K-FAC registration
    def register_layers(self, layer_collection):
        """One fully connected block per layer (model.py:107-119)."""
        for name in self.layers:
            inputs, outputs = self._layer_tokens[name]
            layer_collection.register_fully_connected(params=(name + "/weights", name + "/bias"), inputs=inputs,
                                                      outputs=outputs)

    # ------------------------------------------------------------------ variables
    def get_variables(self):
        if self._engine is not None:
            self._params = self._engine.get_params()
        return {k: v.copy() for k, v in self._params.items()}

    def set_variables(self, params):
        for k, v in self._params.items():
            if tuple(np.shape(params[k])) != v.shape:
                raise ValueError("variable %s: expected shape %s, got %s" % (k, v.shape, np.shape(params[k])))
        self._params = {k: np.asarray(params[k], np.float32).copy() for k in self._params}
        if self._engine is not None:
            self._engine.set_params(self._params)

    @property
    def engine(self):
        return self._engine

    # ------------------------------------------------------------------ used by Session
    def _build_engine(self, session, num_envs, num_steps, objective):
        if session.group is not None or (torch.distributed.is_available() and torch.distributed.is_initialized()
                                         and torch.distributed.get_world_size() > 1):
            raise NotImplementedError("MLPModel trains on one GPU: data-parallel learners are not implemented for it")
        kw = dict(num_envs=num_envs, num_steps=num_steps, obs_dim=self.obs_dim, hidden_sizes=self.hidden_sizes,
                  num_actions=self.num_actions)
        if objective is not None:
            if getattr(objective, "_separate", None) is not None:
                raise NotImplementedError("optimize_separate is not implemented for MLPModel: use optimize_shared")
            kw.update(gamma=objective.discount_factor, entropy_beta=objective.entropy_regularization_strength,
                      value_loss_weight=objective._baseline_loss_weight)
            kw.update(objective._optimizer.engine_overrides())
        else:
            kw.update(acktr=False)
        if "seed" not in self.engine_options:
            base = self.random_seed if self.random_seed is not None else int.from_bytes(__import__("os").urandom(4), "little")
            kw["seed"] = (int(base) * 1000003) & 0x7FFFFFFFFFFFFFFF
        kw.update(self.engine_options)
        cfg = eng.MLPEngineConfig(**kw)
        old = self._engine
        if old is not None:
            self._params = old.get_params()
        e = eng.MLPEngine(cfg, session.device)
        e.set_params(self._params)
        if old is not None and old.config.acktr == cfg.acktr:
            e.load_state_dict(old.state_dict())      # the learner state does not depend on the batch shape
        e.is_learner = objective is not None
        self._engine = e
        self._engine_key = (num_envs, num_steps, id(objective) if objective is not None else None)
        if objective is not None and objective._global_step is not None:
            objective._global_step.bind(e)
        return e

    def _engine_for_feed(self, session, feed, objective):
        obs = feed.get(self._observations_placeholder)
        if obs is None:
            raise ValueError("observations_placeholder must be fed")
        shape = tuple(obs.shape) if hasattr(obs, "shape") else np.shape(obs)
        if len(shape) != 2 + len(self.obs_shape) or tuple(shape[2:]) != self.obs_shape:
            raise ValueError("observations must have shape [environments, steps] + %s, got %s" % (self.obs_shape, shape))
        key = (shape[0], shape[1], id(objective))
        if self._engine is None or self._engine_key != key:
            self._build_engine(session, shape[0], shape[1], objective)
        return self._engine

    def _train_feed(self, feed):
        names = ("observations", "bootstrap_observations", "actions", "rewards", "terminals")
        phs = (self._observations_placeholder, self._bootstrap_observations_placeholder, self._actions_placeholder,
               self._rewards_placeholder, self._terminals_placeholder)
        e, t = self._engine.num_envs, self._engine.num_steps
        out = []
        for name, ph in zip(names, phs):
            if ph not in feed:
                raise ValueError("placeholder '%s' must be fed for a train step (a2c_acktr.py:117-126)" % name)
            v = feed[ph]
            if not isinstance(v, torch.Tensor):
                v = np.asarray(v, dtype=ph.dtype if ph.dtype != np.bool_ else np.bool_)
            if name == "observations":
                v = v.reshape(e, t, self.obs_dim)
            elif name == "bootstrap_observations":
                v = v.reshape(e, self.obs_dim)
            out.append(v)
        return out

    def _act(self, session, feed, greedy):
        obs = feed.get(self._observations_placeholder)
        if obs is None:
            raise ValueError("observations_placeholder must be fed")
        if not isinstance(obs, torch.Tensor):
            obs = torch.from_numpy(np.ascontiguousarray(np.asarray(obs, np.float32)))
        lead = tuple(obs.shape[:obs.dim() - len(self.obs_shape)])
        flat = obs.reshape(-1, self.obs_dim)
        e = self._engine
        if e is None:
            e = self._build_engine(session, flat.shape[0], 1, None)
        if flat.shape[0] > e.rows + e.num_envs:
            raise ValueError("too many observations (%d) for the engine's batch (%d)" % (flat.shape[0], e.rows + e.num_envs))
        actions, logits, values = e.act(flat, greedy=greedy, want_logits=True)
        torch.cuda.current_stream(session.device).synchronize()
        shaped = actions.cpu().numpy().reshape(lead)
        # DistributionPolicy.sample / mode squeeze the last (step) axis: valid for a step dimension of 1 (policies.py:86-87)
        if len(lead) == 2 and lead[1] == 1:
            shaped = shaped.reshape(lead[0])
        return {"sample": shaped, "mode": shaped, "logits": logits.cpu().numpy().reshape(lead + (self.num_actions,)),
                "value": values.cpu().numpy().reshape(lead)}

    def _bootstrap_only(self, session, feed):
        obs = feed.get(self._bootstrap_observations_placeholder)
        if obs is None:
            raise ValueError("bootstrap_observations_placeholder must be fed")
        return self._act(session, {self._observations_placeholder: obs}, greedy=True)["value"]
