"""Host-side handles of the native learner engines (include/acx.h `acx_learner_*`, `acx_mlp_*`).

torch is used for device memory (the arena is one uint8 CUDA tensor, every buffer a view into it),
the current CUDA stream and `torch.distributed`; all arithmetic runs in libacx.so.  There is no CPU
path: constructing an `Engine` without a CUDA device raises.

The hyper-parameters default to the literals of the reference's example
(actorcritic/examples/atari/a2c_acktr.py:52,57,64-71,76,240-251).
"""
import contextlib
import ctypes
import os
import dataclasses

import numpy as np
import torch

from . import _lib

LAYERS = ("conv1", "conv2", "conv3", "fc4", "fc_policy", "fc_baseline")
A_FACTORS = ("conv1", "conv2", "conv3", "fc4", "heads")
OBS_SHAPE = (84, 84, 4)
OBS_BYTES = 84 * 84 * 4

SCALAR_NAMES = ("policy_loss", "baseline_loss", "mean_entropy", "loss", "clip_coeff", "fisher_norm", "grad_norm",
                "learning_rate")


@dataclasses.dataclass
class EngineConfig:
    num_envs: int = 32
    num_steps: int = 20
    num_actions: int = 4
    conv3_filters: int = 32                 # a2c_acktr.py:52 (32 for ACKTR, 64 for A2C)
    acktr: bool = True
    gamma: float = 0.99                     # :57
    entropy_beta: float = 0.01              # :57
    value_loss_weight: float = 0.5          # :76
    lr_start: float = 0.25                  # :68  (A2C: 0.0007, :71)
    lr_end: float = 0.025
    lr_decay_steps: float = None            # :64  1e7 / (num_envs * num_steps)
    cov_ema_decay: float = 0.99             # :245
    damping: float = 0.01
    momentum: float = 0.9
    norm_constraint: float = 0.0001
    invert_every: int = 10
    num_cold_updates: int = 30              # :244
    cold_lr: float = 0.0003                 # :240
    cold_momentum: float = 0.9
    clip_norm: float = 0.5                  # :241 / :251
    rms_decay: float = 0.9                  # TF-1 RMSPropOptimizer defaults (:250)
    rms_epsilon: float = 1e-10
    num_locations_mode: str = "true"        # or "input_div_stride" (SURVEY A.7-U1)
    world_size: int = 1
    gemm_impl: int = 0
    precision: int = 0
    use_graphs: bool = True                 # replay each update as CUDA graphs (captured on the second use of a variant)
    conv_impl: int = 0                      # 0 = gather-form conv2/conv3 input gradient (acx_conv), 1 = GEMM + col2im
    num_lanes: int = 0                      # 0 = default (5 concurrent lanes inside an update), 1 = serial
    seed: int = 0
    cov_init: str = "zero"                  # SURVEY A.7-U3: "zero" (kfac 0.1.x) | "identity" (older tf.contrib.kfac)
    zero_debias: bool = True                # U3
    inv_init: str = "zero"                  # U3: "zero" | "identity"

    @staticmethod
    def a2c(num_envs=16, num_steps=5, num_actions=4, **kw):
        """The reference's A2C configuration (a2c_acktr.py:52,71,250-251,309-310)."""
        base = dict(num_envs=num_envs, num_steps=num_steps, num_actions=num_actions, conv3_filters=64, acktr=False,
                    lr_start=0.0007, lr_end=0.00007)
        base.update(kw)
        return EngineConfig(**base)

    def to_c(self):
        c = _lib.LearnerConfig()
        c.num_envs, c.num_steps, c.num_actions = self.num_envs, self.num_steps, self.num_actions
        c.conv3_filters, c.acktr = self.conv3_filters, int(self.acktr)
        c.gamma, c.entropy_beta, c.value_loss_weight = self.gamma, self.entropy_beta, self.value_loss_weight
        c.lr_start, c.lr_end = self.lr_start, self.lr_end
        steps = self.lr_decay_steps
        c.lr_decay_steps = float(steps) if steps is not None else 1e7 / (self.num_envs * self.num_steps * self.world_size)
        c.cov_ema_decay, c.damping, c.momentum = self.cov_ema_decay, self.damping, self.momentum
        c.norm_constraint = self.norm_constraint
        c.invert_every, c.num_cold_updates = self.invert_every, self.num_cold_updates
        c.cold_lr, c.cold_momentum, c.clip_norm = self.cold_lr, self.cold_momentum, self.clip_norm
        c.rms_decay, c.rms_epsilon = self.rms_decay, self.rms_epsilon
        if self.num_locations_mode not in ("true", "input_div_stride"):
            raise ValueError("num_locations_mode must be 'true' or 'input_div_stride'")
        c.num_locations_mode = 0 if self.num_locations_mode == "true" else 1
        c.world_size, c.gemm_impl, c.precision, c.seed = self.world_size, self.gemm_impl, self.precision, self.seed
        c.use_graphs = int(bool(self.use_graphs))
        c.num_lanes = int(self.num_lanes)
        c.conv_impl = int(self.conv_impl)
        for name in ("cov_init", "inv_init"):
            if getattr(self, name) not in ("zero", "identity"):
                raise ValueError("%s must be 'zero' or 'identity'" % name)
        c.cov_init_identity = int(self.cov_init == "identity")
        c.no_zero_debias = int(not self.zero_debias)
        c.inv_init_identity = int(self.inv_init == "identity")
        return c


def param_shapes(num_actions, c3):
    """Variable shapes of AtariModel (envs/atari/model.py:137-170; HWIO conv kernels, [in, out] fc weights)."""
    return {
        "conv1/weights": (8, 8, 4, 32), "conv1/bias": (32,),
        "conv2/weights": (4, 4, 32, 64), "conv2/bias": (64,),
        "conv3/weights": (3, 3, 64, c3), "conv3/bias": (c3,),
        "fc4/weights": (49 * c3, 512), "fc4/bias": (512,),
        "fc_policy/weights": (512, num_actions), "fc_policy/bias": (num_actions,),
        "fc_baseline/weights": (512, 1), "fc_baseline/bias": (1,),
    }


def flatten_params(params, num_actions, c3):
    """dict of reference-named variables -> the engine's flat vector: per layer [K+1, C] (weight rows in
    (kh, kw, cin) order = the HWIO variable reshaped, then the bias row)."""
    shapes = param_shapes(num_actions, c3)
    parts = []
    for layer in LAYERS:
        w = np.asarray(params[layer + "/weights"], np.float32)
        b = np.asarray(params[layer + "/bias"], np.float32)
        if tuple(w.shape) != shapes[layer + "/weights"] or tuple(b.shape) != shapes[layer + "/bias"]:
            raise ValueError("bad shape for layer %s: %s / %s" % (layer, w.shape, b.shape))
        parts.append(w.reshape(-1, w.shape[-1]).ravel())
        parts.append(b.ravel())
    return np.concatenate(parts)


def unflatten_params(flat, num_actions, c3):
    shapes = param_shapes(num_actions, c3)
    out, off = {}, 0
    flat = np.asarray(flat)
    for layer in LAYERS:
        for kind in ("weights", "bias"):
            shape = shapes[layer + "/" + kind]
            n = int(np.prod(shape))
            out[layer + "/" + kind] = flat[off:off + n].reshape(shape).copy()
            off += n
    return out


def orthogonal_init(num_actions=4, c3=32, seed=None):
    """envs/atari/model.py:132-135: orthogonal kernels with gains sqrt(2) (trunk), 0.01 (policy), 1.0 (value);
    zero biases.  QR-based like tf.orthogonal_initializer; the random stream is numpy's, not TensorFlow's."""
    rng = np.random.default_rng(seed)
    gains = {"conv1": 2.0 ** 0.5, "conv2": 2.0 ** 0.5, "conv3": 2.0 ** 0.5, "fc4": 2.0 ** 0.5, "fc_policy": 0.01,
             "fc_baseline": 1.0}
    params = {}
    for key, shape in param_shapes(num_actions, c3).items():
        layer, kind = key.split("/")
        if kind == "bias":
            params[key] = np.zeros(shape, np.float32)
            continue
        rows, cols = int(np.prod(shape[:-1])), int(shape[-1])
        a = rng.standard_normal((max(rows, cols), min(rows, cols)))
        q, r = np.linalg.qr(a)
        q = q * np.sign(np.diag(r))
        if rows < cols:
            q = q.T
        params[key] = (gains[layer] * q).reshape(shape).astype(np.float32)
    return params


class PendingScalars:
    """Result of `Engine.update(fetch="async")`: the update's scalars once their device-to-host copy has landed."""

    def __init__(self, pinned, event):
        self._pinned, self._event = pinned, event

    def done(self):
        return self._event.query()

    def result(self):
        self._event.synchronize()
        return dict(zip(SCALAR_NAMES, self._pinned.tolist()))


class _ArenaEngine:
    """What the learner handles of libacx share: one device arena (every buffer a view into it), the engine's stream,
    parameters, schedule state, the train-step inputs, scalar read-back and acting.  A subclass names its C API prefix
    (`_API`), its observation dtype and its parameter layout."""

    _API = None
    _OBS_DTYPE = torch.uint8

    def _fn(self, name):
        return getattr(self.lib, self._API + name)

    def _open(self, config, device, obs_shape):
        if not torch.cuda.is_available():
            raise _lib.AcxError("actorcritic_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = _lib.load()
        self.config = config
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self._c = config.to_c()
        # the engine launches on its own (non-default) stream: CUDA graphs cannot be captured on the legacy stream
        self.stream = torch.cuda.Stream(self.device)
        with torch.cuda.device(self.device):
            nbytes = self._fn("arena_bytes")(ctypes.byref(self._c))
            if nbytes == 0:
                raise _lib.AcxError(self.lib.acx_last_error().decode())
            self.arena = torch.empty(nbytes + 256, dtype=torch.uint8, device=self.device)
            self._arena_off = (-self.arena.data_ptr()) % 256
            base = self.arena.data_ptr() + self._arena_off
            self._h = self._fn("create")(ctypes.byref(self._c), ctypes.c_void_p(base), ctypes.c_size_t(nbytes))
            if not self._h:
                raise _lib.AcxError(self.lib.acx_last_error().decode())
        self.is_learner = True          # the models mark the engine they build for acting only (no objective yet)
        self.num_params = int(self._fn("num_params")(self._h))
        self.num_envs, self.num_steps = config.num_envs, config.num_steps
        self.rows = config.num_envs * config.num_steps
        self._views = {}
        self.obs_shape = tuple(obs_shape)
        n, e, a = self.rows, config.num_envs, config.num_actions
        self.observations = self.buffer("observations", self._OBS_DTYPE, (n + e,) + self.obs_shape)
        self.actions = self.buffer("actions", torch.uint8, (e, config.num_steps))
        self.rewards = self.buffer("rewards", torch.float32, (e, config.num_steps))
        self.terminals = self.buffer("terminals", torch.uint8, (e, config.num_steps))
        self.bucket = self.buffer("reduce_bucket", torch.float32)
        self.scalars = self.buffer("scalars", torch.float32)
        self.logits = self.buffer("logits", torch.float32, (n + e, a))
        self.values = self.buffer("values", torch.float32, (n + e,))
        self._pinned_scalars = torch.empty(16, dtype=torch.float32).pin_memory()

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            self._fn("destroy")(h)

    # ------------------------------------------------------------------ buffers
    def buffer(self, name, dtype=torch.float32, shape=None):
        key = (name, dtype, shape)
        if key in self._views:
            return self._views[key]
        nbytes = ctypes.c_size_t(0)
        ptr = self._fn("buffer")(self._h, name.encode(), ctypes.byref(nbytes))
        if not ptr:
            raise KeyError(self.lib.acx_last_error().decode())
        off = ptr - self.arena.data_ptr()
        view = self.arena[off:off + nbytes.value].view(dtype)
        if shape is not None:
            view = view.view(shape)
        self._views[key] = view
        return view

    def _stream(self):
        return ctypes.c_void_p(self.stream.cuda_stream)

    @contextlib.contextmanager
    def on_stream(self):
        """Run the enclosed torch ops on the engine's stream, ordered after what the caller's current stream has
        queued and before what it queues next.  Inside `with torch.cuda.stream(engine.stream)` this is free."""
        cur = torch.cuda.current_stream(self.device)
        if cur == self.stream:
            yield
            return
        self.stream.wait_stream(cur)
        with torch.cuda.stream(self.stream):
            yield
        cur.wait_stream(self.stream)

    # ------------------------------------------------------------------ parameters / state
    def set_params(self, params):
        flat = params if isinstance(params, np.ndarray) and params.ndim == 1 else self._flatten(params)
        flat = np.ascontiguousarray(flat, np.float32)
        if flat.size != self.num_params:
            raise ValueError("expected %d parameters, got %d" % (self.num_params, flat.size))
        with self.on_stream():
            _lib.check(self._fn("set_params")(self._h, flat.ctypes.data_as(ctypes.c_void_p), self._stream()))

    def get_params_flat(self):
        out = np.empty(self.num_params, np.float32)
        with self.on_stream():
            _lib.check(self._fn("get_params")(self._h, out.ctypes.data_as(ctypes.c_void_p), self._stream()))
        return out

    def get_params(self):
        return self._unflatten(self.get_params_flat())

    def layer_matrix(self, kind, layer):
        """[K+1, C] device view of "params" / "grads" / "precon" for one layer."""
        return self.buffer("%s/%s" % (kind, layer), torch.float32).view(-1, self._layer_cols(layer))

    def factor(self, kind, which, name):
        """Square device view: kind in {"stats","sums","inv"}, which in {"A","G"}."""
        v = self.buffer("%s/%s/%s" % (kind, which, name), torch.float32)
        d = int(round(v.numel() ** 0.5))
        return v.view(d, d)

    @property
    def global_step(self):
        return int(self._fn("global_step")(self._h))

    def get_state(self):
        gs, nc, iv = ctypes.c_int64(0), ctypes.c_int64(0), ctypes.c_int(0)
        _lib.check(self._fn("get_state")(self._h, ctypes.byref(gs), ctypes.byref(nc), ctypes.byref(iv)))
        return dict(global_step=gs.value, num_cov_updates=nc.value, inverses_valid=bool(iv.value))

    def set_state(self, global_step, num_cov_updates=0, inverses_valid=False):
        with self.on_stream():
            _lib.check(self._fn("set_state")(self._h, int(global_step), int(num_cov_updates), int(bool(inverses_valid)),
                                             self._stream()))

    def refresh_derived(self):
        """Re-derive the bf16 operand planes after writing "params" / "inverses" on the device."""
        with self.on_stream():
            _lib.check(self._fn("refresh_weights")(self._h, self._stream()))

    def wait_pending_ema(self):
        """A split exchange's EMA (Engine._split_exchange) may still be reading the statistics / writing the running sums on
        its own stream: order the engine's stream after it before anything else touches them."""
        if getattr(self, "_ema_pending", False):
            self.stream.wait_event(self._ema_done)
            self._ema_pending = False

    def state_dict(self):
        """Everything `tf.train.Saver` would save for this path (a2c_acktr.py:101): parameters, optimiser slots,
        K-FAC running sums, stored inverses and the schedule counters - as host tensors."""
        self.wait_pending_ema()
        torch.cuda.synchronize(self.device)
        sd = {k: self.buffer(k, torch.float32).cpu().clone() for k in ("params", "velocity", "accum", "factor_sums",
                                                                       "inverses")}
        sd.update(self.get_state())
        sd["config"] = dataclasses.asdict(self.config)
        return sd

    def load_state_dict(self, sd):
        self.wait_pending_ema()
        for k in ("params", "velocity", "accum", "factor_sums", "inverses"):
            self.buffer(k, torch.float32).copy_(sd[k].to(self.device))
        self.refresh_derived()
        self.set_state(sd["global_step"], sd["num_cov_updates"], sd["inverses_valid"])

    # ------------------------------------------------------------------ one update
    def load_batch(self, observations, bootstrap_observations, actions, rewards, terminals, non_blocking=True):
        """Copy the five train-step inputs (ActorCriticModel placeholders, model.py:97-105) into the arena.
        Accepts host (numpy / pinned torch) or device tensors; layouts [E,T,*obs_shape], [E,*obs_shape] (uint8 for
        AtariModel, float32 for MLPModel), [E,T] u8, [E,T] f32, [E,T] bool/u8."""
        n = self.rows

        def as_t(x, dtype):
            t = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x))
            if t.dtype == torch.bool:
                t = t.to(torch.uint8)
            if t.dtype != dtype:
                t = t.to(dtype)
            return t

        with self.on_stream():
            self.observations[:n].view(self.num_envs, self.num_steps, *self.obs_shape).copy_(
                as_t(observations, self._OBS_DTYPE), non_blocking=non_blocking)
            self.observations[n:].copy_(as_t(bootstrap_observations, self._OBS_DTYPE), non_blocking=non_blocking)
            self.actions.copy_(as_t(actions, torch.uint8), non_blocking=non_blocking)
            self.rewards.copy_(as_t(rewards, torch.float32), non_blocking=non_blocking)
            self.terminals.copy_(as_t(terminals, torch.uint8), non_blocking=non_blocking)

    def _fetched(self, fetch):
        if not fetch:
            return None
        if fetch == "async":
            return self.fetch_scalars_async()
        return self.fetch_scalars()

    def fetch_scalars_async(self):
        """Start the device-to-host copy of this update's scalars (losses, clip coefficient, learning rate ...) and return
        a handle; `handle.result()` waits for THAT copy only, so the host can enqueue the next update before it reads the
        numbers of this one (`update(fetch="async")`).  Four pinned slots are cycled: resolve a handle before four more
        updates have been fetched."""
        if getattr(self, "_pending_slots", None) is None:
            self._pending_slots = [torch.empty(16, dtype=torch.float32).pin_memory() for _ in range(4)]
            self._pending_events = [torch.cuda.Event() for _ in range(4)]
            self._pending_next = 0
        k = self._pending_next % 4
        self._pending_next += 1
        with self.on_stream():
            self._pending_slots[k].copy_(self.scalars, non_blocking=True)
            self._pending_events[k].record(self.stream)
        return PendingScalars(self._pending_slots[k], self._pending_events[k])

    def fetch_scalars(self):
        with self.on_stream():
            self._pinned_scalars.copy_(self.scalars, non_blocking=True)
        self.stream.synchronize()
        vals = self._pinned_scalars.tolist()
        return dict(zip(SCALAR_NAMES, vals))

    # ------------------------------------------------------------------ acting
    def act(self, observations, uniform=None, greedy=False, want_logits=False, out=None):
        """Forward + categorical sample / argmax on [rows, *obs_shape] device observations
        (ActorCriticModel.sample_actions / select_max_actions, model.py:135-169).

        `out` (int32 [rows], optional): where the actions go.  A rollout loop that passes the same observation buffer and
        the same `out` every step has stable pointers, which lets the library replay the whole acting step as one CUDA
        graph (acx_learner_act / acx_mlp_act); without `out` every call returns fresh tensors."""
        if not observations.is_cuda:
            observations = observations.to(self.device, non_blocking=True)
        observations = observations.to(self._OBS_DTYPE).contiguous()
        rows = observations.shape[0]
        actions = out if out is not None else torch.empty(rows, dtype=torch.int32, device=self.device)
        logits = torch.empty((rows, self.config.num_actions), dtype=torch.float32, device=self.device) if want_logits else None
        values = torch.empty(rows, dtype=torch.float32, device=self.device) if want_logits else None
        with self.on_stream():
            _lib.check(self._fn("act")(
                self._h, ctypes.c_void_p(observations.data_ptr()), rows,
                ctypes.c_void_p(uniform.data_ptr()) if uniform is not None else None, int(bool(greedy)),
                ctypes.c_void_p(actions.data_ptr()),
                ctypes.c_void_p(logits.data_ptr()) if want_logits else None,
                ctypes.c_void_p(values.data_ptr()) if want_logits else None, self._stream()))
        if want_logits:
            return actions, logits, values
        return actions


class Engine(_ArenaEngine):
    """One learner per process / GPU (AtariModel's Nature-CNN, include/acx.h `acx_learner_*`)."""

    _API = "acx_learner_"

    def __init__(self, config, device=None):
        self._open(config, device, OBS_SHAPE)

    def _flatten(self, params):
        return flatten_params(params, self.config.num_actions, self.config.conv3_filters)

    def _unflatten(self, flat):
        return unflatten_params(flat, self.config.num_actions, self.config.conv3_filters)

    def _layer_cols(self, layer):
        c = self.config
        return {"conv1": 32, "conv2": 64, "conv3": c.conv3_filters, "fc4": 512, "fc_policy": c.num_actions,
                "fc_baseline": 1}[layer]

    # --- double-buffered host feed: the H2D copy of the next batch overlaps the current update ---------------
    def _ensure_staging(self):
        if getattr(self, "_staging", None) is not None:
            return
        n, e, t = self.rows, self.num_envs, self.num_steps
        mk = lambda shape, dt: torch.empty(shape, dtype=dt, device=self.device)     # noqa: E731
        self._staging = [dict(observations=mk((e, t) + OBS_SHAPE, torch.uint8), bootstrap_observations=mk((e,) + OBS_SHAPE, torch.uint8),
                              actions=mk((e, t), torch.uint8), rewards=mk((e, t), torch.float32), terminals=mk((e, t), torch.uint8))
                         for _ in range(2)]
        self._copy_stream = torch.cuda.Stream(self.device)
        self._ready = [torch.cuda.Event() for _ in range(2)]
        self._free = [torch.cuda.Event() for _ in range(2)]
        self._stage_put = 0
        self._stage_get = 0
        del n

    def stage_batch(self, batch):
        """Start the asynchronous host-to-device copy of a batch (pinned host tensors) into one of two staging slots on
        a dedicated copy stream; `update(staged=True)` consumes the slots in order.  At most two batches in flight."""
        self._ensure_staging()
        if self._stage_put - self._stage_get >= 2:
            raise _lib.AcxError("stage_batch: both staging slots hold batches that update(staged=True) has not consumed yet")
        k = self._stage_put % 2
        slot = self._staging[k]
        with torch.cuda.stream(self._copy_stream):
            if self._stage_put >= 2:
                self._copy_stream.wait_event(self._free[k])
            for name, dst in slot.items():
                src = batch[name]
                if not isinstance(src, torch.Tensor):
                    src = torch.from_numpy(np.ascontiguousarray(src))
                if src.dtype == torch.bool:
                    src = src.to(torch.uint8)
                dst.copy_(src, non_blocking=True)
            self._ready[k].record(self._copy_stream)
        self._stage_put += 1

    def _consume_staged(self):
        if getattr(self, "_staging", None) is None or self._stage_get >= self._stage_put:
            raise _lib.AcxError("update(staged=True) without a staged batch (call stage_batch first)")
        k = self._stage_get % 2
        slot = self._staging[k]
        with self.on_stream():
            self.stream.wait_event(self._ready[k])
            self.load_batch(slot["observations"], slot["bootstrap_observations"], slot["actions"], slot["rewards"],
                            slot["terminals"])
            self._free[k].record(self.stream)
        self._stage_get += 1

    def phase1(self, fisher_labels=None, fisher_eps=None):
        fl = ctypes.c_void_p(fisher_labels.data_ptr()) if fisher_labels is not None else None
        fe = ctypes.c_void_p(fisher_eps.data_ptr()) if fisher_eps is not None else None
        with self.on_stream():
            self.wait_pending_ema()      # the previous update's EMA (split exchange) still reads the statistics
            _lib.check(self.lib.acx_learner_phase1(self._h, fl, fe, self._stream()))

    def allreduce(self, group=None, overlap=None):
        """The collective of the data-parallel path (SURVEY 8(e3)): sum of [A | G | grads | scalars] over the ranks.
        With `overlap` the input-factor prefix A - three quarters of the bucket, complete long before the backward
        pass ends - is all-reduced on a second communicator and stream as soon as the library raises its event
        (acx_learner_wait_input_factors), while phase 1 is still running; only [G | grads | scalars] is reduced after it."""
        if self.config.world_size <= 1:
            return
        dist = torch.distributed
        if self._peers_ready(group):
            # the exchange runs inside phase 2 as one kernel over NVLink peer memory (csrc/peer.cu): nothing to issue here
            # except, for updates with factor statistics and no inverse refresh, the input-factor prefix on the side stream
            self._plan_peer_exchange(group)
            return
        early = False
        if overlap is None:
            # Opt-in (ACX_DP_OVERLAP=1 or overlap=True).  Measured on one 8 x B200 box it does not pay: 2 ranks 1.097 ms/update
            # without vs 1.110 with, 8 ranks 1.154 vs 1.158 and a slower end-to-end loop (second collective's host cost) -
            # the 18 MB all-reduce over NVSwitch is short and its CTAs compete with the backward pass for SMs.
            overlap = os.environ.get("ACX_DP_OVERLAP", "0") != "0"
        if overlap and dist.get_backend(group) == "nccl":
            if getattr(self, "_comm_stream", None) is None:
                self._comm_stream = torch.cuda.Stream(self.device)
                self._comm_group = dist.new_group(ranks=dist.get_process_group_ranks(group or dist.group.WORLD), backend="nccl")
                self._comm_done = torch.cuda.Event()
                self._bucket_a = self.buffer("input_factor_stats", torch.float32)
                self._bucket_rest = self.bucket[self._bucket_a.numel():]
            rc = self.lib.acx_learner_wait_input_factors(self._h, ctypes.c_void_p(self._comm_stream.cuda_stream))
            if rc > 0:
                _lib.check(rc)
            early = rc == 0
        if not overlap and self._split_exchange(group):
            return
        with self.on_stream():
            if early:
                with torch.cuda.stream(self._comm_stream):
                    dist.all_reduce(self._bucket_a, op=dist.ReduceOp.SUM, group=self._comm_group)
                    self._comm_done.record(self._comm_stream)
                dist.all_reduce(self._bucket_rest, op=dist.ReduceOp.SUM, group=group)
                self.stream.wait_event(self._comm_done)
            else:
                dist.all_reduce(self.bucket, op=dist.ReduceOp.SUM, group=group)

    def _peers_ready(self, group):
        """One-time set-up of the peer exchange (NCCL groups on one node, ACX_PEER != 0): every rank exports its arena with CUDA
        IPC, maps the others' and hands the bases to the library.  All ranks agree on the outcome (a rank that cannot map a
        peer sends everybody back to NCCL)."""
        state = getattr(self, "_peer_state", None)
        if state is not None:
            return state
        dist = torch.distributed
        ok = os.environ.get("ACX_PEER", "1") != "0" and dist.get_backend(group) == "nccl" and self.config.world_size <= 8
        bases = None
        if ok:
            handle = (ctypes.c_ubyte * 64)()
            offset = ctypes.c_ulonglong(0)
            base = self.arena.data_ptr() + self._arena_off
            rc = self.lib.acx_peer_export(ctypes.c_void_p(base), handle, ctypes.byref(offset))
            mine = (bytes(handle), int(offset.value), os.uname().nodename) if rc == 0 else None
            everyone = [None] * self.config.world_size
            dist.all_gather_object(everyone, mine, group=group)
            rank = dist.get_rank(group)
            ok = all(x is not None and x[2] == everyone[rank][2] for x in everyone)
            if ok:
                bases = (ctypes.c_void_p * self.config.world_size)()
                with torch.cuda.device(self.device):
                    for k, x in enumerate(everyone):
                        if k == rank:
                            bases[k] = base
                            continue
                        ptr = self.lib.acx_peer_import((ctypes.c_ubyte * 64).from_buffer_copy(x[0]), ctypes.c_ulonglong(x[1]))
                        if not ptr:
                            ok = False
                            break
                        bases[k] = ptr
        flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=self.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
        ok = bool(flag.item())
        if ok:
            _lib.check(self.lib.acx_learner_set_peers(self._h, dist.get_rank(group), self.config.world_size, bases))
            torch.cuda.synchronize(self.device)
            dist.barrier(group=group)      # every rank's flags are zero and mapped before the first kernel signals
        self._peer_state = ok
        return ok

    def _plan_peer_exchange(self, group):
        """With peers: updates that carry factor statistics and do not refresh the inverses keep the split exchange - the
        input-factor prefix A is summed by NCCL on a side stream UNDER phase 2, which itself sums [G | grads | scalars] over
        peer memory; the side stream then waits for that (acx_learner_wait_reduced), scales the statistics and runs the EMA.
        Everything else (cold / A2C updates, refresh updates) sums the whole bucket inside phase 2."""
        dist = torch.distributed
        self._after_phase2 = None
        if not self.config.acktr or os.environ.get("ACX_DP_SPLIT", "1") == "0":
            return
        has_factors, will_invert = ctypes.c_int(0), ctypes.c_int(0)
        _lib.check(self.lib.acx_learner_update_plan(self._h, ctypes.byref(has_factors), ctypes.byref(will_invert)))
        if not has_factors.value or will_invert.value:
            return
        if getattr(self, "_split_stream", None) is None:
            self._split_stream = torch.cuda.Stream(self.device)
            self._split_group = dist.new_group(ranks=dist.get_process_group_ranks(group or dist.group.WORLD), backend="nccl")
            self._p1_done, self._rest_done = torch.cuda.Event(), torch.cuda.Event()
            self._ema_done = torch.cuda.Event()
            self._split_a = self.buffer("input_factor_stats", torch.float32)
            self._split_rest = self.bucket[self._split_a.numel():]
        with self.on_stream():
            self._p1_done.record(self.stream)

        def after_phase2():     # enqueued behind the launch of phase 2, whose graph raises `reduced`
            with torch.cuda.stream(self._split_stream):
                self._split_stream.wait_event(self._p1_done)
                # ACX_PEER_PREFIX=1: the prefix over peer memory too (its own flag channel) - measured slower at 2 ranks (0.816 vs
                # 0.786 ms/update): the spinning CTAs of a second exchange kernel take more from phase 2 than NCCL's few do
                if os.environ.get("ACX_PEER_PREFIX", "0") != "0":
                    _lib.check(self.lib.acx_learner_peer_reduce_prefix(self._h, ctypes.c_void_p(self._split_stream.cuda_stream)))
                else:
                    dist.all_reduce(self._split_a, op=dist.ReduceOp.SUM, group=self._split_group)
                _lib.check(self.lib.acx_learner_wait_reduced(self._h, ctypes.c_void_p(self._split_stream.cuda_stream)))
                _lib.check(self.lib.acx_learner_ema(self._h, ctypes.c_void_p(self._split_stream.cuda_stream)))
                self._ema_done.record(self._split_stream)
        self._after_phase2 = after_phase2
        self._ema_external = True
        self._ema_pending = True

    def _split_exchange(self, group):
        """NCCL groups, K-FAC learners, covariance updates: phase 2 reads only [grads | scalars] of the bucket, so only
        [G | grads | scalars] (4.5 MB at conv3 = 32) is all-reduced on the engine's stream; the input-factor prefix A (13.6 MB)
        is all-reduced on a second stream and communicator UNDER phase 2, followed there by the statistics' 1/k scaling and
        the EMA (acx_learner_ema).  The engine's stream waits for that only before an inverse refresh and before the next
        phase 1 overwrites the statistics.  Same arithmetic in the same order as the single all-reduce: bit-identical
        (tools/dp_overlap_check.py).  ACX_DP_SPLIT=0 switches it off."""
        dist = torch.distributed
        if (not self.config.acktr or os.environ.get("ACX_DP_SPLIT", "1") == "0" or dist.get_backend(group) != "nccl"):
            return False
        has_factors, will_invert = ctypes.c_int(0), ctypes.c_int(0)
        _lib.check(self.lib.acx_learner_update_plan(self._h, ctypes.byref(has_factors), ctypes.byref(will_invert)))
        if not has_factors.value:
            return False
        if getattr(self, "_split_stream", None) is None:
            self._split_stream = torch.cuda.Stream(self.device)
            self._split_group = dist.new_group(ranks=dist.get_process_group_ranks(group or dist.group.WORLD), backend="nccl")
            self._p1_done, self._rest_done = torch.cuda.Event(), torch.cuda.Event()
            self._ema_done = torch.cuda.Event()
            self._split_a = self.buffer("input_factor_stats", torch.float32)
            self._split_rest = self.bucket[self._split_a.numel():]
        with self.on_stream():
            self._p1_done.record(self.stream)
            dist.all_reduce(self._split_rest, op=dist.ReduceOp.SUM, group=group)
            self._rest_done.record(self.stream)
            with torch.cuda.stream(self._split_stream):
                self._split_stream.wait_event(self._p1_done)
                dist.all_reduce(self._split_a, op=dist.ReduceOp.SUM, group=self._split_group)
                self._split_stream.wait_event(self._rest_done)      # the G statistics travel with the gradients
                _lib.check(self.lib.acx_learner_ema(self._h, ctypes.c_void_p(self._split_stream.cuda_stream)))
                self._ema_done.record(self._split_stream)
            if will_invert.value:
                self.stream.wait_event(self._ema_done)
        self._ema_external = True
        self._ema_pending = True
        return True

    def phase2(self):
        external = bool(getattr(self, "_ema_external", False))
        if self.config.world_size > 1:
            _lib.check(self.lib.acx_learner_set_external_ema(self._h, int(external)))
        self._ema_external = False
        with self.on_stream():
            _lib.check(self.lib.acx_learner_phase2(self._h, self._stream()))
        after, self._after_phase2 = getattr(self, "_after_phase2", None), None
        if after is not None:
            after()

    def update(self, batch=None, fisher_labels=None, fisher_eps=None, fetch=True, group=None, staged=False):
        """The reference's `session.run([..., optimize_op], feed_dict)` (a2c_acktr.py:117-126)."""
        if staged:
            self._consume_staged()
        elif batch is not None:
            self.load_batch(batch["observations"], batch["bootstrap_observations"], batch["actions"], batch["rewards"],
                            batch["terminals"])
        if self.config.world_size == 1:
            # nothing happens between the phases on a single GPU: both as one captured graph (acx_learner_update)
            fl = ctypes.c_void_p(fisher_labels.data_ptr()) if fisher_labels is not None else None
            fe = ctypes.c_void_p(fisher_eps.data_ptr()) if fisher_eps is not None else None
            with self.on_stream():
                _lib.check(self.lib.acx_learner_update(self._h, fl, fe, self._stream()))
        else:
            self.phase1(fisher_labels, fisher_eps)
            self.allreduce(group)
            self.phase2()
        return self._fetched(fetch)

    def update_separate(self, batch, policy_spec, baseline_spec, step_increments=(1, 1)):
        """objectives.py:31-54 `optimize_separate`: the gradient of the policy loss and the gradient of the baseline loss,
        both at the current parameters, each applied by its own optimizer (nn.standalone_spec records) with its own slots.
        `step_increments`: how often each `minimize` was handed the global step (it increments it once).  A2C-type
        engines only (acktr=False)."""
        from . import ops
        if self.config.acktr:
            raise _lib.AcxError("optimize_separate runs on a first-order engine (acktr=False)")
        if batch is not None:
            self.load_batch(batch["observations"], batch["bootstrap_observations"], batch["actions"], batch["rewards"],
                            batch["terminals"])
        if getattr(self, "_sep_slots", None) is None:
            def slot(kind):   # TF-1: RMSProp's `ms` starts at one, Momentum's accumulator at zero
                fill = torch.ones if kind == "rmsprop" else torch.zeros
                return fill(self.num_params, dtype=torch.float32, device=self.device)
            self._sep_slots = [slot(policy_spec[0]), slot(baseline_spec[0])]
        params = self.buffer("params", torch.float32)[: self.num_params]
        grads = self.buffer("grads", torch.float32)[: self.num_params]
        gs = self.global_step
        with self.on_stream(), torch.cuda.stream(self.stream):
            _lib.check(self.lib.acx_learner_set_loss_weights(self._h, 1.0, 0.0))
            _lib.check(self.lib.acx_learner_phase1(self._h, None, None, self._stream()))
            g_policy = grads.clone()
            scalars = self.bucket[-4:].clone()
            _lib.check(self.lib.acx_learner_set_loss_weights(self._h, 0.0, 1.0))
            _lib.check(self.lib.acx_learner_phase1(self._h, None, None, self._stream()))
            _lib.check(self.lib.acx_learner_set_loss_weights(self._h, 1.0, float(self.config.value_loss_weight)))
            norms = []
            for (kind, lr, hp, clip), g, slot_t in ((policy_spec, g_policy, self._sep_slots[0]),
                                                    (baseline_spec, grads, self._sep_slots[1])):
                step_fn = ops.clip_rmsprop_step if kind == "rmsprop" else ops.clip_momentum_step
                norms.append(step_fn(params, slot_t, g, lr.value_at(gs), clip_norm=clip, **hp))
            _lib.check(self.lib.acx_learner_refresh_weights(self._h, self._stream()))
        self.set_state(gs + int(sum(step_increments)), 0, False)
        vals = scalars.cpu().tolist()
        return dict(policy_loss=vals[0], baseline_loss=vals[1], mean_entropy=vals[2], loss=vals[0] + vals[1],
                    clip_coeff=float("nan"), fisher_norm=float("nan"), grad_norm=float(norms[0]),
                    learning_rate=float(policy_spec[1].value_at(gs)), baseline_grad_norm=float(norms[1]))

    # ------------------------------------------------------------------ stage timing
    STAGES = ("forward", "loss_heads", "backward", "factors", "ema_or_cold", "inverse", "precondition", "apply")

    def set_profiling(self, enable=True):
        _lib.check(self.lib.acx_learner_set_profiling(self._h, int(bool(enable))))

    def stage_ms(self):
        arr = (ctypes.c_float * 8)()
        _lib.check(self.lib.acx_learner_stage_ms(self._h, arr))
        return dict(zip(self.STAGES, [float(x) for x in arr]))


# ---------------------------------------------------------------------------------------------------------------------
# fully connected models (MLPModel, include/acx.h `acx_mlp_*`)
# ---------------------------------------------------------------------------------------------------------------------
def mlp_layers(num_hidden):
    """Block names of a fully connected model with `num_hidden` hidden layers, in the order of the flat parameter vector."""
    return tuple("fc%d" % (i + 1) for i in range(num_hidden)) + ("fc_policy", "fc_baseline")


def mlp_param_shapes(obs_dim, hidden_sizes, num_actions):
    """nn.fully_connected_params layout: weights [in, out], bias [out]."""
    ins = [int(obs_dim)] + [int(h) for h in hidden_sizes]
    outs = [int(h) for h in hidden_sizes] + [int(num_actions), 1]
    ins.append(ins[-1])                     # both heads read the last hidden layer
    shapes = {}
    for name, k, c in zip(mlp_layers(len(hidden_sizes)), ins, outs):
        shapes[name + "/weights"], shapes[name + "/bias"] = (k, c), (c,)
    return shapes


@dataclasses.dataclass
class MLPEngineConfig:
    num_envs: int = 16
    num_steps: int = 5
    obs_dim: int = 4
    hidden_sizes: tuple = (64, 64)
    num_actions: int = 2
    acktr: bool = True
    gamma: float = 0.99
    entropy_beta: float = 0.01
    value_loss_weight: float = 0.5
    lr_start: float = 0.25
    lr_end: float = 0.025
    lr_decay_steps: float = None            # None: 1e7 / (num_envs * num_steps), as EngineConfig
    cov_ema_decay: float = 0.99
    damping: float = 0.01
    momentum: float = 0.9
    norm_constraint: float = 0.0001
    invert_every: int = 10
    num_cold_updates: int = 30
    cold_lr: float = 0.0003
    cold_momentum: float = 0.9
    clip_norm: float = 0.5
    rms_decay: float = 0.9
    rms_epsilon: float = 1e-10
    use_graphs: bool = True
    seed: int = 0

    def to_c(self):
        c = _lib.MLPConfig()
        c.num_envs, c.num_steps, c.obs_dim, c.num_actions = self.num_envs, self.num_steps, self.obs_dim, self.num_actions
        if not 1 <= len(self.hidden_sizes) <= 4:
            raise ValueError("1 to 4 hidden layers")
        c.num_hidden = len(self.hidden_sizes)
        for i, h in enumerate(self.hidden_sizes):
            c.hidden[i] = int(h)
        c.acktr = int(self.acktr)
        c.gamma, c.entropy_beta, c.value_loss_weight = self.gamma, self.entropy_beta, self.value_loss_weight
        c.lr_start, c.lr_end = self.lr_start, self.lr_end
        steps = self.lr_decay_steps
        c.lr_decay_steps = float(steps) if steps is not None else 1e7 / (self.num_envs * self.num_steps)
        c.cov_ema_decay, c.damping, c.momentum = self.cov_ema_decay, self.damping, self.momentum
        c.norm_constraint = self.norm_constraint
        c.invert_every, c.num_cold_updates = self.invert_every, self.num_cold_updates
        c.cold_lr, c.cold_momentum, c.clip_norm = self.cold_lr, self.cold_momentum, self.clip_norm
        c.rms_decay, c.rms_epsilon = self.rms_decay, self.rms_epsilon
        c.use_graphs, c.seed = int(bool(self.use_graphs)), self.seed
        return c


class MLPEngine(_ArenaEngine):
    """Learner of a fully connected actor-critic model on flat float32 observations [rows, obs_dim]: one update
    (`update`) is one captured CUDA graph of acx_mlp_update."""

    _API = "acx_mlp_"
    _OBS_DTYPE = torch.float32

    def __init__(self, config, device=None):
        self._open(config, device, (config.obs_dim,))
        self.layers = mlp_layers(len(config.hidden_sizes))
        self._shapes = mlp_param_shapes(config.obs_dim, config.hidden_sizes, config.num_actions)

    def _flatten(self, params):
        parts = []
        for layer in self.layers:
            w = np.asarray(params[layer + "/weights"], np.float32)
            b = np.asarray(params[layer + "/bias"], np.float32)
            if w.shape != self._shapes[layer + "/weights"] or b.shape != self._shapes[layer + "/bias"]:
                raise ValueError("bad shape for layer %s: %s / %s" % (layer, w.shape, b.shape))
            parts += [w.ravel(), b.ravel()]
        return np.concatenate(parts)

    def _unflatten(self, flat):
        out, off = {}, 0
        for layer in self.layers:
            for kind in ("weights", "bias"):
                shape = self._shapes[layer + "/" + kind]
                n = int(np.prod(shape))
                out[layer + "/" + kind] = np.asarray(flat[off:off + n]).reshape(shape).copy()
                off += n
        return out

    def _layer_cols(self, layer):
        return self._shapes[layer + "/bias"][0]

    # Session.run drives a train step as phase1 / allreduce / phase2: here the whole update is one call (one graph), so
    # phase1 only takes the Fisher samples and phase2 runs it; the loss scalars are read after phase2.
    def phase1(self, fisher_labels=None, fisher_eps=None):
        self._fisher = (fisher_labels, fisher_eps)

    def allreduce(self, group=None):
        pass

    def phase2(self):
        fl, fe = getattr(self, "_fisher", (None, None))
        self._fisher = (None, None)
        self.update(None, fl, fe, fetch=False)

    def update(self, batch=None, fisher_labels=None, fisher_eps=None, fetch=True):
        """The reference's `session.run([..., optimize_op], feed_dict)` (a2c_acktr.py:117-126) for this model."""
        if batch is not None:
            self.load_batch(batch["observations"], batch["bootstrap_observations"], batch["actions"], batch["rewards"],
                            batch["terminals"])
        fl = ctypes.c_void_p(fisher_labels.data_ptr()) if fisher_labels is not None else None
        fe = ctypes.c_void_p(fisher_eps.data_ptr()) if fisher_eps is not None else None
        with self.on_stream():
            _lib.check(self.lib.acx_mlp_update(self._h, fl, fe, self._stream()))
        return self._fetched(fetch)


# ---------------------------------------------------------------------------------------------------------------------
# convolutional models on square images (CNNModel, include/acx.h `acx_cnn_*`: the fully connected learner with a conv trunk)
# ---------------------------------------------------------------------------------------------------------------------
def cnn_layers(num_conv, num_hidden):
    """Block names in the order of the flat parameter vector: conv1 .. convK, fc(K+1) .. fc(K+L), the heads."""
    return (tuple("conv%d" % (i + 1) for i in range(num_conv)) + tuple("fc%d" % (num_conv + i + 1) for i in range(num_hidden))
            + ("fc_policy", "fc_baseline"))


def cnn_conv_geometry(obs_hw, obs_channels, conv_layers):
    """[(hw_in, c_in, filters, kernel, stride, hw_out)] per conv layer (VALID)."""
    out, hw, c = [], int(obs_hw), int(obs_channels)
    for f, k, s in conv_layers:
        o = (hw - int(k)) // int(s) + 1
        out.append((hw, c, int(f), int(k), int(s), o))
        hw, c = o, int(f)
    return out


def cnn_param_shapes(obs_hw, obs_channels, conv_layers, hidden_sizes, num_actions):
    """nn.conv2d_params (HWIO [k, k, c_in, filters]) for the conv layers, nn.fully_connected_params ([in, out]) after them."""
    geo = cnn_conv_geometry(obs_hw, obs_channels, conv_layers)
    names = cnn_layers(len(geo), len(hidden_sizes))
    shapes = {}
    for name, (_, c, f, k, _, _) in zip(names, geo):
        shapes[name + "/weights"], shapes[name + "/bias"] = (k, k, c, f), (f,)
    hw, c = geo[-1][5], geo[-1][2]
    ins = [hw * hw * c] + [int(h) for h in hidden_sizes]
    outs = [int(h) for h in hidden_sizes] + [int(num_actions), 1]
    ins.append(ins[-1])
    for name, k, c in zip(names[len(geo):], ins, outs):
        shapes[name + "/weights"], shapes[name + "/bias"] = (k, c), (c,)
    return shapes


@dataclasses.dataclass
class CNNEngineConfig(MLPEngineConfig):
    obs_hw: int = 84
    obs_channels: int = 4
    obs_u8: bool = True
    conv_layers: tuple = ((32, 8, 4), (64, 4, 2), (64, 3, 1))   # (filters, kernel, stride) per layer, VALID
    hidden_sizes: tuple = (512,)
    obs_dim: int = None                                          # derived: obs_hw * obs_hw * obs_channels

    def to_c(self):
        if not 1 <= len(self.conv_layers) <= 3:
            raise ValueError("1 to 3 conv layers")
        c = _lib.CNNConfig()
        c.mlp = MLPEngineConfig.to_c(dataclasses.replace(self, obs_dim=self.obs_hw * self.obs_hw * self.obs_channels))
        c.obs_hw, c.obs_channels, c.obs_u8, c.num_conv = self.obs_hw, self.obs_channels, int(bool(self.obs_u8)), len(self.conv_layers)
        for i, (f, k, s) in enumerate(self.conv_layers):
            c.filters[i], c.kernel[i], c.stride[i] = int(f), int(k), int(s)
        return c


class CNNEngine(MLPEngine):
    """Learner of a convolutional actor-critic model on square images [rows, H, H, C] (uint8 or float32 as configured):
    acx_cnn_create / acx_cnn_act, and every other call of the fully connected learner (acx_mlp_*) on the same handle."""

    _CNN_CALLS = ("arena_bytes", "create", "act")

    def __init__(self, config, device=None):
        self._OBS_DTYPE = torch.uint8 if config.obs_u8 else torch.float32
        self._open(config, device, (config.obs_hw, config.obs_hw, config.obs_channels))
        self.layers = cnn_layers(len(config.conv_layers), len(config.hidden_sizes))
        self._shapes = cnn_param_shapes(config.obs_hw, config.obs_channels, config.conv_layers, config.hidden_sizes,
                                        config.num_actions)

    def _fn(self, name):
        return getattr(self.lib, ("acx_cnn_" if name in self._CNN_CALLS else "acx_mlp_") + name)

    def _layer_cols(self, layer):
        return self._shapes[layer + "/bias"][0]
