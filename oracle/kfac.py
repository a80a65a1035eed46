"""Oracle for the K-FAC part of the ACKTR update (torch-CPU, dtype selectable; float64 for parity).

PARITY UNPINNED: the arithmetic lives in tensorflow/kfac 0.1.x ("latest version (0.1.1)",
README.md:27-31, requirements.txt:3, no commit pin) which is neither vendored under
/root/reference nor installable here.  This restates its published algorithm as SURVEY A.5
records it and anchors on the reference's call sites:
  registration  envs/atari/model.py:219-246, policies.py:146-158, baselines.py:55-66
  schedule      kfac_utils.py:38-53
  hyper-params  a2c_acktr.py:240-247
Unpinned choices (SURVEY A.7 U1-U6) are explicit parameters of KfacConfig.
"""
import dataclasses
import math

import numpy as np
import torch

from . import network as net

TRUE_LOCATIONS = {"conv1": 400, "conv2": 81, "conv3": 49, "fc4": 1, "fc_policy": 1, "fc_baseline": 1}
# kfac 0.1.x num_conv_locations = prod(input spatial) // prod(strides)  (SURVEY A.7-U1)
INPUT_DIV_STRIDE_LOCATIONS = {"conv1": 84 * 84 // 16, "conv2": 20 * 20 // 4, "conv3": 9 * 9 // 1,
                              "fc4": 1, "fc_policy": 1, "fc_baseline": 1}
# the two heads are registered with the same `inputs` tensor (envs/atari/model.py:243,246) => one shared factor
A_FACTOR_OF = {"conv1": "conv1", "conv2": "conv2", "conv3": "conv3", "fc4": "fc4",
               "fc_policy": "heads", "fc_baseline": "heads"}
A_FACTORS = ("conv1", "conv2", "conv3", "fc4", "heads")


@dataclasses.dataclass
class KfacConfig:
    learning_rate_start: float = 0.25          # a2c_acktr.py:68
    learning_rate_end: float = 0.025
    decay_steps: float = 1e7 / (32 * 20)       # a2c_acktr.py:64
    cov_ema_decay: float = 0.99                # a2c_acktr.py:245
    damping: float = 0.01
    momentum: float = 0.9
    norm_constraint: float = 1e-4
    invert_every: int = 10
    num_cold_updates: int = 30                 # a2c_acktr.py:244
    cold_learning_rate: float = 3e-4           # a2c_acktr.py:240
    cold_momentum: float = 0.9
    clip_norm: float = 0.5                     # a2c_acktr.py:241
    num_locations_mode: str = "true"           # or "input_div_stride" (U1)
    zero_debias: bool = True                   # U3
    cov_init: str = "zero"                     # U3 ("zero" | "identity")
    inv_init: str = "zero"                     # U3 ("zero" | "identity"): initial value of the stored inverses

    def locations(self, layer):
        table = TRUE_LOCATIONS if self.num_locations_mode == "true" else INPUT_DIV_STRIDE_LOCATIONS
        return table[layer]


def schedule_events(global_step, num_cold_updates, invert_every):
    """What ONE call of ColdStartPeriodicInvUpdateKfacOpt.apply_gradients does when it starts at `global_step`, as coded
    (kfac_utils.py:38-53; pinned by tests/golden/schedule.npz, recorded from the reference class itself):
      :41-44  global_step < num_cold_updates ? cold optimizer (increments global_step) : covariance updates
      :47-50  then, reading the CURRENT global_step: > num_cold_updates and (gs - num_cold_updates) % invert_every == 0
              -> inverse updates
      :52-53  then always KfacOptimizer.apply_gradients (increments global_step).
    Returns dict(cold, cov, inv, kfac_apply, gs_after)."""
    cold = global_step < num_cold_updates
    gs1 = global_step + (1 if cold else 0)
    inv = gs1 > num_cold_updates and (gs1 - num_cold_updates) % invert_every == 0
    return dict(cold=cold, cov=not cold, inv=inv, kfac_apply=True, gs_after=gs1 + 1)


def linear_decay(start, end, step, total_steps):
    """nn.py:154-156 (tf.train.polynomial_decay, power 1, cycle False)."""
    s = min(float(step), float(total_steps))
    return (start - end) * (1.0 - s / float(total_steps)) + end


def append_homog(x):
    return torch.cat([x, torch.ones((x.shape[0], 1), dtype=x.dtype)], 1)


def input_factor(x):
    """A = [x 1]^T [x 1] / rows, symmetrised (SURVEY A.5 'Input factor', U5)."""
    xh = append_homog(x)
    c = xh.T @ xh / x.shape[0]
    return (c + c.T) / 2


def output_factor(g):
    """G = g^T g / rows (SURVEY A.5 'Output factor')."""
    c = g.T @ g / g.shape[0]
    return (c + c.T) / 2


def batch_factors(fwd, fisher_pre_grads):
    """The 11 new covariance contributions of one batch.  fwd from network.forward on the N train
    rows only; fisher_pre_grads from network.backward with the Fisher-sample output gradients."""
    a = {
        "conv1": input_factor(fwd["conv1"]["patches"]),
        "conv2": input_factor(fwd["conv2"]["patches"]),
        "conv3": input_factor(fwd["conv3"]["patches"]),
        "fc4": input_factor(fwd["fc4"]["inputs"]),
        "heads": input_factor(fwd["heads_inputs"]),
    }
    g = {name: output_factor(fisher_pre_grads[name]) for name in net.LAYERS}
    return a, g


def pi_dampings(a, g, lam):
    """pi-adjusted damping of one block (SURVEY A.5 'Damping') from its input and output factors:
    pi = sqrt((tr A / dim A) / (tr G / dim G)) (1 when either trace is not positive), returns (pi sqrt(lam), sqrt(lam) / pi).
    A common scale of A and G (the zero-debias factor) cancels in pi."""
    tr_a = torch.trace(a) / a.shape[0]
    tr_g = torch.trace(g) / g.shape[0]
    pi = math.sqrt(float(tr_a) / float(tr_g)) if float(tr_a) > 0 and float(tr_g) > 0 else 1.0
    root = math.sqrt(lam)
    return pi * root, root / pi


def damped_inverse(s, debias, damp):
    """(debias * sym(S) + damp * I)^-1 of a running sum S, sym(S) = (S + S^T) / 2 (the kernels symmetrise the sums they
    load; a symmetric S is used exactly as it is)."""
    s = torch.as_tensor(s)
    m = 0.5 * (s + s.T) * debias
    return torch.linalg.inv(m + damp * torch.eye(s.shape[0], dtype=s.dtype))


# ------------------------------------------------------------------------------------------------ test factors
# Seeded fp32 running sums for the inverse-refresh tests (tests/test_gpu_kfac_inverse.py), as float64 tensors whose values are
# exactly representable in fp32.
def gram_factor(n, rows, seed, homogeneous=True, scale_octaves=14):
    """S = X^T X / rows, X [rows, n] of small integers times per-column powers of two in [2^-scale_octaves, 1] (the last
    column all ones with `homogeneous`, as the border of an input factor).  rows a power of two: every entry of S is then
    computed exactly and is exactly representable in fp32, so S is exactly PSD with rank min(rows, n), and the extreme
    eigenvalues come from the smaller Gram matrix.  Returns (S, lam_min, lam_max), lam_min = 0 when rows < n."""
    assert rows & (rows - 1) == 0 and rows <= 4096
    rng = np.random.default_rng(seed)
    x = rng.integers(-7, 8, (rows, n)).astype(np.float64) * np.exp2(-rng.integers(0, scale_octaves + 1, n))
    if homogeneous:
        x[:, -1] = 1.0
    x = torch.from_numpy(x)
    s = x.T @ x / rows
    small = s if rows >= n else x @ x.T / rows
    lam = torch.linalg.eigvalsh(small)
    assert torch.equal(s, s.float().double())
    return s, (float(lam[0]) if rows >= n else 0.0), float(lam[-1])


def spectrum_factor(eigenvalues, seed):
    """Q diag(eigenvalues) Q^T with a seeded random orthogonal Q, rounded to fp32 (so its spectrum is the prescribed one
    up to fp32 rounding, relative to the largest eigenvalue)."""
    lam = torch.as_tensor(np.asarray(eigenvalues, np.float64))
    n = lam.shape[0]
    q, r = torch.linalg.qr(torch.from_numpy(np.random.default_rng(seed).standard_normal((n, n))))
    q = q * torch.sign(torch.diagonal(r))
    s = (q * lam) @ q.T
    return (0.5 * (s + s.T)).float().double()


def zero_factor(n):
    """An all-zero running sum: its trace is 0, so pi falls back to 1 for its block."""
    return torch.zeros((n, n), dtype=torch.float64)


def with_antisymmetric_ulp(s):
    """S plus a one-ulp antisymmetric part: above the diagonal every other entry of S moves one fp32 ulp up, its mirror one
    ulp down - what the kernels must symmetrise away (sym of the result equals sym of S up to half an ulp)."""
    s32 = s.float().numpy().copy()
    iu = np.triu_indices(s32.shape[0], 1)
    i, j = iu[0][::2], iu[1][::2]
    s32[i, j] = np.nextafter(s32[i, j], np.float32(np.inf))
    s32[j, i] = np.nextafter(s32[j, i], np.float32(-np.inf))
    return torch.from_numpy(s32).double()


def damping_for_kappa(a, g, kappa, debias=1.0, tnorm=1, lam_min=None, lam_max=None):
    """The `damping` hyper-parameter at which the damped input factor debias * sym(A) + damp_A I of a block reaches the
    condition number `kappa`, with damp_A from the fp64 pi formula (lam = damping / tnorm).  lam_min / lam_max: the extreme
    eigenvalues of sym(A) when known (else computed)."""
    if lam_min is None or lam_max is None:
        lam = torch.linalg.eigvalsh(0.5 * (a + a.T))
        lam_min, lam_max = float(lam[0]), float(lam[-1])
    damp_a = debias * (lam_max - kappa * lam_min) / (kappa - 1.0)
    assert damp_a > 0, "kappa %g is beyond the factor's own condition number" % kappa
    pi = pi_dampings(a, g, 1.0)[0]   # damp_A = pi sqrt(lam)
    return (damp_a / pi) ** 2 * tnorm


class KfacState:
    """Running covariance sums, debias counter, stored inverses, velocities (SURVEY A.5)."""

    def __init__(self, params, cfg, dtype=torch.float64):
        self.cfg, self.dtype = cfg, dtype
        dims_a = {"conv1": 257, "conv2": 513, "conv3": 577,
                  "fc4": params["fc4/weights"].shape[0] + 1, "heads": 513}
        dims_g = {name: params[name + "/weights"].shape[-1] for name in net.LAYERS}

        def init(d):
            return torch.eye(d, dtype=dtype) if cfg.cov_init == "identity" else torch.zeros((d, d), dtype=dtype)
        self.sum_a = {k: init(d) for k, d in dims_a.items()}
        self.sum_g = {k: init(d) for k, d in dims_g.items()}
        self.num_cov_updates = 0

        def init_inv(d):   # kfac 0.1.x: zeros (the K-FAC step is a no-op until the first refresh); older contrib.kfac: identity
            return torch.eye(d, dtype=dtype) if cfg.inv_init == "identity" else torch.zeros((d, d), dtype=dtype)
        self.inv_a = {name: init_inv(dims_a[A_FACTOR_OF[name]]) for name in net.LAYERS}
        self.inv_g = {name: init_inv(dims_g[name]) for name in net.LAYERS}
        self.velocity = {name: torch.zeros_like(net.join_vmat(name, params)) for name in net.LAYERS}

    def update_covs(self, new_a, new_g):
        d = self.cfg.cov_ema_decay
        for k in self.sum_a:
            self.sum_a[k] = d * self.sum_a[k] + (1 - d) * new_a[k]
        for k in self.sum_g:
            self.sum_g[k] = d * self.sum_g[k] + (1 - d) * new_g[k]
        self.num_cov_updates += 1

    def _debias(self):
        if self.cfg.zero_debias and self.cfg.cov_init == "zero":
            if self.num_cov_updates == 0:
                return 1.0
            return 1.0 / (1.0 - self.cfg.cov_ema_decay ** self.num_cov_updates)
        return 1.0

    def cov_a(self, factor):
        return self.sum_a[factor] * self._debias()

    def cov_g(self, layer):
        return self.sum_g[layer] * self._debias()

    def dampings(self, layer):
        """pi-adjusted damping of one block: (damp_A, damp_G)."""
        return pi_dampings(self.cov_a(A_FACTOR_OF[layer]), self.cov_g(layer), self.cfg.damping / self.cfg.locations(layer))

    def update_inverses(self):
        for layer in net.LAYERS:
            damp_a, damp_g = self.dampings(layer)
            self.inv_a[layer] = damped_inverse(self.sum_a[A_FACTOR_OF[layer]], self._debias(), damp_a)
            self.inv_g[layer] = damped_inverse(self.sum_g[layer], self._debias(), damp_g)

    def precondition(self, grads):
        """U_l = A^-1 V_l G^-1 / T~_l with the STORED inverses."""
        return {layer: self.inv_a[layer] @ grads[layer] @ self.inv_g[layer] / self.cfg.locations(layer)
                for layer in net.LAYERS}

    def clip_coeff(self, grads, precon, lr):
        s = sum(float((grads[l] * precon[l]).sum()) for l in net.LAYERS)
        if s <= 0.0:
            return 1.0, s
        return min(1.0, math.sqrt(self.cfg.norm_constraint / (lr * lr * s))), s

    def step(self, params, grads, lr):
        """precondition -> KL clip -> momentum -> theta -= lr * v.  Returns (coeff, s, updates)."""
        precon = self.precondition(grads)
        coeff, s = self.clip_coeff(grads, precon, lr)
        for layer in net.LAYERS:
            self.velocity[layer] = self.cfg.momentum * self.velocity[layer] + coeff * precon[layer]
            new = net.join_vmat(layer, params) - lr * self.velocity[layer]
            w, b = net.split_vmat(layer, new, params)
            params[layer + "/weights"], params[layer + "/bias"] = w, b
        return coeff, s, precon


def global_norm(grads):
    return math.sqrt(sum(float((g * g).sum()) for g in grads.values()))


def clip_by_global_norm(grads, clip_norm):
    """nn.py:185-187 / tf.clip_by_global_norm: g * clip / max(norm, clip)."""
    norm = global_norm(grads)
    scale = clip_norm / max(norm, clip_norm)
    return {k: g * scale for k, g in grads.items()}, norm
