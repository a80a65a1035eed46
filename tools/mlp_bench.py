"""Time the fully connected learner (acx_mlp_update) on the GPU: one JSON line per configuration and optimizer.

Per line: ms per update from CUDA events over the timed updates (after a warm-up past the first inverse refresh, so
every CUDA graph variant is captured), env-steps/s, kernel launches per update (acx_launch_count; a replayed graph
counts its nodes), the GPU's name and power limit read in the same run, whether the batch working set fits L2, and the
float32 oracle (oracle/mlp.py) timed on all host threads as the CPU baseline.  The batch stays in device memory:
this measures the learner, not the host feed.

    python tools/mlp_bench.py [--steps 200] [--warmup 60] [--cpu-updates 10] [--out profiles/mlp_bench.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from actorcritic_b200 import _lib, engine as eng  # noqa: E402
from oracle import kfac as K  # noqa: E402
from oracle import learner as OL  # noqa: E402
from oracle import mlp as OM  # noqa: E402

CONFIGS = {
    "small": dict(obs_dim=8, hidden_sizes=(64, 64), num_actions=4, num_envs=16, num_steps=5),
    "large": dict(obs_dim=128, hidden_sizes=(256, 256), num_actions=8, num_envs=256, num_steps=20),
}


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    name, power = (out[torch.cuda.current_device()].split(", ") + ["?"])[:2] if out else (torch.cuda.get_device_name(), "?")
    return name, power


def batch(cfg, seed=0):
    rng = np.random.default_rng(seed)
    e, t, d = cfg.num_envs, cfg.num_steps, cfg.obs_dim
    return dict(observations=rng.standard_normal((e, t, d)).astype(np.float32),
                bootstrap_observations=rng.standard_normal((e, d)).astype(np.float32),
                actions=rng.integers(0, cfg.num_actions, (e, t)).astype(np.uint8),
                rewards=rng.standard_normal((e, t)).astype(np.float32), terminals=rng.random((e, t)) < 0.05)


def batch_bytes(cfg):
    """Bytes one update streams per batch: fp32 observations, the bf16 plane pairs of the input and every hidden
    activation (N+E rows), the pre-activation gradients (2N rows), rewards / actions / terminals and the head gradients."""
    n = cfg.num_envs * cfg.num_steps
    r = n + cfg.num_envs
    widths = [cfg.obs_dim] + list(cfg.hidden_sizes)
    return (r * cfg.obs_dim * 4 + sum(2 * r * w * 2 for w in widths) + sum(2 * 2 * n * h * 2 for h in cfg.hidden_sizes)
            + n * 6 + 2 * n * (cfg.num_actions + 1) * 4)


def cpu_baseline_ms(cfg, params, updates):
    torch.set_num_threads(os.cpu_count())
    n = cfg.num_envs * cfg.num_steps
    if cfg.acktr:
        ocfg = K.KfacConfig(num_cold_updates=0, invert_every=cfg.invert_every)
    else:
        ocfg = OL.A2CConfig()
    o = OM.MLPOracle(params, len(cfg.hidden_sizes), acktr=cfg.acktr, cfg=ocfg, dtype=torch.float32)
    b = batch(cfg)
    rng = np.random.default_rng(1)
    y, eps = rng.integers(0, cfg.num_actions, n), rng.standard_normal(n)
    o.update(b, y, eps)
    t0 = time.perf_counter()
    for _ in range(updates):
        o.update(b, y, eps)
    return (time.perf_counter() - t0) * 1e3 / updates


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=60)
    ap.add_argument("--cpu-updates", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mlp_bench.py measures on a CUDA device; none found")
    gpu, power = gpu_info()
    l2 = torch.cuda.get_device_properties(0).L2_cache_size
    lines = []
    for size, shape in CONFIGS.items():
        for acktr in (True, False):
            # the reference example's schedule (a2c_acktr.py:240-247): 30 cold updates, inverses every 10 updates
            cfg = eng.MLPEngineConfig(acktr=acktr, seed=1, **shape) if acktr else eng.MLPEngineConfig(
                acktr=False, lr_start=7e-4, lr_end=7e-5, seed=1, **shape)
            e = eng.MLPEngine(cfg)
            rng = np.random.default_rng(0)
            shapes = eng.mlp_param_shapes(cfg.obs_dim, cfg.hidden_sizes, cfg.num_actions)
            params = {k: (0.1 * rng.standard_normal(s)).astype(np.float32) for k, s in shapes.items()}
            e.set_params(params)
            e.load_batch(**batch(cfg))
            for _ in range(max(args.warmup, cfg.num_cold_updates + 2 * cfg.invert_every if acktr else 3)):
                e.update(fetch=False)
            torch.cuda.synchronize()
            l0 = _lib.launch_count()
            start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            start.record(e.stream)
            for _ in range(args.steps):
                e.update(fetch=False)
            end.record(e.stream)
            end.synchronize()
            ms = start.elapsed_time(end) / args.steps
            launches = (_lib.launch_count() - l0) / args.steps
            n = cfg.num_envs * cfg.num_steps
            bb = batch_bytes(cfg)
            rec = dict(config=size, optimizer="acktr" if acktr else "a2c", obs_dim=cfg.obs_dim,
                       hidden_sizes=list(cfg.hidden_sizes), num_actions=cfg.num_actions, num_envs=cfg.num_envs,
                       num_steps=cfg.num_steps, timed_updates=args.steps, ms_per_update=round(ms, 4),
                       env_steps_per_s=round(n / (ms / 1e3), 1), launches_per_update=launches,
                       batch_bytes=bb, l2_bytes=l2, batch_fits_l2=bool(bb < l2), gpu=gpu, power_limit=power,
                       cpu_baseline_ms_per_update=round(cpu_baseline_ms(cfg, params, args.cpu_updates), 3),
                       cpu_threads=os.cpu_count(), scalars=e.fetch_scalars())
            print(json.dumps(rec), flush=True)
            lines.append(rec)
            del e
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
