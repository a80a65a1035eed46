"""Time the convolutional learner (acx_cnn_create + acx_mlp_update) on the GPU: one JSON line per configuration and optimizer.

Per line: ms per update from CUDA events over the timed updates (after a warm-up past the first inverse refresh, so
every CUDA graph variant is captured), env-steps/s, kernel launches per update (acx_launch_count; a replayed graph
counts its nodes), the GPU's name and power limit read in the same run, and the float32 oracle (oracle/cnn.py) timed on
all host threads as the CPU baseline.  At the Nature geometry the same line carries AtariModel's specialised learner
(engine.Engine) timed the same way on the same batch, and the ratio.  The batch stays in device memory: this measures the
learner, not the host feed.

    python tools/cnn_bench.py [--steps 100] [--warmup 60] [--cpu-updates 3] [--out profiles/cnn_bench_1gpu.jsonl]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from actorcritic_b200 import _lib, engine as eng  # noqa: E402
from mlp_bench import gpu_info  # noqa: E402
from oracle import cnn as OC  # noqa: E402
from oracle import kfac as K  # noqa: E402
from oracle import learner as OL  # noqa: E402

CONFIGS = {
    "minatar": dict(obs_hw=10, obs_channels=7, obs_u8=False, conv_layers=((16, 3, 1),), hidden_sizes=(128,), num_actions=6,
                    num_envs=256, num_steps=5),
    "procgen": dict(obs_hw=64, obs_channels=3, obs_u8=True, conv_layers=((32, 8, 4), (64, 4, 2), (64, 3, 1)),
                    hidden_sizes=(256,), num_actions=15, num_envs=64, num_steps=5),
    "nature": dict(obs_hw=84, obs_channels=4, obs_u8=True, conv_layers=((32, 8, 4), (64, 4, 2), (32, 3, 1)),
                   hidden_sizes=(512,), num_actions=6, num_envs=32, num_steps=20),
}


def batch(cfg, seed=0):
    rng = np.random.default_rng(seed)
    e, t = cfg.num_envs, cfg.num_steps
    img = (cfg.obs_hw, cfg.obs_hw, cfg.obs_channels)
    if cfg.obs_u8:
        obs, boot = rng.integers(0, 256, (e, t) + img).astype(np.uint8), rng.integers(0, 256, (e,) + img).astype(np.uint8)
    else:
        obs, boot = rng.standard_normal((e, t) + img).astype(np.float32), rng.standard_normal((e,) + img).astype(np.float32)
    return dict(observations=obs, bootstrap_observations=boot, actions=rng.integers(0, cfg.num_actions, (e, t)).astype(np.uint8),
                rewards=rng.standard_normal((e, t)).astype(np.float32), terminals=rng.random((e, t)) < 0.05)


def params_for(cfg):
    rng = np.random.default_rng(0)
    shapes = eng.cnn_param_shapes(cfg.obs_hw, cfg.obs_channels, cfg.conv_layers, cfg.hidden_sizes, cfg.num_actions)
    return {k: (0.05 * rng.standard_normal(s)).astype(np.float32) for k, s in shapes.items()}


def time_engine(e, cfg, steps, warmup):
    """ms per update and launches per update of `e` with its batch loaded."""
    for _ in range(max(warmup, cfg.num_cold_updates + 2 * cfg.invert_every if cfg.acktr else 3)):
        e.update(fetch=False)
    torch.cuda.synchronize()
    l0 = _lib.launch_count()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record(e.stream)
    for _ in range(steps):
        e.update(fetch=False)
    end.record(e.stream)
    end.synchronize()
    return start.elapsed_time(end) / steps, (_lib.launch_count() - l0) / steps


def cpu_baseline_ms(cfg, params, updates):
    torch.set_num_threads(os.cpu_count())
    n = cfg.num_envs * cfg.num_steps
    ocfg = K.KfacConfig(num_cold_updates=0, invert_every=cfg.invert_every) if cfg.acktr else OL.A2CConfig()
    o = OC.CNNOracle(params, cfg.obs_hw, cfg.obs_channels, cfg.conv_layers, len(cfg.hidden_sizes), obs_u8=cfg.obs_u8,
                     acktr=cfg.acktr, cfg=ocfg, dtype=torch.float32)
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
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=60)
    ap.add_argument("--cpu-updates", type=int, default=3)
    ap.add_argument("--configs", default=",".join(CONFIGS))
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "cnn_bench_1gpu.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("cnn_bench.py measures on a CUDA device; none found")
    gpu, power = gpu_info()
    lines = []
    for size in args.configs.split(","):
        shape = CONFIGS[size]
        for acktr in (True, False):
            # the reference example's schedule (a2c_acktr.py:240-247): 30 cold updates, inverses every 10 updates
            opt = dict(seed=1) if acktr else dict(acktr=False, lr_start=7e-4, lr_end=7e-5, seed=1)
            cfg = eng.CNNEngineConfig(**opt, **shape)
            e = eng.CNNEngine(cfg)
            params = params_for(cfg)
            e.set_params(params)
            b = batch(cfg)
            e.load_batch(**b)
            ms, launches = time_engine(e, cfg, args.steps, args.warmup)
            n = cfg.num_envs * cfg.num_steps
            rec = dict(config=size, optimizer="acktr" if acktr else "a2c", obs_shape=[cfg.obs_hw, cfg.obs_hw, cfg.obs_channels],
                       obs_dtype="uint8" if cfg.obs_u8 else "float32", conv_layers=[list(c) for c in cfg.conv_layers],
                       hidden_sizes=list(cfg.hidden_sizes), num_actions=cfg.num_actions, num_envs=cfg.num_envs,
                       num_steps=cfg.num_steps, timed_updates=args.steps, ms_per_update=round(ms, 4),
                       env_steps_per_s=round(n / (ms / 1e3), 1), launches_per_update=launches, gpu=gpu, power_limit=power)
            scalars = e.fetch_scalars()
            del e
            if size == "nature":   # AtariModel's learner on the same model, batch and schedule
                a = eng.Engine(eng.EngineConfig(conv3_filters=cfg.conv_layers[2][0], **opt, **{
                    k: shape[k] for k in ("num_envs", "num_steps", "num_actions")}))
                a.set_params(params)
                a.load_batch(**b)
                ams, alaunches = time_engine(a, cfg, args.steps, args.warmup)
                rec.update(atari_engine_ms_per_update=round(ams, 4), atari_engine_launches_per_update=alaunches,
                           cnn_over_atari_engine=round(ms / ams, 3))
                del a
            rec.update(cpu_baseline_ms_per_update=round(cpu_baseline_ms(cfg, params, args.cpu_updates), 3),
                       cpu_threads=os.cpu_count(), scalars=scalars)
            print(json.dumps(rec), flush=True)
            lines.append(rec)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
