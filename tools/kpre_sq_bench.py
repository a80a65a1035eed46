"""Time K-PRE at any square size and stack depth (acx_preprocess_stack_sq_u8) on the GPU, and one CNNModel ACKTR
iteration on the device-resident frames it produces.  One JSON line per case.

Kernel lines: E in {256, 1024, 4096} x (S, k) in {(64, 2), (84, 4), (96, 4), (128, 1)}; at (84, 4) the specialised K-PRE
(acx_preprocess_stack_u8) runs alternately with the S x S kernel in the same process.  Each timed pass is one CUDA graph
of `--calls` in-place stack steps (no host launch cost in the window), timed with CUDA events; the line reports the median
over `--reps` passes.  Bytes per call = E x (2 raw frames of 100 800 B + old and new stack of S*S*k B each), from the
shapes; TB/s = bytes / time.  The same inputs are read on every call: at E = 256 the raw frames (52 MB) fit the 126 MB L2
and are served from there after the first call (`l2_resident` true); at E = 1024 (206 MB) and 4096 (826 MB) they do not.

Iteration line: MultiEnvAgent over DeviceAtariMultiEnv(size=64, num_stacked_frames=2), 64 environments x 5 steps (a pool
of 5 frames, so the rollout is replayed as one CUDA graph), with a
CNNModel (conv (32,8,4), (64,4,2), (64,3,1), fc 256, 15 actions) trained by ColdStartPeriodicInvUpdateKfacOpt through
Session.run: ms per rollout + update from a host clock around iterations that end in a device synchronise, after a
warm-up past the graph capture of the rollout and the first inverse refresh.

The GPU's name and power limit are read in the same run.

    python tools/kpre_sq_bench.py [--calls 50] [--reps 7] [--iters 100] [--out profiles/kpre_sq_1gpu.jsonl]
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

from actorcritic_b200 import ops  # noqa: E402
from mlp_bench import gpu_info  # noqa: E402

RAW_BYTES = 210 * 160 * 3
L2_BYTES = 126 * 2 ** 20
ENVS = (256, 1024, 4096)
SHAPES = ((64, 2), (84, 4), (96, 4), (128, 1))


def graph_of(fn, calls, stream):
    fn()                                     # tables, attributes and modules are set up outside the capture
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        for _ in range(calls):
            fn()
    return g


def time_graph(g, stream):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        start.record()
        g.replay()
        end.record()
    end.synchronize()
    return start.elapsed_time(end)


def kernel_lines(calls, reps, gpu, power):
    stream = torch.cuda.Stream()
    for e in ENVS:
        g = torch.Generator(device="cuda").manual_seed(e)
        a = torch.randint(0, 256, (e, 210, 160, 3), dtype=torch.uint8, device="cuda", generator=g)
        b = torch.randint(0, 256, (e, 210, 160, 3), dtype=torch.uint8, device="cuda", generator=g)
        for size, k in SHAPES:
            stack_sq = torch.zeros((e, size, size, k), dtype=torch.uint8, device="cuda")
            variants = {"sq": graph_of(lambda: ops.preprocess_stack_sq(a, b, stack_sq, out=stack_sq), calls, stream)}
            if (size, k) == (84, 4):
                stack_kpre = torch.zeros_like(stack_sq)
                variants["kpre"] = graph_of(lambda: ops.preprocess_stack(a, b, stack_kpre, out=stack_kpre), calls, stream)
            times = {name: [] for name in variants}
            for name, gr in variants.items():        # warm-up pass of each
                time_graph(gr, stream)
            for _ in range(reps):                     # alternate the variants within each repetition
                for name, gr in variants.items():
                    times[name].append(time_graph(gr, stream) / calls)
            if "kpre" in variants:
                assert torch.equal(stack_sq, stack_kpre), "the S x S kernel and K-PRE disagree at 84 x 84 x 4"
            nbytes = e * (2 * RAW_BYTES + 2 * size * size * k)
            for name, ts in times.items():
                ms = float(np.median(ts))
                line = dict(case="kernel", kernel={"sq": "preprocess_sq_kernel", "kpre": "K-PRE"}[name], num_envs=e, size=size,
                            num_stacked_frames=k, bytes_per_call=nbytes, ms_per_call=round(ms, 5),
                            tb_per_s=round(nbytes / (ms * 1e-3) / 1e12, 3), ms_min=round(min(ts), 5), ms_max=round(max(ts), 5),
                            raw_bytes=2 * e * RAW_BYTES, l2_resident=2 * e * RAW_BYTES < L2_BYTES, calls_per_pass=calls,
                            passes=reps, gpu=gpu, power_limit=power)
                print(json.dumps(line), flush=True)
                yield line
        del a, b
        torch.cuda.empty_cache()


def iteration_line(iters, warmup, gpu, power):
    import actorcritic_b200 as ac
    from actorcritic_b200 import agents, kfac, nn, objectives
    from actorcritic_b200.cnn import CNNModel
    from actorcritic_b200.envs.atari.device_env import DeviceAtariMultiEnv
    from actorcritic_b200.kfac_utils import ColdStartPeriodicInvUpdateKfacOpt
    e, t = 64, 5
    env = DeviceAtariMultiEnv(e, num_actions=15, pool_frames=t, terminal_prob=0.01, seed=0, size=64, num_stacked_frames=2)
    model = CNNModel(env.observation_space, env.action_space, conv_layers=((32, 8, 4), (64, 4, 2), (64, 3, 1)),
                     hidden_sizes=(256,), random_seed=0)
    objective = objectives.A2CObjective(model, discount_factor=0.99, entropy_regularization_strength=0.01)
    global_step = ac.GlobalStep()
    lc = kfac.LayerCollection()
    model.register_layers(lc)
    model.register_predictive_distributions(lc)
    cold = nn.ClipGlobalNormOptimizer(nn.MomentumOptimizer(learning_rate=0.0003, momentum=0.9), clip_norm=0.5)
    opt = ColdStartPeriodicInvUpdateKfacOpt(num_cold_updates=2, cold_optimizer=cold, invert_every=10,
                                            learning_rate=nn.linear_decay(0.25, 0.025, global_step, 1e6), cov_ema_decay=0.99,
                                            damping=0.01, layer_collection=lc, momentum=0.9, norm_constraint=0.0001)
    optimize_op = objective.optimize_shared(opt, baseline_loss_weight=0.5, global_step=global_step)
    agent = agents.MultiEnvAgent(env, model, num_steps=t)

    def one(session):
        obs, act, rew, term, nxt, _ = agent.interact(session)
        session.run(optimize_op, feed_dict={model.observations_placeholder: obs, model.bootstrap_observations_placeholder: nxt,
                                            model.actions_placeholder: act, model.rewards_placeholder: rew,
                                            model.terminals_placeholder: term})

    with ac.Session() as session:
        for _ in range(warmup):
            one(session)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(iters):
            one(session)
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3 / iters
        graph_replayed = getattr(agent, "_graph_state", 0) == 2
    line = dict(case="iteration", what="MultiEnvAgent rollout + CNNModel ACKTR update", env="DeviceAtariMultiEnv(size=64, "
                "num_stacked_frames=2)", num_envs=e, num_steps=t, conv_layers=[[32, 8, 4], [64, 4, 2], [64, 3, 1]],
                hidden_sizes=[256], num_actions=15, ms_per_iteration=round(ms, 4), env_steps_per_s=round(e * t / (ms * 1e-3), 1),
                iterations=iters, warmup=warmup, rollout_graph_replayed=graph_replayed, gpu=gpu, power_limit=power)
    print(json.dumps(line), flush=True)
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=30)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "kpre_sq_1gpu.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("kpre_sq_bench.py measures on a CUDA device; none is available")
    gpu, power = gpu_info()
    lines = list(kernel_lines(args.calls, args.reps, gpu, power))
    lines.append(iteration_line(args.iters, args.warmup, gpu, power))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for line in lines:
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
