#!/usr/bin/env python
"""bench.py - the ACKTR learner update of jrobine/actor-critic on B200 (one process per GPU).

A step = one learner update = the reference's `session.run([..., optimize_op], feed_dict)`
(actorcritic/examples/atari/a2c_acktr.py:117-126) in its steady state: forward of the 32x20 train rows and
the 32 bootstrap rows, returns/advantages, A2C loss, backward, Fisher-sample backward, the 11 K-FAC factor
statistics, their EMA, the inverse refresh every 10th update, preconditioning, KL clip, momentum, apply.
Weak scaling: 32 environments x 20 steps PER GPU (8 GPUs = BASELINE.json's 256 x 20 configuration), one NCCL
all-reduce of [gradients | factor statistics | loss scalars] per update.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Prints ONE JSON line (rank 0).  `value` = env-steps/s (updates/s x envs x steps, whole job) with the inputs
resident in HBM; `e2e` = the same with the five train-step inputs coming from pinned host memory every step and
the loss scalars read back; `roofline` = the factor-statistics GEMM stage timed live with CUDA events;
`cpu_baseline` = the CPU restatement of the reference's update (oracle/, fp32 torch-CPU, all host threads)
timed on this box.  `--impl reference` times that CPU restatement alone (TensorFlow-1.x + tensorflow/kfac, the
reference's real dependencies, are not installable offline - see DESIGN.md).

`--dump-outputs DIR` writes, after the timed steps of `value`, what the last of them computed as DIR/<name>.npy
(float32): the updated parameters (one file per variable, e.g. conv1_weights), the forward's logits and values of
that step's rows, and its scalars (policy_loss, ..., learning_rate).  Inputs, initial parameters and Fisher samples
are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))



def ncu_traffic(raw_file):
    """dram__bytes_read.sum + dram__bytes_write.sum (bytes, one launch) parsed from a committed `ncu --page raw` text dump
    under profiles/ (None if the file or the metrics are missing)."""
    path = os.path.join(ROOT, "profiles", raw_file)
    if not os.path.exists(path):
        return None
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    total, seen = 0.0, 0
    for line in open(path):
        f = line.split()
        if len(f) >= 3 and f[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum") and f[1] in unit:
            total += float(f[2].replace(",", "")) * unit[f[1]]
            seen += 1
    return int(total) if seen == 2 else None

METRIC = "acktr_learner_env_steps_per_sec"
UNIT = "env-steps/s"
FRAMESKIP = 4   # a2c_acktr.py:195 - emulator frames per env-step


def positive_int(text):
    value = int(text)
    if value < 1:
        raise argparse.ArgumentTypeError("must be at least 1, got %d" % value)
    return value


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=50, help="timed updates of each timed leg")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=32)
    ap.add_argument("--num-steps", type=int, default=20)
    ap.add_argument("--conv3", type=int, default=32)
    ap.add_argument("--precision", type=int, default=0)
    ap.add_argument("--no-graphs", action="store_true")
    ap.add_argument("--conv-impl", type=int, default=0, help="0 = gather-form conv dgrad (default), 1 = dgrad GEMM + col2im")
    ap.add_argument("--lanes", type=int, default=0, help="concurrent lanes inside an update (0 = library default 5, 1 = serial)")
    ap.add_argument("--invert-every", type=int, default=10, help="diagnostic only: the reference uses 10 (a2c_acktr.py:245)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the conv3 = 64 and A2C 16 x 5 extra keys")
    ap.add_argument("--cpu-budget-s", type=float, default=15.0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed update computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs applies to --impl native")
    return args


DUMP_LIMIT_BYTES = 63 * 10 ** 6    # array data: with the .npy headers a dump stays within 64 MB


def dump_outputs(out_dir, arrays):
    """Write each array as out_dir/<name>.npy in float32.  Should the arrays exceed DUMP_LIMIT_BYTES together, each is
    replaced by a sample of its flattened elements, the same share of every array, at positions drawn from a fixed
    seed, so that two runs with the same arguments sample the same elements."""
    arrays = {k: np.asarray(v, np.float32) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if total > DUMP_LIMIT_BYTES:
            keep = max(1, a.size * DUMP_LIMIT_BYTES // total)
            a = a.ravel()[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=p["hbm_gbs"], tensor_burst=p["bf16_tflops"], tensor_sustained=p["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tensor_burst=1590.0, tensor_sustained=1400.0, source="fallback (B200_PROFILING.md)")


def workload_name(args, world):
    return "ACKTR Nature-CNN, %d envs x %d steps per GPU (%d x %d total), conv3=%d, 4 actions, factor EMA every update, " \
           "inverse refresh every 10 updates" % (args.envs_per_gpu, args.num_steps, args.envs_per_gpu * world,
                                                 args.num_steps, args.conv3)


def make_config(args, world):
    """The `config` object of the JSON line - identical for the native and the reference arm."""
    return {"workload": workload_name(args, world), "envs_per_gpu": args.envs_per_gpu, "num_steps": args.num_steps,
            "total_envs": args.envs_per_gpu * world, "conv3": args.conv3, "num_actions": 4,
            "schedule": "steady state after the cold phase: covariance EMA every update, inverse refresh every %d" % args.invert_every,
            "inputs": "synthetic uint8 observations (iid uniform), 8 batches rotated (152 MB per GPU > 126 MB L2)",
            "parallelism": "dp%d: environments sharded over the GPUs, one all-reduce of gradients + factor statistics per update" % world}


def update_gflop(c3):
    """Algorithmic GFLOP of one 32 x 20 learner update, symmetric-half counting (SURVEY 8(d))."""
    return {32: 78.2, 64: 100.2}.get(c3)


def algorithmic_flops(n_rows, e_rows, c3, num_actions=4):
    """Per-update algorithmic FLOPs (MAC = 2) of each stage, SURVEY 8(d)."""
    mac = 3276800 + 2654208 + 903168 * c3 // 32 + 49 * c3 * 512 + 512 * (num_actions + 1)
    dgrad_mac = 2654208 + 903168 * c3 // 32 + 49 * c3 * 512 + 512 * (num_actions + 1)      # no conv1 input gradient
    dims = [(n_rows * 400, 257), (n_rows * 81, 513), (n_rows * 49, 577), (n_rows, 49 * c3 + 1), (n_rows, 513)]
    a_half = sum(r * d * (d + 1) for r, d in dims)
    gdims = [(n_rows * 400, 32), (n_rows * 81, 64), (n_rows * 49, c3), (n_rows, 512), (n_rows, num_actions), (n_rows, 1)]
    g_half = sum(r * d * (d + 1) for r, d in gdims)
    layers = [(257, 32), (513, 64), (577, c3), (49 * c3 + 1, 512), (513, num_actions), (513, 1)]
    precon = sum(2 * d * d * c + 2 * d * c * c for d, c in layers)
    inverse = sum(2 * d ** 3 + 2 * c ** 3 for d, c in layers)     # Gauss-Jordan: 2 n^3
    return dict(forward=2.0 * mac * (n_rows + e_rows), backward=2.0 * mac * n_rows + 2.0 * dgrad_mac * 2 * n_rows,
                factors=float(a_half + g_half), precondition=float(precon), inverse=float(inverse))


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        return dict(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), power_w_max=float(max(power)),
                    samples=len(sm), reasons=sorted(reasons))


def make_batches(count, envs, steps, seed):
    import synth
    return [synth.rollout(seed + i, envs, steps, 4, terminal_prob=0.05, obs_kind="uniform") for i in range(count)]


def cpu_reference_rate(args, budget_s, warmup=1, steps=None, envs=None, c3=None, acktr=True, t_count=None):
    """The CPU restatement of the reference's update (oracle/learner.py, fp32, reference_cost=True: materialised
    patch matrices, [E,T,T] discount matrices, two towers, separate Fisher backward, dense inverses) on a bounded
    sample: whole updates in the steady state (ACKTR: covariances every update, inverses every 10th; A2C: RMSProp)."""
    import torch
    import synth
    from oracle import kfac as K
    from oracle import learner as OL
    from oracle import network as onet
    torch.set_num_threads(os.cpu_count() or 1)
    envs = args.envs_per_gpu if envs is None else envs
    t_count = args.num_steps if t_count is None else t_count
    c3 = args.conv3 if c3 is None else c3
    params = onet.init_params(4, c3, 0)
    cfg = K.KfacConfig(decay_steps=1e7 / (envs * t_count)) if acktr else OL.A2CConfig(decay_steps=1e7 / (envs * t_count))
    o = OL.OracleLearner(params, 4, c3, acktr=acktr, cfg=cfg, dtype=torch.float32, reference_cost=True)
    batch = synth.rollout(1, envs, t_count, 4)
    n = envs * t_count
    y_hat, eps = synth.fisher_samples(2, n)
    if acktr:
        # reach the first inverse refresh outside the timed sample (9 cheap "updates" would be the honest way, but each
        # costs ~1 s; instead run the covariance + inverse update once directly)
        o.global_step = 30
        info = o.compute(batch, y_hat, eps, need_fisher=True)
        o.kfac.update_covs(info["new_a"], info["new_g"])
        o.kfac.update_inverses()
        o.global_step = 40
    for _ in range(warmup):
        o.update(batch, y_hat, eps)
    times = []
    t_begin = time.perf_counter()
    while True:
        t0 = time.perf_counter()
        o.update(batch, y_hat, eps)
        times.append(time.perf_counter() - t0)
        if steps is not None and len(times) >= steps:
            break
        if steps is None and (time.perf_counter() - t_begin > budget_s or len(times) >= 50):
            break
    sec = float(np.mean(times))
    return dict(sec_per_update=sec, updates=len(times), env_steps_per_sec=n / sec, cores=torch.get_num_threads(),
                gs_end=o.global_step)


def run_reference(args, rank, world):
    """`--impl reference`: the reference's own CPU implementation of the path (its TensorFlow-1.x + tensorflow/kfac
    dependencies are not installable offline, so: the oracle's reference-cost restatement, fp32 torch-CPU) on all host
    threads of rank 0, on the native arm's workload: envs_per_gpu x n_gpus environments x num_steps, the same number of
    warm-up and timed updates."""
    if rank != 0:
        return
    warmup = max(3, args.warmup)
    total_envs = args.envs_per_gpu * args.gpus
    r = cpu_reference_rate(args, budget_s=1e9, warmup=warmup, steps=max(1, args.steps), envs=total_envs)
    n = total_envs * args.num_steps
    line = {
        "impl": "reference", "metric": METRIC, "value": r["env_steps_per_sec"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": warmup, "ms_per_step": r["sec_per_update"] * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "updates_per_sec": 1.0 / r["sec_per_update"], "env_frames_per_sec": r["env_steps_per_sec"] * FRAMESKIP,
        "config": make_config(args, args.gpus),
        "note": "CPU restatement of the reference's TF+kfac update (oracle/learner.py, fp32 torch-CPU, reference_cost=True); the "
                "reference itself needs TensorFlow 1.x + tensorflow/kfac, not installable offline (DESIGN.md section 2)",
        "cpu_baseline": {"value": r["env_steps_per_sec"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                         "sample": "%d whole %dx%d ACKTR updates (%d rows each), steady state incl. inverse refresh every 10"
                                   % (r["updates"], total_envs, args.num_steps, n)},
        "e2e": {"value": r["env_steps_per_sec"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def run_native(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from actorcritic_b200 import engine as eng
    from actorcritic_b200 import _lib

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = None
    if world > 1:
        # keep this rank's host threads - and with them the pinned staging buffers they first touch - on the CPUs next to its
        # GPU: eight ranks copying 19 MB per step from one NUMA node cost the end-to-end loop 0.15 ms per step in round 1
        try:
            import pynvml
            pynvml.nvmlInit()
            pr = torch.cuda.get_device_properties(local_rank)
            try:    # CUDA_VISIBLE_DEVICES may renumber the devices: find the NVML handle by PCI address
                hnd = pynvml.nvmlDeviceGetHandleByPciBusId(b"%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id))
            except Exception:  # noqa: BLE001
                hnd = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
            pynvml.nvmlDeviceSetCpuAffinity(hnd)
            numa = "rank pinned to the CPUs of GPU %d (nvmlDeviceSetCpuAffinity: %d CPUs)" % (local_rank, len(os.sched_getaffinity(0)))
        except Exception as exc:  # noqa: BLE001
            numa = "not pinned (%r)" % (exc,)
        dist.init_process_group("nccl", device_id=dev)
    peaks = load_peaks()
    envs, t_count, c3 = args.envs_per_gpu, args.num_steps, args.conv3
    n = envs * t_count
    cfg = eng.EngineConfig(num_envs=envs, num_steps=t_count, conv3_filters=c3, precision=args.precision,
                           world_size=world, seed=1234 + rank, use_graphs=not args.no_graphs,
                           invert_every=args.invert_every, num_lanes=args.lanes, conv_impl=args.conv_impl)
    e = eng.Engine(cfg, dev)
    e.set_params(eng.orthogonal_init(4, c3, seed=0))
    # synthetic inputs: 8 resident batches (8 x 19 MB > L2) + the same in pinned host memory for the e2e leg
    batches = make_batches(8, envs, t_count, seed=1000 * (rank + 1))
    keys = ("observations", "bootstrap_observations", "actions", "rewards", "terminals")
    host = [{k: torch.from_numpy(np.ascontiguousarray(b[k] if b[k].dtype != bool else b[k].astype(np.uint8))).pin_memory()
             for k in keys} for b in batches]
    resident = [{k: v.to(dev) for k, v in hb.items()} for hb in host]
    h2d_bytes = sum(v.numel() * v.element_size() for v in host[0].values())
    torch.cuda.synchronize()

    def step(i, src, fetch):
        if src is host:
            # public-API path: the batch after this one is already being copied on the copy stream (stage_batch), this
            # one is consumed from its staging slot; every step copies its own 18.97 MB from pinned host memory and
            # reads its own loss scalars back (fetch="async": the read of step i is waited for after step i+1 has been
            # enqueued, so the host never idles the GPU; every handle is resolved inside the timed region)
            e.stage_batch(host[(i + 1) % len(host)])
            return e.update(staged=True, fetch="async" if fetch else False)
        # device-resident inputs: the same public call (on one GPU both phases replay as one CUDA graph; data parallel:
        # phase 1, the exchange, phase 2)
        return e.update(src[i % len(src)], fetch=bool(fetch))

    # prime: post-cold state, then enough updates to pass TWO inverse refreshes (not part of warm-up or timing): the
    # library captures the CUDA graph of a schedule variant on its second use, so after 23 updates (refreshes at
    # global_step 40 and 50) both the plain and the refreshing update replay as graphs from the first timed step on,
    # whatever --warmup is
    e.set_state(30, 0, False)
    for i in range(23):
        step(i, resident, False)
    torch.cuda.synchronize()
    assert e.get_state()["inverses_valid"]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(src, fetch, steps, warmup, window=False):
        # window: cudaProfilerStart / Stop around the timed region (ACX_BENCH_NCU=1 with `ncu --profile-from-start off`: the
        # launch list of exactly the steps `value` is measured on; a number printed by such a run is never a bench value)
        # everything is launched on the engine's stream (events are recorded on that stream too)
        with torch.cuda.stream(e.stream):
            for i in range(warmup):
                step(i, src, fetch)
            barrier()
            if window:
                torch.cuda.profiler.start()
            launches0 = _lib.launch_count()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            last = None
            pending = None
            for i in range(steps):
                out = step(i, src, fetch)
                if isinstance(out, eng.PendingScalars):
                    if pending is not None:
                        last = pending.result()
                    pending = out
                else:
                    last = out
            if pending is not None:
                last = pending.result()
            ev1.record()
            barrier()
            if window:
                torch.cuda.profiler.stop()
        ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), _lib.launch_count() - launches0, last

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_dev, launches, _ = timed(resident, False, args.steps, max(3, args.warmup), window=bool(os.environ.get("ACX_BENCH_NCU")))
    if args.dump_outputs and rank == 0:
        # every rank holds the same parameters after an update; logits and values are those of rank 0's environments
        outputs = {name.replace("/", "_"): v for name, v in e.get_params().items()}
        outputs.update(logits=e.logits.cpu().numpy(), values=e.values.cpu().numpy(), **e.fetch_scalars())
        dump_outputs(args.dump_outputs, outputs)
    e.stage_batch(host[0])        # prologue of the double-buffered feed (the copy of step 0's batch)
    ms_e2e, _, scal = timed(host, True, args.steps, 3)
    clocks = sampler.stop() if rank == 0 else None

    # stage timing (CUDA events inside the engine, one host sync per step)
    e.set_profiling(True)
    stage_sum = {}
    prof_steps = min(args.steps, 20)
    for i in range(prof_steps):
        step(i, resident, False)
        torch.cuda.synchronize()
        for k, v in e.stage_ms().items():
            stage_sum.setdefault(k, []).append(v)
    e.set_profiling(False)
    stage_ms = {k: float(np.mean(v)) for k, v in stage_sum.items()}
    stage_ms["inverse_per_refresh"] = float(np.sum(stage_sum["inverse"]) / max(1, sum(1 for x in stage_sum["inverse"] if x > 0.01)))
    flops = algorithmic_flops(n, envs, c3)

    # conv1 input factor A1 = P1^T P1 (gemm_tc_kernel<1>, SYRK panel mode, 256 x 256 output, K = N*400 patch rows), timed alone
    # and live as the update runs it: the patch operand is read in place (acx_gather_t) from the engine's row-pair bf16 copy
    # of the last update's observations (36 MB: L2 resident), results stored back in (kh, kw, c) order.  Events are recorded by
    # the library around the kernel itself on the launching stream.
    from actorcritic_b200 import ops
    lib = _lib.load()
    k_rows = n * 400
    pairs_copy = e.buffer("obs_pairs", torch.bfloat16)
    ga1 = ops.nature_cnn_gather([pairs_copy], "conv1", n)
    lib.acx_gemm_enable_timing(1)
    durs = []
    with torch.cuda.stream(e.stream):
        for i in range(13):
            ops.gemm([pairs_copy], [pairs_copy], 256, 256, k_rows, trans=True, symmetric=True, pairs=[(0, 0)],
                     alpha=1.0 / (255.0 * 255.0 * k_rows), a_gather=ga1, perm_m=1, perm_n=1)
            ms = ctypes.c_float(0)
            _lib.check(lib.acx_gemm_last_ms(ctypes.byref(ms)))
            if i >= 3:
                durs.append(ms.value)
    lib.acx_gemm_enable_timing(0)
    syrk_ms = float(np.mean(durs))
    syrk_flops = float(k_rows) * 256 * 257          # rows * d * (d + 1), symmetric half (SURVEY 8(d))
    syrk_tflops = syrk_flops / (syrk_ms * 1e-3) / 1e12
    # the largest HBM-bound launch of the update: the row-pair copy itself (obs_pairs_bf16_kernel: uint8 observations read
    # once, bf16 copy written once = 3 bytes per observation byte), timed with CUDA events over the 8 resident batches
    # (152 MB > L2, so every launch reads its observations from HBM)
    obs_all = [torch.cat([b["observations"].reshape(-1, 84, 84, 4), b["bootstrap_observations"].reshape(-1, 84, 84, 4)]) for b in resident]
    pc_out = torch.empty((obs_all[0].shape[0], 42, 84, 2, 4), dtype=torch.bfloat16, device=dev)
    with torch.cuda.stream(e.stream):
        sp = ctypes.c_void_p(e.stream.cuda_stream)
        for ob in obs_all[:3]:
            _lib.check(lib.acx_obs_pairs_bf16(ob.data_ptr(), pc_out.data_ptr(), ob.shape[0], sp))
        p0, p1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record(e.stream)
        for ob in obs_all:
            _lib.check(lib.acx_obs_pairs_bf16(ob.data_ptr(), pc_out.data_ptr(), ob.shape[0], sp))
        p1e.record(e.stream)
    torch.cuda.synchronize()
    pairs_ms = p0.elapsed_time(p1e) / len(obs_all)
    pairs_bytes = 3 * obs_all[0].numel()
    del obs_all, pc_out

    # dominant launch of the update since the gather-form input gradient replaced dgrad GEMM + col2im: conv_tc_kernel on
    # conv3 / conv2 (true + Fisher rows = 2N samples), each timed alone with CUDA events on the launching stream on
    # operands of the update's own shapes; the longer of the two is reported as `roofline`
    # plane pairs / gradient planes of the backward pass per precision preset (learner.cu init_dims): the default keeps
    # activations and gradients on 2 bf16 planes and accumulates 3 plane pairs; preset 5 is the former 3-plane / 6-pair one
    npairs = {0: 3, 4: 3, 1: 3, 2: 3, 3: 1, 5: 6}.get(args.precision, 3)
    gplanes = {0: 2, 4: 2, 1: 2, 2: 2, 3: 1, 5: 3}.get(args.precision, 2)
    s2 = 2 * n

    def time_conv_dgrad(geom, mask_samples):
        hw_in, c_in, k, stride, hw_out, c_out = geom
        gen = torch.Generator(device=dev).manual_seed(7)
        gpl = [pl.reshape(s2, hw_out, hw_out, c_out)
               for pl in ops.split_planes(torch.randn((s2 * hw_out * hw_out, c_out), device=dev, generator=gen) * 1e-3, gplanes)]
        wd = ops.conv_dgrad_weights(torch.randn((k * k * c_in, c_out), device=dev, generator=gen) * 0.05, geom)
        act_mask = torch.rand((mask_samples, hw_in, hw_in, c_in), device=dev, generator=gen).to(torch.bfloat16)
        kw = dict(dgrad=True, mask=act_mask, mask_samples=mask_samples, pairs=ops.PAIRS[npairs])
        out = ops.conv(gpl, wd, geom, s2, out_planes=gplanes, **kw)
        durs = []
        with torch.cuda.stream(e.stream):
            for i in range(4):   # first round = warm-up; 10 back-to-back launches per measurement (no host gap inside)
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ev0.record()
                for _ in range(10):
                    ops.conv(gpl, wd, geom, s2, outs=out, **kw)
                ev1.record()
                ev1.synchronize()
                if i >= 1:
                    durs.append(ev0.elapsed_time(ev1) / 10.0)
        m = k // stride
        hq = hw_in // stride
        return dict(ms=float(np.mean(durs)),
                    flops=2.0 * s2 * hw_out * hw_out * (k * k * c_in) * c_out,            # useful MACs x 2 (SURVEY 8(d))
                    issued=2.0 * npairs * s2 * 128 * (stride * stride * c_in) * (m * m * c_out),   # 128-row tiles x plane pairs
                    rows_used=hq * hq)

    dg = {"conv2": time_conv_dgrad((20, 32, 4, 2, 9, 64), n), "conv3": time_conv_dgrad((9, 64, 3, 1, 7, c3), n)} \
        if c3 in (32, 64) and args.conv_impl == 0 else {}
    dom = max(dg, key=lambda kk: dg[kk]["ms"]) if dg else None

    # K-PRE (BASELINE.json config 5): raw 210x160x3 frame pairs -> gray -> 84x84 -> frame-stack push, HBM bound
    pre = {}
    if rank == 0:
        for pe in (64, 128, 256, 512, 1024, 2048, 4096):
            ra = torch.randint(0, 256, (pe, 210, 160, 3), dtype=torch.uint8, device=dev)
            rb = torch.randint(0, 256, (pe, 210, 160, 3), dtype=torch.uint8, device=dev)
            stk = torch.randint(0, 256, (pe, 84, 84, 4), dtype=torch.uint8, device=dev)
            out = torch.empty_like(stk)
            for _ in range(3):
                ops.preprocess_stack(ra, rb, stk, out=out, out_env_stride=28224)
            torch.cuda.synchronize()
            reps = 20 if pe <= 1024 else 10
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for _ in range(reps):
                ops.preprocess_stack(ra, rb, stk, out=out, out_env_stride=28224)
            ev1.record()
            torch.cuda.synchronize()
            ms = ev0.elapsed_time(ev1) / reps
            gbs = pe * 258048 / (ms * 1e-3) / 1e9
            pre["envs_%d" % pe] = {"ms": ms, "env_steps_per_sec": pe / (ms * 1e-3), "GB/s": gbs, "frac_hbm": gbs / peaks["hbm"]}
            del ra, rb, stk, out
        pre["note"] = ("258048 algorithmic bytes per env-step (ncu: dram__bytes = algorithmic, profiles/r1_prof_kpre_raw.txt); frac_hbm is "
                       "against the measured read+write COPY bandwidth of MEASURED_PEAKS.json - K-PRE is 89 % reads, which is why it can "
                       "reach ~1.0 of that figure (ncu: 80 % of the DRAM peak); 64 envs (16.5 MB) fit L2 and are launch bound")

    # rollout side of the path (agents.py:202-216): T x (K-PRE on E raw frame pairs + forward on E rows + sample)
    from actorcritic_b200.envs.atari.device_env import DeviceAtariMultiEnv
    from actorcritic_b200.agents import MultiEnvAgent

    class _EngineModel:          # what MultiEnvAgent needs from a model whose engine already exists
        engine = e
    # pool_frames = T: every rollout reads the same synthetic frames, so the agent replays the whole rollout
    # (T x (K-PRE, acting forward, sample) + bookkeeping) as ONE CUDA graph after its second call
    env = DeviceAtariMultiEnv(envs, pool_frames=t_count, seed=rank, device=dev)
    agent = MultiEnvAgent(env, _EngineModel(), t_count)
    with torch.cuda.stream(e.stream):
        for _ in range(4):
            agent.interact(None)
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(10):
            agent.interact(None)
        ev1.record()
        torch.cuda.synchronize()
    rollout_ms = ev0.elapsed_time(ev1) / 10

    total_envs = envs * world
    ms_step = ms_dev / args.steps
    # the other long launch of the update: the conv2 input-factor SYRK A2 = P2^T P2 / rows (gemm_tc_kernel<1>, MN-major
    # operands, upper 128-tiles only, split-K, 3 plane pairs on 2 planes), timed like the conv1 SYRK on operands of the
    # update's shape.  Informational (`roofline.factor_syrk`): a failure here must not cost the bench line.
    factor_syrk = None
    try:
        rows2 = n * 81
        gen = torch.Generator(device=dev).manual_seed(11)
        x2 = ops.split_planes(torch.rand((n * 400, 32), device=dev, generator=gen), 2)    # act1-shaped planes [N, 20, 20, 32]
        ga2 = ops.nature_cnn_gather(x2, "conv2", n)
        torch.cuda.synchronize()
        lib.acx_gemm_enable_timing(1)
        d2 = []
        with torch.cuda.stream(e.stream):
            for i in range(9):
                ops.gemm(x2, x2, 512, 512, rows2, trans=True, symmetric=True, pairs=ops.PAIRS[3], alpha=1.0 / rows2, a_gather=ga2)
                ms = ctypes.c_float(0)
                _lib.check(lib.acx_gemm_last_ms(ctypes.byref(ms)))
                if i >= 3:
                    d2.append(ms.value)
        lib.acx_gemm_enable_timing(0)
        ms2 = float(np.mean(d2))
        alg = float(rows2) * 512 * 513                       # rows * d * (d + 1): the symmetric half (SURVEY 8(d))
        issued = 3.0 * 10 * 2.0 * rows2 * 128 * 128           # 3 plane pairs x 10 upper 128-tiles of the 4 x 4 tile grid
        factor_syrk = {"kernel": "gemm_tc_kernel<1>: conv2 input factor A2 = P2^T P2 (512 x 512, K = %d patch rows read in place from the "
                                 "act1 planes by 5-D TMA box loads - no patch matrix -, 3 plane pairs, upper tiles, split-K; the split-K "
                                 "finalize is a separate launch)" % rows2,
                       "bound": "tensor", "launch_ms": ms2, "algorithmic_gflop_per_launch": alg / 1e9,
                       "achieved": alg / (ms2 * 1e-3) / 1e12, "peak": peaks["tensor_burst"], "unit": "TFLOP/s",
                       "frac": alg / (ms2 * 1e-3) / 1e12 / peaks["tensor_burst"],
                       "issued_gflop_per_launch": issued / 1e9, "issued_frac": issued / (ms2 * 1e-3) / 1e12 / peaks["tensor_burst"],
                       # dram__bytes_read.sum + dram__bytes_write.sum of one launch (ncu --set full, profiles/r2_prof_syrk_conv2_gather_raw.txt;
                       # algorithmic: the two act1 planes read once = 2 x N x 20 x 20 x 32 x 2 B = 33 MB)
                       "traffic": ncu_traffic("r2_prof_syrk_conv2_gather_raw.txt"),
                       "algorithmic_bytes_per_launch": 2 * n * 400 * 32 * 2,
                       "ncu": "profiles/r2_prof_syrk_conv2_gather_details.txt (this kernel); the same product on a materialised patch "
                              "matrix: profiles/r2_prof_syrk_conv2_details.txt (tensor pipe active 57.6 % of cycles, shared-memory "
                              "operand wavefronts 45.6 % of peak, DRAM 27 %)"}
        del x2
    except Exception as exc:  # noqa: BLE001
        factor_syrk = {"error": repr(exc)}
        try:
            lib.acx_gemm_enable_timing(0)
        except Exception:  # noqa: BLE001
            pass

    value = total_envs * t_count / (ms_step * 1e-3)
    e2e_value = total_envs * t_count / (ms_e2e / args.steps * 1e-3)
    # `roofline` = the dominant (longest) launch of the update; `hbm_kernel` inside it = the largest HBM-bound launch
    hbm_kernel = {
        "bound": "hbm",
        "kernel": "obs_pairs_bf16_kernel: uint8 observations [%d, 84, 84, 4] -> row-pair interleaved bf16 copy (what replaced the "
                  "conv1 patch matrix) - the largest HBM-bound launch of the update" % (n + envs),
        "achieved": pairs_bytes / (pairs_ms * 1e-3) / 1e9, "peak": peaks["hbm"], "unit": "GB/s",
        "frac": pairs_bytes / (pairs_ms * 1e-3) / 1e9 / peaks["hbm"],
        "traffic": None, "algorithmic_bytes_per_launch": pairs_bytes, "launch_ms": pairs_ms,
        "conv1_factor_syrk": {"kernel": "gemm_tc_kernel<1> (SYRK panel mode): conv1 input factor A1 = P1^T P1, 256 x 256 output, K = %d patch "
                                        "rows read in place from the row-pair copy" % k_rows,
                              "launch_ms": syrk_ms, "algorithmic_gflop_per_launch": syrk_flops / 1e9, "achieved_tflops": syrk_tflops,
                              "frac_of_burst_bf16_peak": syrk_tflops / peaks["tensor_burst"],
                              "round1": "on the materialised patch matrix (131 MB from HBM): 39 us"}}
    # the whole update against the tensor roofline: algorithmic GFLOP (symmetric-half counting, SURVEY 8(d)) over the
    # device-timed step; inside a long loop the sustained peak is the relevant denominator
    per_gpu_gflop = update_gflop(c3) * n / 640.0 if update_gflop(c3) else None
    update_block = None
    if per_gpu_gflop:
        ach = per_gpu_gflop / ms_step          # GFLOP / ms = TFLOP/s, per GPU
        update_block = {"bound": "tensor", "algorithmic_gflop_per_update_per_gpu": per_gpu_gflop, "ms_per_step": ms_step,
                        "achieved": ach, "unit": "TFLOP/s", "peak": peaks["tensor_sustained"], "frac": ach / peaks["tensor_sustained"],
                        "frac_of_burst": ach / peaks["tensor_burst"],
                        "note": "every launch of the update (%d per update at this size: 22 tensor-core kernels, HBM- and latency-bound "
                                "helpers, the inverse refresh amortised over 10 updates) against the dense bf16 peak" % round(launches / max(1, args.steps))}
    if dom is None:   # im2col route / unsupported conv3 width: the largest launch is the HBM-bound conv1 factor SYRK
        roofline = dict(hbm_kernel, stage_ms=stage_ms, update=update_block)
    else:
        roofline = {"bound": "tensor",
                     "kernel": "conv_tc_kernel (conv.cu): %s input gradient in gather form, %d samples (true + Fisher rows), "
                               "%d bf16 plane pairs into one fp32 TMEM accumulator - with the conv2 input-factor SYRK (`factor_syrk`) the longest launch of the update" % (dom, s2, npairs),
                     "achieved": dg[dom]["flops"] / (dg[dom]["ms"] * 1e-3) / 1e12, "peak": peaks["tensor_burst"], "unit": "TFLOP/s",
                     "frac": dg[dom]["flops"] / (dg[dom]["ms"] * 1e-3) / 1e12 / peaks["tensor_burst"],
                     # dram__bytes_read.sum + dram__bytes_write.sum of one launch (profiles/r1_prof_conv_dgrad2_raw.txt)
                     "traffic": ncu_traffic({("conv2", 3): "r1_prof_conv_dgrad2_raw.txt",
                                             ("conv3", 6): "r1_prof_conv_dgrad3_6pairs_raw.txt"}.get((dom, npairs), "none")),
                     "algorithmic_gflop_per_launch": dg[dom]["flops"] / 1e9, "launch_ms": dg[dom]["ms"],
                     "issued_gflop_per_launch": dg[dom]["issued"] / 1e9,
                     "issued_tflops": dg[dom]["issued"] / (dg[dom]["ms"] * 1e-3) / 1e12,
                     "issued_frac": dg[dom]["issued"] / (dg[dom]["ms"] * 1e-3) / 1e12 / peaks["tensor_burst"],
                     "note": "fp32-grade products from bf16 tensor cores cost %d plane pairs (hi*hi + hi*lo + lo*hi), and a sample's %d "
                             "output cells fill %d of a tile's 128 rows: the tensor pipe executes %.1fx the algorithmic FLOPs the fraction is charged on"
                             % (npairs, dg[dom]["rows_used"], dg[dom]["rows_used"], dg[dom]["issued"] / dg[dom]["flops"]),
                     "conv_dgrad_launches": {kk: {"launch_ms": v["ms"], "algorithmic_gflop": v["flops"] / 1e9,
                                                  "issued_gflop": v["issued"] / 1e9} for kk, v in dg.items()},
                     "peak_source": peaks["source"] + ", dense bf16 (cuBLAS) burst",
                     "hbm_kernel": hbm_kernel,
                     "factor_syrk": factor_syrk,
                     "update": update_block,
                     "stage_ms": stage_ms,
                     "stage_note": "stage times are taken with the lanes serialised (profiling mode); factor statistics are "
                                   "issued from inside the forward / backward stages",
                     "stage_tflops": {k: flops[k] / (stage_ms[k] * 1e-3) / 1e12 for k in ("forward", "backward", "precondition")
                                      if stage_ms.get(k, 0) > 0}}
    # The dominant kernel = the longest launch of the dominant kernel family.  gemm_tc_kernel<1> (MN-major operands: the
    # factor SYRKs and the weight gradients) is 13 launches and 29 % of the summed kernel time of an update
    # (profiles/r2_launches_update.txt); its longest launch - the conv2 input-factor SYRK, 50 us - is also the longest launch
    # of the whole update (the conv2 input gradient on conv_tc_kernel, round 1's headline, is 46 us: `roofline.conv_dgrad`).
    if isinstance(roofline, dict) and dom is not None and isinstance(factor_syrk, dict) and "frac" in factor_syrk \
            and factor_syrk["launch_ms"] >= dg[dom]["ms"]:
        conv_block = {k: roofline[k] for k in ("bound", "kernel", "achieved", "peak", "unit", "frac", "traffic",
                                               "algorithmic_gflop_per_launch", "launch_ms", "issued_gflop_per_launch",
                                               "issued_tflops", "issued_frac", "note", "conv_dgrad_launches")}
        rest = {k: v for k, v in roofline.items() if k not in conv_block and k != "factor_syrk"}
        roofline = dict(factor_syrk)
        roofline["peak_source"] = peaks["source"] + ", dense bf16 (cuBLAS) burst"
        roofline["note"] = ("fp32-grade products from bf16 tensor cores cost 3 plane pairs (hi*hi + hi*lo + lo*hi) and the symmetric "
                            "product is computed on 10 of 16 128-tiles: the tensor pipe executes 3.75x the algorithmic FLOPs the "
                            "fraction is charged on (`issued_frac`)")
        roofline.update(rest)
        roofline["conv_dgrad"] = conv_block
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16x2 planes (3 plane pairs), fp32 accumulate" if args.precision == 0 else "bf16 planes, precision preset %d" % args.precision,
        "data": "synthetic",
        "updates_per_sec": 1e3 / ms_step,
        # emulator frames per second of the whole loop on the device: T x (K-PRE + acting forward + sample) + one update
        "env_frames_per_sec": total_envs * t_count * FRAMESKIP / ((ms_step + rollout_ms) * 1e-3),
        "env_frames_per_sec_learner_only": value * FRAMESKIP,
        "config": make_config(args, world),
        "engine": {"host_affinity": numa, "exchange": None if world == 1 else (
                       "one kernel over NVLink peer memory inside phase 2's graph (csrc/peer.cu) for [G | grads | scalars]; the input-factor "
                       "prefix by NCCL on a side stream under phase 2" if getattr(e, "_peer_state", False) else "NCCL all-reduce between the phases"),
                   "precision": args.precision, "cuda_graphs": not args.no_graphs, "lanes": args.lanes if args.lanes > 0 else 5,
                   "patches": "never stored: conv input factors / weight gradients read their patch operands in place (5-D TMA box loads from "
                              "the activations; conv1 from a row-pair interleaved bf16 copy of the observations)"
                              if os.environ.get("ACX_GATHER", "1") != "0" else "materialised P1 / P2 / P3 (ACX_GATHER=0)",
                   "conv": "conv2/conv3 input gradient in gather form on the tensor cores (no patch-gradient matrix, no col2im)" if args.conv_impl == 0 else "dgrad GEMM + col2im",
                   "inverse": "fp32 blocked Gauss-Jordan, all factor tiles resident in shared memory, one persistent kernel (kfac_inv.cu)",
                   "l2": "8 resident input batches rotated (152 MB > 126 MB L2); per-step intermediates ~0.4 GB"},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 64,
                "ms_per_step": ms_e2e / args.steps,
                "note": "Engine.stage_batch + Engine.update(staged=True, fetch='async'): pinned host -> staging slot on a copy stream "
                        "(double buffered); the loss scalars of every step are read back (64 B, own event), the host waits for "
                        "step i's numbers after enqueuing step i+1; all reads complete inside the timed region"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline,
        "preprocess": pre,
        "rollout": {"ms_per_%d_steps" % t_count: rollout_ms, "env_steps_per_sec": envs * t_count / (rollout_ms * 1e-3),
                    "note": "per GPU, MultiEnvAgent.interact on the device-resident synthetic environment: T x (K-PRE on E raw frame "
                            "pairs -> stacks, Nature-CNN forward on E rows, categorical sample) + the [E,T] rollout tensors, replayed "
                            "as one CUDA graph; not part of `value`"},
        "env_steps_per_sec_with_rollout": total_envs * t_count / ((ms_step + rollout_ms) * 1e-3),
        "losses": scal,
    }
    if world > 1 and not args.no_extra:
        # (1) the collective on the critical path, timed alone: [G | grads | scalars] (what phase 2 waits for) and the
        # input-factor prefix A (reduced under phase 2 on a second communicator), each as K back-to-back all-reduces
        coll = {}
        try:
            a_part = e.buffer("input_factor_stats", torch.float32)
            rest = e.bucket[a_part.numel():]
            for name, buf in (("critical_G_grads_scalars", rest), ("input_factor_prefix_A", a_part)):
                with torch.cuda.stream(e.stream):
                    for _ in range(3):
                        dist.all_reduce(buf, op=dist.ReduceOp.SUM)
                    barrier()
                    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    c0.record()
                    for _ in range(20):
                        dist.all_reduce(buf, op=dist.ReduceOp.SUM)
                    c1.record()
                    barrier()
                t = torch.tensor([c0.elapsed_time(c1) / 20 * 1e3], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                coll[name] = {"bytes": buf.numel() * 4, "us": float(t.item())}
            # restore a sane state (the buckets now hold sums of sums): one more full update rewrites them
            step(0, resident, False)
        except Exception as exc:  # noqa: BLE001
            coll["error"] = repr(exc)
        line["collective"] = coll
        # (2) strong scaling of BASELINE.json configs[3]: 256 environments x 20 steps sharded over the ranks
        try:
            if 256 % world == 0:
                es = 256 // world
                cfg_s = eng.EngineConfig(num_envs=es, num_steps=t_count, conv3_filters=c3, precision=args.precision,
                                         world_size=world, seed=4321 + rank, use_graphs=not args.no_graphs,
                                         invert_every=args.invert_every, num_lanes=args.lanes, conv_impl=args.conv_impl)
                del resident, host
                torch.cuda.empty_cache()
                e2 = eng.Engine(cfg_s, dev)
                e2.set_params(eng.orthogonal_init(4, c3, seed=0))
                bs = make_batches(4, es, t_count, seed=5000 * (rank + 1))
                rs = [{k: torch.from_numpy(np.ascontiguousarray(b[k] if b[k].dtype != bool else b[k].astype(np.uint8))).to(dev)
                       for k in keys} for b in bs]
                e2.set_state(30, 0, False)

                def step2(i):
                    e2.update(rs[i % 4], fetch=False)

                with torch.cuda.stream(e2.stream):
                    for i in range(23 + 3):
                        step2(i)
                    barrier()
                    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    s0.record()
                    for i in range(args.steps):
                        step2(i)
                    s1.record()
                    barrier()
                t = torch.tensor([s0.elapsed_time(s1) / args.steps], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                line["strong_256x20"] = {"envs_per_rank": es, "total_envs": 256, "ms_per_step": float(t.item()),
                                         "value": 256 * t_count / (float(t.item()) * 1e-3), "unit": UNIT, "scaling": "strong",
                                         "steps": args.steps}
                del e2, rs
        except Exception as exc:  # noqa: BLE001
            line["strong_256x20"] = {"error": repr(exc)}
    if rank == 0 and world == 1 and not args.no_extra:
        # the other single-GPU configurations of BASELINE.json as extra keys (same timing rules, own CPU baseline):
        # configs[2] at the class-default conv3 = 64 (the 3137 x 3137 factor) and configs[1] = A2C 16 x 5
        del resident, host
        torch.cuda.empty_cache()

        def extra_line(cfg_x, label, cpu_kw):
            ex = eng.Engine(cfg_x, dev)
            ex.set_params(eng.orthogonal_init(4, cfg_x.conv3_filters, seed=0))
            bx = make_batches(8, cfg_x.num_envs, cfg_x.num_steps, seed=77)
            rx = [{k: torch.from_numpy(np.ascontiguousarray(b[k] if b[k].dtype != bool else b[k].astype(np.uint8))).to(dev)
                   for k in keys} for b in bx]
            if cfg_x.acktr:
                ex.set_state(30, 0, False)
            with torch.cuda.stream(ex.stream):
                for i in range(23 + 3):
                    ex.update(rx[i % 8], fetch=False)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for i in range(args.steps):
                    ex.update(rx[i % 8], fetch=False)
                e1.record()
                torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / args.steps
            rows = cfg_x.num_envs * cfg_x.num_steps
            out = {"workload": label, "ms_per_step": ms, "value": rows / (ms * 1e-3), "unit": UNIT, "steps": args.steps}
            g = update_gflop(cfg_x.conv3_filters) if cfg_x.acktr else None
            if g:
                out["roofline_update"] = {"algorithmic_gflop": g * rows / 640.0, "achieved_tflops": g * rows / 640.0 / ms,
                                          "frac": g * rows / 640.0 / ms / peaks["tensor_sustained"], "peak": peaks["tensor_sustained"]}
            if not args.no_cpu_baseline:
                rc = cpu_reference_rate(args, min(args.cpu_budget_s, 8.0), **cpu_kw)
                out["cpu_baseline"] = {"value": rc["env_steps_per_sec"], "unit": UNIT, "cores": rc["cores"], "kind": "port",
                                       "sample": "%d whole updates of the CPU restatement, %.3f s each" % (rc["updates"], rc["sec_per_update"])}
            del ex, rx
            torch.cuda.empty_cache()
            return out

        try:
            line["acktr_conv3_64"] = extra_line(
                eng.EngineConfig(num_envs=envs, num_steps=t_count, conv3_filters=64, seed=7),
                "ACKTR Nature-CNN %d envs x %d steps, conv3 = 64 (class default: 3137 x 3137 fc4 input factor)" % (envs, t_count),
                dict(c3=64))
            line["a2c_16x5"] = extra_line(
                eng.EngineConfig.a2c(16, 5, seed=7),
                "A2C Nature-CNN (no K-FAC) 16 envs x 5 steps, conv3 = 64, RMSProp + global-norm clip (BASELINE.json configs[1])",
                dict(envs=16, t_count=5, c3=64, acktr=False))
        except Exception as exc:  # noqa: BLE001  (informational keys must not cost the bench line)
            line["extra_error"] = repr(exc)
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            r = cpu_reference_rate(args, args.cpu_budget_s)
            line["cpu_baseline"] = {"value": r["env_steps_per_sec"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                                    "sample": "%d whole %dx%d ACKTR updates of the CPU restatement (oracle/learner.py, fp32), "
                                              "%.2f s each" % (r["updates"], envs, t_count, r["sec_per_update"])}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line):
    """The one JSON line goes to the real stdout; everything else this process (or NCCL, which announces its version
    on stdout) prints is diverted to stderr."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, data)
    else:
        sys.stdout.write(data.decode())
        sys.stdout.flush()


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        # launched without torchrun: re-launch ourselves under torch.distributed.run
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29511", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd, stdout=_REAL_STDOUT))
    run_native(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
