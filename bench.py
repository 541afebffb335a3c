#!/usr/bin/env python
"""Benchmark of the evacuation hot path (BASELINE.json metric: pedestrian-steps/s and env-steps/s).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # the reference algorithm on the host CPUs

A "step" is one pass of the hot path over one batch: ONE `env.step(actions)` == one fused kernel
launch advancing every environment of the batch by one time step (agent step, Vicsek alignment,
noise, enslaving, integration, reflection, statuses, rewards, observation encoding, auto-reset).

Workload at N=1: BASELINE.json configs[1] (C2): 4096 envs x 60 pedestrians, rel positions + ohe
statuses Box observation [62,6], enslaving 1.0, noise 0.2, RandomAgent-like U[-1,1]^2 actions,
in-kernel Philox noise, same-step auto-reset.  N>1: the same per-rank batch on every rank
(environments are independent -> weak scaling, no data-path collective; NCCL only all-gathers the
episode statistics after the timed region).

Timing of `value` (timing rules: inputs larger than L2): `--sets` (24) independent C2 batches are
stepped round-robin, one batch per step, so every step finds its state in HBM, not in L2; the K
launches are one CUDA graph, timed with CUDA events around the replay, max over ranks.  Beside it:
`l2_flushed` (one batch, 256 MiB memset before every step, per-step events -- code cold too),
`l2_resident` (one batch stepped K times, graph replay), `rollout` (K steps in ONE launch).

Prints ONE JSON line (rank 0).  Keys follow the driver contract, plus `roofline`, `roofline_fp32`,
`cpu_baseline`, `e2e`, `clocks`, `gpu_launches`, `l2_flushed`, `l2_resident`, `rollout`.

`--dump-outputs DIR` (C2 only) also writes what the last timed step returned to its caller -- observation, reward,
terminated, truncated of the batch it stepped, rank 0 -- as DIR/<name>.npy (float32), so that two builds can be compared
output for output: actions and seeds depend only on the arguments.  Nothing is written into the source tree (it may be
read-only): log files go to a temporary directory and no bytecode is cached.
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_PED = 60
ENVS_PER_GPU = 4096
ENV_KW = dict(number_of_pedestrians=N_PED, enslaving_degree=1.0, noise_coef=0.2, is_new_exiting_reward=True,
              is_new_followers_reward=True)
WRAP_KW = dict(positions="rel", statuses="ohe", type="Box")
WORKLOAD = "C2: 4096 envs x 60 pedestrians per GPU, rel positions + ohe statuses (Box [62,6]), enslaving 1.0, noise 0.2"


def algorithmic_bytes_per_env_step(n: int, obs_bytes: int) -> int:
    """SURVEY.md 8(d): read+write of pos (8N) + dir (8N) + status (N) + agent/time (24), action in (8),
    reward (4) + flags (2), obs out.  N=60 rel+ohe: 3590 B."""
    return 2 * (17 * n + 24) + 14 + obs_bytes


def algorithmic_flops_per_env_step(n: int) -> int:
    """SURVEY.md 8(d): 8 flop per ordered pair over the full N x N + 120 per pedestrian. N=60: 36000."""
    return 8 * n * n + 120 * n


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)", p
    return 6650.0, "fallback (B200_PROFILING.md)", {}


# ---------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons with NVML during the timed region."""

    def __init__(self, index: int, period=0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as exc:  # pragma: no cover
            self.nv, self.err = None, repr(exc)

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------------
# CPU side: the reference's own per-env step loop (src/env/__init__.py:18-21 -> src/env/env/env.py:141-171) on the host
# cores.  kind = "reference": the UNMODIFIED reference, imported through oracle/ref_shim.py from $EVAC_REFERENCE_ROOT,
# /root/reference or baseline/_ref (the pip --target install made by oracle/install_reference.py, which travels to the GPU
# box); kind = "port": oracle/evac_oracle.py (bit-identical to the reference on tests/golden/) when no copy is reachable.
def cpu_kind():
    from oracle import ref_shim

    if os.environ.get("EVAC_BENCH_CPU_KIND") == "port":  # A/B and tests: force the port although the reference is reachable
        return "port"
    return "reference" if ref_shim.reference_available() else "port"


_LOG_DIR = None


def _log_dir():
    """One scratch log directory per process: the reference opens a log file per env (env.py:23-31), this package's
    single-env face one when an episode ends; neither belongs in the working directory."""
    global _LOG_DIR
    if _LOG_DIR is None:
        import atexit
        import shutil
        import tempfile

        _LOG_DIR = tempfile.mkdtemp(prefix="evac_bench_logs_")
        atexit.register(shutil.rmtree, _LOG_DIR, ignore_errors=True)
    return _LOG_DIR


def _make_cpu_env(kind, n_ped, env_kw=None, wrap_kw=None):
    kw = dict(ENV_KW) if env_kw is None else dict(env_kw)
    if n_ped is not None:
        kw["number_of_pedestrians"] = n_ped
    WRAP_KW_ = WRAP_KW if wrap_kw is None else wrap_kw
    if kind == "reference":
        import warnings

        from oracle import ref_shim

        warnings.filterwarnings("ignore")
        ref = ref_shim.load_reference()
        cfg = ref.EnvConfig(wandb_enabled=False, giff_freq=10 ** 9, path_logs=_log_dir(), **kw)
        return ref.setup_env(cfg, ref.EnvWrappersConfig(**WRAP_KW_))
    from oracle.evac_oracle import OracleConfig, OracleEnv

    class _Port:  # same call shape as the reference env
        def __init__(self):
            self.env = OracleEnv(OracleConfig(**kw, **WRAP_KW_))

        def reset(self):
            return self.env.reset(), {}

        def step(self, a):
            return self.env.step(a)

    return _Port()


def _cpu_worker(args, n_ped=None, kind="port"):
    n_envs, steps, warmup, seed, barrier = args
    np.random.seed(seed)
    envs = []
    for _ in range(n_envs):
        e = _make_cpu_env(kind, n_ped)
        e.reset()
        envs.append(e)
    rs = np.random.RandomState(seed + 1)

    def one_step():
        for e in envs:  # the reference's user loop (README.md:79-86): RandomAgent action, step, reset when the episode ends
            _, _, term, trunc, _ = e.step(rs.uniform(-1, 1, 2).astype(np.float32))
            if term or trunc:
                e.reset()

    for _ in range(warmup):
        one_step()
    if barrier is not None:
        barrier.wait()
    t0 = time.perf_counter()
    for _ in range(steps):
        one_step()
    dt = time.perf_counter() - t0
    global _LOG_DIR
    if _LOG_DIR is not None:  # (forked workers leave through os._exit: atexit handlers do not run there)
        import logging
        import shutil

        logging.shutdown()
        shutil.rmtree(_LOG_DIR, ignore_errors=True)
        _LOG_DIR = None
    return dt


def cpu_baseline_single_core(target_seconds=12.0):
    """The CPU step loop on ONE core: one env x 60 pedestrians (C1-like loop with the C2 wrappers), ~target_seconds;
    the reference itself when reachable (and the port beside it), else the port."""
    kind = cpu_kind()
    t = _cpu_worker((1, 200, 20, 0, None), kind=kind)
    steps = max(200, int(200 * target_seconds / max(t, 1e-3)))
    steps = min(steps, 200000)
    t = _cpu_worker((1, steps, 20, 0, None), kind=kind)
    env_sps = steps / t
    # SURVEY 8(d)(iii): the large-crowd config (C4) on one core, 1 env x 4096 pedestrians, a handful of steps (~1 step/s)
    t4 = _cpu_worker((1, 5, 1, 0, None), n_ped=4096, kind=kind)
    what = ("the UNMODIFIED reference (src/env through oracle/ref_shim.py)" if kind == "reference" else
            "oracle/evac_oracle.py (NumPy fp64 port, bit-identical to the reference on tests/golden; no copy of the reference reachable)")
    out = {"value": env_sps * N_PED, "unit": "pedestrian-steps/s", "env_steps_per_s": env_sps, "cores": 1, "kind": kind,
           "sample": f"{what}, 1 env x {N_PED} pedestrians, {steps} steps in {t:.1f} s on 1 core, rel+ohe Box observation, RandomAgent actions",
           "c4_1x4096": {"value": 5 * 4096 / t4, "unit": "pedestrian-steps/s", "env_steps_per_s": 5 / t4,
                         "sample": f"1 env x 4096 pedestrians, 5 steps in {t4:.1f} s on 1 core"}}
    if kind == "reference":  # the port on the same core, same loop (it is the checker of the parity tests)
        tp = _cpu_worker((1, 2000, 20, 0, None), kind="port")
        out["port_same_core"] = {"value": 2000 / tp * N_PED, "unit": "pedestrian-steps/s", "env_steps_per_s": 2000 / tp}
    return out


def c1_leg(dev, seeds=8, steps=2000):
    """BASELINE.md section 3 item 1 / BASELINE.json configs[0] (C1): `EnvConfig(number_of_pedestrians=60)`, one 2000-step episode
    per seed 0..7 (`np.random.seed(s)`, RandomAgent-like actions from `RandomState(1000 + s)`), 1 process / 1 core, with the
    default wrappers (abs / no / Dict), rel + ohe + Box and grav (alpha 3) -- the reference's own README loop
    (README.md:69-90), timed (a) on the CPU implementation (reference when reachable, else the port) and (b) through THIS
    repo's drop-in single-env API (`setup_env(EnvConfig(60), wrap)`: NumPy in / NumPy out, rng="numpy" = the global MT19937
    stream consumed like the reference, one fused kernel launch + one D2H copy per step).  Median over the seeds."""
    import evacuation_b200 as eb

    kind = cpu_kind()
    out = {"cpu_kind": kind, "cores": 1, "seeds": seeds, "steps_per_episode": steps, "cases": {}}
    for name, wrap in (("abs_no_dict", {}), ("rel_ohe_box", WRAP_KW), ("grav_alpha3_dict", dict(positions="grav", alpha=3))):
        rates = {"cpu": [], "gpu": []}
        for arm in ("cpu", "gpu"):
            for seed in range(seeds):
                if arm == "cpu":
                    env = _make_cpu_env(kind, None, env_kw=dict(number_of_pedestrians=N_PED), wrap_kw=wrap)
                else:
                    env = eb.setup_env(eb.EnvConfig(number_of_pedestrians=N_PED, wandb_enabled=False, path_logs=_log_dir()),
                                       eb.EnvWrappersConfig(**wrap), device=dev)
                np.random.seed(seed)
                rs = np.random.RandomState(1000 + seed)
                acts = rs.uniform(-1, 1, size=(steps, 2)).astype(np.float32)
                env.reset()
                if arm == "gpu" and seed == 0:
                    for t in range(20):  # module load / first-launch costs are not the step
                        env.step(acts[t])
                    np.random.seed(seed)
                    env.reset()
                done = 0
                t0 = time.perf_counter()
                for t in range(steps):
                    _, _, term, trunc, _ = env.step(acts[t])
                    done += 1
                    if term or trunc:
                        break
                rates[arm].append(done / (time.perf_counter() - t0))
                if arm == "gpu":
                    env.unwrapped.close()
        cpu, gpu = float(np.median(rates["cpu"])), float(np.median(rates["gpu"]))
        out["cases"][name] = {"cpu_env_steps_per_s": cpu, "gpu_single_env_steps_per_s": gpu, "cpu_us_per_step": 1e6 / cpu,
                              "gpu_single_env_us_per_step": 1e6 / gpu, "speedup_single_env": gpu / cpu}
    global _LOG_DIR
    if _LOG_DIR is not None:
        import shutil

        shutil.rmtree(_LOG_DIR, ignore_errors=True)
        _LOG_DIR = None
    return out


def run_reference_arm(args):
    """--impl reference: the reference's CPU implementation of the path on all host cores, same workload (C2), same metric.
    Every step advances a bounded sample of the 4096-env batch: all 4096 envs when K + W steps of them fit in about a
    minute, else as many as do (the metric is rate-normalised).  At least ~10 s are timed regardless of --steps: the K-step
    measurement is repeated back to back and the mean is reported."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    kind = cpu_kind()
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    t_cal = _cpu_worker((1, 60, 5, 99, None), kind=kind)
    rate = 60.0 / max(t_cal, 1e-6)  # env-steps/s of one core
    steps_all = max(args.steps + args.warmup, 1)
    envs_per_worker = int(max(1, min(-(-ENVS_PER_GPU // cores), rate * 60.0 / steps_all)))
    est = envs_per_worker * args.steps / rate
    min_seconds = float(os.environ.get("EVAC_BENCH_MIN_SECONDS", "10"))
    passes = int(max(1, min(50, np.ceil(min_seconds / max(est, 1e-3)))))
    ctx = mp.get_context("fork")
    barrier = ctx.Barrier(cores)
    queue = ctx.Queue()

    def work(w):
        queue.put(_cpu_worker((envs_per_worker, args.steps * passes, args.warmup, 100 + w, barrier), kind=kind))

    procs = [ctx.Process(target=work, args=(w,)) for w in range(cores)]
    for p in procs:
        p.start()
    times = [queue.get() for _ in procs]
    for p in procs:
        p.join()
    t = max(times) / passes  # mean duration of one K-step pass
    env_steps = cores * envs_per_worker * args.steps
    value = env_steps * N_PED / t
    what = ("UNMODIFIED reference (kind=reference: src/env imported through oracle/ref_shim.py)" if kind == "reference" else
            "oracle port (kind=port: no copy of the reference reachable on this box)")
    sample = (f"{what}, {cores} worker processes x {envs_per_worker} envs x {N_PED} pedestrians = {cores * envs_per_worker} of the "
              f"{ENVS_PER_GPU} envs per step, {passes} back-to-back passes of {args.steps} steps, mean pass time {t:.2f} s (max over workers)")
    line = {
        "impl": "reference", "metric": "pedestrian-steps/s", "value": value, "unit": "pedestrian-steps/s", "env_steps_per_s": env_steps / t,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": f"{cores * envs_per_worker} envs per step on the host CPUs", "passes": passes},
        "cpu_baseline": {"value": value, "unit": "pedestrian-steps/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "pedestrian-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def _nccl_output_to_stderr():
    """stdout must stay the ONE JSON line.  With NCCL_DEBUG=VERSION (set on the GPU boxes) NCCL prints its version
    banner on stdout and ignores NCCL_DEBUG_FILE (debug.cc: the file is only opened above VERSION), so raise the level
    to WARN and send NCCL's output to stderr.  An explicit INFO / TRACE request is kept."""
    if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")


# ---------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    import evacuation_b200 as eb

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        _nccl_output_to_stderr()
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    E, K, W = args.envs, args.steps, max(args.warmup, 3)

    from evacuation_b200.distributed import allgather_episode_totals, bind_host_to_device, shard_offset

    # one process per GPU: run on the cores of the GPU's own socket so that the page-locked buffers of the e2e leg are
    # local to it (EVAC_BENCH_NO_NUMA_BIND=1 switches this off for A/B runs)
    numa = {"bound": False} if os.environ.get("EVAC_BENCH_NO_NUMA_BIND") else bind_host_to_device(local_rank)

    env = eb.setup_env(eb.EnvConfig(**ENV_KW), eb.EnvWrappersConfig(**WRAP_KW), num_envs=E, device=dev, seed=args.seed,
                       auto_reset=True, env_index_offset=shard_offset(rank, E))
    u = env.unwrapped
    env.reset()
    obs_dim = u.obs_dim
    # RandomAgent-like actions resident in HBM before the timed region (one [E,2] table per step)
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    actions = torch.rand((W + K, E, 2), generator=g, device=dev) * 2 - 1

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for s in range(W):
        env.step(actions[s])
    # ---- timed region A (headline `value`): inputs larger than L2.  R independent C2 batches ("sets": own state, own
    # observation / reward / flag buffers, 14.7 MB of algorithmic traffic each) are stepped round-robin, one batch per
    # step, so that by the time a set is stepped again the R-1 other sets (R x 14.7 MB >= 2.5 x the 126 MB L2) have
    # evicted it: every step reads its state from HBM, while the kernel code stays hot as in any real run.  The K
    # launches are captured in ONE CUDA graph (no host in the loop) and the replay is bracketed by CUDA events.
    R = max(1, args.sets)
    sets = [env]
    for r in range(1, R):
        er = eb.setup_env(eb.EnvConfig(**ENV_KW), eb.EnvWrappersConfig(**WRAP_KW), num_envs=E, device=dev, seed=args.seed + 7919 * r,
                          auto_reset=True, env_index_offset=shard_offset(rank, E))
        er.reset()
        for s in range(W):
            er.step(actions[s])
        sets.append(er)
    # Episode phase: the work of a step falls as an episode ages (pedestrians turn EXITING / ESCAPED and leave the pairwise
    # pass: ~15 % fewer instructions by step 500), so every timed leg starts from the SAME state -- reset + W warm-up steps,
    # snapshotted here (evac_save_state) and restored before each timed replay -- which is also the phase the CPU arm times
    # (`--impl reference`: reset, W warm-up steps, K timed steps).  Warm-up replays therefore never age the measured batches.
    snaps = [x.unwrapped.save_state() for x in sets]

    def restore(which=None):
        for x, img in zip(sets, snaps):
            if which is None or x is which:
                x.unwrapped.load_state(img)

    # decoy batches: stepped (untimed) between the restore and the timed steps, they turn the L2 over with the traffic of the
    # very kernel (12 x 14.7 MB per round > 126 MB), so the timed steps find the restored state in HBM and the L2 in the state a
    # long run leaves it in -- a memset flush would leave 126 MB of dirty lines to write back under the first timed steps
    decoys = []
    for r in range(12):
        er = eb.setup_env(eb.EnvConfig(**ENV_KW), eb.EnvWrappersConfig(**WRAP_KW), num_envs=E, device=dev, seed=args.seed + 104729 * (r + 1),
                          auto_reset=True, env_index_offset=shard_offset(rank, E))
        er.reset()
        er.step(actions[0])
        decoys.append(er)
    n_warm = 240

    def decoy_steps():
        for s in range(n_warm):
            decoys[s % len(decoys)].unwrapped.step(actions[s % (W + K)])

    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2 (the `l2_flushed` leg)
    sampler = ClockSampler(local_rank)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    side = torch.cuda.Stream(device=dev)
    # Graph 1 (`ms_per_step_incl_graph_launch`): exactly the K step launches, CUDA events around the replay.  A replay pays the
    # launch latency of the graph itself once -- ~0.4 us per step at the driver's K = 20, nothing at K = 2000.
    graph_a = torch.cuda.CUDAGraph()
    torch.cuda.synchronize(dev)
    launches0 = sum(x.unwrapped.launch_count for x in sets)
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph_a, stream=side):
            for s in range(K):
                last = sets[s % R].unwrapped.step(actions[W + s])  # (the batch's own output buffers: every replay refills them)
    torch.cuda.synchronize(dev)
    # kernel nodes recorded into the graph (the library counts launches at capture time) = launches of the K timed steps
    launches = sum(x.unwrapped.launch_count for x in sets) - launches0
    # Graph 2 (headline `value`): ONE chain of nodes -- [restore every measured batch] [n_warm untimed steps on the decoy
    # batches] event [the K timed steps] event -- with two event-record nodes (external events) around the K timed kernels.
    # The timed steps then run with the device continuously busy (no graph-launch latency, no idle gap in front of the first
    # kernel, code hot) however small K is: a K = 20 replay lasts only 0.18 ms.
    g0, g1 = torch.cuda.Event(enable_timing=True, external=True), torch.cuda.Event(enable_timing=True, external=True)
    graph_b, ingraph_ok = torch.cuda.CUDAGraph(), True
    try:
        with torch.cuda.stream(side):
            with torch.cuda.graph(graph_b, stream=side):
                restore()
                decoy_steps()
                g0.record()
                for s in range(K):
                    sets[s % R].unwrapped.step(actions[W + s])
                g1.record()
    except Exception:  # pragma: no cover  (no external-event support: fall back to graph 1)
        ingraph_ok = False
    torch.cuda.synchronize(dev)
    graph_a.replay()  # untimed: graph upload
    barrier()
    sampler.start()
    restore()
    decoy_steps()  # plain launches queued in front of the timed replay: the host runs ahead, the device never idles
    e0.record()
    graph_a.replay()
    e1.record()
    if ingraph_ok:
        graph_b.replay()
    barrier()
    outer_ms = e0.elapsed_time(e1)
    kernel_ms = outer_ms
    timed_by = "CUDA events around the replay of a graph of the K step launches"
    if ingraph_ok:
        try:
            inner = g0.elapsed_time(g1)
            if 0.0 < inner <= outer_ms:
                kernel_ms = inner
                timed_by = (f"CUDA event-record nodes inside one graph: measured batches restored to reset + W steps, {n_warm} untimed steps "
                            "on 12 decoy batches (L2 turned over), event, the K timed steps, event")
        except Exception:  # pragma: no cover
            pass
    if args.dump_outputs and rank == 0:  # the last timed step's results, before any other leg reuses the batches
        obs, reward, terminated, truncated, _ = last
        dump_outputs(args.dump_outputs, {"obs": obs, "reward": reward, "terminated": terminated, "truncated": truncated})
    del graph_b
    del graph_a
    restore(env)
    for er in sets[1:] + decoys:
        er.unwrapped.close()
    sets, snaps = [env], snaps[:1]
    # ---- timed region A' (`l2_flushed`): one set, L2 flushed (256 MiB memset) before every step, per-step CUDA events
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    barrier()
    # head start for the host: the device spins ~30 ms while the first steps are enqueued, so that a host thread that is
    # briefly descheduled (N ranks + samplers share the box's cores) never leaves a gap INSIDE a per-step event pair
    if not os.environ.get("EVAC_BENCH_NO_HEADSTART"):
        torch.cuda._sleep(int(0.03 * 1.9e9))
    for s in range(K):
        flush.zero_()
        starts[s].record()
        env.step(actions[W + s])
        ends[s].record()
    barrier()
    flushed_ms = sum(a.elapsed_time(b) for a, b in zip(starts, ends))
    del flush
    # ---- timed region B: the same K per-step launches captured in ONE CUDA graph and replayed (state
    # L2-resident, no host launch overhead) -- how a device-side rollout loop drives the per-step API
    restore(env)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        env.step(actions[W])
        torch.cuda.synchronize(dev)
        with torch.cuda.graph(graph, stream=side):
            for s in range(K):
                env.step(actions[W + s])
    torch.cuda.synchronize(dev)
    graph.replay()
    restore(env)
    barrier()
    e0.record()
    graph.replay()
    e1.record()
    barrier()
    resident_ms = e0.elapsed_time(e1)
    # ---- timed region C: K steps inside ONE launch (state resident on chip, on-device RandomAgent)
    env.rollout(8, agent="random")
    restore(env)
    barrier()
    e0.record()
    env.rollout(K, agent="random")
    e1.record()
    barrier()
    rollout_ms = e0.elapsed_time(e1)
    clocks = sampler.stop()

    # ---- e2e: reference-shaped host call -- NumPy actions in, NumPy obs / reward / flags out
    env_h = eb.setup_env(eb.EnvConfig(**ENV_KW), eb.EnvWrappersConfig(**WRAP_KW), num_envs=E, device=dev, seed=args.seed,
                         auto_reset=True, batched=False, rng="philox", env_index_offset=shard_offset(rank, E))
    env_h.reset()
    host_actions = actions[W:W + K].cpu().numpy()
    for s in range(3):  # warm-up of the host face (K may be below 3)
        env_h.step(host_actions[s % K])
    barrier()
    t0 = time.perf_counter()
    for s in range(K):
        env_h.step(host_actions[s])
    torch.cuda.synchronize(dev)
    e2e_s = time.perf_counter() - t0
    barrier()

    def maxr(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- north-star config C5 (65 536 envs in total, policy in the loop) on THIS run's ranks, strong scaling
    c5 = None
    if not args.no_c5:
        try:
            c5 = c5_leg(args, dev, world, rank, barrier)
        except Exception as exc:  # pragma: no cover
            c5 = {"error": repr(exc)}
    per_rank_us = [1e3 * kernel_ms / K]
    if world > 1:
        t = torch.zeros(world, dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(t, torch.tensor([1e3 * kernel_ms / K], dtype=torch.float64, device=dev))
        per_rank_us = [float(x) for x in t.tolist()]
    kernel_ms, outer_ms, flushed_ms, resident_ms, rollout_ms, e2e_s = (maxr(kernel_ms), maxr(outer_ms), maxr(flushed_ms), maxr(resident_ms),
                                                                        maxr(rollout_ms), maxr(e2e_s))
    if c5 is not None and "ms" in c5:
        c5_by_rank = [c5["ms"]]
        if world > 1:
            t = torch.zeros(world, dtype=torch.float64, device=dev)
            dist.all_gather_into_tensor(t, torch.tensor([c5["ms"]], dtype=torch.float64, device=dev))
            c5_by_rank = [float(x) for x in t.tolist()]
        c5["ms"] = maxr(c5["ms"])
        c5["finite"] = bool(maxr(0.0 if c5["finite"] else 1.0) == 0.0)
        c5["ms_per_iteration_by_rank"] = [x / c5["steps"] for x in c5_by_rank]
    totals = allgather_episode_totals(u)  # the only collective: finished-episode statistics

    if rank == 0:
        hbm_peak, peak_src, peaks = load_peaks()
        total_envs = E * world
        env_steps = total_envs * K
        value = env_steps * N_PED / (kernel_ms * 1e-3)
        bytes_launch = algorithmic_bytes_per_env_step(N_PED, obs_dim * 4) * E
        flops_launch = algorithmic_flops_per_env_step(N_PED) * E
        launch_s = kernel_ms * 1e-3 / K
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):  # dram__bytes of the dominant kernel, captured by ncu IN THE TIMED REGIME (rotating batches, no cache flush)
            with open(tpath) as f:
                tj = json.load(f)
            traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
        fp32_peak = 148 * 128 * 2 * 1.965e9 / 1e12  # nominal, SURVEY.md 8(d); measured FMA probe in profiles/
        line = {
            "metric": "pedestrian-steps/s", "value": value, "unit": "pedestrian-steps/s", "env_steps_per_s": env_steps / (kernel_ms * 1e-3),
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": kernel_ms / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "envs_per_gpu": E, "pedestrians": N_PED, "obs": "rel+ohe Box [62,6] f32",
                       "actions": "U[-1,1]^2 table resident in HBM", "noise": "in-kernel Philox2x32-10", "auto_reset": True,
                       "l2": f"inputs larger than L2: {R} independent C2 batches ({R} x {bytes_launch / 1e6:.1f} MB algorithmic traffic vs 126 MB L2) "
                             "stepped round-robin, one batch per step, K launches in one CUDA graph",
                       "timed_by": timed_by, "ms_per_step_incl_graph_launch": outer_ms / K, "untimed_warmup_steps_in_graph": n_warm,
                       "episode_phase": f"every timed leg starts from reset + {W} warm-up steps (state snapshot restored before the timed replay)",
                       "sets": R, "pdl": bool(int(os.environ.get("EVAC_PDL", "0") or 0)),
                       "parallelism": f"env-sharded x{world}, no data-path collective"},
            "roofline": {"bound": "hbm", "achieved": bytes_launch / launch_s / 1e9, "peak": hbm_peak, "unit": "GB/s",
                         "frac": bytes_launch / launch_s / 1e9 / hbm_peak, "traffic": traffic, "traffic_over_algorithmic": (traffic / bytes_launch) if traffic else None,
                         "traffic_source": traffic_src, "peak_source": peak_src,
                         "kernel": "evac_warp_kernel<WMODE_REL_OHE_BOX> (one warp per environment)", "algorithmic_bytes_per_launch": bytes_launch},
            "roofline_fp32": {"bound": "fp32", "achieved": flops_launch / launch_s / 1e12, "peak": fp32_peak, "unit": "TFLOP/s",
                              "frac": flops_launch / launch_s / 1e12 / fp32_peak, "peak_source": "nominal 148 SM x 128 lanes x 2 x 1.965 GHz",
                              "algorithmic_flops_per_launch": flops_launch},
            "l2_flushed": {"value": env_steps * N_PED / (flushed_ms * 1e-3), "unit": "pedestrian-steps/s", "ms_per_step": flushed_ms / K,
                           "note": "ONE batch, L2 flushed (256 MiB memset) before every step, per-step CUDA events (kernel code cold as well)"},
            "l2_resident": {"value": env_steps * N_PED / (resident_ms * 1e-3), "unit": "pedestrian-steps/s", "ms_per_step": resident_ms / K,
                            "note": "the same K per-step launches captured in one CUDA graph and replayed; no L2 flush (state stays L2-resident)"},
            "rollout": {"value": env_steps * N_PED / (rollout_ms * 1e-3), "unit": "pedestrian-steps/s", "ms_per_step": rollout_ms / K,
                        "note": "K steps in ONE launch (evac_rollout), on-device RandomAgent, obs written after the last step"},
            "e2e": {"value": env_steps * N_PED / e2e_s, "unit": "pedestrian-steps/s", "h2d_bytes_per_step": E * 8,
                    "d2h_bytes_per_step": E * (obs_dim * 4 + 4 + 1 + 1), "ms_per_step": 1e3 * e2e_s / K,
                    "api": "setup_env(..., batched=False).step(numpy actions) -> numpy obs, reward, flags (evac_step_host)",
                    "host_affinity": numa},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "us_per_step_by_rank": per_rank_us,
            "build_id": _build_id(),
            "episodes_finished_all_ranks": float(totals[:, 0].sum()),
        }
        if c5 is not None and "ms" in c5:
            ms5 = c5.pop("ms")
            c5.update({"metric": "pedestrian-steps/s", "value": c5["total_envs"] * c5["steps"] * N_PED / (ms5 * 1e-3), "unit": "pedestrian-steps/s",
                       "env_steps_per_s": c5["total_envs"] * c5["steps"] / (ms5 * 1e-3), "ms_per_iteration": ms5 / c5["steps"], "n_gpus": world,
                       "scaling": "strong", "target": "north_star: >= 1e10 pedestrian-steps/s on 8 x B200"})
        if c5 is not None:
            line["c5"] = c5
        # the secondary legs must never cost the contract line: a failure is reported inside it
        try:
            line["roofline_pairwise"] = pairwise_probe(local_rank)
        except Exception as exc:  # pragma: no cover
            line["roofline_pairwise"] = {"error": repr(exc)}
        if world == 1 and not args.no_extra:
            try:
                line["other_workloads"] = other_workloads(dev)
            except Exception as exc:  # pragma: no cover
                line["other_workloads"] = {"error": repr(exc)}
        if world == 1 and not args.no_cpu:
            try:
                line["cpu_baseline"] = cpu_baseline_single_core(args.cpu_seconds)
            except Exception as exc:  # pragma: no cover
                line["cpu_baseline"] = {"error": repr(exc), "kind": "port", "cores": 1}
            try:
                line["c1_single_env"] = c1_leg(dev)
            except Exception as exc:  # pragma: no cover
                line["c1_single_env"] = {"error": repr(exc)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def _build_id():
    from evacuation_b200 import _native as nat

    return nat.build_id()


DUMP_BYTES = 64 * 10 ** 6 - 4096  # at most 64 MB in all, .npy headers included
DUMP_SAMPLE_SEED = 0


def dump_outputs(directory, arrays):
    """Write every [E, ...] tensor as <directory>/<name>.npy in float32 (flags as 0 / 1).  When they exceed DUMP_BYTES in
    all, the same fixed, seeded sample of environments (rows, ascending) is kept from each."""
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    rows = len(next(iter(arrays.values())))
    keep = min(rows, DUMP_BYTES // (sum(a.nbytes for a in arrays.values()) // rows))
    if keep < rows:
        idx = np.sort(np.random.default_rng(DUMP_SAMPLE_SEED).choice(rows, size=keep, replace=False))
        arrays = {k: a[idx] for k, a in arrays.items()}
    os.makedirs(directory, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(directory, f"{k}.npy"), a)


def pairwise_probe(device_index):
    """north_star: ">= 50 % of the FP32 roofline on the pairwise alignment kernel".  Standalone launches of the SAME
    `pairwise_pass` device function the fused step uses (probe_pairwise_kernel<32, 2>: one warp per environment, two
    pedestrians per lane), N = 60, at the bench batch and at the C5 batch; 8 algorithmic flops per ordered pair (SURVEY 8d);
    peak = the FFMA2 probe measured in the same process (nominal 148 x 128 x 2 x 1.965 GHz = 74.4 TFLOP/s beside it)."""
    import ctypes as C

    from evacuation_b200 import _native as nat

    lib = nat.load()
    ms, fl, pairs = C.c_float(), C.c_double(), C.c_double()
    peak = 0.0
    for _ in range(3):
        nat.check(lib.evac_probe_fma(device_index, 1, 20000, C.byref(ms), C.byref(fl)))
        peak = max(peak, fl.value / (ms.value * 1e-3) / 1e12)
    out = {"bound": "fp32", "unit": "TFLOP/s", "peak": peak, "peak_source": "FFMA2 probe (evac_probe_fma) in this process",
           "peak_nominal": 148 * 128 * 2 * 1.965e9 / 1e12, "kernel": "probe_pairwise_kernel<32,2>: pairwise_pass<2,false,4> of the fused step, standalone",
           "flops_per_ordered_pair": 8, "cases": {}}
    for E, reps in ((ENVS_PER_GPU, 200), (65536, 50)):
        best = 0.0
        for _ in range(3):
            nat.check(lib.evac_probe_pairwise(device_index, E, N_PED, reps, C.byref(ms), C.byref(pairs)))
            best = max(best, pairs.value / (ms.value * 1e-3))
        out["cases"][f"{E}x{N_PED}"] = {"achieved": best * 8 / 1e12, "frac": best * 8 / 1e12 / peak, "frac_of_nominal": best * 8 / out["peak_nominal"] / 1e12,
                                         "ordered_pairs_per_s": best}
    head = out["cases"][f"{ENVS_PER_GPU}x{N_PED}"]
    out["achieved"], out["frac"] = head["achieved"], head["frac"]
    # beside it, NOT the fused kernel's shape: 16 lanes x 4 pedestrians per environment, two environments per warp (fewer LDS
    # and loop instructions per evaluated pair; needs many warps: better at 65 536 envs, worse at 4096)
    os.environ["EVAC_PROBE_HALFWARP"] = "2"
    try:
        var = {}
        for E, reps in ((ENVS_PER_GPU, 200), (65536, 50)):
            best = 0.0
            for _ in range(3):
                nat.check(lib.evac_probe_pairwise(device_index, E, N_PED, reps, C.byref(ms), C.byref(pairs)))
                best = max(best, pairs.value / (ms.value * 1e-3))
            var[f"{E}x{N_PED}"] = {"achieved": best * 8 / 1e12, "frac": best * 8 / 1e12 / peak}
        out["variant_16x4_two_envs_per_warp"] = var
        # ... and 8 lanes x 8 pedestrians per environment, four environments per warp: one broadcast LDS.128 pair per 64 packed
        # math instructions instead of per 16 -- the same pairwise_pass device function (PPT = 8) as a standalone kernel; this is
        # the mapping that crosses the north-star's 50 % at its own batch (65 536 x 60).  The fused step keeps 32 x 2: the step as
        # a whole needs its 7 resident warps per scheduler (DESIGN.md section 8: the half-warp step kernel measured slower).
        os.environ["EVAC_PROBE_HALFWARP"] = "8"
        var = {}
        for E, reps in ((ENVS_PER_GPU, 200), (65536, 50)):
            best = 0.0
            for _ in range(3):
                nat.check(lib.evac_probe_pairwise(device_index, E, N_PED, reps, C.byref(ms), C.byref(pairs)))
                best = max(best, pairs.value / (ms.value * 1e-3))
            var[f"{E}x{N_PED}"] = {"achieved": best * 8 / 1e12, "frac": best * 8 / 1e12 / peak}
        out["variant_8x8_four_envs_per_warp"] = var
        out["best_standalone"] = {"mapping": "8 lanes x 8 pedestrians, four environments per warp", "case": f"65536x{N_PED}", **var[f"65536x{N_PED}"],
                                  "target": 0.5, "met": bool(var[f"65536x{N_PED}"]["frac"] >= 0.5)}
    finally:
        os.environ.pop("EVAC_PROBE_HALFWARP", None)
    return out


def c5_leg(args, dev, world, rank, barrier):
    """BASELINE config 5 inside the contract run, for EVERY --gpus N: 65 536 envs x 60 pedestrians in TOTAL, sharded over the
    ranks (strong scaling), the RPO transformer-embedding policy in the rollout loop (rpo_agent.py:180-203: fused CUDA
    policy -> fused env step -> reward normaliser, 4 launches per iteration, CUDA-graph replayed, dropout active).  Returns
    this rank's device time; the caller takes the max over ranks."""
    import torch

    import evacuation_b200 as eb
    from evacuation_b200.distributed import shard_offset
    from evacuation_b200.rollout import FusedRPOTransformerPolicy, PolicyRollout, RPOTransformerPolicy

    total = 65536
    E = total // world
    K5, W5 = int(min(max(args.steps, 1), 64)), int(min(max(args.warmup, 3), 16))
    env = eb.setup_env(eb.EnvConfig(**ENV_KW), eb.EnvWrappersConfig(**WRAP_KW), num_envs=E, device=dev, seed=args.seed, auto_reset=True,
                       env_index_offset=shard_offset(rank, E))
    torch.manual_seed(1)  # every rank holds the same policy replica
    net = RPOTransformerPolicy(env.unwrapped.obs_dim, N_PED).to(dev)
    pol = FusedRPOTransformerPolicy(net, N_PED, device=dev, seed=args.seed, env_index_offset=shard_offset(rank, E))
    ro = PolicyRollout(env, pol, use_graph=True, store=False)
    ro.reset()
    ro.run(W5)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    ro.run(K5)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    out = {"ms": ms, "steps": K5, "warmup": W5, "total_envs": total, "envs_per_gpu": E, "finite": bool(torch.isfinite(ro.out["value"]).all()),
           "gpu_launches": int((ro.launches_per_iteration or 0) * K5), "launches_per_iteration": ro.launches_per_iteration,
           "workload": "C5: 65536 envs x 60 pedestrians in total, env-sharded, RPO transformer-embedding policy (2 blocks, 3 heads, d_ff 96, dropout 0.1 "
                       "active, MLP heads 372-64-64, random init seed 1) in the loop; one CUDA graph per iteration (4 kernels)",
           "l2": "working set 4.5 KB per env: larger than L2 from 32768 envs per GPU; no flush"}
    env.unwrapped.close()
    del ro, pol, net
    torch.cuda.empty_cache()
    return out


def other_workloads(dev):
    """Secondary BASELINE.json configs (parity-test cases, not the bench line): a short device-timed measurement of
    each so that one bench run documents them.  Two regimes per workload, labelled:
      per_step : K calls of `env.step(actions)` (one launch each, observation written every step) captured in one CUDA graph;
                 where one batch's working set is smaller than L2, R independent batches are stepped round-robin so that
                 every step finds its state in HBM (same rule as the headline value);
      rollout  : K steps inside ONE `evac_rollout` launch (state resident on chip, on-device RandomAgent, observation written
                 after the last step only) -- the steady state of the kernel, NOT a per-step number.
    HBM fractions use the algorithmic bytes of SURVEY 8(d) and are only quoted for the per_step regime (a rollout step moves
    no state).  Config 5 additionally with the RPO transformer-embedding policy in the loop."""
    import torch

    import evacuation_b200 as eb

    hbm_peak, _, _ = load_peaks()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def measure(env_kw, wrap_kw, E, K, R=1, **kw):
        n = env_kw["number_of_pedestrians"]
        sets = []
        for r in range(R):
            env = eb.setup_env(eb.EnvConfig(**env_kw), eb.EnvWrappersConfig(**wrap_kw), num_envs=E, device=dev, seed=7 + r, auto_reset=True, **kw)
            env.reset()
            env.rollout(64, agent="random")
            sets.append(env)
        snaps = [x.unwrapped.save_state() for x in sets]
        g = torch.Generator(device=dev).manual_seed(99)
        acts = torch.rand((K, E, 2), generator=g, device=dev) * 2 - 1
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        graph, side = torch.cuda.CUDAGraph(), torch.cuda.Stream(device=dev)
        torch.cuda.synchronize(dev)
        with torch.cuda.stream(side):
            for env in sets:
                env.unwrapped.step(acts[0])
            torch.cuda.synchronize(dev)
            with torch.cuda.graph(graph, stream=side):
                for s_ in range(K):
                    sets[s_ % R].unwrapped.step(acts[s_])
        torch.cuda.synchronize(dev)
        graph.replay()  # untimed: graph upload
        for x, img in zip(sets, snaps):  # every timed replay starts from the same crowd (64 steps after reset): a crowd flocks
            x.unwrapped.load_state(img)  # and escapes as an episode ages, and the cost of a step follows it
        flush.zero_()                    # (the restored state leaves the L2)
        torch.cuda.synchronize(dev)
        e0.record()
        graph.replay()
        e1.record()
        torch.cuda.synchronize(dev)
        us_step = 1e3 * e0.elapsed_time(e1) / K
        del graph
        env = sets[0]
        env.unwrapped.load_state(snaps[0])
        torch.cuda.synchronize(dev)
        e0.record()
        env.rollout(K, agent="random")
        e1.record()
        torch.cuda.synchronize(dev)
        us_roll = 1e3 * e0.elapsed_time(e1) / K
        obs_bytes = env.unwrapped.obs_dim * 4
        bytes_step = algorithmic_bytes_per_env_step(n, obs_bytes) * E
        for env in sets:
            env.unwrapped.close()
        return {"envs": E, "pedestrians": n, "batches_round_robin": R,
                "per_step": {"us_per_step": us_step, "pedestrian_steps_per_s": E * n / us_step * 1e6, "env_steps_per_s": E / us_step * 1e6,
                             "algorithmic_bytes_per_step": bytes_step, "hbm_GBps": bytes_step / us_step / 1e3,
                             "hbm_frac": bytes_step / us_step / 1e3 / hbm_peak},
                "rollout": {"us_per_step": us_roll, "pedestrian_steps_per_s": E * n / us_roll * 1e6, "env_steps_per_s": E / us_roll * 1e6,
                            "note": "K steps in one launch; observation written after the last step only"}}

    fp32_peak = 148 * 128 * 2 * 1.965e9
    out = {}
    out["c3_grav_4096x60"] = measure(dict(number_of_pedestrians=60, enslaving_degree=0.5, noise_coef=0.5), dict(positions="grav", alpha=3), 4096, 192, R=24)
    out["c4_large_crowd_256x4096_cells"] = measure(dict(number_of_pedestrians=4096), WRAP_KW, 256, 20, R=4)
    ap = measure(dict(number_of_pedestrians=4096), WRAP_KW, 256, 4, R=1, neighbor_search="brute")
    for reg in ("per_step", "rollout"):  # all pairs: the only large-crowd leg whose work IS the algorithmic 8 N^2 flops
        ap[reg]["fp32_frac_algorithmic"] = 256 * algorithmic_flops_per_env_step(4096) / (ap[reg]["us_per_step"] * 1e-6) / fp32_peak
    out["c4_large_crowd_256x4096_all_pairs"] = ap
    out["large_crowd_32x32768_cluster"] = measure(dict(number_of_pedestrians=32768), WRAP_KW, 32, 8, R=4)  # one env per thread-block cluster
    c5 = measure(ENV_KW, WRAP_KW, 65536, 48, R=2)
    for reg in ("per_step", "rollout"):
        c5[reg]["fp32_frac_algorithmic"] = 65536 * algorithmic_flops_per_env_step(60) / (c5[reg]["us_per_step"] * 1e-6) / fp32_peak
    out["c5_env_only_65536x60"] = c5
    # config 5, one rank's share of the 8-GPU job (65536 / 8 envs) with the policy in the loop: the fused CUDA policy
    # (evac_policy_forward: embedding kernel + heads kernel, NormalizeObservation / ClipAction fused) and, beside it, the
    # same loop with the PyTorch restatement of the policy (library GEMMs / SDPA).  (65536 envs on this GPU: the `c5` object.)
    from evacuation_b200.rollout import FusedRPOTransformerPolicy, PolicyRollout, RPOTransformerPolicy

    def policy_loop_ms(E, fused, steps):
        env = eb.setup_env(eb.EnvConfig(**ENV_KW), eb.EnvWrappersConfig(**WRAP_KW), num_envs=E, device=dev, seed=7, auto_reset=True)
        torch.manual_seed(1)
        net = RPOTransformerPolicy(env.unwrapped.obs_dim, N_PED).to(dev)  # train mode: dropout active like the reference's rollouts
        pol = FusedRPOTransformerPolicy(net, N_PED, device=dev, seed=1) if fused else net
        ro = PolicyRollout(env, pol, use_graph=True, store=False)
        ro.reset()
        ro.run(4)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        e0.record()
        ro.run(steps)
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / steps
        assert bool(torch.isfinite(ro.out["value"]).all())
        env.unwrapped.close()
        return ms

    for E, fused, steps, key in ((8192, True, 64, "c5_policy_loop_8192x60"), (8192, False, 8, "c5_policy_loop_8192x60_torch_policy")):
        ms = policy_loop_ms(E, fused, steps)
        out[key] = {"envs": E, "pedestrians": N_PED, "ms_per_step": ms, "pedestrian_steps_per_s": E * N_PED / ms * 1e3, "env_steps_per_s": E / ms * 1e3,
                    "note": ("fused CUDA policy (evac_policy_forward: NormalizeObservation + 2 transformer blocks, heads + Normal sampling + ClipAction) "
                             "-> fused env step -> evac_normalize_reward: 4 launches per iteration, CUDA-graph replayed, dropout active") if fused else
                            "the same loop with the PyTorch restatement of the policy (library GEMMs / SDPA), CUDA-graph replayed"}
    return out


def run_c5(args):
    """--workload c5: BASELINE config 5 -- 65 536 envs x 60 pedestrians in TOTAL, sharded over the ranks (strong scaling),
    with the RPO transformer-embedding policy in the rollout loop (fused CUDA policy -> fused env step -> reward
    normaliser, CUDA-graph replayed, dropout active).  Same launch / timing contract as the default workload; NCCL only
    all-gathers the finished-episode statistics after the timed region.  Not the driver's bench line (that is C2)."""
    import torch
    import torch.distributed as dist

    import evacuation_b200 as eb
    from evacuation_b200.distributed import allgather_episode_totals, shard_offset
    from evacuation_b200.rollout import FusedRPOTransformerPolicy, PolicyRollout, RPOTransformerPolicy

    world, rank, local_rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        _nccl_output_to_stderr()
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    total = 65536
    E, K, W = total // world, args.steps, max(args.warmup, 3)
    env = eb.setup_env(eb.EnvConfig(**ENV_KW), eb.EnvWrappersConfig(**WRAP_KW), num_envs=E, device=dev, seed=args.seed, auto_reset=True,
                       env_index_offset=shard_offset(rank, E))
    torch.manual_seed(1)  # every rank holds the same policy replica
    net = RPOTransformerPolicy(env.unwrapped.obs_dim, N_PED).to(dev)
    pol = FusedRPOTransformerPolicy(net, N_PED, device=dev, seed=args.seed, env_index_offset=shard_offset(rank, E))
    ro = PolicyRollout(env, pol, use_graph=True, store=False)
    ro.reset()
    ro.run(W)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    sampler = ClockSampler(local_rank)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = env.unwrapped.launch_count + pol.launch_count
    barrier()
    sampler.start()
    e0.record()
    ro.run(K)
    e1.record()
    barrier()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1)
    launches = env.unwrapped.launch_count + pol.launch_count - l0
    finite = bool(torch.isfinite(ro.out["value"]).all())
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    totals = allgather_episode_totals(env.unwrapped)
    if rank == 0:
        line = {"metric": "pedestrian-steps/s", "value": total * K * N_PED / (ms * 1e-3), "unit": "pedestrian-steps/s",
                "env_steps_per_s": total * K / (ms * 1e-3), "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": "C5: 65536 envs x 60 pedestrians in total with the RPO transformer-embedding policy in the rollout loop",
                           "envs_per_gpu": E, "policy": "2 blocks, 3 heads, d_ff 96, dropout 0.1 active, MLP heads 372-64-64, random init seed 1",
                           "loop": "evac_policy_forward (embedding + heads kernels) -> evac_step -> evac_normalize_reward, one CUDA graph per iteration",
                           "l2": "working set (obs + normaliser statistics, 4.5 KB per env) exceeds L2 only at >= 32768 envs per GPU; no flush",
                           "parallelism": f"env-sharded x{world}, policy replicated, no data-path collective"},
                "gpu_launches": int(launches), "clocks": clocks, "finite": finite, "episodes_finished_all_ranks": float(totals[:, 0].sum())}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=ENVS_PER_GPU, help="environments per GPU")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--sets", type=int, default=24, help="independent batches stepped round-robin so that the inputs exceed L2")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extra", action="store_true", help="skip the other_workloads leg (secondary BASELINE configs)")
    ap.add_argument("--no-c5", action="store_true", help="skip the C5 leg (65536 envs in total with the policy in the loop)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--workload", default="c2", choices=["c2", "c5"], help="c2 = the bench line; c5 = config 5 with the policy in the loop")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs (C2, rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "c2"):
        ap.error("--dump-outputs writes the outputs of the C2 path (--impl ours --workload c2)")
    if args.impl == "reference":
        run_reference_arm(args)
    elif args.workload == "c5":
        run_c5(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    sys.dont_write_bytecode = True  # (the tree may be read-only)
    main()
