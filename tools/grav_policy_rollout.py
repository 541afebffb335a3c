"""The gravity-encoding rollout loop (N = 60, RPOLinearNetwork on 6 floats) on a B200: the CUDA-graph loop of three library launches
per step (heads with the fused NormalizeObservation, env step, reward normaliser; `PolicyRollout.run(T)`) against the one-launch loop
(`evac_rollout_policy`, `PolicyRollout.run(T, steps_per_launch=K)`) at K = 16 / 64 / 256, storage on; and the evaluation mode
(`fused_policy_rollout` with the clipped mean, a frozen normaliser, no storage, status counts) at the same K.

CUDA events around `--steps` iterations after a warm-up of the same shape; each configuration is timed `--reps` times, alternated,
and the median is reported.  Every timed run is checked: the storage, both normalisers and the env's state image of each one-launch
run are torch.equal to the graph loop's from the same seeds; the evaluation's status counts are equal across K.  One JSON line per
(mode, E, K) to <out_dir>/grav_policy_rollout.jsonl, preceded by the card's name and power limit read in the same run.

Usage: python tools/grav_policy_rollout.py OUT_DIR [--sizes 4096,8192,65536] [--steps 256] [--reps 3]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import evacuation_b200 as eb
from evacuation_b200.rollout import FusedRPOLinearPolicy, PolicyRollout, RPOLinearPolicy, VectorNormalizer, fused_policy_rollout

N = 60
KS = (16, 64, 256)


def make_env(E, auto_reset=True):
    return eb.setup_env(eb.EnvConfig(number_of_pedestrians=N, is_new_exiting_reward=True), eb.EnvWrappersConfig(positions="grav", type="Dict"),
                        num_envs=E, seed=1, auto_reset=auto_reset)


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def state(ro):
    n, u = ro.norm, ro.env.unwrapped
    return [ro.next_done, n.obs_mean, n.obs_var, n.obs_count, n.returns, n.ret_mean, n.ret_var, n.ret_count, ro.policy.calls,
            u.save_state(), u.flat_observation]


def train_mode(net, E, steps, reps, warmup):
    """ms per iteration of the graph loop and of the one-launch loop at each K; every timed run checked against the graph loop's."""
    ros = {k: PolicyRollout(make_env(E), FusedRPOLinearPolicy(net, 6, device="cuda", seed=1), use_graph=True, store=True) for k in (1, *KS)}
    for k, ro in ros.items():
        ro.reset()
        ro.run(warmup, steps_per_launch=k)
    times = {k: [] for k in ros}
    equal = True
    for _ in range(reps):
        bufs = {}
        for k, ro in ros.items():
            ms, bufs[k] = timed(lambda: ro.run(steps, steps_per_launch=k))
            times[k].append(ms / steps)
        for k in KS:
            equal &= all(torch.equal(bufs[1][key], bufs[k][key]) for key in bufs[1])
            equal &= all(torch.equal(a, b) for a, b in zip(state(ros[1]), state(ros[k])))
    return {k: statistics.median(v) for k, v in times.items()}, bool(equal)


def eval_mode(net, E, steps, reps):
    """ms per step of the evaluation launches (actor only, frozen normaliser, status counts) at each K, from the same reset."""
    pol = FusedRPOLinearPolicy(net, 6, device="cuda", seed=1).eval()
    norm = VectorNormalizer(E, 6, device="cuda")
    times, counts = {k: [] for k in KS}, {}
    for _ in range(reps):
        for k in KS:
            env = make_env(E, auto_reset=False)
            env.reset()
            nd = torch.zeros(E, device="cuda")
            trace = torch.empty((steps, E, 4), dtype=torch.int16, device="cuda")
            fused_policy_rollout(env, pol, k, nd, normalizer=norm, norm_update=False, normalize_reward=False, sample=False,
                                 status_counts=trace[:k])  # warm-up of this launch shape
            env.reset()
            nd.zero_()

            def run():
                for t in range(0, steps, k):
                    fused_policy_rollout(env, pol, k, nd, normalizer=norm, norm_update=False, normalize_reward=False, sample=False,
                                         status_counts=trace[t:t + k])
            ms, _ = timed(run)
            times[k].append(ms / steps)
            counts[k] = trace
    equal = all(torch.equal(counts[KS[0]], counts[k]) for k in KS)
    return {k: statistics.median(v) for k, v in times.items()}, bool(equal)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--sizes", default="4096,8192,65536")
    ap.add_argument("--steps", type=int, default=256)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=32)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("grav_policy_rollout.py measures on the GPU; no CUDA device is visible")
    if any(args.steps % k for k in KS):
        raise SystemExit(f"--steps must be a multiple of {KS}")
    os.makedirs(args.out_dir, exist_ok=True)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    card = {"gpu": q.stdout.strip() or torch.cuda.get_device_name(), "torch_name": torch.cuda.get_device_name()}
    torch.manual_seed(1)
    net = RPOLinearPolicy(6).cuda()
    with open(os.path.join(args.out_dir, "grav_policy_rollout.jsonl"), "w") as f:
        def emit(rec):
            print(json.dumps(rec), flush=True)
            f.write(json.dumps(rec) + "\n")
        emit(card)
        for E in (int(s) for s in args.sizes.split(",")):
            tr, eq = train_mode(net, E, args.steps, args.reps, args.warmup)
            for k, ms in tr.items():
                emit(dict(mode="train", E=E, N=N, steps_per_launch=k, us_per_step=round(ms * 1e3, 3),
                          speedup_vs_graph=round(tr[1] / ms, 3), equal_to_graph_loop=eq))
            ev, eq = eval_mode(net, E, args.steps, args.reps)
            for k, ms in ev.items():
                emit(dict(mode="eval", E=E, N=N, steps_per_launch=k, us_per_step=round(ms * 1e3, 3), equal_across_K=eq))


if __name__ == "__main__":
    main()
