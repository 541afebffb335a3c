"""The linear RPO policy (RPOLinearNetwork on the flattened observation) in the rollout loop, for the gravity-encoding (K = 6) and the
Dict rel + ohe (K = 364) configs at N = 60: ms per iteration of `PolicyRollout` with the fused policy (3 launches: heads with the
fused NormalizeObservation, env step, reward normaliser) against the same loop with the torch `RPOLinearPolicy` (both CUDA-graph
replayed after the same warm-up, alternated), the fused heads kernel alone (with the normaliser, and without it on an already
normalised observation), and the env step alone (CUDA events over many launches).  One JSON line per (config, E), preceded by
the card's name / power limit / max SM clock read in the same run.

Usage: python tools/linear_rollout.py [--out FILE.jsonl] [--sizes 4096,8192,65536] [--steps 200] [--reps 3]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import evacuation_b200 as eb
from evacuation_b200.rollout import FusedRPOLinearPolicy, PolicyRollout, RPOLinearPolicy, VectorNormalizer

CONFIGS = {"grav": dict(positions="grav", type="Dict"), "dict_rel_ohe": dict(positions="rel", statuses="ohe", type="Dict")}
N = 60


def make_env(cfg, E):
    return eb.setup_env(eb.EnvConfig(number_of_pedestrians=N, is_new_exiting_reward=True), eb.EnvWrappersConfig(**CONFIGS[cfg]),
                        num_envs=E, seed=1, auto_reset=True)


def events_ms(fn, n):
    """Mean ms per call of `fn` over n calls on the current stream (CUDA events, after one warm call)."""
    fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def loop_ms(ro, steps, warmup):
    ro.run(warmup)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    ro.run(steps)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def measure(cfg, E, steps, reps, warmup=8):
    torch.manual_seed(1)
    K = make_env(cfg, 1).unwrapped.obs_dim
    net = RPOLinearPolicy(K).cuda()
    fused = FusedRPOLinearPolicy(net, K, device="cuda", seed=1)
    ro_f = PolicyRollout(make_env(cfg, E), fused, use_graph=True, store=False)
    ro_t = PolicyRollout(make_env(cfg, E), net, use_graph=True, store=False)
    ro_f.reset(); ro_t.reset()
    fused_ms, torch_ms = [], []
    for _ in range(reps):  # alternated, so that both loops see the same machine state
        fused_ms.append(loop_ms(ro_f, steps, warmup))
        torch_ms.append(loop_ms(ro_t, steps, warmup))
    # the heads kernel alone: with the fused normaliser (the loop's launch) and without it on a normalised observation
    x = make_env(cfg, E)
    x.reset()
    raw = x.unwrapped.flat_observation
    norm = VectorNormalizer(E, K, device="cuda")
    o = dict(action=torch.empty((E, 2), device="cuda"), action_clipped=torch.empty((E, 2), device="cuda"), logprob=torch.empty(E, device="cuda"),
             value=torch.empty(E, device="cuda"))
    xn = torch.empty((E, K), device="cuda")
    heads_norm = events_ms(lambda: fused.forward(raw, normalizer=norm, obs_norm=xn, **o), 200)
    heads_plain = events_ms(lambda: fused.forward(xn, **o), 200)
    acts = torch.rand((E, 2), device="cuda") * 2 - 1
    env_ms = events_ms(lambda: x.step(acts), 200)
    f, t = min(fused_ms), min(torch_ms)
    return dict(config=cfg, N=N, K=K, E=E, steps=steps, reps=reps, fused_loop_ms=fused_ms, torch_loop_ms=torch_ms,
                fused_launches_per_iteration=ro_f.launches_per_iteration, torch_launches_per_iteration=ro_t.launches_per_iteration,
                speedup_best=t / f, heads_norm_us=heads_norm * 1e3, heads_plain_us=heads_plain * 1e3, env_step_us=env_ms * 1e3,
                fused_finite=bool(torch.isfinite(ro_f.next_obs).all()), torch_finite=bool(torch.isfinite(ro_t.next_obs).all()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="4096,8192,65536")
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tools/linear_rollout.py measures on a CUDA device; none is visible")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    lines = [dict(kind="device", torch_name=torch.cuda.get_device_name(), nvidia_smi=smi.stdout.strip().splitlines())]
    for cfg in CONFIGS:
        for E in (int(s) for s in args.sizes.split(",")):
            lines.append(measure(cfg, E, args.steps, args.reps))
            print(json.dumps(lines[-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write("".join(json.dumps(l) + "\n" for l in lines))
    print(json.dumps(lines[0]))


if __name__ == "__main__":
    main()
