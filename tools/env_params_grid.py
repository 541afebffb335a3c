"""Per-environment parameters on a B200: the reference's noise x enslaving grid as ONE handle against one uniform handle per
grid point, and the per-env step kernel against the uniform one.

  python tools/env_params_grid.py OUT_DIR [--replicas R] [--steps T] [--reps K]

1. Grid: noise in {0.05, 0.2, 0.5, 0.8} x enslaving in {1, 0.5, 0.1} (12 points), R environments each.  One handle of 12 R
   environments with per-env parameters against 12 uniform handles of R environments (env_index_offset = point x R, so their
   random streams are the grid handle's).  For the random and wacuum agents, the per-step status counts of
   rollout(..., status_counts=True) must be bit-identical.  Then the time per step of the one launch against the 12 launches.
2. Per-env against uniform kernel, alternated, with the per-env records set to the uniform handle's values: 4096 x 60 rel +
   ohe Box per step (rollout of 1) and in a K = 100 rollout, and 4096 x 60 grav (alpha through the per-env record).
Every result is one JSON line in OUT_DIR/env_params_grid.jsonl, with the card's name and power limit read in the same run.
Needs a GPU; fails without one."""
import argparse
import itertools
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import evacuation_b200 as eb  # noqa: E402

NOISES, ENSLAVINGS = (0.05, 0.2, 0.5, 0.8), (1.0, 0.5, 0.1)
REL_OHE_BOX = dict(positions="rel", statuses="ohe", type="Box")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = (s.strip() for s in q.stdout.splitlines()[0].split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def make(E, wrap, offset=0, seed=7, **env_kw):
    wrap = dict(wrap)
    if "alpha" in env_kw:
        wrap["alpha"] = env_kw.pop("alpha")
    env = eb.setup_env(eb.EnvConfig(number_of_pedestrians=60, max_timesteps=200, **env_kw), eb.EnvWrappersConfig(**wrap), num_envs=E,
                       device="cuda:0", seed=seed, env_index_offset=offset, batched=True, auto_reset=True)
    env.unwrapped.reset()
    return env.unwrapped


def time_us(fns, steps_per_call, calls, reps):
    """Median microseconds per step of each fn, reps rounds alternating between the fns, `calls` calls per timed window."""
    times = [[] for _ in fns]
    for fn in fns:  # warm-up
        fn()
    torch.cuda.synchronize()
    for _ in range(reps):
        for i, fn in enumerate(fns):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(calls):
                fn()
            b.record()
            b.synchronize()
            times[i].append(a.elapsed_time(b) * 1e3 / (calls * steps_per_call))
    return [(float(np.median(t)), float(np.min(t)), float(np.max(t))) for t in times]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--replicas", type=int, default=256)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--reps", type=int, default=15)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures on the GPU")
    os.makedirs(args.out_dir, exist_ok=True)
    path = os.path.join(args.out_dir, "env_params_grid.jsonl")
    info = card()
    out = open(path, "w")

    def emit(rec):
        rec = {**rec, **info}
        out.write(json.dumps(rec) + "\n")
        out.flush()
        print(json.dumps(rec))

    # ---- 1. grid: one handle against 12
    R, points = args.replicas, list(itertools.product(NOISES, ENSLAVINGS))
    E = R * len(points)
    for agent in ("random", "wacuum"):
        grid = make(E, REL_OHE_BOX)
        grid.set_env_params(noise_coef=np.repeat([p[0] for p in points], R), enslaving_degree=np.repeat([p[1] for p in points], R))
        grid.reset()
        singles = [make(R, REL_OHE_BOX, offset=i * R, noise_coef=n, enslaving_degree=s) for i, (n, s) in enumerate(points)]
        for u in singles:
            u.reset()
        grid.rollout(args.steps, agent=agent, status_counts=True)
        want = grid.last_status_counts.clone()
        got = []
        for u in singles:
            u.rollout(args.steps, agent=agent, status_counts=True)
            got.append(u.last_status_counts.clone())
        same = bool(torch.equal(want, torch.cat(got, dim=1)))
        assert same, f"{agent}: status counts of the grid handle differ from the 12 uniform handles"
        escaped = want[-1, :, 0].view(len(points), R).to(torch.float64).mean(dim=1).tolist()
        per_step = time_us([lambda: grid.rollout(1, agent=agent), lambda: [u.rollout(1, agent=agent) for u in singles]], 1, 200, args.reps)
        emit({"what": "grid_one_handle_vs_12", "agent": agent, "replicas": R, "envs": E, "status_counts_bit_identical": same,
              "mean_escaped_after_steps": dict(zip([f"noise={n},enslaving={s}" for n, s in points], escaped)), "steps": args.steps,
              "us_per_step_one_handle": per_step[0], "us_per_step_12_handles": per_step[1]})
        del grid, singles

    # ---- 2. per-env kernel against the uniform kernel.  The per-env handle's records hold the uniform handle's own values
    # (set_env_params(**uni.env_params())), so both run the same dynamics and the per-env record load is the only difference.
    for label, wrap, extra in (("rel_ohe_box", REL_OHE_BOX, {}), ("grav", dict(positions="grav"), dict(alpha=3.0))):
        uni, per = make(4096, wrap, **extra), make(4096, wrap, **extra)
        per.set_env_params(**uni.env_params())
        for k, calls in ((1, 400), (100, 8)):
            if label == "grav" and k == 100:
                continue
            t = time_us([lambda: uni.rollout(k, agent="random"), lambda: per.rollout(k, agent="random")], k, calls, args.reps)
            emit({"what": "per_env_vs_uniform_kernel", "obs": label, "envs": 4096, "pedestrians": 60, "steps_per_launch": k,
                  "per_env_values": "equal to the uniform handle's", "us_per_step_uniform": t[0], "us_per_step_per_env": t[1]})
    out.close()
    print("wrote", path)


if __name__ == "__main__":
    main()
