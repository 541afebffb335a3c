"""Evaluation of trained fused policies on a B200 (`rollout.evaluate_policy`: one replayed CUDA graph of the frozen-normaliser policy
forward + one table-agent step per step, status counts recorded):

  * the transformer policy (Box rel + ohe, N = 60, K = 372) and the flat linear policy (Dict rel + ohe, N = 60, K = 364) at 8192 and
    65 536 environments;
  * the gravity-encoding linear policy (K = 6, N = 60) at 4096 / 8192 / 65 536 environments: the per-step loop against the one-launch
    evaluation of `evac_rollout_policy` (`fused_policy_rollout`, 256 steps per launch);
  * the frozen tensor-core heads alone (K = 364, 8192 environments): 64-column against 128-column tiles (EVAC_POLICY_TC=128 pins the
    latter).

Times are CUDA events around whole calls, per step.  `us_per_step` divides a call of --steps steps (graph capture included) by the
steps; `us_per_step_marginal` is (t(2 steps) - t(steps)) / steps, the replay cost without the capture.  The configurations of one
group are alternated over --reps rounds and the median reported.  Every timed run is checked against an untimed reference run from the
same start: status counts and the env's state image torch.equal (the grav per-step loop also against the one-launch evaluation), the
heads' outputs torch.equal to the same tiling's untimed call.  One JSON line per measurement to <out_dir>/policy_eval.jsonl, preceded
by the card's name and power limit read in the same run.

Usage: python tools/policy_eval.py OUT_DIR [--steps 64] [--reps 3]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import evacuation_b200 as eb
from evacuation_b200.rollout import (FusedRPOLinearPolicy, FusedRPOTransformerPolicy, RPOLinearPolicy, RPOTransformerPolicy, VectorNormalizer,
                                     evaluate_policy, fused_policy_rollout)

N = 60
WRAP = {"tf": dict(positions="rel", statuses="ohe", type="Box"), "flat": dict(positions="rel", statuses="ohe", type="Dict"),
        "grav": dict(positions="grav", type="Dict")}


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def make_env(kind, E):
    cfg = eb.EnvConfig(number_of_pedestrians=N, is_new_exiting_reward=True, max_timesteps=2000)
    env = eb.setup_env(cfg, eb.EnvWrappersConfig(**WRAP[kind]), num_envs=E, seed=1, auto_reset=False, batched=True, rng="philox")
    env.unwrapped.reset()
    return env


def frozen_normalizer(E, K):
    n = VectorNormalizer(E, K, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(2)
    n.obs_mean.copy_(torch.randn(E, K, device="cuda", generator=g) * 0.3)
    n.obs_var.copy_(torch.rand(E, K, device="cuda", generator=g) * 2 + 0.05)
    n.obs_count.fill_(100.0)
    return n


def make_policy(kind, K):
    torch.manual_seed(1)
    if kind == "tf":
        return FusedRPOTransformerPolicy(RPOTransformerPolicy(K, N).cuda(), N, device="cuda", seed=1)
    return FusedRPOLinearPolicy(RPOLinearPolicy(K).cuda(), K, device="cuda", seed=1)


class Case:
    """One evaluation configuration on its own env: run(T) from the saved start, checked against the untimed reference of T steps."""

    def __init__(self, kind, E, one_launch=False):
        self.env, self.E, self.one_launch = make_env(kind, E), E, one_launch
        u = self.env.unwrapped
        self.K = u.obs_dim
        self.pol, self.norm = make_policy(kind, self.K), frozen_normalizer(E, self.K)
        self.start, self.obs0 = u.save_state().clone(), u.flat_observation.clone()
        self.ref = {}

    def run(self, T):
        u = self.env.unwrapped
        u.load_state(self.start)
        u.flat_observation.copy_(self.obs0)
        trace = torch.empty((T, self.E, 4), dtype=torch.int16, device="cuda")

        def go():
            if self.one_launch:
                nd = torch.zeros(self.E, device="cuda")
                for t in range(0, T, 256):
                    fused_policy_rollout(self.env, self.pol, min(256, T - t), nd, normalizer=self.norm, norm_update=False,
                                         normalize_reward=False, sample=False, status_counts=trace[t:t + 256])
            else:
                evaluate_policy(self.env, self.pol, T, normalizer=self.norm, status_counts=trace)
        ms = timed(go)
        out = (trace, u.save_state())
        if T not in self.ref:
            self.ref[T] = out  # the untimed reference (warm-up of this shape)
            return None, True
        return ms, all(torch.equal(a, b) for a, b in zip(out, self.ref[T]))


def measure(cases, steps, reps):
    """{name: (median us per step of a call, median marginal us per step, all checks passed)}; names alternated within each round."""
    for c in cases.values():
        c.run(steps); c.run(2 * steps)
    t1, t2, ok = {k: [] for k in cases}, {k: [] for k in cases}, {k: True for k in cases}
    for _ in range(reps):
        for k, c in cases.items():
            a, e1 = c.run(steps)
            b, e2 = c.run(2 * steps)
            t1[k].append(a * 1e3 / steps); t2[k].append((b - a) * 1e3 / steps)
            ok[k] &= e1 and e2
    return {k: (statistics.median(t1[k]), statistics.median(t2[k]), ok[k]) for k in cases}


def heads_tilings(E, iters, reps):
    """The frozen tensor-core heads alone (K = 364): 64- against 128-column tiles at E environments, us per forward."""
    K = 364
    x = (torch.randn(E, K, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3)) * 1.5)
    norm = frozen_normalizer(E, K)
    pols = {}
    for name, hook in (("cols64", "1"), ("cols128", "128")):
        os.environ["EVAC_POLICY_TC"] = hook  # read at evac_policy_create
        pols[name] = make_policy("flat", K)
    os.environ.pop("EVAC_POLICY_TC")
    outs = {k: dict(obs_norm=torch.empty(E, K, device="cuda"), mean=torch.empty(E, 2, device="cuda"), value=torch.empty(E, device="cuda"))
            for k in pols}

    def fwd(k):
        pols[k].forward(x, normalizer=norm, sample=False, norm_update=False, advance=False, **outs[k])
    ref = {}
    for k in pols:
        fwd(k)
        torch.cuda.synchronize()
        ref[k] = {n: t.clone() for n, t in outs[k].items()}
    times, ok = {k: [] for k in pols}, {k: True for k in pols}
    for _ in range(reps):
        for k in pols:
            ms = timed(lambda: [fwd(k) for _ in range(iters)])
            times[k].append(ms * 1e3 / iters)
            ok[k] &= all(torch.equal(outs[k][n], ref[k][n]) for n in outs[k])
    diff = max(float((ref["cols64"][n] - ref["cols128"][n]).abs().max()) for n in ("mean", "value"))
    same_obs_norm = torch.equal(ref["cols64"]["obs_norm"], ref["cols128"]["obs_norm"])
    return {k: (statistics.median(v), ok[k]) for k, v in times.items()}, diff, same_obs_norm


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--heads-iters", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("policy_eval.py measures on the GPU; no CUDA device is visible")
    os.makedirs(args.out_dir, exist_ok=True)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    with open(os.path.join(args.out_dir, "policy_eval.jsonl"), "w") as f:
        def emit(rec):
            print(json.dumps(rec), flush=True)
            f.write(json.dumps(rec) + "\n")
        emit({"gpu": q.stdout.strip() or torch.cuda.get_device_name(), "torch_name": torch.cuda.get_device_name(), "steps": args.steps,
              "reps": args.reps})
        for kind in ("tf", "flat"):
            for E in (8192, 65536):
                r = measure({kind: Case(kind, E)}, args.steps, args.reps)[kind]
                emit(dict(policy=kind, E=E, N=N, path="evaluate_policy", us_per_step=round(r[0], 2), us_per_step_marginal=round(r[1], 2),
                          equal_to_reference=r[2]))
                torch.cuda.empty_cache()
        steps_g = max(args.steps, 256)
        for E in (4096, 8192, 65536):
            cases = {"evaluate_policy": Case("grav", E), "one_launch_K256": Case("grav", E, one_launch=True)}
            r = measure(cases, steps_g, args.reps)
            same = all(torch.equal(a, b) for a, b in zip(cases["evaluate_policy"].ref[steps_g], cases["one_launch_K256"].ref[steps_g]))
            for k, v in r.items():
                emit(dict(policy="grav", E=E, N=N, path=k, us_per_step=round(v[0], 2), us_per_step_marginal=round(v[1], 2),
                          equal_to_reference=v[2], paths_bit_identical=same))
            torch.cuda.empty_cache()
        h, diff, same_on = heads_tilings(8192, args.heads_iters, args.reps)
        for k, (us, ok) in h.items():
            emit(dict(kernel="frozen tensor-core heads", K=364, E=8192, tiling=k, us_per_forward=round(us, 2), equal_to_reference=ok,
                      max_abs_diff_64_vs_128=diff, obs_norm_identical=same_on))


if __name__ == "__main__":
    main()
