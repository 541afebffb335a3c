"""Latency of the reference-shaped single environment through the drop-in API (`setup_env(EnvConfig(60), wrap).step(a)`, NumPy in /
NumPy out, rng="numpy"): microseconds per step for the three wrapper sets of BASELINE.md section 3 item 1.
Usage: python tools/single_env_latency.py"""
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import evacuation_b200 as eb

out = {}
for name, wrap in (("abs_no_dict", {}), ("rel_ohe_box", dict(positions="rel", statuses="ohe", type="Box")), ("grav_alpha3", dict(positions="grav", alpha=3))):
    env = eb.setup_env(eb.EnvConfig(number_of_pedestrians=60, wandb_enabled=False), eb.EnvWrappersConfig(**wrap), device="cuda:0")
    np.random.seed(0)
    acts = np.random.RandomState(1).uniform(-1, 1, size=(3000, 2)).astype(np.float32)
    env.reset()
    for t in range(50):
        env.step(acts[t])
    np.random.seed(0)
    env.reset()
    t0 = time.perf_counter()
    n = 0
    for t in range(2000):
        _, _, term, trunc, _ = env.step(acts[t])
        n += 1
        if term or trunc:
            env.reset()
    out[name + "_us_per_step"] = round(1e6 * (time.perf_counter() - t0) / n, 2)
    env.unwrapped.close()
print(json.dumps(out))
