"""Per-step timing in the bench's regime (R independent C2 batches stepped round-robin in one CUDA graph, inputs larger than
L2) for the library selected by EVAC_B200_LIB (default: the in-tree build) -- compares two builds in one process per build.
Usage: python tools/step_bench.py [E] [K] [R] [mode]   (mode: rel_ohe_box | grav)"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import evacuation_b200 as eb

E = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
K = int(sys.argv[2]) if len(sys.argv) > 2 else 960
R = int(sys.argv[3]) if len(sys.argv) > 3 else 24
mode = sys.argv[4] if len(sys.argv) > 4 else "rel_ohe_box"
wrap = dict(positions="rel", statuses="ohe", type="Box") if mode == "rel_ohe_box" else dict(positions="grav", alpha=3)
kw = dict(number_of_pedestrians=60, enslaving_degree=1.0, noise_coef=0.2, is_new_exiting_reward=True, is_new_followers_reward=True)
dev = torch.device("cuda", 0)
sets = []
acts = torch.rand((8 + K, E, 2), device=dev) * 2 - 1
for r in range(R):
    env = eb.setup_env(eb.EnvConfig(**kw), eb.EnvWrappersConfig(**wrap), num_envs=E, device=dev, seed=r, auto_reset=True)
    env.reset()
    for s in range(8):
        env.step(acts[s])
    sets.append(env)
out = {"lib": os.path.basename(os.environ.get("EVAC_B200_LIB", "libevac_b200.so")), "E": E, "K": K, "R": R, "mode": mode}
for label, k in (("graph", K), ("graph_k20", 20)):
    g, side = torch.cuda.CUDAGraph(), torch.cuda.Stream(device=dev)
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            for s in range(k):
                sets[s % R].unwrapped.step(acts[8 + s])
    torch.cuda.synchronize()
    g.replay()
    torch.cuda.synchronize()
    best = []
    for rep in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda._sleep(int(2e-3 * 1.9e9))
        e0.record(); g.replay(); e1.record()
        torch.cuda.synchronize()
        best.append(1e3 * e0.elapsed_time(e1) / k)
    out[label + "_us"] = [round(x, 3) for x in best]
# K steps in one launch (state on chip)
sets[0].rollout(8, agent="random")
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
torch.cuda.synchronize(); e0.record(); sets[0].rollout(400, agent="random"); e1.record(); torch.cuda.synchronize()
out["rollout_us"] = round(1e3 * e0.elapsed_time(e1) / 400, 3)
print(json.dumps(out))
