"""Fused policy forwards (embedding kernel + tensor-core heads) for compute-sanitizer, one per column tiling of the heads: E
environments (64-column tiles) and 38000 (128-column tiles, chosen from 296 row tiles of 128 environments up).
Usage: python tools/san_policy.py [E]"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from evacuation_b200.rollout import FusedRPOTransformerPolicy, RPOTransformerPolicy

small = int(sys.argv[1]) if len(sys.argv) > 1 else 300
torch.manual_seed(0)
net = RPOTransformerPolicy(372, 60).cuda().eval()
for E in (small, 38000):
    x = torch.randn(E, 372, device="cuda").clamp_(-1, 1)
    fused = FusedRPOTransformerPolicy(net, 60, device="cuda", max_envs=E).eval()
    mean, val, act, lp = (torch.empty(s, device="cuda") for s in ((E, 2), (E,), (E, 2), (E,)))
    fused.forward(x, mean=mean, value=val, action=act, logprob=lp)
    torch.cuda.synchronize()
    with torch.no_grad():
        ref = net.actor_mean(net.embed(x))
    print(E, "envs: max |mean - torch| =", float((mean - ref).abs().max()))
