"""Standalone pairwise pass in the mappings of evac_probe_pairwise: EVAC_PROBE_HALFWARP unset = 32 lanes x 2 pedestrians (the fused
step's), 2 = 16 x 4, 8 = 8 x 8.  Prints one JSON line: TFLOP/s (8 flop per ordered pair) and fraction of the FFMA2 peak
measured in the same process.  Usage: [EVAC_PROBE_HALFWARP=2|8] python tools/probe_pairwise_shapes.py"""
import ctypes as C, json, os, sys
sys.path.insert(0, os.getcwd())
from evacuation_b200 import _native as nat
lib = nat.load()
ms, fl, pairs = C.c_float(), C.c_double(), C.c_double()
best = 0.0
for _ in range(3):
    nat.check(lib.evac_probe_fma(0, 1, 20000, C.byref(ms), C.byref(fl)))
    best = max(best, fl.value / (ms.value * 1e-3) / 1e12)
out = {"variant": os.environ.get("EVAC_PROBE_HALFWARP", "warp"), "ffma2_peak": round(best, 2)}
for (E, n, reps) in ((4096, 60, 200), (65536, 60, 50), (65536, 64, 50)):
    b = 0.0
    for _ in range(3):
        nat.check(lib.evac_probe_pairwise(0, E, n, reps, C.byref(ms), C.byref(pairs)))
        b = max(b, pairs.value / (ms.value * 1e-3))
    out[f"E{E}_N{n}_tflops"] = round(b * 8 / 1e12, 2)
    out[f"E{E}_N{n}_frac"] = round(b * 8 / 1e12 / best, 4)
print(json.dumps(out))
