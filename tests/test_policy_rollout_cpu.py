"""CPU checks of the one-launch policy rollout's boundary (no GPU needed): the ctypes mirror of EvacPolicyRolloutIO against the
header as a C compiler lays it out, and the device-free argument validation of `PolicyRollout.run(steps_per_launch=...)` and
`fused_policy_rollout`."""
import ctypes as C
import os
import subprocess

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_rollout_io_mirror_matches_the_header_layout(tmp_path):
    from evacuation_b200 import _native as nat
    from evacuation_b200.build import find_nvcc

    nvcc = find_nvcc()
    names = [f for f, _ in nat.EvacPolicyRolloutIO._fields_]
    src = tmp_path / "layout.cpp"
    src.write_text('#include <cstdio>\n#include <cstddef>\n#include "evac_b200.h"\nint main() {\n'
                   '  printf("sizeof %zu\\n", sizeof(EvacPolicyRolloutIO));\n'
                   + "".join(f'  printf("{n} %zu\\n", offsetof(EvacPolicyRolloutIO, {n}));\n' for n in names) + "  return 0;\n}\n")
    exe = tmp_path / "layout"
    res = subprocess.run([nvcc, "-x", "c++", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    got = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(got["sizeof"]) == C.sizeof(nat.EvacPolicyRolloutIO)
    for n in names:
        assert int(got[n]) == getattr(nat.EvacPolicyRolloutIO, n).offset, n
    assert "evac_rollout_policy" in nat.SIGNATURES


def test_launch_sizes():
    from evacuation_b200.rollout import policy_launch_sizes

    assert policy_launch_sizes(131, 64) == [64, 64, 3]
    assert policy_launch_sizes(128, 64) == [64, 64]
    assert policy_launch_sizes(5, 7) == [5]
    assert policy_launch_sizes(3, 1) == [1, 1, 1]
    for n, k in ((0, 4), (-1, 4), (5, 0)):
        with pytest.raises(ValueError):
            policy_launch_sizes(n, k)


def test_tensor_validation_without_a_device():
    from evacuation_b200.rollout import VectorNormalizer, check_policy_rollout_tensors

    E, T = 8, 5
    norm = VectorNormalizer(E, 6, device="cpu")
    nd = torch.zeros(E)
    check_policy_rollout_tensors(E, 6, norm, nd, obs_norm=torch.empty(T, E, 6), action=torch.empty(T, E, 2), value=torch.empty(T, E),
                                 status_counts=torch.empty(T, E, 4, dtype=torch.int16))
    with pytest.raises(ValueError):
        check_policy_rollout_tensors(E + 1, 6, norm, torch.zeros(E + 1))                   # the normaliser holds E environments
    with pytest.raises(ValueError):
        check_policy_rollout_tensors(E, 6, VectorNormalizer(E, 6, device="cpu", dtype=torch.float64), nd)
    with pytest.raises(ValueError):
        check_policy_rollout_tensors(E, 6, norm, torch.zeros(E, dtype=torch.float64))     # next_done is float32
    with pytest.raises(ValueError):
        check_policy_rollout_tensors(E, 6, norm, nd, action=torch.empty(T, E, 3))
    with pytest.raises(ValueError):
        check_policy_rollout_tensors(E, 6, norm, nd, status_counts=torch.empty(T, E, 4, dtype=torch.int32))
    with pytest.raises(ValueError):
        check_policy_rollout_tensors(E, 6, norm, nd, obs_norm=torch.empty(E, T, 6).transpose(0, 1))  # not contiguous
    n2 = VectorNormalizer(E, 6, device="cpu")
    n2.obs_count = torch.full((), 1e-4, dtype=torch.float32)
    with pytest.raises(ValueError):
        check_policy_rollout_tensors(E, 6, n2, nd)                                         # the counts are float64 scalars
