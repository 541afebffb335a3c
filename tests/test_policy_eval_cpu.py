"""CPU checks of the evaluation boundary (no GPU needed): the ctypes mirror of EvacPolicyIO, `norm_frozen` included, against the
header as a C compiler lays it out, and the device-free argument validation of `evaluate_policy`."""
import ctypes as C
import os
import subprocess
import types

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_policy_io_mirror_matches_the_header_layout(tmp_path):
    from evacuation_b200 import _native as nat
    from evacuation_b200.build import find_nvcc

    names = [f for f, _ in nat.EvacPolicyIO._fields_]
    assert names[-1] == "norm_frozen"
    src = tmp_path / "layout.cpp"
    src.write_text('#include <cstdio>\n#include <cstddef>\n#include "evac_b200.h"\nint main() {\n'
                   '  printf("sizeof %zu\\n", sizeof(EvacPolicyIO));\n  printf("abi %d\\n", EVAC_ABI_VERSION);\n'
                   + "".join(f'  printf("{n} %zu\\n", offsetof(EvacPolicyIO, {n}));\n' for n in names) + "  return 0;\n}\n")
    exe = tmp_path / "layout"
    res = subprocess.run([find_nvcc(), "-x", "c++", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    got = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(got["abi"]) == nat.EVAC_ABI_VERSION == 6
    assert int(got["sizeof"]) == C.sizeof(nat.EvacPolicyIO)
    for n in names:
        assert int(got[n]) == getattr(nat.EvacPolicyIO, n).offset, n


def _fake_policy(obs_dim, A=2):
    """A stand-in that passes the fused-policy type check without a device."""
    from evacuation_b200.rollout import FusedRPOLinearPolicy

    p = FusedRPOLinearPolicy.__new__(FusedRPOLinearPolicy)
    p.obs_dim, p.A = obs_dim, A
    return p


def test_evaluation_argument_validation_without_a_device():
    from evacuation_b200.rollout import RPOLinearPolicy, VectorNormalizer, check_evaluation_args, evaluate_policy

    E, D, T = 8, 364, 5
    pol = _fake_policy(D)
    norm = VectorNormalizer(E, D, device="cpu")
    ok = dict(obs_norm=torch.empty(T, E, D), action=torch.empty(T, E, 2), status_counts=torch.empty(T, E, 4, dtype=torch.int16))
    check_evaluation_args(E, D, pol, T, norm, **ok)
    check_evaluation_args(E, D, pol, T)
    with pytest.raises(NotImplementedError):                                        # a torch module has no fused forward
        check_evaluation_args(E, D, RPOLinearPolicy(D), T)
    with pytest.raises(NotImplementedError):                                        # ... and evaluate_policy refuses it first
        evaluate_policy(types.SimpleNamespace(unwrapped=types.SimpleNamespace(num_envs=E, obs_dim=D)), RPOLinearPolicy(D), T)
    with pytest.raises(ValueError):
        check_evaluation_args(E, 6, pol, T)                                         # the policy reads another width
    with pytest.raises(ValueError):
        check_evaluation_args(E, D, _fake_policy(D, A=3), T)                         # the env takes 2 actions
    with pytest.raises(ValueError):
        check_evaluation_args(E, D, pol, 0)
    with pytest.raises(ValueError):
        check_evaluation_args(E, D, pol, T, VectorNormalizer(E + 1, D, device="cpu"))  # the normaliser holds E environments
    with pytest.raises(ValueError):
        check_evaluation_args(E, D, pol, T, VectorNormalizer(E, D, device="cpu", dtype=torch.float64))
    with pytest.raises(ValueError):
        check_evaluation_args(E, D, pol, T + 1, **ok)                               # outputs hold num_steps rows
    with pytest.raises(ValueError):
        check_evaluation_args(E, D, pol, T, status_counts=torch.empty(T, E, 4, dtype=torch.int32))
    with pytest.raises(ValueError):
        check_evaluation_args(E, D, pol, T, obs_norm=torch.empty(T, E, 6))
    with pytest.raises(ValueError):
        check_evaluation_args(E, D, pol, T, action=torch.empty(E, T, 2).transpose(0, 1))  # not contiguous


def test_one_launch_choice_is_made_from_the_handle_and_the_policy():
    from evacuation_b200.config import EnvConfig
    from evacuation_b200.rollout import FusedRPOTransformerPolicy, one_launch_evaluation_supported

    def env(N=60, precision="fp32", positions="grav"):
        return types.SimpleNamespace(unwrapped=types.SimpleNamespace(precision=precision, cfg=EnvConfig(number_of_pedestrians=N),
                                                                     _positions=positions))

    assert one_launch_evaluation_supported(env(), _fake_policy(6))
    assert one_launch_evaluation_supported(env(N=64), _fake_policy(6))
    assert not one_launch_evaluation_supported(env(N=65), _fake_policy(6))               # CTA kernel
    assert not one_launch_evaluation_supported(env(precision="fp64"), _fake_policy(6))
    assert not one_launch_evaluation_supported(env(positions="rel"), _fake_policy(6))
    assert not one_launch_evaluation_supported(env(), _fake_policy(6, A=3))
    assert not one_launch_evaluation_supported(env(), _fake_policy(364))
    tf = FusedRPOTransformerPolicy.__new__(FusedRPOTransformerPolicy)
    tf.obs_dim, tf.A = 6, 2
    assert not one_launch_evaluation_supported(env(), tf)
