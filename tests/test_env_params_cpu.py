"""Field validation and broadcasting of EvacuationEnv.set_env_params (merge_env_params), without a device; and the Python
record matching the C struct of include/evac_b200.h."""
import ctypes
import os
import re

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from evacuation_b200 import _native as nat  # noqa: E402
from evacuation_b200.env import ENV_PARAM_FIELDS, merge_env_params  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
E = 5


def _current():
    return {k: np.full(E, 2000 if k == "max_timesteps" else (1 if k.startswith("is_") else 0.25)) for k in ENV_PARAM_FIELDS}


def test_fields_are_the_c_record():
    header = open(os.path.join(ROOT, "include", "evac_b200.h")).read()
    body = re.search(r"typedef struct EvacEnvParams \{(.*?)\} EvacEnvParams;", header, re.S).group(1)
    declared = re.findall(r"(double|int32_t)\s+(\w+);", body)
    assert [n for _, n in declared] == list(ENV_PARAM_FIELDS)
    assert [t for t, _ in declared] == ["double" if f[1] == ctypes.c_double else "int32_t" for f in nat.EvacEnvParams._fields_]
    assert ctypes.sizeof(nat.EvacEnvParams) == 56


def test_scalars_broadcast_and_sequences_of_every_kind_are_taken():
    cur = _current()
    out = merge_env_params(cur, E, dict(noise_coef=0.5, enslaving_degree=[0.1, 0.2, 0.3, 0.4, 0.5],
                                        alpha=np.arange(E, dtype=np.float32) + 2.5, intrinsic_reward_coef=torch.linspace(0, 1, E),
                                        is_new_exiting_reward=[True, False, True, False, True], max_timesteps=np.int64(17)))
    assert out["noise_coef"].tolist() == [0.5] * E
    assert out["enslaving_degree"].tolist() == [0.1, 0.2, 0.3, 0.4, 0.5]
    assert out["alpha"].tolist() == [2.5, 3.5, 4.5, 5.5, 6.5]
    assert np.allclose(out["intrinsic_reward_coef"], np.linspace(0, 1, E))
    assert out["is_new_exiting_reward"].tolist() == [1, 0, 1, 0, 1] and out["max_timesteps"].tolist() == [17] * E
    assert out["max_timesteps"].dtype == np.int32 and out["noise_coef"].dtype == np.float64


def test_unnamed_fields_keep_their_values_and_the_input_is_not_modified():
    cur = _current()
    cur["noise_coef"] = np.linspace(0.05, 0.8, E)
    keep = {k: v.copy() for k, v in cur.items()}
    out = merge_env_params(cur, E, dict(enslaving_degree=0.5))
    assert out["noise_coef"].tolist() == keep["noise_coef"].tolist()
    assert all(np.array_equal(cur[k], keep[k]) for k in cur)
    assert all(np.array_equal(out[k], cur[k]) for k in cur if k != "enslaving_degree")


@pytest.mark.parametrize("fields", [dict(width=2.0), dict(height=1.0), dict(step_size=0.02), dict(to_pedestrian=0.2), dict(eps=1e-6),
                                    dict(to_leader=0.3), dict(number_of_pedestrians=5), dict(positions="rel"), dict(noise=0.1),
                                    dict(noise_coef=[0.1] * (E - 1)), dict(noise_coef=np.zeros((E, 1))), dict(alpha=np.zeros((1, E))),
                                    dict(max_timesteps=2.5), dict(is_new_exiting_reward=[0.5] * E), dict(max_timesteps=2**40)])
def test_refused(fields):
    with pytest.raises(ValueError):
        merge_env_params(_current(), E, fields)
