"""EvacuationEnv -- host-side mirror of the reference's gymnasium environment
(src/env/env/env.py:34-171) whose reset/step run as ONE fused CUDA kernel over a batch of
independent environments (csrc/evac_kernels.cuh behind the C ABI of include/evac_b200.h).

Two faces, one code path:

* ``num_envs == 1`` (default): reference-shaped values -- ``reset() -> (obs, {})`` and
  ``step(action) -> (obs, reward: float, terminated: bool, truncated: bool, {})`` with NumPy
  observations (Dict or Box as selected by the wrappers), through the host-buffer entry
  point ``evac_step_host``.  With ``rng="numpy"`` (the default for this face) the reset layout
  and the per-step noise are drawn from the GLOBAL ``np.random`` stream in exactly the
  order the reference consumes it (pedestrians.py:17-18, area.py:124), so
  ``np.random.seed(s); env.reset(); env.step(a) ...`` retraces the reference's trajectory.
* ``num_envs > 1``: batched torch CUDA tensors in and out, counter-based (Philox) random
  streams inside the kernel, optional same-step auto-reset.

There is no CPU fallback: constructing the environment without the CUDA library or without
a GPU raises.
"""
from __future__ import annotations

import ctypes as C
import logging
import os
from typing import Optional

import numpy as np
import torch

from . import _native as nat
from .config import EnvConfig
from .spaces import Box, Dict
from .statuses import Status, SwitchDistances

log = logging.getLogger(__name__)

_TORCH_STATE_DTYPE = {"fp32": torch.float32, "fp64": torch.float64}


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


# Per-environment dynamics and reward parameters (EvacuationEnv.set_env_params; EvacEnvParams in include/evac_b200.h):
# the EnvConfig / EnvWrappersConfig fields that enter one environment's own arithmetic.
ENV_PARAM_FIELDS = tuple(name for name, _ in nat.EvacEnvParams._fields_)
_ENV_PARAM_DTYPE = np.dtype(nat.EvacEnvParams)  # the C record, field for field
# fields that stay uniform over a batch, and why
_ENV_PARAM_EXCLUDED = {
    **dict.fromkeys(("width", "height", "to_pedestrian"), "it sizes the neighbour-search grid"),
    **dict.fromkeys(("to_leader", "step_size"), "it places the WacuumCleaner's lanes"),
    **dict.fromkeys(("eps", "to_exit", "to_escape"), "the reference's parameter sweeps do not vary it"),
    **dict.fromkeys(("number_of_pedestrians", "positions", "statuses", "type"), "it is a shape"),
}


def merge_env_params(current: dict, num_envs: int, fields: dict) -> dict:
    """`current` (field -> [E] array, every field of ENV_PARAM_FIELDS) updated with `fields`: each value is a scalar
    (broadcast to every environment) or a length-E sequence, NumPy array or tensor.  Returns new [E] arrays (float64 for the
    reals, int32 for the flags and max_timesteps).  ValueError for an unknown or excluded field name, a wrong length or a
    non-integer value of an integer field.  The value ranges are checked by the library (evac_set_env_params)."""
    out = {k: np.array(current[k], dtype=_ENV_PARAM_DTYPE[k], copy=True) for k in ENV_PARAM_FIELDS}
    for name, value in fields.items():
        if name in _ENV_PARAM_EXCLUDED:
            raise ValueError(f"`{name}` cannot be set per environment: {_ENV_PARAM_EXCLUDED[name]}")
        if name not in out:
            raise ValueError(f"unknown per-environment parameter `{name}`; the fields are {', '.join(ENV_PARAM_FIELDS)}")
        v = np.asarray(value.detach().cpu().numpy() if torch.is_tensor(value) else value)
        if v.ndim != 0 and v.shape != (num_envs,):
            raise ValueError(f"`{name}`: expected a scalar or {num_envs} values, got shape {v.shape}")
        dt = _ENV_PARAM_DTYPE[name]
        if dt.kind == "i":
            vf = v.astype(np.float64)
            if not np.all(np.isfinite(vf) & (vf == np.round(vf)) & (np.abs(vf) < 2**31)):
                raise ValueError(f"`{name}` takes integer values")
        out[name][...] = v.astype(dt)
    return out


class _Pedestrians:
    """`env.unwrapped.pedestrians` (src/env/env/pedestrians.py): live views of the device state."""

    def __init__(self, env: "EvacuationEnv"):
        self._env = env
        self.num = env.cfg.number_of_pedestrians
        self.memory = {"positions": [], "statuses": []}  # pedestrians.py:14 (trajectory of the tracked environment)

    def save(self):
        """pedestrians.py:33-35: append the tracked environment's positions / statuses (host copies)."""
        st = self._env.get_state()
        e = self._env.tracked_env
        self.memory["positions"].append(st["positions"][e].cpu().numpy().astype(np.float64))
        self.memory["statuses"].append(st["statuses"][e].cpu().numpy())

    def _fetch(self, key):
        v = self._env.get_state()[key]
        if not self._env.batched:
            v = v[0].cpu().numpy()
        return v

    @property
    def positions(self):
        return self._fetch("positions")

    @property
    def directions(self):
        return self._fetch("directions")

    @property
    def statuses(self):
        """uint8 codes with the reference's enum values (Status.X.value)."""
        env = self._env
        if not env.batched and env._host_statuses is not None:  # came back with the last step's result block
            return np.array(env._host_statuses[0], dtype=np.uint8)
        return self._fetch("statuses")

    @property
    def status_stats(self):  # pedestrians.py:37-44
        env = self._env
        if not env.batched and env._host_statuses is not None:
            h = env._host_statuses[0]
            return {k: int(np.count_nonzero(h == v)) for k, v in (("escaped", 4), ("exiting", 3), ("following", 2), ("viscek", 1))}
        s = self._env.get_state()["statuses"]
        out = {k: (s == v).sum(dim=1) for k, v in
               (("escaped", 4), ("exiting", 3), ("following", 2), ("viscek", 1))}
        if not self._env.batched:
            out = {k: int(v[0]) for k, v in out.items()}
        return out


class _Agent:
    def __init__(self, env: "EvacuationEnv"):
        self._env = env
        self.enslaving_degree = env.cfg.enslaving_degree
        self.start_position = np.zeros(2, dtype=np.float32)
        self.start_direction = np.zeros(2, dtype=np.float32)
        self.memory = {"position": []}  # area.py:24

    def save(self):  # area.py:32-33
        self.memory["position"].append(self._env.get_state()["agent_position"][self._env.tracked_env].cpu().numpy().copy())

    @property
    def position(self):
        v = self._env.get_state()["agent_position"]
        return v if self._env.batched else v[0].cpu().numpy()

    @property
    def direction(self):
        v = self._env.get_state()["agent_direction"]
        return v if self._env.batched else v[0].cpu().numpy()


class _Exit:
    def __init__(self):
        self.position = np.array([0, -1], dtype=np.float32)  # area.py:36-39


class _Area:
    def __init__(self, cfg: EnvConfig):
        self.width, self.height = cfg.width, cfg.height
        self.step_size, self.noise_coef, self.eps = cfg.step_size, cfg.noise_coef, cfg.eps
        self.exit = _Exit()


class _Time:
    def __init__(self, env: "EvacuationEnv"):
        self._env = env
        self.max_timesteps = env.cfg.max_timesteps
        self.n_episodes = 0  # resets seen by this Python object (area.py:49-51)

    @property
    def overall_timesteps(self):
        v = self._env.accumulators()[1]
        return v if self._env.batched else int(v[0])

    @property
    def now(self):
        v = self._env.get_state()["now"]
        return v if self._env.batched else int(v[0])


class EvacuationEnv:
    """Evacuation environment, batched on one B200.  Continuous action and observation space."""

    metadata = {"render_modes": ["human", "rgb_array"], "render_fps": 4}

    def __init__(self, cfg: EnvConfig, num_envs: int = 1, device=None, seed: int = 0,
                 auto_reset: Optional[bool] = None, precision: str = "fp32", env_index_offset: int = 0,
                 rng: Optional[str] = None, batched: Optional[bool] = None, neighbor_search: str = "auto"):
        if isinstance(cfg, type):  # README.md:72 passes the class itself
            cfg = cfg()
        if precision not in nat.PREC:
            raise ValueError(f"Invalid value of `precision`='{precision}'. Must be 'fp32' or 'fp64'.")
        self.cfg = cfg
        self.num_envs = int(num_envs)
        self.batched = (self.num_envs > 1) if batched is None else bool(batched)
        self.rng = rng if rng is not None else ("philox" if self.batched else "numpy")
        if self.rng not in ("numpy", "philox"):
            raise ValueError(f"Invalid value of `rng`='{self.rng}'. Must be 'numpy' or 'philox'.")
        self.auto_reset = self.batched if auto_reset is None else bool(auto_reset)
        self.precision = precision
        if neighbor_search not in nat.SEARCH:
            raise ValueError(f"Invalid value of `neighbor_search`='{neighbor_search}'. Must be 'auto', 'brute' or 'cells'.")
        self.neighbor_search = neighbor_search
        self.seed_value = int(seed)
        self.env_index_offset = int(env_index_offset)
        nat.load()  # fail loudly now if the CUDA library is missing
        if not torch.cuda.is_available():
            raise nat.EvacNativeError("no CUDA device available: evacuation_b200 has no CPU fallback")
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        if self.device.type != "cuda":
            raise ValueError("evacuation_b200 runs on CUDA devices only")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())

        # fused observation pipeline, switched by the wrappers
        self._positions, self._statuses, self._obs_type, self._alpha = "abs", "no", "Dict", 3.0
        self._h = None
        self._host_statuses = None  # numpy-rng face: statuses after the last step (for the |fv| draw)
        # per-environment parameters (set_env_params): [E] arrays of every field, or None (uniform: the construction config);
        # _env_params_mode counts the switches between the two, which select different kernel instances (PolicyRollout
        # re-captures its graph after one)
        self._env_params = None
        self._env_params_mode = 0

        n = cfg.number_of_pedestrians
        self.pedestrians = _Pedestrians(self)
        self.agent = _Agent(self)
        self.area = _Area(cfg)
        self.time = _Time(self)
        self.intrinsic_reward_coef = cfg.intrinsic_reward_coef
        self.action_space = Box(low=-1.0, high=1.0, shape=(2,), dtype=np.float32)  # env.py:69
        self.observation_space = Dict({  # env.py:86-96
            "agent_position": Box(low=-1, high=1, shape=(2,), dtype=np.float32),
            "pedestrians_positions": Box(low=-1, high=1, shape=(n, 2), dtype=np.float32),
            "exit_position": Box(low=-1, high=1, shape=(2,), dtype=np.float32),
        })
        self.render_mode = cfg.render_mode
        self.experiment_name = cfg.experiment_name
        # ---- logging / trajectory capture (env.py:23-31,45-64): host-side, off the per-step device path
        self.draw = bool(cfg.draw)
        self.giff_freq = cfg.giff_freq
        self.save_next_episode_anim = False
        self.wandb_enabled = bool(cfg.wandb_enabled)
        self.path_giff, self.path_png = cfg.path_giff, cfg.path_png
        self.tracked_env = 0  # index of the environment whose trajectory `draw` records
        self._file_logging = False

    # ------------------------------------------------------------------ plumbing
    @property
    def unwrapped(self):
        return self

    def _stream(self):
        # every library call on torch's current stream goes through here: the host face (evac_step_host, its own non-blocking
        # stream) must wait for that work once before its next step
        self._host_sync_needed = True
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _configure_obs(self, **kw):
        """Called by the wrappers: switch on an encoding inside the fused kernel."""
        state = self.get_state() if self._h is not None else None
        for k, v in kw.items():
            setattr(self, "_" + k, v)
        if "alpha" in kw and self._env_params is not None:  # a wrapper's alpha applies to every environment
            self._env_params["alpha"][:] = float(kw["alpha"])
        if self._h is not None:
            self.close()
            self._handle()
            self.set_state(**state)

    def _handle(self):
        if self._h is not None:
            return self._h
        lib = nat.load()
        c = nat.EvacConfig()
        nat.check(lib.evac_default_config(C.byref(c)))
        cfg = self.cfg
        c.number_of_pedestrians = cfg.number_of_pedestrians
        c.width, c.height, c.step_size = cfg.width, cfg.height, cfg.step_size
        c.noise_coef, c.eps, c.enslaving_degree = cfg.noise_coef, cfg.eps, cfg.enslaving_degree
        c.is_new_exiting_reward = int(cfg.is_new_exiting_reward)
        c.is_new_followers_reward = int(cfg.is_new_followers_reward)
        c.intrinsic_reward_coef = cfg.intrinsic_reward_coef
        c.is_termination_agent_wall_collision = int(cfg.is_termination_agent_wall_collision)
        c.init_reward_each_step = cfg.init_reward_each_step
        c.max_timesteps = cfg.max_timesteps
        if self._positions not in nat.POS or self._statuses not in nat.STAT or self._obs_type not in nat.OBS:
            raise ValueError(f"invalid observation mode {self._positions}/{self._statuses}/{self._obs_type}")
        c.positions, c.statuses, c.obs_type = nat.POS[self._positions], nat.STAT[self._statuses], nat.OBS[self._obs_type]
        c.alpha = float(self._alpha)
        c.to_leader, c.to_pedestrian = SwitchDistances.to_leader, SwitchDistances.to_pedestrian
        c.to_exit, c.to_escape = SwitchDistances.to_exit, SwitchDistances.to_escape
        c.auto_reset = int(self.auto_reset)
        c.precision = nat.PREC[self.precision]
        c.neighbor_search = nat.SEARCH[self.neighbor_search]
        h = C.c_void_p()
        nat.check(lib.evac_create(C.byref(c), self.num_envs, self.device.index, C.c_uint64(self.seed_value),
                                  C.c_int64(self.env_index_offset), C.byref(h)))
        self._h = h
        if self._env_params is not None:  # a re-created handle (observation wrappers, reset(seed=...)) keeps them
            self._upload_env_params(self._env_params)
        self._obs_dim = lib.evac_obs_dim(h)
        E, dev = self.num_envs, self.device
        self._obs = torch.empty((E, self._obs_dim), dtype=torch.float32, device=dev)
        self._reward = torch.empty(E, dtype=torch.float32, device=dev)
        self._terminated = torch.empty(E, dtype=torch.uint8, device=dev)
        self._truncated = torch.empty(E, dtype=torch.uint8, device=dev)
        # zero-copy bool views of the flag bytes and the structured view of the observation rows
        self._terminated_b, self._truncated_b = self._terminated.view(torch.bool), self._truncated.view(torch.bool)
        self._obs_view = self._structure(self._obs)
        # page-locked host buffers of the single-env / host face (evac_step_host copies straight into them)
        self._host = None
        return h

    def close(self):
        if self._h is not None:
            torch.cuda.synchronize(self.device)
            nat.load().evac_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def obs_dim(self) -> int:
        """Floats per environment in one flat observation row."""
        self._handle()
        return self._obs_dim

    @property
    def flat_observation(self) -> torch.Tensor:
        """The [E, obs_dim] float32 device buffer the kernel writes: gymnasium `FlattenObservation` of the wrapped
        observation (Dict keys in sorted order / Box rows row-major), valid after reset() and after every batched step()."""
        self._handle()
        return self._obs

    @property
    def num_cells(self) -> int:
        """Cells of the neighbour-search grid the handle is pinned to (0 = all-pairs tiles).  N <= 64 under
        neighbor_search="auto" also reports 0: every warp chooses per step between the all-pairs loop and the cell masks
        of the sparse pass; "cells" pins it to the sparse pass (whenever exact), "brute" to the all-pairs loop."""
        return int(nat.load().evac_num_cells(self._handle()))

    @property
    def launch_count(self) -> int:
        return int(nat.load().evac_launch_count(self._handle()))

    # ------------------------------------------------------------------ state access
    def get_state(self) -> dict:
        """Copy of the full simulation state as torch tensors on the env's device."""
        h, lib = self._handle(), nat.load()
        E, N, dev = self.num_envs, self.cfg.number_of_pedestrians, self.device
        dt = _TORCH_STATE_DTYPE[self.precision]
        st = dict(positions=torch.empty((E, N, 2), dtype=dt, device=dev),
                  directions=torch.empty((E, N, 2), dtype=dt, device=dev),
                  statuses=torch.empty((E, N), dtype=torch.uint8, device=dev),
                  agent_position=torch.empty((E, 2), dtype=torch.float32, device=dev),
                  agent_direction=torch.empty((E, 2), dtype=torch.float32, device=dev),
                  now=torch.empty(E, dtype=torch.int32, device=dev))
        nat.check(lib.evac_get_state(h, _ptr(st["positions"]), _ptr(st["directions"]), _ptr(st["statuses"]),
                                     _ptr(st["agent_position"]), _ptr(st["agent_direction"]), _ptr(st["now"]),
                                     self._stream()))
        return st

    def set_state(self, positions=None, directions=None, statuses=None, agent_position=None,
                  agent_direction=None, now=None):
        """Overwrite (parts of) the state.  statuses=None with new positions => recomputed from the
        positions like pedestrians.py:21-26."""
        h, lib = self._handle(), nat.load()
        E, N, dev = self.num_envs, self.cfg.number_of_pedestrians, self.device
        dt = _TORCH_STATE_DTYPE[self.precision]

        def prep(x, shape, dtype):
            if x is None:
                return None
            t = torch.as_tensor(np.asarray(x) if not torch.is_tensor(x) else x)
            return t.to(device=dev, dtype=dtype).reshape(shape).contiguous()

        p, d = prep(positions, (E, N, 2), dt), prep(directions, (E, N, 2), dt)
        s = prep(statuses, (E, N), torch.uint8)
        ap, ad = prep(agent_position, (E, 2), torch.float32), prep(agent_direction, (E, 2), torch.float32)
        nw = prep(now, (E,), torch.int32)
        nat.check(lib.evac_set_state(h, _ptr(p), _ptr(d), _ptr(s), _ptr(ap), _ptr(ad), _ptr(nw), self._stream()))
        self._host_statuses = None

    def save_state(self) -> torch.Tensor:
        """Checkpoint: the complete device state of the batch (pedestrians, agent, time, episode indices, accumulators,
        scripted-agent state, finished-episode statistics) as one uint8 tensor on the env's device.  `load_state(image)` on
        an env created with the same configuration / num_envs / seed resumes bit-identically (Philox streams are
        counter-based); `torch.save(image.cpu(), path)` makes it a file."""
        h, lib = self._handle(), nat.load()
        image = torch.empty(int(lib.evac_state_bytes(h)), dtype=torch.uint8, device=self.device)
        nat.check(lib.evac_save_state(h, _ptr(image), self._stream()))
        return image

    def load_state(self, image: torch.Tensor) -> None:
        h, lib = self._handle(), nat.load()
        image = torch.as_tensor(image).to(device=self.device, dtype=torch.uint8).contiguous()
        if image.numel() != int(lib.evac_state_bytes(h)):
            raise ValueError(f"state image has {image.numel()} bytes, this environment needs {int(lib.evac_state_bytes(h))}")
        nat.check(lib.evac_load_state(h, _ptr(image), self._stream()))
        self._host_statuses = None

    def set_env_params(self, *uniform, **fields):
        """Per-environment dynamics and reward parameters: one batch runs a whole parameter grid, or a policy trains over a
        range of them (domain randomisation).  `fields` are EnvConfig / EnvWrappersConfig names (ENV_PARAM_FIELDS: noise_coef,
        enslaving_degree, alpha, intrinsic_reward_coef, init_reward_each_step, is_new_exiting_reward, is_new_followers_reward,
        is_termination_agent_wall_collision, max_timesteps); each value is a scalar or a length-E sequence / array / tensor.
        Fields not named keep their current per-environment values.  `set_env_params(None)` returns to the construction
        config.  Stream-ordered like step(): steps already enqueued use the old values.  Environment e then computes, bit for
        bit, what environment e of an env constructed with e's values (same num_envs, seed, env_index_offset) computes.
        The parameters are configuration: save_state() / load_state() do not carry them.  An observation wrapper applied
        afterwards that sets alpha (GravityEncoding(alpha=...)) sets it for every environment."""
        if uniform:
            if len(uniform) != 1 or uniform[0] is not None or fields:
                raise TypeError("set_env_params takes keyword fields, or the single positional argument None")
            params = None
        else:
            params = merge_env_params(self.env_params(), self.num_envs, fields)
        self._handle()
        self._upload_env_params(params)
        if (params is None) != (self._env_params is None):
            self._env_params_mode += 1
        self._env_params = params

    def _upload_env_params(self, params):
        rec = None
        if params is not None:
            rec = np.zeros(self.num_envs, dtype=_ENV_PARAM_DTYPE)
            for k in ENV_PARAM_FIELDS:
                rec[k] = params[k]
        nat.check(nat.load().evac_set_env_params(self._h, None if rec is None else C.c_void_p(rec.ctypes.data), self._stream()))

    def env_params(self) -> dict:
        """field -> [E] NumPy array of the per-environment parameters (the construction config's values when uniform)."""
        rec = np.zeros(self.num_envs, dtype=_ENV_PARAM_DTYPE)
        nat.check(nat.load().evac_get_env_params(self._handle(), C.c_void_p(rec.ctypes.data)))
        return {k: rec[k].copy() for k in ENV_PARAM_FIELDS}

    def accumulators(self):
        """(acc [E,3] float64: episode_reward, episode_intrinsic_reward, episode_status_reward; overall_timesteps [E] int64)
        of the running episodes (env.py:65-67,168-170)."""
        h, lib = self._handle(), nat.load()
        acc = torch.empty((self.num_envs, 3), dtype=torch.float64, device=self.device)
        overall = torch.empty(self.num_envs, dtype=torch.int64, device=self.device)
        nat.check(lib.evac_get_accumulators(h, _ptr(acc), _ptr(overall), self._stream()))
        return acc, overall

    # ------------------------------------------------------------------ logging (env.py:23-31,114-127)
    def _setup_logging(self):
        if self._file_logging:
            return
        os.makedirs(self.cfg.path_logs, exist_ok=True)
        handler = logging.FileHandler(os.path.join(self.cfg.path_logs, f"logs_{self.experiment_name}.log"), mode="w")
        handler.setFormatter(logging.Formatter("%(asctime)s - %(name)s - %(levelname)s - %(message)s"))
        log.addHandler(handler)
        log.setLevel(logging.DEBUG if self.cfg.verbose else logging.INFO)
        self._file_logging = True

    def episode_log(self, env_index: int = 0) -> dict:
        """The per-episode logging dict of env.py:115-125 for the RUNNING episode of one environment."""
        acc, overall = self.accumulators()
        st = self.get_state()
        s = st["statuses"][env_index]
        return {
            "episode_intrinsic_reward": float(acc[env_index, 1]), "episode_status_reward": float(acc[env_index, 2]),
            "episode_reward": float(acc[env_index, 0]), "episode_length": int(st["now"][env_index]),
            "escaped_pedestrians": int((s == 4).sum()), "exiting_pedestrians": int((s == 3).sum()),
            "following_pedestrians": int((s == 2).sum()), "viscek_pedestrians": int((s == 1).sum()),
            "overall_timesteps": int(overall[env_index]),
        }

    def _log_finished_episode(self):
        """What the reference does at the top of reset() (env.py:114-127): log the episode that just ended."""
        d = self.episode_log(self.tracked_env)
        self._setup_logging()
        log.info("\t".join(f"{k}={v}" for k, v in d.items()))
        if self.wandb_enabled:
            try:
                import wandb

                if wandb.run is not None:
                    wandb.log(d)
            except ImportError:
                pass
        return d

    # ------------------------------------------------------------------ observation structure
    def _structure(self, flat):
        """flat: torch [E,D] (batched face) or numpy [D] (single-env face) -> Dict / Box observation."""
        N = self.cfg.number_of_pedestrians
        lead = flat.shape[:-1]
        if self._positions == "grav":  # gravity_encoding.py:52-57
            return {"agent_position": flat[..., 0:2], "grad_potential_exit": flat[..., 2:4],
                    "grad_potential_pedestrians": flat[..., 4:6]}
        sc = {"no": 0, "ohe": 4, "cat": 1}[self._statuses]
        if self._obs_type == "Box":
            return flat.reshape(*lead, N + 2, 2 + sc)
        obs = {"agent_position": flat[..., 0:2], "exit_position": flat[..., 2:4],
               "pedestrians_positions": flat[..., 4:4 + 2 * N].reshape(*lead, N, 2)}
        if sc == 4:
            obs["pedestrians_statuses"] = flat[..., 4 + 2 * N:].reshape(*lead, N, 4)
        elif sc == 1:
            obs["pedestrians_statuses"] = flat[..., 4 + 2 * N:]
        return obs

    def _emit_obs(self):
        if self.batched:
            return self._obs_view
        o = self._obs.cpu().numpy()
        return self._structure(o[0] if self.num_envs == 1 else o)

    # ------------------------------------------------------------------ gymnasium API
    def reset(self, seed=None, options=None):
        """env.py:106-139.  `seed` re-keys the Philox streams (rng="philox"); like in the reference
        it does NOT touch the global NumPy stream that rng="numpy" draws from."""
        lib = nat.load()
        if self.save_next_episode_anim or (self.time.n_episodes + 1) % self.giff_freq == 0:  # env.py:110-112
            self.draw = True
            self.save_next_episode_anim = True
        if self.time.n_episodes > 0 and self._h is not None and not self.batched:
            self.last_episode_log = self._log_finished_episode()
        if seed is not None and self.rng == "philox" and int(seed) != self.seed_value:
            self.close()
            self.seed_value = int(seed)
        h = self._handle()
        self.time.n_episodes += 1
        E, N = self.num_envs, self.cfg.number_of_pedestrians
        if self.rng == "philox":
            nat.check(lib.evac_reset(h, None, _ptr(self._obs), self._stream()))
        else:
            nat.check(lib.evac_reset(h, None, None, self._stream()))  # zero time / accumulators
            pos = np.empty((E, N, 2))
            dirs = np.empty((E, N, 2))
            for e in range(E):  # pedestrians.py:17-20, env after env like a SyncVectorEnv would
                pos[e] = np.random.uniform(-1.0, 1.0, size=(N, 2))
                d = np.random.uniform(-1.0, 1.0, size=(N, 2))
                dirs[e] = (d.T / np.linalg.norm(d, axis=1)).T
            self.set_state(positions=pos, directions=dirs, agent_position=np.zeros((E, 2), np.float32),
                           agent_direction=np.zeros((E, 2), np.float32), now=np.zeros(E, np.int32))
            nat.check(lib.evac_observe(h, _ptr(self._obs), self._stream()))
        self._host_statuses = None
        if self.draw:
            self.pedestrians.memory = {"positions": [], "statuses": []}
            self.agent.memory = {"position": []}
            self.pedestrians.save()
        return self._emit_obs(), {}

    def _numpy_noise(self, out=None):
        """area.py:124: one U(-c/2, c/2) draw per VISCEK/FOLLOWER pedestrian, ascending index, from
        the global NumPy stream; scattered into the dense [E,N] table the kernel consumes."""
        E, N, c = self.num_envs, self.cfg.number_of_pedestrians, self.cfg.noise_coef
        if self._host_statuses is None:
            self._host_statuses = self.get_state()["statuses"].cpu().numpy()
        noise = np.zeros((E, N), dtype=np.float32) if out is None else out
        # ONE draw for the whole batch, environment-major then ascending pedestrian index: MT19937 hands out the same values as one
        # call per environment would (a double costs two words wherever the call boundary falls)
        fv = self._host_statuses.reshape(E, N) <= 2  # VISCEK = 1, FOLLOWER = 2 (statuses are 1..4)
        if self._env_params is not None:  # per-env noise_coef: the same draws, each scaled by its environment's coefficient
            c = np.repeat(self._env_params["noise_coef"], np.count_nonzero(fv, axis=1))
            noise[fv] = np.random.uniform(low=-c / 2, high=c / 2)
        else:
            noise[fv] = np.random.uniform(low=-c / 2, high=c / 2, size=int(np.count_nonzero(fv)))
        return noise

    def step(self, action, noise=None):
        """env.py:141-171 for every environment of the batch in one kernel launch.

        `noise` (optional): dense [E,N] angular-noise table (injection protocol, include/evac_b200.h)."""
        h, lib = self._handle(), nat.load()
        E, N = self.num_envs, self.cfg.number_of_pedestrians
        if self.batched:
            act = action
            if not (torch.is_tensor(act) and act.is_cuda and act.dtype == torch.float32 and act.is_contiguous()
                    and act.numel() == 2 * E):  # fast path: a ready [E,2] float32 CUDA tensor is used in place
                act = act if torch.is_tensor(act) else torch.as_tensor(np.asarray(act, dtype=np.float32))
                act = act.to(device=self.device, dtype=torch.float32).reshape(E, 2).contiguous()
            nz = None
            if noise is None and self.rng == "numpy":
                noise = self._numpy_noise()
            if noise is not None:
                nz = noise if torch.is_tensor(noise) else torch.as_tensor(np.asarray(noise, dtype=np.float32))
                nz = nz.to(device=self.device, dtype=torch.float32).reshape(E, N).contiguous()
            nat.check(lib.evac_step(h, _ptr(act), _ptr(nz), _ptr(self._obs), _ptr(self._reward),
                                    _ptr(self._terminated), _ptr(self._truncated), self._stream()))
            if self.rng == "numpy":
                self._host_statuses = None
            if self.draw:  # env.py:153-155 (host copies of the tracked environment; off by default)
                self.pedestrians.save()
                self.agent.save()
            return (self._obs_view, self._reward, self._terminated_b, self._truncated_b, {})
        # ---- single-env face: host buffers through evac_step_host
        if self._host is None:
            # ONE page-locked block [obs | reward | terminated | truncated | statuses]: evac_step_host fills it with a single
            # D2H copy; the actions (and the injected noise) are staged in page-locked arrays too, so the library copies straight
            # from them.  Pointers are taken once (ctypes / data_ptr conversions are a measurable part of a step).
            D = self.obs_dim
            blk = torch.empty(E * D * 4 + E * 4 + 2 * E + E * N, dtype=torch.uint8, pin_memory=True)
            o0, r0, t0, s0 = E * D * 4, E * D * 4 + E * 4, E * D * 4 + E * 4 + E, E * D * 4 + E * 4 + 2 * E
            self._host_block = blk
            self._host = dict(obs=blk[:o0].view(torch.float32).view(E, D), rew=blk[o0:r0].view(torch.float32), term=blk[r0:t0], trunc=blk[t0:s0],
                              status=blk[s0:].view(E, N))
            self._host_np = {k: v.numpy() for k, v in self._host.items()}
            self._host_np["term_b"], self._host_np["trunc_b"] = self._host_np["term"].view(np.bool_), self._host_np["trunc"].view(np.bool_)
            self._act_pin = torch.empty((E, 2), dtype=torch.float32, pin_memory=True)
            self._act_np = self._act_pin.numpy()
            self._noise_pin = torch.empty((E, N), dtype=torch.float32, pin_memory=True)
            self._noise_np = self._noise_pin.numpy()
            self._host_ptrs = tuple(_ptr(t) for t in (self._act_pin, self._host["obs"], self._host["rew"], self._host["term"], self._host["trunc"],
                                                      self._host["status"], self._noise_pin))
        self._act_np[...] = np.asarray(action, dtype=np.float32).reshape(E, 2)
        if noise is None and self.rng == "numpy":
            noise = self._numpy_noise(out=self._noise_np)
        pn = None
        if noise is not None:
            if noise is not self._noise_np:
                self._noise_np[...] = np.asarray(noise, dtype=np.float32).reshape(E, N)
            pn = self._host_ptrs[6]
        # outputs alias the page-locked buffers and are valid until the next step (the reference's
        # observations alias live state in the same way, env.py:100-102)
        hn = self._host_np
        obs, rew, term, trunc = hn["obs"], hn["rew"], hn["term"], hn["trunc"]
        if getattr(self, "_host_sync_needed", True):  # only after work was queued on torch's stream (reset, set_state, ...)
            torch.cuda.current_stream(self.device).synchronize()
            self._host_sync_needed = False
        pa, po, pr, pt, pu, ps = self._host_ptrs[:6]
        want_statuses = self.rng == "numpy" or E == 1  # (a large Philox batch does not pay the extra N bytes per env)
        nat.check(lib.evac_step_host(h, pa, pn, po, pr, pt, pu, ps if want_statuses else None))
        # the statuses after the step came back in the same copy (no get_state round trip): the next step's noise draw
        # (area.py:124: one value per VISCEK / FOLLOWER pedestrian) and `pedestrians.statuses` read them from here
        self._host_statuses = hn["status"] if want_statuses else None
        if self.draw:
            self.pedestrians.save()
            self.agent.save()
            if E == 1 and (bool(term[0]) or bool(trunc[0])):  # env.py:164-165
                try:
                    self.save_animation()
                except ImportError as exc:
                    log.warning("animation skipped: %s", exc)
        if E == 1:
            return self._structure(obs[0]), float(rew[0]), bool(term[0]), bool(trunc[0]), {}
        return self._structure(obs), rew, hn["term_b"], hn["trunc_b"], {}

    def rollout(self, num_steps: int, agent: str = "random", actions=None, noise=None, obs_every_step: bool = False,
                status_counts: bool = False):
        """`num_steps` consecutive steps in ONE kernel launch, state resident on chip.

        agent: "random" (RandomAgent, random_agent.py:8-9), "rotating" (rotating_agent.py:12-16), "wacuum"
        (WacuumCleaner, baseline_wacuum_cleaner.py:7-80, state machine on device) or "table" with actions
        [num_steps,E,2].  Returns (obs, reward_sum[E], terminated_any[E], truncated_any[E]); obs is [E,...] after the
        last step or [num_steps,E,...].  `status_counts=True` also records `pedestrians.status_stats` after every step
        into `self.last_status_counts` ([num_steps,E,4] int16 tensor: escaped, exiting, following, viscek)."""
        h, lib = self._handle(), nat.load()
        E, N, dev = self.num_envs, self.cfg.number_of_pedestrians, self.device
        kind = nat.AGENT[agent]
        act = nz = None
        if kind == 0:
            act = torch.as_tensor(actions).to(device=dev, dtype=torch.float32).reshape(num_steps, E, 2).contiguous()
        if noise is not None:
            nz = torch.as_tensor(noise).to(device=dev, dtype=torch.float32).reshape(num_steps, E, N).contiguous()
        obs = self._obs
        if obs_every_step:
            obs = torch.empty((num_steps, E, self.obs_dim), dtype=torch.float32, device=dev)
        trace = torch.empty((num_steps, E, 4), dtype=torch.int16, device=dev) if status_counts else None
        nat.check(lib.evac_rollout(h, int(num_steps), kind, _ptr(act), _ptr(nz), _ptr(obs), int(obs_every_step),
                                   _ptr(self._reward), _ptr(self._terminated), _ptr(self._truncated), _ptr(trace), self._stream()))
        self._host_statuses = None
        self.last_status_counts = trace
        return self._structure(obs), self._reward, self._terminated_b, self._truncated_b

    def efficiency_curve(self, num_steps: int, agent="random", chunk: int = 250, normalizer=None):
        """The "quantification of evacuation efficiency" statistic of src/plotting_old/plot.py:165-201: the number of
        escaped pedestrians after every step, mean and standard deviation over the environments (one episode each,
        from a fresh reset) -> (mean[num_steps], std[num_steps]) float64 tensors; `1 - mean / N` is the plotted
        "% NOT evacuated".  Everything runs on the device (`evac_rollout` with the scripted `agent`); create the env
        with auto_reset=False so that finished episodes stay at N escaped.

        `agent` may also be a trained fused policy (`FusedRPOTransformerPolicy` or `FusedRPOLinearPolicy`): it acts with the clipped
        actor mean, on the observation normalised by `normalizer` (a `VectorNormalizer`, used frozen; None = the raw observation), in
        chunks of `chunk` steps that record the status counts.  The gravity-encoding linear policy on a one-warp handle (float32,
        N <= 64) runs one `evac_rollout_policy` launch per chunk; every other pair runs `rollout.evaluate_policy`, one replayed
        CUDA graph of policy forward + step per step."""
        self.reset()
        fused = not isinstance(agent, str)
        if fused:
            from .rollout import evaluate_policy, fused_policy_rollout, one_launch_evaluation_supported
            one_launch = one_launch_evaluation_supported(self, agent)
            next_done = torch.zeros(self.num_envs, dtype=torch.float32, device=self.device)
        means, stds = [], []
        done = 0
        while done < num_steps:
            k = min(chunk, num_steps - done)
            if fused:
                trace = torch.empty((k, self.num_envs, 4), dtype=torch.int16, device=self.device)
                if one_launch:
                    fused_policy_rollout(self, agent, k, next_done, normalizer=normalizer, norm_update=False, normalize_reward=False,
                                         sample=False, status_counts=trace)
                else:
                    evaluate_policy(self, agent, k, normalizer=normalizer, status_counts=trace)
                self._host_statuses = None
                self.last_status_counts = trace
            else:
                self.rollout(k, agent=agent, status_counts=True)
            esc = self.last_status_counts[:, :, 0].to(torch.float64)
            means.append(esc.mean(dim=1)); stds.append(esc.std(dim=1, unbiased=False))
            done += k
        return torch.cat(means), torch.cat(stds)

    def episode_statistics(self):
        """(stats [E,9] float32, finished [E] bool, totals [10] float64) -- per-env record of the last
        finished episode in the key order of env.py:115-125 (`_native.EPISODE_STAT_KEYS`)."""
        h, lib = self._handle(), nat.load()
        E, dev = self.num_envs, self.device
        stats = torch.empty((E, nat.NUM_EPISODE_STATS), dtype=torch.float32, device=dev)
        fin = torch.empty(E, dtype=torch.uint8, device=dev)
        tot = torch.empty(1 + nat.NUM_EPISODE_STATS, dtype=torch.float64, device=dev)
        nat.check(lib.evac_episode_stats(h, _ptr(stats), _ptr(fin), _ptr(tot), self._stream()))
        return stats, fin.bool(), tot

    # ------------------------------------------------------------------ rendering (env.py:173-324), host-side
    def _render_kw(self):
        return dict(width=self.area.width, height=self.area.height, exit_position=self.area.exit.position,
                    to_exit=SwitchDistances.to_exit, to_escape=SwitchDistances.to_escape, to_leader=SwitchDistances.to_leader)

    def render(self):
        """PNG of the tracked environment's current state: `<path_png>/<experiment_name>_<now>.png` (env.py:173-240).
        Rasterised with Pillow (evacuation_b200/render.py); returns the file name."""
        from . import render as R

        st = self.get_state()
        e = self.tracked_env
        now = int(st["now"][e])
        path = os.path.join(self.path_png, f"{self.experiment_name}_{now}.png")
        R.save_png(path, st["positions"][e].cpu().numpy(), st["statuses"][e].cpu().numpy(), st["agent_position"][e].cpu().numpy(),
                   title=f"{self.experiment_name}. Timesteps: {now}", **self._render_kw())
        log.info("Env is rendered and png image is saved to %s", path)
        return path

    def save_animation(self):
        """GIF of the recorded trajectory (`draw=True`): `<path_giff>/<experiment_name>_ep-<n_episodes>.gif`, one frame per
        step, 20 ms per frame (env.py:241-324).  Returns the file name."""
        from . import render as R

        pos, sts, ag = self.pedestrians.memory["positions"], self.pedestrians.memory["statuses"], self.agent.memory["position"]
        path = os.path.join(self.path_giff, f"{self.experiment_name}_ep-{self.time.n_episodes}.gif")
        R.save_gif(path, pos, sts, ag, title=f"{self.experiment_name}\nn_episodes = {self.time.n_episodes}", **self._render_kw())
        log.info("Env is rendered and gif animation is saved to %s", path)
        if self.save_next_episode_anim:  # env.py:322-324
            self.save_next_episode_anim = False
            self.draw = False
        return path


__all__ = ["EvacuationEnv", "Status"]
