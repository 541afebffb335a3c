"""Rollout-loop glue around the fused step kernel (SURVEY.md section 8 row f1, BASELINE config 5).

The caller of the hot path in the reference is the cleanrl-style rollout loop of
`src/agents/rpo_agent.py:180-203`: policy forward -> `envs.step(action)` -> per-env gymnasium
wrappers (`wrapping()`, rpo_agent.py:24-33: FlattenObservation, ClipAction, NormalizeObservation,
clip(-1, 1), NormalizeReward(gamma), clip(-100, 100)).  Everything here is the device-resident,
batched equivalent of that glue so that the loop never leaves the GPU:

* `VectorNormalizer`   -- per-environment running mean / variance of observations and of the discounted
  return (gymnasium `RunningMeanStd`, batch of one sample per step and env), with the two clips;
* `RPOTransformerPolicy` -- the RPO transformer-embedding actor-critic
  (`src/agents/networks/rpo_transformer_agent_network.py:36-163`,
  `rpo_linear_agent_network.py:19-61`) restated in plain PyTorch (library GEMMs / SDPA: this is
  the consumer of the step kernel, not a kernel target of this tier);
* `RPOLinearPolicy`    -- the bare `RPOLinearNetwork` on the flattened observation (the gravity-encoding
  and flat-observation configs), restated the same way;
* `FusedRPOTransformerPolicy` / `FusedRPOLinearPolicy` -- their forward passes as the library's kernels;
* `PolicyRollout`      -- policy -> step -> normalise, one iteration captured in a CUDA graph
  and replayed (the tiny-GEMM policy is otherwise launch-bound);
* `evaluate_policy`    -- a trained fused policy evaluated (actor mean, frozen normaliser) on any handle, the same way.

The environment step is the CUDA path; there is no CPU fallback here either.
"""
from __future__ import annotations

import math
from typing import Optional

import torch
import torch.nn as nn
import torch.nn.functional as F


# ---------------------------------------------------------------------------------------------
class VectorNormalizer:
    """NormalizeObservation + clip(-1,1) + NormalizeReward(gamma) + clip(-100,100), one independent
    running estimate per environment (the reference wraps every env before vectorising them).

    gymnasium's `RunningMeanStd.update` with a batch of one sample x (batch_var = 0, batch_count = 1):
        delta = x - mean;  tot = count + 1
        mean' = mean + delta / tot
        var'  = (var * count + delta^2 * count / tot) / tot
    starting from mean = 0, var = 1, count = 1e-4; normalised value = (x - mean') / sqrt(var' + 1e-8).
    """

    def __init__(self, num_envs: int, obs_dim: int, gamma: float = 0.99, device="cuda", epsilon: float = 1e-8,
                 obs_clip: float = 1.0, reward_clip: float = 100.0, dtype=torch.float32):
        self.gamma, self.epsilon, self.obs_clip, self.reward_clip = gamma, epsilon, obs_clip, reward_clip
        self.obs_mean = torch.zeros((num_envs, obs_dim), dtype=dtype, device=device)
        self.obs_var = torch.ones((num_envs, obs_dim), dtype=dtype, device=device)
        self.ret_mean = torch.zeros(num_envs, dtype=dtype, device=device)
        self.ret_var = torch.ones(num_envs, dtype=dtype, device=device)
        self.returns = torch.zeros(num_envs, dtype=dtype, device=device)
        # the observation and return estimators see exactly one sample per call, so they share one count
        # per stream; kept as device scalars so that a captured CUDA graph advances them
        self.obs_count = torch.full((), 1e-4, dtype=torch.float64, device=device)
        self.ret_count = torch.full((), 1e-4, dtype=torch.float64, device=device)

    @staticmethod
    def _update(mean, var, count, x):
        tot = count + 1.0
        w_new = (1.0 / tot).to(mean.dtype)
        w_old = (count / tot).to(mean.dtype)
        delta = x - mean
        mean.add_(delta * w_new)
        var.mul_(w_old).add_(delta * delta * (w_old * w_new))
        count.add_(1.0)

    def observation(self, obs: torch.Tensor) -> torch.Tensor:
        """obs [E, D] (flattened like FlattenObservation) -> normalised, clipped copy."""
        self._update(self.obs_mean, self.obs_var, self.obs_count, obs)
        out = (obs - self.obs_mean) * torch.rsqrt(self.obs_var + self.epsilon)
        return out.clamp_(-self.obs_clip, self.obs_clip)

    def reward(self, reward: torch.Tensor, terminated: torch.Tensor) -> torch.Tensor:
        """NormalizeReward.step: returns = returns * gamma * (1 - terminated) + reward; reward / sqrt(var(returns) + eps)."""
        self.returns.mul_(self.gamma * (1.0 - terminated.to(self.returns.dtype))).add_(reward)
        self._update(self.ret_mean, self.ret_var, self.ret_count, self.returns)
        out = reward * torch.rsqrt(self.ret_var + self.epsilon)
        return out.clamp_(-self.reward_clip, self.reward_clip)


# ---------------------------------------------------------------------------------------------
def _ortho(layer: nn.Linear, std: float = math.sqrt(2.0), bias: float = 0.0) -> nn.Linear:
    nn.init.orthogonal_(layer.weight, std)  # networks/utils.py:4-7
    nn.init.constant_(layer.bias, bias)
    return layer


class _SetAttention(nn.Module):
    """The reference's attention variant (rpo_transformer_agent_network.py:36-75): projections to
    d_model * num_heads, then the softmax runs over the sequence with the d_model axis acting as the
    batch-of-heads axis and num_heads as the contracted feature axis; scale = sqrt(d_model)."""

    def __init__(self, d_model: int, num_heads: int):
        super().__init__()
        self.d_model, self.num_heads = d_model, num_heads
        self.Wq = nn.Linear(d_model, d_model * num_heads)
        self.Wk = nn.Linear(d_model, d_model * num_heads)
        self.Wv = nn.Linear(d_model, d_model * num_heads)
        self.dense = nn.Linear(d_model * num_heads, d_model)

    def forward(self, x):  # [B, S, D]
        B, S, D = x.shape
        H = self.num_heads

        def split(t):  # [B, S, H*D] -> [B, D, S, H]
            return t.view(B, S, H, D).permute(0, 3, 1, 2)

        # one GEMM for the three projections (K = 6 GEMMs are launch / tail bound); parameter names stay the reference's
        qkv = F.linear(x, torch.cat([self.Wq.weight, self.Wk.weight, self.Wv.weight]), torch.cat([self.Wq.bias, self.Wk.bias, self.Wv.bias]))
        q, k, v = (split(t) for t in qkv.split(H * D, dim=-1))
        if x.is_cuda:
            # zero-padding the contracted axis (H = 3) to 8 changes neither the scores nor the outputs but lets SDPA take
            # its fused kernel instead of the batched-GEMM + softmax fallback (2.6 -> 1.1 ms at 8192 envs on B200)
            pad = (-H) % 8
            q, k, v = (F.pad(t, (0, pad)) for t in (q, k, v))
            out = F.scaled_dot_product_attention(q, k, v, scale=1.0 / math.sqrt(D))[..., :H]
        else:
            out = F.scaled_dot_product_attention(q, k, v, scale=1.0 / math.sqrt(D))  # [B, D, S, H]
        out = out.transpose(1, 2).reshape(B, S, D * H)
        return self.dense(out)


def _layer_norm(x, ln: nn.LayerNorm):
    """LayerNorm over a 6-wide last axis written as elementwise ops: torch's row-wise kernel launches one block per
    row and takes 2.2 ms for the 5e5 rows of an 8192-env batch (half of the whole policy forward on B200)."""
    mu = x.mean(dim=-1, keepdim=True)
    xc = x - mu
    var = (xc * xc).mean(dim=-1, keepdim=True)
    return xc * torch.rsqrt(var + ln.eps) * ln.weight + ln.bias


class _Block(nn.Module):
    """rpo_transformer_agent_network.py:78-131: attention -> dropout -> (resid) -> LayerNorm -> FF (Linear, Dropout,
    ReLU, Linear) -> dropout -> (resid) -> LayerNorm."""

    def __init__(self, d_model: int, num_heads: int, d_ff: int, dropout: float, use_resid: bool):
        super().__init__()
        self.d_model, self.use_resid = d_model, use_resid
        self.attention = _SetAttention(d_model, num_heads)
        self.ff = nn.Sequential(nn.Linear(d_model, d_ff), nn.Dropout(dropout), nn.ReLU(), nn.Linear(d_ff, d_model))
        self.norm1, self.norm2 = nn.LayerNorm(d_model), nn.LayerNorm(d_model)
        self.dropout = nn.Dropout(dropout)

    def forward(self, x):
        shape = x.shape
        if x.dim() == 2:
            x = x.view(shape[0], -1, self.d_model)
        a = self.dropout(self.attention(x))
        x = _layer_norm(x + a if self.use_resid else a, self.norm1)
        f = self.dropout(self.ff(x))
        x = _layer_norm(x + f if self.use_resid else f, self.norm2)
        return x.view(shape)


def _rpo_heads(module: nn.Module, obs_dim: int, action_dim: int, num_hidden: int) -> None:
    """RPOLinearNetwork's parameters (rpo_linear_agent_network.py:23-42) as `critic`, `actor_mean`, `actor_logstd` of `module`."""
    module.critic = nn.Sequential(_ortho(nn.Linear(obs_dim, num_hidden)), nn.Tanh(), _ortho(nn.Linear(num_hidden, num_hidden)), nn.Tanh(),
                                  _ortho(nn.Linear(num_hidden, 1), std=1.0))
    module.actor_mean = nn.Sequential(_ortho(nn.Linear(obs_dim, num_hidden)), nn.Tanh(), _ortho(nn.Linear(num_hidden, num_hidden)), nn.Tanh(),
                                      _ortho(nn.Linear(num_hidden, action_dim), std=0.01))
    module.actor_logstd = nn.Parameter(torch.zeros(1, action_dim))


def _rpo_action_and_value(module: nn.Module, x, action: Optional[torch.Tensor]):
    """rpo_linear_agent_network.py:47-61 on the heads' input x: (action, logprob, entropy, value)."""
    mean = module.actor_mean(x)
    std = torch.exp(module.actor_logstd.expand_as(mean))
    if action is None:
        action = mean + std * torch.randn_like(mean)  # Normal(mean, std).sample()
    else:  # RPO: perturb the mean when re-evaluating stored actions
        mean = mean + torch.empty_like(mean).uniform_(-module.rpo_alpha, module.rpo_alpha)
    var = std * std
    logprob = (-((action - mean) ** 2) / (2 * var) - torch.log(std) - 0.5 * math.log(2 * math.pi)).sum(1)
    entropy = (0.5 + 0.5 * math.log(2 * math.pi) + torch.log(std)).sum(1)
    return action, logprob, entropy, module.critic(x)


class RPOLinearPolicy(nn.Module):
    """RPOLinearNetwork (rpo_linear_agent_network.py:19-61) directly on the flattened observation: the policy of the reference's
    gravity-encoding (6 floats) and flat rel / ohe observation configs.  Parameter names are the reference's."""

    def __init__(self, obs_dim: int, action_dim: int = 2, num_hidden: int = 64, rpo_alpha: float = 0.5):
        super().__init__()
        self.rpo_alpha = rpo_alpha
        _rpo_heads(self, obs_dim, action_dim, num_hidden)

    def get_value(self, x):
        return self.critic(x)

    def get_action_and_value(self, x, action: Optional[torch.Tensor] = None):
        return _rpo_action_and_value(self, x, action)


class RPOTransformerPolicy(nn.Module):
    """RPOTransformerEmbedding (rpo_transformer_agent_network.py:133-163) over RPOLinearNetwork
    (rpo_linear_agent_network.py:19-61).  `obs_dim` = (N + 2) * d_model flattened MatrixObs row."""

    def __init__(self, obs_dim: int, number_of_pedestrians: int, action_dim: int = 2, num_hidden: int = 64, rpo_alpha: float = 0.5,
                 num_blocks: int = 2, num_heads: int = 3, dim_feedforward: int = 96, dropout: float = 0.1, use_resid: bool = False,
                 chunk: int = 8192):
        super().__init__()
        d_model = obs_dim // (number_of_pedestrians + 2)
        self.rpo_alpha, self.chunk = rpo_alpha, chunk
        self.embedding = nn.Sequential(*[_Block(d_model, num_heads, dim_feedforward, dropout, use_resid) for _ in range(num_blocks)])
        _rpo_heads(self, obs_dim, action_dim, num_hidden)

    def embed(self, x):
        if x.shape[0] <= self.chunk:
            return self.embedding(x)
        return torch.cat([self.embedding(c) for c in x.split(self.chunk)], dim=0)  # bounds the attention workspace

    def get_value(self, x):
        return self.critic(self.embed(x))

    def get_action_and_value(self, x, action: Optional[torch.Tensor] = None):
        return _rpo_action_and_value(self, self.embed(x), action)


# ---------------------------------------------------------------------------------------------
_FLAT_BLOCK_KEYS = ("attention.Wq.weight", "attention.Wq.bias", "attention.Wk.weight", "attention.Wk.bias",
                    "attention.Wv.weight", "attention.Wv.bias", "attention.dense.weight", "attention.dense.bias",
                    "ff.0.weight", "ff.0.bias", "ff.3.weight", "ff.3.bias", "norm1.weight", "norm1.bias", "norm2.weight", "norm2.bias")
_FLAT_HEAD_KEYS = ("critic.0.weight", "critic.0.bias", "critic.2.weight", "critic.2.bias", "critic.4.weight", "critic.4.bias",
                   "actor_mean.0.weight", "actor_mean.0.bias", "actor_mean.2.weight", "actor_mean.2.bias",
                   "actor_mean.4.weight", "actor_mean.4.bias", "actor_logstd")


def flatten_policy_weights(state_dict, num_blocks: int):
    """The reference module's `state_dict()` -> the flat float32 vector `evac_policy_load_weights` documents
    (include/evac_b200.h).  Works on the unmodified reference `RPOTransformerEmbedding` and on `RPOTransformerPolicy`; with
    num_blocks = 0 on `RPOLinearPolicy` (the heads only)."""
    parts = [state_dict[f"embedding.{b}.{k}"] for b in range(num_blocks) for k in _FLAT_BLOCK_KEYS]
    parts += [state_dict[k] for k in _FLAT_HEAD_KEYS]
    return torch.cat([p.detach().to(torch.float32).reshape(-1).cpu() for p in parts]).contiguous()


class _FusedRPOPolicy:
    """What the fused policies share: the `evac_policy` handle, weight snapshots, the device call counter and `forward`.
    There is no CPU fallback: construction fails without the CUDA library / a device."""

    def __init__(self, cfg, module, obs_dim: int, device, seed: int, env_index_offset: int):
        import ctypes as C

        from . import _native as nat

        self._C, self._nat, self._lib = C, nat, nat.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise nat.EvacNativeError(f"{type(self).__name__} needs a CUDA device (no CPU fallback)")
        self.cfg, self.num_blocks, self.obs_dim, self.A = cfg, cfg.num_blocks, int(obs_dim), cfg.action_dim
        self.seed, self.env_index_offset = int(seed), int(env_index_offset)
        self._h = C.c_void_p()
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        nat.check(self._lib.evac_policy_create(C.byref(cfg), idx, C.byref(self._h)))
        self.calls = torch.zeros((), dtype=torch.int64, device=self.device)  # device-side stream offset (graph-replay safe)
        self.training = True  # like the reference's rollouts (the module is never put in eval mode)
        self.load_from(module)

    def load_from(self, module) -> None:
        flat = flatten_policy_weights(module.state_dict(), self.num_blocks)
        want = self._lib.evac_policy_num_weights(self._h)
        if flat.numel() != want:
            raise ValueError(f"policy weights: expected {want} floats, module has {flat.numel()}")
        self._nat.check(self._lib.evac_policy_load_weights(self._h, flat.data_ptr(), flat.numel()))

    def train(self, mode: bool = True):
        self.training = bool(mode)
        return self

    def eval(self):
        return self.train(False)

    def reserve(self, max_envs: int) -> None:
        self._nat.check(self._lib.evac_policy_reserve(self._h, int(max_envs)))

    @property
    def launch_count(self) -> int:
        return int(self._lib.evac_policy_launch_count(self._h))

    def _ptr(self, t, dtype=torch.float32):
        if t is None:
            return None
        if not (t.is_cuda and t.is_contiguous() and t.dtype == dtype):
            raise ValueError(f"expected a contiguous CUDA {dtype} tensor, got {t.dtype} on {t.device}")
        return t.data_ptr()

    def forward(self, obs, *, embedding=None, mean=None, value=None, action=None, action_clipped=None, logprob=None, entropy=None,
                given_action=None, sample=True, normalizer: Optional["VectorNormalizer"] = None, obs_norm=None, advance=True,
                norm_update=True):
        """One fused forward on the current stream; every output is an optional preallocated tensor.  `norm_update=False` uses
        `normalizer`'s statistics frozen (evaluation): they and `normalizer.obs_count` stay as they are, `obs_norm` is still written.
        Frozen together with `training` on the transformer policy raises NotImplementedError (evaluation runs without dropout)."""
        E = obs.shape[0]
        if obs.numel() != E * self.obs_dim:
            raise ValueError(f"obs must hold [E, {self.obs_dim}] values, got {tuple(obs.shape)}")
        io = self._nat.EvacPolicyIO()
        io.num_envs, io.obs = E, self._ptr(obs)
        if normalizer is not None:
            io.norm_mean, io.norm_var = self._ptr(normalizer.obs_mean), self._ptr(normalizer.obs_var)
            io.norm_count, io.obs_norm = self._ptr(normalizer.obs_count, torch.float64), self._ptr(obs_norm)
            io.norm_eps, io.norm_clip = normalizer.epsilon, normalizer.obs_clip
            io.norm_frozen = int(not norm_update)
        io.embedding, io.mean, io.value = self._ptr(embedding), self._ptr(mean), self._ptr(value)
        io.action, io.action_clipped = self._ptr(action), self._ptr(action_clipped)
        io.logprob, io.entropy, io.given_action = self._ptr(logprob), self._ptr(entropy), self._ptr(given_action)
        io.sample, io.training = int(sample), int(self.training)
        io.seed, io.offset, io.offset_device = self.seed, 0, self.calls.data_ptr()
        io.env_index_offset = self.env_index_offset
        st = torch.cuda.current_stream(self.device).cuda_stream
        self._nat.check(self._lib.evac_policy_forward(self._h, self._C.byref(io), self._C.c_void_p(st)))
        if normalizer is not None and norm_update:
            normalizer.obs_count.add_(1.0)
        if advance:
            self.calls.add_(1)

    # ---- the reference module's surface (rpo_linear_agent_network.py:44-61)
    def get_value(self, x):
        v = torch.empty(x.shape[0], device=self.device)
        self.forward(x.contiguous(), value=v, sample=False)
        return v.unsqueeze(1)

    def get_action_and_value(self, x, action: Optional[torch.Tensor] = None):
        """(action, logprob, entropy, value[E,1]) like the module; `action` given = evaluate its log-probability
        (without the RPO mean perturbation, which belongs to the trainer's update pass)."""
        E = x.shape[0]
        o = {k: torch.empty(s, device=self.device) for k, s in (("action", (E, self.A)), ("logprob", (E,)), ("entropy", (E,)), ("value", (E,)))}
        self.forward(x.contiguous(), given_action=None if action is None else action.contiguous(), **o)
        return o["action"], o["logprob"], o["entropy"], o["value"].unsqueeze(1)

    def __del__(self):
        try:
            if getattr(self, "_h", None) is not None and self._h.value:
                self._lib.evac_policy_destroy(self._h)
                self._h = None
        except Exception:
            pass


class FusedRPOTransformerPolicy(_FusedRPOPolicy):
    """Forward-only CUDA implementation of `RPOTransformerPolicy` (= the reference's `RPOTransformerEmbedding`):
    two hand-written kernels behind `evac_policy_forward` (csrc/evac_policy.cuh) instead of ~60 library launches --
    the transformer blocks run one warp per environment out of registers, the actor / critic heads 32 environments
    per CTA, Normal sampling, log-probability and ClipAction included.  Optionally fuses the per-env
    NormalizeObservation + clip of `VectorNormalizer` into its prologue (`normalizer=`).

    Weights are snapshotted from a torch module (`load_from`); call it again after an optimiser step.  There is no
    CPU fallback: construction fails without the CUDA library / a device."""

    def __init__(self, module: "RPOTransformerPolicy", number_of_pedestrians: int, device="cuda", seed: int = 0,
                 env_index_offset: int = 0, max_envs: int = 0):
        from . import _native as nat

        blk = module.embedding[0]
        self.S, self.D = number_of_pedestrians + 2, blk.d_model
        cfg = nat.EvacPolicyConfig()
        nat.check(nat.load().evac_policy_default_config(cfg, number_of_pedestrians, self.D))
        cfg.num_heads, cfg.dim_feedforward = blk.attention.num_heads, blk.ff[0].out_features
        cfg.num_blocks, cfg.use_resid = len(module.embedding), int(blk.use_resid)
        cfg.dropout, cfg.layer_norm_eps = float(blk.dropout.p), float(blk.norm1.eps)
        cfg.num_hidden, cfg.action_dim = module.critic[0].out_features, module.actor_mean[4].out_features
        super().__init__(cfg, module, self.S * self.D, device, seed, env_index_offset)
        if max_envs:
            self.reserve(max_envs)

    # ---- the reference module's surface (rpo_transformer_agent_network.py:155-163)
    def embed(self, x):
        out = torch.empty((x.shape[0], self.S * self.D), device=self.device)
        self.forward(x.contiguous(), embedding=out)
        return out


class FusedRPOLinearPolicy(_FusedRPOPolicy):
    """Forward-only CUDA implementation of `RPOLinearPolicy` (the reference's RPOLinearNetwork on the flattened observation):
    ONE kernel per forward -- the critic / actor MLPs on the tensor cores when `obs_dim` is a multiple of 4, else on the CUDA
    cores, with Normal sampling, log-probability and ClipAction -- and with `normalizer=` the per-env NormalizeObservation + clip
    of `VectorNormalizer` fused into the kernel's load of the observation.  `forward` takes the transformer class's keywords;
    `embedding=` is rejected (ValueError): this network has none.  `train()` / `eval()` are accepted (there is no dropout)."""

    def __init__(self, module: "RPOLinearPolicy", obs_dim: int, device="cuda", seed: int = 0, env_index_offset: int = 0):
        from . import _native as nat

        cfg = nat.EvacPolicyConfig()
        nat.check(nat.load().evac_policy_default_linear_config(cfg, int(obs_dim)))
        cfg.num_hidden, cfg.action_dim = module.critic[0].out_features, module.actor_mean[4].out_features
        super().__init__(cfg, module, obs_dim, device, seed, env_index_offset)


def normalize_reward_fused(norm: "VectorNormalizer", reward: torch.Tensor, terminated: torch.Tensor, out: torch.Tensor,
                           truncated: Optional[torch.Tensor] = None, done_out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """`VectorNormalizer.reward` as ONE kernel (evac_normalize_reward); `terminated` / `truncated` are the uint8/bool flag
    tensors of step().  With `truncated` and `done_out` the same pass writes next_done = float(terminated | truncated)."""
    import ctypes as C

    from . import _native as nat

    lib = nat.load()
    u8 = lambda t: None if t is None else (t.view(torch.uint8) if t.dtype == torch.bool else t).data_ptr()
    st = torch.cuda.current_stream(reward.device).cuda_stream
    nat.check(lib.evac_normalize_reward(reward.shape[0], reward.data_ptr(), u8(terminated), u8(truncated), norm.returns.data_ptr(),
                                        norm.ret_mean.data_ptr(), norm.ret_var.data_ptr(), norm.ret_count.data_ptr(), out.data_ptr(),
                                        None if done_out is None else done_out.data_ptr(), norm.gamma, norm.epsilon,
                                        norm.reward_clip, C.c_void_p(st)))
    norm.ret_count.add_(1.0)
    return out


def policy_launch_sizes(num_steps: int, steps_per_launch: int) -> list:
    """Iterations of each `evac_rollout_policy` launch: `steps_per_launch` each, the last launch the remainder."""
    if int(num_steps) < 1 or int(steps_per_launch) < 1:
        raise ValueError(f"num_steps and steps_per_launch must be >= 1, got {num_steps}, {steps_per_launch}")
    n, k = int(num_steps), int(steps_per_launch)
    return [k] * (n // k) + ([n % k] if n % k else [])


def check_policy_rollout_tensors(num_envs: int, obs_dim: int, normalizer: Optional["VectorNormalizer"] = None, next_done=None,
                                 **outputs) -> None:
    """The shapes and dtypes `fused_policy_rollout` needs (ValueError otherwise): the normaliser's [E, obs_dim] / [E] float32 statistics
    and float64 scalar counts, next_done [E] float32, and every given per-step output as [T, E, ...] of its dtype.  Device-free."""
    E, D = int(num_envs), int(obs_dim)

    def want(name, t, shape, dtype):
        if t is None:
            return
        if tuple(t.shape) != tuple(shape) or t.dtype != dtype or not t.is_contiguous():
            raise ValueError(f"{name}: expected a contiguous {dtype} tensor of shape {tuple(shape)}, got {t.dtype} {tuple(t.shape)}")

    want("next_done", next_done, (E,), torch.float32)
    if normalizer is not None:
        n = normalizer
        want("obs_mean", n.obs_mean, (E, D), torch.float32); want("obs_var", n.obs_var, (E, D), torch.float32)
        for k in ("returns", "ret_mean", "ret_var"):
            want(k, getattr(n, k), (E,), torch.float32)
        want("obs_count", n.obs_count, (), torch.float64); want("ret_count", n.ret_count, (), torch.float64)
    T = None
    for k, t in outputs.items():
        if t is None:
            continue
        T = t.shape[0] if T is None else T
        tail, dtype = {"obs_norm": ((D,), torch.float32), "action": ((2,), torch.float32), "status_counts": ((4,), torch.int16)}.get(k, ((), torch.float32))
        want(k, t, (T, E, *tail), dtype)


def fused_policy_rollout(env, policy: "FusedRPOLinearPolicy", num_steps: int, next_done: torch.Tensor, *, normalizer: Optional["VectorNormalizer"] = None,
                         norm_update: bool = True, normalize_reward: bool = True, sample: bool = True, obs_norm=None, action=None, logprob=None, value=None, reward_norm=None,
                         dones=None, status_counts=None) -> None:
    """`num_steps` iterations of the gravity-encoding rollout loop (rpo_agent.py:180-203) in ONE step-kernel launch
    (`evac_rollout_policy`): the fused linear policy (with `normalizer`'s NormalizeObservation, updated or, `norm_update=False`,
    frozen), ClipAction, the env step with same-step auto-reset and (`normalize_reward`) its NormalizeReward, for every environment
    of `env`.  Reads the raw
    observation from, and leaves the last one in, `env.unwrapped.flat_observation`; advances the normaliser's counts and
    `policy.calls` by `num_steps`.  The per-step outputs are optional [num_steps, E, ...] tensors.  Supported: a handle of the
    one-warp kernel (float32, N <= 64) with positions = grav and a `FusedRPOLinearPolicy` on its 6 values with action_dim 2;
    anything else raises NotImplementedError."""
    import ctypes as C

    from . import _native as nat

    if not isinstance(policy, _FusedRPOPolicy):
        raise NotImplementedError(f"the one-launch rollout runs the fused linear policy, not {type(policy).__name__}")
    u = env.unwrapped
    E = u.num_envs
    if int(num_steps) < 1:
        raise ValueError(f"num_steps must be >= 1, got {num_steps}")
    check_policy_rollout_tensors(E, u.obs_dim, normalizer, next_done, obs_norm=obs_norm, action=action, logprob=logprob, value=value,
                                 reward_norm=reward_norm, dones=dones, status_counts=status_counts)
    for k, t in (("obs_norm", obs_norm), ("action", action), ("logprob", logprob), ("value", value), ("reward_norm", reward_norm),
                 ("dones", dones), ("status_counts", status_counts)):
        if t is not None and t.shape[0] != num_steps:
            raise ValueError(f"{k}: expected {num_steps} steps, got {t.shape[0]}")
    p = lambda t: None if t is None else t.data_ptr()
    io = nat.EvacPolicyRolloutIO()
    io.obs, io.next_done = p(u.flat_observation), p(next_done)
    if normalizer is not None:
        n = normalizer
        io.norm_mean, io.norm_var, io.norm_count = p(n.obs_mean), p(n.obs_var), p(n.obs_count)
        io.norm_eps, io.norm_clip, io.norm_update = n.epsilon, n.obs_clip, int(bool(norm_update))
        if normalize_reward:
            io.returns, io.ret_mean, io.ret_var, io.ret_count = p(n.returns), p(n.ret_mean), p(n.ret_var), p(n.ret_count)
            io.gamma, io.eps, io.clip = n.gamma, n.epsilon, n.reward_clip
    io.sample, io.seed, io.offset, io.offset_device = int(bool(sample)), policy.seed, 0, p(policy.calls)
    io.env_index_offset = policy.env_index_offset
    io.obs_norm, io.action, io.logprob, io.value = p(obs_norm), p(action), p(logprob), p(value)
    io.reward_norm, io.dones, io.status_counts = p(reward_norm), p(dones), p(status_counts)
    io.reward_sum, io.terminated, io.truncated = p(u._reward), p(u._terminated), p(u._truncated)
    st = torch.cuda.current_stream(u.device).cuda_stream
    nat.check(nat.load().evac_rollout_policy(u._handle(), policy._h, int(num_steps), C.byref(io), C.c_void_p(st)))


def one_launch_evaluation_supported(env, policy) -> bool:
    """Whether `evac_rollout_policy` runs `policy` on `env` (include/evac_b200.h): a handle of the one-warp step kernel (float32,
    N <= 64) with positions = grav, and a `FusedRPOLinearPolicy` on its 6 values with action_dim 2.  Device-free."""
    u = env.unwrapped
    return (u.precision == "fp32" and u.cfg.number_of_pedestrians <= 64 and u._positions == "grav"
            and isinstance(policy, FusedRPOLinearPolicy) and policy.obs_dim == 6 and policy.A == 2)


def check_evaluation_args(num_envs: int, obs_dim: int, policy, num_steps: int, normalizer: Optional["VectorNormalizer"] = None,
                          **outputs) -> None:
    """What `evaluate_policy` needs before it touches a device: a fused policy (NotImplementedError otherwise) on the env's
    obs_dim values with 2 actions, num_steps >= 1, and the normaliser and the per-step outputs of `check_policy_rollout_tensors`,
    each output with num_steps rows (ValueError otherwise)."""
    if not isinstance(policy, _FusedRPOPolicy):
        raise NotImplementedError(f"evaluate_policy runs a fused policy (FusedRPOTransformerPolicy, FusedRPOLinearPolicy), "
                                  f"not {type(policy).__name__}")
    if policy.obs_dim != int(obs_dim) or policy.A != 2:
        raise ValueError(f"the policy reads {policy.obs_dim} values and acts with {policy.A}; the env has obs_dim {obs_dim} and 2 actions")
    if int(num_steps) < 1:
        raise ValueError(f"num_steps must be >= 1, got {num_steps}")
    check_policy_rollout_tensors(num_envs, obs_dim, normalizer, **outputs)
    for k, t in outputs.items():
        if t is not None and t.shape[0] != num_steps:
            raise ValueError(f"{k}: expected {num_steps} steps, got {t.shape[0]}")


def _snapshot(env, tensors):
    """The env's checkpoint image and copies of `tensors`: what one captured iteration mutates, for `_restore`."""
    return env.unwrapped.save_state(), [(t, t.clone()) for t in tensors]


def _restore(env, snap):
    image, tensors = snap
    env.unwrapped.load_state(image)
    for t, saved in tensors:
        t.copy_(saved)


def _capture_graph(env, iteration, tensors, count):
    """One `iteration()` recorded into a CUDA graph -> (graph, kernels counted by `count()` while recording).

    The warm-up outside the capture (lazy initialisation: function attributes, library autotuning) and the capture itself execute /
    record real iterations, so the env state and `tensors` (everything else an iteration mutates) are snapshotted and restored: the
    first replay starts exactly where the caller left the environments."""
    device = env.unwrapped.device
    snap = _snapshot(env, tensors)
    rng_state = torch.cuda.get_rng_state(device)
    side = torch.cuda.Stream(device=device)
    side.wait_stream(torch.cuda.current_stream(device))
    with torch.cuda.stream(side):
        for _ in range(2):
            iteration()
    torch.cuda.current_stream(device).wait_stream(side)
    torch.cuda.synchronize(device)
    graph = torch.cuda.CUDAGraph()
    before = count()
    with torch.cuda.graph(graph):
        iteration()
    launches = count() - before
    _restore(env, snap)
    torch.cuda.set_rng_state(rng_state, device)
    torch.cuda.synchronize(device)
    return graph, launches


@torch.no_grad()
def evaluate_policy(env, policy, num_steps: int, *, normalizer: Optional["VectorNormalizer"] = None, obs_norm=None, action=None,
                    status_counts=None) -> None:
    """`num_steps` evaluation steps of a trained fused policy (`FusedRPOTransformerPolicy` or `FusedRPOLinearPolicy`) on every
    environment of `env`, whatever kernel its handle runs (one-warp, CTA cell list, cluster, float64).

    Per step: `evac_policy_forward` on the env's raw observation with training off, the actor mean as the action and `normalizer`'s
    statistics frozen (None = the raw observation), then one table-agent step (`evac_rollout`) on the clipped action.  One step is
    captured in a CUDA graph and replayed; the capture does not advance the environments.  The per-step outputs are optional
    [num_steps, E, ...] tensors: `obs_norm` the observation the policy saw, `action` the actor mean before ClipAction,
    `status_counts` (int16) the escaped / exiting / following / viscek counts after the step.  `policy.calls`, `policy.training` and
    the normaliser are left as they are."""
    u = env.unwrapped
    E, D = u.num_envs, u.obs_dim
    T = int(num_steps)
    check_evaluation_args(E, D, policy, T, normalizer, obs_norm=obs_norm, action=action, status_counts=status_counts)
    from . import _native as nat

    lib, dev = nat.load(), u.device
    policy.reserve(E)  # the transformer's embedding scratch, allocated before the capture
    x = u.flat_observation  # the raw observation: every step rewrites this buffer in place
    step_act = torch.empty((E, 2), device=dev) if action is not None else None
    step_clip = torch.empty((E, 2), device=dev)
    step_norm = torch.empty((E, D), device=dev) if obs_norm is not None and normalizer is not None else None
    step_counts = torch.empty((1, E, 4), dtype=torch.int16, device=dev) if status_counts is not None else None
    p = lambda t: None if t is None else t.data_ptr()

    def iteration():
        policy.forward(x, action=step_act, action_clipped=step_clip, sample=False, normalizer=normalizer, obs_norm=step_norm,
                       norm_update=False, advance=False)
        nat.check(lib.evac_rollout(u._handle(), 1, nat.AGENT["table"], p(step_clip), None, p(x), 0, p(u._reward), p(u._terminated),
                                   p(u._truncated), p(step_counts), u._stream()))

    training = policy.training
    policy.training = False
    try:
        graph, _ = _capture_graph(env, iteration, [x, u._reward, u._terminated, u._truncated], lambda: 0)
    finally:
        policy.training = training
    for t in range(T):
        if obs_norm is not None and normalizer is None:
            obs_norm[t].copy_(x)  # without a normaliser the policy sees the raw observation
        graph.replay()
        if step_norm is not None:
            obs_norm[t].copy_(step_norm)
        if action is not None:
            action[t].copy_(step_act)
        if status_counts is not None:
            status_counts[t].copy_(step_counts[0])
    u._host_statuses = None


# ---------------------------------------------------------------------------------------------
class PolicyRollout:
    """policy forward -> ClipAction -> fused env step (same-step auto-reset) -> normalise, `num_steps` times.

    One iteration is captured in a CUDA graph (`use_graph=True`) and replayed; storage tensors follow
    rpo_agent.py:160-163 (obs, actions, logprobs, rewards, dones, values)."""

    def __init__(self, env, policy, gamma: float = 0.99, use_graph: bool = True, store: bool = True):
        self.env, self.policy, self.store, self.use_graph = env, policy, store, use_graph
        u = env.unwrapped
        self.E, self.D, self.device = u.num_envs, u.obs_dim, u.device
        self.norm = VectorNormalizer(self.E, self.D, gamma=gamma, device=self.device)
        self.next_obs = torch.zeros((self.E, self.D), device=self.device)
        self.next_done = torch.zeros(self.E, device=self.device)
        self.out = {k: torch.zeros(s, device=self.device) for k, s in
                    (("action", (self.E, 2)), ("logprob", (self.E,)), ("value", (self.E,)), ("reward", (self.E,)))}
        self._graph = None
        self._graph_params_mode = None  # env's _env_params_mode at capture: uniform and per-env steps are different kernels
        self.launches_per_iteration = None
        # fused policy: NormalizeObservation runs in the policy's first kernel on the env's raw observation buffer, so `next_obs`
        # (the normalised observation the policy saw) is produced INSIDE the iteration
        self.fused = isinstance(policy, _FusedRPOPolicy)
        self._raw_obs = None
        self._act_clipped = torch.zeros((self.E, 2), device=self.device)
        if self.fused:
            policy.reserve(self.E)

    def reset(self):
        self.env.reset()
        obs = self.env.unwrapped.flat_observation  # Box or Dict: the env's persistent [E, D] buffer (step() rewrites it)
        if self.fused:
            self._raw_obs = obs
        else:
            self.next_obs.copy_(self.norm.observation(obs))
        self.next_done.zero_()

    @torch.no_grad()
    def _iteration(self):
        if self.fused:
            # transformer: 4 launches (policy embedding, policy heads (+ sampling, ClipAction), env step, reward normaliser);
            # linear: 3 (the heads with the normaliser fused into their load of the observation, env step, reward normaliser)
            self.policy.forward(self._raw_obs, normalizer=self.norm, obs_norm=self.next_obs, action=self.out["action"],
                                action_clipped=self._act_clipped, logprob=self.out["logprob"], value=self.out["value"])
            _, reward, term, trunc, _ = self.env.step(self._act_clipped)
            assert self.env.unwrapped.flat_observation.data_ptr() == self._raw_obs.data_ptr()
            normalize_reward_fused(self.norm, reward, term, self.out["reward"], truncated=trunc, done_out=self.next_done)
            return
        action, logprob, _, value = self.policy.get_action_and_value(self.next_obs)
        _, reward, term, trunc, _ = self.env.step(action.clamp(-1.0, 1.0).contiguous())  # ClipAction
        self.out["action"].copy_(action); self.out["logprob"].copy_(logprob); self.out["value"].copy_(value.flatten())
        self.out["reward"].copy_(self.norm.reward(reward, term))
        self.next_obs.copy_(self.norm.observation(self.env.unwrapped.flat_observation))
        self.next_done.copy_(torch.logical_or(term, trunc).to(self.next_done.dtype))

    def _mutated(self):
        """Everything one `_iteration()` mutates besides the env state: normaliser statistics, the loop's carried tensors, the
        policy's stream offset and the observation buffer."""
        u = self.env.unwrapped
        tensors = [self.next_obs, self.next_done, u.flat_observation, *self.out.values(), self._act_clipped,
                   self.norm.obs_mean, self.norm.obs_var, self.norm.obs_count, self.norm.returns, self.norm.ret_mean, self.norm.ret_var, self.norm.ret_count]
        if self.fused:
            tensors.append(self.policy.calls)
        return tensors

    def _capture(self):
        # the first run() starts exactly where reset() left the environments (ADVICE r1: the warm-up used to advance them by two steps)
        count = lambda: self.env.unwrapped.launch_count + (self.policy.launch_count if self.fused else 0)
        self._graph, launches = _capture_graph(self.env, self._iteration, self._mutated(), count)
        # kernels of THIS library recorded into one graph replay: the handles count launches at capture time; the fused loop's
        # evac_normalize_reward is a handle-less entry point (+1)
        self.launches_per_iteration = launches + (1 if self.fused else 0)
        self._graph_params_mode = self.env.unwrapped._env_params_mode

    def run(self, num_steps: int, steps_per_launch: int = 1):
        """Returns the storage dict ([T, E, ...]) when `store`, else None.

        `steps_per_launch` > 1 (the gravity-encoding config with a `FusedRPOLinearPolicy`): each launch of `evac_rollout_policy` runs
        that many iterations in the step kernel (the last launch the remainder), bit-identical to the per-step loop and writing the
        storage in place; `self.out` and `self.next_obs` are not updated on this path.  Switching between the two paths mid-run
        continues the same trajectory.  Anything else raises NotImplementedError; 1 is the CUDA-graph loop."""
        if steps_per_launch != 1:
            return self._run_fused(num_steps, steps_per_launch)
        if self._graph is not None and self._graph_params_mode != self.env.unwrapped._env_params_mode:
            self._graph = None  # set_env_params switched between the uniform and the per-env step kernel: capture again
        if self.use_graph and self._graph is None:
            self._capture()
        buf = None
        if self.store:
            buf = dict(obs=torch.empty((num_steps, self.E, self.D), device=self.device), actions=torch.empty((num_steps, self.E, 2), device=self.device),
                       logprobs=torch.empty((num_steps, self.E), device=self.device), rewards=torch.empty((num_steps, self.E), device=self.device),
                       dones=torch.empty((num_steps, self.E), device=self.device), values=torch.empty((num_steps, self.E), device=self.device))
        for t in range(num_steps):
            if buf is not None:
                buf["dones"][t].copy_(self.next_done)
                if not self.fused:
                    buf["obs"][t].copy_(self.next_obs)
            if self._graph is not None:
                self._graph.replay()
            else:
                self._iteration()
            if buf is not None:
                if self.fused:
                    buf["obs"][t].copy_(self.next_obs)
                buf["actions"][t].copy_(self.out["action"]); buf["logprobs"][t].copy_(self.out["logprob"])
                buf["values"][t].copy_(self.out["value"]); buf["rewards"][t].copy_(self.out["reward"])
        return buf

    def _new_storage(self, num_steps):
        return dict(obs=torch.empty((num_steps, self.E, self.D), device=self.device), actions=torch.empty((num_steps, self.E, 2), device=self.device),
                    logprobs=torch.empty((num_steps, self.E), device=self.device), rewards=torch.empty((num_steps, self.E), device=self.device),
                    dones=torch.empty((num_steps, self.E), device=self.device), values=torch.empty((num_steps, self.E), device=self.device))

    def _run_fused(self, num_steps, steps_per_launch):
        sizes = policy_launch_sizes(num_steps, steps_per_launch)
        if not isinstance(self.policy, FusedRPOLinearPolicy):
            raise NotImplementedError(f"steps_per_launch > 1 runs the fused linear policy, not {type(self.policy).__name__}")
        if self._raw_obs is None:
            raise ValueError("call reset() first")
        buf = self._new_storage(num_steps) if self.store else None
        t = 0
        for k in sizes:
            o = {} if buf is None else dict(obs_norm=buf["obs"][t:t + k], action=buf["actions"][t:t + k], logprob=buf["logprobs"][t:t + k],
                                            value=buf["values"][t:t + k], reward_norm=buf["rewards"][t:t + k], dones=buf["dones"][t:t + k])
            fused_policy_rollout(self.env, self.policy, k, self.next_done, normalizer=self.norm, **o)
            t += k
        return buf


__all__ = ["VectorNormalizer", "RPOTransformerPolicy", "RPOLinearPolicy", "FusedRPOTransformerPolicy", "FusedRPOLinearPolicy", "PolicyRollout",
           "flatten_policy_weights", "normalize_reward_fused", "fused_policy_rollout", "evaluate_policy"]
