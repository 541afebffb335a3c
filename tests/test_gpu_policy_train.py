"""GPU tests of the fused policy in training mode (the mode of the config-5 rollout loop: the reference's rollouts never call
.eval()) against float64, with the random streams restated: the embedding kernel's dropout masks and the heads' Normal draws
come from evac_testlib (dropout_masks, policy_normal), which tests/test_host_cpu.py::test_policy_streams_match_their_numpy_restatement
pins to the kernels' own stream functions.  The references are the plain-PyTorch restatements `RPOTransformerPolicy` /
`RPOLinearPolicy` (pinned to the reference network's goldens by tests/test_rollout_cpu.py) evaluated on the CPU, with the
restated masks multiplied in where `_Block` calls `self.dropout` (attention output, block output) and `ff[1]` (hidden layer).

Bars.  Embedding: |kernel - f64| <= 2e-5 + 4 |torch32 - f64| elementwise, torch32 being the same masked forward in float32:
dropout can leave a LayerNorm row almost constant, and there float32 rounding is amplified for any implementation.  Sampling:
action - mean = exp(logstd) z to float32 rounding of the Box-Muller terms, 2e-6 (1 + r) with r the Box-Muller radius."""
import copy
import math

import numpy as np
import pytest
import torch
import torch.nn as nn

import evac_testlib as T

pytestmark = pytest.mark.gpu

SEED = 2 ** 32 + 0x5EED          # both seed words are used
ENV_OFFSET = 2 ** 31 - 5         # global env indices cross 2^31 inside the larger batches
HALF_LOG_2PI = 0.5 * math.log(2 * math.pi)


def _mods():
    from evacuation_b200.rollout import FusedRPOLinearPolicy, FusedRPOTransformerPolicy, PolicyRollout, RPOLinearPolicy, RPOTransformerPolicy
    return FusedRPOTransformerPolicy, FusedRPOLinearPolicy, PolicyRollout, RPOTransformerPolicy, RPOLinearPolicy


def _perturb(net, seed):
    """Non-trivial LayerNorm affine, biases and log-std (the defaults are 1 / 0 / 0)."""
    torch.manual_seed(seed)
    with torch.no_grad():
        for name, p in net.named_parameters():
            if "norm" in name or name.endswith("bias") or name == "actor_logstd":
                p.add_(0.3 * torch.randn_like(p))
    return net


def _transformer(n_ped, d_model, p, seed=0, **kw):
    torch.manual_seed(seed)
    return _perturb(_mods()[3]((n_ped + 2) * d_model, n_ped, dropout=p, **kw), seed + 1)


class _Mask(nn.Module):
    """Stands in for nn.Dropout: multiplies by the given masks in turn."""

    def __init__(self, *masks):
        super().__init__()
        self.masks, self.calls = masks, 0

    def forward(self, x):
        m = self.masks[self.calls % len(self.masks)]
        self.calls += 1
        return x * m


def _masked_forward(net, x, masks, dtype):
    """(embedding, mean, value) of `net` in `dtype` on the CPU with the restated masks (per block: attention, hidden, output)."""
    m = copy.deepcopy(net).cpu().to(dtype)
    for blk, (ma, mh, mo) in zip(m.embedding, masks):
        blk.dropout = _Mask(torch.as_tensor(ma, dtype=dtype), torch.as_tensor(mo, dtype=dtype))
        blk.ff[1] = _Mask(torch.as_tensor(mh, dtype=dtype))
    with torch.no_grad():
        emb = m.embed(x.detach().cpu().to(dtype))
        return emb, m.actor_mean(emb), m.critic(emb).flatten()


def _within(got, f64, t32, base, name):
    """|got - f64| <= base + 4 |t32 - f64| elementwise; returns (max, median) of |got - f64|."""
    got, f64, t32 = (np.asarray(v, dtype=np.float64) for v in (got, f64, t32))
    err, ref_err = np.abs(got - f64), np.abs(t32 - f64)
    bad = err > base + 4 * ref_err
    assert not bad.any(), f"{name}: {int(bad.sum())} of {bad.size} beyond the bar, worst {float(err[bad].max()):.3g} (torch32 there {float(ref_err[bad][np.argmax(err[bad])]):.3g})"
    return float(err.max()), float(np.median(err))


def _sampling_bar(sd, rad, act):
    """|action - (mean + sd z)| allowed: float32 rounding of the Box-Muller terms and of the stored action."""
    return sd * 2e-6 * (1 + rad) + 2.0 ** -23 * np.abs(act)


# ---------------------------------------------------------------------------------------------------------------------------
# (a) the training-mode embedding against float64
TRAIN_SHAPES = [
    (60, 6, {}, 0.1, 1003),      # the default network, the last 4-warp CTA partial
    (60, 6, {}, 0.5, 37),
    (60, 3, {}, 0.1, 37), (60, 2, {}, 0.5, 37),
    (60, 6, dict(num_heads=1), 0.1, 37), (60, 6, dict(num_heads=2), 0.5, 1), (60, 6, dict(num_heads=4), 0.1, 37),
    (60, 6, dict(dim_feedforward=10), 0.1, 37), (60, 6, dict(dim_feedforward=33, num_blocks=3), 0.5, 37),   # F padded to F4
    (60, 6, dict(num_blocks=1), 0.1, 1),
    (60, 6, dict(use_resid=True), 0.1, 37), (20, 6, dict(use_resid=True, num_hidden=12), 0.5, 1003),
    (1, 6, {}, 0.1, 37), (31, 6, {}, 0.5, 37), (62, 6, {}, 0.1, 1003),   # S = 3, 33, 64: lane row rb invalid / at the limit
]


@pytest.mark.parametrize("n_ped,d_model,kw,p,E", TRAIN_SHAPES)
def test_training_embedding_matches_float64_with_restated_masks(n_ped, d_model, kw, p, E):
    Fused = _mods()[0]
    net = _transformer(n_ped, d_model, p, seed=n_ped + 7 * d_model + E, **kw)
    S, K = n_ped + 2, (n_ped + 2) * d_model
    fused = Fused(net, n_ped, device="cuda", seed=SEED, env_index_offset=ENV_OFFSET)
    assert fused.training
    g = torch.Generator().manual_seed(E)
    x = (torch.randn(E, K, generator=g) * 0.7).clamp_(-1, 1).cuda()
    given = (torch.rand(E, net.actor_mean[4].out_features, generator=g) * 2 - 1).cuda()
    for _ in range(3):   # advance the device call counter: the checked call draws stream offset 3
        fused.forward(x, embedding=torch.empty_like(x))
    assert int(fused.calls) == 3
    emb, mean, value, lp = torch.empty_like(x), torch.empty_like(given), torch.empty(E, device="cuda"), torch.empty(E, device="cuda")
    fused.forward(x, embedding=emb, mean=mean, value=value, logprob=lp, given_action=given)
    torch.cuda.synchronize()

    blk = net.embedding[0]
    masks = T.dropout_masks(SEED, 3, ENV_OFFSET, E, len(net.embedding), S, d_model, blk.ff[0].out_features, p)
    e64 = _masked_forward(net, x, masks, torch.float64)[0].numpy()
    e32 = _masked_forward(net, x, masks, torch.float32)[0].numpy()
    mx, med = _within(emb.cpu().numpy(), e64, e32, 2e-5, "embedding")
    print(f"embedding vs float64: max {mx:.3g}, median {med:.3g}")
    # the heads on the kernel's own embedding, in float64 (the bars of test_gpu_policy.py's float64 heads test)
    net64 = copy.deepcopy(net).double()
    with torch.no_grad():
        ek = emb.cpu().double()
        mean64, val64 = net64.actor_mean(ek), net64.critic(ek).flatten()
    assert float((mean.cpu().double() - mean64).abs().max()) < 2e-6
    assert float((value.cpu().double() - val64).abs().max() / val64.abs().max().clamp_min(1.0)) < 6e-6
    ls = net.actor_logstd.detach().double().flatten()
    lp64 = (-0.5 * ((given.cpu().double() - mean64) / ls.exp()) ** 2 - ls - HALF_LOG_2PI).sum(1)
    np.testing.assert_allclose(lp.cpu().numpy(), lp64.numpy(), rtol=1e-5, atol=5e-5)


# ---------------------------------------------------------------------------------------------------------------------------
# (b) sampling is exact
SAMPLING_CASES = [("transformer", tc, A, NH, 257) for tc in ("1", "0") for A in (1, 2, 3) for NH in (12, 64)]
SAMPLING_CASES += [("transformer", "1", 2, 64, 38000), ("transformer", "0", 3, 64, 38000)]   # 64 -> 128-column tiles
SAMPLING_CASES += [("linear6", "1", A, NH, 257) for A in (1, 3) for NH in (12, 64)]           # K = 6: the CUDA cores
SAMPLING_CASES += [("linear364", tc, A, NH, 257) for tc in ("1", "0") for A in (1, 3) for NH in (12, 64)]
SAMPLING_CASES += [("linear364", "1", 3, 64, 38000), ("linear364", "0", 2, 12, 38000)]


@pytest.mark.parametrize("kind,tc,A,NH,E", SAMPLING_CASES)
def test_sampled_actions_are_the_restated_normal_draws(kind, tc, A, NH, E, monkeypatch):
    FusedT, FusedL, _, Torch, Linear = _mods()
    monkeypatch.setenv("EVAC_POLICY_TC", tc)   # read at evac_policy_create: "0" keeps the heads on the CUDA cores
    if kind == "transformer":
        net = _transformer(60, 6, 0.1, seed=A * 100 + NH, action_dim=A, num_hidden=NH)
        fused, K = FusedT(net, 60, device="cuda", seed=SEED, env_index_offset=ENV_OFFSET), 372
    else:
        K = int(kind[len("linear"):])
        torch.manual_seed(A * 100 + NH)
        net = _perturb(Linear(K, action_dim=A, num_hidden=NH), A + NH)
        fused = FusedL(net, K, device="cuda", seed=SEED, env_index_offset=ENV_OFFSET)
    x = (torch.randn(E, K, generator=torch.Generator().manual_seed(E)) * 0.7).clamp_(-1, 1).cuda()
    fused.calls.fill_(2 ** 32 - 1)   # the two calls straddle the carry into the offset's upper word
    ls = net.actor_logstd.detach().double().flatten().numpy()
    sd = np.exp(ls)
    env_g = (ENV_OFFSET + np.arange(E)) & 0xFFFFFFFF
    means = []
    for off in (2 ** 32 - 1, 2 ** 32):
        o = {k: torch.empty(s, device="cuda") for k, s in (("mean", (E, A)), ("action", (E, A)), ("action_clipped", (E, A)),
                                                            ("logprob", (E,)), ("entropy", (E,)))}
        fused.forward(x, **o)
        torch.cuda.synchronize()
        mean, act = o["mean"].cpu().double().numpy(), o["action"].cpu().double().numpy()
        z, rad = T.policy_normal(SEED, off, env_g, A)
        err = np.abs((act - mean) - sd * z)
        bar = _sampling_bar(sd, rad, act)
        assert (err <= bar).all(), (off, float((err / bar).max()), np.argwhere(err > bar)[:5])
        zk = (act - mean) / sd
        np.testing.assert_allclose(o["logprob"].cpu().numpy(), (-0.5 * zk ** 2 - ls - HALF_LOG_2PI).sum(1), rtol=1e-5, atol=1e-5)
        np.testing.assert_allclose(o["entropy"].cpu().numpy(), np.full(E, (0.5 + HALF_LOG_2PI + ls).sum()), rtol=1e-6, atol=1e-6)
        assert torch.equal(o["action_clipped"], o["action"].clamp(-1, 1))
        means.append(o["mean"])
    assert int(fused.calls) == 2 ** 32 + 1
    if kind != "transformer":   # no dropout: the same means on both calls, only the draws moved
        assert torch.equal(means[0], means[1])


# ---------------------------------------------------------------------------------------------------------------------------
# (c) the production loop, replayed
def test_graph_captured_rollout_replays_from_its_stored_observations():
    """PolicyRollout(use_graph=True, store=True) with the training-mode transformer policy, an auto-reset inside the run: for every
    step t the stored normalised observation, the call index t, the restated masks and the restated Normal draw give the stored
    value, action and log-probability in float64 -- every replay advanced the counter, and the stored observation is the one the
    policy saw."""
    import evacuation_b200 as eb

    FusedT, _, Rollout, _, _ = _mods()
    E, N, Tn = 64, 60, 8
    env = eb.setup_env(eb.EnvConfig(number_of_pedestrians=N, max_timesteps=5), eb.EnvWrappersConfig(positions="rel", statuses="ohe", type="Box"),
                       num_envs=E, seed=5, auto_reset=True)
    net = _transformer(N, 6, 0.1, seed=21)
    pol = FusedT(net, N, device="cuda", seed=SEED, env_index_offset=ENV_OFFSET)
    ro = Rollout(env, pol, use_graph=True, store=True)
    ro.reset()
    buf = ro.run(Tn)
    torch.cuda.synchronize()
    assert int(pol.calls) == Tn
    # the 5th step truncates every episode and resets it in the same step: steps 5 .. 7 see fresh episodes
    assert bool((buf["dones"][:5] == 0).all()) and bool((buf["dones"][5] == 1).all())
    ls = net.actor_logstd.detach().double().flatten().numpy()
    sd = np.exp(ls)
    env_g = (ENV_OFFSET + np.arange(E)) & 0xFFFFFFFF
    errs = []
    for t in range(Tn):
        obs = buf["obs"][t]
        assert float(obs.abs().max()) <= 1.0
        masks = T.dropout_masks(SEED, t, ENV_OFFSET, E, 2, N + 2, 6, 96, 0.1)
        _, m64, v64 = (v.numpy() for v in _masked_forward(net, obs, masks, torch.float64))
        _, m32, v32 = (v.numpy() for v in _masked_forward(net, obs, masks, torch.float32))
        errs.append(_within(buf["values"][t].cpu().numpy(), v64, v32, 2e-5 * (1 + np.abs(v64)), f"value, step {t}"))
        z, rad = T.policy_normal(SEED, t, env_g, 2)
        act = buf["actions"][t].cpu().double().numpy()
        _within(act, m64 + sd * z, m32 + sd * z, 2e-5 + _sampling_bar(sd, rad, act), f"action, step {t}")
        lp64 = (-0.5 * z ** 2 - ls - HALF_LOG_2PI).sum(1)
        lp_bar = (2e-6 * (1 + rad) * (1 + np.abs(z))).sum(1) + 1e-5 * (1 + np.abs(lp64))
        lp = buf["logprobs"][t].cpu().double().numpy()
        assert (np.abs(lp - lp64) <= lp_bar).all(), (t, float(np.abs(lp - lp64).max()))
    print("value vs float64 per step (max, median):", ", ".join(f"({a:.3g}, {b:.3g})" for a, b in errs))
