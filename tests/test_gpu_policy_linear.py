"""GPU tests of the fused linear RPO policy (num_blocks = 0: RPOLinearNetwork, rpo_linear_agent_network.py:19-61, on the
flattened observation; csrc/evac_policy.cuh / evac_policy_tc.cuh through `evac_policy_forward`) against its plain-PyTorch
restatement `RPOLinearPolicy`, whose heads are the code `tests/test_rollout_cpu.py` pins to the reference golden through
`RPOTransformerPolicy`.  Float64 bars are those of test_gpu_policy.py::test_heads_on_tensor_cores_match_the_cuda_core_path_and_float64,
the normaliser bars those of test_gpu_policy.py::test_fused_normalizer_prologue_matches_vector_normalizer.

Shapes: grav K = 6 (CUDA cores), Dict rel + ohe N = 60 K = 364 and Box rel + ohe N = 60 K = 372 (tensor cores), Dict abs + cat
N = 7 K = 25 (CUDA cores), K = 1 (the smallest accepted; K = 0 raises)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _mods():
    from evacuation_b200.rollout import FusedRPOLinearPolicy, PolicyRollout, RPOLinearPolicy, VectorNormalizer, normalize_reward_fused
    return FusedRPOLinearPolicy, PolicyRollout, RPOLinearPolicy, VectorNormalizer, normalize_reward_fused


def _net(K, seed=0, **kw):
    _, _, Torch, _, _ = _mods()
    torch.manual_seed(seed)
    net = Torch(K, **kw).cuda().eval()
    with torch.no_grad():  # non-trivial biases and log-std (the defaults are 0)
        for name, p in net.named_parameters():
            if name.endswith("bias") or name == "actor_logstd":
                p.add_(0.3 * torch.randn_like(p))
    return net


def _run(net, K, x, tc, monkeypatch, seed=7, **fwd):
    """mean, value, action, logprob of one fused forward; EVAC_POLICY_TC=0 (read at evac_policy_create) keeps the heads on the
    CUDA cores."""
    Fused = _mods()[0]
    monkeypatch.setenv("EVAC_POLICY_TC", tc)
    fused = Fused(net, K, device="cuda", seed=seed).eval()
    E, A = x.shape[0], net.actor_mean[4].out_features
    o = dict(mean=torch.empty((E, A), device="cuda"), value=torch.empty(E, device="cuda"), action=torch.empty((E, A), device="cuda"),
             logprob=torch.empty(E, device="cuda"))
    fused.forward(x, **o, **fwd)
    torch.cuda.synchronize()
    return o


def _check_float64(net, x, o):
    net64 = _mods()[2](x.shape[1], action_dim=net.actor_mean[4].out_features, num_hidden=net.critic[0].out_features).double().cuda().eval()
    net64.load_state_dict({k: v.double() for k, v in net.state_dict().items()})
    with torch.no_grad():
        mean64, val64 = net64.actor_mean(x.double()), net64.critic(x.double()).flatten()
    assert float((o["mean"].double() - mean64).abs().max()) < 2e-6
    assert float((o["value"].double() - val64).abs().max() / val64.abs().max().clamp_min(1.0)) < 6e-6


SHAPES = [(6, {}), (364, {}), (372, {}), (25, {}), (1, {}), (364, dict(num_hidden=12)), (364, dict(num_hidden=32)),
          (6, dict(num_hidden=12)), (6, dict(action_dim=1)), (364, dict(action_dim=3)), (25, dict(action_dim=3, num_hidden=32))]


@pytest.mark.parametrize("K,kw", SHAPES)
def test_linear_heads_match_float64_on_both_kernels(K, kw, monkeypatch):
    net = _net(K, seed=K, **kw)
    x = (torch.randn(129, K, device="cuda") * 0.7).clamp_(-1, 1)
    outs = {tc: _run(net, K, x, tc, monkeypatch) for tc in ("1", "0")}
    for tc in ("1", "0"):
        _check_float64(net, x, outs[tc])
    # the sampled action is mean + std * noise with noise keyed by (seed, call, env): identical streams on both kernels
    np.testing.assert_allclose(outs["1"]["action"].cpu().numpy(), outs["0"]["action"].cpu().numpy(), rtol=0, atol=2e-6)
    np.testing.assert_allclose(outs["1"]["logprob"].cpu().numpy(), outs["0"]["logprob"].cpu().numpy(), rtol=0, atol=2e-5)


@pytest.mark.parametrize("K", [6, 364])
@pytest.mark.parametrize("E", [1, 5, 129, 4096, 38000])
def test_linear_heads_batch_sizes(K, E, monkeypatch):
    """E = 38000 crosses the tensor-core kernel's switch from 64- to 128-column tiles (296 row tiles)."""
    net = _net(K, seed=3)
    x = (torch.randn(E, K, device="cuda") * 0.7).clamp_(-1, 1)
    outs = {tc: _run(net, K, x, tc, monkeypatch) for tc in ("1", "0")}
    for tc in ("1", "0"):
        _check_float64(net, x, outs[tc])
    np.testing.assert_allclose(outs["1"]["action"].cpu().numpy(), outs["0"]["action"].cpu().numpy(), rtol=0, atol=2e-6)


@pytest.mark.parametrize("K,E,tc", [
    (364, 50, "1"),       # tensor cores, a batch the normaliser-free kernel runs in 64-column tiles
    (364, 38000, "1"),    # tensor cores, a batch the normaliser-free kernel runs in 128-column tiles
    (372, 4096, "1"),
    (364, 50, "0"), (364, 38000, "0"),   # CUDA cores
    (6, 4096, "1"), (25, 129, "1"), (1, 40, "1"),   # K not a multiple of 4: CUDA cores either way
])
def test_fused_normalizer_matches_vector_normalizer(K, E, tc, monkeypatch):
    """NormalizeObservation + clip fused into the heads' X load == VectorNormalizer.observation over 12 calls with drifting
    inputs: the normalised observation, the statistics (a double or racing update would move them) and the count; the heads
    see the normalised observation."""
    Fused, _, _, Norm, _ = _mods()
    net = _net(K, seed=5)
    monkeypatch.setenv("EVAC_POLICY_TC", tc)
    fused = Fused(net, K, device="cuda", seed=1).eval()
    n_ref, n_fused = Norm(E, K, device="cuda"), Norm(E, K, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(0)
    for t in range(12):
        raw = torch.randn(E, K, device="cuda", generator=g) * (1 + t) + 0.5
        want = n_ref.observation(raw)
        got, mean, val = torch.empty_like(raw), torch.empty((E, 2), device="cuda"), torch.empty(E, device="cuda")
        fused.forward(raw, normalizer=n_fused, obs_norm=got, mean=mean, value=val, sample=False)
        torch.testing.assert_close(got, want, rtol=0, atol=1e-6)
        torch.testing.assert_close(n_fused.obs_mean, n_ref.obs_mean, rtol=1e-6, atol=1e-7)
        torch.testing.assert_close(n_fused.obs_var, n_ref.obs_var, rtol=1e-6, atol=1e-7)
        assert float(n_fused.obs_count) == float(n_ref.obs_count)
        with torch.no_grad():
            torch.testing.assert_close(mean, net.actor_mean(want), rtol=0, atol=2e-5)
            torch.testing.assert_close(val, net.critic(want).flatten(), rtol=1e-5, atol=8e-5)


def test_fused_normalizer_without_head_outputs_still_updates():
    Fused, _, _, Norm, _ = _mods()
    net = _net(364, seed=2)
    fused = Fused(net, 364, device="cuda").eval()
    n_ref, n_fused = Norm(70, 364, device="cuda"), Norm(70, 364, device="cuda")
    raw = torch.randn(70, 364, device="cuda") * 2
    want, got = n_ref.observation(raw), torch.empty_like(raw)
    fused.forward(raw, normalizer=n_fused, obs_norm=got)
    torch.testing.assert_close(got, want, rtol=0, atol=1e-6)
    torch.testing.assert_close(n_fused.obs_mean, n_ref.obs_mean, rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("K", [6, 364])
def test_linear_sampling_statistics_logprob_and_streams(K):
    Fused = _mods()[0]
    net = _net(K, seed=9)
    fused = Fused(net, K, device="cuda", seed=7).eval()
    E = 20000
    x = (torch.randn(E, K, device="cuda") * 0.7).clamp_(-1, 1)
    mean, act, clip, lp, ent, val = (torch.empty(s, device="cuda") for s in ((E, 2), (E, 2), (E, 2), (E,), (E,), (E,)))
    fused.forward(x, mean=mean, action=act, action_clipped=clip, logprob=lp, entropy=ent, value=val)
    std = torch.exp(net.actor_logstd.detach()).expand_as(mean)
    zs = ((act - mean) / std).cpu().numpy()
    assert abs(zs.mean()) < 0.03 and abs(zs.std() - 1.0) < 0.03 and abs(np.corrcoef(zs[:, 0], zs[:, 1])[0, 1]) < 0.03
    assert abs((np.abs(zs) > 1.96).mean() - 0.05) < 0.01
    dist = torch.distributions.Normal(mean, std)
    np.testing.assert_allclose(lp.cpu().numpy(), dist.log_prob(act).sum(1).cpu().numpy(), rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(ent.cpu().numpy(), dist.entropy().sum(1).cpu().numpy(), rtol=1e-6)
    assert torch.equal(clip, act.clamp(-1, 1))
    # the device-side call counter advances the stream: a second call draws different numbers, same means
    act2, mean2 = torch.empty_like(act), torch.empty_like(mean)
    fused.forward(x, mean=mean2, action=act2)
    assert torch.equal(mean, mean2) and not torch.equal(act, act2)
    # same (seed, offset, global env index) -> same numbers, whatever the batch split (sharding invariance)
    fa = Fused(net, K, device="cuda", seed=7).eval()
    fb = Fused(net, K, device="cuda", seed=7, env_index_offset=100).eval()
    a_full, a_part = torch.empty((E, 2), device="cuda"), torch.empty((50, 2), device="cuda")
    fa.forward(x, action=a_full)
    fb.forward(x[100:150].contiguous(), action=a_part)
    assert torch.equal(a_full[100:150], a_part)
    # the module surface: get_value / get_action_and_value
    v = fa.get_value(x)
    with torch.no_grad():
        torch.testing.assert_close(v, net.critic(x), rtol=1e-5, atol=8e-5)
    a, lp2, ent2, v2 = fa.get_action_and_value(x, act)
    assert torch.equal(a, act) and torch.equal(v2, v)
    np.testing.assert_allclose(lp2.cpu().numpy(), dist.log_prob(act).sum(1).cpu().numpy(), rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("K", [6, 364])
def test_linear_nan_rows_propagate_to_their_env_only(K):
    Fused, _, _, Norm, _ = _mods()
    net = _net(K, seed=4)
    fused = Fused(net, K, device="cuda").eval()
    x = (torch.randn(40, K, device="cuda") * 0.5).clamp_(-1, 1)
    x[3, K // 2] = float("nan")
    mean, val = torch.empty((40, 2), device="cuda"), torch.empty(40, device="cuda")
    fused.forward(x, mean=mean, value=val, sample=False)
    bad = torch.zeros(40, dtype=torch.bool, device="cuda")
    bad[3] = True
    assert torch.equal(torch.isnan(mean).any(dim=1), bad) and torch.equal(torch.isnan(val), bad)
    with torch.no_grad():
        np.testing.assert_allclose(mean[~bad].cpu().numpy(), net.actor_mean(x[~bad]).cpu().numpy(), rtol=0, atol=2e-5)
    # through the fused normaliser: NaN enters the statistics of that element only, like VectorNormalizer
    n_ref, n_fused = Norm(40, K, device="cuda"), Norm(40, K, device="cuda")
    want, got = n_ref.observation(x), torch.empty_like(x)
    fused.forward(x, normalizer=n_fused, obs_norm=got, mean=mean, value=val, sample=False)
    torch.testing.assert_close(got, want, rtol=0, atol=1e-6, equal_nan=True)
    torch.testing.assert_close(n_fused.obs_mean, n_ref.obs_mean, rtol=1e-6, atol=1e-7, equal_nan=True)
    assert torch.equal(torch.isnan(mean).any(dim=1), bad) and torch.equal(torch.isnan(val), bad)


def _env(kind, E, seed):
    import evacuation_b200 as eb
    if kind == "grav":
        return eb.setup_env(eb.EnvConfig(number_of_pedestrians=60, is_new_exiting_reward=True), eb.EnvWrappersConfig(positions="grav", type="Dict"),
                            num_envs=E, seed=seed, auto_reset=True)
    return eb.setup_env(eb.EnvConfig(number_of_pedestrians=60, is_new_exiting_reward=True), eb.EnvWrappersConfig(positions="rel", statuses="ohe", type="Dict"),
                        num_envs=E, seed=seed, auto_reset=True)


@pytest.mark.parametrize("kind,K", [("grav", 6), ("dict", 364)])
def test_policy_rollout_with_the_fused_linear_policy(kind, K):
    """The loop of the gravity-encoding / flat-observation configs: heads with the fused normaliser -> env step -> reward
    normaliser, 3 library launches per iteration, CUDA-graph replayed; in eval mode with the mean as the action it retraces the
    PyTorch loop."""
    Fused, Rollout, Torch, Norm, norm_reward = _mods()
    E, T = 96, 20
    assert _env(kind, 1, 0).unwrapped.obs_dim == K
    torch.manual_seed(1)
    net = Torch(K).cuda()
    # (1) the production loop: graph-captured, sampling on
    pol = Fused(net, K, device="cuda", seed=1)
    env = _env(kind, E, 5)
    ro = Rollout(env, pol, use_graph=True, store=True)
    ro.reset()
    buf = ro.run(T)
    torch.cuda.synchronize()
    assert ro.launches_per_iteration == 3
    for k in ("obs", "actions", "logprobs", "rewards", "values", "dones"):
        assert torch.isfinite(buf[k]).all(), k
    assert float(buf["obs"].abs().max()) <= 1.0 and not torch.equal(buf["actions"][0], buf["actions"][1])
    # the capture's warm-up and recorded iterations do not advance the environments: the same run without the graph, bit for bit
    assert int(pol.calls) == T and abs(float(ro.norm.obs_count) - (1e-4 + T)) < 1e-9
    assert bool((buf["dones"][0] == 0).all())
    pol_e = Fused(net, K, device="cuda", seed=1)
    ro_e = Rollout(_env(kind, E, 5), pol_e, use_graph=False, store=True)
    ro_e.reset()
    buf_e = ro_e.run(T)
    for k in buf:
        assert torch.equal(buf[k], buf_e[k]), k
    # (2) eval-mode retrace against torch: same env seed, actions = clipped means
    env_a, env_b = _env(kind, E, 7), _env(kind, E, 7)
    fused = Fused(net, K, device="cuda").eval()
    net.eval()
    na, nb = Norm(E, K, device="cuda"), Norm(E, K, device="cuda")
    env_a.reset(); env_b.reset()
    oa, ob = env_a.unwrapped.flat_observation, env_b.unwrapped.flat_observation
    mean, val, clip, xn = torch.empty((E, 2), device="cuda"), torch.empty(E, device="cuda"), torch.empty((E, 2), device="cuda"), torch.empty((E, K), device="cuda")
    for t in range(15):
        fused.forward(oa, normalizer=na, obs_norm=xn, mean=mean, value=val, action_clipped=clip, sample=False)
        with torch.no_grad():
            xb = nb.observation(ob)
            mb = net.actor_mean(xb)
        np.testing.assert_allclose(xn.cpu().numpy(), xb.cpu().numpy(), rtol=0, atol=2e-6)
        np.testing.assert_allclose(mean.cpu().numpy(), mb.cpu().numpy(), rtol=0, atol=2e-5)
        assert torch.equal(clip, mean.clamp(-1, 1))
        act = mb.clamp(-1, 1).contiguous()  # both envs take the SAME action so that the traces stay comparable
        _, ra, ta, _, _ = env_a.step(act)
        _, rb, tb, _, _ = env_b.step(act)
        assert torch.equal(oa, ob) and torch.equal(ra, rb)
        got_r = norm_reward(na, ra, ta, torch.empty(E, device="cuda"))
        np.testing.assert_allclose(got_r.cpu().numpy(), nb.reward(rb, tb).cpu().numpy(), rtol=1e-6, atol=1e-7)


def test_rollout_capture_does_not_advance_the_environments_linear():
    """After reset() the first run(T) of the graph-captured loop records exactly T transitions from the reset state."""
    Fused, Rollout, Torch, _, _ = _mods()
    E, T = 6, 5
    env = _env("dict", E, 4)
    torch.manual_seed(3)
    pol = Fused(Torch(364).cuda(), 364, device="cuda", seed=9).eval()
    ro = Rollout(env, pol, use_graph=True, store=True)
    ro.reset()
    ro.run(T)
    st = env.unwrapped.get_state()
    assert bool((st["now"] == T).all()), st["now"]
    assert int(pol.calls) == T and abs(float(ro.norm.ret_count) - (1e-4 + T)) < 1e-9


def test_unsupported_linear_policies_raise():
    Fused, _, Torch, _, _ = _mods()
    with pytest.raises(NotImplementedError):
        Fused(Torch(4097), 4097, device="cuda")      # wider than the 4096-float limit
    with pytest.raises(NotImplementedError):
        Fused(Torch(0), 0, device="cuda")            # below the smallest accepted width (1)
    with pytest.raises(NotImplementedError):
        Fused(Torch(364, num_hidden=128), 364, device="cuda")
    with pytest.raises(NotImplementedError):
        Fused(Torch(364, action_dim=4), 364, device="cuda")
    fused = Fused(Torch(364).cuda(), 364, device="cuda")
    x = torch.zeros(4, 364, device="cuda")
    with pytest.raises(ValueError):
        fused.forward(x, embedding=torch.empty_like(x))
    with pytest.raises(ValueError):
        fused.forward(torch.zeros(4, 372, device="cuda"))
