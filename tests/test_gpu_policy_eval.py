"""GPU tests of evaluation with a trained fused policy: the frozen observation normaliser of `evac_policy_forward`
(`EvacPolicyIO.norm_frozen`, `forward(norm_update=False)`) on every heads kernel and the embedding kernel, and
`rollout.evaluate_policy` / `EvacuationEnv.efficiency_curve(agent=policy)` on every kind of handle.

(1) the frozen forward: statistics untouched, obs_norm = the frozen formula, embedding / mean / value bit-identical to the
    normaliser-free forward on that obs_norm, a NaN row confined to its environment, frozen + dropout refused;
(2) grav, N <= 64: evaluate_policy is the one-launch evaluation of evac_rollout_policy bit for bit;
(3) transformer and flat linear policy at N = 60, grav linear at N = 200 (CTA cell-list kernel): teacher-forced actions, the
    frozen formula on a replay's raw observations, a table-agent replay, the efficiency curve, nothing of the policy or the
    normaliser moved."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _mods():
    import evacuation_b200 as eb
    from evacuation_b200 import rollout as ro
    return eb, ro


def _lin(K, seed=0, **kw):
    torch.manual_seed(seed)
    net = _mods()[1].RPOLinearPolicy(K, **kw).cuda().eval()
    with torch.no_grad():  # non-trivial biases and log-std, a larger action spread
        for name, p in net.named_parameters():
            if name.endswith("bias") or name == "actor_logstd":
                p.add_(0.3 * torch.randn_like(p))
        net.actor_mean[4].weight.mul_(60.0)
    return net


def _tf(N, seed=0):
    torch.manual_seed(seed)
    net = _mods()[1].RPOTransformerPolicy(6 * (N + 2), N).cuda()
    with torch.no_grad():
        net.actor_mean[4].weight.mul_(60.0)
    return net


def _frozen_normalizer(E, K, seed):
    n = _mods()[1].VectorNormalizer(E, K, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(seed)
    n.obs_mean.copy_(torch.randn(E, K, device="cuda", generator=g) * 0.3)
    n.obs_var.copy_(torch.rand(E, K, device="cuda", generator=g) * 2 + 0.05)
    n.obs_count.fill_(123.0)
    return n


def _stats(n):
    return n.obs_mean.clone(), n.obs_var.clone(), n.obs_count.clone()


def _same_stats(n, saved):
    return torch.equal(n.obs_mean, saved[0]) and torch.equal(n.obs_var, saved[1]) and torch.equal(n.obs_count, saved[2])


def _want(raw, saved, eps):
    return ((raw - saved[0]) * torch.rsqrt(saved[1] + eps)).clamp(-1, 1)


def _policy(kind, K, monkeypatch, tc):
    """(fused policy, torch module); EVAC_POLICY_TC is read at evac_policy_create: 0 = CUDA-core heads, 128 = 128-column tiles."""
    _, ro = _mods()
    monkeypatch.setenv("EVAC_POLICY_TC", tc)
    if kind == "tf":
        net = _tf(60, seed=K)
        return ro.FusedRPOTransformerPolicy(net, 60, device="cuda", seed=3).eval(), net
    net = _lin(K, seed=K)
    return ro.FusedRPOLinearPolicy(net, K, device="cuda", seed=3), net


FORWARD = [  # (policy, K, E, EVAC_POLICY_TC)
    ("tf", 372, 257, "1"),      # embedding kernel + tensor-core heads
    ("tf", 372, 257, "0"),      # embedding kernel + CUDA-core heads
    ("lin", 364, 50, "1"),      # tensor cores, 64-column tiles (below 296 row tiles)
    ("lin", 364, 38000, "1"),   # tensor cores, 128-column tiles
    ("lin", 364, 50, "128"),    # tensor cores, 128-column tiles pinned at a small batch
    ("lin", 364, 50, "0"),      # CUDA cores
    ("lin", 25, 129, "1"),      # K not a multiple of 4: CUDA cores
    ("lin", 6, 129, "1"),
]


@pytest.mark.parametrize("kind,K,E,tc", FORWARD)
def test_frozen_forward_reads_the_statistics_only(kind, K, E, tc, monkeypatch):
    pol, _ = _policy(kind, K, monkeypatch, tc)
    norm = _frozen_normalizer(E, K, seed=K)
    saved = _stats(norm)
    g = torch.Generator(device="cuda").manual_seed(E)
    raw = torch.randn(E, K, device="cuda", generator=g) * 1.5 + 0.2
    raw[1] = 0.0  # exact zeros and values far outside the clip
    raw[2] *= 50.0

    def run(x, normalizer=None):
        o = dict(mean=torch.empty(E, 2, device="cuda"), value=torch.empty(E, device="cuda"))
        if kind == "tf":
            o["embedding"] = torch.empty(E, K, device="cuda")
        on = torch.empty(E, K, device="cuda") if normalizer is not None else None
        calls = pol.calls.clone()
        pol.forward(x, normalizer=normalizer, obs_norm=on, sample=False, norm_update=False, advance=False, **o)
        torch.cuda.synchronize()
        assert torch.equal(pol.calls, calls)
        return on, o

    on, got = run(raw, norm)
    assert _same_stats(norm, saved)
    assert float((on - _want(raw, saved, norm.epsilon)).abs().max()) <= 2e-6
    _, ref = run(on)
    for k in got:
        assert torch.equal(got[k], ref[k]), k
    # a NaN observation value: NaN in its obs_norm, no finite mean of its environment, every other environment as before
    bad = raw.clone()
    bad[3, K // 2] = float("nan")
    on_b, got_b = run(bad, norm)
    assert _same_stats(norm, saved)
    assert bool(torch.isnan(on_b[3, K // 2]))
    assert not bool(torch.isfinite(got_b["mean"][3]).any())
    keep = torch.ones(E, dtype=torch.bool, device="cuda")
    keep[3] = False
    assert torch.equal(on_b[keep], on[keep])
    for k in got:
        assert torch.equal(got_b[k][keep], got[k][keep]), k
    if kind == "tf":  # evaluation runs without dropout
        pol.train()
        with pytest.raises(NotImplementedError):
            pol.forward(raw, normalizer=norm, mean=torch.empty(E, 2, device="cuda"), sample=False, norm_update=False)
        assert _same_stats(norm, saved)


def _grav_env(E, N, seed, auto_reset, max_timesteps):
    eb, _ = _mods()
    cfg = eb.EnvConfig(number_of_pedestrians=N, is_new_exiting_reward=True, is_termination_agent_wall_collision=True, max_timesteps=max_timesteps)
    return eb.setup_env(cfg, eb.EnvWrappersConfig(positions="grav", type="Dict"), num_envs=E, seed=seed, auto_reset=auto_reset,
                        batched=True, rng="philox")


def _image(u):
    """save_state() into a zeroed buffer (the image's padding is left as the buffer found it)"""
    from evacuation_b200 import _native as nat
    img = torch.zeros(int(nat.load().evac_state_bytes(u._handle())), dtype=torch.uint8, device=u.device)
    nat.check(nat.load().evac_save_state(u._handle(), img.data_ptr(), u._stream()))
    return img


def _outputs(T, E, K):
    return dict(obs_norm=torch.empty(T, E, K, device="cuda"), action=torch.empty(T, E, 2, device="cuda"),
                status_counts=torch.empty(T, E, 4, dtype=torch.int16, device="cuda"))


@pytest.mark.parametrize("N,per_env,with_norm,auto_reset", [(60, False, True, True), (60, True, True, False), (33, True, False, True),
                                                            (1, False, True, False), (1, True, False, True)])
def test_grav_evaluation_is_the_one_launch_evaluation_bit_for_bit(N, per_env, with_norm, auto_reset):
    _, ro = _mods()
    E, T = 96, 40
    net = _lin(6, seed=N)
    pol = ro.FusedRPOLinearPolicy(net, 6, device="cuda", seed=4, env_index_offset=9)
    envs = [_grav_env(E, N, seed=N, auto_reset=auto_reset, max_timesteps=23 if auto_reset else 500) for _ in range(2)]
    for env in envs:
        if per_env:
            r = np.random.RandomState(E)
            env.unwrapped.set_env_params(alpha=r.choice([2.0, 3.0, 2.5], E), noise_coef=r.uniform(0.05, 0.6, E),
                                         max_timesteps=r.randint(5, 40, E))
        env.unwrapped.reset()
    a, b = envs[0].unwrapped, envs[1].unwrapped
    b.load_state(a.save_state())
    b.flat_observation.copy_(a.flat_observation)
    norm = _frozen_normalizer(E, 6, seed=N) if with_norm else None
    saved = None if norm is None else _stats(norm)
    oa, ob = _outputs(T, E, 6), _outputs(T, E, 6)
    ro.fused_policy_rollout(envs[0], pol, T, torch.zeros(E, device="cuda"), normalizer=norm, norm_update=False, normalize_reward=False,
                            sample=False, **oa)
    calls = pol.calls.clone()
    ro.evaluate_policy(envs[1], pol, T, normalizer=norm, **ob)
    torch.cuda.synchronize()
    for k in oa:
        assert torch.equal(oa[k], ob[k]), k
    assert torch.equal(_image(a), _image(b)) and torch.equal(a.flat_observation, b.flat_observation)
    assert torch.equal(pol.calls, calls)
    if norm is not None:
        assert _same_stats(norm, saved)


EVAL = [  # (policy, N, wrappers)
    ("tf", 60, dict(positions="rel", statuses="ohe", type="Box")),    # K = 372: embedding + tensor-core heads, one-warp step
    ("lin", 60, dict(positions="rel", statuses="ohe", type="Dict")),  # K = 364: tensor-core heads
    ("lin", 200, dict(positions="grav", type="Dict")),                # K = 6 on the CTA cell-list step kernel
]


@pytest.mark.parametrize("kind,N,wrap", EVAL)
def test_evaluation_is_teacher_forced_and_replays_through_the_table_agent(kind, N, wrap):
    eb, ro = _mods()
    E, T = 96, 40
    cfg = eb.EnvConfig(number_of_pedestrians=N, is_new_exiting_reward=True, max_timesteps=500)
    make = lambda: eb.setup_env(cfg, eb.EnvWrappersConfig(**wrap), num_envs=E, seed=21, auto_reset=False, batched=True, rng="philox")
    env = make()
    u = env.unwrapped
    K = u.obs_dim
    if kind == "tf":
        net = _tf(N, seed=1)
        pol = ro.FusedRPOTransformerPolicy(net, N, device="cuda", seed=4)   # training mode, as the reference leaves it
    else:
        net = _lin(K, seed=1)
        pol = ro.FusedRPOLinearPolicy(net, K, device="cuda", seed=4)
    assert pol.training
    u.reset()
    start, obs0 = u.save_state().clone(), u.flat_observation.clone()
    norm = _frozen_normalizer(E, K, seed=2)
    saved, calls = _stats(norm), pol.calls.clone()
    o = _outputs(T, E, K)
    ro.evaluate_policy(env, pol, T, normalizer=norm, **o)
    torch.cuda.synchronize()
    final_obs, final_image = u.flat_observation.clone(), _image(u)
    assert _same_stats(norm, saved) and torch.equal(pol.calls, calls) and pol.training
    # the actions: the actor mean of evac_policy_forward (training off, no normaliser) on the stored obs_norm, step by step (the
    # tensor-core tiling follows the batch size), bit for bit
    pol.eval()
    for t in range(T):
        mean = torch.empty(E, 2, device="cuda")
        pol.forward(o["obs_norm"][t], mean=mean, sample=False, advance=False)
        assert torch.equal(mean, o["action"][t]), t
        assert torch.equal(mean.clamp(-1, 1), o["action"][t].clamp(-1, 1))
    pol.train()
    # the observations: the frozen formula on a per-step replay's raw observations (step 0: the reset observation); the capture of
    # the graph did not advance the environments, so the replay from `start` is the evaluated trajectory
    acts = o["action"].clamp(-1, 1).contiguous()
    u.load_state(start)
    u.flat_observation.copy_(obs0)
    raw = torch.empty(T, E, K, device="cuda")
    raw[0] = obs0
    for t in range(T - 1):
        u.rollout(1, agent="table", actions=acts[t:t + 1])
        raw[t + 1] = u.flat_observation
    assert float((o["obs_norm"] - _want(raw, saved, norm.epsilon)).abs().max()) <= 2e-6
    # the env: the clipped actions through the table agent reproduce counts, state image and final observation
    u.load_state(start)
    u.rollout(T, agent="table", actions=acts, status_counts=True)
    assert torch.equal(u.last_status_counts, o["status_counts"])
    assert torch.equal(_image(u), final_image) and torch.equal(u.flat_observation, final_obs)
    # efficiency_curve(agent=policy) from a fresh reset, in chunks, equals the curve of that replay
    esc = o["status_counts"][:, :, 0].to(torch.float64)
    mean_c, std_c = make().unwrapped.efficiency_curve(T, agent=pol, normalizer=norm, chunk=16)
    assert torch.equal(mean_c, esc.mean(dim=1)) and torch.equal(std_c, esc.std(dim=1, unbiased=False))
    assert _same_stats(norm, saved) and torch.equal(pol.calls, calls) and pol.training
