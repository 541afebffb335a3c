"""GPU tests of `evac_rollout_policy` (`PolicyRollout.run(T, steps_per_launch=K)`, `EvacuationEnv.efficiency_curve(agent=policy)`):
the gravity-encoding rollout loop with the fused linear policy as the agent of the one-warp step kernel, K iterations per launch.

(a) bit-identity with the CUDA-graph loop of three library launches per step (heads + fused normaliser, env step, reward
    normaliser) on every storage tensor, the carried state, both normalisers, both counts, the policy's call counter, the env's
    checkpoint image, episode statistics and the last observation;
(b) evaluation (sample = 0, frozen normaliser) teacher-forced against evac_policy_forward, the frozen normaliser restated in torch
    and a replay of the recorded clipped actions through evac_rollout(agent="table");
(c) the refusals."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _mods():
    import evacuation_b200 as eb
    from evacuation_b200.rollout import FusedRPOLinearPolicy, PolicyRollout, RPOLinearPolicy, VectorNormalizer, fused_policy_rollout
    return eb, FusedRPOLinearPolicy, PolicyRollout, RPOLinearPolicy, VectorNormalizer, fused_policy_rollout


def _env(E, N, seed=5, search="auto", max_timesteps=23, env_index_offset=0, auto_reset=True, **wrap):
    eb = _mods()[0]
    wrap = wrap or dict(positions="grav", type="Dict")
    cfg = eb.EnvConfig(number_of_pedestrians=N, is_new_exiting_reward=True, is_termination_agent_wall_collision=True,
                       max_timesteps=max_timesteps)
    return eb.setup_env(cfg, eb.EnvWrappersConfig(**wrap), num_envs=E, seed=seed, auto_reset=auto_reset, neighbor_search=search,
                        env_index_offset=env_index_offset, batched=True, rng="philox")


def _net(NH, seed=0, **kw):
    torch.manual_seed(seed)
    net = _mods()[3](6, num_hidden=NH, **kw).cuda()
    with torch.no_grad():  # non-trivial biases, a larger action spread (agent-wall terminations) and log-std
        for name, p in net.named_parameters():
            if name.endswith("bias") or name == "actor_logstd":
                p.add_(0.3 * torch.randn_like(p))
        net.actor_mean[4].weight.mul_(60.0)
    return net


def _per_env(env, E):
    r = np.random.RandomState(E)
    env.unwrapped.set_env_params(alpha=r.choice([2.0, 3.0, 2.5], E), noise_coef=r.uniform(0.05, 0.6, E),
                                 max_timesteps=r.randint(5, 40, E))


def _image(u):
    """save_state() into a zeroed buffer: the image rounds each region up to 16 bytes, and save_state leaves that padding as
    torch.empty found it"""
    from evacuation_b200 import _native as nat
    img = torch.zeros(int(nat.load().evac_state_bytes(u._handle())), dtype=torch.uint8, device=u.device)
    nat.check(nat.load().evac_save_state(u._handle(), img.data_ptr(), u._stream()))
    return img


def _state(ro):
    u = ro.env.unwrapped
    n = ro.norm
    stats, fin, tot = u.episode_statistics()
    return dict(next_done=ro.next_done, obs_mean=n.obs_mean, obs_var=n.obs_var, obs_count=n.obs_count, returns=n.returns,
                ret_mean=n.ret_mean, ret_var=n.ret_var, ret_count=n.ret_count, calls=ro.policy.calls, image=_image(u),
                stats=stats, fin=fin, tot=tot, obs=u.flat_observation)


def _pair(E, N, NH, search, per_env, seed=5):
    _, Fused, Rollout, _, _, _ = _mods()
    net = _net(NH, seed=NH)
    ros = []
    for _ in range(2):
        env = _env(E, N, seed=seed, search=search, env_index_offset=1000)
        if per_env:
            _per_env(env, E)
        ro = Rollout(env, Fused(net, 6, device="cuda", seed=11, env_index_offset=77), use_graph=True, store=True)
        ro.reset()
        ros.append(ro)
    # the same image in both handles: pedestrian slots >= N of a fresh handle are never written by a reset and carry whatever the
    # allocation held; the step kernels read and write them back but never use them
    ros[1].env.unwrapped.load_state(ros[0].env.unwrapped.save_state())
    return ros


def _run_k(ro, T, K):
    """run(T) with K iterations per evac_rollout_policy launch (steps_per_launch = 1 selects the graph loop: K = 1 runs one-step
    launches of the fused kernel directly)."""
    return ro._run_fused(T, 1) if K == 1 else ro.run(T, steps_per_launch=K)


CASES = [  # (K, T, E, N, num_hidden, neighbour search, per-env parameters)
    (7, 24, 96, 60, 64, "auto", False),
    (1, 5, 1, 1, 12, "brute", False),
    (64, 131, 96, 33, 32, "cells", True),
    (7, 40, 4096, 64, 64, "cells", True),
    (64, 70, 4096, 60, 12, "brute", False),
    (7, 30, 1, 64, 32, "auto", True),
    (64, 100, 96, 60, 64, "brute", True),
]


@pytest.mark.parametrize("K,T,E,N,NH,search,per_env", CASES)
def test_fused_rollout_is_the_three_launch_loop_bit_for_bit(K, T, E, N, NH, search, per_env):
    ref, got = _pair(E, N, NH, search, per_env)
    # two consecutive runs each
    bufs_r = [ref.run(T), ref.run(T // 2 + 1)]
    bufs_g = [_run_k(got, T, K), _run_k(got, T // 2 + 1, K)]
    torch.cuda.synchronize()
    assert ref.launches_per_iteration == 3
    for br, bg in zip(bufs_r, bufs_g):
        for k in br:
            assert torch.equal(br[k], bg[k]), k
    sr, sg = _state(ref), _state(got)
    for k in sr:
        assert torch.equal(sr[k], sg[k]), k
    if E > 1:  # the loop reached terminations / truncations: auto-resets inside launches
        assert float(bufs_r[0]["dones"].sum()) > 0 and int(sr["tot"][0]) > 0


def test_switching_paths_mid_run_continues_the_trajectory():
    ref, got = _pair(96, 60, 64, "auto", True, seed=8)
    a = [ref.run(9), ref.run(13), ref.run(20)]
    b = [got.run(9, steps_per_launch=4), got.run(13), got.run(20, steps_per_launch=64)]
    torch.cuda.synchronize()
    for br, bg in zip(a, b):
        for k in br:
            assert torch.equal(br[k], bg[k]), k
    sr, sg = _state(ref), _state(got)
    for k in sr:
        assert torch.equal(sr[k], sg[k]), k


def test_store_off_keeps_the_same_state_and_launch_counts():
    ref, got = _pair(96, 60, 64, "auto", False)
    got.store = False
    ref.run(30)
    u = got.env.unwrapped
    before = u.launch_count
    assert got.run(30, steps_per_launch=16) is None
    assert u.launch_count - before == 2 * 2  # two launches of 16 + 14 steps, each the step kernel + the counter kernel
    sr, sg = _state(ref), _state(got)
    for k in sr:
        assert torch.equal(sr[k], sg[k]), k


def _frozen_normalizer(E, seed):
    Norm = _mods()[4]
    n = Norm(E, 6, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(seed)
    n.obs_mean.copy_(torch.randn(E, 6, device="cuda", generator=g) * 0.3)
    n.obs_var.copy_(torch.rand(E, 6, device="cuda", generator=g) * 2 + 0.05)
    n.obs_count.fill_(123.0)
    return n


@pytest.mark.parametrize("NH,with_norm", [(64, True), (32, False)])
def test_evaluation_is_teacher_forced_and_replays_through_the_table_agent(NH, with_norm):
    eb, Fused, _, _, _, rollout = _mods()
    E, N, T = 257, 60, 90
    net = _net(NH, seed=3)
    pol = Fused(net, 6, device="cuda", seed=4, env_index_offset=9).eval()
    env = _env(E, N, seed=21, auto_reset=False, max_timesteps=500)
    u = env.unwrapped
    u.reset()
    start = u.save_state().clone()
    obs0 = u.flat_observation.clone()
    norm = _frozen_normalizer(E, 1) if with_norm else None
    frozen = None if norm is None else (norm.obs_mean.clone(), norm.obs_var.clone(), norm.obs_count.clone())
    o = dict(obs_norm=torch.empty(T, E, 6, device="cuda"), action=torch.empty(T, E, 2, device="cuda"), value=torch.empty(T, E, device="cuda"),
             status_counts=torch.empty(T, E, 4, dtype=torch.int16, device="cuda"))
    next_done = torch.zeros(E, device="cuda")
    rollout(env, pol, T, next_done, normalizer=norm, norm_update=False, normalize_reward=False, sample=False, **o)
    torch.cuda.synchronize()
    final_obs, final_image = u.flat_observation.clone(), _image(u)
    if norm is not None:  # frozen: nothing moved
        assert torch.equal(norm.obs_mean, frozen[0]) and torch.equal(norm.obs_var, frozen[1]) and torch.equal(norm.obs_count, frozen[2])
    # the heads: evac_policy_forward without a normaliser on the recorded obs_norm, bit for bit (the same CUDA-core sums)
    ref = Fused(net, 6, device="cuda", seed=4, env_index_offset=9).eval()
    x = o["obs_norm"].reshape(T * E, 6).contiguous()
    mean, value = torch.empty(T * E, 2, device="cuda"), torch.empty(T * E, device="cuda")
    ref.forward(x, mean=mean, value=value, sample=False)
    assert torch.equal(mean.view(T, E, 2), o["action"]) and torch.equal(value.view(T, E), o["value"])
    # the observations: the frozen formula on the replayed raw observation (step 0: the reset observation)
    acts = o["action"].clamp(-1, 1).contiguous()
    u.load_state(start)
    u.flat_observation.copy_(obs0)
    raw = torch.empty(T, E, 6, device="cuda")
    raw[0] = obs0
    for t in range(T - 1):  # per-step replay for the raw observation sequence (same kernel as a rollout of one step)
        u.rollout(1, agent="table", actions=acts[t:t + 1])
        raw[t + 1] = u.flat_observation
    if norm is None:
        assert torch.equal(o["obs_norm"], raw)
    else:
        want = ((raw - frozen[0]) * torch.rsqrt(frozen[1] + norm.epsilon)).clamp(-1, 1)
        assert float((o["obs_norm"] - want).abs().max()) < 2e-6
    # the env: replaying the clipped actions through the table agent reproduces counts, state image and final observation
    u.load_state(start)
    u.rollout(T, agent="table", actions=acts, status_counts=True)
    assert torch.equal(u.last_status_counts, o["status_counts"])
    assert torch.equal(_image(u), final_image) and torch.equal(u.flat_observation, final_obs)
    # efficiency_curve(agent=policy) from a fresh reset equals the curve of that replay
    esc = o["status_counts"][:, :, 0].to(torch.float64)
    env2 = _env(E, N, seed=21, auto_reset=False, max_timesteps=500)
    mean_c, std_c = env2.unwrapped.efficiency_curve(T, agent=pol, normalizer=norm, chunk=32)
    assert torch.equal(mean_c, esc.mean(dim=1)) and torch.equal(std_c, esc.std(dim=1, unbiased=False))
    assert float(mean_c[-1]) > 0


def test_refusals():
    eb, Fused, Rollout, Torch, Norm, rollout = _mods()
    E = 8
    net = _net(64)
    pol = Fused(net, 6, device="cuda")
    nd = torch.zeros(E, device="cuda")

    def call(env, p=pol, steps=3, **kw):
        env.reset()
        rollout(env, p, steps, nd, **kw)

    with pytest.raises(NotImplementedError):
        call(_env(E, 60, positions="rel", statuses="ohe", type="Box"))
    with pytest.raises(NotImplementedError):
        call(_env(E, 60, positions="rel", statuses="ohe", type="Dict"))
    with pytest.raises(NotImplementedError):
        call(_env(E, 65))
    env64 = eb.setup_env(eb.EnvConfig(number_of_pedestrians=60), eb.EnvWrappersConfig(positions="grav", type="Dict"), num_envs=E,
                         precision="fp64", auto_reset=True)
    with pytest.raises(NotImplementedError):
        call(env64)
    from evacuation_b200.rollout import FusedRPOTransformerPolicy, RPOTransformerPolicy
    torch.manual_seed(0)
    tf = FusedRPOTransformerPolicy(RPOTransformerPolicy(6 * 62, 60).cuda(), 60, device="cuda")
    with pytest.raises(NotImplementedError):
        call(_env(E, 60), p=tf)
    with pytest.raises(NotImplementedError):
        call(_env(E, 60), p=Fused(Torch(364).cuda(), 364, device="cuda"))
    for A in (1, 3):
        with pytest.raises(NotImplementedError):
            call(_env(E, 60), p=Fused(Torch(6, action_dim=A).cuda(), 6, device="cuda"))
    with pytest.raises(NotImplementedError):  # the torch policy has no one-launch path
        ro = Rollout(_env(E, 60), net, use_graph=False)
        ro.reset()
        ro.run(4, steps_per_launch=2)
    bad_e = Norm(E + 1, 6, device="cuda")
    with pytest.raises(ValueError):
        call(_env(E, 60), normalizer=bad_e)
    bad_t = Norm(E, 6, device="cuda", dtype=torch.float64)
    with pytest.raises(ValueError):
        call(_env(E, 60), normalizer=bad_t)
    with pytest.raises(ValueError):
        call(_env(E, 60), steps=0)
    ro = Rollout(_env(E, 60), pol, use_graph=False)
    ro.reset()
    with pytest.raises(ValueError):
        ro.run(0, steps_per_launch=4)
