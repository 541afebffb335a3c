"""Per-environment dynamics and reward parameters (EvacuationEnv.set_env_params, evac_set_env_params).

The random streams are keyed by (seed, global env index, episode, step), not by these parameters, so environment e of a
handle with per-env parameters must equal environment e of a uniform handle built with e's values (same E, seed and
env_index_offset) bit for bit: observations, rewards, flags, state, accumulators and finished-episode records, for every
kernel family (one-warp, CTA fp32 cell list / brute, fp64, cluster), per step and in rollouts."""
import itertools

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import evacuation_b200 as eb  # noqa: E402

REL_OHE_BOX = dict(positions="rel", statuses="ohe", type="Box")
ABS_CAT_DICT = dict(positions="abs", statuses="cat", type="Dict")
GRAV = dict(positions="grav")
NOISES, ENSLAVINGS = (0.05, 0.2, 0.5, 0.8), (1.0, 0.5, 0.1)  # the reference's sweep (SURVEY.md section 2 row 17)


def _make(N, wrap, E, env_kw=None, seed=7, offset=0, **kw):
    env_kw = dict(env_kw or {})
    wrap = dict(wrap)
    if "alpha" in env_kw:
        wrap["alpha"] = env_kw.pop("alpha")
    env = eb.setup_env(eb.EnvConfig(number_of_pedestrians=N, **env_kw), eb.EnvWrappersConfig(**wrap), num_envs=E, device="cuda:0",
                       seed=seed, env_index_offset=offset, batched=True, auto_reset=kw.pop("auto_reset", True), **kw)
    return env, env.unwrapped


def _bits(t):
    t = t.contiguous()
    return t.view(torch.int32) if t.dtype == torch.float32 else (t.view(torch.int64) if t.dtype == torch.float64 else t)


def _run(u, steps, actions=None, agent=None, chunk=None):
    """Per-step outputs (or per-rollout-chunk outputs with `agent`), then state, accumulators and the finished-episode
    records collected after every call."""
    u.reset()
    out = {"obs0": u.flat_observation.clone()}
    rec = []
    if agent is None:
        for t in range(steps):
            _, r, te, tr, _ = u.step(actions[t])
            rec.append((u.flat_observation.clone(), r.clone(), te.clone(), tr.clone(), *u.episode_statistics()[:2]))
    else:
        for _ in range(steps // chunk):
            _, r, te, tr = u.rollout(chunk, agent=agent, status_counts=True)
            rec.append((u.flat_observation.clone(), r.clone(), te.clone(), tr.clone(), *u.episode_statistics()[:2],
                        u.last_status_counts.clone()))
    out["steps"] = rec
    out["state"] = u.get_state()
    out["acc"] = u.accumulators()
    torch.cuda.synchronize()
    return out


def _rows_equal(a, b, rows, what):
    ra, rb = a[rows], b[rows]
    if ra.dtype == torch.bool:
        ra, rb = ra.to(torch.uint8), rb.to(torch.uint8)
    assert torch.equal(_bits(ra), _bits(rb)), what


def _compare(mixed, uni, rows):
    _rows_equal(mixed["obs0"], uni["obs0"], rows, "reset observation")
    for t, (m, r) in enumerate(zip(mixed["steps"], uni["steps"])):
        for k, (x, y) in enumerate(zip(m, r)):
            if x.dim() == 3:  # status_counts [K, E, 4]
                x, y = x.transpose(0, 1), y.transpose(0, 1)
            if k == 4:  # finished-episode statistics: only rows that finished an episode carry a record
                fin = m[5][rows]
                assert torch.equal(fin, r[5][rows]), f"call {t}: finished flags"
                _rows_equal(x[rows][fin], y[rows][fin], slice(None), f"call {t}: episode statistics")
                continue
            _rows_equal(x, y, rows, f"call {t}: output {k}")
    for k in mixed["state"]:
        _rows_equal(mixed["state"][k], uni["state"][k], rows, f"state {k}")
    for x, y in zip(mixed["acc"], uni["acc"]):
        _rows_equal(x, y, rows, "accumulators")


def _check(N, wrap, E, per_env, steps, env_kw=None, agent=None, chunk=None, actions=None, **kw):
    """Environment e of one handle with `per_env` (field -> E values) against environment e of the uniform handle of e's values.
    Returns the handle and its outputs."""
    keys = sorted(per_env)
    vals = [tuple(per_env[k][e] for k in keys) for e in range(E)]
    if agent is None and actions is None:
        actions = torch.as_tensor(np.random.RandomState(1).uniform(-1, 1, (steps, E, 2)).astype(np.float32), device="cuda:0")
    _, mu = _make(N, wrap, E, env_kw, **kw)
    mu.set_env_params(**per_env)
    mixed = _run(mu, steps, actions, agent, chunk)
    for combo in sorted(set(vals)):
        _, uu = _make(N, wrap, E, {**(env_kw or {}), **dict(zip(keys, combo))}, **kw)
        uni = _run(uu, steps, actions, agent, chunk)
        rows = torch.tensor([v == combo for v in vals], device="cuda:0")
        _compare(mixed, uni, rows)
        del uu
    return mu, mixed


def _grid(E):
    combos = list(itertools.product(NOISES, ENSLAVINGS))
    return {"noise_coef": [combos[e % 12][0] for e in range(E)], "enslaving_degree": [combos[e % 12][1] for e in range(E)]}


# ---- 1. the reference's noise x enslaving grid on the one-warp kernel
@pytest.mark.parametrize("N,wrap,alphas", [(60, REL_OHE_BOX, None), (10, ABS_CAT_DICT, None), (33, GRAV, (2, 3, 4, 5, 2.5))])
def test_grid_one_warp_kernel(N, wrap, alphas):
    E = 96
    per_env = _grid(E)
    if alphas:  # 2.5: the powf path of the gravity encoding
        per_env["alpha"] = [alphas[(e // 12) % len(alphas)] for e in range(E)]
    _check(N, wrap, E, per_env, 300, env_kw=dict(max_timesteps=90, is_new_exiting_reward=True))


# ---- 2. the other kernel families
@pytest.mark.parametrize("N,precision,search,wrap", [(200, "fp32", "auto", REL_OHE_BOX), (200, "fp32", "brute", REL_OHE_BOX),
                                                     (60, "fp64", "auto", REL_OHE_BOX), (60, "fp64", "auto", GRAV)])
def test_cta_and_fp64_kernels(N, precision, search, wrap):
    E = 24
    per_env = _grid(E)
    per_env["intrinsic_reward_coef"] = [(0.0, 0.5)[e % 2] for e in range(E)]
    if wrap is GRAV:
        per_env["alpha"] = [(2, 3.5, 5)[e % 3] for e in range(E)]
    _check(N, wrap, E, per_env, 12, env_kw=dict(max_timesteps=5), precision=precision, neighbor_search=search)


def test_cluster_kernel(monkeypatch):
    monkeypatch.setenv("EVAC_CLUSTER", "4")
    E = 4
    _check(9000, REL_OHE_BOX, E, {"noise_coef": [0.05, 0.8, 0.2, 0.5], "enslaving_degree": [1.0, 0.1, 0.5, 1.0],
                                  "is_new_exiting_reward": [0, 1, 1, 0]}, 3, env_kw=dict(max_timesteps=2))


# ---- 3. evac_rollout with the scripted agents and status counts
@pytest.mark.parametrize("agent", ["random", "rotating", "wacuum"])
def test_rollout_agents_status_counts(agent):
    E = 48
    _check(60, REL_OHE_BOX, E, _grid(E), 150, env_kw=dict(max_timesteps=70), agent=agent, chunk=50)


# ---- 4. reward knobs and horizon
def test_reward_knobs_and_horizon():
    E = 36
    per_env = {"max_timesteps": [(5, 17, 200)[e % 3] for e in range(E)],
               "is_new_exiting_reward": [(e // 3) % 2 for e in range(E)],
               "is_new_followers_reward": [(e // 6) % 2 for e in range(E)],
               "is_termination_agent_wall_collision": [(e // 12) % 2 for e in range(E)],
               "intrinsic_reward_coef": [(0.0, 1.0)[(e // 18) % 2] for e in range(E)],
               "init_reward_each_step": [(-1.0, 0.0, -0.5)[(e // 2) % 3] for e in range(E)]}
    # the agents of the 200-step envs walk right, (1, 0), and hit the wall at x = 1 after about 100 steps: with the wall flag
    # they terminate there, without it they stay (and take the -5 collision reward every step)
    steps = 150
    acts = np.random.RandomState(1).uniform(-1, 1, (steps, E, 2)).astype(np.float32)
    acts[:, 2::3] = (1.0, 0.0)
    acts = torch.as_tensor(acts, device="cuda:0")
    wall = torch.tensor([e % 3 == 2 and per_env["is_termination_agent_wall_collision"][e] == 1 for e in range(E)], device="cuda:0")
    free = torch.tensor([e % 3 == 2 and per_env["is_termination_agent_wall_collision"][e] == 0 for e in range(E)], device="cuda:0")
    for N, wrap in ((60, REL_OHE_BOX), (200, REL_OHE_BOX)):
        mu, out = _check(N, wrap, E, per_env, steps, actions=acts)
        assert mu.env_params()["max_timesteps"].tolist() == per_env["max_timesteps"]
        term = torch.stack([o[2] for o in out["steps"]])  # [steps, E]
        assert bool(term[90:, wall].any(dim=0).all()), "every wall-terminating agent must terminate on its collision"
        assert not bool(term[:, free].any()), "agents without wall termination never terminate here"


# ---- 5. semantics
def test_equal_values_give_the_uniform_bits_and_none_returns_to_uniform():
    E, N, steps = 16, 60, 40
    acts = torch.as_tensor(np.random.RandomState(2).uniform(-1, 1, (steps, E, 2)).astype(np.float32), device="cuda:0")
    _, ref = _make(N, REL_OHE_BOX, E)
    want = _run(ref, steps, acts)
    rows = torch.ones(E, dtype=torch.bool, device="cuda:0")
    # the per-env kernel with every record equal to the construction config
    _, a = _make(N, REL_OHE_BOX, E)
    a.set_env_params(**a.env_params())
    _compare(_run(a, steps, acts), want, rows)
    # back to uniform: the construction values, the uniform kernel, the bits of a fresh handle
    _, b = _make(N, REL_OHE_BOX, E)
    b.set_env_params(noise_coef=np.linspace(0.05, 0.8, E), max_timesteps=9)
    b.set_env_params(None)
    assert b.env_params()["noise_coef"].tolist() == [0.2] * E and b.env_params()["max_timesteps"].tolist() == [2000] * E
    _compare(_run(b, steps, acts), want, rows)


def test_partial_update_round_trip_and_errors():
    E = 8
    _, u = _make(10, ABS_CAT_DICT, E)
    noise = np.linspace(0.05, 0.8, E)
    u.set_env_params(noise_coef=noise)
    u.set_env_params(enslaving_degree=torch.full((E,), 0.5), max_timesteps=17)
    p = u.env_params()
    assert p["noise_coef"].tolist() == noise.tolist() and p["enslaving_degree"].tolist() == [0.5] * E
    assert p["max_timesteps"].tolist() == [17] * E and p["alpha"].tolist() == [3.0] * E
    _, v = _make(10, ABS_CAT_DICT, E)
    v.set_env_params(**p)
    q = v.env_params()
    assert all(np.array_equal(p[k], q[k]) for k in p)
    for bad in (dict(width=2.0), dict(step_size=0.02), dict(noise_coef=[0.1] * (E - 1)), dict(max_timesteps=0)):
        with pytest.raises(ValueError):
            u.set_env_params(**bad)
    assert all(np.array_equal(u.env_params()[k], p[k]) for k in p)  # a refused update changes nothing


def test_gravity_wrapper_alpha_applies_to_every_environment():
    E = 6
    env = eb.setup_env(eb.EnvConfig(number_of_pedestrians=10), eb.EnvWrappersConfig(), num_envs=E, device="cuda:0", batched=True)
    u = env.unwrapped
    u.set_env_params(alpha=[2.0, 3.0, 4.0, 5.0, 2.5, 3.0], noise_coef=0.5)
    eb.GravityEncoding(env, alpha=4.0)
    p = u.env_params()
    assert p["alpha"].tolist() == [4.0] * E and p["noise_coef"].tolist() == [0.5] * E


# ---- 6. a switch of parameters mid-run == checkpoint of a uniform P1 handle resumed in a uniform P2 handle
def test_switch_mid_run_equals_checkpoint_into_other_config():
    E, N, t, steps = 24, 60, 25, 60
    # the same fields in both (set_env_params keeps the fields it is not given)
    P1 = dict(noise_coef=0.8, enslaving_degree=0.1, is_new_exiting_reward=True, intrinsic_reward_coef=0.0, max_timesteps=40)
    P2 = dict(noise_coef=0.05, enslaving_degree=0.5, is_new_exiting_reward=False, intrinsic_reward_coef=0.5, max_timesteps=15)
    acts = torch.as_tensor(np.random.RandomState(3).uniform(-1, 1, (steps, E, 2)).astype(np.float32), device="cuda:0")
    _, m = _make(N, REL_OHE_BOX, E)
    m.set_env_params(**P1)
    m.reset()
    got = []
    for s in range(steps):
        if s == t:
            m.set_env_params(**P2)
        _, r, te, tr, _ = m.step(acts[s])
        got.append((m.flat_observation.clone(), r.clone(), te.clone(), tr.clone()))
    _, u1 = _make(N, REL_OHE_BOX, E, P1)
    _, u2 = _make(N, REL_OHE_BOX, E, P2)
    u1.reset()
    want = []
    for s in range(steps):
        if s == t:
            u2.load_state(u1.save_state())
        u = u1 if s < t else u2
        _, r, te, tr, _ = u.step(acts[s])
        want.append((u.flat_observation.clone(), r.clone(), te.clone(), tr.clone()))
    for s, (g, w) in enumerate(zip(got, want)):
        for x, y in zip(g, w):
            assert torch.equal(_bits(x.to(torch.uint8) if x.dtype == torch.bool else x), _bits(y.to(torch.uint8) if y.dtype == torch.bool else y)), s
    for k, x in m.get_state().items():
        assert torch.equal(_bits(x), _bits(u2.get_state()[k])), k


# ---- 7. sharding: two half handles with their parameter slices == one handle
def test_sharding_with_parameter_slices():
    E = 24
    per_env = _grid(E)
    per_env["alpha"] = [(2, 2.5, 4)[e % 3] for e in range(E)]
    _, whole = _make(33, GRAV, E)
    whole.set_env_params(**per_env)
    want = _run(whole, 120, agent="random", chunk=40)
    halves = []
    for off in (0, E // 2):
        _, h = _make(33, GRAV, E // 2, offset=off)
        h.set_env_params(**{k: v[off:off + E // 2] for k, v in per_env.items()})
        halves.append(_run(h, 120, agent="random", chunk=40))
    cat = lambda a, b, dim=0: torch.cat([a, b], dim=dim)  # noqa: E731
    joined = {"obs0": cat(halves[0]["obs0"], halves[1]["obs0"]),
              "steps": [tuple(cat(x, y, 1 if k == 6 else 0) for k, (x, y) in enumerate(zip(a, b)))  # 6: status counts [K, E, 4]
                        for a, b in zip(halves[0]["steps"], halves[1]["steps"])],
              "state": {k: cat(halves[0]["state"][k], halves[1]["state"][k]) for k in want["state"]},
              "acc": tuple(cat(x, y) for x, y in zip(halves[0]["acc"], halves[1]["acc"]))}
    _compare(joined, want, torch.ones(E, dtype=torch.bool, device="cuda:0"))


# ---- 8. the host face draws its NumPy noise with the env's current noise_coef
def test_host_face_numpy_noise_uses_the_env_noise_coef():
    runs = []
    for per_env in (True, False):
        env = eb.setup_env(eb.EnvConfig(number_of_pedestrians=10, noise_coef=0.2 if per_env else 0.5), eb.EnvWrappersConfig(), device="cuda:0")
        if per_env:
            env.unwrapped.set_env_params(noise_coef=0.5)
        np.random.seed(11)
        obs, _ = env.reset()
        acts = np.random.RandomState(5).uniform(-1, 1, (40, 2)).astype(np.float32)
        trace = [np.concatenate([v.ravel() for v in obs.values()])]
        for a in acts:
            obs, r, te, tr, _ = env.step(a)
            trace.append(np.concatenate([np.concatenate([v.ravel() for v in obs.values()]), [r, te, tr]]))
        runs.append(trace)
    assert all(np.array_equal(a, b) for a, b in zip(*runs))


# ---- 9. PolicyRollout: graph replay on a mixed handle, and re-capture after a uniform -> per-env switch
def test_policy_rollout_graph_on_mixed_handle():
    from evacuation_b200.rollout import FusedRPOTransformerPolicy, PolicyRollout, RPOTransformerPolicy

    E, N = 48, 10
    torch.manual_seed(0)
    net = RPOTransformerPolicy((N + 2) * 6, N).cuda()
    per_env = _grid(E)

    def loop(use_graph, switch):
        _, u = _make(N, REL_OHE_BOX, E, dict(max_timesteps=30))
        if not switch:
            u.set_env_params(**per_env)
        pol = FusedRPOTransformerPolicy(net, N, seed=4).eval()
        ro = PolicyRollout(u, pol, use_graph=use_graph)
        ro.reset()
        bufs = [ro.run(12)]
        graph = ro._graph
        if switch:
            u.set_env_params(**per_env)
            bufs.append(ro.run(12))
            if use_graph:
                assert ro._graph is not graph, "switching to per-env parameters must re-capture the graph"
            u.set_env_params(noise_coef=0.3)  # a value-only update: the captured graph reads the new values
            graph = ro._graph
            bufs.append(ro.run(12))
            assert ro._graph is graph
        return bufs

    for switch in (False, True):
        got, want = loop(True, switch), loop(False, switch)
        for g, w in zip(got, want):
            for k in w:
                assert torch.equal(_bits(g[k]), _bits(w[k])), (switch, k)
