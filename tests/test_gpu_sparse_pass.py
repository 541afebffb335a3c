"""The one-warp kernel's sparse neighbour pass (N <= 64, 2-D cell masks, evac_warp.cuh) against the all-pairs loop.

neighbor_search="auto" takes the sparse pass per warp and step unless the all-pairs loop is cheaper or a source direction
is NaN; "cells" takes it whenever it is exact; "brute" always runs the all-pairs loop.  All three must give the same bits:
states, observations, rewards and flags, over per-step calls and K-step rollouts, with same-step auto-resets, escaped /
exiting pedestrians, a NaN direction, dense blobs next to sparse crowds in one batch, and pairs just inside the vision
radius across cell boundaries."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

WRAPS = {
    "rel_ohe_box": dict(positions="rel", statuses="ohe", type="Box"),
    "grav": dict(positions="grav", alpha=3),
    "abs_cat_dict": dict(positions="abs", statuses="cat", type="Dict"),
}
MAX_T = 40


def _boundary_pairs(n, width, height, vision, rs):
    """Pairs just inside the vision radius straddling a cell edge in x, in y and diagonally (the grid of warp_cell_grid)."""
    gx = max(1, min(32, int(np.floor(2 * width / (vision * (1 + 1e-4))))))
    gy = max(1, min(32, int(np.floor(2 * height / (vision * (1 + 1e-4))))))
    d = vision * (1 - 1e-6)
    pos = rs.uniform(-1, 1, (n, 2)) * [width, height]
    for i in range(0, n - 1, 2):
        kx, ky = rs.randint(1, gx) if gx > 1 else 0, rs.randint(1, gy) if gy > 1 else 0
        bx, by = -width + kx * 2 * width / gx, -height + ky * 2 * height / gy
        ang = (0.0, 0.5 * np.pi, 0.25 * np.pi)[(i // 2) % 3]
        c = np.array([bx if ang != 0.5 * np.pi else rs.uniform(-0.9, 0.9) * width,
                      by if ang != 0.0 else rs.uniform(-0.9, 0.9) * height])
        off = 0.5 * d * np.array([np.cos(ang), np.sin(ang)])
        pos[i], pos[i + 1] = c - off, c + off
    return np.clip(pos, [-width, -height], [width, height])


def _layouts(n, E, width, height, vision, seed):
    """E environments: uniform crowds, a dense blob, half blob / half uniform, near-radius pairs across cell edges, and one
    with a zero direction (NaN unit vector) and pedestrians at / near the exit (EXITING, ESCAPED)."""
    rs = np.random.RandomState(seed)
    pos = rs.uniform(-1, 1, (E, n, 2)) * [width, height]
    blob = np.array([0.3 * width, -0.2 * height])
    pos[1] = blob + rs.normal(0, 0.02, (n, 2))
    pos[2, : n // 2] = blob + rs.normal(0, 0.02, (n // 2, 2))
    pos[3] = _boundary_pairs(n, width, height, vision, rs)
    pos = np.clip(pos, [-width, -height], [width, height])
    ang = rs.uniform(0, 2 * np.pi, (E, n))
    dirs = 0.01 * np.stack([np.cos(ang), np.sin(ang)], axis=-1)
    if E > 4:
        pos[4, 0] = [0.0, -0.995]                     # ESCAPED
        pos[4, n // 2] = [0.05, -0.8]                 # EXITING
        if n > 2:
            pos[4, n - 1] = [0.5, 0.5]                # VISCEK (far from the exit and from the agent) ...
            dirs[4, n - 1] = 0.0                      # ... with a zero direction -> NaN unit vector, poisons every sum
    return pos.astype(np.float32), dirs.astype(np.float32)


def _run(search, n, wrap, E, pos, dirs, now, steps, mode, width=1.0, height=1.0):
    import evacuation_b200 as eb

    env_kw = dict(number_of_pedestrians=n, width=width, height=height, is_new_exiting_reward=True, intrinsic_reward_coef=0.3,
                  enslaving_degree=0.6, noise_coef=0.4, max_timesteps=MAX_T, wandb_enabled=False)
    env = eb.setup_env(eb.EnvConfig(**env_kw), eb.EnvWrappersConfig(**wrap), num_envs=E, batched=True, auto_reset=True,
                       seed=11, neighbor_search=search)
    u = env.unwrapped
    u.reset()
    assert (u.num_cells > 0) == (search == "cells")
    u.set_state(positions=pos, directions=dirs, agent_position=np.zeros((E, 2), np.float32),
                agent_direction=np.zeros((E, 2), np.float32), now=now)
    rs = np.random.RandomState(5)
    out = {"obs": [], "rew": [], "term": [], "trunc": []}

    def keep(obs, r, tm, tr):
        flat = torch.cat([obs[k].reshape(E, -1) for k in sorted(obs)], 1) if isinstance(obs, dict) else obs.reshape(E, -1)
        out["obs"].append(flat.cpu().numpy().copy())
        out["rew"].append(r.cpu().numpy().copy())
        out["term"].append(tm.cpu().numpy().copy())
        out["trunc"].append(tr.cpu().numpy().copy())

    if mode == "step":
        for s in range(steps):
            obs, r, tm, tr, _ = env.step(torch.as_tensor(rs.uniform(-1, 1, (E, 2)).astype(np.float32)))
            keep(obs, r, tm, tr)
    else:
        for chunk in (steps // 2, steps - steps // 2):
            keep(*u.rollout(chunk, agent="random"))
    st = u.get_state()
    for k in ("positions", "directions", "statuses"):
        out[k] = st[k].cpu().numpy()
    u.close()
    return out


def _assert_same(a, b):
    for k in a:
        x, y = np.asarray(a[k]), np.asarray(b[k])
        assert x.shape == y.shape and np.array_equal(x, y, equal_nan=True), k


@pytest.mark.parametrize("mode", ["step", "rollout"])
@pytest.mark.parametrize("search", ["auto", "cells"])
@pytest.mark.parametrize("wrap", list(WRAPS))
@pytest.mark.parametrize("n", [1, 2, 33, 60, 64])
def test_sparse_pass_is_bit_identical_to_all_pairs(n, wrap, search, mode):
    E, steps = 6, 12
    pos, dirs = _layouts(n, E, 1.0, 1.0, 0.1, seed=n)
    now = np.array([0, 3, MAX_T - 4, 0, 0, MAX_T - 7], np.int32)  # two environments auto-reset inside the window
    got = _run(search, n, WRAPS[wrap], E, pos, dirs, now, steps, mode)
    ref = _run("brute", n, WRAPS[wrap], E, pos, dirs, now, steps, mode)
    _assert_same(got, ref)
    if n > 2:
        assert np.isnan(ref["directions"][4]).any()  # the NaN source poisoned its environment (the all-pairs fallback)


@pytest.mark.parametrize("n,width,height,vision", [(60, 1.0, 1.0, 2.5),     # one cell
                                                   (60, 1.0, 1.0, 0.03),    # 66 x 66 -> the 32 x 32 cap
                                                   (64, 1.5, 0.8, 0.1),     # 29 x 15
                                                   (33, 0.4, 1.3, 0.07),    # 11 x 37 -> 11 x 32
                                                   (60, 1.0, 1.0, 0.35)])   # 5 x 5
@pytest.mark.parametrize("search", ["auto", "cells"])
def test_sparse_pass_grid_shapes(n, width, height, vision, search, monkeypatch):
    import evacuation_b200 as eb

    monkeypatch.setattr(eb.SwitchDistances, "to_pedestrian", vision)
    E, steps = 6, 10
    pos, dirs = _layouts(n, E, width, height, vision, seed=100 + n)
    now = np.array([0, 0, MAX_T - 3, 0, 0, 0], np.int32)
    wrap = WRAPS["rel_ohe_box"]
    got = _run(search, n, wrap, E, pos, dirs, now, steps, "step", width, height)
    ref = _run("brute", n, wrap, E, pos, dirs, now, steps, "step", width, height)
    _assert_same(got, ref)
