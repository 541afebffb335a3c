"""CPU tests of the rollout-loop glue (evacuation_b200/rollout.py): the policy restatement against a golden
produced by the unmodified reference network, and the per-env running normalisers against a NumPy restatement of
gymnasium's RunningMeanStd."""
import os

import numpy as np
import pytest
import torch

from evacuation_b200.rollout import RPOTransformerPolicy, VectorNormalizer

HERE = os.path.dirname(os.path.abspath(__file__))


def _load_policy():
    z = np.load(os.path.join(HERE, "golden", "policy", "policy_transformer.npz"))
    n = int(z["number_of_pedestrians"])
    x = torch.as_tensor(z["x"])
    net = RPOTransformerPolicy(x.shape[1], n).eval()
    sd = {k[2:]: torch.as_tensor(z[k]) for k in z.files if k.startswith("w:")}
    missing, unexpected = net.load_state_dict(sd, strict=True)  # same parameter names / shapes as the reference module
    assert not missing and not unexpected
    return z, x, net


def test_policy_matches_reference_network_golden():
    z, x, net = _load_policy()
    with torch.no_grad():
        emb = net.embed(x)
        np.testing.assert_allclose(emb.numpy(), z["embedding"], rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(net.actor_mean(emb).numpy(), z["actor_mean"], rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(net.get_value(x).numpy(), z["value"], rtol=1e-5, atol=1e-6)
        # log-probability / entropy of the action the reference sampled
        a = torch.as_tensor(z["sampled_action"])
        mean = net.actor_mean(emb)
        std = torch.exp(net.actor_logstd.expand_as(mean))
        lp = torch.distributions.Normal(mean, std).log_prob(a).sum(1)
        np.testing.assert_allclose(lp.numpy(), z["logprob_of_sampled"], rtol=1e-5, atol=1e-6)
        _, lp2, ent, v = net.get_action_and_value(x)
        np.testing.assert_allclose(ent.numpy(), z["entropy"], rtol=1e-6)
        np.testing.assert_allclose(v.numpy(), z["value"], rtol=1e-5, atol=1e-6)


def test_policy_chunking_is_transparent():
    z, x, net = _load_policy()
    net.chunk = 2
    with torch.no_grad():
        np.testing.assert_allclose(net.embed(x).numpy(), z["embedding"], rtol=1e-5, atol=1e-6)


class _RMS:  # gymnasium.wrappers.normalize.RunningMeanStd restated (float64)
    def __init__(self, shape):
        self.mean, self.var, self.count = np.zeros(shape), np.ones(shape), 1e-4

    def update(self, x):
        bm, bv, bc = x.mean(axis=0), x.var(axis=0), x.shape[0]
        delta = bm - self.mean
        tot = self.count + bc
        self.mean = self.mean + delta * bc / tot
        m2 = self.var * self.count + bv * bc + delta ** 2 * self.count * bc / tot
        self.var, self.count = m2 / tot, tot


def test_vector_normalizer_matches_gymnasium_running_mean_std():
    E, D, T, gamma = 3, 5, 40, 0.99
    rs = np.random.RandomState(0)
    norm = VectorNormalizer(E, D, gamma=gamma, device="cpu", dtype=torch.float64)
    obs_rms = [_RMS((D,)) for _ in range(E)]
    ret_rms = [_RMS(()) for _ in range(E)]
    returns = np.zeros(E)
    for t in range(T):
        obs = rs.normal(0.3, 2.0, (E, D))
        rew = rs.normal(-1, 3, E)
        term = rs.rand(E) < 0.1
        got_o = norm.observation(torch.as_tensor(obs)).numpy()
        got_r = norm.reward(torch.as_tensor(rew), torch.as_tensor(term)).numpy()
        for e in range(E):
            obs_rms[e].update(obs[e][None])
            want_o = np.clip((obs[e] - obs_rms[e].mean) / np.sqrt(obs_rms[e].var + 1e-8), -1, 1)
            np.testing.assert_allclose(got_o[e], want_o, rtol=1e-9, atol=1e-12)
            returns[e] = returns[e] * gamma * (1 - term[e]) + rew[e]
            ret_rms[e].update(np.array([returns[e]]))
            want_r = np.clip(rew[e] / np.sqrt(ret_rms[e].var + 1e-8), -100, 100)
            np.testing.assert_allclose(got_r[e], want_r, rtol=1e-9, atol=1e-12)


@pytest.mark.parametrize("tag", ["unit", "wide"])
def test_wacuum_cleaner_matches_reference_trace(tag):
    """The sweep baseline (single-env NumPy face and the batched torch state machine) against the action trace of the
    unmodified reference class (tests/golden/policy/gen_wacuum_golden.py)."""
    from types import SimpleNamespace as NS

    from evacuation_b200.agents import WacuumCleaner

    z = np.load(os.path.join(HERE, "golden", "policy", "wacuum_actions.npz"))
    w, h, step = z[tag + "_cfg"]
    area = NS(width=w, height=h, step_size=step, exit=NS(position=np.array([0, -1], dtype=np.float32)))
    env = NS(area=area, num_envs=2, device="cpu")
    env.unwrapped = env
    single, batched = WacuumCleaner(env), WacuumCleaner.batched(env)
    for pos, want in zip(z[tag + "_pos"], z[tag + "_act"]):
        got = single.act({"agent_position": pos})
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-7)
        gb = batched.act(torch.as_tensor(np.stack([pos, pos]))).numpy()
        np.testing.assert_allclose(gb[0], want, rtol=0, atol=1e-7)
        np.testing.assert_allclose(gb[1], want, rtol=0, atol=1e-7)


def test_flat_weight_order_of_the_fused_policy_covers_the_reference_state_dict():
    """`flatten_policy_weights` (the vector `evac_policy_load_weights` documents in include/evac_b200.h) consumes every
    parameter of the reference module exactly once, in the documented order."""
    from evacuation_b200.rollout import _FLAT_BLOCK_KEYS, _FLAT_HEAD_KEYS, flatten_policy_weights

    z, x, net = _load_policy()
    sd = {k[2:]: torch.as_tensor(z[k]) for k in z.files if k.startswith("w:")}   # names of the unmodified reference module
    flat = flatten_policy_weights(sd, 2)
    assert flat.dtype == torch.float32 and flat.numel() == sum(v.numel() for v in sd.values())
    names = [f"embedding.{b}.{k}" for b in range(2) for k in _FLAT_BLOCK_KEYS] + list(_FLAT_HEAD_KEYS)
    assert sorted(names) == sorted(sd.keys())
    off = 0
    for n in names:
        v = sd[n].reshape(-1)
        assert torch.equal(flat[off:off + v.numel()], v), n
        off += v.numel()
    # D = 6, H = 3, F = 96, NH = 64, A = 2: the count formula of evac_policy_num_weights
    D, H, F, NH, A, K = 6, 3, 96, 64, 2, x.shape[1]
    block = 3 * (H * D * D + H * D) + (D * H * D + D) + (F * D + F) + (D * F + D) + 4 * D
    heads = 2 * (NH * K + NH + NH * NH + NH) + (NH + 1) + (A * NH + A) + A
    assert flat.numel() == 2 * block + heads


def test_fused_policy_fails_loudly_without_a_cuda_device():
    """No CPU fallback: constructing the fused policy on a machine without a GPU raises."""
    if torch.cuda.is_available():
        pytest.skip("needs a machine without a GPU")
    from evacuation_b200._native import EvacNativeError
    from evacuation_b200.rollout import FusedRPOTransformerPolicy

    net = RPOTransformerPolicy(372, 60)
    with pytest.raises(EvacNativeError):
        FusedRPOTransformerPolicy(net, 60, device="cpu")
    with pytest.raises((EvacNativeError, RuntimeError, AssertionError)):
        FusedRPOTransformerPolicy(net, 60, device="cuda")


def test_vector_env_fails_loudly_without_a_cuda_device():
    if torch.cuda.is_available():
        pytest.skip("needs a machine without a GPU")
    import evacuation_b200 as eb
    from evacuation_b200._native import EvacNativeError

    with pytest.raises((EvacNativeError, RuntimeError, AssertionError)):
        eb.EvacuationVectorEnv(eb.EnvConfig(number_of_pedestrians=10), eb.EnvWrappersConfig(positions="rel", statuses="ohe", type="Box"),
                               num_envs=4)


def _policy_variants():
    z = np.load(os.path.join(HERE, "golden", "policy", "policy_variants.npz"))
    for i in range(int(z["num_variants"])):
        pre = f"v{i}:"
        n, d, heads, dff, blocks, resid, nh = (int(v) for v in z[pre + "cfg"])
        sd = {k[len(pre) + 2:]: torch.as_tensor(z[k]) for k in z.files if k.startswith(pre + "w:")}
        kw = dict(num_heads=heads, dim_feedforward=dff, num_blocks=blocks, use_resid=bool(resid), num_hidden=nh)
        yield i, n, d, kw, sd, {k: z[pre + k] for k in ("x", "embedding", "actor_mean", "value", "action", "logprob")}


def test_policy_restatement_matches_reference_network_variants():
    """Residual blocks, 1 / 2 / 4 heads, d_model 3 / 2, 1 / 3 blocks, narrow feed-forward, 62 and 64 rows: outputs of the
    unmodified reference module (tests/golden/policy/gen_policy_variants_golden.py)."""
    seen = 0
    for i, n, d, kw, sd, g in _policy_variants():
        net = RPOTransformerPolicy((n + 2) * d, n, **kw).eval()
        missing, unexpected = net.load_state_dict(sd, strict=True)
        assert not missing and not unexpected
        x = torch.as_tensor(g["x"])
        with torch.no_grad():
            emb = net.embed(x)
            np.testing.assert_allclose(emb.numpy(), g["embedding"], rtol=1e-5, atol=2e-6, err_msg=f"variant {i}")
            np.testing.assert_allclose(net.actor_mean(emb).numpy(), g["actor_mean"], rtol=1e-5, atol=2e-6)
            np.testing.assert_allclose(net.get_value(x).numpy(), g["value"], rtol=1e-5, atol=2e-6)
            _, lp, _, _ = net.get_action_and_value(x, torch.as_tensor(g["action"]))
        seen += 1
    assert seen == 6


def test_hidden_dropout_words_are_unbiased_and_uncorrelated():
    """The fused policy's hidden-layer dropout (csrc/evac_policy.cuh, feed-forward loop) takes four 16-bit words per row and
    group of four features from ONE fmix32 word and a cheap second mix of it (multiply + xor-shift); an element is dropped
    when its word is below round(p * 65536).  The word schedule is evac_testlib's restatement, which
    tests/test_host_cpu.py::test_policy_streams_match_their_numpy_restatement pins to the kernel's code: every word drops at
    rate p, the indicators of different words are uncorrelated, and the number of dropped features per row is binomial
    [torch.nn.Dropout(0.1) of rpo_transformer_agent_network.py:98]."""
    import evac_testlib as T

    rng = np.random.default_rng(0)
    keys = rng.integers(0, 2 ** 32, size=200000, dtype=np.uint64)
    p = 0.1
    drop = T.drop_hidden_words(keys, 96) < T.drop_threshold(p)  # dim_feedforward 96 = 24 groups
    rates = drop.mean(0)
    assert abs(drop.mean() - p) < 5e-4 and np.abs(rates - p).max() < 4e-3
    c = np.corrcoef(drop[:, :16].T.astype(np.float64))
    assert np.abs(c - np.eye(16)).max() < 0.012
    cnt = drop.sum(1)
    assert abs(cnt.mean() - 96 * p) < 0.05 and abs(cnt.var() - 96 * p * (1 - p)) < 0.2
