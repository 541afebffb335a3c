"""CPU checks of the linear RPO policy (RPOLinearNetwork on the flattened observation, rpo_linear_agent_network.py:19-61):
its torch restatement's parameter names and formulas, and the flat weight vector the library's num_blocks = 0 policy loads."""
import pytest
import torch

from evacuation_b200.rollout import RPOLinearPolicy, RPOTransformerPolicy, _FLAT_HEAD_KEYS, flatten_policy_weights


def test_linear_policy_state_dict_keys_are_the_transformer_head_keys():
    lin = RPOLinearPolicy(364)
    heads = [k for k in RPOTransformerPolicy(372, 60).state_dict() if not k.startswith("embedding.")]
    assert list(lin.state_dict()) == heads
    assert set(lin.state_dict()) == set(_FLAT_HEAD_KEYS)


@pytest.mark.parametrize("K,NH,A", [(6, 64, 2), (364, 64, 2), (25, 32, 3), (1, 12, 1)])
def test_flat_linear_weights_have_the_header_length(K, NH, A):
    """include/evac_b200.h: the heads part of the layout, 2 (NH K + NH + NH NH + NH) + (NH + 1) + (A NH + A) + A floats."""
    flat = flatten_policy_weights(RPOLinearPolicy(K, action_dim=A, num_hidden=NH).state_dict(), num_blocks=0)
    assert flat.dtype == torch.float32 and flat.numel() == 2 * (NH * K + NH + NH * NH + NH) + (NH + 1) + (A * NH + A) + A


def test_linear_policy_logprob_and_entropy_match_torch_distributions_in_float64():
    torch.manual_seed(0)
    net = RPOLinearPolicy(6, action_dim=3).double()
    with torch.no_grad():
        net.actor_logstd.add_(0.4 * torch.randn_like(net.actor_logstd))
    x = torch.rand(257, 6, dtype=torch.float64) * 2 - 1
    action, logprob, entropy, value = net.get_action_and_value(x)
    mean = net.actor_mean(x)
    dist = torch.distributions.Normal(mean, torch.exp(net.actor_logstd.expand_as(mean)))
    torch.testing.assert_close(logprob, dist.log_prob(action).sum(1), rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(entropy, dist.entropy().sum(1), rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(value, net.critic(x), rtol=0, atol=0)
    assert action.shape == (257, 3) and value.shape == (257, 1)
    # a given action is evaluated against the RPO-perturbed mean: mean + U(-rpo_alpha, rpo_alpha)
    gen = torch.get_rng_state()
    _, lp_given, _, _ = net.get_action_and_value(x, action)
    torch.set_rng_state(gen)
    pert = mean + torch.empty_like(mean).uniform_(-net.rpo_alpha, net.rpo_alpha)
    want = torch.distributions.Normal(pert, torch.exp(net.actor_logstd.expand_as(mean))).log_prob(action).sum(1)
    torch.testing.assert_close(lp_given, want, rtol=1e-12, atol=1e-12)
    assert bool(torch.isfinite(lp_given).all())
