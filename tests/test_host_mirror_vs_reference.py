"""The host-side policy containers (mjrl_b200.policies / utils.fc_network) against the reference classes, on the CPU.
The reference's outputs are stored in tests/golden/host_containers.npz (oracle/make_golden_host.py); the inputs are
drawn here from the same seeded generators, in the same order."""
import pickle
import types

import numpy as np
import pytest
import torch

from conftest import golden_equal, load_golden


@pytest.fixture(scope="module")
def ref():
    return load_golden("host_containers")


SHAPES = [(6, 2, (32, 32)), (17, 6, (128, 128)), (5, 3, (64, 64))]      # mlp0_ .. mlp2_ in the fixture


@pytest.mark.parametrize("shape", SHAPES)
def test_policy_container_matches_reference(ref, shape):
    from mjrl_b200.policies.gaussian_mlp import MLP
    obs_dim, act_dim, hidden = shape
    i = SHAPES.index(shape)
    r = {k[len("mlp%d_" % i):]: v for k, v in ref.items() if k.startswith("mlp%d_" % i)}
    mine = MLP(types.SimpleNamespace(observation_dim=obs_dim, action_dim=act_dim), hidden_sizes=hidden, seed=7,
               init_log_std=-0.25, min_log_std=-2.0)
    assert mine.d == r["d"] and repr([tuple(s) for s in mine.param_shapes]) == str(r["param_shapes"])
    assert list(mine.param_sizes) == list(r["param_sizes"])
    assert golden_equal(mine.get_param_values(), r, "init")                        # same init draws, same layout
    # set_param_values: layout, clamp of log_std, new / old sets
    rng = np.random.RandomState(1)
    th = rng.randn(mine.d).astype(np.float32)
    th[-act_dim:] = np.linspace(-4.0, 1.0, act_dim)                                   # some entries below min_log_std
    for j, flags in enumerate(((True, True), (True, False), (False, True))):
        mine.set_param_values(th * (1 + flags[0] + 2 * flags[1]), *flags)
        assert golden_equal(mine.get_param_values(), r, "set%d_params" % j)
        old_m = np.concatenate([p.data.numpy().ravel() for p in mine.old_params])
        assert golden_equal(old_m, r, "set%d_old" % j)
        assert golden_equal(mine.log_std_val, r, "set%d_log_std_val" % j)
    assert mine.get_param_values()[-act_dim:].min() >= -2.0
    # sampling: same mean, same global-RNG draw
    o = rng.randn(obs_dim)
    np.random.seed(5); a_m, info_m = mine.get_action(o)
    assert golden_equal(a_m, r, "action") and golden_equal(info_m["mean"], r, "action_mean")
    assert golden_equal(info_m["evaluation"], r, "action_evaluation") and golden_equal(info_m["log_std"], r, "action_log_std")
    # small-input helpers
    obs, act = rng.randn(50, obs_dim).astype(np.float32), rng.randn(50, act_dim).astype(np.float32)
    mine.set_param_values(th, True, False)                                            # new != old
    np.testing.assert_allclose(mine.log_likelihood(obs, act), r["log_likelihood"], rtol=1e-6, atol=1e-6)
    nm, om = mine.new_dist_info(obs, act), mine.old_dist_info(obs, act)
    for a, b in zip(nm[:2] + om[:2], (r["new_ll"], r["new_mean"], r["old_ll"], r["old_mean"])):
        np.testing.assert_allclose(a.detach().numpy(), b, rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(mine.likelihood_ratio(nm, om).detach().numpy(), r["likelihood_ratio"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(float(mine.mean_kl(nm, om)), float(r["mean_kl"]), rtol=1e-5, atol=1e-7)
    # pickling keeps the weights and keeps working
    clone = pickle.loads(pickle.dumps(mine))
    assert np.array_equal(clone.get_param_values(), mine.get_param_values())
    clone.set_param_values(th * 0.5)
    assert np.array_equal(clone.get_param_values()[:-act_dim], (th * 0.5)[:-act_dim])


def test_fc_network_matches_reference(ref):
    from mjrl_b200.utils.fc_network import FCNetwork
    rng = np.random.RandomState(0)
    tr = dict(in_shift=rng.randn(7), in_scale=0.5 + rng.rand(7), out_shift=rng.randn(3), out_scale=0.5 + rng.rand(3))
    for i, (hidden, nl) in enumerate((((16, 8), "tanh"), ((32, 32), "relu"), ((), "tanh"))):
        k = "fc%d_" % i
        torch.manual_seed(3); b = FCNetwork(7, 3, hidden, nl, **tr)
        assert repr([tuple(p.shape) for p in b.parameters()]) == str(ref[k + "param_shapes"])
        assert golden_equal(np.concatenate([p.data.numpy().ravel() for p in b.parameters()]), ref, k + "params")
        assert repr(list(b.state_dict().keys())) == str(ref[k + "state_dict_keys"])
        x = torch.from_numpy(rng.randn(9, 7).astype(np.float32))
        assert golden_equal(b(x).detach().numpy(), ref, k + "output")
        assert repr(b.layer_sizes) == str(ref[k + "layer_sizes"])
        assert repr(sorted(b.transformations)) == str(ref[k + "transformations"])


def test_linear_policy_container_matches_reference(ref):
    from mjrl_b200.policies.gaussian_linear import LinearPolicy
    mine = LinearPolicy(types.SimpleNamespace(observation_dim=11, action_dim=4), seed=3)
    assert mine.d == ref["lin_d"]
    th = np.random.RandomState(2).randn(mine.d).astype(np.float32)
    mine.set_param_values(th)
    assert golden_equal(mine.get_param_values(), ref, "lin_params")
    o = np.random.RandomState(4).randn(11)
    np.random.seed(9); a_m = mine.get_action(o)[0]
    np.testing.assert_allclose(a_m, ref["lin_action"], rtol=1e-6, atol=1e-6)
