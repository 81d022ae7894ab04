"""TEST INFRASTRUCTURE ONLY -- golden vectors of the reference's host-side containers and of one NPG step, produced by
importing the UNMODIFIED reference (oracle/ref_shim.py; needs a reference checkout, e.g. through $MJRL_REF):

    python -m oracle.make_golden_host    ->  tests/golden/host_containers.npz, tests/golden/npg_11x3_ragged.npz

host_containers.npz pins mjrl_b200.policies (MLP, LinearPolicy) and mjrl_b200.utils.fc_network.FCNetwork
(tests/test_host_mirror_vs_reference.py); npg_11x3_ragged.npz pins the oracle's NPG step on shapes that no other
fixture has (tests/test_oracle.py::test_live_reference_npg_step).  The inputs are not stored: the tests draw them
from the same seeded generators, in the same order, as this script.  An array the tests compare bit for bit and
that has more than DIGEST_ABOVE entries is stored as its digest (see `digest`) to keep the fixtures small.
"""
import copy
import hashlib
import os

import numpy as np
import torch

from oracle import npg_oracle as O
from oracle import ref_shim

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
MLP_SHAPES = [(6, 2, (32, 32)), (17, 6, (128, 128)), (5, 3, (64, 64))]
FC_CASES = [((16, 8), "tanh"), ((32, 32), "relu"), ((), "tanh")]
DIGEST_ABOVE, SAMPLE = 1024, 128


def _flat(values):
    return np.concatenate([np.asarray(v).ravel() for v in values])


def digest(a):
    """{"@shape", "@sample", "@sha256"} of an array: its shape, SAMPLE entries at seeded positions (which locate a
    mismatch) and the sha256 of its bytes (which pins every bit).  tests/conftest.py's golden_equal checks them."""
    a = np.ascontiguousarray(a)
    idx = np.sort(np.random.RandomState(0).choice(a.size, SAMPLE, replace=False))
    return {"@shape": np.array(a.shape, np.int64), "@sample": a.ravel()[idx],
            "@sha256": np.array(hashlib.sha256(a.tobytes()).hexdigest())}


def exact(out, key, a):
    """Store an array that the tests compare bit for bit: whole when small, else as its digest."""
    a = np.asarray(a)
    if a.size <= DIGEST_ABOVE:
        out[key] = a
    else:
        out.update({key + k: v for k, v in digest(a).items()})


def policy_container(R, i, obs_dim, act_dim, hidden):
    out, k = {}, "mlp%d_" % i
    ref = R.MLP(R.EnvSpec(obs_dim, act_dim, 10), hidden_sizes=hidden, seed=7, init_log_std=-0.25, min_log_std=-2.0)
    out[k + "d"] = np.int64(ref.d)
    out[k + "param_shapes"] = np.array(repr([tuple(s) for s in ref.param_shapes]))
    out[k + "param_sizes"] = np.array(list(ref.param_sizes), np.int64)
    exact(out, k + "init", ref.get_param_values())
    rng = np.random.RandomState(1)
    th = rng.randn(ref.d).astype(np.float32)
    th[-act_dim:] = np.linspace(-4.0, 1.0, act_dim)
    for j, flags in enumerate(((True, True), (True, False), (False, True))):
        ref.set_param_values(th * (1 + flags[0] + 2 * flags[1]), *flags)
        exact(out, k + "set%d_params" % j, ref.get_param_values())
        exact(out, k + "set%d_old" % j, _flat([p.data.numpy() for p in ref.old_params]))
        exact(out, k + "set%d_log_std_val" % j, ref.log_std_val)
    o = rng.randn(obs_dim)
    np.random.seed(5)
    a, info = ref.get_action(o)
    exact(out, k + "action", a)
    for name in ("mean", "evaluation", "log_std"):
        exact(out, k + "action_" + name, info[name])
    obs, act = rng.randn(50, obs_dim).astype(np.float32), rng.randn(50, act_dim).astype(np.float32)
    ref.set_param_values(th, True, False)
    out[k + "log_likelihood"] = ref.log_likelihood(obs, act)
    nr, orr = ref.new_dist_info(obs, act), ref.old_dist_info(obs, act)
    for tag, info in (("new", nr), ("old", orr)):
        out[k + tag + "_ll"] = info[0].detach().numpy()
        out[k + tag + "_mean"] = info[1].detach().numpy()
    out[k + "likelihood_ratio"] = ref.likelihood_ratio(nr, orr).detach().numpy()
    out[k + "mean_kl"] = np.float64(float(ref.mean_kl(nr, orr)))
    return out


def fc_networks(R):
    from mjrl.utils.fc_network import FCNetwork
    out = {}
    rng = np.random.RandomState(0)
    tr = dict(in_shift=rng.randn(7), in_scale=0.5 + rng.rand(7), out_shift=rng.randn(3), out_scale=0.5 + rng.rand(3))
    for i, (hidden, nl) in enumerate(FC_CASES):
        k = "fc%d_" % i
        torch.manual_seed(3)
        a = FCNetwork(7, 3, hidden, nl, **tr)
        out[k + "param_shapes"] = np.array(repr([tuple(p.shape) for p in a.parameters()]))
        exact(out, k + "params", _flat([p.data.numpy() for p in a.parameters()]))
        out[k + "state_dict_keys"] = np.array(repr(list(a.state_dict().keys())))
        x = torch.from_numpy(rng.randn(9, 7).astype(np.float32))
        exact(out, k + "output", a(x).detach().numpy())
        out[k + "layer_sizes"] = np.array(repr(a.layer_sizes))
        out[k + "transformations"] = np.array(repr(sorted(a.transformations)))
    return out


def linear_policy(R):
    ref = R.LinearPolicy(R.EnvSpec(11, 4, 10), seed=3)
    th = np.random.RandomState(2).randn(ref.d).astype(np.float32)
    ref.set_param_values(th)
    o = np.random.RandomState(4).randn(11)
    np.random.seed(9)
    out = {"lin_d": np.int64(ref.d), "lin_action": ref.get_action(o)[0]}
    exact(out, "lin_params", ref.get_param_values())
    return out


def npg_step(R):
    obs_dim, act_dim, hidden = 11, 3, (64, 64)
    paths = O.synthetic_paths(obs_dim, act_dim, 30, 300, seed=3, ragged=True)
    es = R.EnvSpec(obs_dim, act_dim, 300)
    pol = R.MLP(es, hidden_sizes=hidden, seed=9)
    bl = R.MLPBaseline(es, reg_coef=1e-3, epochs=1)
    out = {"theta0": pol.get_param_values(),
           "vf_w": _flat([p.data.numpy() for p in bl.model.parameters()]).astype(np.float32)}
    ref_paths = copy.deepcopy(paths)
    R.process_samples.compute_returns(ref_paths, 0.995)
    R.process_samples.compute_advantages(ref_paths, bl, 0.995, 0.97)
    exact(out, "returns", np.concatenate([p["returns"] for p in ref_paths]))
    exact(out, "advantages", np.concatenate([p["advantages"] for p in ref_paths]))
    R.NPG(None, pol, bl, normalized_step_size=0.05).train_from_paths(ref_paths)
    out["new_params"] = pol.get_param_values()
    out["meta"] = np.array(repr(dict(obs_dim=obs_dim, act_dim=act_dim, hidden=hidden, n_paths=30, horizon=300,
                                     path_seed=3, ragged=True, policy_seed=9, gamma=0.995, lam=0.97, npg_step=0.05)))
    return out


def main():
    R = ref_shim.load()
    torch.set_num_threads(1)          # bitwise-repeatable reference outputs
    host = {}
    for i, shape in enumerate(MLP_SHAPES):
        host.update(policy_container(R, i, *shape))
    host.update(fc_networks(R))
    host.update(linear_policy(R))
    for name, out in (("host_containers", host), ("npg_11x3_ragged", npg_step(R))):
        path = os.path.join(GOLDEN_DIR, name + ".npz")
        np.savez_compressed(path, **out)
        print("%-24s %3d arrays  %.0f KB" % (os.path.basename(path), len(out), os.path.getsize(path) / 1024))


if __name__ == "__main__":
    main()
