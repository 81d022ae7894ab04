"""CPU tests of PPO-clip and behaviour cloning: the fp32 oracle against the reference fixtures, the minibatch index draw
against the reference's np.random.choice loop, and the agents' host logic."""
import numpy as np
import pytest

from conftest import load_golden
from oracle import ppo_bc_oracle as PB

CASES = ["ppo_17x6_h128", "ppo_6x2_h32", "ppo_clipheavy_6x2_h64", "ppo_39x28_h256", "bc_mse_17x6_h128",
         "bc_mle_tr_11x3_h64"]


def initial_theta(meta):
    """theta_0 of a fixture case from this package's host policy (the reference's init draws) and, for BC with
    set_transforms, the BC constructor."""
    from mjrl_b200.policies.gaussian_mlp import MLP
    from mjrl_b200.utils.gym_env import EnvSpec
    pol = MLP(EnvSpec(meta["obs_dim"], meta["act_dim"], meta["horizon"]), hidden_sizes=meta["hidden"],
              seed=meta["policy_seed"])
    if meta["kind"] == "bc" and meta["set_transforms"]:
        from mjrl_b200.algos.behavior_cloning import BC
        BC(PB.case_paths(meta, 0), pol, set_transforms=True)
    return pol


@pytest.mark.parametrize("n", [250, 1000, 12345, 2 ** 31 - 5])
def test_one_randint_equals_the_choice_loop(n):
    """epochs x int(N/mb) calls of np.random.choice(N, size=mb) == one np.random.randint call: values and the global
    generator state afterwards."""
    from mjrl_b200.algos.ppo_clip import minibatch_indices
    mb, epochs = 64, 3
    per_epoch = min(int(n / mb), 40)
    np.random.seed(5)
    np.random.rand(3)
    want = np.stack([np.random.choice(n, size=mb) for _ in range(epochs * per_epoch)])
    after_want = np.random.get_state()
    np.random.seed(5)
    np.random.rand(3)
    got = np.random.randint(0, n, size=epochs * per_epoch * mb).reshape(-1, mb)
    after_got = np.random.get_state()
    assert np.array_equal(got, want)
    assert after_got[2] == after_want[2] and np.array_equal(after_got[1], after_want[1])
    if n <= 100000:
        np.random.seed(9)
        ref = np.stack([np.random.choice(n, size=mb) for _ in range(epochs * int(n / mb))])
        np.random.seed(9)
        blk = minibatch_indices(n, mb, epochs)
        assert blk.dtype == np.int32 and np.array_equal(blk, ref)


@pytest.mark.parametrize("n,mb,epochs,rows", [(1000, 64, 10, 150), (127, 64, 2, 2), (63, 64, 5, 0), (640, 64, 1, 10),
                                             (100, 7, 3, 42)])
def test_index_block_shape(n, mb, epochs, rows):
    from mjrl_b200.algos.ppo_clip import minibatch_indices
    blk = minibatch_indices(n, mb, epochs)
    assert blk.shape == (rows, mb) and blk.dtype == np.int32
    assert rows == 0 or (blk.min() >= 0 and blk.max() < n)


def _order_of_calls(agent_cls, monkeypatch, **kw):
    from mjrl_b200.policies.gaussian_mlp import MLP
    from mjrl_b200.utils import process_samples
    from mjrl_b200.utils.gym_env import EnvSpec
    calls = []

    class Baseline:
        def fit_begin(self, paths, return_errors=False):
            calls.append("fit_begin")

        def fit_defer(self):
            calls.append("fit_defer")

        def fit(self, paths, return_errors=False):
            calls.append("fit")

        def _bind(self, eng):
            pass

    for name in ("returns_on", "returns_write_back", "advantages_on"):
        monkeypatch.setattr(process_samples, name, lambda *a, **k: None)
    agent = agent_cls(None, MLP(EnvSpec(4, 2, 10), hidden_sizes=(32, 32), seed=1), Baseline(), **kw)
    agent.train_from_paths = lambda paths: calls.append("train") or [0.0] * 4
    agent._update_resident(None, [dict(rewards=np.zeros(3))], 0.995, 0.97)
    return calls


def test_ppo_fits_the_baseline_after_its_minibatch_draws(monkeypatch):
    """The reference draws PPO's minibatch indices before the baseline fit's permutations: no fit overlap for PPO,
    unchanged overlap for NPG / TRPO / DAPG."""
    from mjrl_b200.algos.dapg import DAPG
    from mjrl_b200.algos.npg_cg import NPG
    from mjrl_b200.algos.ppo_clip import PPO
    from mjrl_b200.algos.trpo import TRPO
    assert _order_of_calls(PPO, monkeypatch) == ["train", "fit"]
    assert _order_of_calls(NPG, monkeypatch) == ["fit_begin", "train", "fit_defer"]
    assert _order_of_calls(TRPO, monkeypatch) == ["fit_begin", "train", "fit_defer"]
    assert _order_of_calls(DAPG, monkeypatch, demo_paths=None) == ["fit_begin", "train", "fit_defer"]
    with pytest.raises(NotImplementedError):
        PPO(None, _order_of_calls.__globals__["np"] and __import__("mjrl_b200.policies.gaussian_mlp", fromlist=["MLP"]).MLP(
            __import__("mjrl_b200.utils.gym_env", fromlist=["EnvSpec"]).EnvSpec(4, 2, 10), (32, 32)), None).update_from_rollouts({})


def test_agents_refuse_what_the_kernel_does_not_run():
    from mjrl_b200.algos.behavior_cloning import BC
    from mjrl_b200.algos.ppo_clip import PPO
    from mjrl_b200.policies.gaussian_linear import LinearPolicy
    from mjrl_b200.policies.gaussian_mlp import MLP
    from mjrl_b200.utils.gym_env import EnvSpec
    pol = MLP(EnvSpec(4, 2, 10), hidden_sizes=(32, 32), seed=1)
    with pytest.raises(NotImplementedError, match="optimizer"):
        BC([], pol, optimizer=object())
    with pytest.raises(ValueError, match="loss_type"):
        BC([], pol, loss_type="RWR")
    with pytest.raises(ValueError, match="64"):
        BC([], pol, batch_size=128)
    with pytest.raises(ValueError, match="64"):
        PPO(None, pol, None, mb_size=65)
    with pytest.raises(NotImplementedError, match="LinearPolicy"):
        PPO(None, LinearPolicy(EnvSpec(4, 2, 10), seed=0), None)


@pytest.mark.parametrize("case", CASES)
def test_oracle_matches_reference_fixture(case):
    g = load_golden(case)
    meta = g["meta"]
    pol = initial_theta(meta)
    theta0 = pol.get_param_values()
    assert PB.compare(theta0, g, "theta0", meta) == 0.0
    if meta["kind"] == "ppo":
        assert np.mean(g["clipfrac1"]) > (0.1 if "clipheavy" in case else -1)
    spec = PB.case_spec(meta, g)
    res = PB.run_case(meta, spec, theta0)
    for call, r in enumerate(res, 1):
        assert r["step"] == int(g["step%d" % call])
        assert len(r["loss"]) == len(g["loss%d" % call])
        if meta["kind"] == "ppo" and call == 2:
            # From the second call on the reference's old network aliases the new one: set_param_values builds both from
            # one numpy buffer, so the in-place Adam steps move old_model too (DESIGN 2.7).  Until the first step the two
            # agree; this package keeps the old policy fixed, as PPO defines it.
            np.testing.assert_allclose(r["loss"][0], g["loss2"][0], rtol=1e-5, atol=1e-7)
            continue
        np.testing.assert_allclose(r["loss"], g["loss%d" % call], rtol=1e-4, atol=1e-6)
        for key in ("theta", "m", "v"):
            assert PB.compare(r[key], g, "%s%d" % (key, call), meta) < (1e-5 if key == "theta" else 1e-3), (key, call)
        if meta["kind"] == "ppo":
            np.testing.assert_allclose(r["surr"][:2], g["surr%d" % call], rtol=1e-4, atol=1e-6)
            np.testing.assert_allclose(r["surr"][2], g["kl%d" % call], rtol=1e-3, atol=1e-9)
            np.testing.assert_allclose(r["clipfrac"], g["clipfrac%d" % call], atol=1.0 / meta["mb"] + 1e-6)
        else:
            np.testing.assert_allclose(r["bcloss"], g["bcloss%d" % call], rtol=1e-5)
    assert np.array_equal(np.random.randint(0, 1 << 30, size=4), g["rng_after"])
