"""GPU tests of PPO-clip and behaviour cloning (csrc/policy_sgd.cu behind mjrl_b200.algos.ppo_clip.PPO and
mjrl_b200.algos.behavior_cloning.BC) against the reference fixtures and the fp32 oracle."""
import numpy as np
import pytest

from conftest import load_golden
from oracle import npg_oracle as O
from oracle import ppo_bc_oracle as PB
from test_ppo_bc_cpu import CASES, initial_theta

pytestmark = pytest.mark.gpu


def _run_agent(meta, calls=2, record=True):
    """Our agent on a fixture case: returns the policy, the agent and one dict per call."""
    from mjrl_b200.algos.behavior_cloning import BC
    from mjrl_b200.algos.ppo_clip import PPO
    pol = initial_theta(meta)
    out = []
    if meta["kind"] == "ppo":
        agent = PPO(None, pol, None, clip_coef=meta["clip"], epochs=meta["epochs"], mb_size=meta["mb"],
                    learn_rate=meta["lr"])
    else:
        agent = BC(PB.case_paths(meta, 0), pol, epochs=meta["epochs"], batch_size=meta["mb"], lr=meta["lr"],
                   loss_type=meta["loss"], set_transforms=False)
    agent.record_minibatch_stats = record
    np.random.seed(meta["rng_seed"])
    for call in range(calls):
        r = {}
        if meta["kind"] == "ppo":
            agent.train_from_paths(PB.case_paths(meta, call))
            st = agent.last_stats
            r["surr"] = (st["surr_before"], st["surr_after"], st["kl_dist"])
            r["clipfrac"] = agent.last_clip_frac
        else:
            agent.train()
            r["bcloss"] = (agent.logger.log["loss_before"][-1], agent.logger.log["loss_after"][-1])
        r["loss"] = agent.last_minibatch_loss
        r["theta"] = pol.get_param_values()
        r["m"], r["v"], r["step"] = agent.adam.m.copy(), agent.adam.v.copy(), agent.adam.step
        out.append(r)
    return pol, agent, out


@pytest.mark.parametrize("case", CASES)
def test_matches_reference(cuda_device, case):
    g = load_golden(case)
    meta = g["meta"]
    _, _, got = _run_agent(meta)
    oracle = PB.run_case(meta, PB.case_spec(meta, g), initial_theta(meta).get_param_values())
    for call, (r, o) in enumerate(zip(got, oracle), 1):
        assert r["step"] == o["step"] == int(g["step%d" % call])
        if meta["kind"] == "ppo" and call == 2:
            # the reference's old network aliases the new one from the second call on (DESIGN 2.7): the fp32 oracle,
            # which keeps the old policy fixed as this package does, is the yardstick here
            np.testing.assert_allclose(r["loss"][:3], o["loss"][:3], rtol=1e-3, atol=1e-6)
            if "clipheavy" not in case:
                # (at learn_rate 2e-2 with a quarter of the rows clipped, last-bit differences grow step by step over
                # the 60 steps of a call; the first call above holds the 1e-4 gate, here the onset is checked)
                assert PB.compare(r["theta"], {"t": o["theta"]}, "t", meta) < 1e-3
                np.testing.assert_allclose(r["surr"], o["surr"], rtol=1e-2, atol=1e-5)
            continue
        # per-step minibatch losses over the first steps; theta after the first call within 1e-4
        k = min(8, len(r["loss"]))
        np.testing.assert_allclose(r["loss"][:k], g["loss%d" % call][:k], rtol=1e-3, atol=1e-6)
        tol = 1e-4 if call == 1 else max(1e-3, 20 * PB.compare(o["theta"], g, "theta2", meta))
        assert PB.compare(r["theta"], g, "theta%d" % call, meta) < tol, call
        if meta["kind"] == "ppo":
            np.testing.assert_allclose(r["surr"][:2], g["surr%d" % call], rtol=1e-3, atol=1e-6)
            np.testing.assert_allclose(r["surr"][2], g["kl%d" % call], rtol=1e-3, atol=1e-8)
            assert abs(float(np.mean(r["clipfrac"])) - float(np.mean(g["clipfrac%d" % call]))) < 0.02
        else:
            np.testing.assert_allclose(r["bcloss"], g["bcloss%d" % call], rtol=1e-3)
    if "clipheavy" in case:
        assert float(np.mean(got[0]["clipfrac"])) > 0.1


def test_mse_leaves_log_std_untouched(cuda_device):
    g = load_golden("bc_mse_17x6_h128")
    meta = g["meta"]
    pol = initial_theta(meta)
    from mjrl_b200.algos.behavior_cloning import BC
    agent = BC(PB.case_paths(meta, 0), pol, epochs=1, batch_size=64, loss_type='MSE', save_logs=False)
    A = meta["act_dim"]
    ls0 = pol.get_param_values()[-A:].copy()
    agent.adam.m[-A:] = np.float32(0.25)
    agent.adam.v[-A:] = np.float32(0.5)
    m0, v0 = agent.adam.m[-A:].copy(), agent.adam.v[-A:].copy()
    np.random.seed(0)
    agent.train()
    assert np.array_equal(pol.get_param_values()[-A:], ls0)
    assert np.array_equal(agent.adam.m[-A:], m0) and np.array_equal(agent.adam.v[-A:], v0)
    assert agent.adam.step > 0 and not np.array_equal(pol.get_param_values()[:-A], initial_theta(meta).get_param_values()[:-A])


def test_repeat_is_bit_identical(cuda_device):
    meta = load_golden("ppo_clipheavy_6x2_h64")["meta"]
    _, _, a = _run_agent(meta)
    _, _, b = _run_agent(meta)
    for x, y in zip(a, b):
        for k in ("theta", "m", "v", "loss", "clipfrac"):
            assert np.array_equal(x[k], y[k]), k


def test_engine_growth_and_shared_policy(cuda_device):
    """PPO on a small batch, then on one large enough to replace the engine; BC before PPO on one shared policy: the
    Adam state follows the agents through engine replacement and shared engines."""
    from mjrl_b200 import runtime
    from mjrl_b200.algos.behavior_cloning import BC
    from mjrl_b200.algos.ppo_clip import PPO
    from mjrl_b200.policies.gaussian_mlp import MLP
    from mjrl_b200.utils.gym_env import EnvSpec
    runtime.shutdown()
    obs_dim, act_dim, hidden = 9, 3, (64, 64)
    spec = O.PolicySpec(obs_dim, act_dim, hidden)
    pol = MLP(EnvSpec(obs_dim, act_dim, 100), hidden_sizes=hidden, seed=21)
    theta = pol.get_param_values()
    demo = O.synthetic_paths(obs_dim, act_dim, 3, 100, seed=4)
    small = O.synthetic_paths(obs_dim, act_dim, 4, 100, seed=5)
    big = O.synthetic_paths(obs_dim, act_dim, 60, 400, seed=6)          # 24 000 rows > the first engine's capacity
    for ps, s in ((small, 1), (big, 2)):
        rng = np.random.RandomState(s)
        for p in ps:
            p["advantages"] = rng.randn(len(p["rewards"]))
    bc = BC(demo, pol, epochs=2, batch_size=64, lr=1e-3, loss_type='MLE', save_logs=False)
    ppo = PPO(None, pol, None, epochs=1, mb_size=64, learn_rate=3e-4)
    np.random.seed(8)
    bc.train()
    ppo.train_from_paths(small)
    eng_small = ppo._engine
    bc.train()                                        # BC's own Adam state goes back into the shared engine
    ppo.train_from_paths(big)
    assert ppo._engine is not eng_small               # the engine was replaced by a larger one
    # oracle: the same sequence uninterrupted, one Adam state per agent
    np.random.seed(8)
    adam_bc, adam_ppo = PB.AdamState(spec.d), PB.AdamState(spec.d)

    def bc_call(th):
        obs = np.concatenate([p["observations"] for p in demo]); act = np.concatenate([p["actions"] for p in demo])
        idx = PB.minibatch_indices(obs.shape[0], 64, 2)
        return spec.clamp(PB.train(spec, th, adam_bc, obs, act, idx, 1e-3, "mle")[0])

    def ppo_call(th, ps):
        obs = np.concatenate([p["observations"] for p in ps]); act = np.concatenate([p["actions"] for p in ps])
        adv = np.concatenate([p["advantages"] for p in ps])
        adv = ((adv - adv.mean()) / (adv.std() + 1e-6)).astype(np.float32)
        _, llo = PB.log_likelihood(spec, th, obs, act)
        idx = PB.minibatch_indices(obs.shape[0], 64, 1)
        return spec.clamp(PB.train(spec, th, adam_ppo, obs, act, idx, 3e-4, "ppo", adv, llo)[0])

    th = ppo_call(bc_call(theta), small)
    th = ppo_call(bc_call(th), big)
    assert ppo.adam.step == adam_ppo.step and bc.adam.step == adam_bc.step
    assert PB.compare(pol.get_param_values(), {"t": th}, "t", None) < 1e-3
    runtime.shutdown()


def test_cfg3_full_size_properties(cuda_device):
    """cfg3 policy shape (17 -> 128 x 128 -> 6), 1e6 samples, one epoch: the surrogate improves, the KL is finite,
    the clip fraction is reported and a repeat from the same state is bit-identical."""
    from mjrl_b200.engine import Engine
    obs_dim, act_dim, hidden, N = 17, 6, (128, 128), 1_000_000
    spec = O.PolicySpec(obs_dim, act_dim, hidden)
    theta = O.init_policy_params(spec, 3)
    rng = np.random.RandomState(0)
    obs, act = rng.randn(N, obs_dim), 0.1 * rng.randn(N, act_dim)
    adv = rng.randn(N)
    eng = Engine(obs_dim, act_dim, hidden, max_samples=N + 64, max_paths=8)
    eng.upload_flat(obs, act, np.zeros(N), np.array([N], np.int32), np.zeros(1, np.uint8))
    eng.set_advantages(adv)
    eng.process_paths()
    np.random.seed(1)
    idx = PB.minibatch_indices(N, 64, 1).astype(np.int32)
    runs = []
    for _ in range(2):
        eng.set_params(theta)
        eng.adam_set(np.zeros(spec.d, np.float32), np.zeros(spec.d, np.float32), 0)
        before = eng.eval()
        loss, clip = eng.policy_sgd("ppo", idx, 3e-4, 0.2, want_outputs=True)
        after = eng.eval()
        runs.append((eng.get_params(), eng.adam_get(), loss, clip, before, after, eng.last_sgd_ms()))
    (t1, a1, l1, c1, b1, f1, ms), (t2, a2, l2, c2, b2, f2, _) = runs
    assert f1[0] > b1[0] and np.isfinite(f1[1]) and f1[1] > 0
    assert len(c1) == len(idx) and 0.0 <= float(c1.mean()) < 1.0
    assert np.array_equal(t1, t2) and np.array_equal(a1[0], a2[0]) and np.array_equal(a1[1], a2[1])
    assert np.array_equal(l1, l2) and np.array_equal(c1, c2) and f1 == f2
    print("cfg3 1e6 x 1 epoch: %d steps, %.2f us/step, surr %.5f -> %.5f, kl %.3g, clip frac %.3f" % (
        len(idx), 1e3 * ms / len(idx), b1[0], f1[0], f1[1], float(c1.mean())))
    eng.close()
