"""CPU tests: the oracle restatement (oracle/npg_oracle.py) against (a) known-answer vectors and
(b) the golden fixtures produced by the real reference (oracle/make_golden.py), and (c) one reference
NPG step on shapes of its own (oracle/make_golden_host.py).  Tolerances: bit-exact for returns/GAE/indexing; fp32
autograd flavour == reference to ~1e-6; fp64 closed form == reference to fp32 rounding."""
import numpy as np
import pytest
import torch

from conftest import ALL_CASES, golden_equal, golden_paths, load_golden, one_minus_cos, rel
from oracle import npg_oracle as O


def spec_of(g):
    m = g["meta"]
    return O.PolicySpec(m["obs_dim"], m["act_dim"], m["hidden"])


def vf_of(g, w="vf_w0"):
    vf = O.VFState(g["meta"]["obs_dim"], (128, 128))
    vf.w = g[w].copy()
    return vf


def test_known_answers():
    k = load_golden("kat")
    assert np.array_equal(O.discount_sum(k["ds_in"], 0.5), [3.25, 4.5, 5.0, 4.0])
    assert np.array_equal(O.discount_sum(k["ds_in"], 0.5), k["ds_out"])
    f32 = O.discount_sum(k["ds_in"].astype(np.float32), 0.5)
    assert f32.dtype == np.float32 and np.array_equal(f32, k["ds_f32_out"])
    assert O.discount_sum(np.zeros(0), 0.9).shape == (0,)
    r, b = k["gae_r"], k["gae_b"]
    assert np.array_equal(O.discount_sum(r, 0.9), k["gae_ret"])
    assert np.array_equal(O.gae_path(r, b, False, 0.9, 0.5), k["gae_adv_term0"])
    assert np.array_equal(O.gae_path(r, b, True, 0.9, 0.5), k["gae_adv_term1"])
    np.testing.assert_allclose(k["gae_adv_term1"], [1.243625, -0.3475, 3.45, -3.0], rtol=1e-12)
    assert np.array_equal(O.discount_sum(r, 0.9) - b, k["nogae_adv"])
    A = np.array([[4.0, 1.0], [1.0, 3.0]])
    bb = np.array([1.0, 2.0])
    assert np.array_equal(O.cg_solve(lambda v: A.dot(v), bb, 1), k["cg_1"])
    np.testing.assert_allclose(O.cg_solve(lambda v: A.dot(v), bb, 2), [1 / 11, 7 / 11], rtol=1e-12)
    feat = O.vf_features([dict(observations=k["feat_obs"], rewards=np.zeros(2))])
    assert np.array_equal(feat, k["feat_out"])
    for dims, d in (((6, 2, (32, 32)), 1348), ((8, 2, (64, 64)), 4868), ((17, 6, (128, 128)), 19596),
                    ((39, 28, (256, 256)), 83256), ((376, 17, ()), 6426)):
        assert O.PolicySpec(*dims).d == d


@pytest.mark.parametrize("case", ALL_CASES)
def test_golden_returns_gae_bitexact(case):
    g = load_golden(case)
    paths = golden_paths(g)
    vf = vf_of(g)
    assert np.array_equal(O.init_policy_params(spec_of(g), g["meta"]["policy_seed"]), g["theta0"])
    O.compute_returns(paths, g["meta"]["gamma"])
    O.compute_advantages(paths, lambda p: O.vf_predict(vf, p), g["meta"]["gamma"], g["meta"]["lam"])
    cat = lambda k: np.concatenate([p[k] for p in paths])
    assert np.array_equal(cat("returns"), g["returns"])
    np.testing.assert_allclose(cat("baseline"), g["baseline"], rtol=0, atol=2e-6)
    # GAE is bit-exact given the reference's own baseline predictions
    k = 0
    for p in paths:
        T = len(p["rewards"])
        adv = O.gae_path(p["rewards"], g["baseline"][k:k + T], p["terminated"], g["meta"]["gamma"], g["meta"]["lam"])
        assert np.array_equal(adv, g["advantages"][k:k + T])
        assert np.array_equal(p["returns"] - g["baseline"][k:k + T], g["advantages_nogae"][k:k + T])
        k += T
    np.testing.assert_allclose(O.whiten(g["advantages"]), g["adv_white"], rtol=0, atol=1e-12)
    stats, _ = O.path_stats(paths, None)
    np.testing.assert_allclose(stats, g["base_stats"], rtol=1e-12)


@pytest.mark.parametrize("case", ALL_CASES)
def test_golden_gradients(case):
    g = load_golden(case)
    paths = golden_paths(g)
    spec = spec_of(g)
    obs = np.concatenate([p["observations"] for p in paths])
    act = np.concatenate([p["actions"] for p in paths])
    adv = g["adv_white"]
    th = g["theta0"]
    for kw, tol in ((dict(dtype=torch.float32, autograd=True), 2e-6), (dict(dtype=torch.float64), 2e-6)):
        a = adv.astype(np.float32) if kw["dtype"] == torch.float32 else adv
        assert rel(O.flat_vpg(spec, th, obs, act, a, **kw), g["vpg"]) < tol
        assert rel(O.fvp(spec, th, obs, g["fvp_vec"], g["meta"]["damping"], **kw), g["fvp_out"]) < tol
        assert rel(O.flat_vpg(spec, g["theta_pert"], obs, act, a, theta_old=th, **kw), g["vpg_pert"]) < 5e-6
    # the FVP does not depend on the actions (SURVEY headline 3)
    assert abs(float(O.surrogate(spec, th, th, obs, act, adv)) - g["surr0"]) < 1e-6
    assert abs(float(O.surrogate(spec, g["theta_pert"], th, obs, act, adv)) - g["surr_pert"]) < 2e-5 * max(1, abs(g["surr_pert"]))
    assert abs(float(O.mean_kl(spec, g["theta_pert"], th, obs)) - g["kl_pert"]) < 1e-5 * max(1.0, g["kl_pert"])


@pytest.mark.parametrize("case", ALL_CASES)
def test_golden_updates(case):
    g = load_golden(case)
    paths = golden_paths(g)
    m = g["meta"]
    spec = spec_of(g)
    obs = np.concatenate([p["observations"] for p in paths])
    act = np.concatenate([p["actions"] for p in paths])
    adv, th = g["adv_white"], g["theta0"]
    well_conditioned = obs.shape[0] > 4 * spec.d / max(1, spec.act_dim) or len(m["hidden"]) == 0
    o = O.policy_update(spec, th, obs, act, adv, "npg", step_size=m["npg_step"])
    if well_conditioned:
        assert rel(o["new_params"], g["npg_theta"]) < 1e-4
    # N < d cases (rank-deficient Fisher + 1e-4 damping) amplify fp32 thread-order noise ~1e3x
    # (even the reference's own fp32 CG is 1.4e-4 in cosine from the fp64 solution on pm_40x25_ragged)
    stol = 2e-3 if well_conditioned else 3e-2
    ctol = 1e-4 if well_conditioned else 5e-3
    assert one_minus_cos(o["npg_grad"], g["cg_x"]) < ctol
    assert one_minus_cos(o["new_params"] - th, g["npg_theta"] - th) < ctol
    assert abs(o["alpha"] / g["npg_alpha"] - 1) < stol
    assert abs(o["kl_dist"] / g["npg_kl_dist"] - 1) < 3 * stol
    for tag, kl in (("trpo", 0.01), ("trpo_big", 0.5)):
        t = O.policy_update(spec, th, obs, act, adv, "trpo", kl_dist=kl)
        assert t["backtracks"] == int(g[tag + "_backtracks"])
        assert one_minus_cos(t["new_params"] - th, g[tag + "_theta"] - th) < ctol
        assert abs(t["alpha"] / g[tag + "_alpha"] - 1) < stol
    demo = golden_paths(g, demo=True)
    d_obs = np.concatenate([p["observations"] for p in demo])
    d_act = np.concatenate([p["actions"] for p in demo])
    batch = O.dapg_batch(obs, act, adv, d_obs, d_act, 1.0, 0.95, 3.0)
    dd = O.policy_update(spec, th, obs, act, adv, "dapg", kl_dist=0.01, grad_batch=batch)
    assert one_minus_cos(dd["new_params"] - th, g["dapg_theta"] - th) < ctol
    assert abs(dd["alpha"] / g["dapg_alpha"] - 1) < stol
    sub = O.policy_update(spec, th, obs, act, adv, "npg", step_size=m["npg_step"], hvp_idx=list(g["sub_idx"]))
    assert one_minus_cos(sub["new_params"] - th, g["sub_theta"] - th) < ctol


@pytest.mark.parametrize("case", [c for c in ALL_CASES if c != "cheetah_24x500"])
def test_golden_baseline_fit(case):
    g = load_golden(case)
    paths = golden_paths(g)
    O.compute_returns(paths, g["meta"]["gamma"])
    vf = vf_of(g)
    e = O.vf_fit(vf, paths, list(g["fit_perms"][:2]), 2, 64, 1e-3, 1e-3, return_errors=True)
    np.testing.assert_allclose(e, g["fit1_err"], rtol=1e-4)
    assert rel(vf.w, g["fit1_w"]) < 1e-5
    O.vf_fit(vf, paths, list(g["fit_perms"][2:4]), 2, 64, 1e-3, 1e-3)
    # Adam normalises near-zero gradients of dead ReLU units, so raw weights drift (2e-3 after 440 steps on
    # swim_40x250) in directions that do not change the function: gate the second call on predictions.
    assert rel(vf.w, g["fit2_w"]) < 2e-2
    assert vf.t == int(g["fit2_step"])
    assert rel(vf.v, g["fit2_v"]) < 1e-3
    pred = np.concatenate([O.vf_predict(vf, p) for p in paths])
    np.testing.assert_allclose(pred, g["fit2_predict"], rtol=0, atol=1e-4)


def test_fit_torch_flavour_equals_explicit_adam():
    g = load_golden("swim_40x250")
    paths = golden_paths(g)
    O.compute_returns(paths, g["meta"]["gamma"])
    a, b = vf_of(g), vf_of(g)
    O.vf_fit(a, paths, list(g["fit_perms"][:1]), 1, 64, 1e-3, 1e-3)
    O.vf_fit_torch(b, paths, list(g["fit_perms"][:1]), 1, 64, 1e-3, 1e-3)
    assert a.t == b.t and rel(a.w, b.w) < 1e-5


def test_fit_needs_two_batches():
    paths = O.synthetic_paths(3, 1, 2, 50, seed=0)
    O.compute_returns(paths, 0.9)
    with pytest.raises(ValueError):
        O.vf_fit(O.VFState(3), paths, [np.arange(100)])


def test_live_reference_npg_step():
    """Shapes not in the other goldens: oracle (fp32 autograd flavour) vs one NPG step of the reference, whose
    initial weights, returns, advantages and new parameters are stored in tests/golden/npg_11x3_ragged.npz."""
    g = load_golden("npg_11x3_ragged")
    torch.set_num_threads(1)
    obs_dim, act_dim, hidden = 11, 3, (64, 64)
    paths = O.synthetic_paths(obs_dim, act_dim, 30, 300, seed=3, ragged=True)
    spec = O.PolicySpec(obs_dim, act_dim, hidden)
    th = g["theta0"]
    vf = O.VFState(obs_dim)
    vf.w = g["vf_w"].copy()
    O.compute_returns(paths, 0.995)
    O.compute_advantages(paths, lambda p: O.vf_predict(vf, p), 0.995, 0.97)
    assert golden_equal(np.concatenate([p["returns"] for p in paths]), g, "returns")
    assert golden_equal(np.concatenate([p["advantages"] for p in paths]), g, "advantages")
    obs = np.concatenate([p["observations"] for p in paths])
    act = np.concatenate([p["actions"] for p in paths])
    adv = O.whiten(np.concatenate([p["advantages"] for p in paths]))
    o = O.policy_update(spec, th, obs, act, adv, "npg", step_size=0.05)
    assert rel(o["new_params"], g["new_params"]) < 1e-4
