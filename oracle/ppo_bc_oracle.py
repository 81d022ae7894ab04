"""TEST INFRASTRUCTURE ONLY -- a small torch-fp32 restatement of the PPO-clip and behaviour-cloning minibatch loops
(mjrl/algos/ppo_clip.py:48-102, mjrl/algos/behavior_cloning.py:74-136) on a flat parameter vector.

Gradients come from torch autograd through the same expressions the reference builds; the Adam update is torch.optim.Adam's
single-tensor arithmetic written out, so the optimizer state (m, v, step) can be carried across calls and compared.  The
GPU tests use it for shapes and sizes that have no reference fixture; tests/test_ppo_bc_oracle.py pins it to the fixtures
that oracle/make_golden_ppo_bc.py wrote from the reference itself."""
import math

import numpy as np
import torch

from oracle import npg_oracle as O

BETA1, BETA2, EPS = 0.9, 0.999, 1e-8


def minibatch_indices(num_samples, mb_size, epochs):
    """The reference's epochs x int(N / mb) calls of np.random.choice(N, size=mb) as ONE np.random.randint call: same
    values, same global RNG state afterwards (the legacy bounded-integer path draws per value and buffers nothing)."""
    steps = epochs * int(num_samples / mb_size)
    return np.random.randint(0, num_samples, size=steps * mb_size).reshape(steps, mb_size)


class AdamState:
    def __init__(self, d):
        self.m, self.v, self.step = np.zeros(d, np.float32), np.zeros(d, np.float32), 0


def _adam(p, g, m, v, t, lr):
    m.lerp_(g, 1 - BETA1)
    v.mul_(BETA2).addcmul_(g, g, value=1 - BETA2)
    bc1, bc2 = 1 - BETA1 ** t, 1 - BETA2 ** t
    denom = (v.sqrt() / math.sqrt(bc2)).add_(EPS)
    p.addcdiv_(m, denom, value=-lr / bc1)


def _mean_ll(spec, params, obs, act):
    layers, log_std = params[:-1], params[-1]
    h = (obs - torch.from_numpy(spec.in_shift)) / (torch.from_numpy(spec.in_scale) + 1e-8)
    for i in range(0, len(layers) - 2, 2):
        h = torch.tanh(h @ layers[i].T + layers[i + 1])
    mu = (h @ layers[-2].T + layers[-1]) * torch.from_numpy(spec.out_scale) + torch.from_numpy(spec.out_shift)
    z = (act - mu) / torch.exp(log_std)
    ll = -0.5 * torch.sum(z ** 2, dim=1) - torch.sum(log_std) - 0.5 * spec.act_dim * np.log(2 * np.pi)
    return mu, ll


def _split(spec, theta):
    th = torch.from_numpy(np.array(theta, np.float32))
    layers, log_std = spec.split(th)
    out = []
    for W, b in layers:
        out += [W.clone(), b.clone()]
    return out + [log_std.clone()]


def train(spec, theta, adam, obs, act, idx, lr, loss, adv=None, ll_old=None, clip_coef=0.2):
    """len(idx) sequential Adam steps; loss in ("ppo", "mle", "mse").  Returns (theta, per-step minibatch losses, per-step
    fraction of rows whose gradient the clip zeroed).  `adam` is updated in place.  No log_std clamp inside the chain."""
    params = [p.requires_grad_(True) for p in _split(spec, theta)]
    sizes = [p.numel() for p in params]
    bounds = np.concatenate([[0], np.cumsum(sizes)])
    m = [torch.from_numpy(adam.m[lo:hi].copy()).reshape(p.shape) for p, lo, hi in zip(params, bounds[:-1], bounds[1:])]
    v = [torch.from_numpy(adam.v[lo:hi].copy()).reshape(p.shape) for p, lo, hi in zip(params, bounds[:-1], bounds[1:])]
    obs_t, act_t = torch.from_numpy(np.asarray(obs, np.float32)), torch.from_numpy(np.asarray(act, np.float32))
    losses, clipped = [], []
    for rows in idx:
        rows = torch.as_tensor(np.asarray(rows, np.int64))
        for p in params:
            p.grad = None
        mu, ll = _mean_ll(spec, params, obs_t[rows], act_t[rows])
        if loss == "ppo":
            a = torch.from_numpy(np.asarray(adv, np.float32))[rows]
            lr_ = torch.exp(ll - torch.from_numpy(np.asarray(ll_old, np.float32))[rows])
            lc = torch.clamp(lr_, min=1 - clip_coef, max=1 + clip_coef)
            val = -torch.mean(torch.min(lr_ * a, lc * a))
            with torch.no_grad():
                live = ((lr_ >= 1 - clip_coef) & (lr_ <= 1 + clip_coef)) | (lr_ * a < lc * a)
                clipped.append(1.0 - float(live.float().mean()))
        elif loss == "mle":
            val = -torch.mean(ll)
        else:
            val = torch.mean((mu - act_t[rows]) ** 2)
        val.backward()
        losses.append(float(val.detach()))
        adam.step += 1
        with torch.no_grad():
            for p, mm, vv in zip(params, m, v):
                if p.grad is not None:               # MSE: log_std is not in the graph, torch's Adam skips it
                    _adam(p, p.grad, mm, vv, adam.step, lr)
    flat = lambda ts: np.concatenate([t.detach().reshape(-1).numpy() for t in ts]).astype(np.float32)
    adam.m, adam.v = flat(m), flat(v)
    return flat(params), np.array(losses, np.float32), np.array(clipped, np.float32)


def log_likelihood(spec, theta, obs, act):
    with torch.no_grad():
        mu, ll = _mean_ll(spec, _split(spec, theta), torch.from_numpy(np.asarray(obs, np.float32)),
                          torch.from_numpy(np.asarray(act, np.float32)))
    return mu.numpy(), ll.numpy()


def bc_loss(spec, theta, obs, act, loss):
    mu, ll = log_likelihood(spec, theta, obs, act)
    if loss == "mle":
        return float(-np.mean(ll, dtype=np.float32))
    return float(np.mean((mu - np.asarray(act, np.float32)) ** 2, dtype=np.float32))


def ppo_eval(spec, theta_new, theta_old, obs, act, adv, spec_old=None):
    """(surrogate, mean KL) of CPI_surrogate / kl_old_new (batch_reinforce.py:40-52) in fp32."""
    s = O.surrogate(spec, theta_new, theta_old, obs, act, adv, dtype=torch.float32, spec_old=spec_old)
    k = O.mean_kl(spec, theta_new, theta_old, obs, dtype=torch.float32, spec_old=spec_old)
    return float(s), float(k)


# ---------------------------------------------------------------------------------------------
# fixture cases (oracle/make_golden_ppo_bc.py writes them, the tests regenerate their inputs)
# ---------------------------------------------------------------------------------------------
def case_paths(meta, call):
    """The batch of call 0 / 1 of a fixture case (PPO: two batches, BC: the same demonstrations twice), with seeded
    advantages."""
    seed = meta["path_seed"] + (call if meta["kind"] == "ppo" else 0)
    paths = O.synthetic_paths(meta["obs_dim"], meta["act_dim"], meta["n_paths"], meta["horizon"], seed=seed,
                              ragged=meta["ragged"])
    rng = np.random.RandomState(meta["adv_seed"] + call)
    for p in paths:
        p["advantages"] = rng.randn(len(p["rewards"]))
    return paths


def block_bounds(meta):
    h1, h2 = meta["hidden"]
    sizes = [h1 * meta["obs_dim"], h1, h2 * h1, h2, meta["act_dim"] * h2, meta["act_dim"], meta["act_dim"]]
    return np.concatenate([[0], np.cumsum(sizes)])


def compare(a, g, key, meta):
    """Relative error of `a` against the fixture vector `key`: over the whole vector, or over the stored sample and
    the per-block norms (the larger of the two)."""
    a = np.asarray(a, np.float64)
    if key in g:
        b = np.asarray(g[key], np.float64)
        return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-30))
    idx = np.sort(np.random.RandomState(0).choice(a.size, g[key + "@sample"].size, replace=False))
    b = np.asarray(g[key + "@sample"], np.float64)
    e1 = float(np.linalg.norm(a[idx] - b) / (np.linalg.norm(b) + 1e-30))
    bb = block_bounds(meta)
    norms = np.array([np.linalg.norm(a[lo:hi]) for lo, hi in zip(bb[:-1], bb[1:])])
    e2 = float(np.max(np.abs(norms - g[key + "@norms"]) / (g[key + "@norms"] + 1e-30)))
    return max(e1, e2)


def case_spec(meta, g):
    kw = {}
    if meta.get("set_transforms"):
        kw = dict(in_shift=g["in_shift"], in_scale=g["in_scale"], out_shift=g["out_shift"], out_scale=g["out_scale"])
    return O.PolicySpec(meta["obs_dim"], meta["act_dim"], meta["hidden"], **kw)


def run_case(meta, spec, theta0, calls=2):
    """The fixture's two consecutive calls restated in fp32 (global numpy RNG seeded as the generator did).  Returns one
    dict per call: theta (clamped, as set_param_values leaves it), adam (m, v, step), losses, clipfrac and
    surr / kl (PPO) or bc loss before / after."""
    np.random.seed(meta["rng_seed"])
    adam = AdamState(spec.d)
    theta = np.array(theta0, np.float32)
    out = []
    for call in range(calls):
        paths = case_paths(meta, call)
        obs = np.concatenate([p["observations"] for p in paths])
        act = np.concatenate([p["actions"] for p in paths])
        n = obs.shape[0]
        r = {}
        if meta["kind"] == "ppo":
            adv = np.concatenate([p["advantages"] for p in paths])
            adv = ((adv - np.mean(adv)) / (np.std(adv) + 1e-6)).astype(np.float32)
            _, ll_old = log_likelihood(spec, theta, obs, act)
            idx = minibatch_indices(n, meta["mb"], meta["epochs"])
            new, r["loss"], r["clipfrac"] = train(spec, theta, adam, obs, act, idx, meta["lr"], "ppo", adv, ll_old,
                                                  meta["clip"])
            r["surr"] = (ppo_eval(spec, theta, theta, obs, act, adv)[0],) + ppo_eval(spec, new, theta, obs, act, adv)
        else:
            loss = meta["loss"].lower()
            before = bc_loss(spec, theta, obs, act, loss)
            idx = minibatch_indices(n, meta["mb"], meta["epochs"])
            new, r["loss"], _ = train(spec, theta, adam, obs, act, idx, meta["lr"], loss)
            r["bcloss"] = (before, bc_loss(spec, spec.clamp(new), obs, act, loss))
        theta = spec.clamp(new)
        r["theta"], r["m"], r["v"], r["step"] = theta, adam.m.copy(), adam.v.copy(), adam.step
        out.append(r)
    return out
