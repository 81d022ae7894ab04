"""Bit-exact fixture of the tensor-core baseline fit (vf_fit_tc_kernel): w, m, v, the Adam step counter and the fit errors
after two consecutive fits from a seeded state, for the single-SM shape (K = 21) and the K-split cluster shapes with one
(K = 43) and six (K = 380) helper CTAs, at step counts that straddle the kernel's prefetch distance and buffer parity.

    python tools/make_fit_tc_bits.py [OUT.npz]        (default tests/golden/fit_tc_bits.npz; needs the GPU)

The fit is chaotic (a last-bit difference grows to ~1e-1 in the weights over a full fit), so any change of rounding
anywhere in the kernel shows up here; a schedule change that keeps every operation's inputs and order does not.
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

OBS_DIMS = (17, 39, 376)                  # K = obs_dim + 4 = 21 (head only), 43 (one helper), 380 (six helpers)
STEPS = (2, 3, 4, 37, 301)                # Adam steps per fit = N / 64 - 1
SAMPLE = 64                               # entries kept verbatim next to each digest


def case_key(obs_dim, steps):
    return "k%d_s%d_" % (obs_dim + 4, steps)


def run_case(obs_dim, steps):
    """Two fits of `steps` Adam steps each from a seeded state; returns the arrays the fixture pins."""
    from mjrl_b200.engine import Engine
    n = 64 * (steps + 1)
    rng = np.random.RandomState(1000 * obs_dim + steps)
    eng = Engine(obs_dim, 6, (128, 128), max_samples=n + 8, max_paths=n // 64 + 1)
    try:
        eng.upload_flat(rng.randn(n, obs_dim), rng.randn(n, 6), rng.randn(n), np.full(n // 64, 64, np.int32),
                        np.zeros(n // 64, np.uint8))
        eng.compute_returns(0.995)
        d = eng.vf_d
        w = (0.1 * rng.randn(d)).astype(np.float32)
        m = (1e-3 * rng.randn(d)).astype(np.float32)
        v = (1e-6 * rng.rand(d)).astype(np.float32)
        eng.vf_set_state(w, m, v, 7)
        eng.vf_set_tensor_cores(True)
        errs = []
        for _ in range(2):                # the second fit starts from the first one's Adam state and step counter
            errs.extend(eng.vf_fit(rng.permutation(n).astype(np.int32), 64, 1e-3, 1e-3, return_errors=True))
        w, m, v, step = eng.vf_get_state()
    finally:
        eng.close()
    return {"w": w, "m": m, "v": v, "step": np.int64(step), "errors": np.array(errs, np.float64)}


def digest(a):
    """shape, seeded sample and sha256 of an array (the form tests/conftest.py:golden_equal reads)"""
    a = np.ascontiguousarray(a)
    idx = np.sort(np.random.RandomState(0).choice(a.size, SAMPLE, replace=False))
    return {"@shape": np.array(a.shape, np.int64), "@sample": a.ravel()[idx],
            "@sha256": np.array(hashlib.sha256(a.tobytes()).hexdigest())}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden", "fit_tc_bits.npz")
    out = {}
    for obs_dim in OBS_DIMS:
        for steps in STEPS:
            r = run_case(obs_dim, steps)
            k = case_key(obs_dim, steps)
            for name in ("w", "m", "v"):
                out.update({k + name + s: x for s, x in digest(r[name]).items()})
            out[k + "step"] = r["step"]
            out[k + "errors"] = r["errors"]
            print("%s step %d errors %s w sha %s" % (k, r["step"], r["errors"], out[k + "w@sha256"]))
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    np.savez_compressed(out_path, **out)
    print("wrote", out_path)


if __name__ == "__main__":
    main()
