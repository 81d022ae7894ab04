import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def load_golden(name):
    g = dict(np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False))
    if "meta" in g:
        g["meta"] = eval(str(g["meta"]))      # repr() of a plain dict written by oracle/make_golden.py
    return g


def golden_equal(a, g, key):
    """`a` equals, bit for bit, the array a fixture stores under `key`: whole, or for a large array (stored by
    oracle/make_golden_host.py's `exact`) its shape, its entries at the seeded sample positions and the sha256 of its
    bytes."""
    import hashlib
    a = np.ascontiguousarray(a)
    if key in g:
        return np.array_equal(a, g[key])
    sample = g[key + "@sample"]
    if a.shape != tuple(g[key + "@shape"]) or a.dtype != sample.dtype:
        return False
    idx = np.sort(np.random.RandomState(0).choice(a.size, sample.size, replace=False))
    return np.array_equal(a.ravel()[idx], sample) and hashlib.sha256(a.tobytes()).hexdigest() == str(g[key + "@sha256"])


def golden_paths(g, demo=False):
    """Regenerate the synthetic trajectories a golden file was produced from and verify the checksum."""
    from oracle import npg_oracle as O
    m = g["meta"]
    if demo:
        return O.synthetic_paths(m["obs_dim"], m["act_dim"], max(2, m["n_paths"] // 4), m["horizon"],
                                 seed=m["demo_seed"])
    paths = O.synthetic_paths(m["obs_dim"], m["act_dim"], m["n_paths"], m["horizon"], seed=m["path_seed"],
                              ragged=m["ragged"])
    cs = [np.concatenate([p[k].ravel() for p in paths]).sum() for k in ("observations", "actions", "rewards")]
    assert np.array_equal(np.array(cs), g["input_checksum"]), "synthetic input generator drifted"
    assert np.array_equal(np.array([len(p["rewards"]) for p in paths], np.int32), g["path_len"])
    return paths


MLP_CASES = ["pm_5x50", "pm_40x25_ragged", "swim_40x250", "cheetah_24x500"]
ALL_CASES = MLP_CASES + ["linear_30x200"]


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-300))


def one_minus_cos(a, b):
    a, b = np.asarray(a, np.float64).ravel(), np.asarray(b, np.float64).ravel()
    return float(1.0 - a.dot(b) / (np.linalg.norm(a) * np.linalg.norm(b)))


@pytest.fixture(scope="session")
def cuda_device():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")
