"""The tensor-core baseline fit reproduces, bit for bit, a fixture written by tools/make_fit_tc_bits.py: the weights,
both Adam moments, the step counter and the fit errors after two consecutive fits, for the single-SM shape and the
K-split shapes with one and six helper CTAs, at step counts on both sides of the kernel's prefetch distance and
minibatch-buffer parity.  A change of the kernel's schedule must leave every one of these bits where it was."""
import numpy as np
import pytest

from conftest import golden_equal, load_golden
from tools.make_fit_tc_bits import OBS_DIMS, STEPS, case_key, run_case

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("steps", STEPS)
@pytest.mark.parametrize("obs_dim", OBS_DIMS)
def test_fit_tc_bits(cuda_device, obs_dim, steps):
    g = load_golden("fit_tc_bits")
    k = case_key(obs_dim, steps)
    r = run_case(obs_dim, steps)
    assert int(r["step"]) == int(g[k + "step"])
    assert np.array_equal(r["errors"], g[k + "errors"]), (r["errors"], g[k + "errors"])
    for name in ("w", "m", "v"):
        assert golden_equal(r[name], g, k + name), "%s differs from the fixture (K = %d, %d steps)" % (name, obs_dim + 4, steps)
