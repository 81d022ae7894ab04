"""CPU tests of the boundary: the shared library loads here (no GPU) and exports exactly the symbols
include/mjrl_b200.h declares; creating an engine without a device fails loudly (no CPU fallback)."""
import os
import re

from conftest import ROOT


def header_symbols():
    src = open(os.path.join(ROOT, "include", "mjrl_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(mjb_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    import __graft_entry__
    __graft_entry__.build()
    from mjrl_b200 import _native
    lib = _native.load()
    declared = header_symbols()
    assert declared == _native.exported_symbols()
    for name in declared:
        assert getattr(lib, name) is not None
    assert lib.mjb_version() == 1
    # the dynamic symbol table of the .so itself: exactly the declared entry points carry the mjb_ prefix
    import subprocess
    out = subprocess.run(["nm", "-D", "--defined-only", _native.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = sorted({ln.split()[-1] for ln in out.splitlines() if ln.split() and ln.split()[-1].startswith("mjb_")})
    assert exported == declared, (set(exported) ^ set(declared))


def test_header_cites_reference():
    src = open(os.path.join(ROOT, "include", "mjrl_b200.h")).read()
    for cite in ("utils/process_samples.py", "algos/npg_cg.py", "utils/cg_solve.py", "baselines/mlp_baseline.py",
                 "algos/trpo.py", "algos/dapg.py", "policies/gaussian_mlp.py"):
        assert cite in src


def test_no_cpu_fallback():
    """Without a CUDA device, creating an engine raises MjbError.  Checked in a child process with every device
    hidden, so that it holds on machines with a GPU too."""
    import subprocess
    import sys
    code = ("from mjrl_b200.engine import Engine, MjbError\n"
            "try:\n"
            "    Engine(4, 2, (32, 32))\n"
            "except MjbError:\n"
            "    raise SystemExit(0)\n"
            "raise SystemExit('an engine was created without a CUDA device')\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


def test_product_never_imports_oracle():
    """The oracle is test infrastructure: nothing under mjrl_b200/ may import it."""
    for dirpath, _, files in os.walk(os.path.join(ROOT, "mjrl_b200")):
        for f in files:
            if f.endswith(".py"):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text.replace("# oracle", ""), os.path.join(dirpath, f)


def test_host_classes_construct_on_cpu():
    import numpy as np
    from mjrl_b200.algos.dapg import DAPG
    from mjrl_b200.algos.npg_cg import NPG
    from mjrl_b200.algos.trpo import TRPO
    from mjrl_b200.baselines.mlp_baseline import MLPBaseline
    from mjrl_b200.policies.gaussian_linear import LinearPolicy
    from mjrl_b200.policies.gaussian_mlp import MLP
    from mjrl_b200.utils.cg_solve import cg_solve
    from mjrl_b200.utils.gym_env import EnvSpec
    es = EnvSpec(6, 2, 50)
    pol = MLP(es, hidden_sizes=(32, 32), seed=500)
    assert pol.d == 1348 and LinearPolicy(EnvSpec(376, 17, 10), seed=0).d == 6426
    th = pol.get_param_values()
    th[-2:] = -7.0
    pol.set_param_values(th)
    assert np.all(pol.get_param_values()[-2:] == -3.0)          # min_log_std clamp (gaussian_mlp.py:73-75)
    bl = MLPBaseline(es)
    feat = bl._features([dict(observations=np.array([[0.0, 20, -30, 0, 0, 0], [1, 2, 3, 0, 0, 0]]), rewards=np.zeros(2))])
    assert np.allclose(feat[1, -4:], [1e-3, 1e-6, 1e-9, 1e-12]) and feat[0, 1] == 1.0 and feat[0, 2] == -1.0
    for cls, kw in ((NPG, {}), (TRPO, {}), (DAPG, dict(demo_paths=None))):
        a = cls(None, pol, bl, **kw)
        assert a.FIM_invert_args == {'iters': 10, 'damping': 1e-4}
    A = np.array([[4.0, 1.0], [1.0, 3.0]])
    assert np.allclose(cg_solve(lambda v: A.dot(v), np.array([1.0, 2.0]), cg_iters=2), [1 / 11, 7 / 11])


def test_host_permutation_is_numpys():
    """mjb_host_permutation reproduces np.random.permutation(n) of the global RandomState bit for bit -- the order
    AND the generator state afterwards (MLPBaseline.fit's minibatch order, optimize_model.py:22)."""
    import numpy as np
    from mjrl_b200 import runtime
    for seed, n in [(0, 2), (1, 3), (2, 64), (3, 1000), (4, 4096), (5, 4097), (123, 65536), (7, 250000), (8, 1000003)]:
        np.random.seed(seed)
        np.random.rand(seed % 5)                          # start from an arbitrary position inside the MT block
        want = np.random.permutation(n)
        after_want = np.random.randint(0, 1 << 30, size=5)
        np.random.seed(seed)
        np.random.rand(seed % 5)
        got = runtime.global_permutation(n)
        after_got = np.random.randint(0, 1 << 30, size=5)
        assert got.dtype == np.int32 and np.array_equal(got, want), (seed, n)
        assert np.array_equal(after_got, after_want), (seed, n)
    # a gaussian cached in the state (has_gauss) survives the round trip
    np.random.seed(11)
    np.random.randn(3)
    a = np.random.permutation(1000); x = np.random.randn()
    np.random.seed(11)
    np.random.randn(3)
    b = runtime.global_permutation(1000); y = np.random.randn()
    assert np.array_equal(a, b) and x == y
