"""The reference's own Python API tests, UNMODIFIED (src/kernel/tests/yask_kernel_api_test.py and
yask_kernel_api_exception_test.py of the reference, byte-compiled by oracle/build_ref.sh into oracle/_ref/ship/tests next to
the compiled C++ API tests), run against the
`yask_kernel` module of this engine (pybind11, yask_b200/csrc/yk_pybind.cpp) on the GPU: vars are filled through NumPy
buffers, read back, the solution runs 1 + 4 steps, stats are read -- every assert in those scripts must hold."""
import glob
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "oracle", "_ref", "ship", "tests")
MODS = sorted(glob.glob(os.path.join(ROOT, "yask_b200", "lib", "python", "*", "yask_kernel*.so")))


def _run(script, mod):
    path = os.path.join(BIN, script)
    if not os.path.exists(path):
        pytest.skip(f"{script} was not built (oracle/build_ref.sh)")
    env = dict(os.environ, PYTHONPATH=os.path.dirname(mod))
    return subprocess.run([sys.executable, path], env=env, capture_output=True, text=True, timeout=600)


@pytest.mark.skipif(not MODS, reason="python modules not built")
@pytest.mark.parametrize("mod", MODS, ids=[os.path.basename(os.path.dirname(m)) for m in MODS])
def test_reference_python_api_test_unmodified(mod):
    r = _run("ref_yask_kernel_api_test.pyc", mod)
    assert r.returncode == 0, (r.stdout[-3000:] + r.stderr[-3000:])
    assert "End of YASK Python kernel API test." in r.stdout


@pytest.mark.skipif(not MODS, reason="python modules not built")
def test_reference_python_exception_test_unmodified():
    mod = [m for m in MODS if os.sep + "iso3dfd" + os.sep in m] or MODS
    r = _run("ref_yask_kernel_api_exception_test.pyc", mod[0])
    assert r.returncode == 0, (r.stdout[-3000:] + r.stderr[-3000:])
    assert "End of YASK Python kernel API test with exception." in r.stdout


TT_SCRIPT = r"""
import numpy as np
import yask_kernel as yk
kfac = yk.yk_factory(); env = kfac.new_env()
def run(bt, steps):
    s = kfac.new_solution(env)
    for d in s.get_domain_dim_names():
        s.set_overall_domain_size(d, 72)
    s.set_block_size(s.get_step_dim_name(), bt)
    s.prepare_solution()
    rng = np.random.default_rng(3)
    for v in s.get_vars():
        names = v.get_dim_names()
        for t in ([0, 1] if "t" in names else [0]):
            first = [t if d == "t" else v.get_first_rank_domain_index(d) for d in names]
            last = [t if d == "t" else v.get_last_rank_domain_index(d) for d in names]
            shape = [l - f + 1 for f, l in zip(first, last)]
            a = (rng.random(shape, dtype=np.float32) * (0.25 if v.get_name() == "v" else 2.0) - (0.0 if v.get_name() == "v" else 1.0)).astype(np.float32)
            assert v.set_elements_in_slice(a.data, first, last) == a.size
    s.run_solution(0, steps - 1)
    p = s.get_var("p")
    tl = p.get_last_valid_step_index()
    names = p.get_dim_names()
    first = [tl if d == "t" else p.get_first_rank_domain_index(d) for d in names]
    last = [tl if d == "t" else p.get_last_rank_domain_index(d) for d in names]
    out = np.zeros([l - f + 1 for f, l in zip(first, last)], dtype=np.float32)
    assert p.get_elements_in_slice(out.data, first, last) == out.size
    st = s.get_stats()
    s.end_solution()
    return out, st.get_num_steps_done()
a, na = run(2, 5)
b, nb = run(1, 5)
assert na == nb == 5
assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), "temporal blocking changed the result"
assert np.isfinite(a).all() and np.abs(a).max() > 0
print("OK temporal tile through the Python API")
"""


@pytest.mark.parametrize("radius", [1, 2])
def test_temporal_blocking_through_the_python_api(radius):
    """set_block_size(step dim, 2) on the radius-suffixed iso3dfd modules: same bits as without it (5 steps = 2 fused + 1)."""
    mod = [m for m in MODS if os.sep + f"iso3dfd_r{radius}" + os.sep in m]
    if not mod:
        pytest.skip("module not built")
    env = dict(os.environ, PYTHONPATH=os.path.dirname(mod[0]))
    r = subprocess.run([sys.executable, "-c", TT_SCRIPT], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "OK temporal tile" in r.stdout, (r.stdout[-3000:] + r.stderr[-3000:])
