"""The C++ host mirror of the reference API (yask_b200/include/yask_kernel_api.hpp + libyask_kernel.<s>.b200.so).

* `yk_driver.<stencil>` is oracle/ref_driver.cpp -- the program that drives the UNMODIFIED reference through its
  public yk_* API to make the golden fixtures -- compiled unchanged against OUR header and library.  Feeding it the
  fixtures' inputs must reproduce the reference's outputs.
* `ref_kernel_api_test.<stencil>` / `ref_kernel_api_exception_test` are the reference's own API tests
  (src/kernel/tests/*.cpp of the reference), compiled unmodified against our header and libraries by oracle/build_ref.sh
  into oracle/_ref/ship/tests.
"""
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from tests.helpers import field_ulps, golden_cases, load_golden, regen_inputs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "tests", "_bin")
REF_TESTS = os.path.join(ROOT, "oracle", "_ref", "ship", "tests")


def _bin(name, where=BIN):
    p = os.path.join(where, name)
    if not os.path.exists(p):
        pytest.skip(f"{name} not built (run __graft_entry__.build())")
    return p


def test_cpp_api_fails_loudly_without_a_device():
    from yask_b200 import capi
    if capi.device_count() > 0:
        pytest.skip("a CUDA device is present")
    r = subprocess.run([_bin("yk_driver.iso3dfd"), "info", "32", "32", "32"], capture_output=True, text=True)
    assert r.returncode != 0 and "no CUDA device" in (r.stdout + r.stderr)
    r = subprocess.run([_bin("ref_kernel_api_exception_test.iso3dfd", REF_TESTS)], capture_output=True, text=True)
    # first expected exception (run before prepare) is raised with the reference's message
    assert "run_solution() called without calling prepare_solution() first" in r.stdout + r.stderr


def _drive(stencil, n, steps, ins, radius=None):
    exe = _bin(f"yk_driver.{stencil}")
    # the library's radius is fixed by its name; YASK_B200_RADIUS overrides it like the reference's `make radius=<r>`
    env = dict(os.environ, YASK_B200_RADIUS=str(radius)) if radius else None
    with tempfile.TemporaryDirectory() as d:
        for (name, t), a in ins.items():
            np.ascontiguousarray(a).tofile(os.path.join(d, f"{name}.t{t}.in"))
        n3 = list(n) + [1] * (3 - len(n))
        r = subprocess.run([exe, "run"] + [str(i) for i in n3] + [str(steps), d], capture_output=True, text=True, env=env)
        assert r.returncode == 0, r.stdout + r.stderr
        outs = {}
        for fn in os.listdir(d):
            if fn.endswith(".out"):
                outs[fn[:-4]] = np.fromfile(os.path.join(d, fn), dtype=next(iter(ins.values())).dtype)
        return outs


def _driver_cases():
    """Fixtures of the solutions that have a C++ API library (Makefile YK_STENCILS); iso3dfd: default build only."""
    out = []
    for p in golden_cases(""):
        meta, _ = load_golden(p)
        if meta["stencil"] in ("awp_elastic", "ssg", "test_3d") or (meta["stencil"] == "iso3dfd" and "strict" not in meta["ref_tag"]):
            out.append(p)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("path", _driver_cases())
def test_same_driver_source_reproduces_reference_outputs(path):
    meta, arrays = load_golden(path)
    ins = regen_inputs(meta)
    radius = re.search(r"-r(\d+)[-.]", meta["ref_tag"])          # iso3dfd fixtures of the reference built at another radius
    outs = _drive(meta["stencil"], meta["n"], meta["steps"], ins, radius=radius and int(radius.group(1)))
    for key, ref in arrays.items():
        got = outs[key].reshape(ref.shape)
        if meta["stencil"] == "iso3dfd":
            assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))      # default fp_mode = reference GCC build
        elif "strict" in meta["ref_tag"]:
            assert field_ulps(got, ref) <= 4.0    # driver runs the default (fused) mode; strict parity is tested through the C ABI
        else:
            assert field_ulps(got, ref) <= 4.0


@pytest.mark.gpu
@pytest.mark.parametrize("stencil", ["test_3d", "iso3dfd", "awp_elastic", "ssg"])   # the reference runs it on test_3d
def test_reference_kernel_api_test_passes_unmodified(stencil):
    r = subprocess.run([_bin(f"ref_kernel_api_test.{stencil}", REF_TESTS)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-2000:])
    assert "End of YASK C++ kernel API test." in r.stdout


@pytest.mark.gpu
def test_reference_kernel_api_exception_test_passes_unmodified():
    r = subprocess.run([_bin("ref_kernel_api_exception_test.iso3dfd", REF_TESTS)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-2000:])


# ---- command-line harness (yask_b200/csrc/yk_main.cpp -> yask_b200/bin/yask_kernel.<stencil>.b200.exe) -----------
def _exe(stencil):
    p = os.path.join(ROOT, "yask_b200", "bin", f"yask_kernel.{stencil}.b200.exe")
    if not os.path.exists(p):
        pytest.skip("harness not built (run __graft_entry__.build())")
    return p


def test_harness_help_and_loud_failure_without_device():
    r = subprocess.run([_exe("iso3dfd"), "-help"], capture_output=True, text=True)
    assert r.returncode == 0 and "-trial_steps" in r.stdout and "-g<dim>" in r.stdout
    from yask_b200 import capi
    if capi.device_count() == 0:
        r = subprocess.run([_exe("iso3dfd"), "-g", "64"], capture_output=True, text=True)
        assert r.returncode != 0 and "no CUDA device" in r.stdout + r.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("stencil,args", [("iso3dfd", ["-g", "128"]), ("awp_elastic", ["-g", "64"]), ("ssg", ["-gx", "48", "-gy", "40", "-gz", "64"])])
def test_harness_prints_the_reference_report_keys(stencil, args):
    """A reference-style command line (its CPU tuning flags included) runs and prints the report lines that
    the reference's log scrapers key on (yask_main.cpp:513-536)."""
    cmd = [_exe(stencil)] + args + ["-trial_steps", "4", "-num_trials", "3", "-no-pre_auto_tune", "-no-auto_tune", "-outer_threads", "8",
                                    "-b", "64", "-sleep", "0"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    for key in ("num-trials:", "best-throughput (num-points/sec):", "mid-throughput (num-points/sec):", "best-elapsed-time (sec):",
                "num-points-per-step:", "stencil-name:", "yask-version:", "Num MPI ranks:", "num-temporal-block-steps:", "YASK DONE"):
        assert key in r.stdout, key
    line = [l for l in r.stdout.splitlines() if "best-num-steps-done" in l][0]
    assert line.split()[-1] == "4"


@pytest.mark.gpu
def test_harness_validate_iso3dfd():
    r = subprocess.run([_exe("iso3dfd"), "-g", "96", "-validate"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "TEST PASSED" in r.stdout, r.stdout + r.stderr


def _run_ranks(exe, args, world, port):
    """Start the harness once per rank the way mpirun/torchrun would (RANK / WORLD_SIZE / LOCAL_RANK in the environment);
    the ranks meet in the library's shared-memory mailbox.  Ranks share the box's devices round-robin."""
    import torch
    ndev = max(1, torch.cuda.device_count())
    procs = []
    for r in range(world):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE=str(world), LOCAL_RANK=str(r % ndev), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port),
                   YASK_JOB_ID=f"pytest_{os.getpid()}_{port}")
        procs.append(subprocess.Popen([exe] + args, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    outs = []
    for p in procs:
        o, e = p.communicate(timeout=300)
        outs.append((p.returncode, o, e))
    return outs


@pytest.mark.gpu
def test_harness_two_ranks_validate_and_report():
    """The reference's multi-rank command line (`-nrx 2`, one process per rank) through the C++ API only: prepare_solution()
    wires the ranks (yb_comm + CUDA IPC), -validate compares the sweep kernel with the direct kernel across the rank
    boundary, the timing run reports from rank 0 with the global point count."""
    outs = _run_ranks(_exe("iso3dfd"), ["-g", "96", "-nrx", "2", "-validate"], 2, 29561)
    for rc, o, e in outs:
        assert rc == 0, o + e
    assert "TEST PASSED" in outs[0][1] and "num-ranks:              2" in outs[0][1]
    assert "TEST PASSED" not in outs[1][1]          # only rank 0 prints
    outs = _run_ranks(_exe("awp_elastic"), ["-g", "64", "-trial_steps", "3", "-num_trials", "2"], 2, 29562)   # rank grid chosen by the library
    for rc, o, e in outs:
        assert rc == 0, o + e
    assert "YASK DONE" in outs[0][1] and "num-ranks:              2" in outs[0][1]
    line = [l for l in outs[0][1].splitlines() if "global-domain-size" in l][0]
    assert "x=64" in line


@pytest.mark.gpu
def test_yask_sh_launcher_two_ranks(tmp_path):
    """The yask.sh-style launcher (yask_b200/scripts/yask.sh): reference option names, log file, closing checks; -ranks 2 starts
    one process per rank without mpirun."""
    sh = os.path.join(ROOT, "yask_b200", "scripts", "yask.sh")
    _exe("iso3dfd")
    r = subprocess.run([sh, "-stencil", "iso3dfd", "-ranks", "2", "-log_dir", str(tmp_path), "-v", "-g", "96"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "YASK passed internal validation test." in r.stdout and "YASK ran successfully." in r.stdout
    logs = [f for f in os.listdir(tmp_path) if f.endswith(".log")]
    assert len(logs) == 1 and logs[0].startswith("yask.iso3dfd.b200.") and ".r2." in logs[0]
