"""The primal entry points as a C/C++ caller sees them: a translation unit that includes only
include/clp_b200.h, compiled with g++ and linked against the shared library."""
import os
import subprocess

import pytest

from conftest import ROOT

SRC = os.path.join(ROOT, "tests", "cabi", "primal_consumer.cpp")
LIBDIR = os.path.join(ROOT, "clp_b200", "_lib")


def _build(tmp_path):
    exe = str(tmp_path / "primal_consumer")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), SRC,
                           "-L", LIBDIR, "-lclp_b200", f"-Wl,-rpath,{LIBDIR}", "-o", exe])
    return exe


def test_primal_consumer_host_only(tmp_path):
    # devices hidden: the primal entries answer CLPB_NO_DEVICE, chgObjCoefficients / getProblem are host only
    out = subprocess.run([_build(tmp_path)], capture_output=True, text=True, timeout=120,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert out.returncode == 0, out.stdout + out.stderr
    assert "primal consumer ok (host only)" in out.stdout


def test_chg_obj_coefficients_python_host_only():
    import numpy as np

    import clp_b200
    from conftest import load_golden

    lp = load_golden("afiro")
    s = clp_b200.ClpSimplex()
    s.loadLP(lp)
    c = lp.objective * 1.03 + 0.5
    s.chgObjCoefficients(c)
    np.testing.assert_array_equal(s.getProblem().objective, c)
    with pytest.raises(ValueError):
        s.chgObjCoefficients(c[:-1])


@pytest.mark.gpu
def test_primal_consumer_solves_and_resolves_hot(tmp_path):
    out = subprocess.run([_build(tmp_path), "gpu"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "primal consumer ok (gpu)" in out.stdout
