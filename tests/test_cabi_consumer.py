"""A C++ translation unit that includes only include/clp_b200.h, compiled with g++ and linked against
the shared library: the boundary as a C/C++ caller sees it (not ctypes)."""
import os
import subprocess

import pytest

from conftest import ROOT

SRC = os.path.join(ROOT, "tests", "cabi", "consumer.cpp")
LIBDIR = os.path.join(ROOT, "clp_b200", "_lib")


def _build(tmp_path):
    exe = str(tmp_path / "consumer")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), SRC,
                           "-L", LIBDIR, "-lclp_b200", f"-Wl,-rpath,{LIBDIR}", "-o", exe])
    return exe


def test_cpp_consumer_host_only(tmp_path):
    # the devices are hidden, so that the no-device answer is checked on machines with a GPU too
    out = subprocess.run([_build(tmp_path)], capture_output=True, text=True, timeout=120,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert out.returncode == 0, out.stdout + out.stderr
    assert "consumer ok (host only)" in out.stdout


@pytest.mark.gpu
def test_cpp_consumer_solves_and_steps(tmp_path):
    out = subprocess.run([_build(tmp_path), "gpu"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "consumer ok (gpu)" in out.stdout
