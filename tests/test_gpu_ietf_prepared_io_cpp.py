"""PreparedInputs and the PreparedPublics overloads that take it, of the C++ header (include/vrfs_b200.hpp) compiled against the
C ABI, built in a temporary directory."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "ark_ec_vrfs_b200")
SRC = os.path.join(ROOT, "tests", "cpp", "test_ietf_prepared_io_mirror.cpp")


def build(tmp_path):
    from ark_ec_vrfs_b200 import build as b
    b.build()
    exe = str(tmp_path / "test_ietf_prepared_io_mirror")
    subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-o", exe, SRC, "-L" + PKG, "-lvrfs_b200", "-Wl,-rpath," + PKG], check=True)
    return exe


@pytest.mark.gpu
def test_ietf_prepared_io_mirror_builds(tmp_path):
    assert os.path.exists(build(tmp_path))


@pytest.mark.gpu
def test_ietf_prepared_io_mirror_runs(tmp_path):
    r = subprocess.run([build(tmp_path)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "all ok" in r.stdout, r.stdout + r.stderr
