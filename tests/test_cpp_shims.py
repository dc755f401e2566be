"""The header-only C++ shims (include/epivo_shims.hpp) compile against stand-in matrix/point types
and, on a GPU box, drive the C ABI like the reference drivers would."""
import os
import subprocess

import pytest

from epivo_b200 import build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bindir(tmp_path_factory):
    """the test executables are built outside the repository tree, which may be read-only"""
    return str(tmp_path_factory.mktemp("cpp"))


def _compile(bindir):
    lib = build.build()
    src = os.path.join(ROOT, "tests", "cpp", "shim_test.cpp")
    exe = os.path.join(bindir, "shim_test.bin")
    cmd = ["g++", "-O1", "-std=c++11", "-I", os.path.join(ROOT, "include"), src, "-o", exe,
           lib, "-Wl,-rpath," + os.path.dirname(lib), "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64", "-lcudart"]
    p = subprocess.run(cmd, capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    return exe


def _compile_dropin(bindir):
    """tests/cpp/dropin_test.cpp: the reference's literal call lines against include/epivo_dropin.hpp, with stand-in
    cv:: types and the oracle's Eigen stand-in (neither OpenCV nor Eigen exists in this image)."""
    lib = build.build()
    shim = os.path.join(ROOT, "oracle", "ref_shim")
    exe = os.path.join(bindir, "dropin_test.bin")
    cmd = ["g++", "-O1", "-std=c++11", "-I", os.path.join(ROOT, "include"), "-I", shim,
           os.path.join(ROOT, "tests", "cpp", "dropin_test.cpp"), os.path.join(shim, "standin_impl.cpp"), "-o", exe,
           lib, "-Wl,-rpath," + os.path.dirname(lib), "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64", "-lcudart"]
    p = subprocess.run(cmd, capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    return exe


def test_shims_compile_and_link(bindir):
    _compile(bindir)


def test_dropin_literal_call_lines_compile(bindir):
    """kitti_E.cpp:98-104,120,196 and kitti_ba.cpp:602,641,702,715,881 compile with only the include added."""
    _compile_dropin(bindir)


@pytest.mark.gpu
def test_dropin_literal_call_lines_run(bindir):
    exe = _compile_dropin(bindir)
    p = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert p.returncode == 0, p.stdout + p.stderr
    assert "dropin ok" in p.stdout


@pytest.mark.gpu
def test_shims_run_like_a_reference_driver(bindir):
    exe = _compile(bindir)
    p = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert p.returncode == 0, p.stdout + p.stderr
    assert "shims ok" in p.stdout
