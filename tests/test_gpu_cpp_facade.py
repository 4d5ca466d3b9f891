"""Builds tests/cpp/test_facade.cpp (the C++ mirror of the reference API, include/acb200.hpp) with
g++ against libacb200.so and runs it on the GPU.  The programs are built in a per-test temporary
directory: the repository tree may be read-only, or shared with other users."""
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
SRC = ROOT / "tests" / "cpp" / "test_facade.cpp"


def _build(out_dir):
    exe = out_dir / "test_facade"
    libdir = ROOT / "aho-corasick_b200"
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-I", str(ROOT / "include"), str(SRC), "-o", str(exe),
           "-L", str(libdir), "-lacb200", f"-Wl,-rpath,{libdir}"]
    subprocess.check_call(cmd)
    return exe


def test_cpp_packed_host_checks(tmp_path):
    """-m "not gpu": acb200::packed on host-only searchers (construction contract, error behaviour)."""
    src = ROOT / "tests" / "cpp" / "test_packed_host.cpp"
    exe = tmp_path / "test_packed_host"
    libdir = ROOT / "aho-corasick_b200"
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", str(ROOT / "include"), str(src), "-o",
                           str(exe), "-L", str(libdir), "-lacb200", f"-Wl,-rpath,{libdir}"])
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "all checks passed" in r.stdout, r.stdout + r.stderr


def test_cpp_facade_compiles(tmp_path):
    """-m "not gpu": the header and the test program must at least build and link."""
    assert _build(tmp_path).exists()


@pytest.mark.gpu
def test_cpp_facade_runs(tmp_path):
    exe = _build(tmp_path)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "all checks passed" in r.stdout
