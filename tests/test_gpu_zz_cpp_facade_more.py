"""Second C++ facade program (tests/cpp/test_facade_more.cpp: OverlappingState, replace_all*,
acb200::packed) on the GPU; and, without a GPU, both facade programs linked against the dry-run
library of tests/emu/ (the kernel sources executed on the CPU).  The programs are built in a per-test
temporary directory, not in the repository tree."""
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
CPP = ROOT / "tests" / "cpp"


def _build(src, exe, libdir, libname):
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-I", str(ROOT / "include"), str(src), "-o", str(exe),
                           "-L", str(libdir), f"-l{libname}", f"-Wl,-rpath,{libdir}"])


@pytest.mark.gpu
def test_cpp_facade_more_runs(tmp_path):
    exe = tmp_path / "test_facade_more"
    _build(CPP / "test_facade_more.cpp", exe, ROOT / "aho-corasick_b200", "acb200")
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "all checks passed" in r.stdout, r.stdout + r.stderr


@pytest.mark.parametrize("prog", ["test_facade", "test_facade_more"])
def test_cpp_facade_programs_on_the_dry_run_library(prog, tmp_path):
    sys.path.insert(0, str(ROOT / "tests" / "emu"))
    import build_emu
    lib = build_emu.build()
    exe = tmp_path / f"{prog}_emu"
    _build(CPP / f"{prog}.cpp", exe, lib.parent, "acb200_emu")
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "all checks passed" in r.stdout, r.stdout + r.stderr
