"""The restart calls of the two language facades: the C++ class (include/digital_filter.hpp: save_restart / load_restart) and the
Fortran module's by-reference entry points (dfb_save_restart_f / dfb_load_restart_f, made as a Fortran compiler makes them by
tests/fortran_restart_mimic.c).  CPU: both compile and link.  GPU: save -> destroy -> load into a fresh handle -> continue, bitwise
against the uninterrupted run, on the reference's default plane read from files in the reference's formats."""
import os
import subprocess

import pytest

from conftest import ROOT

LIBDIR = os.path.join(ROOT, "digital-filtering_b200", "lib")


@pytest.fixture(scope="module")
def restart_bin(dfb, tmp_path_factory):
    out = str(tmp_path_factory.mktemp("restart_facades"))          # a temporary directory: the tree may be read-only
    common = ["-I" + os.path.join(ROOT, "include"), "-L" + LIBDIR, "-ldfb200", "-Wl,-rpath," + LIBDIR]
    subprocess.run(["/usr/bin/g++", "-std=c++17", "-Wall", os.path.join(ROOT, "tests", "restart_cpp_test.cpp")] + common +
                   ["-o", os.path.join(out, "restart_cpp_test")], check=True, capture_output=True)
    subprocess.run(["/usr/bin/gcc", "-std=c11", "-Wall", os.path.join(ROOT, "tests", "fortran_restart_mimic.c")] + common +
                   ["-o", os.path.join(out, "fortran_restart_mimic")], check=True, capture_output=True)
    return out


def test_restart_facades_compile_and_link(restart_bin):
    assert all(os.path.exists(os.path.join(restart_bin, b)) for b in ("restart_cpp_test", "fortran_restart_mimic"))


def test_fortran_module_binds_the_restart_entry_points():
    f = open(os.path.join(ROOT, "fortran", "digital_filtering.f90")).read()
    for name in ("dfb_save_restart_f", "dfb_load_restart_f"):
        assert f"bind(C, name='{name}')" in f
    assert "public :: save_restart, load_restart" in f


@pytest.mark.gpu
def test_cpp_facade_resumes_bitwise(restart_bin, default_data, tmp_path):
    r = subprocess.run([os.path.join(restart_bin, "restart_cpp_test"), str(tmp_path / "cpp.dfbr")], cwd=default_data / "run",
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "RESTART_OK 3" in r.stdout, (r.stdout, r.stderr)


@pytest.mark.gpu
def test_fortran_calling_convention_resumes_bitwise(restart_bin, default_data, tmp_path):
    r = subprocess.run([os.path.join(restart_bin, "fortran_restart_mimic"), str(default_data / "files" / "RST.dat"), str(default_data / "line.dat"),
                        str(tmp_path / "fortran.dfbr")], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "RESTART_OK 3" in r.stdout, (r.stdout, r.stderr)
