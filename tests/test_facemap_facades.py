"""The face maps of the two language facades: the C++ class (include/digital_filter.hpp: face_map_interp / FaceMap) and the Fortran
module's by-reference entry points (dfb_facemap_create_f, dfb_interp_to_host_f, dfb_interp_to_cells_f, made as a Fortran compiler makes
them by tests/fortran_facemap_mimic.c).  CPU: both compile and link, and the module binds the entry points.  GPU: on the reference's
default plane, faces equal to the cells return the fields bit for bit and the device path equals the host path."""
import os
import subprocess

import pytest

from conftest import ROOT

LIBDIR = os.path.join(ROOT, "digital-filtering_b200", "lib")
CUDA = "/usr/local/cuda"


@pytest.fixture(scope="module")
def facemap_bin(dfb, tmp_path_factory):
    out = str(tmp_path_factory.mktemp("facemap_facades"))          # a temporary directory: the tree may be read-only
    common = ["-I" + os.path.join(ROOT, "include"), "-I" + CUDA + "/include", "-L" + LIBDIR, "-ldfb200", "-Wl,-rpath," + LIBDIR,
              "-L" + CUDA + "/lib64", "-lcudart", "-Wl,-rpath," + CUDA + "/lib64"]
    for cc, std, src, exe in (("/usr/bin/g++", "-std=c++17", "facemap_cpp_test.cpp", "facemap_cpp_test"),
                              ("/usr/bin/gcc", "-std=c11", "fortran_facemap_mimic.c", "fortran_facemap_mimic")):
        r = subprocess.run([cc, std, "-Wall", os.path.join(ROOT, "tests", src)] + common + ["-o", os.path.join(out, exe)],
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    return out


def test_facemap_facades_compile_and_link(facemap_bin):
    assert all(os.path.exists(os.path.join(facemap_bin, b)) for b in ("facemap_cpp_test", "fortran_facemap_mimic"))


def test_fortran_module_binds_the_facemap_entry_points():
    f = open(os.path.join(ROOT, "fortran", "digital_filtering.f90")).read()
    for name in ("dfb_facemap_create_f", "dfb_facemap_served_f", "dfb_facemap_destroy_f", "dfb_interp_to_host_f", "dfb_interp_to_cells_f"):
        assert f"bind(C, name='{name}')" in f
    assert "public :: facemap_create, interp_to_host, interp_to_cells, facemap_destroy" in f


@pytest.mark.gpu
def test_cpp_facade_face_maps(facemap_bin, default_data):
    r = subprocess.run([os.path.join(facemap_bin, "facemap_cpp_test")], cwd=default_data / "run", capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "FACEMAP_OK" in r.stdout, (r.returncode, r.stdout, r.stderr)


@pytest.mark.gpu
def test_fortran_calling_convention_face_maps(facemap_bin, default_data):
    r = subprocess.run([os.path.join(facemap_bin, "fortran_facemap_mimic"), str(default_data / "files" / "RST.dat"),
                        str(default_data / "line.dat")], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "FACEMAP_OK" in r.stdout, (r.returncode, r.stdout, r.stderr)
