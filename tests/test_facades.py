"""The two language facades over the C ABI.
  C++      include/digital_filter.hpp, used exactly like the reference's test/cpp-main.cpp
  Fortran  fortran/digital_filtering.f90 -- no Fortran compiler in the image, so its binding is
           exercised by tests/fortran_abi_mimic.c (same struct image, same by-reference calls)
CPU: both compile and link against libdfb200.so.  GPU: both run on the reference's default plane, read from files in the
reference's formats that the `default_data` fixture writes from the stored tables."""
import os
import subprocess

import pytest

from conftest import ROOT

BIN = os.path.join(ROOT, "tests", "_bin")
LIBDIR = os.path.join(ROOT, "digital-filtering_b200", "lib")


def _build(dfb):
    os.makedirs(BIN, exist_ok=True)
    common = ["-I" + os.path.join(ROOT, "include"), "-L" + LIBDIR, "-ldfb200", "-Wl,-rpath," + LIBDIR]
    subprocess.run(["/usr/bin/g++", "-std=c++17", "-Wall", os.path.join(ROOT, "examples", "cpp-main.cpp")] + common +
                   ["-o", os.path.join(BIN, "cpp-test")], check=True, capture_output=True)
    subprocess.run(["/usr/bin/gcc", "-std=c11", "-Wall", os.path.join(ROOT, "tests", "fortran_abi_mimic.c")] + common +
                   ["-lm", "-o", os.path.join(BIN, "fortran_abi_mimic")], check=True, capture_output=True)


def test_facades_compile_and_link(dfb):
    _build(dfb)
    assert os.path.exists(os.path.join(BIN, "cpp-test")) and os.path.exists(os.path.join(BIN, "fortran_abi_mimic"))


REF_MAIN = "/root/reference/digital-filtering-c++/test/cpp-main.cpp"


def _build_reference_main():
    """The reference's OWN driver (test/cpp-main.cpp: DFConfig config; DIGITAL_FILTER df(config); df.get_rms();), byte for byte,
    compiled against the B200 facade: staged (never committed) as <stage>/test/cpp-main.cpp beside <stage>/df -> include/df, whose
    df.hpp stands where the reference's stands.  Only possible where /root/reference exists (the build container); the binary lands
    in tests/_bin (git-ignored) and travels to the GPU box."""
    import shutil
    stage = os.path.join(BIN, "refmain")
    os.makedirs(os.path.join(stage, "test"), exist_ok=True)
    shutil.copyfile(REF_MAIN, os.path.join(stage, "test", "cpp-main.cpp"))
    link = os.path.join(stage, "df")
    if os.path.islink(link) or os.path.exists(link):
        os.unlink(link)
    os.symlink(os.path.join(ROOT, "include", "df"), link)
    subprocess.run(["/usr/bin/g++", "-std=c++17", os.path.join(stage, "test", "cpp-main.cpp"), "-L" + LIBDIR, "-ldfb200",
                    "-Wl,-rpath," + LIBDIR, "-o", os.path.join(BIN, "ref-cpp-main")], check=True, capture_output=True)
    assert open(os.path.join(stage, "test", "cpp-main.cpp"), "rb").read() == open(REF_MAIN, "rb").read()
    shutil.rmtree(stage)                     # only the binary stays (and travels); no reference source is kept in the tree


def test_reference_main_compiles_unchanged(dfb):
    if not os.path.exists(REF_MAIN):
        pytest.skip("/root/reference is only present in the build container")
    _build_reference_main()
    assert os.path.exists(os.path.join(BIN, "ref-cpp-main"))


def test_fortran_module_mirrors_the_c_struct():
    """field order of `type, bind(C) :: dfb_config_c` == field order of `struct dfb_config`"""
    import re
    h = open(os.path.join(ROOT, "include", "dfb200.h")).read()
    body = h[h.index("typedef struct dfb_config {") + len("typedef struct dfb_config {"):h.index("} dfb_config;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    c_fields = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl or decl.startswith("typedef"):
            continue
        names = re.sub(r"^(const\s+)?(unsigned\s+)?\w+\s*\*?", "", decl, count=1)
        c_fields += [n.strip().lstrip("*").strip() for n in names.split(",") if n.strip()]
    f = open(os.path.join(ROOT, "fortran", "digital_filtering.f90")).read()
    fb = f[f.index("type, bind(C) :: dfb_config_c"):f.index("end type dfb_config_c")]
    f_fields = []
    for ln in fb.splitlines()[1:]:
        if "::" in ln:
            f_fields += [n.strip() for n in ln.split("::")[1].split(",")]
    assert [x.lower() for x in c_fields] == [x.lower() for x in f_fields], (c_fields, f_fields)


@pytest.mark.gpu
def test_cpp_facade_runs_the_reference_example(dfb, default_data):
    _build(dfb)
    r = subprocess.run([os.path.join(BIN, "cpp-test")], cwd=default_data / "run", capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert "Ny=510 Nz=400" in r.stdout
    rms = float(r.stdout.split("=")[-1].split()[0])
    assert 20.0 < rms < 80.0          # sqrt(mean R11) of the M6 DNS profile on this plane is ~50 m/s


@pytest.mark.gpu
def test_reference_main_runs_unchanged(dfb, O):
    """test/cpp-main.cpp of the reference, unmodified, on the GPU: constructor + get_rms() (500 steps of dt = 1e-5, df.cpp:584-611)
    + plot_rms()'s file in the reference's place and format."""
    exe = os.path.join(BIN, "ref-cpp-main")
    if os.path.exists(REF_MAIN):
        _build_reference_main()
    if not os.path.exists(exe) or not O.have_ref():
        pytest.skip("the staged build of the reference's main did not travel")
    os.makedirs(O.REF_RUN, exist_ok=True)
    out = os.path.join(O.REF_FILES, "cpp_vel_fluc_rms.csv")
    if os.path.exists(out):
        os.unlink(out)
    r = subprocess.run([exe], cwd=O.REF_RUN, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    assert "Finished plotting to file: ../files/cpp_vel_fluc_rms.csv" in r.stdout
    lines = open(out).read().splitlines()
    assert lines[0] == "z, y, u'_rms, v'_rms, w'_rms, T'_rms, rho'_rms " and len(lines) == 1 + 510 * 400
    # u'_rms over the plane ~ sqrt(mean R11) of the M6 DNS profile (tens of m/s); the wall row has R = 0
    import numpy as np
    vals = np.array([[float(x) for x in ln.split(", ")] for ln in lines[1::37]])
    assert np.all(np.isfinite(vals)) and 20.0 < np.sqrt(np.mean(vals[:, 2] ** 2)) < 80.0


@pytest.mark.gpu
def test_fortran_calling_convention(dfb, default_data):
    _build(dfb)
    r = subprocess.run([os.path.join(BIN, "fortran_abi_mimic"), str(default_data / "files" / "RST.dat"), str(default_data / "line.dat")],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, (r.stdout, r.stderr)
    tok = r.stdout.split()
    assert tok[0] == "OK" and (int(tok[1]), int(tok[2])) == (510, 400) and float(tok[3]) > 1.0
    assert "BATCH_OK 3" in r.stdout           # create_digital_filter_batch / filter_batch / face_map through the by-reference entry points
