"""The host side of the per-cell profiles on the CPU, through tests/profiles_shim.cpp (csrc/setup.cpp, profiles.cpp, stepplan.cpp,
restart.cpp and fluxtables.cpp built with g++, no CUDA): the per-cell constants against numpy and, for the row tables broadcast along the
span, against the row constants bit for bit; a slab's columns; every refusal; the restart fingerprint; the flux correction's per-cell
tables against numpy for both modes."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import profiles_model as PM
from oracle_harness import package
from shims import CSRC
from conftest import ROOT

D = C.POINTER(C.c_double)
FP_PROFILE_96x160 = 0x30964925d0e2b739        # the parent's fingerprint of this plane without profiles (test_time_scales_host.py)


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    lib = str(tmp_path_factory.mktemp("profiles") / "libprofiles.so")
    srcs = [os.path.join(CSRC, s) for s in ("setup.cpp", "profiles.cpp", "stepplan.cpp", "restart.cpp", "fluxtables.cpp")]
    subprocess.run(["/usr/bin/g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"), "-I", "/usr/local/cuda/include",
                    "-I", CSRC, "-shared", "-fPIC", "-Wl,--no-undefined", *srcs, os.path.join(ROOT, "tests", "profiles_shim.cpp"), "-o", lib],
                   check=True)
    L = C.CDLL(lib)
    L.pr_plane.argtypes = [C.c_void_p, C.POINTER(C.c_int), D, D, D, C.c_char_p, C.c_int]
    L.pr_consts.argtypes = [C.c_void_p, D, D, D, C.c_char_p, C.c_int]
    L.pr_fingerprint.argtypes = [C.c_void_p, D, C.POINTER(C.c_uint64), C.c_char_p, C.c_int]
    L.pr_flux.argtypes = [C.c_void_p, D, C.c_int, D, D, D, D, D, C.c_char_p, C.c_int]
    return L


@pytest.fixture(scope="module")
def dfbm():
    return package()


class Plane:
    """a plane's dfb_config (as dfb_config_init + fill_config make it) with its plan's sizes, rows and vertices"""

    def __init__(self, shim, dfbm, plane, **kw):
        self.plane = plane
        self.c = dfbm.dfb_config()
        self.c.struct_bytes = C.sizeof(self.c)
        self.c.grid_file_len = self.c.vel_fluc_file_len = self.c.line_file_len = -1
        self.c.device = -1
        self.keep = dfbm.fill_config(self.c, dfbm.DFConfig.from_plane(plane, **kw))
        dims, err = (C.c_int * 4)(), C.create_string_buffer(512)
        assert shim.pr_plane(self.ref(), dims, None, None, None, err, 512) == 0, err.value
        self.Ny, self.NzG, self.k0, self.k1 = dims
        self.rows, self.vy, self.vz = np.zeros((8, self.Ny)), np.zeros(self.Ny + 1), np.zeros(self.NzG + 1)
        assert shim.pr_plane(self.ref(), dims, _d(self.rows), _d(self.vy), _d(self.vz), err, 512) == 0

    def ref(self):
        return C.byref(self.c)


def _d(a):
    return a.ctypes.data_as(D) if a is not None else None


def consts(shim, p, cells):
    """(rc, per-cell constants [7][Ny][W], row constants [Ny][8], message)"""
    cells = np.ascontiguousarray(cells, dtype=np.float64)
    out, rowc, err = np.zeros((7, p.Ny, p.k1 - p.k0)), np.zeros((p.Ny, 8)), C.create_string_buffer(1024)
    rc = shim.pr_consts(p.ref(), _d(cells), _d(out), _d(rowc), err, 1024)
    return rc, out, rowc, err.value.decode()


@pytest.fixture(scope="module")
def planes(shim, dfbm, W):
    p = W.plane_profile(96, 160, 24, 10)
    return dict(profile=Plane(shim, dfbm, p), slab=Plane(shim, dfbm, p, k_begin=48, k_end=112),
                ragged=Plane(shim, dfbm, W.plane_ragged(40, 56, 8, seed=3)))


@pytest.mark.parametrize("which", ["profile", "slab", "ragged"])
def test_broadcast_rows_give_the_row_constants(shim, planes, which):
    p = planes[which]
    rc, out, rowc, err = consts(shim, p, PM.broadcast(p.rows, p.NzG))
    assert rc == 0, err
    for c in range(7):
        assert np.array_equal(out[c], np.repeat(rowc[:, c:c + 1], p.k1 - p.k0, axis=1)), c


@pytest.mark.parametrize("which", ["profile", "slab", "ragged"])
def test_band_constants_match_numpy(shim, planes, which):
    p = planes[which]
    cells = PM.band_cells(PM.band_rows(p.plane), p.NzG)
    rc, out, _, err = consts(shim, p, cells)
    assert rc == 0, err
    ref = PM.consts(cells)[:, :, p.k0:p.k1]
    assert np.array_equal(out, ref)
    # the bands really differ, and each band's columns are its own row table's
    e = PM.band_edges(p.NzG)
    assert not np.array_equal(cells[0, :, e[0]], cells[0, :, e[2]])


def test_slab_takes_its_own_columns(shim, planes):
    whole, slab = planes["profile"], planes["slab"]
    cells = PM.band_cells(PM.band_rows(whole.plane), whole.NzG)
    _, a, _, _ = consts(shim, whole, cells)
    _, b, _, _ = consts(shim, slab, cells)
    assert np.array_equal(a[:, :, slab.k0:slab.k1], b)


QUANTITY = ["R11", "R21", "R22", "R33", "Us", "Ts", "rhos", "Ms"]


@pytest.mark.parametrize("q", range(8))
@pytest.mark.parametrize("bad", [np.nan, np.inf, -np.inf])
def test_non_finite_input_is_refused(shim, dfbm, planes, q, bad):
    p = planes["profile"]
    cells = PM.broadcast(p.rows, p.NzG)
    cells[q, 17, 33] = bad
    rc, _, _, err = consts(shim, p, cells)
    assert rc == dfbm.ERR_ARG and err.startswith("%d dfb_set_profiles: %s at row 17, column 33 is not finite" % (dfbm.ERR_ARG, QUANTITY[q])), err


@pytest.mark.parametrize("q, value, const", [
    (0, -1.0, "sqrt(R11)"),                        # R11 < 0
    (2, 0.0, "sqrt(R22 - b^2)"),                   # R22 < b^2 (R21 != 0)
    (3, -1e-3, "sqrt(R33)"),                       # R33 < 0
    (4, 0.0, "-0.2 Ms^2 / Us"),                    # Us = 0
])
def test_non_finite_constant_is_refused(shim, dfbm, planes, q, value, const):
    p = planes["profile"]
    cells = PM.broadcast(p.rows, p.NzG)
    cells[q, 40, 150] = value
    rc, _, _, err = consts(shim, p, cells)
    assert rc == dfbm.ERR_ARG, err
    assert ("dfb_set_profiles: %s at row 40, column 150 gives %s = " % (QUANTITY[q], const)) in err, err


def test_the_first_refusal_is_reported(shim, dfbm, planes):
    p = planes["profile"]
    cells = PM.broadcast(p.rows, p.NzG)
    cells[4, 60, 2] = 0.0
    cells[0, 5, 7] = -1.0                          # earlier in row-major (row, column) order
    _, _, _, err = consts(shim, p, cells)
    assert "R11 at row 5, column 7" in err, err


# ---- the restart fingerprint ----
def fingerprint(shim, p, cells):
    fp, err = C.c_uint64(), C.create_string_buffer(512)
    c = None if cells is None else np.ascontiguousarray(cells, dtype=np.float64)
    assert shim.pr_fingerprint(p.ref(), _d(c), C.byref(fp), err, 512) == 0, err.value
    return fp.value


def test_fingerprint(shim, planes):
    p = planes["profile"]
    assert fingerprint(shim, p, None) == FP_PROFILE_96x160              # without profiles: the parent's fingerprint
    cells = PM.band_cells(PM.band_rows(p.plane), p.NzG)
    fa = fingerprint(shim, p, cells)
    assert fa != FP_PROFILE_96x160 and fa == fingerprint(shim, p, cells)
    other = cells.copy()
    other[5, 3, 4] = np.nextafter(other[5, 3, 4], np.inf)                # one ulp of one Ts
    assert fingerprint(shim, p, other) not in (fa, FP_PROFILE_96x160)
    fb = fingerprint(shim, p, PM.broadcast(p.rows, p.NzG))               # profiles equal to the rows are still profiles
    assert fb not in (fa, FP_PROFILE_96x160)
    # a slab hashes the whole-plane table, so every slab layout of a plane shares its fingerprint's profile part
    assert fingerprint(shim, planes["slab"], cells) == fa


# ---- the flux correction's per-cell tables ----
def flux(shim, p, cells, mode):
    n = None if cells is None else np.ascontiguousarray(cells, dtype=np.float64)
    t = dict(wy=np.zeros(p.Ny), hz=np.zeros(p.NzG), wz=np.zeros((p.Ny, p.NzG)) if cells is not None else None)
    d, mean, err = C.c_double(), C.c_double(), C.create_string_buffer(512)
    rc = shim.pr_flux(p.ref(), _d(n), mode, _d(t["wy"]), _d(t["hz"]), _d(t["wz"]), C.byref(d), C.byref(mean), err, 512)
    t["D"], t["mean"] = d.value, mean.value
    return rc, t, err.value.decode()


@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("which", ["profile", "ragged"])
def test_flux_tables_match_numpy(shim, planes, which, mode):
    p = planes[which]
    cells = PM.band_cells(PM.band_rows(p.plane), p.NzG)
    rc, t, err = flux(shim, p, cells, mode)
    assert rc == 0, err
    R11, Us, rhos, Ms = cells[0], cells[4], cells[6], cells[7]
    hy, hz = np.diff(p.vy), np.diff(p.vz)
    g = rhos * (1.0 + 0.2 * Ms * Ms) if mode == 1 else np.ones_like(R11)
    assert np.array_equal(t["wy"], hy) and np.array_equal(t["hz"], hz)
    assert np.array_equal(t["wz"], g * hz[None, :])
    A = np.outer(hy, hz).astype(np.longdouble)
    Dref = float((A * (g * np.sqrt(R11)).astype(np.longdouble)).sum())
    mref = float((A * (rhos * Us if mode == 1 else Us).astype(np.longdouble)).sum())
    assert t["D"] == pytest.approx(Dref, rel=1e-13) and t["mean"] == pytest.approx(mref, rel=1e-13)
    # the row tables broadcast give the row path's D and mean flux to rounding
    _, r, _ = flux(shim, p, None, mode)
    _, b, _ = flux(shim, p, PM.broadcast(p.rows, p.NzG), mode)
    assert b["D"] == pytest.approx(r["D"], rel=1e-13) and b["mean"] == pytest.approx(r["mean"], rel=1e-13)


def test_flux_refuses_profiles_without_R11(shim, dfbm, planes):
    p = planes["profile"]
    cells = PM.broadcast(p.rows, p.NzG)
    cells[0] = 0.0
    cells[1] = 0.0
    rc, _, err = flux(shim, p, cells, 2)
    assert rc == dfbm.ERR_ARG and "R11 is zero on every cell" in err, err
