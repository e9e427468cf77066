"""The host tables of the inflow mass-flux correction on the CPU, through tests/flux_shim.cpp (csrc/setup.cpp and csrc/fluxtables.cpp built
with g++, no CUDA): the row weights g_j hy_j, sqrt(R11_j), the column widths hz_k, D and the mean flux against numpy for both modes, on
the reference's default plane, a profile plane and a plane whose columns have different widths; and the refusals."""
import ctypes as C

import numpy as np
import pytest

from oracle_harness import package
from shims import build_shim

D = C.POINTER(C.c_double)


def flux_shim(tmp_path_factory):
    L = build_shim(tmp_path_factory, "flux", "fluxtables.cpp")
    L.fx_dims.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_char_p, C.c_int]
    L.fx_tables.argtypes = [C.c_void_p, C.c_int] + [D] * 8 + [C.c_char_p, C.c_int]
    L.fx_fma.argtypes = [C.c_longlong, D, D, D, D]
    return L


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    return flux_shim(tmp_path_factory)


@pytest.fixture(scope="module")
def dfbm():
    return package()


class Cfg:
    """a dfb_config as dfb_config_init + fill_config make it, kept alive with its arrays"""

    def __init__(self, dfbm, config):
        self.c = dfbm.dfb_config()
        self.c.struct_bytes = C.sizeof(self.c)
        self.c.grid_file_len = self.c.vel_fluc_file_len = self.c.line_file_len = -1
        self.c.device = -1
        self.keep = dfbm.fill_config(self.c, config)

    def ref(self):
        return C.byref(self.c)


def _d(a):
    return a.ctypes.data_as(D)


def tables(shim, cfg, mode):
    """(rc, dict of the plan's rows / vertices and the library's tables, error message)"""
    Ny, NzG, err = C.c_int(), C.c_int(), C.create_string_buffer(512)
    assert shim.fx_dims(cfg.ref(), C.byref(Ny), C.byref(NzG), err, 512) == 0, err.value
    ny, nz = Ny.value, NzG.value
    t = dict(rows=np.zeros((8, ny)), vert_y=np.zeros(ny + 1), vert_z=np.zeros(nz + 1), wy=np.zeros(ny), rc0=np.zeros(ny), hz=np.zeros(nz))
    d, mean = C.c_double(), C.c_double()
    rc = shim.fx_tables(cfg.ref(), mode, *[_d(t[k]) for k in ("rows", "vert_y", "vert_z", "wy", "rc0", "hz")], C.byref(d), C.byref(mean),
                        err, 512)
    t["D"], t["mean"] = d.value, mean.value
    return rc, t, err.value.decode()


def np_tables(t, mode):
    """the definition, restated: cells [vert_y[j], vert_y[j+1]) x [vert_z[k], vert_z[k+1]); g = rhos (1 + 0.2 Ms^2) or 1"""
    R11, Us, rhos, Ms = t["rows"][0], t["rows"][4], t["rows"][6], t["rows"][7]
    hy, hz = np.diff(t["vert_y"]), np.diff(t["vert_z"])
    g = rhos * (1.0 + 0.2 * Ms * Ms) if mode == 1 else np.ones_like(hy)
    A = np.outer(hy, hz).astype(np.longdouble)
    rc0 = np.sqrt(R11)
    Dref = float((A * (g * rc0)[:, None].astype(np.longdouble)).sum())
    flux = rhos * Us if mode == 1 else Us
    mean = float((A * flux[:, None].astype(np.longdouble)).sum())
    return dict(wy=g * hy, rc0=rc0, hz=hz, D=Dref, mean=mean, g=g)


def configs(dfbm, W, default_data):
    return {
        "default": Cfg(dfbm, dfbm.DFConfig(vel_fluc_file=str(default_data / "files" / "RST.dat"), line_file=str(default_data / "line.dat"))),
        "profile": Cfg(dfbm, dfbm.DFConfig.from_plane(W.plane_profile(96, 160, 24, 10))),
        "ragged_hz": Cfg(dfbm, dfbm.DFConfig.from_plane(W.plane_ragged(40, 56, 8, seed=3))),
    }


@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("which", ["default", "profile", "ragged_hz"])
def test_tables_match_numpy(shim, dfbm, W, default_data, which, mode):
    cfg = configs(dfbm, W, default_data)[which]
    rc, t, err = tables(shim, cfg, mode)
    assert rc == 0, err
    ref = np_tables(t, mode)
    assert np.array_equal(t["rc0"], ref["rc0"])                     # sqrt(R11): the epilogue's rc0, bit for bit
    assert np.array_equal(t["hz"], ref["hz"])
    assert np.allclose(t["wy"], ref["wy"], rtol=2e-16, atol=0)
    assert t["D"] == pytest.approx(ref["D"], rel=1e-13) and t["D"] > 0
    assert t["mean"] == pytest.approx(ref["mean"], rel=1e-13) and t["mean"] > 0
    if which == "ragged_hz":
        assert np.ptp(t["hz"]) > 0.1 * t["hz"].mean()                # the columns really differ in width
    if mode == 1 and which == "default":
        # the density term dominates near the boundary-layer edge of the reference's plane (Ms up to 5.8)
        assert ref["g"].max() / t["rows"][6][np.argmax(ref["g"])] > 6.0


def test_modes_differ_only_in_the_weights(shim, dfbm, W, default_data):
    cfg = configs(dfbm, W, default_data)["profile"]
    _, m, _ = tables(shim, cfg, 1)
    _, v, _ = tables(shim, cfg, 2)
    assert np.array_equal(m["rc0"], v["rc0"]) and np.array_equal(m["hz"], v["hz"])
    assert np.array_equal(v["wy"], np.diff(v["vert_y"]))
    assert not np.array_equal(m["wy"], v["wy"]) and m["D"] != v["D"]


@pytest.mark.parametrize("mode", [0, 3, -1])
def test_unknown_mode_is_refused(shim, dfbm, W, default_data, mode):
    rc, _, err = tables(shim, configs(dfbm, W, default_data)["profile"], mode)
    assert rc == dfbm.ERR_ARG and "unknown flux correction mode %d" % mode in err, err


def test_slab_is_refused(shim, dfbm, W):
    cfg = Cfg(dfbm, dfbm.DFConfig.from_plane(W.plane_profile(96, 160, 24, 10), k_begin=0, k_end=96))
    rc, _, err = tables(shim, cfg, 1)
    assert rc == dfbm.ERR_ARG and "whole plane" in err and "slab" in err, err


def test_plane_without_R11_is_refused(shim, dfbm, W):
    p = W.plane_profile(32, 48, 6, 6)
    p["rows"] = np.array(p["rows"], dtype=np.float64)
    p["rows"][0] = 0.0
    p["rows"][1] = 0.0                                            # R21 = 0 too: the plane stays valid
    rc, _, err = tables(shim, Cfg(dfbm, dfbm.DFConfig.from_plane(p)), 2)
    assert rc == dfbm.ERR_ARG and "R11 is zero on every row" in err, err


def test_fma_helper_is_correctly_rounded(shim):
    # 1 + 2^-30 squared needs the unrounded product: the exact result minus 1 is 2^-29 + 2^-60
    a = np.array([1.0 + 2.0 ** -30])
    out = np.zeros(1)
    shim.fx_fma(1, _d(a), _d(a), _d(np.array([-1.0])), _d(out))
    assert out[0] == 2.0 ** -29 + 2.0 ** -60 and a[0] * a[0] - 1.0 == 2.0 ** -29
