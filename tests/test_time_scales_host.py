"""Per-row time scales on the CPU, through tests/time_scales_shim.cpp (csrc/setup.cpp and csrc/restart.cpp built with g++, no CUDA):
dfb_time_scales_from_lengths against a numpy restatement of its formula (the u_min clamp at the wall, a trimmed Ny), the refusal of
entries that are not finite or not > 0, and the restart fingerprint -- the same as before this feature without rows, different with
rows, and different for different rows."""
import ctypes as C

import numpy as np
import pytest

from oracle_harness import package
from shims import build_shim

D = C.POINTER(C.c_double)


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    L = build_shim(tmp_path_factory, "time_scales", "restart.cpp")
    L.ts_plan.argtypes = [C.c_void_p, C.POINTER(C.c_int), D, D, D, C.c_int, C.c_char_p, C.c_int]
    L.ts_from_lengths.argtypes = [C.c_void_p, D, C.c_double, D, C.c_char_p, C.c_int]
    L.ts_fingerprint.argtypes = [C.c_void_p, D, C.POINTER(C.c_uint64), C.c_char_p, C.c_int]
    return L


@pytest.fixture(scope="module")
def dfbm():
    return package()


def _d(a):
    return None if a is None else a.ctypes.data_as(D)


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


def plan(shim, cfg):
    Ny, d_i, err = C.c_int(), C.c_double(), C.create_string_buffer(512)
    assert shim.ts_plan(cfg.ref(), C.byref(Ny), C.byref(d_i), None, None, 0, err, 512) == 0, err.value
    yc, Us = np.zeros(Ny.value), np.zeros(Ny.value)
    assert shim.ts_plan(cfg.ref(), C.byref(Ny), C.byref(d_i), _d(yc), _d(Us), Ny.value, err, 512) == 0, err.value
    return Ny.value, d_i.value, yc, Us


def from_lengths(shim, cfg, Ix, u_min, Ny):
    out, err = np.zeros((3, Ny)), C.create_string_buffer(512)
    rc = shim.ts_from_lengths(cfg.ref(), _d(np.asarray(Ix, dtype=np.float64)), u_min, _d(out), err, 512)
    return rc, out, err.value.decode()


def np_from_lengths(Ix, u_min, yc, Us, d_i):
    out = []
    for f in range(3):
        inn, outer = Ix[2 * f], Ix[2 * f + 1]
        Ixj = inn + (outer - inn) * 0.5 * (1 + np.tanh((yc / d_i - 0.2) / 0.03))
        out.append(Ixj / np.maximum(Us, u_min))
    return np.stack(out)


def fingerprint(shim, cfg, rows=None):
    fp, err = C.c_uint64(), C.create_string_buffer(512)
    r = None if rows is None else np.ascontiguousarray(rows, dtype=np.float64)
    rc = shim.ts_fingerprint(cfg.ref(), _d(r), C.byref(fp), err, 512)
    return rc, fp.value, err.value.decode()


IX = [2e-4, 1.6e-3, 1e-4, 8e-4, 1.5e-4, 1.2e-3]


@pytest.fixture(scope="module")
def default_cfg(dfbm, default_data, tmp_path_factory):
    """the reference's default plane with a fluctuation file that ends at 60 % of its rows: the setup trims the rows above its last
    y / d_i (df.cpp:282-288)"""
    head, rows = [], []
    for line in open(default_data / "files" / "RST.dat").read().splitlines():
        (rows if line.strip() and line.split()[0].replace(".", "").isdigit() else head).append(line)
    keep = rows[:int(len(rows) * 0.6)]
    head = [h.replace("i=%d" % len(rows), "i=%d" % len(keep)) for h in head]
    short = tmp_path_factory.mktemp("ts_trim") / "RST.dat"
    short.write_text("\n".join(head + keep) + "\n")
    full = Cfg(dfbm, dfbm.DFConfig(vel_fluc_file=str(default_data / "files" / "RST.dat"), line_file=str(default_data / "line.dat")))
    cfg = Cfg(dfbm, dfbm.DFConfig(vel_fluc_file=str(short), line_file=str(default_data / "line.dat")))
    cfg.untrimmed = full
    return cfg


@pytest.mark.parametrize("which", ["profile", "default_trimmed"])
def test_from_lengths_matches_numpy(shim, dfbm, W, default_cfg, which):
    cfg = default_cfg if which == "default_trimmed" else Cfg(dfbm, dfbm.DFConfig.from_plane(W.plane_profile(96, 160, 24, 10)))
    Ny, d_i, yc, Us = plan(shim, cfg)
    if which == "default_trimmed":
        assert Ny < plan(shim, cfg.untrimmed)[0]                           # rows beyond the DNS data were trimmed
    assert Us[0] < Us[-1]
    for u_min in (1e-3, 0.5 * Us[Ny // 4] + 0.5 * Us[0], 10.0 * Us[-1]):   # no clamp, a clamp near the wall, every row clamped
        rc, got, err = from_lengths(shim, cfg, IX, u_min, Ny)
        assert rc == 0, err
        ref = np_from_lengths(IX, u_min, yc, Us, d_i)
        assert np.allclose(got, ref, rtol=1e-14, atol=0), np.max(np.abs(got / ref - 1))
        clamped = Us < u_min                                               # these rows divide by u_min: a real clamp is tested
        assert clamped.any() == (u_min > 1e-3) and np.any(np_from_lengths(IX, 1e-3, yc, Us, d_i)[:, clamped] > ref[:, clamped] * 1.01) == (u_min > 1e-3)
    # far from the wall the blend is the outer length, at the wall the inner one
    rc, got, _ = from_lengths(shim, cfg, IX, 1e-3, Ny)
    assert got[0, -1] == pytest.approx(IX[1] / Us[-1], rel=1e-4) and got[2, 0] == pytest.approx(IX[4] / max(Us[0], 1e-3), rel=1e-4)


@pytest.mark.parametrize("bad", [("u_min", 0.0), ("u_min", -1.0), ("u_min", np.nan), ("Ix", 0.0), ("Ix", np.inf), ("Ix", -1e-3)])
def test_from_lengths_refuses_bad_inputs(shim, dfbm, W, bad):
    cfg = Cfg(dfbm, dfbm.DFConfig.from_plane(W.plane_profile(32, 48, 6, 6)))
    Ny = plan(shim, cfg)[0]
    Ix, u_min = list(IX), 1.0
    if bad[0] == "u_min":
        u_min = bad[1]
    else:
        Ix[3] = bad[1]
    rc, _, err = from_lengths(shim, cfg, Ix, u_min, Ny)
    assert rc == dfbm.ERR_ARG and bad[0] in err, err


# fingerprint of W.plane_profile(96, 160, 24, 10) with the default config values, as the library computed it before per-row time
# scales existed: a handle without rows must keep it, so that existing restart files still load
FP_PROFILE_96x160 = 0x30964925d0e2b739


def test_fingerprint_without_rows_is_unchanged(shim, dfbm, W):
    cfg = Cfg(dfbm, dfbm.DFConfig.from_plane(W.plane_profile(96, 160, 24, 10)))
    rc, fp, err = fingerprint(shim, cfg)
    assert rc == 0, err
    assert fp == FP_PROFILE_96x160, hex(fp)


def test_fingerprint_changes_with_rows(shim, dfbm, W):
    p = W.plane_profile(96, 160, 24, 10)
    cfg = Cfg(dfbm, dfbm.DFConfig.from_plane(p))
    Ny = plan(shim, cfg)[0]
    fp0 = fingerprint(shim, cfg)[1]
    Lt = np.asarray(p["scales"], dtype=np.float64)[:, 2]
    uniform = np.repeat(Lt[:, None], Ny, axis=1)
    rows = uniform * np.linspace(0.5, 1.5, Ny)[None, :]
    fps = {fingerprint(shim, cfg, r)[1] for r in (uniform, rows)}
    other = rows.copy()
    other[2, Ny - 1] = np.nextafter(other[2, Ny - 1], 1.0)                  # one ulp of one entry
    fps.add(fingerprint(shim, cfg, other)[1])
    assert len(fps) == 3 and fp0 not in fps                                 # rows equal to the scalar Lt are rows all the same
    assert fingerprint(shim, cfg, rows)[1] == fingerprint(shim, cfg, rows.copy())[1]


@pytest.mark.parametrize("value", [0.0, -1e-4, np.nan, np.inf])
def test_check_names_field_and_row(shim, dfbm, W, value):
    cfg = Cfg(dfbm, dfbm.DFConfig.from_plane(W.plane_profile(32, 48, 6, 6)))
    Ny = plan(shim, cfg)[0]
    rows = np.full((3, Ny), 1e-4)
    rows[1, 7] = value
    rc, _, err = fingerprint(shim, cfg, rows)
    assert rc == dfbm.ERR_ARG and "field 1 (v), row 7" in err, err
