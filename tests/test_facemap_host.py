"""Face maps (csrc/facemap.cpp) on the CPU: bilinear point maps against scipy's RegularGridInterpolator, their edges and wall flag,
area maps against a brute-force overlap computation, conservation over faces that tile the plane, and which slab serves which face.
facemap.cpp and csrc/setup.cpp are built with g++ against no CUDA library (tests/facemap_shim.cpp)."""
import ctypes as C

import numpy as np
import pytest
from scipy.interpolate import RegularGridInterpolator

from oracle_harness import package
from shims import build_shim

POINT, AREA = 0, 1
WALL_ZERO = 1
D = C.POINTER(C.c_double)


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    L = build_shim(tmp_path_factory, "facemap", "facemap.cpp")
    L.fm_build.restype = C.c_void_p
    L.fm_build.argtypes = [C.c_void_p, C.c_int, C.c_int, D, D, D, D, C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_int]
    L.fm_free.argtypes = [C.c_void_p]
    L.fm_sizes.argtypes = [C.c_void_p, C.POINTER(C.c_longlong)]
    L.fm_arrays.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), D]
    L.fm_geom.argtypes = [C.c_void_p, C.c_int, D]
    return L


@pytest.fixture(scope="module")
def dfbm():
    return package()


class Map:
    """one build_face_map result: served [n], taps(i) -> (global cells (j, k), weights) in the map's order, geometry of the plane"""

    def __init__(self, L, dfbm, config, kind, yf, zf, hy=None, hz=None, own=(0, 0), flags=0):
        c = dfbm.dfb_config()
        c.struct_bytes = C.sizeof(c)
        c.grid_file_len = c.vel_fluc_file_len = c.line_file_len = -1
        c.device = -1
        keep = dfbm.fill_config(c, config)
        arr = [None if a is None else np.ascontiguousarray(a, dtype=np.float64) for a in (yf, zf, hy, hz)]
        ptrs = [None if a is None else a.ctypes.data_as(D) for a in arr]
        err = C.create_string_buffer(1024)
        n = len(arr[0])
        h = L.fm_build(C.byref(c), kind, n, *ptrs, own[0], own[1], flags, err, 1024)
        del keep
        if not h:
            code, msg = err.value.decode().split(" ", 1)
            raise dfbm.DfbError(int(code), msg)
        s = (C.c_longlong * 8)()
        L.fm_sizes(h, s)
        self.Ny, self.NzG, self.k0, self.k1, self.periodic, self.n, self.n_served, ntaps = list(s)
        self.W = self.k1 - self.k0
        self.served = np.zeros(n, dtype=np.int32)
        self.ptr = np.zeros(n + 1, dtype=np.int32)
        self.idx = np.zeros(max(ntaps, 1), dtype=np.int32)
        self.w = np.zeros(max(ntaps, 1))
        L.fm_arrays(h, self.served.ctypes.data_as(C.POINTER(C.c_int)), self.ptr.ctypes.data_as(C.POINTER(C.c_int)),
                    self.idx.ctypes.data_as(C.POINTER(C.c_int)), self.w.ctypes.data_as(D))
        self.geom = []
        for which, m in enumerate((self.Ny, self.NzG, self.Ny + 1, self.NzG + 1)):
            g = np.zeros(m)
            L.fm_geom(h, which, g.ctypes.data_as(D))
            self.geom.append(g)
        self.yc, self.zc, self.vy, self.vz = self.geom
        L.fm_free(h)
        self.kind = kind
        if kind == POINT:
            self.ptr = np.arange(n + 1, dtype=np.int32) * 4

    def taps(self, i):
        a, b = self.ptr[i], self.ptr[i + 1]
        cell = self.idx[a:b]
        return np.stack([cell // self.W, cell % self.W + self.k0], axis=1), self.w[a:b]

    def apply(self, F):
        """sum of w * F[j, k] over each face's taps in the map's order, F the global [Ny][NzG] field; NaN for unserved faces"""
        out = np.full(self.n, np.nan)
        for i in np.nonzero(self.served)[0]:
            jk, w = self.taps(i)
            acc = 0.0
            for (j, k), wt in zip(jk, w):
                acc += wt * F[j, k]
            out[i] = acc
        return out


def default_config(dfbm, data, **kw):
    """the reference's default plane (tanh vertex grid), from input files in its formats"""
    return dfbm.DFConfig(vel_fluc_file=str(data / "files" / "RST.dat"), line_file=str(data / "line.dat"), **kw)


def planes(W):
    return {"stretched": W.plane_profile(48, 64, 8, 6), "odd_nz": W.plane_profile(40, 37, 6, 6)}


def close(got, ref, tol):
    scale = np.maximum(np.abs(ref), np.sqrt(np.mean(ref * ref)))
    return float(np.max(np.abs(got - ref) / scale))


def configs(dfbm, W, data):
    out = {"default": default_config(dfbm, data)}
    for name, p in planes(W).items():
        out[name] = dfbm.DFConfig.from_plane(p)
        out[name + "_periodic"] = dfbm.DFConfig.from_plane(p, periodic_z=1)
    return out


# ---------------------------------------------------------------------------------------------
# point maps
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["default", "stretched", "odd_nz", "stretched_periodic", "odd_nz_periodic"])
def test_point_against_scipy(shim, dfbm, W, default_data, name):
    cfg = configs(dfbm, W, default_data)[name]
    rng = np.random.default_rng(7)
    probe = Map(shim, dfbm, cfg, POINT, [0.0], [0.0])
    yc, zc, vz = probe.yc, probe.zc, probe.vz
    n = 4000
    yf = rng.uniform(yc[0], yc[-1], n)
    if probe.periodic:                   # the whole span, seam included: against the grid padded with the wrapped columns
        Lz = vz[-1] - vz[0]
        zf = rng.uniform(vz[0], vz[-1], n)
        zgrid = np.concatenate([[zc[-1] - Lz], zc, [zc[0] + Lz]])
    else:
        zf = rng.uniform(zc[0], zc[-1], n)
        zgrid = zc
    m = Map(shim, dfbm, cfg, POINT, yf, zf)
    assert m.n_served == n and m.served.all()
    for _ in range(2):
        F = rng.standard_normal((m.Ny, m.NzG))
        Fg = np.concatenate([F[:, -1:], F, F[:, :1]], axis=1) if m.periodic else F
        ref = RegularGridInterpolator((yc, zgrid), Fg, method="linear")(np.stack([yf, zf], axis=1))
        assert close(m.apply(F), ref, 1e-14) <= 1e-14
    assert np.all(m.w >= 0) and np.all(m.w <= 1)


@pytest.mark.parametrize("name", ["default", "stretched_periodic", "odd_nz"])
def test_point_at_cell_centres(shim, dfbm, W, default_data, name):
    cfg = configs(dfbm, W, default_data)[name]
    probe = Map(shim, dfbm, cfg, POINT, [0.0], [0.0])
    jj, kk = np.meshgrid(np.arange(probe.Ny), np.arange(probe.NzG), indexing="ij")
    m = Map(shim, dfbm, cfg, POINT, probe.yc[jj.ravel()], probe.zc[kk.ravel()])
    for i, (j, k) in enumerate(zip(jj.ravel(), kk.ravel())):
        jk, w = m.taps(i)
        nz = w != 0
        assert nz.sum() == 1 and w[nz][0] == 1.0 and tuple(jk[nz][0]) == (j, k)
        assert np.all(jk[~nz] == (j, k))                     # zero-weight taps read the face's own cell


def test_point_edges_and_wall(shim, dfbm, W):
    p = planes(W)["stretched"]
    cfg = dfbm.DFConfig.from_plane(p)
    probe = Map(shim, dfbm, cfg, POINT, [0.0], [0.0])
    yc, zc, vy, vz = probe.yc, probe.zc, probe.vy, probe.vz
    rng = np.random.default_rng(3)
    F = rng.standard_normal((probe.Ny, probe.NzG))
    k = 10
    zmid = 0.5 * (zc[k] + zc[k + 1])
    # above the top row: the top row; below the first centre: the first row; beyond the spanwise edges: the edge columns
    ys = np.array([yc[-1] + 1.0, yc[-1], 0.5 * (vy[0] + yc[0]), vy[0] - 1.0, yc[3]])
    zs = np.array([zmid, zmid, zmid, zmid, vz[-1] + 5.0])
    m = Map(shim, dfbm, cfg, POINT, np.r_[ys, yc[3]], np.r_[zs, vz[0] - 5.0])
    got = m.apply(F)
    rowz = lambda j: RegularGridInterpolator((zc,), F[j])([zmid])[0]
    assert close(got[:4], np.array([rowz(-1), rowz(-1), rowz(0), rowz(0)]), 1e-15) <= 1e-15
    assert got[4] == F[3, -1] and got[5] == F[3, 0]
    # DFB_MAP_WALL_ZERO: linear to 0 at vert_y[0], 0 below it; unchanged above the first centre
    s = np.array([0.0, 0.25, 0.5, 1.0])
    yw = np.r_[vy[0] + s * (yc[0] - vy[0]), vy[0] - 1e-3, yc[5]]
    mw = Map(shim, dfbm, cfg, POINT, yw, np.full(len(yw), zc[k]), flags=WALL_ZERO)
    got = mw.apply(F)
    assert close(got[:4], s * F[0, k], 1e-15) <= 1e-15
    assert got[4] == 0.0 and got[5] == F[5, k]
    jk, w = mw.taps(4)
    assert np.all(w == 0) and np.all(jk[:, 1] == k)


# ---------------------------------------------------------------------------------------------
# area maps
# ---------------------------------------------------------------------------------------------
def brute_area(m, yf, zf, hy, hz):
    """dense [n][Ny][NzG] weights: overlap of each face with every cell, the first / last cell extended to -inf / +inf (wrapping in
    z on a periodic plane), over the face area"""
    vy, vz = m.vy.copy(), m.vz.copy()
    Lz = vz[-1] - vz[0]
    ylo_c, yhi_c = vy[:-1].copy(), vy[1:].copy()
    ylo_c[0], yhi_c[-1] = -np.inf, np.inf
    out = np.zeros((len(yf), m.Ny, m.NzG))
    for i in range(len(yf)):
        a, b = yf[i] - hy[i] / 2, yf[i] + hy[i] / 2
        oy = np.clip(np.minimum(b, yhi_c) - np.maximum(a, ylo_c), 0, None)
        c, d = zf[i] - hz[i] / 2, zf[i] + hz[i] / 2
        if m.periodic:
            oz = np.zeros(m.NzG)
            for s in range(-2, 3):
                oz += np.clip(np.minimum(d - s * Lz, vz[1:]) - np.maximum(c - s * Lz, vz[:-1]), 0, None)
        else:
            zlo_c, zhi_c = vz[:-1].copy(), vz[1:].copy()
            zlo_c[0], zhi_c[-1] = -np.inf, np.inf
            oz = np.clip(np.minimum(d, zhi_c) - np.maximum(c, zlo_c), 0, None)
        out[i] = np.outer(oy / oy.sum(), oz / oz.sum())         # the face area as the sum of its overlaps (hy hz to rounding)
    return out


def dense(m, i):
    D_ = np.zeros((m.Ny, m.NzG))
    jk, w = m.taps(i)
    for (j, k), wt in zip(jk, w):
        D_[j, k] += wt
    return D_


@pytest.mark.parametrize("name", ["default", "stretched", "odd_nz_periodic"])
def test_area_against_brute_force(shim, dfbm, W, default_data, name):
    cfg = configs(dfbm, W, default_data)[name]
    probe = Map(shim, dfbm, cfg, POINT, [0.0], [0.0])
    vy, vz = probe.vy, probe.vz
    rng = np.random.default_rng(11)
    n = 300
    Ly, Lz = vy[-1] - vy[0], vz[-1] - vz[0]
    yf = rng.uniform(vy[0] - 0.05 * Ly, vy[-1] + 0.05 * Ly, n)   # some faces reach outside the plane
    zf = rng.uniform(vz[0] - 0.05 * Lz, vz[-1] + 0.05 * Lz, n)
    hy = rng.uniform(0.001, 0.1, n) * Ly
    hz = rng.uniform(0.001, 0.1, n) * Lz
    m = Map(shim, dfbm, cfg, AREA, yf, zf, hy, hz)
    assert m.served.all()
    B = brute_area(m, yf, zf, hy, hz)
    for i in range(n):
        jk, w = m.taps(i)
        assert np.all(w > 0)
        assert abs(w.sum() - 1.0) <= 1e-15, (i, w.sum() - 1)
        assert np.max(np.abs(dense(m, i) - B[i])) <= 1e-15, i
        order = jk[:, 0] * m.NzG + jk[:, 1]
        assert np.all(np.diff(order) > 0)                     # fixed order: row-major over the plane, each cell once


def test_area_tiling_conserves(shim, dfbm, W):
    """faces that tile the plane at another resolution carry the plane's integral: sum(face area * value) = sum(cell area * value)"""
    for periodic in (0, 1):
        cfg = dfbm.DFConfig.from_plane(planes(W)["stretched"], periodic_z=periodic)
        probe = Map(shim, dfbm, cfg, POINT, [0.0], [0.0])
        vy, vz = probe.vy, probe.vz
        ey = np.linspace(vy[0], vy[-1], 31)
        ez = np.linspace(vz[0], vz[-1], 23) + (0.3 * (vz[1] - vz[0]) if periodic else 0.0)   # periodic: tiles across the seam
        yy, zz = np.meshgrid(0.5 * (ey[1:] + ey[:-1]), 0.5 * (ez[1:] + ez[:-1]), indexing="ij")
        hy, hz = np.meshgrid(np.diff(ey), np.diff(ez), indexing="ij")
        m = Map(shim, dfbm, cfg, AREA, yy.ravel(), zz.ravel(), hy.ravel(), hz.ravel())
        F = np.random.default_rng(5).standard_normal((m.Ny, m.NzG))
        cell_area = np.outer(np.diff(vy), np.diff(vz))
        total = float((cell_area * F).sum())
        faces = float((hy.ravel() * hz.ravel() * m.apply(F)).sum())
        assert abs(faces - total) <= 1e-13 * float((cell_area * np.abs(F)).sum()), (periodic, faces, total)


def test_area_face_equal_to_cell(shim, dfbm, W, default_data):
    for cfg in (default_config(dfbm, default_data), dfbm.DFConfig.from_plane(planes(W)["odd_nz"], periodic_z=1)):
        probe = Map(shim, dfbm, cfg, POINT, [0.0], [0.0])
        vy, vz = probe.vy, probe.vz
        jj, kk = np.meshgrid(np.arange(probe.Ny), np.arange(probe.NzG), indexing="ij")
        j, k = jj.ravel(), kk.ravel()
        m = Map(shim, dfbm, cfg, AREA, 0.5 * (vy[j] + vy[j + 1]), 0.5 * (vz[k] + vz[k + 1]), vy[j + 1] - vy[j], vz[k + 1] - vz[k])
        for i in range(len(j)):
            jk, w = m.taps(i)
            assert len(w) == 1 and w[0] == 1.0 and tuple(jk[0]) == (j[i], k[i]), i


# ---------------------------------------------------------------------------------------------
# which slab serves which face
# ---------------------------------------------------------------------------------------------
def slabs(NzG, cuts):
    """16-aligned cuts, each slab widened by 16 columns on each side within the plane: [(k_begin, k_end, own_begin, own_end)]"""
    return [(max(0, a - 16), min(NzG, b + 16), a, b) for a, b in zip(cuts[:-1], cuts[1:])]


@pytest.mark.parametrize("kind", [POINT, AREA])
@pytest.mark.parametrize("periodic", [0, 1])
def test_slabs_serve_every_face_once(shim, dfbm, W, kind, periodic):
    p = W.plane_profile(32, 96, 6, 6)
    whole_cfg = dfbm.DFConfig.from_plane(p, periodic_z=periodic)
    probe = Map(shim, dfbm, whole_cfg, POINT, [0.0], [0.0])
    yc, zc, vy, vz = probe.yc, probe.zc, probe.vy, probe.vz
    rng = np.random.default_rng(21 + kind + 2 * periodic)
    n = 3000
    yf = rng.uniform(vy[0], vy[-1], n)
    # a periodic plane's faces within half a cell of the seam need both edge columns: only a whole-plane handle serves them
    zf = rng.uniform(zc[0], zc[-1], n) if periodic else rng.uniform(vz[0] - 1e-4, vz[-1] + 1e-4, n)
    ext = dict(hy=rng.uniform(0.2, 3.0, n) * np.diff(vy).mean(), hz=rng.uniform(0.2, 3.0, n) * np.diff(vz).mean()) if kind == AREA else {}
    if kind == AREA and periodic:        # ... as do area faces across the seam
        zf = vz[0] + 0.5 * ext["hz"] + rng.uniform(0, 1, n) * (vz[-1] - vz[0] - ext["hz"])
    whole = Map(shim, dfbm, whole_cfg, kind, yf, zf, **ext)
    assert whole.served.all()
    for cuts in ([0, 48, 96], [0, 16, 48, 64, 96]):
        count = np.zeros(n, dtype=int)
        for k0, k1, o0, o1 in slabs(96, cuts):
            m = Map(shim, dfbm, dfbm.DFConfig.from_plane(p, periodic_z=periodic, k_begin=k0, k_end=k1), kind, yf, zf, own=(o0, o1), **ext)
            count += m.served
            for i in np.nonzero(m.served)[0][::7]:             # the same taps as the whole plane's, in the same order
                a, wa = m.taps(i)
                b, wb = whole.taps(i)
                nz = wb != 0
                assert np.array_equal(a[wa != 0], b[nz]) and np.array_equal(wa, wb), i
        assert np.all(count == 1), np.nonzero(count != 1)[0][:5]


def test_unwidened_slab_refuses_seam_face(shim, dfbm, W):
    p = W.plane_profile(32, 96, 6, 6)
    probe = Map(shim, dfbm, dfbm.DFConfig.from_plane(p), POINT, [0.0], [0.0])
    zc, yc = probe.zc, probe.yc
    cfg = dfbm.DFConfig.from_plane(p, k_begin=32, k_end=64)
    with pytest.raises(dfbm.DfbError) as e:                  # right half of column 63: bilinear with column 64
        Map(shim, dfbm, cfg, POINT, [yc[4]], [0.5 * (zc[63] + zc[64]) - 1e-9 * (zc[64] - zc[63])])
    assert e.value.code == dfbm.ERR_ARG and "columns 63..64" in str(e.value) and "[32, 64)" in str(e.value)
    with pytest.raises(dfbm.DfbError) as e:                  # left half of column 32: bilinear with column 31
        Map(shim, dfbm, cfg, POINT, [yc[4]], [0.25 * zc[31] + 0.75 * zc[32]])
    assert "columns 31..32" in str(e.value)
    # a face on the centre of the slab's last column needs no other column
    m = Map(shim, dfbm, cfg, POINT, [yc[4]], [zc[63]])
    assert m.served.all()
    # periodic: a face between the centres of columns 95 and 0 names the seam
    pc = dfbm.DFConfig.from_plane(p, periodic_z=1, k_begin=0, k_end=80)
    with pytest.raises(dfbm.DfbError) as e:
        Map(shim, dfbm, pc, POINT, [yc[4]], [probe.vz[0] + 1e-3 * (zc[1] - zc[0])])
    assert "columns 0..95 (across the periodic seam)" in str(e.value)


def test_bad_arguments(shim, dfbm, W):
    cfg = dfbm.DFConfig.from_plane(planes(W)["stretched"])
    one = [1e-4]
    cases = [
        dict(kind=2, yf=one, zf=one),
        dict(kind=POINT, yf=one, zf=one, flags=2),
        dict(kind=AREA, yf=one, zf=one, hy=one, hz=one, flags=WALL_ZERO),
        dict(kind=POINT, yf=[np.nan], zf=one),
        dict(kind=POINT, yf=one, zf=[np.inf]),
        dict(kind=POINT, yf=one, zf=one, hy=one, hz=one),
        dict(kind=AREA, yf=one, zf=one),
        dict(kind=AREA, yf=one, zf=one, hy=[0.0], hz=one),
        dict(kind=AREA, yf=one, zf=one, hy=one, hz=[-1.0]),
        dict(kind=POINT, yf=one, zf=one, own=(10, 5)),
    ]
    for c in cases:
        kw = dict(c)
        with pytest.raises(dfbm.DfbError) as e:
            Map(shim, dfbm, cfg, kw.pop("kind"), kw.pop("yf"), kw.pop("zf"), **kw)
        assert e.value.code == dfbm.ERR_ARG, c
    with pytest.raises(dfbm.DfbError) as e:                  # the own columns must lie in the slab
        Map(shim, dfbm, dfbm.DFConfig.from_plane(planes(W)["stretched"], k_begin=16, k_end=48), POINT, one, one, own=(0, 32))
    assert "own columns" in str(e.value)
