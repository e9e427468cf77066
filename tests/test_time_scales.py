"""Per-row temporal scales (dfb_set_time_scales) on the GPU: bands of rows equal handles whose scalar Lt is the band's, bit for bit, on
every kernel form, periodic planes, batches and slabs; rows equal to the scalar Lt are the scalar path bit for bit, and clearing them
continues like a handle that never set them; the oracle's blend applied row by row matches at the 1e-12 gate, also over 200 steps of
changing dt without synchronisation through every host-driven call; attached steps and graph replays; the delivered temporal
correlation per row; restart files; refusals."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, normwise_close
from oracle_harness import Model, check

pytestmark = pytest.mark.gpu

FIELDS = (0, 1, 2, 3, 4, 5, 6, 7)          # u', v', w', T', rho', filt u, v, w
K = 30
DTS = [1e-8 * (1 + k % 7) for k in range(K)]
FACTORS = (0.25, 1.0, 4.0)                 # Lt of each band of rows, times the plane's scalar Lt


def profile(W):
    return W.plane_profile(128, 256, 24, 16)


def make(dfb, pl, nplanes=1, seed=91, **kw):
    return dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(pl, seed=seed, device=0, **kw), fetch=False, nplanes=nplanes)


def scaled(pl, factor):
    """the plane with every field's scalar Lt times factor"""
    q = dict(pl)
    q["scales"] = np.array(pl["scales"], dtype=np.float64)
    q["scales"][:, 2] *= factor
    return q


def bands(Ny):
    return [slice(0, Ny // 3), slice(Ny // 3, (2 * Ny) // 3), slice((2 * Ny) // 3, Ny)]


def band_rows(pl, Ny):
    Lt = np.asarray(pl["scales"], dtype=np.float64)[:, 2]
    rows = np.zeros((3, Ny))
    for b, s in enumerate(bands(Ny)):
        rows[:, s] = (Lt * FACTORS[b])[:, None]
    return rows


def snapshot(df):
    return np.stack([df.get(w, plane=p) for p in range(df.nplanes) for w in FIELDS])


FORMS = {"default": ({}, {}), "y_dense": ({"DFB_Y_MODE": "0"}, {}), "y_chunk_rec": ({"DFB_Y_MODE": "1"}, {}),
         "y_run": ({"DFB_Y_MODE": "2"}, {}), "z_direct": ({"DFB_Z_MODE": "0"}, {}), "simple": ({}, dict(kernel_variant=1)),
         "periodic": ({}, dict(periodic_z=1)), "batch3": ({}, dict(nplanes=3))}


def form(monkeypatch, name):
    env, kw = FORMS[name]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    kw = dict(kw)
    return kw.pop("nplanes", 1), kw


# ---- 1. bands of rows equal scalar handles ----
@pytest.mark.parametrize("name", list(FORMS))
def test_row_bands_equal_scalar_handles(dfb, W, monkeypatch, name):
    pl = profile(W)
    nplanes, kw = form(monkeypatch, name)
    h = make(dfb, pl, nplanes, **kw)
    Ny = h.Ny
    h.set_time_scales(band_rows(pl, Ny))
    assert h.info(15) == 1 and np.array_equal(h.time_scales, band_rows(pl, Ny))
    scal = [make(dfb, scaled(pl, f), nplanes, **kw) for f in FACTORS]
    for dt in DTS:
        for d in [h] + scal:
            d.filter(dt)
    got = snapshot(h)
    for b, s in enumerate(bands(Ny)):
        assert np.array_equal(got[:, s], snapshot(scal[b])[:, s]), (name, b)
    for d in [h] + scal:
        d.close()


def test_row_bands_on_slabs_equal_whole_plane(dfb, W):
    """two slabs cut on a multiple of 16 columns, each with the rows, against the whole plane with the rows and its bands against
    scalar handles"""
    pl = profile(W)
    whole = make(dfb, pl)
    rows = band_rows(pl, whole.Ny)
    whole.set_time_scales(rows)
    slabs = [make(dfb, pl, k_begin=0, k_end=112), make(dfb, pl, k_begin=112, k_end=256)]
    for s in slabs:
        s.set_time_scales(rows)
    scal = [make(dfb, scaled(pl, f)) for f in FACTORS]
    for dt in DTS:
        for d in [whole] + slabs + scal:
            d.filter(dt)
    ref = snapshot(whole)
    assert np.array_equal(np.concatenate([snapshot(s) for s in slabs], axis=2), ref)
    for b, s in enumerate(bands(whole.Ny)):
        assert np.array_equal(ref[:, s], snapshot(scal[b])[:, s])
    for d in [whole] + slabs + scal:
        d.close()


# ---- 2. uniform rows are the scalar path ----
@pytest.mark.parametrize("name", list(FORMS))
def test_uniform_rows_equal_scalar_path(dfb, W, monkeypatch, name):
    pl = profile(W)
    nplanes, kw = form(monkeypatch, name)
    a, b = make(dfb, pl, nplanes, **kw), make(dfb, pl, nplanes, **kw)
    Lt = np.asarray(pl["scales"], dtype=np.float64)[:, 2]
    a.set_time_scales(np.repeat(Lt[:, None], a.Ny, axis=1))
    assert np.array_equal(a.time_scales, b.time_scales) and b.info(15) == 0
    for dt in DTS:
        a.filter(dt)
        b.filter(dt)
    assert np.array_equal(snapshot(a), snapshot(b))
    a.close()
    b.close()


def test_clear_mid_run_continues_like_never_set(dfb, W):
    pl = profile(W)
    a, b = make(dfb, pl), make(dfb, pl)
    a.set_time_scales(band_rows(pl, a.Ny))
    for dt in DTS[:10]:
        a.filter(dt)
    a.set_time_scales(None)
    assert a.info(15) == 0
    fo, step = a.get_state()
    b.set_state(fo, step)
    for dt in DTS[10:]:
        a.filter(dt)
        b.filter(dt)
    assert np.array_equal(snapshot(a), snapshot(b))
    a.close()
    b.close()


# ---- 3. against the oracle under identical noise ----
def rows_step(O, plane, rys, hal, fo, dt, Lt_rows, first):
    """the oracle's step (orc_step's order: per field y-sweep, z-sweep, blend; then the RST scaling and T', rho') with the unchanged
    orc_correlate applied row by row with each row's Lt"""
    L, d, i = O.lib(), O._d, O._i
    Ny, Nz = plane["Ny"], plane["Nz"]
    rows = np.ascontiguousarray(plane["rows"], dtype=np.float64)
    fo = [np.array(fo[f], dtype=np.float64).reshape(Ny, Nz).copy() for f in range(3)]
    filt = [np.zeros((Ny, Nz)) for _ in range(3)]
    fluc = [np.zeros((Ny, Nz)) for _ in range(3)]
    T, rho = np.zeros((Ny, Nz)), np.zeros((Ny, Nz))
    for f in range(3):
        M = int(plane["Nz_max"][f])
        N_y = np.ascontiguousarray(plane["N_y"][f], dtype=np.int32)
        N_z = np.ascontiguousarray(plane["N_z"][f], dtype=np.int32)
        ry = np.ascontiguousarray(rys[f], dtype=np.float64)
        rz = O.make_rzs(np.asarray(hal[f]), Ny, Nz, M)
        L.orc_sweep_y(C.c_int(Ny), C.c_int(Nz), C.c_int(int(plane["Ny_max"][f])), C.c_int(M), i(N_y), d(ry), d(rz))
        L.orc_sweep_z(C.c_int(Ny), C.c_int(Nz), C.c_int(M), i(N_z), d(rz), d(filt[f]))
        if not first:
            for j in range(Ny):
                L.orc_correlate(C.c_long(Nz), d(fo[f][j]), d(filt[f][j]), C.c_double(dt), C.c_double(float(Lt_rows[f][j])))
    r = [np.ascontiguousarray(rows[k]) for k in range(8)]
    L.orc_rst_scaling(C.c_int(Ny), C.c_int(Nz), d(r[0]), d(r[1]), d(r[2]), d(r[3]), d(filt[0]), d(filt[1]), d(filt[2]),
                      d(fluc[0]), d(fluc[1]), d(fluc[2]), d(fo[0]), d(fo[1]), d(fo[2]))
    if not first:
        L.orc_sra(C.c_int(Ny), C.c_int(Nz), d(r[7]), d(r[4]), d(r[5]), d(r[6]), d(fluc[0]), d(T), d(rho))
    return dict(fluc=np.stack(fluc), filt_old=np.stack(fo), T=T, rho=rho)


class RowsModel(Model):
    """Model (oracle_harness) whose blend uses per-row time scales"""

    def __init__(self, O, plane, seed, Lt_rows, nplanes=1):
        super().__init__(O, plane, seed, 0, nplanes)
        self.Lt_rows = Lt_rows

    def filter(self, dt, first=False):
        for p in range(self.P):
            rys = [self.noise(p, f, self.step)[0] for f in range(3)]
            hal = [self.noise(p, f, self.step)[1] for f in range(3)]
            o = rows_step(self.O, self.plane, rys, hal, self.fo[p], dt, self.Lt_rows, first)
            self.fo[p] = o["filt_old"]
            self.out[p, :3] = o["fluc"]
            if not first:
                self.out[p, 3], self.out[p, 4] = o["T"], o["rho"]
        self.noise_step = self.step
        self.step += 1


def oracle_plane(O, pl):
    O.half_widths(pl)
    return pl


def profile_rows(pl, Ny):
    """a smooth wall-normal profile: Lt from 0.2 of the scalar value at the wall to 1.5 times it at the top"""
    Lt = np.asarray(pl["scales"], dtype=np.float64)[:, 2]
    return Lt[:, None] * np.linspace(0.2, 1.5, Ny)[None, :] ** 2


@pytest.mark.parametrize("wname,steps", [("512x512_N32", 4), ("1024x2048_profile_N128", 2)])
def test_rows_against_oracle(dfb, W, O, wname, steps):
    pl = oracle_plane(O, W.NAMED[wname]())
    df = make(dfb, pl, seed=7)
    rows = profile_rows(pl, df.Ny)
    df.set_time_scales(rows)
    m = RowsModel(O, pl, 7, rows)
    m.first_step()
    worst = {}
    for s in range(steps):
        dt = 2e-7 * (1 + s)
        df.filter(dt)
        m.filter(dt)
        check(df, m, worst=worst)
    print(wname, "worst normwise ratio", worst)
    df.close()


# ---- 4. dt changing every step, no synchronisation in between ----
@pytest.mark.parametrize("call", ["filter", "filter_batch", "begin_end"])
def test_changing_dt_without_sync(dfb, W, O, call):
    pl = oracle_plane(O, W.plane_profile(48, 96, 8, 8))
    df = make(dfb, pl, seed=5)
    rows = profile_rows(pl, df.Ny)
    df.set_time_scales(rows)
    m = RowsModel(O, pl, 5, rows)
    m.first_step()
    n, Ny, Nz = 200, df.Ny, df.Nz
    dts = [1e-7 * (1 + (7 * k) % 13) for k in range(n)]
    if call == "filter":
        for dt in dts:
            df.filter(dt)
        for dt in dts:
            m.filter(dt)
        check(df, m)
    elif call == "filter_batch":
        out = np.zeros((n, 5, Ny, Nz))
        df.filter_batch(dts, out=out)
        for k, dt in enumerate(dts):
            m.filter(dt)
            for i in range(5):
                assert normwise_close(out[k, i], m.out[0, i], 1e-12)[0], (k, i)
        check(df, m)
    else:
        L = dfb.lib()
        bufs = [np.zeros((5, Ny, Nz)) for _ in range(2)]
        ptrs = lambda b: [C.c_void_p(b[i].ctypes.data) for i in range(5)]   # noqa: E731
        assert L.dfb_filter_to_host_begin(df._h, dts[0], *ptrs(bufs[0])) == 0
        for k in range(1, n + 1):
            if k < n:
                assert L.dfb_filter_to_host_begin(df._h, dts[k], *ptrs(bufs[k % 2])) == 0
            assert L.dfb_filter_to_host_end(df._h) == 0
            m.filter(dts[k - 1])
            got = bufs[(k - 1) % 2]
            for i in range(5):
                assert normwise_close(got[i], m.out[0, i], 1e-12)[0], (k - 1, i)
    df.close()


# ---- 5. attached steps ----
def test_attached_rows(dfb, W):
    import torch
    pl = profile(W)
    rows = band_rows(pl, 128)
    a, b, c = make(dfb, pl), make(dfb, pl), make(dfb, pl)
    for d in (a, b, c):
        d.set_time_scales(rows)
    s = torch.cuda.Stream()
    dt_a = torch.zeros(1, dtype=torch.float64, device="cuda")
    dt_b = torch.zeros(1, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    a.attach_stream(s)
    b.attach_stream(s)
    with pytest.raises(dfb.DfbError) as e:
        a.set_time_scales(rows)
    assert e.value.code == dfb.ERR_STATE
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        a.filter_dev(dt_a)
    with torch.cuda.stream(s):
        for dt in DTS:
            dt_a.fill_(dt)
            g.replay()
            dt_b.fill_(dt)
            b.filter_dev(dt_b)
    for dt in DTS:
        c.filter(dt)
    s.synchronize()
    ga, gb, gc = snapshot(a), snapshot(b), snapshot(c)
    assert np.array_equal(ga, gb)
    for x, y in zip(gb, gc):
        ok, r = normwise_close(x, y, 1e-14)
        assert ok, r
    assert a.step == c.step
    a.attach_stream(None)
    b.attach_stream(None)
    del g
    for d in (a, b, c):
        d.close()


# ---- 6. delivered temporal correlation ----
def test_delivered_temporal_correlation(dfb, W):
    pl = W.plane_profile(48, 256, 6, 8)
    df = make(dfb, pl, seed=3)
    Ny, Nz = df.Ny, df.Nz
    Lt0 = np.asarray(pl["scales"], dtype=np.float64)[:, 2]
    lo = np.arange(Ny) < Ny // 2
    Lt = Lt0[:, None] * np.where(lo, 1.0, 4.0)[None, :]                     # two bands, 4x apart
    df.set_time_scales(Lt)
    dt = 0.3 * Lt0[0] / np.pi                                                # lag-1 correlation exp(-0.15) of u' in the first band
    S, L = 1500, 8
    df.corr_enable(z=dfb.CORR_SUPPORT, y=0, t=L)
    for _ in range(S):
        df.filter(dt)
    R11, R21, R22 = df.table(0), df.table(1), df.table(2)
    bb = np.where(R11 < 1e-10, 0.0, R21 / np.sqrt(np.where(R11 < 1e-10, 1.0, R11)))
    cc = R22 - bb * bb
    m = np.arange(L + 1)

    def expected(Ltf):
        sa = np.exp(-np.pi * dt / (2 * Ltf))                                # [3][Ny]
        e = [sa[f][:, None] ** m[None, :] for f in range(3)]
        w = np.where(bb * bb + cc > 0, bb * bb + cc, 1.0)
        e[1] = (bb[:, None] ** 2 * e[0] + cc[:, None] * sa[1][:, None] ** m[None, :]) / w[:, None]
        return e, sa

    def errors(Ltf):
        e, sa = expected(Ltf)
        out = []
        for f in range(3):
            Rt = df.corr(f, dfb.CORR_T)[0]
            Rz = df.corr(f, dfb.CORR_Z)[0]
            two_z = 2.0 * np.nansum(Rz ** 2, axis=1) - Rz[:, 0] ** 2
            rho1 = sa[f] if f != 1 else np.maximum(sa[0], sa[1])
            two_t = (1 + rho1 ** 2) / (1 - rho1 ** 2)                        # AR(1): sum over all lags of rho^(2|m|)
            sig = np.sqrt(2.0 * two_z * two_t / (Nz * S))
            ok = R11 > 1e-10
            out.append(np.nanmax(np.abs(Rt[ok] - e[f][ok]) / sig[ok, None]))
        return out

    err = errors(Lt)
    assert max(err) < 6.0, err
    scalar = errors(np.repeat(Lt0[:, None], Ny, axis=1))
    assert scalar[0] > 6.0 and scalar[2] > 6.0, scalar                      # the scalar expectation fails the per-row handle
    df.close()


# ---- 7. restart files ----
def test_restart_with_rows(dfb, W, tmp_path):
    pl = profile(W)
    rows = band_rows(pl, 128)
    ref = make(dfb, pl)
    ref.set_time_scales(rows)
    for dt in DTS:
        ref.filter(dt)
    slabs = [make(dfb, pl, k_begin=0, k_end=112), make(dfb, pl, k_begin=112, k_end=256)]
    for s in slabs:
        s.set_time_scales(rows)
    for dt in DTS[:10]:
        for s in slabs:
            s.filter(dt)
    path = str(tmp_path / "rows.rst")
    for s in slabs:
        s.save_restart(path)
    # refused: no rows, other rows; the handle is unchanged
    for other in (None, rows * 1.5):
        h = make(dfb, pl)
        if other is not None:
            h.set_time_scales(other)
        before = snapshot(h), h.step
        with pytest.raises(dfb.DfbError) as e:
            h.load_restart(path)
        assert e.value.code == dfb.ERR_ARG and "filter tables differ" in str(e.value)
        assert np.array_equal(snapshot(h), before[0]) and h.step == before[1]
        h.close()
    whole = make(dfb, pl)
    whole.set_time_scales(rows)
    whole.load_restart(path)
    for dt in DTS[10:]:
        whole.filter(dt)
    assert np.array_equal(snapshot(whole), snapshot(ref))
    # and back: the whole plane saves, slabs resume
    path2 = str(tmp_path / "rows2.rst")
    w2 = make(dfb, pl)
    w2.set_time_scales(rows)
    for dt in DTS[:10]:
        w2.filter(dt)
    w2.save_restart(path2)
    for s in slabs:
        s.load_restart(path2)
        for dt in DTS[10:]:
            s.filter(dt)
    assert np.array_equal(np.concatenate([snapshot(s) for s in slabs], axis=2), snapshot(ref))
    for d in [ref, whole, w2] + slabs:
        d.close()


# ---- 8. refusals ----
def test_refusals_leave_the_handle_unchanged(dfb, W):
    pl = profile(W)
    h, ctl = make(dfb, pl), make(dfb, pl)
    good = band_rows(pl, h.Ny)
    L = dfb.lib()
    for bad_value in (np.nan, 0.0, -1e-5):
        bad = good.copy()
        bad[2, 17] = bad_value
        with pytest.raises(dfb.DfbError) as e:
            h.set_time_scales(bad)
        assert e.value.code == dfb.ERR_ARG and "field 2 (w), row 17" in str(e.value)
    assert h.info(15) == 0
    Ny, Nz = h.Ny, h.Nz
    buf = [np.zeros((Ny, Nz)) for _ in range(5)]
    assert L.dfb_filter_to_host_begin(h._h, 1e-8, *[C.c_void_p(b.ctypes.data) for b in buf]) == 0
    ctl.filter(1e-8)
    assert L.dfb_set_time_scales(h._h, good.ctypes.data_as(C.POINTER(C.c_double))) == dfb.ERR_STATE
    assert L.dfb_filter_to_host_end(h._h) == 0
    out = np.zeros(Ny)
    assert L.dfb_get_table(h._h, 14, 3, out.ctypes.data_as(C.POINTER(C.c_double)), Ny) == dfb.ERR_ARG
    assert L.dfb_get_table(h._h, 14, -1, out.ctypes.data_as(C.POINTER(C.c_double)), Ny) == dfb.ERR_ARG
    assert L.dfb_get_table(h._h, 15, 0, out.ctypes.data_as(C.POINTER(C.c_double)), Ny) == dfb.ERR_ARG
    v = C.c_int64()
    assert L.dfb_info(h._h, 16, 0, C.byref(v)) == dfb.ERR_ARG
    assert h.info(15) == 0
    for dt in DTS:
        h.filter(dt)
        ctl.filter(dt)
    assert np.array_equal(snapshot(h), snapshot(ctl))
    h.close()
    ctl.close()


# ---- facades: the C++ class and the Fortran module's by-reference entry points ----
LIBDIR = os.path.join(ROOT, "digital-filtering_b200", "lib")
CUDA = "/usr/local/cuda"


@pytest.fixture(scope="module")
def facade_bin(dfb, tmp_path_factory):
    out = str(tmp_path_factory.mktemp("time_scales_facades"))
    common = ["-I" + os.path.join(ROOT, "include"), "-I" + CUDA + "/include", "-L" + LIBDIR, "-ldfb200", "-Wl,-rpath," + LIBDIR,
              "-L" + CUDA + "/lib64", "-lcudart", "-Wl,-rpath," + CUDA + "/lib64"]
    for cc, std, src, exe in (("/usr/bin/g++", "-std=c++17", "time_scales_cpp_test.cpp", "time_scales_cpp_test"),
                              ("/usr/bin/gcc", "-std=c11", "fortran_time_scales_mimic.c", "fortran_time_scales_mimic")):
        r = subprocess.run([cc, std, "-Wall", os.path.join(ROOT, "tests", src)] + common + ["-lm", "-o", os.path.join(out, exe)],
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    return out


@pytest.mark.parametrize("exe", ["time_scales_cpp_test", "fortran_time_scales_mimic"])
def test_facades(facade_bin, default_data, exe):
    r = subprocess.run([os.path.join(facade_bin, exe), str(default_data / "files" / "RST.dat"), str(default_data / "line.dat")],
                       cwd=default_data / "run", capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "TIME_SCALES_OK" in r.stdout, (r.returncode, r.stdout, r.stderr)
