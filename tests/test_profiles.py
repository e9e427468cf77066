"""Per-cell profiles (dfb_set_profiles) on the GPU, each check over 30 steps of changing dt.

Column bands: a handle whose profiles take row tables A, B and C on the column bands [0, a), [a, b) and [b, Nz) equals, bit for bit,
handles A, B and C (same seed and geometry, those rows) on their bands in u', v', w', T', rho' and the N2 sums, on every kernel form,
per-cell geometry, periodic planes, a batch, slabs, per-row time scales and the Gaussian shape; and filt_old equals a no-profile twin.
Also: profiles equal to the rows give the rows' bits, setting and clearing mid-run, attached steps and graph replays, the flux
correction with profiles, the oracle band by band at the 1e-12 gate, restart files, refusals and the C++ and Fortran-mimic facades."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import profiles_model as PM
from conftest import ROOT, normwise_close
from oracle_harness import Model
from test_flux_host import flux_shim

pytestmark = pytest.mark.gpu

K = 30
DTS = [1e-8 * (1 + k % 7) for k in range(K)]
D_ = C.POINTER(C.c_double)


def profile(W):
    return W.plane_profile(128, 256, 24, 16)


def with_rows(pl, rows):
    q = dict(pl)
    q["rows"] = np.asarray(rows, dtype=np.float64)
    return q


def make(dfb, pl, nplanes=1, seed=91, **kw):
    return dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(pl, seed=seed, device=0, **kw), fetch=False, nplanes=nplanes)


def snapshot(df):
    return np.stack([df.get(w, plane=p) for p in range(df.nplanes) for w in range(8)])


FORMS = {"default": ({}, {}), "y_dense": ({"DFB_Y_MODE": "0"}, {}), "y_chunk_rec": ({"DFB_Y_MODE": "1"}, {}),
         "y_run": ({"DFB_Y_MODE": "2"}, {}), "z_direct": ({"DFB_Z_MODE": "0"}, {}), "z_rec": ({"DFB_Z_MODE": "1"}, {}),
         "zk8": ({"DFB_ZK": "8"}, {}), "zk16": ({"DFB_ZK": "16"}, {}), "simple": ({}, dict(kernel_variant=1)),
         "per_cell_geometry": ({}, dict(ragged=True)), "periodic": ({}, dict(periodic_z=1)), "batch3": ({}, dict(nplanes=3)),
         "gaussian": ({}, dict(filter_shape=1)), "time_rows": ({}, dict(time_rows=True))}


def build_bands(dfb, W, kw):
    """(plane, profiles handle, [handles A, B, C], no-profile twin, band edges)"""
    kw = dict(kw)
    nplanes = kw.pop("nplanes", 1)
    ragged = kw.pop("ragged", False)
    time_rows = kw.pop("time_rows", False)
    pl = W.plane_ragged(64, 96, 8, seed=3) if ragged else profile(W)     # ragged: per-cell geometry (geom_per_row = 0)
    rows = PM.band_rows(pl)
    prof, twin = make(dfb, pl, nplanes, **kw), make(dfb, pl, nplanes, **kw)
    bands = [make(dfb, with_rows(pl, r), nplanes, **kw) for r in rows]
    Nz = prof.Nz
    prof.set_profiles(PM.band_cells(rows, Nz))
    if time_rows:
        Lt = np.asarray(pl["scales"], dtype=np.float64)[:, 2][:, None] * np.linspace(0.2, 1.5, prof.Ny)[None, :]
        for d in [prof, twin] + bands:
            d.set_time_scales(Lt)
    for d in [prof] + bands:
        d.stats_enable(True)
    return pl, prof, bands, twin, PM.band_edges(Nz)


def check_bands(prof, bands, twin, e, where):
    for p in range(prof.nplanes):
        got = [prof.get(w, plane=p) for w in range(8)]
        for i, b in enumerate(bands):
            for w in range(8):
                ref = b.get(w, plane=p)
                assert np.array_equal(got[w][:, e[i]:e[i + 1]], ref[:, e[i]:e[i + 1]]), (where, p, i, w)
        for w in (5, 6, 7):
            assert np.array_equal(got[w], twin.get(w, plane=p)), (where, p, "filt_old", w)


def check_stats(prof, bands, e):
    for p in range(prof.nplanes):
        for s in range(6):
            got, n = prof.stats(s, plane=p)
            assert n == K
            for i, b in enumerate(bands):
                ref, _ = b.stats(s, plane=p)
                assert np.array_equal(got[:, e[i]:e[i + 1]], ref[:, e[i]:e[i + 1]]), (p, s, i)


@pytest.mark.parametrize("name", list(FORMS))
def test_column_bands(dfb, W, monkeypatch, name):
    env, kw = FORMS[name]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    pl, prof, bands, twin, e = build_bands(dfb, W, kw)
    assert prof.info(19) == 1 and twin.info(19) == 0
    if name == "simple" or name == "per_cell_geometry":
        assert not prof.tuned
    if name.startswith("z") or name.startswith("y"):
        assert prof.tuned
    for s, dt in enumerate(DTS):
        for d in [prof, twin] + bands:
            d.filter(dt)
        check_bands(prof, bands, twin, e, (name, s))
    check_stats(prof, bands, e)
    for d in [prof, twin] + bands:
        d.close()


@pytest.mark.parametrize("slabs", [[(0, 64), (64, 144), (144, 256)], [(0, 128), (128, 256)]])
def test_slabs_equal_the_whole_plane(dfb, W, slabs):
    pl = profile(W)
    cells = PM.band_cells(PM.band_rows(pl), 256)
    whole = make(dfb, pl)
    whole.set_profiles(cells)
    parts = [make(dfb, pl, k_begin=a, k_end=b) for a, b in slabs]
    for (a, b), s in zip(slabs, parts):
        s.set_profiles(cells)
        assert np.array_equal(s.profiles, cells[:, :, a:b])
    for dt in DTS:
        whole.filter(dt)
        for s in parts:
            s.filter(dt)
        ref = snapshot(whole)
        for (a, b), s in zip(slabs, parts):
            assert np.array_equal(snapshot(s), ref[:, :, a:b]), (a, b)
    for d in [whole] + parts:
        d.close()


# ---- invariance ----
@pytest.mark.parametrize("kw", [{}, dict(kernel_variant=1), dict(nplanes=2)])
def test_broadcast_rows_equal_no_profiles(dfb, W, kw):
    kw = dict(kw)
    nplanes = kw.pop("nplanes", 1)
    pl = profile(W)
    a, b = make(dfb, pl, nplanes, **kw), make(dfb, pl, nplanes, **kw)
    a.set_profiles(PM.broadcast(a.rows(), a.Nz))
    assert np.array_equal(a.profiles, PM.broadcast(b.rows(), b.Nz))
    for d in (a, b):
        d.stats_enable(True)
    for dt in DTS:
        a.filter(dt)
        b.filter(dt)
        assert np.array_equal(snapshot(a), snapshot(b))
    for p in range(nplanes):
        for s in range(6):
            assert np.array_equal(a.stats(s, plane=p)[0], b.stats(s, plane=p)[0]), (p, s)
    a.close()
    b.close()


def test_set_and_clear_mid_run(dfb, W):
    pl = profile(W)
    a, b = make(dfb, pl), make(dfb, pl)
    cells = PM.band_cells(PM.band_rows(pl), a.Nz)
    assert a.profiles is None
    for s, dt in enumerate(DTS):
        if s == 5:
            a.set_profiles(cells)
        if s == 15:
            a.set_profiles(None)
            assert a.profiles is None and a.info(19) == 0
        a.filter(dt)
        b.filter(dt)
        x, y = snapshot(a), snapshot(b)
        assert np.array_equal(x[5:], y[5:]), s                    # filt_old never depends on the profiles
        if 5 <= s < 15:
            assert not np.array_equal(x[0], y[0])
        else:
            assert np.array_equal(x, y), s
    a.close()
    b.close()


def test_first_step_takes_the_profiles(dfb, W):
    pl = profile(W)
    rows = PM.band_rows(pl)
    a = make(dfb, pl, skip_first_step=1)
    a.set_profiles(PM.band_cells(rows, a.Nz))
    a.first_step()
    e = PM.band_edges(a.Nz)
    for i, r in enumerate(rows):
        b = make(dfb, with_rows(pl, r))
        for w in range(8):
            assert np.array_equal(a.get(w)[:, e[i]:e[i + 1]], b.get(w)[:, e[i]:e[i + 1]]), (i, w)
        b.close()
    assert not a.get(3).any() and not a.get(4).any()               # quirk 3: T', rho' untouched by the constructor's step
    a.close()


# ---- attached steps and graph replays ----
@pytest.mark.parametrize("kw", [{}, dict(kernel_variant=1), dict(nplanes=2)])
def test_graph_replays_and_attached_steps(dfb, W, kw):
    import torch
    kw = dict(kw)
    nplanes = kw.pop("nplanes", 1)
    pl = profile(W)
    cells = PM.band_cells(PM.band_rows(pl), 256)
    a, b, c, e = (make(dfb, pl, nplanes, **kw) for _ in range(4))
    for d in (a, b, c, e):
        d.set_profiles(cells)
        d.stats_enable(True)
    s = torch.cuda.Stream()
    dt_a = torch.zeros(1, dtype=torch.float64, device="cuda")
    dt_b = torch.zeros(1, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    for d in (a, b, e):
        d.attach_stream(s)
    with pytest.raises(dfb.DfbError) as err:
        a.set_profiles(None)
    assert err.value.code == dfb.ERR_STATE and "attached" in str(err.value) and a.info(19) == 1
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        a.filter_dev(dt_a)
    with torch.cuda.stream(s):
        for dt in DTS:
            dt_a.fill_(dt)
            g.replay()
            dt_b.fill_(dt)
            b.filter_dev(dt_b)
            e.filter(dt)
    for dt in DTS:
        c.filter(dt)
    s.synchronize()
    assert np.array_equal(snapshot(a), snapshot(b))             # graph replays = eager attached steps
    assert np.array_equal(snapshot(e), snapshot(c))             # attached with a host dt = host-driven
    for p in range(nplanes):
        for i in range(6):
            assert np.array_equal(a.stats(i, plane=p)[0], b.stats(i, plane=p)[0])
            assert np.array_equal(e.stats(i, plane=p)[0], c.stats(i, plane=p)[0])
    # a void step changes nothing
    before = snapshot(a)
    bad = torch.full((1,), float("nan"), dtype=torch.float64, device="cuda")
    a.filter_dev(bad)
    with pytest.raises(dfb.DfbError) as err:
        a.sync()
    assert err.value.code == dfb.ERR_ARG and np.array_equal(snapshot(a), before)
    for d in (a, b, e):
        d.attach_stream(None)
    del g
    for d in (a, b, c, e):
        d.close()


# ---- the flux correction with profiles ----
def fma(shim, a, b, c):
    a, b, c = (np.ascontiguousarray(np.broadcast_to(x, np.shape(c)), dtype=np.float64) for x in (a, b, c))
    out = np.zeros_like(c)
    shim.fx_fma(c.size, a.ctypes.data_as(D_), b.ctypes.data_as(D_), c.ctypes.data_as(D_), out.ctypes.data_as(D_))
    return out


@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("kw", [{}, dict(kernel_variant=1), dict(nplanes=3)])
def test_flux_correction(dfb, W, tmp_path_factory, kw, mode):
    shim = flux_shim(tmp_path_factory)
    kw = dict(kw)
    nplanes = kw.pop("nplanes", 1)
    pl = profile(W)
    cells = PM.band_cells(PM.band_rows(pl), 256)
    df, twin = make(dfb, pl, nplanes, **kw), make(dfb, pl, nplanes, **kw)
    df.set_flux_correction(mode)                                  # before the profiles: set_profiles rebuilds the tables
    for d in (df, twin):
        d.set_profiles(cells)
    R11, Us, Ts, rhos, Ms = cells[0], cells[4], cells[5], cells[6], cells[7]
    rc0, rc4 = np.sqrt(R11), -0.5 * (1.4 - 1) * Ms * Ms / Us
    hy, hz = np.diff(df.table(12, n=df.Ny + 1)), np.diff(df.table(13, n=df.Nz + 1))
    g = rhos * (1.0 + 0.2 * Ms * Ms) if mode == 1 else np.ones_like(R11)
    A = (hy[:, None] * hz[None, :] * g)
    Dx = float((A.astype(np.longdouble) * rc0).sum())
    worst = 0.0
    for s, dt in enumerate(DTS):
        df.filter(dt)
        twin.filter(dt)
        for p in range(nplanes):
            a = [df.get(w, plane=p) for w in range(8)]
            b = [twin.get(w, plane=p) for w in range(8)]
            for w in (1, 2, 5, 6, 7):
                assert np.array_equal(a[w], b[w]), (s, p, w)
            c, m, mean = df.flux_info(p)
            u = fma(shim, -c, rc0, b[0])
            assert np.array_equal(a[0], u), (s, p)
            t2 = rc4 * u
            assert np.array_equal(a[3], t2 * Ts) and np.array_equal(a[4], -t2 * rhos), (s, p)
            m_ext = float((A.astype(np.longdouble) * b[0]).sum())
            s_abs = float((A * np.abs(b[0])).sum())
            assert abs(c - m_ext / Dx) * Dx <= 1e-13 * s_abs, (s, p)
            fl = float((A.astype(np.longdouble) * a[0]).sum())
            assert abs(fl) <= 1e-12 * float((A * np.abs(a[0])).sum()), (s, p, fl)
            worst = max(worst, abs(fl) / float((A * np.abs(a[0])).sum()))
            assert mean == pytest.approx(float((hy[:, None] * hz[None, :] * (rhos * Us if mode == 1 else Us)).sum()), rel=1e-12)
    print("flux with profiles, mode %d %s: worst delivered flux / sum A g |u'| %.2e" % (mode, kw, worst))
    df.close()
    twin.close()


# ---- the oracle, band by band ----
def scaled(O, fo, rows, T_rho):
    """orc_rst_scaling and orc_sra of one band's filtered fields (fo: [3][Ny][n]) with the band's rows"""
    L, d = O.lib(), O._d
    Ny, n = fo.shape[1], fo.shape[2]
    filt = [np.ascontiguousarray(fo[f]) for f in range(3)]
    fluc, old = [np.zeros((Ny, n)) for _ in range(3)], [np.zeros((Ny, n)) for _ in range(3)]
    r = [np.ascontiguousarray(rows[k], dtype=np.float64) for k in range(8)]
    L.orc_rst_scaling(C.c_int(Ny), C.c_int(n), d(r[0]), d(r[1]), d(r[2]), d(r[3]), d(filt[0]), d(filt[1]), d(filt[2]),
                      d(fluc[0]), d(fluc[1]), d(fluc[2]), d(old[0]), d(old[1]), d(old[2]))
    T, rho = np.zeros((Ny, n)), np.zeros((Ny, n))
    L.orc_sra(C.c_int(Ny), C.c_int(n), d(r[7]), d(r[4]), d(r[5]), d(r[6]), d(fluc[0]), d(T), d(rho))
    return fluc + [T, rho]


@pytest.mark.parametrize("wname,steps", [("512x512_N32", 4), ("1024x2048_profile_N128", 2)])
def test_against_oracle(dfb, W, O, wname, steps):
    pl = W.NAMED[wname]()
    O.half_widths(pl)
    rows = PM.band_rows(pl)
    df = make(dfb, pl, seed=7)
    df.set_profiles(PM.band_cells(rows, df.Nz))
    m = Model(O, pl, 7, 0)
    m.first_step()
    e = PM.band_edges(df.Nz)
    worst = 0.0
    for s in range(steps):
        dt = 2e-7 * (1 + s)
        df.filter(dt)
        m.filter(dt)
        got = [df.get(w) for w in range(5)]
        for i, r in enumerate(rows):
            ref = scaled(O, m.fo[0][:, :, e[i]:e[i + 1]], r, True)
            for w in range(5):
                ok, ratio = normwise_close(np.ascontiguousarray(got[w][:, e[i]:e[i + 1]]), ref[w])
                worst = max(worst, ratio)
                assert ok, (wname, s, i, w, ratio)
        for f in range(3):
            assert normwise_close(df.get(5 + f), m.fo[0, f])[0]
    print("%s: per-cell profiles against the oracle band by band, worst normwise ratio %.2e" % (wname, worst))
    df.close()


# ---- restart files ----
def test_restart(dfb, W, tmp_path):
    pl = profile(W)
    cells = PM.band_cells(PM.band_rows(pl), 256)
    a = make(dfb, pl)
    a.set_profiles(cells)
    for dt in DTS[:8]:
        a.filter(dt)
    path = str(tmp_path / "prof.rst")
    a.save_restart(path)
    plain = make(dfb, pl)
    for dt in DTS[:8]:
        plain.filter(dt)
    plain_path = str(tmp_path / "plain.rst")
    plain.save_restart(plain_path)
    b = make(dfb, pl)
    b.set_profiles(cells)
    b.load_restart(path)
    slabs = [make(dfb, pl, k_begin=k, k_end=k + 128) for k in (0, 128)]
    for s in slabs:
        s.set_profiles(cells)
        s.load_restart(path)
    for dt in DTS[8:16]:
        for d in [a, b] + slabs:
            d.filter(dt)
    ref = snapshot(a)
    assert np.array_equal(snapshot(b), ref)
    for k, s in zip((0, 128), slabs):
        assert np.array_equal(snapshot(s), ref[:, :, k:k + 128])
    # refused loads, naming the reason; the handle is unchanged
    none, other = make(dfb, pl), make(dfb, pl)
    other_cells = cells.copy()
    other_cells[5, 3, 4] *= 1.0 + 1e-15
    other.set_profiles(other_cells)
    for d, p, why in ((none, path, "saved with per-cell profiles"), (other, path, "differ from the file's"),
                      (b, plain_path, "the file was saved without them")):
        before = snapshot(d)
        with pytest.raises(dfb.DfbError) as e:
            d.load_restart(p)
        assert e.value.code == dfb.ERR_ARG and why in str(e.value), str(e.value)
        assert np.array_equal(snapshot(d), before)
    for d in [a, b, plain, none, other] + slabs:
        d.close()


# ---- refusals ----
def test_refusals(dfb, W):
    import torch
    L = dfb.lib()
    pl = profile(W)
    a = make(dfb, pl)
    good = PM.band_cells(PM.band_rows(pl), a.Nz)
    for q, v, text in ((2, np.nan, "R22 at row 3, column 7 is not finite"), (0, -1.0, "R11 at row 3, column 7 gives sqrt(R11)"),
                       (2, 0.0, "R22 at row 3, column 7 gives sqrt(R22 - b^2)"), (4, 0.0, "Us at row 3, column 7 gives -0.2 Ms^2 / Us")):
        bad = good.copy()
        bad[q, 3, 7] = v
        with pytest.raises(dfb.DfbError) as e:
            a.set_profiles(bad)
        assert e.value.code == dfb.ERR_ARG and text in str(e.value), str(e.value)
        assert a.profiles is None
    with pytest.raises(ValueError):
        a.set_profiles(good[:, :, :-1])
    a.set_profiles(good)
    bufs = np.zeros((5, a.Ny, a.Nz))
    assert L.dfb_filter_to_host_begin(a._h, 1e-8, *[C.c_void_p(bufs[i].ctypes.data) for i in range(5)]) == 0
    with pytest.raises(dfb.DfbError) as e:
        a.set_profiles(None)
    assert e.value.code == dfb.ERR_STATE and "outstanding" in str(e.value)
    assert L.dfb_filter_to_host_end(a._h) == 0
    assert a.info(19) == 1
    # the gather's rebuild of T', rho' uses the row tables: dfb_comm_init refuses a handle with profiles before it reaches NCCL
    uid = (C.c_char * 128)()
    assert L.dfb_comm_init(a._h, uid, 0, 2) == dfb.ERR_STATE
    assert "per-cell profiles" in L.dfb_last_error().decode()
    # the flux correction refuses profiles that leave no sqrt(R11) anywhere
    f = make(dfb, pl)
    f.set_flux_correction(dfb.FLUX_VOLUME)
    zero = good.copy()
    zero[0] = zero[1] = 0.0
    with pytest.raises(dfb.DfbError) as e:
        f.set_profiles(zero)
    assert e.value.code == dfb.ERR_ARG and "R11 is zero on every cell" in str(e.value) and f.profiles is None
    # unknown selectors stay unknown; table 16 checks its quantity
    out = np.zeros(a.Ny * a.Nz)
    assert L.dfb_get_table(a._h, 16, 8, out.ctypes.data_as(D_), out.size) == dfb.ERR_ARG
    assert L.dfb_get_table(a._h, 15, 0, out.ctypes.data_as(D_), out.size) == dfb.ERR_ARG
    a.close()
    f.close()


# ---- facades: the C++ class and the Fortran module's by-reference entry points ----
LIBDIR = os.path.join(ROOT, "digital-filtering_b200", "lib")
CUDA = "/usr/local/cuda"


@pytest.fixture(scope="module")
def facade_bin(dfb, tmp_path_factory):
    out = str(tmp_path_factory.mktemp("profiles_facades"))
    common = ["-I" + os.path.join(ROOT, "include"), "-I" + CUDA + "/include", "-L" + LIBDIR, "-ldfb200", "-Wl,-rpath," + LIBDIR,
              "-L" + CUDA + "/lib64", "-lcudart", "-Wl,-rpath," + CUDA + "/lib64"]
    for cc, std, src, exe in (("/usr/bin/g++", "-std=c++17", "profiles_cpp_test.cpp", "profiles_cpp_test"),
                              ("/usr/bin/gcc", "-std=c11", "fortran_profiles_mimic.c", "fortran_profiles_mimic")):
        r = subprocess.run([cc, std, "-Wall", os.path.join(ROOT, "tests", src)] + common + ["-lm", "-o", os.path.join(out, exe)],
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    return out


@pytest.mark.parametrize("exe", ["profiles_cpp_test", "fortran_profiles_mimic"])
def test_facades(facade_bin, default_data, exe):
    r = subprocess.run([os.path.join(facade_bin, exe), str(default_data / "files" / "RST.dat"), str(default_data / "line.dat")],
                       cwd=default_data / "run", capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "PROFILES_OK" in r.stdout, (r.returncode, r.stdout, r.stderr)
