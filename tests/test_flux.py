"""The inflow mass-flux correction (dfb_set_flux_correction) on the GPU.  Against a twin handle with the correction off (same seed, 30
steps of changing dt) on every kernel form, periodic planes, a batch, the Gaussian shape and per-row time scales: filt_old, v' and w' are
the twin's bit for bit, u' is fma(-c, sqrt(R11), u'_twin) with the reported c, T' and rho' are the rebuild from that u', c is m' / D to
rounding, and the delivered first-order flux is zero to rounding.  Also: the oracle plus a numpy restatement at the 1e-12 gate, batches
against single planes, repeated runs, graph replays and attached steps, void steps, switching off, restart files across modes, N2 and
correlation statistics of the delivered fields, refusals, and the C++ and Fortran-mimic facades."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, normwise_close
from oracle_harness import Model, np_sums
from test_flux_host import flux_shim

pytestmark = pytest.mark.gpu

K = 30
DTS = [1e-8 * (1 + k % 7) for k in range(K)]
D_ = C.POINTER(C.c_double)
WORST = {}


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    return flux_shim(tmp_path_factory)


def profile(W):
    return W.plane_profile(128, 256, 24, 16)


def make(dfb, pl, nplanes=1, seed=91, **kw):
    return dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(pl, seed=seed, device=0, **kw), fetch=False, nplanes=nplanes)


def fma(shim, a, b, c):
    a, b, c = (np.ascontiguousarray(np.broadcast_to(x, np.shape(c)), dtype=np.float64) for x in (a, b, c))
    out = np.zeros_like(c)
    shim.fx_fma(c.size, a.ctypes.data_as(D_), b.ctypes.data_as(D_), c.ctypes.data_as(D_), out.ctypes.data_as(D_))
    return out


class Geometry:
    """what the definition reads, from the handle's own tables: A = hy hz, g per mode, sqrt(R11) and the epilogue's T', rho' factors"""

    def __init__(self, df, mode):
        R11, Us, Ts, rhos, Ms = (df.table(i) for i in (0, 4, 5, 6, 7))
        self.hy, self.hz = np.diff(df.table(12, n=df.Ny + 1)), np.diff(df.table(13, n=df.Nz + 1))
        self.g = rhos * (1.0 + 0.2 * Ms * Ms) if mode == 1 else np.ones(df.Ny)
        self.rc0 = np.sqrt(R11)
        self.rc4 = -0.5 * (1.4 - 1) * Ms * Ms / Us                 # stepplan.cpp, the same expression
        self.Ts, self.rhos = Ts, rhos
        self.w = (self.hy * self.g)[:, None] * self.hz[None, :]     # A g per cell
        self.D = float((self.w.astype(np.longdouble) * self.rc0[:, None]).sum())

    def flux(self, u):
        return float((self.w.astype(np.longdouble) * u).sum()), float((self.w * np.abs(u)).sum())

    def rebuild(self, u):
        t2 = self.rc4[:, None] * u
        return t2 * self.Ts[:, None], -t2 * self.rhos[:, None]


def fields(df, p):
    return [df.get(w, plane=p) for w in range(8)]


def check_against_twin(shim, df, twin, G, where):
    """one step's checks of every plane; returns the worst |c - c_ext| D / sum A g |u'| and delivered flux / sum A g |u'|"""
    wc = wf = 0.0
    for p in range(df.nplanes):
        a, b = fields(df, p), fields(twin, p)
        for w in (1, 2, 5, 6, 7):                                   # v', w', filt_old: untouched
            assert np.array_equal(a[w], b[w]), (where, p, w)
        c, m, mean = df.flux_info(p)
        u = fma(shim, -c, G.rc0[:, None], b[0])
        assert np.array_equal(a[0], u), (where, p)
        T, rho = G.rebuild(u)
        assert np.array_equal(a[3], T) and np.array_equal(a[4], rho), (where, p)
        m_ext, s_abs = G.flux(b[0])
        assert abs(m - m_ext) <= 1e-13 * s_abs, (where, p, m, m_ext)
        r = abs(c - m_ext / G.D) * G.D / s_abs
        assert r <= 1e-13, (where, p, r)
        fl, s_new = G.flux(a[0])
        assert abs(fl) <= 1e-12 * s_new, (where, p, fl, s_new)
        wc, wf = max(wc, r), max(wf, abs(fl) / s_new)
        assert mean > 0
    return wc, wf


FORMS = {"default": ({}, {}), "y_dense": ({"DFB_Y_MODE": "0"}, {}), "y_chunk_rec": ({"DFB_Y_MODE": "1"}, {}),
         "y_run": ({"DFB_Y_MODE": "2"}, {}), "z_direct": ({"DFB_Z_MODE": "0"}, {}), "simple": ({}, dict(kernel_variant=1)),
         "periodic": ({}, dict(periodic_z=1)), "batch3": ({}, dict(nplanes=3)), "gaussian": ({}, dict(filter_shape=1)),
         "time_rows": ({}, {})}


@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("name", list(FORMS))
def test_against_twin(dfb, W, shim, monkeypatch, name, mode):
    env, kw = FORMS[name]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    kw = dict(kw)
    nplanes = kw.pop("nplanes", 1)
    pl = profile(W)
    df, twin = make(dfb, pl, nplanes, **kw), make(dfb, pl, nplanes, **kw)
    if name == "time_rows":
        rows = np.asarray(pl["scales"], dtype=np.float64)[:, 2][:, None] * np.linspace(0.2, 1.5, df.Ny)[None, :]
        df.set_time_scales(rows)
        twin.set_time_scales(rows)
    assert df.flux_correction == dfb.FLUX_OFF
    df.set_flux_correction(mode)
    assert df.flux_correction == mode and twin.flux_correction == dfb.FLUX_OFF
    G = Geometry(df, mode)
    worst = (0.0, 0.0)
    for s, dt in enumerate(DTS):
        df.filter(dt)
        twin.filter(dt)
        r = check_against_twin(shim, df, twin, G, (name, s))
        worst = tuple(max(x, y) for x, y in zip(worst, r))
    WORST[(name, mode)] = worst
    print("flux %s mode %d: worst |c - m'/D| D / sum A g |u'| %.2e, delivered flux / sum A g |u'| %.2e" % (name, mode, *worst))
    df.close()
    twin.close()


# ---- the oracle and a numpy restatement of the correction ----
def corrected(m, G, p):
    u = m.out[p, 0]
    c = float((G.w * u).sum()) / G.D
    u = u - c * G.rc0[:, None]
    T, rho = G.rebuild(u)
    return [u, m.out[p, 1], m.out[p, 2], T, rho]


@pytest.mark.parametrize("wname,steps", [("512x512_N32", 4), ("1024x2048_profile_N128", 2)])
def test_against_oracle(dfb, W, O, wname, steps):
    pl = W.NAMED[wname]()
    O.half_widths(pl)
    df = make(dfb, pl, seed=7)
    df.set_flux_correction(dfb.FLUX_MASS)
    G = Geometry(df, 1)
    m = Model(O, pl, 7, 0)
    m.first_step()
    worst = 0.0
    for s in range(steps):
        dt = 2e-7 * (1 + s)
        df.filter(dt)
        m.filter(dt)
        ref = corrected(m, G, 0)
        for w in range(5):
            ok, r = normwise_close(df.get(w), ref[w])
            worst = max(worst, r)
            assert ok, (wname, s, w, r)
        for f in range(3):
            assert normwise_close(df.get(5 + f), m.fo[0, f])[0]
    print(wname, "flux-corrected outputs against the oracle: worst normwise ratio %.2e" % worst)
    df.close()


# ---- reproducibility ----
def snapshot(df):
    return np.stack([df.get(w, plane=p) for p in range(df.nplanes) for w in range(8)])


def test_batch_planes_equal_single_planes(dfb, W, monkeypatch):
    monkeypatch.setenv("DFB_Y_MODE", "2")                         # one y-sweep form for the batch and the single planes
    pl = profile(W)
    batch = make(dfb, pl, 3)
    singles = [make(dfb, pl, plane_id=p) for p in range(3)]
    assert batch.info(10) == singles[0].info(10) == 2
    for d in [batch] + singles:
        d.set_flux_correction(dfb.FLUX_MASS)
    for dt in DTS[:10]:
        for d in [batch] + singles:
            d.filter(dt)
    for p in range(3):
        for w in range(8):
            assert np.array_equal(batch.get(w, plane=p), singles[p].get(w)), (p, w)
        assert batch.flux_info(p) == singles[p].flux_info(0)
    for d in [batch] + singles:
        d.close()


def test_repeated_runs_are_bitwise(dfb, W):
    pl = profile(W)
    out = []
    for _ in range(2):
        d = make(dfb, pl, 2)
        d.set_flux_correction(dfb.FLUX_VOLUME)
        for dt in DTS[:12]:
            d.filter(dt)
        out.append((snapshot(d), d.flux_info(0), d.flux_info(1)))
        d.close()
    assert np.array_equal(out[0][0], out[1][0]) and out[0][1:] == out[1][1:]


@pytest.mark.parametrize("kw", [{}, dict(kernel_variant=1), dict(nplanes=2)])
def test_graph_replays_and_attached_steps(dfb, W, kw):
    import torch
    kw = dict(kw)
    nplanes = kw.pop("nplanes", 1)
    pl = profile(W)
    a, b, c, e = (make(dfb, pl, nplanes, **kw) for _ in range(4))
    for d in (a, b, c, e):
        d.set_flux_correction(dfb.FLUX_MASS)
    s = torch.cuda.Stream()
    dt_a = torch.zeros(1, dtype=torch.float64, device="cuda")
    dt_b = torch.zeros(1, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    for d in (a, b, e):
        d.attach_stream(s)
    with pytest.raises(dfb.DfbError) as err:
        a.set_flux_correction(dfb.FLUX_OFF)
    assert err.value.code == dfb.ERR_STATE and a.flux_correction == dfb.FLUX_MASS
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        a.filter_dev(dt_a)
    with torch.cuda.stream(s):
        for dt in DTS:
            dt_a.fill_(dt)
            g.replay()
            dt_b.fill_(dt)
            b.filter_dev(dt_b)
            e.filter(dt)                                        # attached, host dt
    for dt in DTS:
        c.filter(dt)
    s.synchronize()
    assert np.array_equal(snapshot(a), snapshot(b))             # graph replays = eager attached steps
    assert np.array_equal(snapshot(e), snapshot(c))             # attached with a host dt = host-driven
    for p in range(nplanes):
        assert a.flux_info(p) == b.flux_info(p) and e.flux_info(p) == c.flux_info(p)
    for x, y in zip(snapshot(b), snapshot(c)):
        assert normwise_close(x, y, 1e-14)[0]
    for d in (a, b, e):
        d.attach_stream(None)
    del g
    for d in (a, b, c, e):
        d.close()


def test_void_step_changes_nothing(dfb, W):
    import torch
    pl = profile(W)
    a = make(dfb, pl)
    a.set_flux_correction(dfb.FLUX_MASS)
    for dt in DTS[:3]:
        a.filter(dt)
    s = torch.cuda.Stream()
    torch.cuda.synchronize()
    a.attach_stream(s)
    before, info = snapshot(a), a.flux_info(0)
    bad = torch.full((1,), float("nan"), dtype=torch.float64, device="cuda")
    a.filter_dev(bad)
    with pytest.raises(dfb.DfbError) as e:
        a.sync()
    assert e.value.code == dfb.ERR_ARG
    assert np.array_equal(snapshot(a), before) and a.flux_info(0) == info
    a.attach_stream(None)
    a.close()


def test_switching_off_continues_like_never_on(dfb, W):
    pl = profile(W)
    a, b = make(dfb, pl), make(dfb, pl)
    a.set_flux_correction(dfb.FLUX_MASS)
    for dt in DTS[:10]:
        a.filter(dt)
        b.filter(dt)
    info = a.flux_info(0)
    a.set_flux_correction(dfb.FLUX_OFF)
    assert a.flux_correction == dfb.FLUX_OFF
    for dt in DTS[10:20]:
        a.filter(dt)
        b.filter(dt)
        assert np.array_equal(snapshot(a), snapshot(b))
    assert a.flux_info(0) == info                                 # the last corrected step's
    a.close()
    b.close()


def test_restart_across_modes(dfb, W, tmp_path):
    pl = profile(W)
    a = make(dfb, pl)
    a.set_flux_correction(dfb.FLUX_MASS)
    for dt in DTS[:8]:
        a.filter(dt)
    path = str(tmp_path / "flux.rst")
    a.save_restart(path)
    ref = make(dfb, pl)                                           # never corrected, same steps
    for dt in DTS[:8]:
        ref.filter(dt)
    ref_path = str(tmp_path / "plain.rst")
    ref.save_restart(ref_path)
    assert open(path, "rb").read() == open(ref_path, "rb").read()     # header, fingerprint and state alike
    off, vol = make(dfb, pl), make(dfb, pl)
    off.load_restart(path)
    vol.set_flux_correction(dfb.FLUX_VOLUME)
    vol.load_restart(ref_path)
    for dt in DTS[8:14]:
        for d in (a, ref, off, vol):
            d.filter(dt)
    assert np.array_equal(snapshot(off), snapshot(ref))
    sa, sv = snapshot(a), snapshot(vol)
    assert np.array_equal(sa[[1, 2, 5, 6, 7]], sv[[1, 2, 5, 6, 7]]) and not np.array_equal(sa[0], sv[0])
    for d in (a, ref, off, vol):
        d.close()


# ---- statistics of the delivered fields ----
@pytest.mark.parametrize("kw", [{}, dict(kernel_variant=1)])
def test_n2_of_delivered_fields(dfb, W, kw):
    pl = profile(W)
    a = make(dfb, pl, **kw)
    a.set_flux_correction(dfb.FLUX_MASS)
    a.stats_enable(True)
    sums = np.zeros((6, a.Ny, a.Nz))
    for dt in DTS[:10]:
        a.filter(dt)
        f = [a.get(w) for w in range(5)]
        for i in range(5):
            sums[i] = sums[i] + f[i] * f[i]                          # mul then add, like the library
        sums[5] = sums[5] + f[0] * f[1]
    for i in range(6):
        got, n = a.stats(i)
        assert n == 10 and np.array_equal(got, sums[i]), i
    a.close()


def test_correlation_of_delivered_fields(dfb, W):
    pl = profile(W)
    a = make(dfb, pl)
    a.set_flux_correction(dfb.FLUX_MASS)
    a.corr_enable(z=8, y=4, t=0)
    steps = [[], [], []]
    for dt in DTS[:8]:
        a.filter(dt)
        for f in range(3):
            steps[f].append(a.get(f))
    for f in range(3):
        ref = np_sums(steps[f], (8, 4, 0))
        for d in (0, 1):
            S, pairs, n = a.corr(f, d, normalized=False)
            assert n == 8 and np.array_equal(pairs, ref[d][1])
            assert normwise_close(S, ref[d][0], 1e-12)[0], (f, d)
    a.close()


# ---- refusals ----
def test_refusals(dfb, W):
    import torch
    L = dfb.lib()
    pl = profile(W)
    a = make(dfb, pl)
    with pytest.raises(dfb.DfbError) as e:
        a.flux_info(0)
    assert e.value.code == dfb.ERR_STATE and "never enabled" in str(e.value)
    for bad in (-1, 3):
        with pytest.raises(dfb.DfbError) as e:
            a.set_flux_correction(bad)
        assert e.value.code == dfb.ERR_ARG and "unknown flux correction mode" in str(e.value)
    assert a.flux_correction == dfb.FLUX_OFF
    slab = make(dfb, pl, k_begin=0, k_end=128)
    with pytest.raises(dfb.DfbError) as e:
        slab.set_flux_correction(dfb.FLUX_MASS)
    assert e.value.code == dfb.ERR_ARG and "whole plane" in str(e.value) and slab.flux_correction == dfb.FLUX_OFF
    slab.set_flux_correction(dfb.FLUX_OFF)
    a.set_flux_correction(dfb.FLUX_VOLUME)
    with pytest.raises(dfb.DfbError) as e:
        a.flux_info(1)
    assert e.value.code == dfb.ERR_ARG
    bufs = np.zeros((5, a.Ny, a.Nz))
    assert L.dfb_filter_to_host_begin(a._h, 1e-8, *[C.c_void_p(bufs[i].ctypes.data) for i in range(5)]) == 0
    with pytest.raises(dfb.DfbError) as e:
        a.set_flux_correction(dfb.FLUX_MASS)
    assert e.value.code == dfb.ERR_STATE
    assert L.dfb_filter_to_host_end(a._h) == 0
    assert a.flux_correction == dfb.FLUX_VOLUME
    s = torch.cuda.Stream()
    torch.cuda.synchronize()
    a.attach_stream(s)
    with pytest.raises(dfb.DfbError) as e:
        a.set_flux_correction(dfb.FLUX_OFF)
    assert e.value.code == dfb.ERR_STATE and "attached" in str(e.value)
    a.attach_stream(None)
    assert a.flux_correction == dfb.FLUX_VOLUME
    a.close()
    slab.close()


def test_worst_values(capsys):
    """the worst values of the twin checks of this run (printed; the gates are asserted step by step above)"""
    if WORST:
        with capsys.disabled():
            wc = max(v[0] for v in WORST.values())
            wf = max(v[1] for v in WORST.values())
            print("\nflux correction, all forms: worst |c - m'/D| D / sum A g |u'| = %.2e, worst delivered |sum A g u'| / sum A g |u'| = %.2e"
                  % (wc, wf))


# ---- facades: the C++ class and the Fortran module's by-reference entry points ----
LIBDIR = os.path.join(ROOT, "digital-filtering_b200", "lib")
CUDA = "/usr/local/cuda"


@pytest.fixture(scope="module")
def facade_bin(dfb, tmp_path_factory):
    out = str(tmp_path_factory.mktemp("flux_facades"))
    common = ["-I" + os.path.join(ROOT, "include"), "-I" + CUDA + "/include", "-L" + LIBDIR, "-ldfb200", "-Wl,-rpath," + LIBDIR,
              "-L" + CUDA + "/lib64", "-lcudart", "-Wl,-rpath," + CUDA + "/lib64"]
    for cc, std, src, exe in (("/usr/bin/g++", "-std=c++17", "flux_cpp_test.cpp", "flux_cpp_test"),
                              ("/usr/bin/gcc", "-std=c11", "fortran_flux_mimic.c", "fortran_flux_mimic")):
        r = subprocess.run([cc, std, "-Wall", os.path.join(ROOT, "tests", src)] + common + ["-lm", "-o", os.path.join(out, exe)],
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    return out


@pytest.mark.parametrize("exe", ["flux_cpp_test", "fortran_flux_mimic"])
def test_facades(facade_bin, default_data, exe):
    r = subprocess.run([os.path.join(facade_bin, exe), str(default_data / "files" / "RST.dat"), str(default_data / "line.dat")],
                       cwd=default_data / "run", capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "FLUX_OK" in r.stdout, (r.returncode, r.stdout, r.stderr)
