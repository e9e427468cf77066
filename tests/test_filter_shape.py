"""The Gaussian filter shape (dfb_set_filter_shape) on the GPU: the constructor's step and three filter(dt) steps against the numpy
restatement of the sweeps with the Gaussian table followed by the oracle's blend, Lund scaling and SRA (tests/shape_model.py), at the
field-wide and the per-row 1e-12 gates, on 512x512 (both lane blockings forced), the 1024x2048 profile, the reference's default plane,
the one-thread-per-cell kernels and a periodic plane; slabs, batches, graph replays and restart files bit for bit; the delivered
spanwise and wall-normal correlations and integral scales against the exact expectation of the Gaussian table; refusals; facades."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, default_plane
from shape_model import ShapeModel, gauss_coef
from test_correlation import PI_BLEND, expected_rho, sample_sigma
from test_random_planes import SEL, gate, magnitudes

pytestmark = pytest.mark.gpu

SEED, PLANE_ID = 57, 2
DTS = (2e-7, 4.5e-7, 1.2e-6)


class AbsShapeModel(ShapeModel):
    """ShapeModel on |noise|: every weight of the Gaussian chain is positive, so its filt is the sum of the magnitudes of the terms"""

    def noise(self, p, f, step):
        rys, hal = ShapeModel.noise(self, p, f, step)
        return np.abs(rys), None if hal is None else np.abs(hal)


def make(dfb, pl, **kw):
    nplanes = kw.pop("nplanes", 1)
    kw.setdefault("seed", SEED)
    kw.setdefault("plane_id", PLANE_ID)
    return dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(pl, device=0, filter_shape=dfb.FILTER_GAUSSIAN, **kw), fetch=False,
                              nplanes=nplanes)


def outputs(dfb, df, dts=DTS):
    """out[step][plane] = the 8 outputs after the constructor's step and each filter(dt)"""
    out = []
    for s in range(len(dts) + 1):
        if s:
            df.filter(dts[s - 1])
        out.append([[df.get(w, plane=p).copy() for w in SEL(dfb)] for p in range(df.nplanes)])
    return out


_refs = {}


def reference(O, name, pl, periodic=False):
    """the restatement's outputs and their term magnitudes for plane `name`, computed once"""
    key = (name, periodic)
    if key not in _refs:
        kw = dict(seed=SEED, plane_id=PLANE_ID, coef=gauss_coef, periodic=periodic)
        m, a = ShapeModel(O, pl, **kw), AbsShapeModel(O, pl, **kw)
        ref, mag = [], []
        for s in range(len(DTS) + 1):
            for x in (m, a):
                x.first_step() if s == 0 else x.filter(DTS[s - 1])
            ref.append([[m.out[0, i].copy() for i in range(5)] + [m.fo[0, f].copy() for f in range(3)]])
            mag.append([magnitudes(pl, *a.fo[0].copy(), s == 0)])
        _refs[key] = (ref, mag)
    return _refs[key]


def plane_named(O, W, name):
    if name == "default":
        return default_plane()
    pl = W.NAMED[name]()
    O.half_widths(pl)
    return pl


# name, plane, environment, config fields
PARITY = [("512", "512x512_N32", {}, {}), ("512_zk8", "512x512_N32", {"DFB_ZK": "8"}, {}), ("512_zk16", "512x512_N32", {"DFB_ZK": "16"}, {}),
          ("512_variant", "512x512_N32", {}, dict(kernel_variant=1)), ("512_periodic", "512x512_N32", {}, dict(periodic_z=1)),
          ("1024x2048", "1024x2048_profile_N128", {}, {}), ("1024x2048_variant", "1024x2048_profile_N128", {}, dict(kernel_variant=1)),
          ("default", "default", {}, {}), ("default_variant", "default", {}, dict(kernel_variant=1))]
_tuned_out = {}


@pytest.mark.parametrize("name,wname,env,kw", PARITY, ids=[p[0] for p in PARITY])
def test_parity_with_the_restatement(dfb, O, W, monkeypatch, name, wname, env, kw):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    pl = plane_named(O, W, wname)
    ref, mag = reference(O, wname, pl, periodic=bool(kw.get("periodic_z")))
    df = make(dfb, pl, **kw)
    assert df.filter_shape == dfb.FILTER_GAUSSIAN and df.step == 1
    info = (df.info(3), df.info(7), df.info(8), df.info(10), df.info(11))
    if kw.get("kernel_variant"):
        assert info[0] == 0
    else:
        assert info == (1, 0, 0, 0, 0), info                      # tuned: direct z form, dense band matrices only
    for N in np.unique(np.concatenate([np.ravel(pl["N_y"]), np.ravel(pl["N_z"])])):
        assert np.max(np.abs(df.table(11, int(N)) - gauss_coef(int(N)))) <= 1e-15, N
    out = outputs(dfb, df)
    worst = {}
    gate(out, ref, mag, name, worst)
    print(f"filter shape parity {name}: dfb_info 3/7/8/10/11 = {info}, worst field-wide "
          f"{max(w[0] for w in worst.values()):.2e} per-row {max(w[1] for w in worst.values()):.2e}")
    if not env and not kw.get("periodic_z"):
        base = wname
        _tuned_out.setdefault(base, {})["variant" if kw.get("kernel_variant") else "tuned"] = out
        both = _tuned_out[base]
        if len(both) == 2:                                         # tuned and one-thread-per-cell kernels on the same noise
            gate(both["tuned"], both["variant"], mag, f"{base}: tuned against kernel_variant 1", {})
    df.close()


def profile(W):
    return W.plane_profile(128, 256, 24, 16)


def snapshot(dfb, df):
    return np.stack([df.get(w, plane=p) for p in range(df.nplanes) for w in SEL(dfb)])


def test_slabs_equal_the_whole_plane(dfb, W):
    pl = profile(W)
    whole = make(dfb, pl)
    slabs = [make(dfb, pl, k_begin=a, k_end=b) for a, b in ((0, 64), (64, 160), (160, 256))]
    for dt in DTS:
        for d in [whole] + slabs:
            d.filter(dt)
    assert np.array_equal(np.concatenate([snapshot(dfb, s) for s in slabs], axis=2), snapshot(dfb, whole))
    for d in [whole] + slabs:
        d.close()


def test_batch_equals_single_planes(dfb, W):
    pl = profile(W)
    batch = make(dfb, pl, nplanes=3)
    assert batch.filter_shape == dfb.FILTER_GAUSSIAN and batch.info(10) == 0
    singles = [make(dfb, pl, plane_id=PLANE_ID + p) for p in range(3)]
    for dt in DTS:
        for d in [batch] + singles:
            d.filter(dt)
    got = snapshot(dfb, batch)
    for p, s in enumerate(singles):
        assert np.array_equal(got[8 * p:8 * (p + 1)], snapshot(dfb, s)), p
    for d in [batch] + singles:
        d.close()


def test_graph_replays_equal_eager_attached_steps(dfb, W):
    import torch
    pl = profile(W)
    a, b = make(dfb, pl), make(dfb, pl)
    s = torch.cuda.Stream()
    dt_a = torch.zeros(1, dtype=torch.float64, device="cuda")
    dt_b = torch.zeros(1, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    a.attach_stream(s)
    b.attach_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        a.filter_dev(dt_a)
    with torch.cuda.stream(s):
        for dt in DTS * 3:
            dt_a.fill_(dt)
            g.replay()
            dt_b.fill_(dt)
            b.filter_dev(dt_b)
    s.synchronize()
    assert np.array_equal(snapshot(dfb, a), snapshot(dfb, b)) and a.step == b.step == 1 + 3 * len(DTS)
    a.attach_stream(None)
    b.attach_stream(None)
    del g
    a.close()
    b.close()


def test_restart_round_trip_and_cross_shape_load(dfb, W, tmp_path):
    pl = profile(W)
    a = make(dfb, pl)
    for dt in DTS[:2]:
        a.filter(dt)
    path = str(tmp_path / "gauss.rst")
    a.save_restart(path)
    for dt in DTS:
        a.filter(dt)
    b = make(dfb, pl)
    b.load_restart(path)
    for dt in DTS:
        b.filter(dt)
    assert np.array_equal(snapshot(dfb, a), snapshot(dfb, b)) and a.step == b.step
    e = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(pl, device=0, seed=SEED, plane_id=PLANE_ID), fetch=False)
    with pytest.raises(dfb.DfbError) as err:
        e.load_restart(path)
    assert err.value.code == dfb.ERR_ARG and "filter shape differs: file Gaussian, handle exponential" in str(err.value)
    path_e = str(tmp_path / "exp.rst")
    e.save_restart(path_e)
    with pytest.raises(dfb.DfbError) as err:
        b.load_restart(path_e)
    assert err.value.code == dfb.ERR_ARG and "filter shape differs: file exponential, handle Gaussian" in str(err.value)
    assert dfb.restart_info(path)["fingerprint"] != dfb.restart_info(path_e)["fingerprint"]
    for d in (a, b, e):
        d.close()


def test_delivered_correlations_and_integral_scales(dfb, W):
    """a periodic row-uniform plane, 300 steps: the normalised z and y correlations at full support against the exact expectation of
    the Gaussian table, the median spanwise integral scale against n dz (n = N_z / 2), and an exponential control at ~0.64 of it"""
    plane = W.plane_profile(256, 1024, 16, 16)
    Lt_u = plane["scales"][0][2]
    dt = 2.0 * Lt_u * np.log(2.0) / PI_BLEND
    S = 300
    ratios = {}
    for shape in (dfb.FILTER_GAUSSIAN, dfb.FILTER_EXPONENTIAL):
        df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=2024, periodic_z=1, filter_shape=shape), fetch=False)
        df.corr_enable(dfb.DFB_CORR_SUPPORT, dfb.DFB_CORR_SUPPORT, 2)
        for _ in range(S):
            df.filter(dt)
        L = df.corr_lags
        Nyr = [df.half_widths(f, 0)[:, 0] for f in range(3)]
        Nzr = [df.half_widths(f, 1)[:, 0] for f in range(3)]
        vz = df.table(13, n=plane["Nz"] + 1)
        wbar = (vz[-1] - vz[0]) / plane["Nz"]
        if shape == dfb.FILTER_GAUSSIAN:
            Lt = df.table(10)
            alpha = [np.exp(-PI_BLEND * dt / Lt[f]) for f in range(3)]
            exp = expected_rho(gauss_coef, Nyr, Nzr, df.rows(), alpha, plane["Nz"], L)
            for f in range(3):
                sig = sample_sigma(exp[f, 0], exp[f, 2], plane["Nz"] * S)
                for d in (0, 1):
                    R = df.corr(f, d)[0]
                    E = exp[f, d]
                    assert np.array_equal(np.isnan(R), np.isnan(E)), (f, d)
                    err = np.nanmax(np.abs(R - E) / sig[:, None])
                    assert err < 6.0, (f, d, err)
                    print(f"Gaussian correlations: field {f} dir {d}: worst |R - E| = {err:.2f} sigma over lags 0..{L[d]}")
        for f in (0, 2):                                            # u' and w': one field's filter each
            n = Nzr[f] / 2.0
            I = df.integral_scales(f, dfb.CORR_Z)
            rows = n >= 4
            ratios[shape, f] = float(np.median(I[rows] / (n[rows] * wbar)))
        df.close()
    print("median spanwise integral scale / (n dz):", {k: round(v, 4) for k, v in ratios.items()})
    for f in (0, 2):
        assert abs(ratios[dfb.FILTER_GAUSSIAN, f] - 1.0) <= 0.03, ratios
        assert abs(ratios[dfb.FILTER_EXPONENTIAL, f] - 0.64) <= 0.04, ratios


def _status(fn, *a):
    try:
        fn(*a)
        return 0, ""
    except Exception as e:                                          # DfbError
        return e.code, str(e)


def test_refusals_leave_the_handle_unchanged(dfb, W, monkeypatch):
    import torch
    pl = profile(W)
    L = dfb.lib()
    base = dfb.DFConfig.from_plane(pl, device=0, seed=SEED)
    fresh = lambda **kw: dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(pl, device=0, seed=SEED, skip_first_step=1, **kw), fetch=False)
    # an unknown shape
    h = fresh()
    for bad in (-1, 2, 7):
        assert _status(h.set_filter_shape, bad)[0] == dfb.ERR_ARG
    # a handle that has stepped
    stepped = dfb.DIGITAL_FILTER(base, fetch=False)
    code, msg = _status(stepped.set_filter_shape, dfb.FILTER_GAUSSIAN)
    assert code == dfb.ERR_STATE and "has stepped" in msg, msg
    # N2, correlation statistics, time-scale rows, face maps, an outstanding _begin, attached, a communicator
    cases = {}
    a = fresh(); a.stats_enable(True); cases["N2 statistics are enabled"] = a
    b = fresh(); b.corr_enable(4, 4, 0); cases["correlation statistics are enabled"] = b
    c = fresh(); c.set_time_scales(np.full((3, c.Ny), 1e-6)); cases["per-row time scales are set"] = c
    d = fresh(); fm = d.facemap(np.array([1e-5]), np.array([1e-5])); cases["face maps"] = d
    for why, x in cases.items():
        code, msg = _status(x.set_filter_shape, dfb.FILTER_GAUSSIAN)
        assert code == dfb.ERR_STATE and why in msg, (why, msg)
        assert x.filter_shape == dfb.FILTER_EXPONENTIAL
    fm.close()
    assert _status(d.set_filter_shape, dfb.FILTER_GAUSSIAN)[0] == 0      # the map is gone: the handle takes the shape
    # a _begin outstanding on a handle whose counter was set back to 0
    g = fresh()
    buf = [np.zeros((g.Ny, g.Nz)) for _ in range(5)]
    assert L.dfb_filter_to_host_begin(g._h, 0.0, *[C.c_void_p(x.ctypes.data) for x in buf]) == 0
    g.set_state(None, 0)
    code, msg = _status(g.set_filter_shape, dfb.FILTER_GAUSSIAN)
    assert code == dfb.ERR_STATE and "dfb_filter_to_host_begin is outstanding" in msg, msg
    assert L.dfb_filter_to_host_end(g._h) == 0
    s = torch.cuda.Stream()
    at = fresh()
    at.attach_stream(s)
    code, msg = _status(at.set_filter_shape, dfb.FILTER_GAUSSIAN)
    assert code == dfb.ERR_STATE and "attached" in msg, msg
    at.attach_stream(None)
    cm = fresh()
    cm.comm_init(dfb.DIGITAL_FILTER.comm_unique_id(), 0, 1)
    code, msg = _status(cm.set_filter_shape, dfb.FILTER_GAUSSIAN)
    assert code == dfb.ERR_STATE and "communicator" in msg, msg
    # the planner's refusal of a recursive form forced by the environment leaves the exponential plan in place
    monkeypatch.setenv("DFB_Y_MODE", "2")
    r = fresh()
    y_form = r.info(10)
    code, msg = _status(r.set_filter_shape, dfb.FILTER_GAUSSIAN)
    assert code == dfb.ERR_ARG and "DFB_Y_MODE=2" in msg and "Gaussian" in msg, msg
    assert r.filter_shape == dfb.FILTER_EXPONENTIAL and r.info(10) == y_form == 2
    monkeypatch.delenv("DFB_Y_MODE")
    # every refused handle steps like a control that never saw the call
    ctl = dfb.DIGITAL_FILTER(base, fetch=False)
    for x in (h, r):
        x.first_step()
    for dt in DTS:
        for x in (h, r, ctl):
            x.filter(dt)
    for x in (h, r):
        assert np.array_equal(snapshot(dfb, x), snapshot(dfb, ctl))
    for x in [h, stepped, g, at, cm, r, ctl] + list(cases.values()):
        x.close()


def test_shape_switch_back_and_inject_mode(dfb, O, W):
    """setting the shape twice rebuilds the plan each time (Gaussian, exponential again: the exponential handle's bits); an inject-mode
    handle takes the shape before its first step and matches the restatement on the model's noise"""
    pl = profile(W)
    O.half_widths(pl)
    cfg = dict(device=0, seed=SEED, plane_id=PLANE_ID)
    x = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(pl, skip_first_step=1, **cfg), fetch=False)
    x.set_filter_shape(dfb.FILTER_GAUSSIAN)
    assert x.info(10) == 0 and x.info(7) == 0
    x.set_filter_shape(dfb.FILTER_EXPONENTIAL)
    ctl = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(pl, **cfg), fetch=False)
    assert tuple(x.info(i) for i in (3, 7, 8, 9, 10, 11)) == tuple(ctl.info(i) for i in (3, 7, 8, 9, 10, 11))
    x.first_step()
    for dt in DTS:
        x.filter(dt)
        ctl.filter(dt)
    assert np.array_equal(snapshot(dfb, x), snapshot(dfb, ctl))
    m = ShapeModel(O, pl, SEED, PLANE_ID, gauss_coef)
    inj = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(pl, noise_mode=dfb.NOISE_INJECT, filter_shape=dfb.FILTER_GAUSSIAN, **cfg), fetch=False)
    assert inj.step == 0 and inj.filter_shape == dfb.FILTER_GAUSSIAN
    from oracle_harness import run
    worst = run(inj, m, DTS)
    print("inject mode, Gaussian: worst", worst)
    for d in (x, ctl, inj):
        d.close()


# ---- facades: the C++ class and the Fortran module's by-reference entry points ----
LIBDIR = os.path.join(ROOT, "digital-filtering_b200", "lib")
CUDA = "/usr/local/cuda"


@pytest.fixture(scope="module")
def facade_bin(dfb, tmp_path_factory):
    out = str(tmp_path_factory.mktemp("filter_shape_facades"))
    common = ["-I" + os.path.join(ROOT, "include"), "-I" + CUDA + "/include", "-L" + LIBDIR, "-ldfb200", "-Wl,-rpath," + LIBDIR,
              "-L" + CUDA + "/lib64", "-lcudart", "-Wl,-rpath," + CUDA + "/lib64"]
    for cc, std, src, exe in (("/usr/bin/g++", "-std=c++17", "filter_shape_cpp_test.cpp", "filter_shape_cpp_test"),
                              ("/usr/bin/gcc", "-std=c11", "fortran_filter_shape_mimic.c", "fortran_filter_shape_mimic")):
        r = subprocess.run([cc, std, "-Wall", os.path.join(ROOT, "tests", src)] + common + ["-lm", "-o", os.path.join(out, exe)],
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    return out


@pytest.mark.parametrize("exe", ["filter_shape_cpp_test", "fortran_filter_shape_mimic"])
def test_facades(facade_bin, default_data, exe):
    r = subprocess.run([os.path.join(facade_bin, exe), str(default_data / "files" / "RST.dat"), str(default_data / "line.dat")],
                       cwd=default_data / "run", capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "FILTER_SHAPE_OK" in r.stdout, (r.returncode, r.stdout, r.stderr)
