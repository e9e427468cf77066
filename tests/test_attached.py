"""Handles attached to a caller's stream (dfb_attach_stream) with dt in device memory (dfb_filter_dev): a captured graph replays
exactly the eager steps, attached steps reproduce host-driven ones, one attached step matches the oracle, the state round-trips through
detach and restart files, void steps change nothing, and the calls attached handles cannot serve are refused."""
import math
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, normwise_close
from oracle_harness import Model, check

pytestmark = pytest.mark.gpu

LIBDIR = os.path.join(ROOT, "digital-filtering_b200", "lib")
K = 50
DTS = [0.0 if k % 5 == 3 else 1e-8 * (1 + k % 7) for k in range(K)]
FIELDS = (0, 1, 2, 3, 4, 5, 6, 7)          # u', v', w', T', rho', filt u, v, w


def torch_dev():
    import torch
    return torch, torch.device("cuda", 0)


def plane(W):
    return W.plane_profile(128, 256, 24, 16)


def make(dfb, W, nplanes=1, pl=None, **kw):
    return dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(pl or plane(W), seed=91, device=0, **kw), fetch=False, nplanes=nplanes)


def snapshot(df):
    return np.stack([df.get(w, plane=p) for p in range(df.nplanes) for w in FIELDS])


def faces(df, n=96):
    vy, vz = df.table(12, n=df.Ny + 1), df.table(13, n=df.Nz + 1)
    rng = np.random.default_rng(5)
    return df.facemap(rng.uniform(vy[0], vy[-1], n), rng.uniform(vz[0], vz[-1], n))


FORMS = {"default": ({}, {}), "y_dense": ({"DFB_Y_MODE": "0"}, {}), "y_chunk_rec": ({"DFB_Y_MODE": "1"}, {}),
         "y_run": ({"DFB_Y_MODE": "2"}, {}), "simple": ({}, dict(kernel_variant=1)), "periodic": ({}, dict(periodic_z=1)),
         "batch4": ({}, dict(nplanes=4))}


@pytest.mark.parametrize("form", list(FORMS))
def test_graph_replays_equal_eager_steps(dfb, W, monkeypatch, form):
    """One dfb_filter_dev + one dfb_interp_to_cells captured with torch.cuda.graph and replayed K times, dt rewritten in device memory
    between replays, against the same sequence run eagerly on a second handle: all fields, filt_old, the faces and the step counter
    bit for bit."""
    torch, dev = torch_dev()
    env, kw = FORMS[form]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    nplanes = kw.pop("nplanes", 1)
    a, b = make(dfb, W, nplanes, **kw), make(dfb, W, nplanes, **kw)
    ma, mb = faces(a), faces(b)
    s = torch.cuda.Stream()
    dt_a = torch.zeros(1, dtype=torch.float64, device=dev)
    dt_b = torch.zeros(1, dtype=torch.float64, device=dev)
    fa = [torch.zeros(ma.n, dtype=torch.float64, device=dev) for _ in range(5)]
    fb = [torch.zeros(mb.n, dtype=torch.float64, device=dev) for _ in range(5)]
    torch.cuda.synchronize()
    a.attach_stream(s)
    b.attach_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        a.filter_dev(dt_a)
        ma.to_cells(fa, plane=nplanes - 1)
    with torch.cuda.stream(s):
        for dt in DTS:
            dt_a.fill_(dt)
            g.replay()
            dt_b.fill_(dt)
            b.filter_dev(dt_b)
            mb.to_cells(fb, plane=nplanes - 1)
    s.synchronize()
    assert a.step == b.step == 1 + K
    assert np.array_equal(snapshot(a), snapshot(b))
    assert all(torch.equal(x, y) for x, y in zip(fa, fb)) and all(bool(x.abs().sum() > 0) for x in fa[:3])
    a.attach_stream(None)
    b.attach_stream(None)
    del g


def test_attached_steps_against_host_driven(dfb, W):
    """Attached dfb_filter(h, dt) reproduces an unattached handle bit for bit over K steps, noise included; dfb_filter_dev agrees with
    it to 1e-14 of the field rms, normwise, at every step, with bitwise equal noise."""
    torch, dev = torch_dev()
    host, att, devdt = make(dfb, W), make(dfb, W), make(dfb, W)
    s = torch.cuda.Stream()
    att.attach_stream(s)
    devdt.attach_stream(s)
    dt_t = torch.zeros(1, dtype=torch.float64, device=dev)
    worst = 0.0
    for k, dt in enumerate(DTS):
        host.filter(dt)
        att.filter(dt)
        with torch.cuda.stream(s):
            dt_t.fill_(dt)
        devdt.filter_dev(dt_t)
        ref = snapshot(host)
        assert np.array_equal(snapshot(att), ref), k
        got = snapshot(devdt)
        for i in range(len(ref)):
            ok, r = normwise_close(got[i], ref[i], 1e-14)
            assert ok, (k, i, r)
            worst = max(worst, r)
        for f in range(3):
            rh = host.get_noise(f)
            assert all(np.array_equal(x, y) for x, y in zip(att.get_noise(f), rh) if x is not None), (k, f)
            assert all(np.array_equal(x, y) for x, y in zip(devdt.get_noise(f), rh) if x is not None), (k, f)
    assert host.step == att.step == devdt.step == 1 + K
    print(f"dfb_filter_dev vs dfb_filter: worst normwise ratio {worst:.3e}")


@pytest.mark.parametrize("name", ["512x512_N32", "1024x2048_profile_N128", "1024x2048_saturated_N128"])
def test_one_attached_step_against_the_oracle(dfb, W, O, name):
    torch, dev = torch_dev()
    pl = O.half_widths(W.NAMED[name]())
    df = make(dfb, W, pl=pl)
    m = Model(O, pl, 91, 0)
    m.first_step()
    s = torch.cuda.Stream()
    df.attach_stream(s)
    dt = 3e-8
    df.filter_dev(torch.full((1,), dt, dtype=torch.float64, device=dev))
    m.filter(dt)
    worst = check(df, m)
    print(name, "worst normwise ratio against the oracle:", worst)
    df.attach_stream(None)


def test_round_trips(dfb, W, tmp_path):
    """attach -> K graph replays -> detach -> M host steps equals K + M host steps (N2 sums and count included); a restart file
    saved after the replays records the device step and the resumed run matches.  The graph holds a host-dt step (dfb_filter while
    attached), whose blend constants are the host's: bit for bit a host-driven step."""
    torch, dev = torch_dev()
    M, DT = 7, 2e-8
    ref, df = make(dfb, W), make(dfb, W)
    ref.stats_enable(True)
    df.stats_enable(True)
    for dt in [DT] * K + DTS[:M]:
        ref.filter(dt)
    s = torch.cuda.Stream()
    torch.cuda.synchronize()
    df.attach_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        df.filter(DT)
    with torch.cuda.stream(s):
        for _ in range(K):
            g.replay()
    s.synchronize()
    path = str(tmp_path / "attached.dfbr")
    df.save_restart(path, stats=True)
    assert dfb.restart_info(path)["step"] == 1 + K
    df.attach_stream(None)
    del g
    for dt in DTS[:M]:
        df.filter(dt)
    assert df.step == ref.step == 1 + K + M
    assert np.array_equal(snapshot(df), snapshot(ref))
    for w in range(6):
        (x, nx), (y, ny) = df.stats(w), ref.stats(w)
        assert nx == ny == K + M and np.array_equal(x, y), w
    resumed = make(dfb, W)
    resumed.load_restart(path, stats=True)
    resumed.attach_stream(s)
    for dt in DTS[:M]:
        resumed.filter(dt)
    assert resumed.step == ref.step
    assert np.array_equal(snapshot(resumed), snapshot(ref))
    for w in range(6):
        (x, nx), (y, ny) = resumed.stats(w), ref.stats(w)
        assert nx == ny and np.array_equal(x, y), w
    resumed.attach_stream(None)


@pytest.mark.parametrize("bad", [math.nan, math.inf, -1e-8])
def test_void_steps_change_nothing(dfb, W, bad):
    torch, dev = torch_dev()
    ref, df = make(dfb, W), make(dfb, W)
    ref.stats_enable(True)
    df.stats_enable(True)
    s = torch.cuda.Stream()
    df.attach_stream(s)
    ref.attach_stream(s)                               # the same device-side blend constants: bitwise comparable
    dt_t = torch.zeros(1, dtype=torch.float64, device=dev)
    dt_r = torch.zeros(1, dtype=torch.float64, device=dev)
    seq = [1e-8, 2e-8, None, 3e-8, None, 1e-8]          # None: a void step
    for dt in seq:
        with torch.cuda.stream(s):
            dt_t.fill_(bad if dt is None else dt)
        df.filter_dev(dt_t)
        if dt is None:
            with pytest.raises(dfb.DfbError) as e:
                df.sync()
            assert e.value.code == dfb.ERR_ARG and "dt must be finite and >= 0" in str(e.value)
            df.sync()                                  # reported once
        else:
            with torch.cuda.stream(s):
                dt_r.fill_(dt)
            ref.filter_dev(dt_r)
        # fields, filt_old, N2 and the step as the reference's, after every step, void or not
        assert df.step == ref.step
        assert np.array_equal(snapshot(df), snapshot(ref))
        for w in range(6):
            (x, nx), (y, ny) = df.stats(w), ref.stats(w)
            assert nx == ny and np.array_equal(x, y), w
        for f in range(3):
            assert all(np.array_equal(x, y) for x, y in zip(df.get_noise(f), ref.get_noise(f)) if x is not None)
    # a void step that no call looked at is reported by the detach, which still detaches
    with torch.cuda.stream(s):
        dt_t.fill_(bad)
    df.filter_dev(dt_t)
    with pytest.raises(dfb.DfbError) as e:
        df.attach_stream(None)
    assert e.value.code == dfb.ERR_ARG
    with pytest.raises(dfb.DfbError) as e:
        df.filter_dev(dt_t)
    assert e.value.code == dfb.ERR_STATE                # detached
    ref.attach_stream(None)
    df.filter(2e-8)
    ref.filter(2e-8)
    assert np.array_equal(snapshot(df), snapshot(ref))


def test_refusals_change_nothing(dfb, W):
    import ctypes as C
    torch, dev = torch_dev()
    L = dfb.lib()
    df = make(dfb, W)
    s = torch.cuda.Stream()
    df.attach_stream(s)
    df.filter(1e-8)
    before, step = snapshot(df), df.step
    h = df._h
    out = np.zeros(5 * df.Ny * df.Nz)
    lags = (C.c_int * 3)(4, 4, 0)
    dts = np.full(2, 1e-8)
    calls = {
        "dfb_comm_init": lambda: L.dfb_comm_init(h, C.create_string_buffer(128), 0, 1),
        "dfb_corr_enable": lambda: L.dfb_corr_enable(h, 1, lags),
        "dfb_stats_enable": lambda: L.dfb_stats_enable(h, 1),
        "dfb_set_timing(h, 1)": lambda: L.dfb_set_timing(h, 1),
        "dfb_filter_to_host_begin": lambda: L.dfb_filter_to_host_begin(h, 1e-8, out.ctypes.data, None, None, None, None),
        "dfb_filter_to_host_end": lambda: L.dfb_filter_to_host_end(h),
        "dfb_filter_batch": lambda: L.dfb_filter_batch(h, 2, dts.ctypes.data_as(C.POINTER(C.c_double)), None),
        "dfb_generate_noise": lambda: L.dfb_generate_noise(h, 3),
        "dfb_get_rms": lambda: L.dfb_get_rms(h, 2, 1e-8),
    }
    for name, call in calls.items():
        assert call() == dfb.ERR_STATE, name
        assert name in L.dfb_last_error().decode(), (name, L.dfb_last_error())
    assert L.dfb_attach_stream(h, C.c_void_p(s.cuda_stream)) == dfb.ERR_STATE          # attached already
    assert L.dfb_set_timing(h, 0) == dfb.OK
    assert df.step == step and np.array_equal(snapshot(df), before)
    df.attach_stream(None)
    # what cannot be attached
    inj = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane(W), device=0, noise_mode=dfb.NOISE_INJECT), fetch=False)
    assert L.dfb_attach_stream(inj._h, C.c_void_p(s.cuda_stream)) == dfb.ERR_STATE
    df.corr_enable(z=4, y=4, t=0)
    assert L.dfb_attach_stream(h, C.c_void_p(s.cuda_stream)) == dfb.ERR_STATE
    df.corr_enable(on=False)
    df.set_timing(True)
    assert L.dfb_attach_stream(h, C.c_void_p(s.cuda_stream)) == dfb.ERR_STATE
    df.set_timing(False)
    assert L.dfb_filter_dev(h, C.c_void_p(1)) == dfb.ERR_STATE                          # not attached
    if torch.cuda.device_count() > 1:
        s1 = torch.cuda.Stream(device=1)
        assert L.dfb_attach_stream(h, C.c_void_p(s1.cuda_stream)) == dfb.ERR_ARG
    df.filter(1e-8)
    assert df.step == step + 1


@pytest.fixture(scope="module")
def capture_bin(dfb, tmp_path_factory):
    out = str(tmp_path_factory.mktemp("attached_capture_gpu"))
    exe = os.path.join(out, "attached_capture_test")
    subprocess.run(["/usr/bin/gcc", "-std=c11", "-Wall", os.path.join(ROOT, "tests", "attached_capture_test.c"),
                    "-I" + os.path.join(ROOT, "include"), "-I/usr/local/cuda/include", "-L" + LIBDIR, "-ldfb200",
                    "-Wl,-rpath," + LIBDIR, "-L/usr/local/cuda/lib64", "-lcudart", "-Wl,-rpath,/usr/local/cuda/lib64", "-o", exe],
                   check=True, capture_output=True)
    return exe


@pytest.mark.parametrize("mode", ["c", "fortran"])
def test_runtime_api_capture_program(capture_bin, default_data, mode):
    """the C program captures with cudaStreamBeginCapture (global mode) and replays against eager steps; mode fortran makes the attach
    and the steps through the by-reference entry points"""
    r = subprocess.run([capture_bin, str(default_data / "files" / "RST.dat"), str(default_data / "line.dat"), mode],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and f"CAPTURE_OK {K}" in r.stdout, (r.stdout, r.stderr)
