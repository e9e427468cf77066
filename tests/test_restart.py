"""Restart files on the GPU (dfb_save_restart / dfb_load_restart): a run that takes n steps, saves, is destroyed and is resumed by a
FRESH handle gives every output of the next n steps bit for bit as the uninterrupted run -- on the y-sweep's forms, periodic planes,
the one-thread-per-cell kernels and inject mode, with variable dt across the restart; across changes of decomposition (slabs <->
whole plane, batch <-> single planes, batch of 8 -> batches of 4); with the N2 and correlation statistics; and every refused load
leaves the handle as it was."""
import os

import numpy as np
import pytest

from conftest import default_plane, normwise_close

pytestmark = pytest.mark.gpu

N = 3                                                        # steps before and after the restart
DTS = [2e-7, 5e-8, 0.0, 1.3e-6, 3e-7, 7e-8]                  # variable dt, also across the restart


def outputs(dfb, df):
    """every output of the last step: u', v', w', T', rho', filt u v w of every plane, [P * 8][Ny][W]"""
    which = (dfb.U_FLUC, dfb.V_FLUC, dfb.W_FLUC, dfb.T_FLUC, dfb.RHO_FLUC, dfb.U_FILT, dfb.V_FILT, dfb.W_FILT)
    return np.stack([df.get(w, plane=p) for p in range(df.nplanes) for w in which])


def make(dfb, plane, nplanes=1, **kw):
    return dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, **kw), fetch=False, nplanes=nplanes)


def steps(dfb, df, dts, inject=None):
    out = []
    for s, dt in enumerate(dts):
        if inject is not None:
            inject(df, s)
        df.filter(dt)
        out.append(outputs(dfb, df))
    return out


def assert_same(got, ref, what):
    for s, (g, r) in enumerate(zip(got, ref)):
        assert g.shape == r.shape and np.array_equal(g, r), (what, s, float(np.max(np.abs(g - r))) if g.shape == r.shape else g.shape)


def _W():
    import _dfb_import  # noqa: F401
    from digital_filtering_b200 import workloads
    return workloads


CASES = {
    "small": (lambda: _W().plane_profile(96, 160, 24, 10), {}),
    "1024x2048_profile": (lambda: _W().NAMED["1024x2048_profile_N128"](), {}),
    "default_plane": (default_plane, {}),
    "periodic_z": (lambda: _W().plane_profile(96, 160, 24, 10), {"periodic_z": 1}),
    "kernel_variant_1": (lambda: _W().plane_profile(96, 160, 24, 10), {"kernel_variant": 1}),
}


@pytest.mark.parametrize("case", list(CASES))
def test_resume_is_bitwise_the_uninterrupted_run(dfb, tmp_path, case):
    mk, kw = CASES[case]
    plane = mk()
    A = make(dfb, plane, seed=11, plane_id=2, **kw)
    if case == "1024x2048_profile":
        assert A.info(10) == 2                               # the run-recursive y-sweep
    if case == "default_plane":
        assert A.info(10) != 2 and A.info(9) > 0             # band matrices
    ref = steps(dfb, A, DTS)[N:]
    A.close()
    B = make(dfb, plane, seed=11, plane_id=2, **kw)
    steps(dfb, B, DTS[:N])
    path = str(tmp_path / "run.dfbr")
    B.save_restart(path)
    info = dfb.restart_info(path)
    assert info["step"] == N + 1 and info["records"] == 1 and info["seed"] == 11 and info["plane_id"] == 2
    B.close()
    C = make(dfb, plane, seed=11, plane_id=2, **kw)
    C.load_restart(path)
    assert C.step == N + 1
    assert_same(steps(dfb, C, DTS[N:]), ref, case)


def test_resume_in_inject_mode(dfb, tmp_path):
    """the same injected noise on both sides of the restart"""
    plane = _W().plane_profile(96, 160, 24, 10)
    probe = make(dfb, plane, noise_mode=dfb.NOISE_INJECT)
    Ny, Nz = probe.Ny, probe.Nz
    ym, zm = [F.Ny_max for F in (probe.u, probe.v, probe.w)], [F.Nz_max for F in (probe.u, probe.v, probe.w)]
    probe.close()
    rng = np.random.default_rng(3)
    noise = [[(rng.standard_normal((Ny + 2 * ym[f], Nz)), rng.standard_normal((Ny, 2 * zm[f]))) for f in range(3)] for _ in range(2 * N + 1)]

    def inject(df, s):
        for f in range(3):
            df.set_noise(f, *noise[s][f])

    def started():
        df = make(dfb, plane, noise_mode=dfb.NOISE_INJECT)
        inject(df, 0)
        df.first_step()
        return df

    A = started()
    ref = steps(dfb, A, DTS, lambda df, s: inject(df, s + 1))[N:]
    B = started()
    steps(dfb, B, DTS[:N], lambda df, s: inject(df, s + 1))
    path = str(tmp_path / "inject.dfbr")
    B.save_restart(path)
    B.close()
    C = make(dfb, plane, noise_mode=dfb.NOISE_INJECT, seed=999)        # inject mode: the seed is not the noise
    C.load_restart(path)
    assert_same(steps(dfb, C, DTS[N:], lambda df, s: inject(df, s + N + 1)), ref, "inject")


# ---- changes of decomposition: every loader against the uninterrupted run of its own layout ----
PLANE_NZ = 160


def _slabs(dfb, plane, cuts, **kw):
    return [make(dfb, plane, k_begin=a, k_end=b, **kw) for a, b in zip(cuts[:-1], cuts[1:])]


def _resume_check(dfb, loaders, refs, path, exact=True, **load):
    for L in loaders:
        L.load_restart(path, **load)
    for L, r in zip(loaders, refs):
        got = steps(dfb, L, DTS[N:])
        if exact:
            assert_same(got, r, "decomposition")
        else:
            for g, x in zip(got, r):
                ok, worst = normwise_close(g, x, 1e-12)
                assert ok, worst


# Slabs cut on 16-column boundaries run the whole plane's kernel forms and reproduce it bit for bit; a slab cut elsewhere (101) takes
# the direct z-sweep, so a file it wrote, or a run it continues, agrees with the other layout to rounding.
@pytest.mark.parametrize("save_cuts, load_cuts, exact", [([0, 64, 160], [0, 160], True), ([0, 160], [0, 48, 112, 160], True),
                                                         ([0, 48, 112, 160], [0, 160], True), ([0, 160], [0, 48, 101, 160], False),
                                                         ([0, 48, 101, 160], [0, 160], False)])
def test_slabs_and_whole_planes_share_one_file(dfb, tmp_path, save_cuts, load_cuts, exact):
    plane = _W().plane_profile(96, PLANE_NZ, 24, 10)
    refs = [steps(dfb, A, DTS)[N:] for A in _slabs(dfb, plane, load_cuts, seed=5)]
    path = str(tmp_path / "slabs.dfbr")
    writers = _slabs(dfb, plane, save_cuts, seed=5)
    for B in writers:
        steps(dfb, B, DTS[:N])
    for B in writers:
        B.save_restart(path)
    assert dfb.restart_info(path)["records"] == len(writers)
    del writers
    _resume_check(dfb, _slabs(dfb, plane, load_cuts, seed=5), refs, path, exact)


def test_batch_of_4_resumes_as_single_planes(dfb, tmp_path):
    plane = _W().plane_profile(96, 160, 24, 10)
    refs = [steps(dfb, make(dfb, plane, seed=8, plane_id=10 + p), DTS)[N:] for p in range(4)]
    B = make(dfb, plane, nplanes=4, seed=8, plane_id=10)
    steps(dfb, B, DTS[:N])
    path = str(tmp_path / "batch.dfbr")
    B.save_restart(path)
    B.close()
    _resume_check(dfb, [make(dfb, plane, seed=8, plane_id=10 + p) for p in range(4)], refs, path)


def test_batch_of_8_resumes_as_two_batches_of_4(dfb, tmp_path):
    plane = _W().plane_profile(96, 160, 24, 10)
    refs = [steps(dfb, make(dfb, plane, nplanes=4, seed=8, plane_id=pid), DTS)[N:] for pid in (0, 4)]
    B = make(dfb, plane, nplanes=8, seed=8)
    steps(dfb, B, DTS[:N])
    path = str(tmp_path / "batch8.dfbr")
    B.save_restart(path)
    B.close()
    _resume_check(dfb, [make(dfb, plane, nplanes=4, seed=8, plane_id=pid) for pid in (0, 4)], refs, path)


# ---- statistics ----
def test_statistics_resume_bitwise(dfb, tmp_path):
    """N2 sums and count; correlation sums, pairs, count and integral scales, with a temporal ring (L_t = 4) spanning the restart"""
    plane = _W().plane_profile(96, 160, 24, 10)

    def started():
        df = make(dfb, plane, seed=21)
        df.stats_enable()
        df.corr_enable(t=4)
        return df

    def stats(df):
        n2 = [df.stats(w) for w in range(6)]
        corr = [df.corr(f, d, normalized=False) for f in range(3) for d in range(3)]
        scales = [df.integral_scales(f, d) for f in range(3) for d in range(3)]
        return n2, corr, scales

    A = started()
    steps(dfb, A, DTS)
    ref = stats(A)
    B = started()
    steps(dfb, B, DTS[:N])
    path = str(tmp_path / "stats.dfbr")
    B.save_restart(path, stats=True, corr=True)
    info = dfb.restart_info(path)
    assert info["stats_count"] == N and info["corr_count"] == N and info["ring_fields"] == N and info["corr_lag_t"] == 4
    B.close()
    C = make(dfb, plane, seed=21)
    C.load_restart(path, stats=True, corr=True)
    assert C.corr_lags == A.corr_lags
    steps(dfb, C, DTS[N:])
    got = stats(C)
    for (g, gc), (r, rc) in zip(got[0], ref[0]):
        assert gc == rc == 2 * N and np.array_equal(g, r)
    for (g, gp, gc), (r, rp, rc) in zip(got[1], ref[1]):
        assert gc == rc == 2 * N and np.array_equal(gp, rp) and np.array_equal(g, r)
    for g, r in zip(got[2], ref[2]):
        assert np.array_equal(g, r, equal_nan=True)


def test_file_of_other_kernel_forms_resumes_to_rounding(dfb, tmp_path, monkeypatch):
    """a file written under DFB_Y_MODE=0 (dense band matrices) loaded into a default handle (run-recursive y-sweep)"""
    plane = _W().plane_profile(96, 160, 24, 10)
    A = make(dfb, plane, seed=4)
    ref = steps(dfb, A, DTS)[N:]
    monkeypatch.setenv("DFB_Y_MODE", "0")
    B = make(dfb, plane, seed=4)
    monkeypatch.delenv("DFB_Y_MODE")
    assert B.info(10) == 0 and A.info(10) != 0
    steps(dfb, B, DTS[:N])
    path = str(tmp_path / "dense.dfbr")
    B.save_restart(path)
    assert dfb.restart_info(path)["y_form"] == 0
    C = make(dfb, plane, seed=4)
    C.load_restart(path)
    for g, r in zip(steps(dfb, C, DTS[N:]), ref):
        ok, worst = normwise_close(g, r, 1e-12)
        assert ok, worst


# ---- refusals: each leaves the handle's next step bitwise as if no load had been attempted ----
def test_refused_loads_and_saves_change_nothing(dfb, tmp_path):
    W = _W()
    plane = W.plane_profile(96, 160, 24, 10)
    X, T = make(dfb, plane, seed=30), make(dfb, plane, seed=30)          # X is refused; T is its untouched twin
    for df in (X, T):
        steps(dfb, df, DTS[:2])

    def file_of(name, pl=plane, what=None, **kw):
        df = make(dfb, pl, **{"seed": 30, **kw})
        df.filter(1e-7)
        if what == "stats":
            df.stats_enable()
            df.filter(1e-7)
        p = str(tmp_path / name)
        df.save_restart(p, stats=what == "stats")
        df.close()
        return p

    def refused(code, text, path, **kw):
        with pytest.raises(dfb.DfbError) as e:
            X.load_restart(path, **kw)
        assert e.value.code == code and text in str(e.value), str(e.value)

    refused(dfb.ERR_ARG, "seed differs: file 31, handle 30", file_of("seed.dfbr", seed=31))
    refused(dfb.ERR_ARG, "geometry differs", file_of("geom.dfbr", W.plane_profile(96, 176, 24, 10)))
    refused(dfb.ERR_ARG, "the filter tables differ", file_of("hw.dfbr", W.plane_profile(96, 160, 24, 12)))
    refused(dfb.ERR_ARG, "are not in the file's planes", file_of("planes.dfbr", plane_id=5))
    refused(dfb.ERR_ARG, "no N2 statistics", file_of("nostats.dfbr"), stats=True)
    good = file_of("good.dfbr")
    trunc = str(tmp_path / "trunc.dfbr")
    with open(good, "rb") as fh:
        data = fh.read()
    with open(trunc, "wb") as fh:
        fh.write(data[:-8])
    refused(dfb.ERR_IO, "truncated", trunc)
    refused(dfb.ERR_IO, "", str(tmp_path / "missing.dfbr"))
    half = str(tmp_path / "half.dfbr")
    S = make(dfb, plane, seed=30, k_begin=0, k_end=64)
    S.filter(1e-7)
    S.save_restart(half)                                                 # the other slab's writer never saved
    refused(dfb.ERR_IO, "no writer record covers columns [64, 160)", half)
    # saves that are refused
    with pytest.raises(dfb.DfbError) as e:
        X.save_restart(str(tmp_path / "x.dfbr"), stats=True)
    assert e.value.code == dfb.ERR_STATE
    with pytest.raises(dfb.DfbError) as e:
        X.save_restart(str(tmp_path / "x.dfbr"), corr=True)
    assert e.value.code == dfb.ERR_STATE
    with pytest.raises(dfb.DfbError) as e:
        S.save_restart(half, corr=True)
    assert e.value.code == dfb.ERR_ARG and "whole plane" in str(e.value)
    with pytest.raises(dfb.DfbError) as e:
        S.load_restart(half, corr=True)
    assert e.value.code == dfb.ERR_ARG and "whole plane" in str(e.value)
    # a save while a dfb_filter_to_host_begin is outstanding (both handles take the same step)
    host = [np.zeros((96, 160)) for _ in range(5)]
    for df in (X, T):
        assert dfb.lib().dfb_filter_to_host_begin(df._h, 1e-7, *[h.ctypes.data for h in host]) == 0
    with pytest.raises(dfb.DfbError) as e:
        X.save_restart(str(tmp_path / "x.dfbr"))
    assert e.value.code == dfb.ERR_STATE and "outstanding" in str(e.value)
    for df in (X, T):
        assert dfb.lib().dfb_filter_to_host_end(df._h) == 0
    assert not os.path.exists(str(tmp_path / "x.dfbr"))
    assert X.step == T.step
    assert_same(steps(dfb, X, DTS[2:5]), steps(dfb, T, DTS[2:5]), "after refusals")
