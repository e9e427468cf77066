"""Half-widths from 0 to the limit of each sweep form.

The tuned z-sweep stages a window of 2 N_z + 1 columns (plus its padding and, in the direct form, the whole coefficient vector) in
shared memory; the run-recursive y-sweep stages 2 N_y + 1 rows per row group.  Where a window does not fit, the planner hands the
rows to another form: the y-sweep's band-matrix kernels, or, for the z-sweep, the general one-thread-per-cell kernels for the whole
handle.  CPU: every plan the planner returns for N_z = 0 .. 1800 fits a B200, and the limits it finds.  GPU (-m gpu): every form
at N = 0, around its blocking and at its limit, and the forms that take over beyond it, against the oracle.  The limits are taken
from the planner (tests/step_plan_shim.cpp, B200 limits), never written down as constants, except where the CPU test pins them."""
import re

import numpy as np
import pytest

from conftest import normwise_close
from test_periodic_z import periodic_step
from test_step_plan import B200, StepPlan, dfbm, explicit_config, explicit_plane, shim  # noqa: F401  (dfbm, shim: fixtures)

TOL = 1e-12
SMEM = B200["smem_optin"]
NZ_SWEEP = 1800                      # beyond the old 256-line limit of both lane blockings
DTS = [2e-7, 8e-7]
gpu = pytest.mark.gpu


def zplane(W, Nz_rows, Nz=400, Ny_rows=None):
    """a plane of len(Nz_rows) rows whose three fields all have these N_z (and N_y = 2 unless given), with the oracle's Ny_max /
    Nz_max; 400 columns take 16 outputs per lane by default (>= 384), 200 take 8"""
    Ny = len(Nz_rows[0]) if isinstance(Nz_rows[0], (list, np.ndarray)) else len(Nz_rows)
    zr = Nz_rows if isinstance(Nz_rows[0], (list, np.ndarray)) else [Nz_rows] * 3
    yr = Ny_rows if Ny_rows is not None else [np.full(Ny, 2)] * 3
    p = explicit_plane(W, Ny, Nz, [np.asarray(r) for r in yr], [np.asarray(r) for r in zr])
    p.update(Ny_max=[int(p["N_y"][f].max()) for f in range(3)], Nz_max=[int(p["N_z"][f].max()) for f in range(3)])
    return p


def natural_z(Nz_rows, Nz, k=None):
    """the lane blocking and z form the planner picks without overrides (stepplan.cpp plan_z)"""
    zk = 16 if Nz >= 384 and max(Nz_rows) >= 24 else 8
    aligned = k is None or (k[0] % 16 == 0 and (k[1] % 16 == 0 or k[1] == Nz))
    return zk, 1 if aligned and min(Nz_rows) >= 1 else 0


def plan(L, dfbm, plane, k=None, **ovr):
    kw = {} if k is None else dict(k_begin=k[0], k_end=k[1])
    return StepPlan(L, dfbm, explicit_config(dfbm, plane, **kw), **ovr)


def forced_fits(L, dfbm, W, N, zk, zmode):
    """does the planner accept N_z = N under DFB_ZK = zk, DFB_Z_MODE = zmode?  (a refusal must be the over-budget error)"""
    try:
        plan(L, dfbm, zplane(W, [N, N]), zk=zk, z_mode=zmode)
        return True
    except dfbm.DfbError as e:
        assert e.code == dfbm.ERR_ARG and "z half-width too large" in str(e), str(e)
        return False


@pytest.fixture(scope="module")
def z_limits(shim, dfbm, W):
    """(outputs per lane, z form) -> largest N_z whose tuned z-sweep fits a B200, as the planner decides it"""
    out = {}
    for zk in (8, 16):
        for zmode in (0, 1):
            N = 1
            while forced_fits(shim, dfbm, W, N + 1, zk, zmode):
                N += 1
            out[(zk, zmode)] = N
    return out


YPLANE = dict(Ny=8, Nz=150)          # the y ladder's limit cases: one 8-row block, partial last column tile


def yplane(W, Ny_rows, Ny=YPLANE["Ny"], Nz=YPLANE["Nz"]):
    yr = Ny_rows if isinstance(Ny_rows[0], (list, np.ndarray)) else [Ny_rows] * 3
    return zplane(W, [np.full(Ny, 2)] * 3, Nz=Nz, Ny_rows=yr)


@pytest.fixture(scope="module")
def y_limits(shim, dfbm, W):
    """largest N_y of the 8-row plane that the run-recursive y-sweep takes: forced (DFB_Y_MODE=2) with two window buffers per CTA,
    forced with one, and by default (windows of a 128-row block twice in shared memory)"""
    out = {}
    for N in range(0, 1000):
        f2 = plan(shim, dfbm, yplane(W, np.full(8, N)), y_mode=2)
        fd = plan(shim, dfbm, yplane(W, np.full(8, N)))
        if f2.s("y_form") == 2:
            out["forced-2buf" if f2.s("r_nbuf") == 2 else "forced-1buf"] = N
        if fd.s("y_form") == 2:
            out["default"] = N
    return out


# ---------------------------------------------------------------------------------------------
# CPU: the planner
# ---------------------------------------------------------------------------------------------
def check_fits(sp):
    assert sp.s("z_smem") <= SMEM and sp.s("box_lines") <= 256
    assert sp.s("n_rtiles") == 0 or sp.s("r_smem") <= SMEM


# unforced planes: (columns, N_z = 0 row beside the N_z row, slab)
UNFORCED = {"zk16-recursive": (400, False, None), "zk16-direct": (400, True, None), "zk16-unaligned-slab": (400, False, (8, 400)),
            "zk16-aligned-slab": (400, False, (16, 208)), "zk8-recursive": (200, False, None), "zk8-direct": (200, True, None),
            "zk8-unaligned-slab": (200, False, (0, 100)), "zk8-aligned-slab": (200, False, (96, 200))}


@pytest.mark.parametrize("case", list(UNFORCED))
def test_unforced_plans_fit_or_take_the_general_kernels(shim, dfbm, W, z_limits, case):
    """N_z = 0 .. 1800 without overrides: the planner returns a tuned plan whose z window (and y window) fits the device exactly when
    N_z is within the limit of the lane blocking and form it picks, and the general kernels (tuned = 0) otherwise -- never a plan
    that cannot launch, never a refusal.  An aligned slab decides as its whole plane does."""
    Nz, zero_row, k = UNFORCED[case]
    for N in range(0, NZ_SWEEP + 1):
        rows = [0, N] if zero_row else [N, N]
        zk, zmode = natural_z(rows, Nz, k)
        sp = plan(shim, dfbm, zplane(W, rows, Nz), k)
        want = N <= z_limits[(zk, zmode)]
        assert sp.s("tuned") == want, (N, zk, zmode, sp.s("z_smem"), sp.s("box_lines"))
        if want:
            assert (sp.s("zk"), sp.s("zmode")) == (zk, zmode), N
            check_fits(sp)
        else:
            assert sp.info() == (0, 0, 0, 0, 0) and len(sp.a("units")) == 0, N
        if case.endswith("aligned-slab") and not case.endswith("unaligned-slab"):
            whole = plan(shim, dfbm, zplane(W, rows, Nz))
            assert (sp.s("tuned"), sp.s("zk"), sp.s("zmode")) == (whole.s("tuned"), whole.s("zk"), whole.s("zmode")), N


@pytest.mark.parametrize("zk", [8, 16])
@pytest.mark.parametrize("zmode", [0, 1], ids=["direct", "recursive"])
def test_forced_plans_fit_or_are_refused(shim, dfbm, W, zk, zmode):
    """N_z = 0 .. 1800 under DFB_ZK and DFB_Z_MODE: a plan that is returned fits; one that would not is DFB_ERR_ARG with the lines and
    shared memory it needs and what the device allows, and stays refused for every larger N_z"""
    refused = False
    for N in range(0 if zmode == 0 else 1, NZ_SWEEP + 1):
        try:
            sp = plan(shim, dfbm, zplane(W, [N, N]), zk=zk, z_mode=zmode)
        except dfbm.DfbError as e:
            assert e.code == dfbm.ERR_ARG
            m = re.search(r"needs (\d+) lines \(at most 256\) and (\d+) bytes of shared memory, the device allows (\d+)", str(e))
            assert m, str(e)
            lines, need, have = (int(x) for x in m.groups())
            assert have == SMEM and (lines > 256 or need > SMEM), (N, lines, need)
            refused = True
            continue
        assert not refused, N
        assert sp.s("tuned") == 1 and (sp.s("zk"), sp.s("zmode")) == (zk, zmode)
        check_fits(sp)
    assert refused


def test_limits_on_a_b200(z_limits, y_limits):
    """the half-widths the tuned kernels take on a B200 (232 448 bytes of opt-in shared memory), as include/dfb200.h and INTEGRATION.md
    state them: the z-sweep's direct form is bounded by shared memory, its recursive form with 8 outputs per lane by the 256-line box
    of a tensor map; the run-recursive y-sweep on an 8-row plane"""
    assert z_limits == {(16, 1): 1120, (16, 0): 544, (8, 1): 888, (8, 0): 720}
    assert y_limits == {"forced-2buf": 204, "forced-1buf": 412, "default": 144}


def test_the_y_form_beyond_the_run_limits(shim, dfbm, W, y_limits):
    """one N_y past the run form's limit goes to the band matrices: chunk-recursive by default, dense when the run form was forced"""
    assert plan(shim, dfbm, yplane(W, np.full(8, y_limits["default"] + 1))).s("y_form") == 1
    sp = plan(shim, dfbm, yplane(W, np.full(8, y_limits["forced-1buf"] + 1)), y_mode=2)
    assert sp.s("y_form") == 0 and sp.s("n_rtiles") == 0


# ---------------------------------------------------------------------------------------------
# GPU: against the oracle
# ---------------------------------------------------------------------------------------------
def handle(dfb, plane, k=None, nplanes=1, **kw):
    if k is not None:
        kw.update(k_begin=k[0], k_end=k[1])
    return dfb.DIGITAL_FILTER(explicit_config(dfb, plane, **kw), nplanes=nplanes)


def forms(df):
    """dfb_info 3 (tuned kernels), 7 (z form), 10 (y form)"""
    return df.info(3), df.info(7), df.info(10)


def against_oracle(dfb, O, plane, seed, periodic=False):
    """constructor step + two filter(dt) steps in inject mode, every output against O.step (periodic_step for a periodic plane) at
    the 1e-12 normwise gate.  Returns (dfb_info 3/7/10, worst ratio per output)."""
    Ny, Nz = plane["Ny"], plane["Nz"]
    df = handle(dfb, plane, noise_mode=dfb.NOISE_INJECT, periodic_z=int(periodic))
    info = forms(df)
    fo = np.zeros((3, Ny, Nz))
    worst = {}
    for s, dt in enumerate([0.0] + DTS):
        rys = [O.noise_rys(seed, 0, f, s, Ny, plane["Ny_max"][f], Nz) for f in range(3)]
        hal = [O.noise_halo(seed, 0, f, s, Ny, plane["Nz_max"][f]) if plane["Nz_max"][f] else np.zeros((Ny, 0)) for f in range(3)]
        for f in range(3):
            df.set_noise(f, rys[f], hal[f] if plane["Nz_max"][f] and not periodic else None)
        df.first_step() if s == 0 else df.filter(dt)
        df.fetch()
        o = periodic_step(O, plane, rys, fo, dt, s == 0) if periodic else O.step(plane, rys, hal, fo, dt, first_step=(s == 0))
        fo = o["filt_old"]
        got = dict(filt=[df.u.filt, df.v.filt, df.w.filt], fluc=[df.u.fluc, df.v.fluc, df.w.fluc], T=[df.T_fluc], rho=[df.rho_fluc])
        for key, arrs in got.items():
            if s == 0 and key in ("T", "rho"):
                continue
            for f, a in enumerate(arrs):
                ok, r = normwise_close(a, o[key][f] if key in ("filt", "fluc") else o[key], TOL)
                worst[key] = max(worst.get(key, 0.0), r)
                assert ok, (plane["name"], s, key, f, r)
    df.close()
    return info, worst


def note(case, info, worst):
    print("half-width limits: %-40s dfb_info 3/7/10 = %s, worst normwise ratio %.2e %s" % (case, info, max(worst.values()), worst))


@gpu
@pytest.mark.parametrize("zk", [8, 16])
@pytest.mark.parametrize("zmode", [0, 1], ids=["direct", "recursive"])
def test_z_ladder_forced(dfb, O, W, monkeypatch, z_limits, zk, zmode):
    """each lane blocking and z form forced, one row per N_z of 0 (direct form only), 1, 2, ZK-1, ZK, ZK+1 and the largest N_z that
    fits; in the direct form the third field has N_z = 0 on every row (Nz_max = 0: no halo is drawn).  601 columns: several strips,
    a partial last one."""
    monkeypatch.setenv("DFB_ZK", str(zk))
    monkeypatch.setenv("DFB_Z_MODE", str(zmode))
    Ns = ([0] if zmode == 0 else []) + [1, 2, zk - 1, zk, zk + 1, z_limits[(zk, zmode)]]
    third = np.zeros(len(Ns), dtype=int) if zmode == 0 else np.full(len(Ns), 3)
    plane = zplane(W, [np.array(Ns), np.array(Ns[::-1]), third], Nz=601)
    info, worst = against_oracle(dfb, O, plane, seed=41)
    note(f"z ladder zk={zk} zmode={zmode}", info, worst)
    assert info[:2] == (1, zmode)


# (ZK, z form) -> unforced plane that takes it: columns, and whether a row has N_z = 0
NATURAL = {(16, 1): (400, False), (16, 0): (400, True), (8, 1): (200, False), (8, 0): (200, True)}
BEYOND = {16: 1800, 8: 1000}           # past the 256-line box of each lane blocking


@gpu
@pytest.mark.parametrize("at", ["limit", "limit+1", "beyond-256-lines"])
@pytest.mark.parametrize("zk,zmode", list(NATURAL), ids=[f"zk{a}-{'recursive' if b else 'direct'}" for a, b in NATURAL])
def test_z_limit_unforced(dfb, O, W, z_limits, zk, zmode, at):
    """without overrides, at the largest N_z the planner's form takes (tuned, that form), one past it and one past the old 256-line
    limit (the general kernels for the whole handle)"""
    Nz, zero_row = NATURAL[(zk, zmode)]
    N = {"limit": z_limits[(zk, zmode)], "limit+1": z_limits[(zk, zmode)] + 1, "beyond-256-lines": BEYOND[zk]}[at]
    plane = zplane(W, [0, N, N] if zero_row else [N, N, N], Nz=Nz)
    info, worst = against_oracle(dfb, O, plane, seed=43)
    note(f"z zk={zk} zmode={zmode} N_z={N} ({at})", info, worst)
    assert info == ((1, zmode, info[2]) if at == "limit" else (0, 0, -1))


@gpu
def test_z_zero_row_beside_600(dfb, O, W):
    """2048 columns, one row with N_z = 0 beside one with N_z = 600: the direct form with 16 outputs per lane needs more shared memory
    than a B200 has, so the handle runs the general kernels"""
    plane = zplane(W, [0, 600], Nz=2048)
    info, worst = against_oracle(dfb, O, plane, seed=45)
    note("z N_z = 0 / 600 on 2048 columns", info, worst)
    assert info == (0, 0, -1)


@gpu
def test_forced_z_override_over_the_budget_is_refused(dfb, W, monkeypatch, z_limits):
    monkeypatch.setenv("DFB_ZK", "16")
    monkeypatch.setenv("DFB_Z_MODE", "0")
    with pytest.raises(dfb.DfbError) as e:
        handle(dfb, zplane(W, [z_limits[(16, 0)] + 1] * 2))
    assert e.value.code == dfb.ERR_ARG and "bytes of shared memory, the device allows" in str(e.value)


# y ladder: case -> rows of the three fields (a callable of the y limits), the form each forced mode must report (None: the default's)
def _zero_rows(L):
    u = np.concatenate([np.zeros(5), np.full(12, 180), np.zeros(3), np.full(9, 17), [0], np.full(10, 64)]).astype(int)
    return [u, u[::-1].copy(), np.zeros(len(u), dtype=int)]           # the third field: Ny_max = 0


YCASES = {
    "zero-rows": (_zero_rows, None),
    "rec-threshold-15-16-17": (lambda L: [np.repeat([15, 16, 17], 8), np.repeat([17, 16, 15], 8), np.full(24, 16)], None),
    "run-limit-2buf": (lambda L: [np.full(8, L["forced-2buf"])] * 3, {"2": (2, 2)}),
    "run-limit-1buf": (lambda L: [np.full(8, L["forced-1buf"])] * 3, {"2": (2, 1)}),
    "run-limit-1buf+1": (lambda L: [np.full(8, L["forced-1buf"] + 1)] * 3, {"2": (0, 0)}),
    "default-run-limit": (lambda L: [np.full(8, L["default"])] * 3, {None: (2, 2)}),
    "default-run-limit+1": (lambda L: [np.full(8, L["default"] + 1)] * 3, {None: (1, 0)}),
    "tall-3000": (lambda L: [np.full(8, 3000)] * 3, {None: (1, 0), "2": (0, 0)}),
}


@gpu
@pytest.mark.parametrize("case", list(YCASES))
@pytest.mark.parametrize("ymode", [None, "0", "1", "2"], ids=["y-default", "y-dense", "y-chunk-recursive", "y-run-recursive"])
def test_y_ladder(dfb, O, W, shim, monkeypatch, y_limits, ymode, case):
    """every y form (forced, and the default's choice) at N_y = 0 (rows, and a whole field), around the chunk-recursive threshold
    (16), at the largest N_y the run form takes with two window buffers, with one, one past it, and N_y = 3000 on 8 rows.  The
    form dfb_info(10) reports is the planner's (and, where the case names one, that form)."""
    rows_of, named = YCASES[case]
    rows = rows_of(y_limits)
    plane = yplane(W, rows, Ny=len(rows[0]))
    sp = plan(shim, dfb, plane, **({} if ymode is None else dict(y_mode=int(ymode))))
    want = (sp.s("y_form"), sp.s("r_nbuf") if sp.s("n_rtiles") else 0)
    if ymode in ("0", "1"):
        assert want[0] == int(ymode)
    if named and ymode in named:
        assert want == named[ymode], want
    if ymode is not None:
        monkeypatch.setenv("DFB_Y_MODE", ymode)
    info, worst = against_oracle(dfb, O, plane, seed=47)
    note(f"y {case} mode={ymode}", info, worst)
    assert info[0] == 1 and info[2] == want[0]


# ---------------------------------------------------------------------------------------------
# GPU: composites at the boundary N_z (16 outputs per lane, direct form: a row with N_z = 0)
# ---------------------------------------------------------------------------------------------
SEL = lambda dfb: (dfb.U_FLUC, dfb.V_FLUC, dfb.W_FLUC, dfb.T_FLUC, dfb.RHO_FLUC, dfb.U_FILT, dfb.V_FILT, dfb.W_FILT)


def generate(dfb, plane, steps=2, plane_id=0, nplanes=1, k=None):
    """generate mode, seed 5: the constructor step and `steps` filter(dt) steps; outputs[step][plane][which]"""
    df = handle(dfb, plane, k=k, seed=5, plane_id=plane_id, nplanes=nplanes)
    info = forms(df)
    out = []
    for s in range(steps + 1):
        if s:
            df.filter(DTS[s - 1])
        out.append([[df.get(w, plane=p).copy() for w in SEL(dfb)] for p in range(nplanes)])
    df.close()
    return info, out


def boundary_plane(W, z_limits, past):
    N = z_limits[(16, 0)] + (1 if past else 0)
    return zplane(W, [np.array([0, N, 5]), np.array([N, 0, N]), np.array([3, 3, N])], Nz=400), N


@gpu
@pytest.mark.parametrize("past", [False, True], ids=["limit", "limit+1"])
def test_periodic_plane_at_the_boundary(dfb, O, W, z_limits, past):
    """periodic_z with Nz_max = Nz = the boundary N_z and N_z = 0 rows, against the periodic restatement"""
    N = z_limits[(16, 0)] + (1 if past else 0)
    plane = zplane(W, [np.array([0, N, 5]), np.array([N, 0, N]), np.array([3, 3, N])], Nz=N)
    info, worst = against_oracle(dfb, O, plane, seed=49, periodic=True)
    note(f"periodic Nz = N_z = {N}", info, worst)
    assert info[:2] == ((0, 0) if past else (1, 0))


@gpu
@pytest.mark.parametrize("past", [False, True], ids=["limit", "limit+1"])
def test_slabs_at_the_boundary(dfb, O, W, z_limits, past):
    """slabs on 16-column boundaries take their plane's decision and reproduce it bit for bit; a slab cut off a 16-column boundary
    against the oracle (generate mode, the oracle on the same counter-based noise)"""
    plane, N = boundary_plane(W, z_limits, past)
    winfo, whole = generate(dfb, plane)
    assert winfo[:2] == ((0, 0) if past else (1, 0))
    for k in [(0, 160), (160, 176), (176, 400)]:
        info, part = generate(dfb, plane, k=k)
        assert info == winfo, (k, info, winfo)
        for s in range(len(whole)):
            for i, a in enumerate(part[s][0]):
                assert np.array_equal(a, whole[s][0][i][:, k[0]:k[1]]), (k, s, i)
    k = (7, 391)
    info, part = generate(dfb, plane, k=k)
    assert info[:2] == ((0, 0) if past else (1, 0))
    Ny, Nz = plane["Ny"], plane["Nz"]
    fo = np.zeros((3, Ny, Nz))
    worst = 0.0
    for s, dt in enumerate([0.0] + DTS):
        rys = [O.noise_rys(5, 0, f, s, Ny, plane["Ny_max"][f], Nz) for f in range(3)]
        hal = [O.noise_halo(5, 0, f, s, Ny, plane["Nz_max"][f]) for f in range(3)]
        o = O.step(plane, rys, hal, fo, dt, first_step=(s == 0))
        fo = o["filt_old"]
        want = list(o["fluc"]) + [o["T"], o["rho"]] + list(o["filt"])
        for i, b in enumerate(want):
            if s == 0 and i in (3, 4):
                continue
            ok, r = normwise_close(part[s][0][i], b[:, k[0]:k[1]], TOL)
            worst = max(worst, r)
            assert ok, (s, i, r)
    note(f"slab {k} at N_z = {N}", info, {"all": worst})


@gpu
@pytest.mark.parametrize("past", [False, True], ids=["limit", "limit+1"])
def test_batch_at_the_boundary(dfb, W, z_limits, past):
    """a batch of 3 planes reproduces single-plane handles with plane_id + p bit for bit"""
    plane, _ = boundary_plane(W, z_limits, past)
    binfo, batch = generate(dfb, plane, plane_id=4, nplanes=3)
    assert binfo[:2] == ((0, 0) if past else (1, 0))
    for p in range(3):
        info, single = generate(dfb, plane, plane_id=4 + p)
        assert info[:2] == binfo[:2]
        if info[2] == binfo[2]:
            for s in range(len(single)):
                for i, a in enumerate(single[s][0]):
                    assert np.array_equal(batch[s][p][i], a), (p, s, i)
        else:
            for s in range(len(single)):
                for i, a in enumerate(single[s][0]):
                    assert normwise_close(batch[s][p][i], a, 1e-13)[0], (p, s, i)
