"""The filter shape on the CPU, through tests/filter_shape_shim.cpp and tests/filter_shape_fp_shim.cpp (csrc/setup.cpp, csrc/stepplan.cpp
and csrc/restart.cpp built with g++, no CUDA): the Gaussian table against numpy's formula and the exponential one against the oracle's,
the integral scales their exact autocorrelations deliver, the step's plan of Gaussian planes (direct forms only, every descriptor
invariant, the random-plane generator's cases among them), the refusal of the recursive forms' overrides, the restart fingerprint of
either shape, and the numpy restatement of the sweeps (tests/shape_model.py) against the oracle's sweeps."""
import ctypes as C

import numpy as np
import pytest

from conftest import normwise_close
from oracle_harness import explicit_config, explicit_plane, package
from shape_model import gauss_coef, sweep_y, sweep_z
from shims import B200, OVR, StepPlan, build_shim, check_noise, check_y, check_z, step_plan_shim, yplane, zplane
from test_random_planes import OVERRIDES, SEEDS, config_of, plane_of, random_case
from test_time_scales_host import FP_PROFILE_96x160, Cfg

D = C.POINTER(C.c_double)
EXP, GAUSS = 0, 1


@pytest.fixture(scope="module")
def sp_shim(tmp_path_factory):
    return step_plan_shim(tmp_path_factory)


@pytest.fixture(scope="module")
def shim(tmp_path_factory, sp_shim):
    L = build_shim(tmp_path_factory, "filter_shape", "stepplan.cpp")
    for name in ("sp_free", "sp_scalar", "sp_array"):        # the accessors of tests/step_plan_shim.cpp, compiled into this library
        fn, ref = getattr(L, name), getattr(sp_shim, name)
        fn.restype, fn.argtypes = ref.restype, ref.argtypes
    L.fs_coefficients.argtypes = [C.c_int, C.c_int, D]
    L.fs_plan.restype = C.c_void_p
    L.fs_plan.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_longlong, C.POINTER(C.c_int), C.c_int, C.c_char_p, C.c_int]
    L.fs_plan_coef.argtypes = [C.c_void_p, C.c_int, D]
    return L


@pytest.fixture(scope="module")
def fp_shim(tmp_path_factory):
    L = build_shim(tmp_path_factory, "filter_shape_fp", "restart.cpp")
    L.fs_fingerprint.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_uint64), C.c_char_p, C.c_int]
    return L


@pytest.fixture(scope="module")
def dfbm():
    return package()


class ShapePlan(StepPlan):
    """StepPlan of the plane in filter shape `shape` (fs_plan: the table rebuilt as dfb_set_filter_shape rebuilds it)"""

    def __init__(self, L, dfbm, config, shape, nplanes=1, **ovr):
        c = dfbm.dfb_config()
        c.struct_bytes = C.sizeof(c)
        c.grid_file_len = c.vel_fluc_file_len = c.line_file_len = -1
        c.device = -1
        keep = dfbm.fill_config(c, config)
        vals = (C.c_int * 5)(*[int(ovr.get(k) or 0) for k in OVR])
        set_bits = sum(1 << i for i, k in enumerate(OVR) if ovr.get(k) is not None)
        err = C.create_string_buffer(512)
        self.L = L
        self.h = L.fs_plan(C.byref(c), shape, nplanes, B200["sms"], B200["smem_optin"], vals, set_bits, err, 512)
        del keep
        if not self.h:
            code, msg = err.value.decode().split(" ", 1)
            raise dfbm.DfbError(int(code), msg)
        self.nplanes = nplanes

    def coef(self, N):
        b = np.zeros(2 * N + 1)
        assert self.L.fs_plan_coef(self.h, N, b.ctypes.data_as(D)) == 1, N
        return b


def table(shim, N, shape):
    b = np.zeros(2 * N + 1)
    shim.fs_coefficients(N, shape, b.ctypes.data_as(D))
    return b


# ---- the tables ----
NS = list(range(0, 65)) + [96, 127, 128, 200, 256, 511, 1120]


def test_gaussian_table_matches_numpy(shim):
    for N in NS:
        b = table(shim, N, GAUSS)
        ref = gauss_coef(N)
        assert np.max(np.abs(b - ref)) <= 1e-15 * np.max(ref), N
        assert abs(np.sum(b * b) - 1.0) <= 1e-14, N
        assert np.array_equal(b, b[::-1]), N                         # mirrored, not recomputed
    assert np.array_equal(table(shim, 0, GAUSS), [1.0])


def test_exponential_table_is_the_oracles(shim, O):
    for N in NS:
        assert np.array_equal(table(shim, N, EXP), O.coeffs(N)), N


def integral_scale(b):
    """the integral scale, in cells, of the exact autocorrelation of table b as dfb_corr_integral_scales defines it: the trapezoidal
    sum of R(0..d*), d* the last lag before R first drops to <= 0"""
    N = (len(b) - 1) // 2
    R = np.array([np.dot(b[:len(b) - d], b[d:]) for d in range(2 * N + 1)]) / np.dot(b, b)
    dstar = len(R) - 1 if np.all(R > 0) else int(np.argmax(R <= 0)) - 1
    return float(np.sum(0.5 * (R[:dstar] + R[1:dstar + 1])))


# integral scale / n (n = N / 2) of either shape, to three digits: the Gaussian delivers the configured length, the exponential ~0.64 of it
DELIVERED = {4: (0.533, 1.000), 8: (0.586, 1.000), 16: (0.620, 0.999), 32: (0.631, 0.999), 64: (0.633, 0.999), 128: (0.634, 0.999),
             256: (0.634, 0.999)}


@pytest.mark.parametrize("N", sorted(DELIVERED))
def test_delivered_integral_scales(shim, N):
    exp_ratio, gauss_ratio = DELIVERED[N]
    assert integral_scale(table(shim, N, EXP)) / (N / 2) == pytest.approx(exp_ratio, abs=1e-3)      # the table's last digit
    assert integral_scale(table(shim, N, GAUSS)) / (N / 2) == pytest.approx(gauss_ratio, abs=1e-3)


# ---- the step's plan of a Gaussian plane ----
def check_direct(sp, what):
    assert sp.s("y_form") == 0 if sp.s("tuned") else True, what
    if sp.s("tuned"):
        assert sp.s("zmode") == 0 and sp.s("n_tiles_rec") == 0 and sp.s("n_rtiles") == 0, (what, sp.info())
        assert len(sp.a("rgroups")) == 0 and len(sp.a("rtiles")) == 0 and len(sp.a("unit_par")) == 0, what
        assert not np.any(sp.a("groups")["rec"]), what
        check_y(sp)
        check_z(sp)
    check_noise(sp)


def hand_planes(W):
    """the planner's decision points of an exponential plane: long runs of equal N (run- and chunk-recursive forms), slabs on and off
    16-column boundaries, windows up to and beyond the direct z-sweep's limit"""
    out = [(W.plane_profile(96, 160, 24, 10), {}), (W.plane_profile(256, 512, 40, 24), {}), (W.plane_profile(128, 400, 64, 32), {}),
           (W.plane_profile(96, 160, 24, 10), dict(k_begin=32, k_end=96)), (W.plane_profile(96, 160, 24, 10), dict(k_begin=5, k_end=77)),
           (W.plane_profile(96, 160, 24, 10), dict(periodic_z=1))]
    out += [(yplane(W, np.full(8, N)), {}) for N in (16, 40, 100, 300)]
    out += [(zplane(W, [N, N]), {}) for N in (20, 300, 544, 545, 900)]
    return out


def test_gaussian_plans_use_the_direct_forms(shim, dfbm, W):
    tuned = untuned = 0
    for i, (pl, kw) in enumerate(hand_planes(W)):
        cfg = explicit_config(dfbm, pl, **kw) if pl.get("explicit_N") else dfbm.DFConfig.from_plane(pl, **kw)
        for nplanes in (1, 4):
            sp = ShapePlan(shim, dfbm, cfg, GAUSS, nplanes)
            check_direct(sp, (i, kw, nplanes))
            tuned, untuned = tuned + sp.s("tuned"), untuned + (1 - sp.s("tuned"))
            ex = ShapePlan(shim, dfbm, cfg, EXP, nplanes)
            assert ex.s("tuned") >= sp.s("tuned")                   # the direct z form's window limit is the tighter one
    assert tuned and untuned
    # beyond the direct z-sweep's limit the handle runs the one-thread-per-cell kernels; the recursive form still takes the exponential
    ex, ga = (ShapePlan(shim, dfbm, explicit_config(dfbm, zplane(W, [700, 700])), s) for s in (EXP, GAUSS))
    assert ex.s("tuned") == 1 and ex.s("zmode") == 1 and ga.s("tuned") == 0


def test_random_plane_cases_plan_the_direct_forms(shim, sp_shim, dfbm, W):
    """the random-plane generator's cases (tests/test_random_planes.py) as Gaussian planes, with their overrides: every plan passes
    the invariants and uses the direct forms; every refusal names the override"""
    from shims import y_limits, z_limits
    limits = dict(z={f"{zk}/{zm}": n for (zk, zm), n in z_limits(sp_shim, dfbm, W).items()}, y=dict(y_limits(sp_shim, dfbm, W)))
    planned = refused = 0
    for s in SEEDS:
        case = random_case(s, limits)
        plane = plane_of(case, W)
        ovr = {OVERRIDES[n]: int(v) for n, v in case["env"].items() if n in OVERRIDES}
        try:
            sp = ShapePlan(shim, dfbm, config_of(dfbm, case, plane), GAUSS, case["P"], **ovr)
        except dfbm.DfbError as e:
            refused += 1
            assert e.code == dfbm.ERR_ARG, (s, str(e))
            assert ("Gaussian" in str(e) and (ovr.get("y_mode") in (1, 2) or ovr.get("z_mode") == 1)) or \
                "z half-width too large" in str(e), (s, ovr, str(e))
            continue
        planned += 1
        check_direct(sp, s)
        for N in np.unique(np.concatenate([np.ravel(plane["N_y"]), np.ravel(plane["N_z"])])):
            assert np.max(np.abs(sp.coef(int(N)) - gauss_coef(int(N)))) <= 1e-15, (s, N)
    assert planned >= 40 and refused >= 1, (planned, refused)


@pytest.mark.parametrize("ovr,msg", [(dict(y_mode=1), "DFB_Y_MODE=1 (chunk-recursive y-sweep)"),
                                     (dict(y_mode=2), "DFB_Y_MODE=2 (run-recursive y-sweep)"),
                                     (dict(z_mode=1), "DFB_Z_MODE=1 (recursive z-sweep)")])
def test_recursive_overrides_are_refused(shim, dfbm, W, ovr, msg):
    cfg = dfbm.DFConfig.from_plane(W.plane_profile(96, 160, 24, 10))
    with pytest.raises(dfbm.DfbError) as e:
        ShapePlan(shim, dfbm, cfg, GAUSS, **ovr)
    assert e.value.code == dfbm.ERR_ARG
    assert str(e.value).endswith(": " + msg + " evaluates the exponential filter recursively: the filter shape is Gaussian (DFB_FILTER_GAUSSIAN), " \
                                 "which runs the direct forms only")
    ShapePlan(shim, dfbm, cfg, EXP, **ovr)                        # the exponential plane takes them
    sp = ShapePlan(shim, dfbm, cfg, GAUSS, y_mode=0, z_mode=0)    # ... and the Gaussian one the direct forms'
    check_direct(sp, ovr)


def test_exponential_plans_are_unchanged(shim, sp_shim, dfbm, W):
    for pl, kw in hand_planes(W):
        cfg = explicit_config(dfbm, pl, **kw) if pl.get("explicit_N") else dfbm.DFConfig.from_plane(pl, **kw)
        a, b = StepPlan(sp_shim, dfbm, cfg), ShapePlan(shim, dfbm, cfg, EXP)
        assert a.info() == b.info() and a.s("tuned") == b.s("tuned")
        for name in ("groups", "tiles", "cmat", "yrec", "ygc", "rgroups", "rtiles", "coef_pad", "coef_pad_ptr", "units", "unit_par"):
            x, y = a.a(name), b.a(name)
            fields = x.dtype.names or (None,)
            assert len(x) == len(y) and all(np.array_equal(x[f], y[f]) if f else np.array_equal(x, y) for f in fields), name


# ---- the restart fingerprint ----
def fingerprint(fp_shim, cfg, shape):
    fp, err = C.c_uint64(), C.create_string_buffer(512)
    assert fp_shim.fs_fingerprint(cfg.ref(), shape, C.byref(fp), err, 512) == 0, err.value
    return fp.value


def test_fingerprint(fp_shim, dfbm, W):
    cfg = Cfg(dfbm, dfbm.DFConfig.from_plane(W.plane_profile(96, 160, 24, 10)))
    assert fingerprint(fp_shim, cfg, EXP) == FP_PROFILE_96x160
    g = fingerprint(fp_shim, cfg, GAUSS)
    assert g != FP_PROFILE_96x160 and g == fingerprint(fp_shim, cfg, GAUSS)


# ---- the numpy restatement of the sweeps against the oracle's ----
def test_restated_sweeps_match_the_oracle(O, W):
    rng = np.random.default_rng(5)
    cases = [explicit_plane(W, 40, 56, [rng.integers(0, 13, 40)] * 3, [rng.integers(0, 17, 40)] * 3)]
    pl = W.plane_profile(96, 160, 24, 10)
    O.half_widths(pl)
    cases.append(pl)
    ragged = explicit_plane(W, 24, 32, [np.full(24, 5)] * 3, [np.full(24, 7)] * 3)
    ragged["N_y"][0] = rng.integers(0, 6, (24, 32))
    ragged["N_z"][0] = rng.integers(0, 8, (24, 32))
    cases.append(ragged)
    for p in cases:
        Ny, Nz = p["Ny"], p["Nz"]
        Nym, Nzm = int(np.max(p["N_y"][0])), int(np.max(p["N_z"][0]))
        N_y, N_z = np.ascontiguousarray(p["N_y"][0], dtype=np.int32), np.ascontiguousarray(p["N_z"][0], dtype=np.int32)
        rys = rng.standard_normal((Ny + 2 * Nym, Nz))
        rz = rng.standard_normal((Ny, Nz + 2 * Nzm))
        ref_y = np.full((Ny, Nz + 2 * Nzm), np.nan)
        O.lib().orc_sweep_y(C.c_int(Ny), C.c_int(Nz), C.c_int(Nym), C.c_int(Nzm), O._i(N_y), O._d(rys), O._d(ref_y))
        got_y = sweep_y(O.coeffs, N_y, Nym, rys)
        ok, r = normwise_close(got_y, ref_y[:, Nzm:Nzm + Nz], 1e-15)
        assert ok, r
        ref_z = np.zeros((Ny, Nz))
        O.lib().orc_sweep_z(C.c_int(Ny), C.c_int(Nz), C.c_int(Nzm), O._i(N_z), O._d(rz), O._d(ref_z))
        ok, r = normwise_close(sweep_z(O.coeffs, N_z, Nzm, rz), ref_z, 1e-15)
        assert ok, r
