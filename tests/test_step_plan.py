"""The step's plan (csrc/stepplan.cpp) on the CPU: which y-sweep form, groups and tiles, which z-sweep form and units, and the noise
tables every handle would get on a B200, with the invariants the kernels rely on.  The planner and csrc/setup.cpp are built with
g++ against no CUDA library (tests/step_plan_shim.cpp), so every check here runs without a GPU."""
import numpy as np
import pytest

from oracle_harness import explicit_config, explicit_plane, package
from shims import StepPlan, check_noise, check_y, check_z, step_plan_shim


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    return step_plan_shim(tmp_path_factory)


@pytest.fixture(scope="module")
def dfbm():
    return package()


def hybrid_plane(W):
    """test_G2_hybrid_y_sweep_run_blocks_and_band_matrices: steady half-widths over most rows, a new one every row in a steep part"""
    Ny, Nz = 320, 3400
    steep = np.arange(40, 104, 1) * 2
    row_N = np.concatenate([np.full(96, 40), steep, np.repeat(np.arange(100, 36, -4) * 2, 10)])[:Ny]
    return explicit_plane(W, Ny, Nz, [row_N, np.full(Ny, 24), row_N[::-1].copy()], [np.full(Ny, 6)] * 3)


def ragged_runs_plane(W):
    """test_G2_both_forms_of_the_y_sweep: runs of length 1..40 of N from 2 to 200, and of N = 0"""
    rng = np.random.default_rng(7)
    runs, Ns = [], [2, 8, 15, 16, 17, 18, 31, 40, 64, 66, 100, 128, 200]
    while sum(runs) < 330:
        runs.append(int(rng.integers(1, 41)))
    row_N = np.concatenate([np.full(r, Ns[int(rng.integers(0, len(Ns)))]) for r in runs])
    row_N = np.concatenate([row_N[:40], np.zeros(6, dtype=int), row_N[40:], [0]])     # and N = 0: a run of 6 rows, a lone last row
    Ny = len(row_N)
    return explicit_plane(W, Ny, 150, [row_N, row_N[::-1].copy(), np.full(Ny, 128)], [np.full(Ny, 4)] * 3)


def wide_plane(W):
    """test_large_half_widths_beyond_128: half-widths up to 300"""
    Ny, Nz = 24, 700
    Nyr = [np.full(Ny, 200), np.full(Ny, 96), np.linspace(20, 260, Ny).astype(int) // 2 * 2]
    Nzr = [np.full(Ny, 300), np.full(Ny, 2), np.full(Ny, 130)]
    return explicit_plane(W, Ny, Nz, Nyr, Nzr)


@pytest.fixture(scope="module")
def default_plane():
    from oracle.oracle import stored_default_plane
    return stored_default_plane()


def config_of(dfbm, W, default_plane, name, **kw):
    if name == "default":
        return dfbm.DFConfig.from_plane(default_plane, **kw)
    if name == "uniform_N160":
        return dfbm.DFConfig.from_plane(W.plane_saturated(512, 1024, 160), **kw)
    return dfbm.DFConfig.from_plane(W.NAMED[name](), **kw)


# (workload, planes of the handle) -> dfb_info 7..11 on a B200 (zmode, chunk-recursive tiles, dense tiles, y form, run tiles)
BENCH = {
    ("512x512_N32", 1): (1, 0, 0, 2, 192),
    ("1024x2048_profile_N128", 1): (1, 0, 0, 2, 1536),
    ("1024x2048_saturated_N128", 1): (1, 0, 0, 2, 1536),
    ("4096x8192_profile_N128", 1): (1, 0, 0, 2, 24576),
    ("4096x8192_saturated_N128", 1): (1, 0, 0, 2, 24576),
    ("default", 1): (1, 0, 336, 0, 0),
    ("default", 8): (1, 0, 40, 3, 130),
    ("uniform_N160", 1): (1, 384, 0, 1, 0),
}


@pytest.mark.parametrize("name,nplanes", list(BENCH), ids=[f"{n}-x{p}" for n, p in BENCH])
def test_form_and_tile_counts_of_the_benchmarked_planes(shim, dfbm, W, default_plane, name, nplanes):
    sp = StepPlan(shim, dfbm, config_of(dfbm, W, default_plane, name), nplanes)
    assert sp.s("tuned") == 1
    assert sp.info() == BENCH[(name, nplanes)]
    check_y(sp)
    check_z(sp)
    check_noise(sp)


# ---- the tests' own hard planes ----
HARD = {
    "hybrid": (hybrid_plane, {}),
    "ragged-y2": (ragged_runs_plane, dict(y_mode=2)),
    "ragged-y1": (ragged_runs_plane, dict(y_mode=1)),
    "ragged-y0": (ragged_runs_plane, dict(y_mode=0)),
    "ragged": (ragged_runs_plane, {}),
    "wide": (wide_plane, {}),
    "wide-y2": (wide_plane, dict(y_mode=2)),
}


@pytest.mark.parametrize("case", list(HARD))
def test_y_z_and_noise_invariants_on_hard_planes(shim, dfbm, W, case):
    make, ovr = HARD[case]
    sp = StepPlan(shim, dfbm, explicit_config(dfbm, make(W)), **ovr)
    assert sp.s("tuned") == 1
    if case == "hybrid":
        assert sp.s("y_form") == 3
    if "y_mode" in ovr:
        assert sp.s("y_form") == ovr["y_mode"] or (case == "wide-y2" and sp.s("y_form") in (2, 3))
    if case == "wide-y2":
        assert sp.s("r_nbuf") == 1                                      # windows too tall for two buffers
    check_y(sp)
    check_z(sp)
    check_noise(sp)


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_forced_y_form_on_a_profile(shim, dfbm, W, mode):
    sp = StepPlan(shim, dfbm, dfbm.DFConfig.from_plane(W.plane_profile(200, 300, 96, 24)), y_mode=mode)
    assert sp.s("y_form") == mode
    check_y(sp)


def test_overrides_their_errors_and_the_fallback_beyond_the_z_window_limit(shim, dfbm, W):
    cfg = dfbm.DFConfig.from_plane(W.NAMED["512x512_N32"]())
    assert StepPlan(shim, dfbm, cfg, zk=16).s("zk") == 16
    assert StepPlan(shim, dfbm, cfg, y_mode=0, y_tk=64).s("tk") == 64
    assert StepPlan(shim, dfbm, cfg, z_mode=0).s("zmode") == 0
    with pytest.raises(dfbm.DfbError, match="DFB_ZK must be 8 or 16") as e:
        StepPlan(shim, dfbm, cfg, zk=4)
    assert e.value.code == dfbm.ERR_ARG
    slab = dfbm.DFConfig.from_plane(W.NAMED["512x512_N32"](), k_begin=8, k_end=512)
    with pytest.raises(dfbm.DfbError, match="DFB_Z_MODE=1 needs slab boundaries"):
        StepPlan(shim, dfbm, slab, z_mode=1)
    plane = explicit_plane(W, 4, 64, [np.full(4, 2)] * 3, [np.full(4, 1000)] * 3)    # 8 outputs per lane: a window of 283 lines
    sp = StepPlan(shim, dfbm, explicit_config(dfbm, plane))
    assert sp.s("tuned") == 0 and sp.info() == (0, 0, 0, 0, 0)                        # the general kernels
    with pytest.raises(dfbm.DfbError, match=r"z half-width too large for the tuned z-sweep under DFB_ZK / DFB_Z_MODE: its staged window "
                                            r"needs 283 lines \(at most 256\) and \d+ bytes of shared memory, the device allows 232448") as e:
        StepPlan(shim, dfbm, explicit_config(dfbm, plane), zk=8)
    assert e.value.code == dfbm.ERR_ARG


def test_periodic_row_count_limit(shim, dfbm, W):
    """a periodic plane whose extended rows wrap is drawn by one CTA row per piece: at most 65535 pieces per array"""
    Ny = 21900                                                          # 3 pieces per padded row
    plane = explicit_plane(W, Ny, 32, [np.full(Ny, 2)] * 3, [np.full(Ny, 2)] * 3)
    with pytest.raises(dfbm.DfbError, match="periodic_z: too many padded rows"):
        StepPlan(shim, dfbm, explicit_config(dfbm, plane, periodic_z=1))


@pytest.mark.parametrize("k0,k1,Nz_zero,want", [(0, 0, False, 1), (16, 400, False, 1), (0, 390, False, 1), (8, 400, False, 0),
                                                 (0, 208, False, 1), (0, 200, False, 0), (0, 0, True, 0)])
def test_z_mode_follows_slab_alignment_and_zero_half_widths(shim, dfbm, W, k0, k1, Nz_zero, want):
    Ny, Nz = 40, 390
    Nzr = np.full(Ny, 12)
    if Nz_zero:
        Nzr[7] = 0
    plane = explicit_plane(W, Ny, Nz, [np.full(Ny, 20)] * 3, [Nzr, Nzr, Nzr])
    if k1 > Nz:
        k1 = Nz
    sp = StepPlan(shim, dfbm, explicit_config(dfbm, plane, k_begin=k0, k_end=k1))
    assert sp.s("zmode") == want
    check_z(sp)
    check_noise(sp)


@pytest.mark.parametrize("periodic", [0, 1])
def test_noise_tables_of_slabs(shim, dfbm, W, periodic):
    plane = explicit_plane(W, 30, 200, [np.full(30, 8)] * 3, [np.full(30, 40), np.full(30, 0), np.full(30, 150)])
    for k0, k1 in [(0, 0), (0, 64), (64, 128), (136, 200), (30, 170)]:
        sp = StepPlan(shim, dfbm, explicit_config(dfbm, plane, k_begin=k0, k_end=k1, periodic_z=periodic), nplanes=2)
        check_noise(sp)
        check_z(sp)


def run_rows(sp):
    rg, rt = sp.a("rgroups"), sp.a("rtiles")
    rows = set()
    for t in rt:
        for g in rg[t["g0"]:t["g0"] + t["ngroups"]]:
            rows.add((int(t["field"]), int(g["j0"]), int(g["nrows"]), int(g["N"])))
    return rows


@pytest.mark.parametrize("name,nplanes", [("1024x2048_profile_N128", 1), ("default", 1), ("default", 8), ("hybrid", 1), ("ragged", 1)])
def test_slabs_on_16_column_boundaries_take_the_planes_forms(shim, dfbm, W, default_plane, name, nplanes):
    """a slab on 16-column boundaries must compute what the whole plane computes in its columns, bit for bit: it takes the plane's
    y-sweep form, z-sweep blocking and form, and the same run groups"""
    def cfg(**kw):
        if name == "hybrid":
            return explicit_config(dfbm, hybrid_plane(W), **kw)
        if name == "ragged":
            return explicit_config(dfbm, ragged_runs_plane(W), **kw)
        return config_of(dfbm, W, default_plane, name, **kw)
    whole = StepPlan(shim, dfbm, cfg(), nplanes)
    NzG = whole.s("NzG")
    want = (whole.s("y_form"), whole.s("zk"), whole.s("zmode"), run_rows(whole))
    q = NzG // 16
    cuts = [0, 16 * (q // 3), 16 * (2 * q // 3), NzG]
    for k0, k1 in zip(cuts[:-1], cuts[1:]):
        sp = StepPlan(shim, dfbm, cfg(k_begin=k0, k_end=k1), nplanes)
        assert (sp.s("y_form"), sp.s("zk"), sp.s("zmode"), run_rows(sp)) == want, (k0, k1)
        check_y(sp)
        check_z(sp)
        check_noise(sp)
