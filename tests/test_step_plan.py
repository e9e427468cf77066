"""The step's plan (csrc/stepplan.cpp) on the CPU: which y-sweep form, groups and tiles, which z-sweep form and units, and the noise
tables every handle would get on a B200, with the invariants the kernels rely on.  The planner and csrc/setup.cpp are built with
g++ against no CUDA library (tests/step_plan_shim.cpp), so every check here runs without a GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "digital-filtering_b200", "csrc")
B200 = dict(sms=148, smem_optin=232448)          # multiprocessors, opt-in shared memory per block (bytes)
OVR = ("y_mode", "y_tk", "y_colgroup", "zk", "z_mode")

I4 = np.dtype("<i4")
DT = {
    "groups": np.dtype({"names": ["field", "j0", "nrows", "Nmax", "cstart", "nchunks", "cmat_off", "rec", "w0", "gc_off"],
                        "formats": ["<i4"] * 6 + ["<i8"] + ["<i4"] * 3}, align=True),
    "tiles": np.dtype([(k, "<i4") for k in ("field", "col0", "g0", "ngroups", "cbegin", "cend")]),
    "rgroups": np.dtype([("j0", "<i4"), ("nrows", "<i4"), ("N", "<i4"), ("pad", "<i4"),
                         ("a", "<f8"), ("a4", "<f8"), ("naN1", "<f8"), ("inv_s", "<f8")]),
    "rtiles": np.dtype([(k, "<i4") for k in ("field", "col0", "g0", "ngroups", "wlo", "wrows")]),
    "units": np.dtype([(k, "<i4") for k in ("j", "c0", "f", "nchunk", "line0", "cbytes", "coff16", "pad")]),
    "slot_jump": np.dtype([("A", "<u8"), ("C", "<u8")]), "jump": np.dtype([("A", "<u8"), ("C", "<u8")]),
    "win": np.dtype([(k, "<i4") for k in ("row", "x0", "x1", "pad")]),
    "off": I4, "np": I4, "N_y_row": I4, "N_z_row": I4, "coef_pad_ptr": np.dtype("<i8"),
}


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    lib = str(tmp_path_factory.mktemp("stepplan") / "libstepplan.so")      # a temporary directory: the tree may be read-only
    srcs = [os.path.join(CSRC, "setup.cpp"), os.path.join(CSRC, "stepplan.cpp"), os.path.join(ROOT, "tests", "step_plan_shim.cpp")]
    subprocess.run(["/usr/bin/g++", "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), "-I", "/usr/local/cuda/include",
                    "-I", CSRC, "-shared", "-fPIC", "-Wl,--no-undefined", *srcs, "-o", lib], check=True)
    L = C.CDLL(lib)
    L.sp_plan.restype = C.c_void_p
    L.sp_plan.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_longlong, C.POINTER(C.c_int), C.c_int, C.c_char_p, C.c_int]
    L.sp_free.argtypes = [C.c_void_p]
    L.sp_scalar.restype = C.c_longlong
    L.sp_scalar.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
    L.sp_array.restype = C.c_void_p
    L.sp_array.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.POINTER(C.c_longlong), C.POINTER(C.c_int)]
    return L


@pytest.fixture(scope="module")
def dfbm():
    import _dfb_import  # noqa: F401
    import digital_filtering_b200
    return digital_filtering_b200


class StepPlan:
    """One plan_step result, read through the shim: .s(name, i) scalars, .a(name, i) numpy arrays (copies)."""

    def __init__(self, L, dfbm, config, nplanes=1, **ovr):
        c = dfbm.dfb_config()
        c.struct_bytes = C.sizeof(c)                  # what dfb_config_init sets
        c.grid_file_len = c.vel_fluc_file_len = c.line_file_len = -1
        c.device = -1
        keep = dfbm.fill_config(c, config)
        vals = (C.c_int * 5)(*[int(ovr.get(k) or 0) for k in OVR])
        set_bits = sum(1 << i for i, k in enumerate(OVR) if ovr.get(k) is not None)
        err = C.create_string_buffer(512)
        self.L = L
        self.h = L.sp_plan(C.byref(c), nplanes, B200["sms"], B200["smem_optin"], vals, set_bits, err, 512)
        del keep
        if not self.h:
            code, msg = err.value.decode().split(" ", 1)
            raise dfbm.DfbError(int(code), msg)
        self.nplanes = nplanes

    def __del__(self):
        if getattr(self, "h", None):
            self.L.sp_free(self.h)

    def s(self, name, i=0):
        return int(self.L.sp_scalar(self.h, name.encode(), i))

    def a(self, name, i=0):
        nb, el = C.c_longlong(), C.c_int()
        p = self.L.sp_array(self.h, name.encode(), i, C.byref(nb), C.byref(el))
        assert p or nb.value == 0, name
        dt = DT.get(name, np.dtype("<f8"))
        assert dt.itemsize == el.value, (name, dt.itemsize, el.value)
        if nb.value == 0:
            return np.zeros(0, dtype=dt)
        return np.frombuffer(C.string_at(p, nb.value), dtype=dt).copy()

    def info(self):
        """dfb_info 7..11: z mode, chunk-recursive tiles, dense tiles, y form, run tiles"""
        return (self.s("zmode"), self.s("n_tiles_rec"), self.s("n_tiles_dense"), self.s("y_form"), self.s("n_rtiles"))


# ---- planes ----
def explicit_plane(W, Ny, Nz, Ny_rows, Nz_rows):
    """row-uniform plane whose half-widths are supplied (dfb_config.N_y / N_z), as tests/test_gpu_parity.py builds them"""
    yc = (np.arange(Ny) + 0.5) * 1e-5
    N_y = np.stack([np.repeat(np.asarray(Ny_rows[f], dtype=np.int32)[:, None], Nz, axis=1) for f in range(3)])
    N_z = np.stack([np.repeat(np.asarray(Nz_rows[f], dtype=np.int32)[:, None], Nz, axis=1) for f in range(3)])
    return dict(name=f"explicit_{Ny}x{Nz}", Ny=Ny, Nz=Nz, d_i=W.D_I, U_e=W.U_E, yc=yc, dy=np.full(Ny, 1e-5), dz=np.full(Ny, 1e-5),
                rows=W.synthetic_rows(yc + 1e-4), scales=W._scales(W.D_I), explicit_N=True, N_y=N_y, N_z=N_z)


def explicit_config(dfbm, plane, **kw):
    cfg = dfbm.DFConfig.from_plane(plane, **kw)
    cfg.geom_per_row = 0
    cfg.yc = cfg.dy = cfg.dz = None
    cfg.N_y, cfg.N_z = plane["N_y"], plane["N_z"]
    return cfg


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
def W():
    import _dfb_import  # noqa: F401
    from digital_filtering_b200 import workloads
    return workloads


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


# ---- invariants ----
def yr_group_cap(N):
    return (min(N * 331 // 1000, 32) if N >= 25 else 8)


def check_y(sp):
    Ny, RC, YR_C, YR_BOX, Y_G, YJ = (sp.s(k) for k in ("Ny", "Y_RC", "YR_C", "YR_BOX", "Y_G", "YJ"))
    Nr = [sp.a("N_y_row", f) for f in range(3)]
    Nymax = [sp.s("Ny_max", f) for f in range(3)]
    We = [sp.s("We", f) for f in range(3)]
    owner = np.zeros((3, Ny), dtype=int)
    rg, rt = sp.a("rgroups"), sp.a("rtiles")
    assert sp.s("n_rtiles") == len(rt)
    blocks = {}
    for t in rt:
        blocks.setdefault((int(t["field"]), int(t["g0"]), int(t["ngroups"]), int(t["wlo"]), int(t["wrows"])), []).append(int(t["col0"]))
    for (f, g0, ng, wlo, wrows), cols in blocks.items():
        assert sorted(cols) == list(range(0, We[f], YR_C))                 # the block's tiles cover the columns [0, We)
        assert 1 <= ng and wrows <= sp.s("r_wrows")
        for g in rg[g0:g0 + ng]:
            j0, nr, N = int(g["j0"]), int(g["nrows"]), int(g["N"])
            assert np.all(Nr[f][j0:j0 + nr] == N) and 1 <= nr <= yr_group_cap(N)
            assert g["pad"] == (1 if nr > YJ else 0)
            assert wlo <= j0 + Nymax[f] - N and j0 + nr - 1 + Nymax[f] + N <= wlo + wrows - 1
            owner[f, j0:j0 + nr] += 1
    assert sum(ng for (_, _, ng, _, _) in blocks) == len(rg)
    if len(rt):
        assert sp.s("r_wrows") % YR_BOX == 0
        assert sp.s("r_smem") == sp.s("run_smem_ctl") + sp.s("r_nbuf") * sp.s("r_wrows") * YR_C * 8 <= B200["smem_optin"]
        assert sp.s("r_grid") == B200["sms"]
    groups, tiles = sp.a("groups"), sp.a("tiles")
    for g in groups:
        f, j0, nr = int(g["field"]), int(g["j0"]), int(g["nrows"])
        assert 1 <= nr <= YJ and g["Nmax"] == Nr[f][j0:j0 + nr].max()
        lo, hi = j0 + Nymax[f] - g["Nmax"], j0 + nr - 1 + Nymax[f] + g["Nmax"]
        assert g["cstart"] == lo // RC and g["cstart"] + g["nchunks"] == hi // RC + 1
        if g["rec"]:
            assert np.all(Nr[f][j0:j0 + nr] == g["Nmax"]) and g["Nmax"] >= 16
        owner[f, j0:j0 + nr] += 1
    assert np.all(owner == 1), np.argwhere(owner != 1)[:5]                 # every (field, row) in exactly one group
    nd, nrec = sp.s("n_tiles_dense"), sp.s("n_tiles_rec")
    assert nd + nrec == len(tiles)
    bands = {}
    for i, t in enumerate(tiles):
        g = groups[t["g0"]:t["g0"] + t["ngroups"]]
        assert 1 <= len(g) <= Y_G and np.all(g["field"] == t["field"])
        assert np.all(g["j0"][1:] == g["j0"][:-1] + g["nrows"][:-1])          # adjacent groups
        assert t["cbegin"] == g["cstart"].min() and t["cend"] == (g["cstart"] + g["nchunks"]).max()
        bands.setdefault((int(t["field"]), int(t["g0"]), int(t["ngroups"]), i >= nd), []).append(int(t["col0"]))
    tk = sp.s("tk")
    for (f, _, _, rec), cols in bands.items():
        assert sorted(cols) == list(range(0, We[f], 128 if rec else tk))
    assert sum(ng for (_, _, ng, _) in bands) == len(groups)
    any_run, any_band = len(rg) > 0, len(groups) > 0
    form = sp.s("y_form")
    assert form == (3 if any_band else 2) if any_run else form in (0, 1)
    if form == 1:
        assert nd == 0 and nrec > 0
    if form in (0, 3):
        assert nrec == 0 and nd > 0


def check_z(sp):
    Ny, W, zk = sp.s("Ny"), sp.s("W"), sp.s("zk")
    units, n_uv, n_items = sp.a("units")[:-1], sp.s("n_uv"), sp.s("n_items")
    strips = list(range(0, W, 32 * zk))
    assert n_uv == Ny * len(strips) and n_items == 2 * n_uv and len(units) == 3 * n_uv
    keys = sorted(zip(units["j"].tolist(), units["c0"].tolist(), units["f"].tolist()))
    assert keys == sorted((j, c0, f) for j in range(Ny) for c0 in strips for f in range(3))   # every (row, strip, field) once
    u, v = units[0:2 * n_uv:2], units[1:2 * n_uv:2]
    assert np.all(u["f"] == 0) and np.all(v["f"] == 1) and np.all(u["j"] == v["j"]) and np.all(u["c0"] == v["c0"])
    assert np.all(units[2 * n_uv:]["f"] == 2)


def check_noise(sp):
    NzG, k0, k1, periodic = sp.s("NzG"), sp.s("k0"), sp.s("k1"), sp.s("periodic")
    n = sp.s("n_arrays")
    np_all = []
    seen = set()
    for i in range(n):
        f, kind, nseg = sp.s("field", i), sp.s("kind", i), sp.s("n_seg", i)
        seen.add((f, kind))
        off, npr, win = sp.a("off", i), sp.a("np", i), sp.a("win", i)
        assert len(off) == len(npr) == len(sp.a("jump", i)) == nseg > 0
        np_all.append(npr)
        if kind == 1:
            M = sp.s("Nz_max", f)
            assert np.all(off == 0) and np.all(npr == M) and nseg == sp.s("Ny")
            assert sp.s("npairs", i) == sp.s("Ny") * M
            continue
        rows_y, We, xk0 = sp.s("rows_y", f), sp.s("We", f), sp.s("xk0", f)
        assert sp.s("npairs", i) == (rows_y * NzG + 1) // 2
        if len(win) == 0:                                               # one piece per padded row: extended columns [0, We)
            assert (xk0 >= 0 and xk0 + We <= NzG) and nseg == rows_y
            win = np.zeros(nseg, dtype=DT["win"])
            win["row"], win["x1"] = np.arange(rows_y), We
        else:
            assert periodic and (xk0 < 0 or xk0 + We > NzG)
        # each piece's pairs cover its window, at most one element beyond each end
        x0, x1 = win["x0"], win["x1"]
        assert np.all(off <= x0) and np.all(x0 - off <= 1) and np.all(off + 2 * npr >= x1) and np.all(off + 2 * npr - x1 <= 1)
        for r in range(rows_y):                                          # the pieces of a row cover [0, We) exactly
            w = np.sort(win[win["row"] == r], order="x0")
            assert len(w) >= 1 and w["x0"][0] == 0 and w["x1"][-1] == We and np.all(w["x0"][1:] == w["x1"][:-1]), r
    for f in range(3):
        M = sp.s("Nz_max", f)
        assert (f, 0) in seen
        assert ((f, 1) in seen) == (not periodic and M > 0 and (k0 - M < 0 or k1 + M > NzG))   # halo only for slabs that touch an edge
    max_np = max(int(a.max()) for a in np_all)
    assert sp.s("max_np") == max_np and len(sp.a("slot_jump")) == max_np
    per_cta = sp.s("NOISE_THREADS") * sp.s("NOISE_PAIRS")
    assert sp.s("chunks") == (max_np + per_cta - 1) // per_cta


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
