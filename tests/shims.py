"""Host-only library code built with g++ against no CUDA library, so that it is checked without a GPU: the builder (once per session
for each shim), the step's plan read through tests/step_plan_shim.cpp (StepPlan) with the invariants its descriptors must hold, and
the largest half-widths each tuned sweep form takes on a B200, as the planner decides them."""
import ctypes as C
import functools
import os
import subprocess

import numpy as np

from conftest import ROOT
from oracle_harness import explicit_config, explicit_plane

CSRC = os.path.join(ROOT, "digital-filtering_b200", "csrc")
B200 = dict(sms=148, smem_optin=232448)          # multiprocessors, opt-in shared memory per block (bytes)
OVR = ("y_mode", "y_tk", "y_colgroup", "zk", "z_mode")

_built = {}


def build_shim(tmp_path_factory, name, source):
    """lib<name>.so from csrc/setup.cpp, csrc/<source> and tests/<name>_shim.cpp, in a temporary directory (the tree may be
    read-only); built once per session"""
    if name not in _built:
        lib = str(tmp_path_factory.mktemp(name) / f"lib{name}.so")
        srcs = [os.path.join(CSRC, "setup.cpp"), os.path.join(CSRC, source), os.path.join(ROOT, "tests", f"{name}_shim.cpp")]
        subprocess.run(["/usr/bin/g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"), "-I", "/usr/local/cuda/include",
                        "-I", CSRC, "-shared", "-fPIC", "-Wl,--no-undefined", *srcs, "-o", lib], check=True)
        _built[name] = C.CDLL(lib)
    return _built[name]


def step_plan_shim(tmp_path_factory):
    L = build_shim(tmp_path_factory, "step_plan", "stepplan.cpp")
    L.sp_plan.restype = C.c_void_p
    L.sp_plan.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_longlong, C.POINTER(C.c_int), C.c_int, C.c_char_p, C.c_int]
    L.sp_free.argtypes = [C.c_void_p]
    L.sp_scalar.restype = C.c_longlong
    L.sp_scalar.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
    L.sp_array.restype = C.c_void_p
    L.sp_array.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.POINTER(C.c_longlong), C.POINTER(C.c_int)]
    return L


# ---------------------------------------------------------------------------------------------
# the step's plan
# ---------------------------------------------------------------------------------------------
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


# ---------------------------------------------------------------------------------------------
# the largest half-widths of each tuned sweep form
# ---------------------------------------------------------------------------------------------
def zplane(W, Nz_rows, Nz=400, Ny_rows=None):
    """a plane of len(Nz_rows) rows whose three fields all have these N_z (and N_y = 2 unless given); 400 columns take 16 outputs
    per lane by default (>= 384), 200 take 8"""
    Ny = len(Nz_rows[0]) if isinstance(Nz_rows[0], (list, np.ndarray)) else len(Nz_rows)
    zr = Nz_rows if isinstance(Nz_rows[0], (list, np.ndarray)) else [Nz_rows] * 3
    yr = Ny_rows if Ny_rows is not None else [np.full(Ny, 2)] * 3
    return explicit_plane(W, Ny, Nz, [np.asarray(r) for r in yr], [np.asarray(r) for r in zr])


YPLANE = dict(Ny=8, Nz=150)          # the y ladder's limit cases: one 8-row block, partial last column tile


def yplane(W, Ny_rows, Ny=YPLANE["Ny"], Nz=YPLANE["Nz"]):
    yr = Ny_rows if isinstance(Ny_rows[0], (list, np.ndarray)) else [Ny_rows] * 3
    return zplane(W, [np.full(Ny, 2)] * 3, Nz=Nz, Ny_rows=yr)


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


@functools.cache
def z_limits(L, dfbm, W):
    """(outputs per lane, z form) -> largest N_z whose tuned z-sweep fits a B200, as the planner decides it"""
    out = {}
    for zk in (8, 16):
        for zmode in (0, 1):
            N = 1
            while forced_fits(L, dfbm, W, N + 1, zk, zmode):
                N += 1
            out[(zk, zmode)] = N
    return out


@functools.cache
def y_limits(L, dfbm, W):
    """largest N_y of the 8-row plane that the run-recursive y-sweep takes: forced (DFB_Y_MODE=2) with two window buffers per CTA,
    forced with one, and by default (windows of a 128-row block twice in shared memory)"""
    out = {}
    for N in range(0, 1000):
        f2 = plan(L, dfbm, yplane(W, np.full(8, N)), y_mode=2)
        fd = plan(L, dfbm, yplane(W, np.full(8, N)))
        if f2.s("y_form") == 2:
            out["forced-2buf" if f2.s("r_nbuf") == 2 else "forced-1buf"] = N
        if fd.s("y_form") == 2:
            out["default"] = N
    return out
