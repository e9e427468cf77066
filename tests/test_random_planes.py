"""Seeded random planes through every decision of the step's plan, against the oracle.

The planner (csrc/stepplan.cpp) decides per handle the y-sweep form of every 32-row block, the run groups and their caps, one or two
window buffers, the dense tile width and the column-group order of the run tiles, the z lane blocking and form (or the general
kernels when a window does not fit) and the noise pieces of slabs and periodic planes; the kernels trust the descriptors it emits.
The hand-picked planes of the other tests pin about a dozen combinations of these decisions.  Here a generator draws planes,
handles and launch settings from numpy.random.default_rng(seed): shapes biased towards strip and tile boundaries, half-width
profiles that land on the group caps and on each form's limit (read from the planner, as tests/test_half_width_limits.py does),
N = 0 rows and fields, per-cell ragged planes, batches, periodic planes, slabs, both kernel variants, both noise modes, the planner's
overrides and the launch knobs that change how work is distributed.

CPU: the committed SEEDS reach every entry of FEATURES (read from each case's plan through tests/step_plan_shim.cpp, B200 limits),
every plan passes the descriptor invariants of tests/shims.py, the drawn cases are pinned by a digest, the oracle work is
bounded, and the per-row gate is checked on hand-made arrays.
GPU (-m gpu): each case's handle reports the shim's plan (dfb_info 3, 7-11) and its constructor step and three filter(dt) steps
match the oracle in every output at the field-wide and at a per-row 1e-12 normwise gate; tuned cases match the one-thread-per-cell
kernels on the same noise; slabs on 16-column boundaries and batches reproduce whole planes and single-plane handles bit for bit.
The per-row gate scales a row by the larger of its own rms and the rms of the magnitudes of the terms its values are summed from
(the oracle's chain on |noise|, see magnitudes()): a row carries its own sqrt(R11), b, c and SRA factors, so an error confined to
near-wall rows is seen, while a row whose values cancel (test_a_cancelling_row_is_gated_by_the_magnitude_of_its_terms) is held to
what fp64 can give it."""
import hashlib
import json

import numpy as np
import pytest

from conftest import normwise_close
from oracle_harness import Model, explicit_config, explicit_plane, package
from shims import OVR, StepPlan, check_noise, check_y, check_z, step_plan_shim, y_limits, yr_group_cap, z_limits

gpu = pytest.mark.gpu
TOL = 1e-12
SEED = 31                                # noise seed of every handle
PLANE_ID = 3
STEPS = 4                                # the constructor's step and three filter(dt) steps
CASE_TAPS = 4e9                          # oracle taps of one case's chain (all steps, all planes of a batch)
TOTAL_TAPS = 1.2e11                      # ... of both chains (values, term magnitudes) of all cases: ~40 s of one host core
DT_MENU = (5e-8, 2e-7, 4.5e-7, 1.2e-6, 3e-6)   # Lt is 1.2e-6 (u) and 4.5e-7 (v, w)
OVERRIDES = {"DFB_Y_MODE": "y_mode", "DFB_Y_TK": "y_tk", "DFB_Y_COLGROUP": "y_colgroup", "DFB_ZK": "zk", "DFB_Z_MODE": "z_mode"}
assert tuple(OVERRIDES.values()) == OVR
KNOBS = {"DFB_Z_BLOCKS_PER_SM": ("1", "2", "3"), "DFB_Y_PERSIST": ("1", "2", "7")}


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    return step_plan_shim(tmp_path_factory)


@pytest.fixture(scope="module")
def dfbm():
    return package()


@pytest.fixture(scope="module")
def limits(shim, dfbm, W):
    return dict(z={f"{zk}/{zm}": n for (zk, zm), n in z_limits(shim, dfbm, W).items()}, y=dict(y_limits(shim, dfbm, W)))


# ---------------------------------------------------------------------------------------------
# the generator
# ---------------------------------------------------------------------------------------------
Y_SMALL = (1, 2, 3, 7, 8, 9, 15, 16, 17, 23, 24, 25, 26, 31, 32, 40, 48, 64, 75, 76, 96, 100, 128)
Z_SMALL = (1, 2, 3, 6, 7, 8, 9, 15, 16, 17, 23, 24, 25, 31, 32, 33, 48, 64, 100, 130, 200)
PRIMES = (2, 3, 5, 7, 11, 13, 17, 31, 61, 127, 257, 509, 1021, 1499)


def _pick(rng, seq):
    return seq[int(rng.integers(len(seq)))]


def _draw_Nz(rng):
    kind = int(rng.integers(5))
    if kind == 0:
        return int(rng.integers(1, 1501))
    if kind == 1:                                                       # a multiple of 16, or one off it
        return max(1, 16 * int(rng.integers(1, 94)) + _pick(rng, (-1, 0, 0, 1)))
    if kind == 2:                                                       # a multiple of a z strip (32 * zk), or one off it
        return max(1, _pick(rng, (256, 512)) * int(rng.integers(1, 3)) + _pick(rng, (-1, 0, 0, 1)))
    if kind == 3:
        return _pick(rng, PRIMES)
    return int(rng.integers(1, 40))


def _profile(rng, Ny, small, limit_vals):
    """one field's half-widths in one direction, row by row"""
    kind = _pick(rng, ("const", "const", "runs", "runs", "runs", "ramp", "zeros", "zero-field", "limit"))
    if kind == "const":
        return np.full(Ny, _pick(rng, small))
    if kind == "zero-field":
        return np.zeros(Ny, dtype=int)
    if kind == "limit":
        return np.full(Ny, _pick(rng, limit_vals))
    if kind == "ramp":                                                  # a new N every row
        N0, step = int(rng.integers(1, 200)), _pick(rng, (-2, -1, 1, 2))
        r = np.abs(N0 + step * np.arange(Ny))
        return np.where(r == 0, 1, r)
    out = []                                                            # runs, or runs with isolated N = 0 rows
    while len(out) < Ny:
        N = _pick(rng, small) if rng.random() < 0.85 else _pick(rng, limit_vals)
        cap = N * 331 // 1000
        L = _pick(rng, (1, 2, 8, 9, max(1, cap - 1), max(1, cap), cap + 1, 32, 33, int(rng.integers(1, 41))))
        out += [N] * L
    out = np.array(out[:Ny])
    if kind == "zeros":
        out[rng.integers(0, Ny, size=max(1, Ny // 20))] = 0
    return out


def _cost(Ny, Nz, Nyr, Nzr, P):
    return STEPS * P * Nz * sum(int(np.sum(2 * Nyr[f] + 2 * Nzr[f] + 2)) for f in range(3))


def random_case(seed, limits):
    """One case, drawn from numpy.random.default_rng(seed); `limits` = the planner's form limits (fixture `limits`).  Everything is
    plain ints, strings and lists, so that the cases can be pinned by a digest."""
    rng = np.random.default_rng(seed)
    Ny = int(rng.integers(1, 9)) if rng.random() < 0.2 else int(rng.integers(1, 301))
    Nz = _draw_Nz(rng)
    zl, yl = limits["z"], limits["y"]
    y_lim = sorted(v + d for v in yl.values() for d in (0, 1))
    z_lim = sorted(v + d for v in zl.values() for d in (0, 1))
    same = rng.random() < 0.3
    Nyr = [_profile(rng, Ny, Y_SMALL, y_lim) for _ in range(3)]
    Nzr = [_profile(rng, Ny, Z_SMALL, z_lim) for _ in range(3)]
    if same:
        Nyr, Nzr = [Nyr[0]] * 3, [Nzr[0]] * 3
    P = _pick(rng, (1, 1, 1, 2, 3, 5))
    while Ny > 1 and _cost(Ny, Nz, Nyr, Nzr, P) > CASE_TAPS:           # bound the oracle's work: fewer rows
        Ny = max(1, Ny * 2 // 3)
        Nyr, Nzr = [r[:Ny] for r in Nyr], [r[:Ny] for r in Nzr]
    while _cost(Ny, Nz, Nyr, Nzr, P) > CASE_TAPS:                       # ... and, on one row, fewer columns
        Nz = max(1, Nz // 2)
    ragged = []
    if rng.random() < 0.08:                                             # a few cells off their row's value: the general kernels
        for _ in range(int(rng.integers(1, 4))):
            f, d, j, k = int(rng.integers(3)), int(rng.integers(2)), int(rng.integers(Ny)), int(rng.integers(Nz))
            base = int((Nyr if d == 0 else Nzr)[f][j])
            ragged.append([f, d, j, k, max(0, base + _pick(rng, (-2, -1, 1, 3)))])
    Nz_max = max(max(int(r.max()) for r in Nzr), max([v for f, d, j, k, v in ragged if d == 1], default=0))
    periodic = int(Nz_max <= Nz and rng.random() < 0.3)
    k = None
    if Nz >= 2 and rng.random() < 0.35:
        if Nz > 32 and rng.random() < 0.5:                              # on 16-column boundaries (or ending at the plane's edge)
            q = (Nz + 15) // 16
            a, b = sorted(int(x) for x in rng.choice(q + 1, size=2, replace=False))
            k = [16 * a, min(Nz, 16 * b)]
        else:
            a, b = sorted(int(x) for x in rng.choice(Nz + 1, size=2, replace=False))
            k = [a, b]
        if k == [0, Nz]:
            k = None
    variant = int(rng.random() < 0.15)
    mode = "inject" if P == 1 and k is None and rng.random() < 0.5 else "generate"
    env = {}
    for name, vals in (("DFB_Y_MODE", ("0", "1", "2")), ("DFB_Y_TK", ("64", "128")), ("DFB_Y_COLGROUP", ("1", "2", "3")),
                       ("DFB_ZK", ("8", "16")), ("DFB_Z_MODE", ("0", "1"))):
        if rng.random() < 0.12:
            env[name] = _pick(rng, vals)
    for name, vals in KNOBS.items():
        if rng.random() < 0.2:
            env[name] = _pick(rng, vals)
    dts = [float(_pick(rng, DT_MENU)) for _ in range(STEPS - 1)]
    return dict(seed=seed, Ny=Ny, Nz=Nz, N_y=[r.astype(int).tolist() for r in Nyr], N_z=[r.astype(int).tolist() for r in Nzr],
                ragged=ragged, P=P, periodic=periodic, k=k, variant=variant, mode=mode, env=env, dts=dts)


def plane_of(case, W):
    p = explicit_plane(W, case["Ny"], case["Nz"], [np.array(r) for r in case["N_y"]], [np.array(r) for r in case["N_z"]])
    for f, d, j, k, v in case["ragged"]:
        p["N_y" if d == 0 else "N_z"][f][j, k] = v
    p.update(Ny_max=[int(p["N_y"][f].max()) for f in range(3)], Nz_max=[int(p["N_z"][f].max()) for f in range(3)])
    return p


def config_of(dfbm, case, plane, k="case", **kw):
    """the case's configuration; k: "case" = its slab, None = the whole plane"""
    k = case["k"] if k == "case" else k
    kw.setdefault("kernel_variant", case["variant"])
    kw.setdefault("plane_id", PLANE_ID)
    if k is not None:
        kw.update(k_begin=k[0], k_end=k[1])
    return explicit_config(dfbm, plane, seed=SEED, periodic_z=case["periodic"],
                           noise_mode=dfbm.NOISE_INJECT if case["mode"] == "inject" else dfbm.NOISE_GENERATE, **kw)


def plan_of(L, dfbm, case, plane, nplanes=None, **kw):
    """the shim's plan of the case (B200 limits, the case's overrides); raises DfbError where the library would refuse"""
    ovr = {OVERRIDES[n]: int(v) for n, v in case["env"].items() if n in OVERRIDES}
    return StepPlan(L, dfbm, config_of(dfbm, case, plane, **kw), case["P"] if nplanes is None else nplanes, **ovr)


def oracle_taps(case, W):
    p = plane_of(case, W)
    return STEPS * case["P"] * int(sum(np.sum(2 * p["N_y"][f] + 2 * p["N_z"][f] + 2) for f in range(3)))


# ---------------------------------------------------------------------------------------------
# what a case's plan exercises
# ---------------------------------------------------------------------------------------------
FEATURES = {
    "y:0", "y:1", "y:2", "y:3",                                         # y-sweep forms: dense, chunk-recursive, run-recursive, both
    "rgroup:1", "rgroup:2-8", "rgroup:>8",                              # run groups of 1 row, of 2..8, of more (the pad flag)
    "rgroup:at-cap-8", "rgroup:at-cap-0.33N", "rgroup:at-cap-32",       # a run group at its exact cap
    "rtile:partial",                                                    # run tiles whose last 32-column tile is partial
    "rbuf:1", "rbuf:2", "tk:64", "colgroup:>1",
    "band:chunk+dense",                                                 # chunk-recursive and dense groups in one plane
    "z:zk8-direct", "z:zk8-recursive", "z:zk16-direct", "z:zk16-recursive",
    "z:partial-strip", "z:narrow",                                      # W % (32 zk) != 0, W < 32 zk
    "general:ragged", "general:window", "general:variant",              # tuned == 0: per-cell half-widths, a z window too large, asked for
    "zero:y-row", "zero:z-row", "zero:y-field", "zero:z-field",         # N = 0 rows and whole fields
    "batch:y0", "batch:y1", "batch:y2", "batch:y3", "batch:5",
    "periodic", "periodic:wrap",                                        # a periodic plane; one whose noise window wraps
    "slab:aligned:halo", "slab:aligned:no-halo", "slab:unaligned:halo", "slab:unaligned:no-halo",
    "mode:inject", "mode:generate",
    "knob:DFB_Z_BLOCKS_PER_SM", "knob:DFB_Y_PERSIST",
    "refused",
}


def features(case, sp):
    """what the case exercises, from its plan (sp: StepPlan, or the DfbError of a refused override)"""
    out = {"mode:" + case["mode"]}
    if isinstance(sp, Exception):
        return out | {"refused"}
    P, env = case["P"], case["env"]
    for d, key in (("y", "N_y_row"), ("z", "N_z_row")):
        rows = [sp.a(key, f) for f in range(3)]
        if any((r == 0).any() and not (r == 0).all() for r in rows):
            out.add(f"zero:{d}-row")
        if any((r == 0).all() for r in rows):
            out.add(f"zero:{d}-field")
    if P == 5:
        out.add("batch:5")
    if case["periodic"]:
        out.add("periodic")
        if any(len(sp.a("win", i)) for i in range(sp.s("n_arrays"))):
            out.add("periodic:wrap")
    if case["k"] is not None:
        k0, k1 = case["k"]
        aligned = k0 % 16 == 0 and (k1 % 16 == 0 or k1 == case["Nz"])
        halo = any(sp.s("kind", i) == 1 for i in range(sp.s("n_arrays")))
        if not case["periodic"] and (halo or max(sp.s("Nz_max", f) for f in range(3)) > 0):
            out.add(f"slab:{'aligned' if aligned else 'unaligned'}:{'halo' if halo else 'no-halo'}")
    if not sp.s("tuned"):
        out.add("general:variant" if case["variant"] else "general:ragged" if case["ragged"] else "general:window")
        return out
    yf, zk, zmode, W = sp.s("y_form"), sp.s("zk"), sp.s("zmode"), sp.s("W")
    out.add(f"y:{yf}")
    if P > 1:
        out.add(f"batch:y{yf}")
    out.add(f"z:zk{zk}-{'recursive' if zmode else 'direct'}")
    if W % (32 * zk):
        out.add("z:partial-strip")
    if W < 32 * zk:
        out.add("z:narrow")
    rg, rt = sp.a("rgroups"), sp.a("rtiles")
    for g in rg:
        n, N = int(g["nrows"]), int(g["N"])
        out.add("rgroup:1" if n == 1 else "rgroup:2-8" if n <= 8 else "rgroup:>8")
        cap = yr_group_cap(N)
        if n == cap > 1:
            out.add("rgroup:at-cap-8" if N < 25 else "rgroup:at-cap-32" if cap == 32 else "rgroup:at-cap-0.33N")
    if len(rt):
        out.add(f"rbuf:{sp.s('r_nbuf')}")
        fields = set(int(f) for f in rt["field"])
        if any(sp.s("We", f) % 32 for f in fields):
            out.add("rtile:partial")
        if "DFB_Y_COLGROUP" in env and max(-(-sp.s("We", f) // 32) for f in fields) > int(env["DFB_Y_COLGROUP"]):
            out.add("colgroup:>1")
    if sp.s("n_tiles_dense") and sp.s("tk") == 64:
        out.add("tk:64")
    groups = sp.a("groups")
    if (groups["rec"] == 1).any() and (groups["rec"] == 0).any():
        out.add("band:chunk+dense")
    if "DFB_Z_BLOCKS_PER_SM" in env:
        out.add("knob:DFB_Z_BLOCKS_PER_SM")
    if "DFB_Y_PERSIST" in env and sp.s("n_tiles_dense"):
        out.add("knob:DFB_Y_PERSIST")
    return out


# The seeds, chosen once: 0..59, and the four that a greedy cover of FEATURES then picked out of 0..599.  Some features come from
# one seed alone (y form 3, a batch in it and one run window buffer: 329; more than one column group: 279; DFB_Y_PERSIST on dense
# tiles: 172; an unaligned slab that draws no halo: 112).
SEEDS = list(range(60)) + [112, 172, 279, 329]
DIGEST = "d1cb6fe3b1d6f862a6089487cfacac791e83b789b8a2be8065a6c529aa60f999"


@pytest.fixture(scope="module")
def cases(shim, dfbm, W, limits):
    """seed -> (case, plane, plan or DfbError)"""
    out = {}
    for s in SEEDS:
        case = random_case(s, limits)
        plane = plane_of(case, W)
        try:
            sp = plan_of(shim, dfbm, case, plane)
        except dfbm.DfbError as e:
            sp = e
        out[s] = (case, plane, sp)
    return out


# ---------------------------------------------------------------------------------------------
# the per-row gate
# ---------------------------------------------------------------------------------------------
def rowwise_close(got, ref, tol=TOL, mag=None):
    """normwise per row: |got - ref| <= tol * max(|ref|, rms of ref's row, rms of mag's row) elementwise, the row scale floored at
    1e-300 (a row that is identically 0 must come out 0).  mag: the magnitude of the terms each value is computed from
    (magnitudes()); where a row's values are small against those terms, fp64 cannot give them to 1e-12 of their own rms.
    Returns (ok, worst ratio, its row)."""
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    if ref.size == 0:
        return True, 0.0, -1
    rms = np.sqrt(np.mean(ref * ref, axis=1, keepdims=True))
    if mag is not None:
        mag = np.asarray(mag, dtype=np.float64)
        rms = np.maximum(rms, np.sqrt(np.mean(mag * mag, axis=1, keepdims=True)))
    ratio = np.max(np.abs(got - ref) / np.maximum(np.abs(ref), np.maximum(rms, 1e-300)), axis=1)
    if np.isnan(ratio).any():
        j = int(np.argmax(np.isnan(ratio)))
        return False, float("nan"), j
    j = int(np.argmax(ratio))
    return bool(ratio[j] <= tol), float(ratio[j]), j


class AbsModel(Model):
    """the oracle's chain on |noise|: every filter weight (b_i = a^|i| / s, sqrt(alpha), sqrt(1 - alpha)) is positive, so its filt
    is, value for value, the sum of the magnitudes of the terms whose sum is the true filt"""

    def noise(self, p, f, step):
        rys, hal = Model.noise(self, p, f, step)
        return np.abs(rys), None if hal is None else np.abs(hal)


def magnitudes(plane, U, V, Wf, first):
    """the 8 outputs' term magnitudes from the filt magnitudes U, V, W of one step: u' = sqrt(R11) u, v' = b u + c v, w' = sqrt(R33) w,
    T' and rho' = row factors times u' (oracle/df_oracle.c orc_rst_scaling, orc_sra); a first step leaves T', rho' at 0"""
    R11, R21, R22, R33, Us, Ts, rhos, Ms = (np.asarray(r, dtype=np.float64)[:, None] for r in plane["rows"])
    b = np.where(R11 < 1e-10, 0.0, R21 / np.sqrt(np.maximum(R11, 1e-300)))
    um = np.sqrt(R11) * U
    t1 = np.abs(-0.5 * (1.4 - 1) * Ms * Ms / Us)
    z = np.zeros_like(U)
    return [um, np.abs(b) * U + np.sqrt(R22 - b * b) * V, np.sqrt(R33) * Wf, z if first else t1 * Ts * um, z if first else t1 * rhos * um,
            U, V, Wf]


# ---------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------
def test_seeds_cover_every_feature(cases):
    seen = set()
    for s, (case, _, sp) in cases.items():
        seen |= features(case, sp)
    missing = sorted(FEATURES - seen)
    assert not missing, f"features no seed reaches any more (the planner moved a boundary?): {missing}"


def test_plans_of_every_seed_pass_the_invariants(cases):
    for s, (case, _, sp) in cases.items():
        if isinstance(sp, Exception):
            continue
        try:
            if sp.s("tuned"):
                check_y(sp)
                check_z(sp)
            check_noise(sp)
        except AssertionError as e:
            raise AssertionError(f"seed {s}: {e}") from None


def test_refusals_are_the_overrides_errors(cases, dfbm):
    for s, (case, _, sp) in cases.items():
        if isinstance(sp, Exception):
            assert sp.code == dfbm.ERR_ARG and any(n in str(sp) for n in ("DFB_ZK", "DFB_Z_MODE")), (s, str(sp))
            assert "DFB_ZK" in case["env"] or "DFB_Z_MODE" in case["env"], s


def test_cases_are_pinned(limits):
    """the drawn cases are a function of the seeds alone: a change to numpy's generator or to random_case shows up here"""
    blob = json.dumps([random_case(s, limits) for s in SEEDS], sort_keys=True).encode()
    assert hashlib.sha256(blob).hexdigest() == DIGEST
    assert random_case(SEEDS[0], limits) == random_case(SEEDS[0], limits) != random_case(SEEDS[1], limits)


def test_oracle_work_is_bounded(cases, W):
    taps = [oracle_taps(case, W) for case, _, _ in cases.values()]
    assert max(taps) <= CASE_TAPS and 2 * sum(taps) <= TOTAL_TAPS, (max(taps), sum(taps))


def test_rowwise_gate_on_hand_made_arrays():
    ref = np.array([[1.0, -2.0, 3.0], [1e-20, 2e-20, -1e-20], [0.0, 0.0, 0.0]])
    assert rowwise_close(ref, ref) == (True, 0.0, 0)
    got = ref.copy()
    got[1, 1] += 2e-20 * 5e-13                                         # small against its own row: passes
    assert rowwise_close(got, ref)[0]
    assert normwise_close(got, ref)[0]
    got[1, 1] = 2e-20 * (1 + 1e-9)                                     # 1e-9 of a row 1e20 times smaller than the field
    ok, r, j = rowwise_close(got, ref)
    assert not ok and j == 1 and 5e-10 < r < 1e-8
    assert normwise_close(got, ref)[0]                                 # ... which the field-wide gate cannot see
    got = ref.copy()
    got[2, 0] = 1e-310                                                 # anything but 0 in a row that is identically 0
    ok, r, j = rowwise_close(got, ref)
    assert not ok and j == 2
    got[2, 0] = np.nan
    assert rowwise_close(got, ref)[:1] == (False,) and rowwise_close(got, ref)[2] == 2
    got = ref.copy()
    got[0, 2] = 3.0 * (1 + 2e-12)                                      # scaled by |ref| where it exceeds the row rms
    ok, r, j = rowwise_close(got, ref)
    assert not ok and j == 0 and abs(r - 2e-12) < 1e-15
    got = ref.copy()
    got[1, 1] = 2e-20 * (1 + 1e-9)
    mag = np.abs(ref)
    mag[1] = 1e-10                                                     # the row's values are differences of terms of 1e-10
    assert rowwise_close(got, ref, mag=mag)[0] and not rowwise_close(got, ref, mag=np.abs(ref))[0]
    assert rowwise_close(np.zeros((2, 0)), np.zeros((2, 0)))[0]


def _row_in_long_double(O, plane, m, f, j):
    """filt of row j at the first step in long double: the oracle's y and z sweeps (oracle/df_oracle.c) on its own noise and
    coefficients, for a row-uniform plane that is not periodic"""
    Nz, Ymax, M = plane["Nz"], plane["Ny_max"][f], plane["Nz_max"][f]
    rys, hal = m.noise(0, f, 0)
    ny, nz = int(plane["N_y"][f][j, 0]), int(plane["N_z"][f][j, 0])
    by, bz = O.coeffs(ny).astype(np.longdouble), O.coeffs(nz).astype(np.longdouble)
    y = (by[:, None] * rys[j + Ymax - ny:j + Ymax + ny + 1].astype(np.longdouble)).sum(0)
    rz = np.concatenate([hal[j, :M].astype(np.longdouble), y, hal[j, M:].astype(np.longdouble)])
    return np.array([(bz * rz[k + M - nz:k + M + nz + 1]).sum() for k in range(Nz)])


def test_a_cancelling_row_is_gated_by_the_magnitude_of_its_terms(O, W, limits):
    """Seed 47: 17 columns, N_z = 721, so each row of a field is 17 almost equal values; in row 103, v' = b u + c v of terms near 4.7
    comes to 0.02.  fp64 cannot give such a row to 1e-12 of its own rms: the oracle itself, which the reference is pinned to bit for
    bit, is 1.3e-12 of it away from the long-double value.  Against the magnitude of the terms (magnitudes()) it is 2e-16 away."""
    case = random_case(47, limits)
    plane = plane_of(case, W)
    assert (case["Nz"], case["N_z"][1][103], case["ragged"], case["periodic"]) == (17, 721, [], 0)
    kw = dict(seed=SEED, plane_id=PLANE_ID)
    m, a = Model(O, plane, **kw), AbsModel(O, plane, **kw)
    m.first_step()
    a.first_step()
    j = 103
    R11, R21, R22 = (float(plane["rows"][i][j]) for i in range(3))
    b = R21 / np.sqrt(R11)
    exact = (np.longdouble(b) * _row_in_long_double(O, plane, m, 0, j) + np.longdouble(np.sqrt(R22 - b * b)) *
             _row_in_long_double(O, plane, m, 1, j)).astype(np.float64)
    vp = m.out[0, 1]
    mag = magnitudes(plane, *a.fo[0], True)[1]
    ok, r, _ = rowwise_close(vp[j:j + 1], exact[None])
    assert not ok and r > 1e-12
    ok, r, _ = rowwise_close(vp[j:j + 1], exact[None], mag=mag[j:j + 1])
    assert ok and r < 1e-14
    assert np.all(mag >= np.abs(vp))                                   # the magnitudes bound the values they were computed beside


# ---------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------
NAMES = ("u'", "v'", "w'", "T'", "rho'", "filt u", "filt v", "filt w")
SEL = lambda dfb: (dfb.U_FLUC, dfb.V_FLUC, dfb.W_FLUC, dfb.T_FLUC, dfb.RHO_FLUC, dfb.U_FILT, dfb.V_FILT, dfb.W_FILT)


def reference(O, case, plane):
    """the oracle's outputs of the whole plane: ref[step][plane] = the 8 outputs, mag[step][plane] = their term magnitudes; and the
    model (for its noise)"""
    kw = dict(seed=SEED, plane_id=PLANE_ID, nplanes=case["P"], periodic=bool(case["periodic"]))
    m, a = Model(O, plane, **kw), AbsModel(O, plane, **kw)
    ref, mag = [], []
    for s in range(STEPS):
        for x in (m, a):
            x.first_step() if s == 0 else x.filter(case["dts"][s - 1])
        ref.append([[m.out[p, i].copy() for i in range(5)] + [m.fo[p, f].copy() for f in range(3)] for p in range(case["P"])])
        mag.append([magnitudes(plane, *a.fo[p].copy(), s == 0) for p in range(case["P"])])     # (the model rewrites fo in place)
    return ref, mag, m


def run(dfb, case, plane, m=None, **kw):
    """the case's handle (its environment set by the caller): dfb_info 3, 7-11 and out[step][plane] = the 8 outputs"""
    nplanes = kw.pop("nplanes", case["P"])
    df = dfb.DIGITAL_FILTER(config_of(dfb, case, plane, **kw), fetch=False, nplanes=nplanes)
    info = (df.info(3),) + tuple(df.info(i) for i in (7, 8, 9, 10, 11))
    out = []
    for s in range(STEPS):
        if case["mode"] == "inject":
            for f in range(3):
                rys, hal = m.noise(0, f, s)
                df.set_noise(f, rys, hal if plane["Nz_max"][f] and not case["periodic"] else None)
            df.first_step() if s == 0 else df.filter(case["dts"][s - 1])
        elif s:
            df.filter(case["dts"][s - 1])
        out.append([[df.get(w, plane=p).copy() for w in SEL(dfb)] for p in range(nplanes)])
    df.close()
    return info, out


def gate(got, ref, mag, what, worst, k=None):
    """every output of every step and plane at the field-wide and the per-row 1e-12 gates; worst[name] = (field-wide, per-row).
    mag[step][plane]: the term magnitudes of ref's outputs (whole plane, like ref when k is given)"""
    for s in range(len(ref)):
        for p in range(len(ref[s])):
            for i, b in enumerate(ref[s][p]):
                mg = mag[s][p][i]
                b, mg = (b, mg) if k is None else (b[:, k[0]:k[1]], mg[:, k[0]:k[1]])
                a = got[s][p][i]
                ok1, r1 = normwise_close(a, b, TOL)
                ok2, r2, j = rowwise_close(a, b, TOL, mg)
                w = worst.setdefault(NAMES[i], [0.0, 0.0])
                w[0], w[1] = max(w[0], r1), max(w[1], r2)
                assert ok1 and ok2, (f"{what}: step {s}, {NAMES[i]}, plane {p}: field-wide ratio {r1:.3e}, per-row {r2:.3e} "
                                     f"(worst row {j}, column {int(np.argmax(np.abs(a[j] - b[j])))} of {b.shape[1]})")


def expected_info(sp):
    """dfb_info 3, 7-11 of a handle with this plan"""
    if not sp.s("tuned"):
        return (0, 0, 0, 0, -1, 0)
    return (1,) + sp.info()


@gpu
@pytest.mark.parametrize("seed", SEEDS)
def test_random_plane(dfb, O, W, shim, limits, monkeypatch, seed):
    case = random_case(seed, limits)
    plane = plane_of(case, W)
    for name, v in case["env"].items():
        monkeypatch.setenv(name, v)                                     # read when a handle is created
    try:
        sp = plan_of(shim, dfb, case, plane)
    except dfb.DfbError as e:
        with pytest.raises(dfb.DfbError) as got:
            run(dfb, case, plane)
        assert got.value.code == dfb.ERR_ARG and str(got.value) == str(e), (seed, str(got.value), str(e))
        print(f"random planes: seed {seed}: refused as planned: {e}")
        return
    ref, mag, m = reference(O, case, plane)
    tag = f"seed {seed}"
    worst = {}
    info, out = run(dfb, case, plane, m)
    assert info == expected_info(sp), (tag, info, expected_info(sp))
    gate(out, ref, mag, tag, worst, case["k"])
    k = case["k"]
    kmag = mag if k is None else [[[x[:, k[0]:k[1]] for x in pl] for pl in st] for st in mag]     # the handle's columns
    if sp.s("tuned"):                                                   # the one-thread-per-cell kernels on the same noise
        vinfo, vout = run(dfb, case, plane, m, kernel_variant=1)
        assert vinfo[0] == 0
        gate(out, vout, kmag, f"{tag} against kernel_variant 1", {})
    if k is not None and k[0] % 16 == 0 and (k[1] % 16 == 0 or k[1] == case["Nz"]):
        _, whole = run(dfb, case, plane, k=None)                        # a slab on 16-column boundaries: the plane's columns, exactly
        for s in range(STEPS):
            for p in range(case["P"]):
                for i in range(8):
                    assert np.array_equal(out[s][p][i], whole[s][p][i][:, k[0]:k[1]]), (tag, "slab", s, p, NAMES[i])
    if case["P"] > 1:                                                   # a batch: P single-plane handles with plane_id + p
        single_sp = plan_of(shim, dfb, case, plane, nplanes=1)
        same = (single_sp.s("tuned"), single_sp.s("y_form"), single_sp.s("tk")) == (sp.s("tuned"), sp.s("y_form"), sp.s("tk"))
        for p in range(case["P"]):
            _, one = run(dfb, case, plane, nplanes=1, plane_id=PLANE_ID + p)
            for s in range(STEPS):
                for i in range(8):
                    if same:
                        assert np.array_equal(out[s][p][i], one[s][0][i]), (tag, "batch", s, p, NAMES[i])
            if not same:
                gate([[st[p]] for st in out], [[st[0]] for st in one], [[st[p]] for st in kmag],
                     f"{tag} batch plane {p} against its single-plane handle", {})
    print(f"random planes: seed {seed:4d} dfb_info 3/7-11 = {info} worst field-wide {max(w[0] for w in worst.values()):.2e} "
          f"per-row {max(w[1] for w in worst.values()):.2e} "
          + " ".join(f"{n}={w[0]:.1e}/{w[1]:.1e}" for n, w in worst.items()))
