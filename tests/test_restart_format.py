"""The restart file's host code (csrc/restart.cpp) on the CPU: header encoding, the fingerprint of the filter tables, the writer-record
check a loader makes, the offsets of row segments in the global layout, and a save by several writers into one file that the library's
dfb_restart_info then reads.  restart.cpp and csrc/setup.cpp are built with g++ against no CUDA library (tests/restart_shim.cpp)."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle_harness import package
from shims import build_shim

DATA_AT = 8192
SEC_STATE, SEC_STATS, SEC_CORR_Z, SEC_CORR_Y, SEC_CORR_T, SEC_RING = range(6)
I64 = C.POINTER(C.c_int64)


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    L = build_shim(tmp_path_factory, "restart", "restart.cpp")
    L.rs_fingerprint.restype = C.c_uint64
    L.rs_fingerprint.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
    L.rs_roundtrip.argtypes = [I64, C.POINTER(C.c_double), I64, C.c_char_p, I64, C.POINTER(C.c_double), I64, C.c_char_p, C.c_char_p, C.c_int]
    L.rs_offset.restype = C.c_longlong
    L.rs_offset.argtypes = [I64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    L.rs_file_bytes.restype = C.c_longlong
    L.rs_file_bytes.argtypes = [I64]
    L.rs_coverage.argtypes = [I64, C.c_int, I64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_int]
    L.rs_save.argtypes = [C.c_char_p, I64, I64, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_double), C.c_char_p, C.c_int]
    L.rs_read.argtypes = [C.c_char_p, I64, I64, C.c_int, C.c_char_p, C.c_int]
    return L


@pytest.fixture(scope="module")
def dfbm():
    return package()


def i64(a):
    a = np.ascontiguousarray(a, dtype=np.int64)
    return a, a.ctypes.data_as(I64)


def header(Ny=5, Nz=7, plane0=10, nplanes=3, step=100, sections=1, lags=(0, 0, 0), n_ring=0, fp=0x1234_5678_9abc_def0, seed=42, at=None):
    """header values in dfb_restart_info's order; at = {index: value} for the others"""
    v = np.zeros(30, dtype=np.int64)
    v[[1, 2, 3, 4, 5, 8, 9]] = [Ny, Nz, plane0, nplanes, seed, step, sections]
    v[11] = np.int64(np.uint64(fp).view(np.int64))
    v[12:15], v[15:18], v[18:21] = [6, 4, 6], [8, 8, 6], [1, 1, 2]
    v[23:26], v[28] = lags, n_ring
    for k, x in (at or {}).items():
        v[k] = x
    return v


def test_header_round_trips(shim, dfbm):
    v = header(Ny=1024, Nz=2048, plane0=7, nplanes=4, step=123456789012, sections=7, lags=(40, 30, 5), n_ring=5, seed=-3,
               fp=0xfedc_ba98_7654_3210, at={6: 1, 7: 1, 10: 3, 21: 999, 22: 1, 26: 998, 27: 1})
    Lt = np.array([1.5e-6, 2.5e-7, np.pi])
    ts = np.arange(65, dtype=np.int64) * 7 + 1
    out, Lt_out, ts_out, ver = np.zeros(30, dtype=np.int64), np.zeros(3), np.zeros(65, dtype=np.int64), C.create_string_buffer(64)
    err = C.create_string_buffer(256)
    vv, pv = i64(v)
    assert shim.rs_roundtrip(pv, Lt.ctypes.data_as(C.POINTER(C.c_double)), ts.ctypes.data_as(I64), b"dfb200 test version", out.ctypes.data_as(I64),
                             Lt_out.ctypes.data_as(C.POINTER(C.c_double)), ts_out.ctypes.data_as(I64), ver, err, 256) == 0, err.value
    assert out[0] == 1 and out[29] == shim.rs_file_bytes(pv)
    assert np.array_equal(out[1:29], v[1:29])
    assert np.array_equal(Lt_out, Lt) and np.array_equal(ts_out, ts) and ver.value == b"dfb200 test version"
    # the file's size: header + records, then state [3][P][Ny][Nz], stats [P][6][Ny][Nz], corr sums [P][3][Ny][L+1] per direction,
    # ring [n_ring][P][3][Ny][Nz]
    P, Ny, Nz = 4, 1024, 2048
    expect = DATA_AT + 8 * (3 * P * Ny * Nz + 6 * P * Ny * Nz + sum(P * 3 * Ny * (L + 1) for L in (40, 30, 5)) + 5 * P * 3 * Ny * Nz)
    assert out[29] == expect


def test_header_refuses_foreign_bytes(shim, tmp_path, dfbm):
    bad = tmp_path / "foreign.bin"
    bad.write_bytes(b"not a restart file" + bytes(9000))
    with pytest.raises(dfbm.DfbError) as e:
        dfbm.restart_info(str(bad))
    assert e.value.code == dfbm.ERR_IO and "magic" in str(e.value)
    with pytest.raises(dfbm.DfbError) as e:
        dfbm.restart_info(str(tmp_path / "missing.bin"))
    assert e.value.code == dfbm.ERR_IO


# ---- fingerprint ----
def _fp(shim, dfbm, cfg):
    c = dfbm.dfb_config()
    c.struct_bytes = C.sizeof(c)                       # what dfb_config_init sets
    c.grid_file_len = c.vel_fluc_file_len = c.line_file_len = -1
    c.device = -1
    keep = dfbm.fill_config(c, cfg)
    err = C.create_string_buffer(512)
    fp = shim.rs_fingerprint(C.byref(c), err, 512)
    del keep
    assert fp != 0, err.value
    return fp


def _explicit(W, Ny=96, Nz=160, per_cell=False):
    plane = W.plane_profile(Ny, Nz, 24, 10)
    rng = np.random.default_rng(5)
    shape = (3, Ny, Nz) if per_cell else (3, Ny)
    plane["N_y"] = rng.integers(1, 12, size=shape).astype(np.int32)
    plane["N_z"] = rng.integers(1, 10, size=shape).astype(np.int32)
    if per_cell:
        for k in ("yc", "dy", "dz"):
            plane[k] = np.repeat(np.asarray(plane[k])[:, None], Nz, axis=1)
    plane["explicit_N"] = True
    return plane


@pytest.mark.parametrize("per_cell", [False, True])
def test_fingerprint_changes_with_exactly_one_input(shim, dfbm, W, per_cell):
    base = _explicit(W, per_cell=per_cell)
    cfg = lambda p, **kw: dfbm.DFConfig.from_plane(p, **kw)          # noqa: E731
    fp0 = _fp(shim, dfbm, cfg(base))
    # what does not decide the numbers of the filter tables: seed, plane id, slab, kernel form
    assert _fp(shim, dfbm, cfg(base, seed=7, plane_id=3, k_begin=37, k_end=101, kernel_variant=1)) == fp0

    def changed(**edit):
        p = {k: (np.array(v, copy=True) if isinstance(v, np.ndarray) else v) for k, v in base.items()}
        for k, f in edit.items():
            f(p)
        return p

    def bump(name, idx, by):
        def f(p):
            p[name][idx] += by
        return f

    one_N = (1, 17, 23) if per_cell else (1, 17)
    variants = {
        "one N_y entry": changed(N_y=bump("N_y", one_N, 2)),
        "one N_z entry": changed(N_z=bump("N_z", one_N, 2)),
        "one row-table value": changed(rows=bump("rows", (4, 10), 1e-9)),
        "one Lt": changed(scales=bump("scales", (2, 2), 1e-9)),
    }
    fps = {k: _fp(shim, dfbm, cfg(p)) for k, p in variants.items()}
    fps["periodic_z"] = _fp(shim, dfbm, cfg(base, periodic_z=1))
    # Ny and Nz: the same plane one row shorter / 16 columns wider
    short = {k: v for k, v in base.items()}
    short["Ny"] = base["Ny"] - 1
    for k in ("yc", "dy", "dz"):
        short[k] = np.asarray(base[k])[:-1]
    short["rows"], short["N_y"], short["N_z"] = base["rows"][:, :-1], base["N_y"][:, :-1], base["N_z"][:, :-1]
    fps["Ny"] = _fp(shim, dfbm, cfg(short))
    if not per_cell:                                    # the same rows, 16 columns wider
        wide = W.plane_profile(96, 176, 24, 10)
        wide.update(N_y=base["N_y"], N_z=base["N_z"], explicit_N=True)
        fps["Nz"] = _fp(shim, dfbm, cfg(wide))
    for k, fp in fps.items():
        assert fp != fp0, k
    assert len(set(fps.values())) == len(fps)


# ---- writer records ----
def _cover(shim, v, recs, p0, p1, k0, k1):
    r = np.array([[a, b, c, d, e, np.uint64(f).view(np.int64) if isinstance(f, np.uint64) else f] for a, b, c, d, e, f in recs],
                 dtype=np.int64).reshape(-1, 6)
    vv, pv = i64(v)
    msg = C.create_string_buffer(512)
    rc = shim.rs_coverage(pv, len(recs), r.ctypes.data_as(I64), p0, p1, k0, k1, msg, 512)
    return rc == 0, msg.value.decode()


def test_records_accept_full_coverage_uneven_and_off_16_column_slabs(shim):
    v = header(Nz=96, plane0=10, nplanes=3, step=100, fp=77)
    for cuts in ([0, 96], [0, 48, 96], [0, 37, 61, 96], [0, 16, 17, 80, 96]):
        recs = [(10, 3, a, b, 100, 77) for a, b in zip(cuts[:-1], cuts[1:])]
        for p0, p1 in ((10, 13), (11, 12), (12, 13)):
            ok, msg = _cover(shim, v, recs[::-1], p0, p1, 0, 96)
            assert ok, (cuts, msg)


def test_records_accept_partial_coverage_of_the_loaders_columns(shim):
    v = header(Nz=96, step=100, fp=77)
    recs = [(10, 3, 0, 37, 100, 77)]
    assert _cover(shim, v, recs, 10, 13, 16, 37)[0]
    assert _cover(shim, v, recs, 10, 13, 0, 37)[0]
    ok, msg = _cover(shim, v, recs, 10, 13, 16, 48)
    assert not ok and "[37, 48)" in msg


def test_records_reject_gaps_stale_steps_and_foreign_fingerprints(shim):
    v = header(Nz=96, step=100, fp=77)
    ok, msg = _cover(shim, v, [(10, 3, 0, 32, 100, 77), (10, 3, 48, 96, 100, 77)], 10, 13, 0, 96)
    assert not ok and "[32, 48)" in msg and "no writer record" in msg
    ok, msg = _cover(shim, v, [], 10, 13, 0, 96)
    assert not ok and "[0, 96)" in msg
    ok, msg = _cover(shim, v, [(10, 3, 0, 48, 99, 77), (10, 3, 48, 96, 100, 77)], 10, 13, 0, 96)
    assert not ok and "stale" in msg and "[0, 48)" in msg and "99" in msg
    ok, msg = _cover(shim, v, [(10, 3, 0, 48, 100, 77), (10, 3, 48, 96, 100, 78)], 10, 13, 0, 96)
    assert not ok and "stale" in msg and "[48, 96)" in msg and "fingerprint" in msg
    # a stale record outside the loader's columns does not matter
    assert _cover(shim, v, [(10, 3, 0, 48, 100, 77), (10, 3, 48, 96, 99, 77)], 10, 13, 0, 48)[0]


# ---- offsets and a save by several writers ----
def test_segment_offsets_are_numpys_index_of_the_global_arrays(shim):
    P, Ny, Nz, L, R = 3, 5, 7, (4, 3, 2), 2
    v = header(Ny=Ny, Nz=Nz, nplanes=P, sections=7, lags=L, n_ring=R)
    vv, pv = i64(v)
    shapes = [(SEC_STATE, (3, P, Ny, Nz)), (SEC_STATS, (P, 6, Ny, Nz)), (SEC_CORR_Z, (P, 3, Ny, L[0] + 1)), (SEC_CORR_Y, (P, 3, Ny, L[1] + 1)),
              (SEC_CORR_T, (P, 3, Ny, L[2] + 1)), (SEC_RING, (R, P, 3, Ny, Nz))]
    base = DATA_AT
    rng = np.random.default_rng(0)
    for sec, shape in shapes:
        for _ in range(40):
            idx = tuple(int(rng.integers(0, s)) for s in shape)
            if sec == SEC_STATE:
                comp, plane, j, k = idx
            elif sec == SEC_STATS:
                plane, comp, j, k = idx
            elif sec == SEC_RING:
                i, plane, f, j, k = idx
                comp = 3 * i + f
            else:
                plane, comp, j, k = idx
            assert shim.rs_offset(pv, sec, comp, plane, j, k) == base + 8 * np.ravel_multi_index(idx, shape), (sec, idx)
        base += 8 * int(np.prod(shape))
    assert base == shim.rs_file_bytes(pv)


def _save(shim, path, v, record, blocks):
    """blocks: (section, comp, plane, rows [nrows, width], k0)"""
    desc = np.array([[s, c, p, r.shape[0], r.shape[1], k0] for s, c, p, r, k0 in blocks], dtype=np.int32)
    data = np.concatenate([np.ascontiguousarray(r, dtype=np.float64).ravel() for _, _, _, r, _ in blocks])
    vv, pv = i64(v)
    rr, pr = i64(record)
    err = C.create_string_buffer(512)
    rc = shim.rs_save(str(path).encode(), pv, pr, len(blocks), desc.ctypes.data_as(C.POINTER(C.c_int)), data.ctypes.data_as(C.POINTER(C.c_double)),
                      err, 512)
    return rc, err.value.decode()


def _read(shim, path):
    out, recs = np.zeros(30, dtype=np.int64), np.zeros((64, 6), dtype=np.int64)
    err = C.create_string_buffer(512)
    n = shim.rs_read(str(path).encode(), out.ctypes.data_as(I64), recs.ctypes.data_as(I64), 64, err, 512)
    return n, out, recs[:max(n, 0)], err.value.decode()


def test_slab_writers_fill_the_global_layout_and_info_reads_it(shim, dfbm, tmp_path):
    P, Ny, Nz = 2, 6, 40
    v = header(Ny=Ny, Nz=Nz, plane0=4, nplanes=P, step=50, sections=3, fp=99)
    state = np.random.default_rng(1).standard_normal((3, P, Ny, Nz))
    stats = np.random.default_rng(2).standard_normal((P, 6, Ny, Nz))
    path = tmp_path / "r.dfbr"
    cuts = [0, 13, 16, 40]                              # uneven, one cut off a 16-column boundary
    for a, b in zip(cuts[:-1], cuts[1:]):
        blocks = [(SEC_STATE, f, p, state[f, p, :, a:b], a) for f in range(3) for p in range(P)]
        blocks += [(SEC_STATS, s, p, stats[p, s, :, a:b], a) for p in range(P) for s in range(6)]
        assert _save(shim, path, v, [4, P, a, b, 50, 99], blocks) == (0, "")
    raw = np.fromfile(path, dtype="<f8", offset=DATA_AT)
    assert np.array_equal(raw[:state.size].reshape(state.shape), state)
    assert np.array_equal(raw[state.size:].reshape(stats.shape), stats)
    n, out, recs, _ = _read(shim, path)
    assert n == 3 and sorted(map(tuple, recs[:, 2:4])) == [(0, 13), (13, 16), (16, 40)]
    info = dfbm.restart_info(str(path))
    assert (info["Ny"], info["Nz"], info["plane_id"], info["nplanes"], info["step"], info["sections"], info["records"]) == (Ny, Nz, 4, P, 50, 3, 3)
    assert info["fingerprint"] == 99 and info["seed"] == 42 and info["bytes"] == os.path.getsize(path)
    assert [info[k] for k in ("Ny_max_u", "Ny_max_v", "Ny_max_w", "Nz_max_u", "Nz_max_v", "Nz_max_w")] == [6, 4, 6, 8, 8, 6]
    # the same writer again replaces its record; a save of another step clears the table
    assert _save(shim, path, v, [4, P, 0, 13, 50, 99], [(SEC_STATE, 0, 0, state[0, 0, :, :13], 0)])[0] == 0
    assert _read(shim, path)[0] == 3
    v2 = v.copy()
    v2[8] = 60
    assert _save(shim, path, v2, [4, P, 0, 13, 60, 99], [(SEC_STATE, 0, 0, state[0, 0, :, :13], 0)])[0] == 0
    n, out, recs, _ = _read(shim, path)
    assert n == 1 and out[8] == 60 and tuple(recs[0, 2:5]) == (0, 13, 60)


def test_truncated_file_is_an_io_error(shim, dfbm, tmp_path):
    v = header(Ny=4, Nz=16, nplanes=1, step=5)
    path = tmp_path / "t.dfbr"
    assert _save(shim, path, v, [10, 1, 0, 16, 5, int(v[11])], [(SEC_STATE, f, 0, np.ones((4, 16)), 0) for f in range(3)])[0] == 0
    os.truncate(path, os.path.getsize(path) - 8)
    n, _, _, err = _read(shim, path)
    assert n == -2 and "truncated" in err
    with pytest.raises(dfbm.DfbError) as e:
        dfbm.restart_info(str(path))
    assert e.value.code == dfbm.ERR_IO
    os.truncate(path, 100)
    assert _read(shim, path)[0] == -2
