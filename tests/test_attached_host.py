"""Attached steps without a GPU: the noise positions the advance kernel computes on the device are the host's own (one shared function,
compiled here for the host) and are the pcg32 stream's; the new entry points are exported; the capture program and its by-reference
(Fortran) mode compile and link; the facades bind the calls."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from oracle_harness import package
from shims import build_shim

LIBDIR = os.path.join(ROOT, "digital-filtering_b200", "lib")
MASK64 = (1 << 64) - 1
MULT = 6364136223846793005


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    L = build_shim(tmp_path_factory, "noise_states", "stepplan.cpp")
    L.ns_states.restype = C.c_int
    u64 = C.POINTER(C.c_ulonglong)
    ip = C.POINTER(C.c_int)
    L.ns_states.argtypes = [C.c_void_p, C.c_int, C.c_ulonglong, C.c_int, C.c_longlong, ip, ip, u64, u64, u64, u64, C.c_char_p, C.c_int]
    return L


def states(L, dfbm, config, nplanes, seed, plane_id, step):
    c = dfbm.dfb_config()
    c.struct_bytes = C.sizeof(c)
    c.grid_file_len = c.vel_fluc_file_len = c.line_file_len = -1
    c.device = -1
    keep = dfbm.fill_config(c, config)
    field, kind = np.zeros(6, np.int32), np.zeros(6, np.int32)
    npairs = np.zeros(6, np.uint64)
    hs, hi, ds = (np.zeros(16 * 6, np.uint64) for _ in range(3))
    err = C.create_string_buffer(512)
    u64 = lambda a: a.ctypes.data_as(C.POINTER(C.c_ulonglong))     # noqa: E731
    ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int))            # noqa: E731
    n = L.ns_states(C.byref(c), nplanes, seed, plane_id, step, ip(field), ip(kind), u64(npairs), u64(hs), u64(hi), u64(ds), err, 512)
    del keep
    assert n > 0, err.value
    return n, field, kind, npairs, hs.reshape(16, 6), hi.reshape(16, 6), ds.reshape(16, 6)


def xsh_rr(s):
    x = (((s >> 18) ^ s) >> 27) & 0xFFFFFFFF
    r = s >> 59
    return ((x >> r) | (x << ((32 - r) & 31))) & 0xFFFFFFFF


@pytest.mark.parametrize("nplanes,periodic,k", [(1, 0, None), (4, 0, None), (1, 1, None), (3, 1, None), (1, 0, (40, 88))])
def test_shared_noise_positions_match_the_stream(shim, W, O, nplanes, periodic, k):
    """For random steps up to 2^40: the host's states (fill_noise_states, what a host-driven step uses) equal the device function's
    (noise_step_state, what step_advance_kernel evaluates), and the first draws from them are the oracle's pcg32 draws of
    (seed, stream ((plane*3 + field)*2 + kind)) advanced by 4 * step * pairs -- batches, periodic planes and slabs."""
    dfbm = package()
    kw = dict(periodic_z=periodic)
    if k:
        kw.update(k_begin=k[0], k_end=k[1])
    cfg = dfbm.DFConfig.from_plane(W.plane_profile(64, 128, 8, 6), **kw)
    rng = np.random.default_rng(nplanes * 10 + periodic)
    steps = [0, 1, 2, (1 << 40) - 1, 1 << 40] + [int(s) for s in rng.integers(0, 1 << 40, 6)]
    for step in steps:
        seed, plane_id = int(rng.integers(0, 1 << 63)), int(rng.integers(0, 50))
        n, field, kind, npairs, hs, hi, ds = states(shim, dfbm, cfg, nplanes, seed, plane_id, step)
        assert np.array_equal(hs[:nplanes, :n], ds[:nplanes, :n])
        for p in range(nplanes):
            for a in range(n):
                stream = ((plane_id + p) * 3 + int(field[a])) * 2 + int(kind[a])
                assert int(hi[p, a]) == ((stream << 1) | 1) & MASK64
                s0 = int(hs[p, a])
                s1 = (s0 * MULT + int(hi[p, a])) & MASK64
                delta = (4 * step * int(npairs[a])) & MASK64
                ref = O.pcg32_draw(seed, stream, delta, 2)
                assert [xsh_rr(s0), xsh_rr(s1)] == [int(v) for v in ref], (step, p, a)


def test_new_entry_points_are_exported(dfb):
    L = dfb.lib()
    for name in ("dfb_attach_stream", "dfb_filter_dev", "dfb_attach_stream_f", "dfb_filter_dev_f"):
        assert hasattr(L, name), name
    h = dfb.lib().dfb_filter_dev(None, None)
    assert h == dfb.ERR_ARG


@pytest.fixture(scope="module")
def capture_bin(dfb, tmp_path_factory):
    out = str(tmp_path_factory.mktemp("attached_capture"))          # a temporary directory: the tree may be read-only
    exe = os.path.join(out, "attached_capture_test")
    subprocess.run(["/usr/bin/gcc", "-std=c11", "-Wall", os.path.join(ROOT, "tests", "attached_capture_test.c"),
                    "-I" + os.path.join(ROOT, "include"), "-I/usr/local/cuda/include", "-L" + LIBDIR, "-ldfb200",
                    "-Wl,-rpath," + LIBDIR, "-L/usr/local/cuda/lib64", "-lcudart", "-Wl,-rpath,/usr/local/cuda/lib64", "-o", exe],
                   check=True, capture_output=True)
    return exe


def test_capture_program_compiles_and_links(capture_bin):
    assert os.path.exists(capture_bin)


def test_facades_bind_the_attached_calls():
    f = open(os.path.join(ROOT, "fortran", "digital_filtering.f90")).read()
    for name in ("dfb_attach_stream_f", "dfb_filter_dev_f"):
        assert f"bind(C, name='{name}')" in f
    assert "public :: attach_stream, filter_dev" in f
    hpp = open(os.path.join(ROOT, "include", "digital_filter.hpp")).read()
    assert "dfb_attach_stream(h_, stream)" in hpp and "dfb_filter_dev(h_, dt_dev)" in hpp
