"""Pins the plain-C restatement (oracle/df_oracle.c) -- CPU only.
  * against the committed golden fixtures generated from the reference's own object code
    (tests/golden/make_golden.py), always;
  * against that object code live (oracle/_ref/libdfref.so), when it is present."""
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, default_plane


def test_default_plane_tables_match_golden(O):
    if not O.have_ref():
        pytest.skip("default-plane setup needs the data files under oracle/_ref")
    g = np.load(os.path.join(GOLDEN, "default_tables.npz"))
    P = O.default_plane()
    assert (P["Ny"], P["Nz"]) == (int(g["Ny"]), int(g["Nz"])) == (510, 400)
    assert np.array_equal(P["rows"], g["rows"]) and np.array_equal(P["scales"], g["scales"])
    assert np.array_equal(P["yc"], g["yc"]) and np.array_equal(P["dy"], g["dy"])
    assert np.array_equal(P["N_y"][:, :, 0], g["N_y"]) and np.array_equal(P["N_z"][:, :, 0], g["N_z"])
    assert list(P["Ny_max"]) == list(g["Ny_max"]) == [212, 160, 212] and list(P["Nz_max"]) == list(g["Nz_max"]) == [6, 4, 6]
    assert P["u_tau"] == float(g["u_tau"]) and P["tau_w"] == float(g["tau_w"])


def test_small_plane_three_steps_match_golden_bitwise(O, W):
    g = np.load(os.path.join(GOLDEN, "small_step.npz"))
    plane = dict(Ny=int(g["Ny"]), Nz=int(g["Nz"]), d_i=float(g["d_i"]), yc=g["yc"], dy=g["dy"], dz=g["dz"], rows=g["rows"], scales=g["scales"])
    O.half_widths(plane)
    assert np.array_equal(plane["N_y"][:, :, 0], g["N_y"]) and np.array_equal(plane["N_z"][:, :, 0], g["N_z"])
    fo = np.zeros((3, plane["Ny"], plane["Nz"]))
    T = rho = None
    for s, dt in enumerate(g["dts"]):
        rys = [g[f"s{s}_rys{f}"] for f in range(3)]
        hal = [g[f"s{s}_halo{f}"] for f in range(3)]
        # the committed noise itself is the oracle's counter-based stream
        for f in range(3):
            assert np.array_equal(rys[f], O.noise_rys(int(g["seed"]), 0, f, s, plane["Ny"], plane["Ny_max"][f], plane["Nz"]))
            assert np.array_equal(hal[f], O.noise_halo(int(g["seed"]), 0, f, s, plane["Ny"], plane["Nz_max"][f]))
        o = O.step(plane, rys, hal, fo, float(dt), first_step=(s == 0))
        fo = o["filt_old"]
        assert np.array_equal(o["filt"], g[f"s{s}_filt"]) and np.array_equal(o["fluc"], g[f"s{s}_fluc"])
        if s > 0:
            assert np.array_equal(o["T"], g[f"s{s}_T"]) and np.array_equal(o["rho"], g[f"s{s}_rho"])


def test_default_plane_step_digest(O):
    d = json.load(open(os.path.join(GOLDEN, "default_step_digest.json")))
    P = default_plane()
    # the half-widths the restatement derives from the stored geometry are the reference's own (default_tables.npz)
    G = O.half_widths(dict(P))
    assert np.array_equal(G["N_y"], P["N_y"]) and np.array_equal(G["N_z"], P["N_z"])
    assert G["Ny_max"] == P["Ny_max"] == [212, 160, 212] and G["Nz_max"] == P["Nz_max"] == [6, 4, 6]
    Ny, Nz, seed = P["Ny"], P["Nz"], d["seed"]
    rys = [O.noise_rys(seed, 0, f, 1, Ny, P["Ny_max"][f], Nz) for f in range(3)]
    hal = [O.noise_halo(seed, 0, f, 1, Ny, P["Nz_max"][f]) for f in range(3)]
    fo = [O.noise_elements(seed, 100 + f, 0, Ny * Nz, 0, Ny * Nz).reshape(Ny, Nz) for f in range(3)]
    o = O.step(P, rys, hal, fo, d["dt"])
    for k, rec in d["outputs"].items():
        assert hashlib.sha256(np.ascontiguousarray(o[k]).tobytes()).hexdigest() == rec["sha256"], k


def test_coefficients_unit_energy_and_symmetry(O):
    for N in (2, 4, 6, 28, 128, 212):
        b = O.coeffs(N)
        assert len(b) == 2 * N + 1 and np.array_equal(b, b[::-1])
        assert abs(np.sum(b * b) - 1.0) < 1e-14        # df.cpp:168-177: sum b^2 = 1


def test_interpolate_clamps_like_reference(O):
    y, f = np.array([0.0, 1.0, 3.0]), np.array([10.0, 20.0, 0.0])
    out = O.linear_interpolate(y, f, np.array([-1.0, 0.0, 0.5, 1.0, 2.0, 3.0, 9.0]))
    assert np.array_equal(out, [10.0, 10.0, 15.0, 20.0, 10.0, 0.0, 0.0])


# ---------------------------------------------------------------------------------------------
# live reference object code
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ref(O):
    if not O.have_ref():
        pytest.skip("oracle/_ref not built")
    r = O.RefFilter()
    yield r
    r.close()


def test_live_default_plane(O, ref):
    P, RP = O.default_plane(), ref.plane()
    for k in ("rows", "scales", "N_y", "N_z"):
        assert np.array_equal(np.asarray(P[k]), np.asarray(RP[k])), k
    by, off, Ns = ref.fvec(0, "by"), ref.ivec(0, "by_offsets"), ref.ivec(0, "N_ys")
    bz, offz, Nzs = ref.fvec(1, "bz"), ref.ivec(1, "bz_offsets"), ref.ivec(1, "N_zs")
    for idx in (0, 399, 400, 77777, 203999):
        assert np.array_equal(by[off[idx] - Ns[idx]:off[idx] + Ns[idx] + 1], O.coeffs(int(Ns[idx])))
        assert np.array_equal(bz[offz[idx] - Nzs[idx]:offz[idx] + Nzs[idx] + 1], O.coeffs(int(Nzs[idx])))


def test_live_replay_of_the_real_filter_call(O, ref):
    """DIGITAL_FILTER::filter(dt) itself (its own random_device-seeded noise, df.cpp:449-468):
    capture filt_old before, read back the noise it drew, replay through the restatement."""
    P = ref.plane()
    fo = ref.outputs()["filt_old"].copy()
    ref.filter(1e-5)
    rys = [ref.fvec(f, "r_ys").reshape(-1, P["Nz"]) for f in range(3)]
    o = O.step(P, rys, ref.halos(), fo, 1e-5)
    r = ref.outputs()
    for k in ("filt", "fluc", "filt_old", "T", "rho"):
        assert np.array_equal(o[k], r[k]), k


def test_live_synthetic_shape(O, W, ref):
    plane = W.plane_profile(64, 48, 16, 12)
    r2 = O.RefFilter()
    try:
        r2.reshape(plane)
        RP = r2.plane()
        O.half_widths(plane)
        assert np.array_equal(plane["N_y"], RP["N_y"]) and np.array_equal(plane["N_z"], RP["N_z"])
        rys = [O.noise_rys(3, 0, f, 0, 64, plane["Ny_max"][f], 48) for f in range(3)]
        hal = [O.noise_halo(3, 0, f, 0, 64, plane["Nz_max"][f]) for f in range(3)]
        fo = np.stack([O.noise_elements(3, 50 + f, 0, 64 * 48, 0, 64 * 48).reshape(64, 48) for f in range(3)])
        r2.inject(rys, hal, fo)
        r2.step_injected(3e-7)
        o, r = O.step(plane, rys, hal, fo, 3e-7), r2.outputs()
        for k in ("filt", "fluc", "filt_old", "T", "rho"):
            assert np.array_equal(o[k], r[k]), k
    finally:
        r2.close()
