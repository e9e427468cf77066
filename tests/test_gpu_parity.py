"""Parity of the CUDA path (through the C ABI) against the CPU checkers -- needs a B200 (-m gpu).

Gates of north_star:
  G1  random field bit-exact against the host pcg32 jump-ahead restatement;
  G2  given identical noise, filtered + scaled fields within 1e-12 of the reference's filter()
      (normwise form, SURVEY section 7: |d| <= 1e-12 * max(|ref|, rms(ref)));
  G3  output Reynolds stresses match the target RST within a stated sampling tolerance.
Nothing here reads /root/reference: the checkers are oracle/libdforacle.so (restatement, pinned
by the CPU tests) and, when it travelled with the snapshot, oracle/_ref/libdfref.so (the reference's
own object code).
"""
import os

import numpy as np
import pytest

from conftest import GOLDEN, default_plane, normwise_close

pytestmark = pytest.mark.gpu
TOL = 1e-12


def inject_and_step(dfb, O, plane, variant, seed, dts, check_first=True):
    """Runs constructor step + len(dts) filter steps in inject mode on the GPU and through the oracle
    restatement with the same (counter-based) noise; returns worst normwise ratio per output."""
    cfg = dfb.DFConfig.from_plane(plane, noise_mode=dfb.NOISE_INJECT, kernel_variant=variant)
    df = dfb.DIGITAL_FILTER(cfg)
    O.half_widths(plane)
    Ny, Nz = plane["Ny"], plane["Nz"]
    for f in range(3):
        assert np.array_equal(df.half_widths(f, 0), plane["N_y"][f]) and np.array_equal(df.half_widths(f, 1), plane["N_z"][f])
    fo = np.zeros((3, Ny, Nz))
    worst = {}
    for s, dt in enumerate([0.0] + list(dts)):
        rys = [O.noise_rys(seed, 0, f, s, Ny, plane["Ny_max"][f], Nz) for f in range(3)]
        hal = [O.noise_halo(seed, 0, f, s, Ny, plane["Nz_max"][f]) for f in range(3)]
        for f in range(3):
            df.set_noise(f, rys[f], hal[f])
        if s == 0:
            df.first_step()
        else:
            df.filter(dt)
        df.fetch()
        o = O.step(plane, rys, hal, fo, dt, first_step=(s == 0))
        fo = o["filt_old"]
        got = dict(filt=np.stack([df.u.filt, df.v.filt, df.w.filt]), fluc=np.stack([df.u.fluc, df.v.fluc, df.w.fluc]),
                   T=df.T_fluc, rho=df.rho_fluc)
        for k in ("filt", "fluc", "T", "rho"):
            if s == 0 and k in ("T", "rho"):
                assert not got[k].any()          # SURVEY quirk 3: T', rho' stay 0 after the constructor
                continue
            for f in range(3) if k in ("filt", "fluc") else [None]:
                a, b = (got[k][f], o[k][f]) if f is not None else (got[k], o[k])
                ok, r = normwise_close(a, b, TOL)
                worst[k] = max(worst.get(k, 0.0), r)
                assert ok, (plane["name"], variant, s, k, f, r)
    df.close()
    return worst


# ---------------------------------------------------------------------------------------------
# G1: RNG
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(40, 36, 8, 6), (33, 51, 6, 4), (64, 130, 16, 12)])
def test_G1_noise_bit_exact(dfb, O, W, shape):
    plane = W.plane_profile(*shape)
    df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=42, plane_id=9))
    Ny, Nz = plane["Ny"], plane["Nz"]
    for step in (0, 1, 7, 123456):
        df.generate_noise(step)
        for f in range(3):
            r_ys, halo = df.get_noise(f)
            F = (df.u, df.v, df.w)[f]
            assert np.array_equal(r_ys, O.noise_rys(42, 9, f, step, Ny, F.Ny_max, Nz)), (step, f)
            assert np.array_equal(halo, O.noise_halo(42, 9, f, step, Ny, F.Nz_max)), (step, f)
    df.close()


def test_G1_noise_bit_exact_default_plane_size(dfb, O, W):
    plane = W.plane_profile(510, 400, 212, 6)
    df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=20261018))
    df.generate_noise(3)
    r_ys, halo = df.get_noise(0)
    assert np.array_equal(r_ys, O.noise_rys(20261018, 0, 0, 3, 510, df.u.Ny_max, 400))
    assert np.array_equal(halo, O.noise_halo(20261018, 0, 0, 3, 510, df.u.Nz_max))
    assert abs(r_ys.mean()) < 5e-3 and abs(r_ys.var() - 1) < 6e-3
    df.close()


# ---------------------------------------------------------------------------------------------
# G2: filtered / scaled fields under identical noise
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", [0, 1], ids=["tuned", "simple"])
@pytest.mark.parametrize("shape", [(40, 36, 8, 6), (37, 45, 10, 4), (72, 530, 20, 16), (130, 1100, 40, 34)])
def test_G2_profile_planes(dfb, O, W, shape, variant):
    inject_and_step(dfb, O, W.plane_profile(*shape), variant, seed=5, dts=[2e-7, 9e-7])


@pytest.mark.parametrize("variant", [0, 1], ids=["tuned", "simple"])
def test_G2_saturated_plane(dfb, O, W, variant):
    inject_and_step(dfb, O, W.plane_saturated(48, 600, 32), variant, seed=6, dts=[3e-7])


@pytest.mark.parametrize("zmode", ["1", "0"], ids=["z-recursive", "z-direct"])
def test_G2_both_forms_of_the_z_sweep(dfb, O, W, monkeypatch, zmode):
    """The tuned z-sweep has two forms (DESIGN section 5): the recursive evaluation of the exponential window (default) and the
    direct Toeplitz sum (slabs cut off a 16-column boundary, N = 0 rows, DFB_Z_MODE=0).  Both must pass the same gate, at N = 128
    and on a plane wide enough for several 512-column strips; the recursive form must also stay well inside it (1e-13)."""
    monkeypatch.setenv("DFB_Z_MODE", zmode)
    plane = W.plane_profile(72, 1100, 128, 128)
    df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, noise_mode=dfb.NOISE_INJECT))
    assert df.tuned and df.info(7) == int(zmode)
    df.close()
    worst = inject_and_step(dfb, O, plane, 0, seed=15, dts=[2e-7, 1e-6])
    assert max(worst.values()) < 1e-13, worst


def test_G2_ragged_per_cell_half_widths(dfb, O, W):
    plane = W.plane_ragged(48, 64, 12, seed=3)
    cfg = dfb.DFConfig.from_plane(plane, noise_mode=dfb.NOISE_INJECT)
    df = dfb.DIGITAL_FILTER(cfg)
    assert not df.tuned                       # not row-uniform -> the general kernels
    df.close()
    inject_and_step(dfb, O, plane, 0, seed=8, dts=[4e-7])


def test_G2_golden_small_plane_from_reference_object_code(dfb, O):
    """committed fixture generated from the reference's own df.cpp (tests/golden/make_golden.py)"""
    g = np.load(os.path.join(GOLDEN, "small_step.npz"))
    plane = dict(name="golden", Ny=int(g["Ny"]), Nz=int(g["Nz"]), d_i=float(g["d_i"]), yc=g["yc"], dy=g["dy"], dz=g["dz"],
                 rows=g["rows"], scales=g["scales"])
    for variant in (0, 1):
        df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, noise_mode=dfb.NOISE_INJECT, kernel_variant=variant))
        for s, dt in enumerate(g["dts"]):
            for f in range(3):
                df.set_noise(f, g[f"s{s}_rys{f}"], g[f"s{s}_halo{f}"])
            df.first_step() if s == 0 else df.filter(float(dt))
            df.fetch()
            for f, F in enumerate((df.u, df.v, df.w)):
                assert normwise_close(F.filt, g[f"s{s}_filt"][f], TOL)[0]
                assert normwise_close(F.fluc, g[f"s{s}_fluc"][f], TOL)[0]
            if s > 0:
                assert normwise_close(df.T_fluc, g[f"s{s}_T"], TOL)[0] and normwise_close(df.rho_fluc, g[f"s{s}_rho"], TOL)[0]
        df.close()


def _default_plane_reference_step(dfb, O):
    """The reference's default plane from its stored setup tables, and the one injected step whose reference outputs
    tests/golden/default_step_digest.json records (sha256 + probes, tests/golden/make_golden.py): noise of step 1 and filt_old
    from the oracle's counter-based stream (seed 20261018), dt = 1e-5.  The oracle's output of that step is checked against the
    reference's sha256 here, so what the GPU is compared with below is the reference's own output, bit for bit.
    Returns (df after the step, oracle output, plane, digest)."""
    import hashlib
    import json
    d = json.load(open(os.path.join(GOLDEN, "default_step_digest.json")))
    P = default_plane()
    Ny, Nz, seed = P["Ny"], P["Nz"], d["seed"]
    rys = [O.noise_rys(seed, 0, f, 1, Ny, P["Ny_max"][f], Nz) for f in range(3)]
    hal = [O.noise_halo(seed, 0, f, 1, Ny, P["Nz_max"][f]) for f in range(3)]
    fo = np.stack([O.noise_elements(seed, 100 + f, 0, Ny * Nz, 0, Ny * Nz).reshape(Ny, Nz) for f in range(3)])
    o = O.step(P, rys, hal, fo, d["dt"])
    for k, rec in d["outputs"].items():
        assert hashlib.sha256(np.ascontiguousarray(o[k]).tobytes()).hexdigest() == rec["sha256"], k
    df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(P, noise_mode=dfb.NOISE_INJECT))
    df.set_state(fo, 1)
    for f in range(3):
        df.set_noise(f, rys[f], hal[f])
    df.filter(d["dt"])
    df.fetch()
    return df, o, P, d


def test_G2_default_plane_against_reference_object_code(dfb, O):
    """config 1: the reference's own default plane (its setup tables, stored) and one step of its filter() on stored-noise
    inputs whose outputs are recorded from the reference's object code: setup tables, half-widths, coefficients and all
    five outputs on the GPU against them."""
    df, o, P, d = _default_plane_reference_step(dfb, O)
    assert (df.Ny, df.Nz) == (510, 400)
    assert np.array_equal(df.rows(), P["rows"])
    for f in range(3):
        assert np.array_equal(df.half_widths(f, 0), P["N_y"][f]) and np.array_equal(df.half_widths(f, 1), P["N_z"][f])
    for N in (2, 6, 28, 212):
        assert np.array_equal(df.table(11, N), O.coeffs(N))
    assert np.array_equal(df.table(10), P["scales"][:, 2])
    got = dict(filt=np.stack([df.u.filt, df.v.filt, df.w.filt]), fluc=np.stack([df.u.fluc, df.v.fluc, df.w.fluc]), T=df.T_fluc, rho=df.rho_fluc)
    for k, rec in d["outputs"].items():
        for f in range(3 if k in ("filt", "fluc") else 1):
            ok, ratio = normwise_close(got[k][f] if k in ("filt", "fluc") else got[k], o[k][f] if k in ("filt", "fluc") else o[k], TOL)
            assert ok, (k, f, ratio)
        probe = got[k].ravel()[[0, 12345, 99999, got[k].size - 1]]   # the reference's values at the recorded cells
        assert np.all(np.abs(probe - rec["probe"]) <= TOL * np.maximum(np.abs(rec["probe"]), rec["rms"])), (k, probe, rec["probe"])
    df.close()


def test_G2_generate_mode_equals_oracle_on_the_same_stream(dfb, O, W):
    """generate mode end to end: device noise (G1) + device filter == oracle noise + oracle filter"""
    plane = W.plane_profile(96, 200, 24, 10)
    df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=77))
    O.half_widths(plane)
    Ny, Nz = 96, 200
    fo = np.zeros((3, Ny, Nz))
    for s, dt in enumerate([0.0, 1e-7, 1e-7, 3e-7]):
        if s > 0:
            df.filter(dt)
        else:
            df.fetch()
        rys = [O.noise_rys(77, 0, f, s, Ny, plane["Ny_max"][f], Nz) for f in range(3)]
        hal = [O.noise_halo(77, 0, f, s, Ny, plane["Nz_max"][f]) for f in range(3)]
        o = O.step(plane, rys, hal, fo, dt, first_step=(s == 0))
        fo = o["filt_old"]
        for f, F in enumerate((df.u, df.v, df.w)):
            ok, r = normwise_close(F.fluc, o["fluc"][f], TOL)
            assert ok, (s, f, r)
    assert df.step == 4
    df.close()


# ---------------------------------------------------------------------------------------------
# slabs, state, properties at full size
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ymode", [None, "1"], ids=["y-default", "y-recursive"])
def test_slabs_reproduce_the_whole_plane_bitwise(dfb, W, monkeypatch, ymode):
    """Slabs whose first column is a multiple of 16 plane columns (what parallel.slab_bounds produces) reproduce the whole plane
    bit for bit, ragged widths included; a slab cut anywhere else takes the direct-form z-sweep and agrees to the G2 tolerance."""
    if ymode is not None:
        monkeypatch.setenv("DFB_Y_MODE", ymode)          # the recursive y kernel must be slab-invariant too (per-column arithmetic)
    plane = W.plane_profile(64, 700, 16, 24) if ymode is None else W.plane_profile(96, 700, 48, 24)
    whole = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=3))
    whole.filter(2e-7); whole.filter(2e-7)
    fields = lambda d: (d.u.fluc, d.v.fluc, d.w.fluc, d.T_fluc, d.rho_fluc)
    for k0, k1 in [(0, 160), (160, 176), (176, 400), (400, 700), (0, 700)]:
        part = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=3, k_begin=k0, k_end=k1))
        part.filter(2e-7); part.filter(2e-7)
        assert (part.Ny, part.Nz) == (plane["Ny"], k1 - k0)
        for a, b in zip(fields(part), fields(whole)):
            assert np.array_equal(a, b[:, k0:k1]), (k0, k1)
        part.close()
    for k0, k1 in [(150, 151), (151, 401), (400, 699), (699, 700)]:
        part = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=3, k_begin=k0, k_end=k1))
        part.filter(2e-7); part.filter(2e-7)
        for a, b in zip(fields(part), fields(whole)):
            ref = b[:, k0:k1]
            assert np.all(np.abs(a - ref) <= TOL * np.maximum(np.abs(ref), np.sqrt(np.mean(b * b)))), (k0, k1)
        part.close()
    whole.close()


def test_checkpoint_resume(dfb, W):
    plane = W.plane_profile(40, 64, 8, 6)
    a = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=11))
    for _ in range(3):
        a.filter(1e-7)
    fo, step = a.get_state()
    a.filter(2e-7)
    b = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=11, skip_first_step=1))
    b.set_state(fo, step)
    b.filter(2e-7)
    assert step == 4 and np.array_equal(a.u.fluc, b.u.fluc) and np.array_equal(a.rho_fluc, b.rho_fluc)
    # rewinding the SAME handle to the step it just finished must not see stale u->v completion stamps
    keep_v = a.v.fluc.copy()
    a.set_state(fo, step)
    a.filter(2e-7)
    assert np.array_equal(a.v.fluc, keep_v)
    a.close(); b.close()


def test_inject_mode_requires_noise(dfb, W):
    df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(W.plane_profile(40, 36, 8, 6), noise_mode=dfb.NOISE_INJECT))
    with pytest.raises(dfb.DfbError) as e:
        df.filter(1e-7)
    assert e.value.code == dfb.ERR_STATE
    df.close()


def test_dns_statistics_file_layout(dfb, default_data, tmp_path):
    """N1: the Fortran caller's configuration (vel_file_offset = 142 header lines + the DNS statistics
    layout, fortran-main.f90:17-19) gives the same tables as the preprocessed RST.dat (RST.cpp:43-50)."""
    RST_DAT, LINE_DAT = str(default_data / "files" / "RST.dat"), str(default_data / "line.dat")
    rst = [ln.split() for ln in open(RST_DAT).read().splitlines()[2:] if ln.strip()]
    stat = tmp_path / "Stat.dat"
    with open(stat, "w") as fh:
        for i in range(142):
            fh.write("# header line %d\n" % i)
        for r in rst:
            cols = ["0"] * 20
            cols[0], cols[1], cols[8], cols[10], cols[9], cols[15] = r[0], r[1], r[2], r[3], r[4], r[5]
            fh.write(" ".join(cols) + "\n")
    a = dfb.DIGITAL_FILTER(dfb.DFConfig(vel_fluc_file=RST_DAT, line_file=LINE_DAT, seed=1))
    b = dfb.DIGITAL_FILTER(dfb.DFConfig(vel_fluc_file=str(stat), line_file=LINE_DAT, seed=1, vel_file_offset=142, vel_file_N_values=330))
    assert (a.Ny, a.Nz) == (b.Ny, b.Nz) == (510, 400)
    assert np.array_equal(a.rows(), b.rows())
    assert np.array_equal(a.u.fluc, b.u.fluc)
    a.close(); b.close()


def test_missing_file_is_an_io_status(dfb):
    with pytest.raises(dfb.DfbError) as e:
        dfb.DIGITAL_FILTER(dfb.DFConfig(vel_fluc_file="/nonexistent/RST.dat"))
    assert e.value.code == dfb.ERR_IO


def test_full_size_properties_1024x2048(dfb, W):
    """BASELINE size (config 3a): size-independent properties instead of a CPU run.
    linearity: filter(2*noise) == 2*filter(noise) exactly (power-of-two scaling commutes with fp64
    rounding); unit variance of the filtered field (sum b^2 = 1); simple == tuned kernels."""
    plane = W.NAMED["1024x2048_profile_N128"]()
    rng = np.random.default_rng(0)
    cfg = dfb.DFConfig.from_plane(plane, noise_mode=dfb.NOISE_INJECT)
    df = dfb.DIGITAL_FILTER(cfg)
    noise = []
    for f, F in enumerate((df.u, df.v, df.w)):
        noise.append((rng.standard_normal((1024 + 2 * F.Ny_max, 2048)), rng.standard_normal((1024, 2 * F.Nz_max))))
        df.set_noise(f, *noise[f])
    df.first_step()
    df.fetch()
    base = [F.filt.copy() for F in (df.u, df.v, df.w)]
    for b in base:
        assert abs(b.var() - 1.0) < 0.05 and abs(b.mean()) < 0.2
    for f in range(3):
        df.set_noise(f, 2.0 * noise[f][0], 2.0 * noise[f][1])
    df.first_step()
    df.fetch()
    for b, F in zip(base, (df.u, df.v, df.w)):
        assert np.array_equal(F.filt, 2.0 * b)
    df.close()
    ds = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, noise_mode=dfb.NOISE_INJECT, kernel_variant=1))
    for f in range(3):
        ds.set_noise(f, *noise[f])
    ds.first_step()
    ds.fetch()
    for b, F in zip(base, (ds.u, ds.v, ds.w)):
        ok, r = normwise_close(F.filt, b, TOL)
        assert ok, r
    ds.close()


# ---------------------------------------------------------------------------------------------
# G3: Reynolds stresses
# ---------------------------------------------------------------------------------------------
def test_G3_reynolds_stresses_recovered(dfb, W):
    """The reference's only validation (get_rms, df.cpp:584-611), automated: time-average u'u',
    v'v', w'w', u'v' over steps and the spanwise direction, compare row-wise with the target RST.
    Stated sampling tolerance: 400 decorrelated steps x 400 columns with a spanwise correlation
    length of ~13 cells give n_eff ~ 12 000 per row: relative sampling noise ~ (2/n_eff)^0.5 = 1.3 %
    for the diagonal terms and ~ ((R11 R22 / R21^2 + 1)/n_eff)^0.5 = 2.5 % for u'v'.  Gates: diagonal
    median < 2 %, p95 < 6 %, max < 12 %; shear median < 4 %, p95 < 10 %, max < 16 %.  (The reference
    itself measured median 0.5 %, max 2-3 % with 100 x 400 samples, BASELINE.md section 2.)"""
    plane = W.plane_profile(128, 400, 24, 6)
    df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=2026), fetch=False)
    rows = plane["rows"]
    acc = np.zeros((4, 128))
    n = 400
    for _ in range(n):
        df.filter(1e-5)          # dt >> Lt: consecutive fields are decorrelated (alpha ~ 0)
        u, v, w = df.get(dfb.U_FLUC), df.get(dfb.V_FLUC), df.get(dfb.W_FLUC)
        acc += np.stack([(u * u).mean(1), (v * v).mean(1), (w * w).mean(1), (u * v).mean(1)])
    acc /= n
    for i, (name, tgt) in enumerate((("R11", rows[0]), ("R22", rows[2]), ("R33", rows[3]), ("R21", rows[1]))):
        rel = np.abs(acc[i] - tgt) / np.abs(tgt)
        lim = (0.04, 0.10, 0.16) if name == "R21" else (0.02, 0.06, 0.12)
        got = (float(np.median(rel)), float(np.percentile(rel, 95)), float(rel.max()))
        assert got[0] < lim[0] and got[1] < lim[1] and got[2] < lim[2], (name, got)
    df.close()


# ---------------------------------------------------------------------------------------------
# "next" rows: N2 running statistics, N4 CSV writer
# ---------------------------------------------------------------------------------------------
def test_N2_running_statistics_match_rms_add(dfb, W):
    """rms_add / plot_rms (df.cpp:571-621) on the device: per-cell sums of squares accumulated step by step
    equal the same accumulation done on the host from the fetched fields, bit for bit."""
    plane = W.plane_profile(40, 96, 8, 6)
    df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=4))
    df.stats_enable(True)
    acc = np.zeros((6, 40, 96))
    for _ in range(7):
        df.filter(3e-7)
        f = [df.u.fluc, df.v.fluc, df.w.fluc, df.T_fluc, df.rho_fluc]
        for i in range(5):
            acc[i] += f[i] * f[i]
        acc[5] += f[0] * f[1]
    for i in range(6):
        got, cnt = df.stats(i)
        assert cnt == 7 and np.array_equal(got, acc[i]), i
    rms, _ = df.stats(0, rms=True)
    assert np.array_equal(rms, np.sqrt(acc[0] / 7))
    df.close()


def test_N4_csv_matches_reference_writer(dfb, O, tmp_path):
    """write_csv (df.cpp:764-803): same header, same fixed 15-decimal format, the reference's cell-centre coordinates
    (df.cpp:776-786 on its own grid, read_grid df.cpp:71-118) and, within the fp64 gate, the reference's outputs of the
    stored default-plane step (_default_plane_reference_step)."""
    import ctypes as C
    df, o, P, _ = _default_plane_reference_step(dfb, O)
    mine = tmp_path / "b200_vel_fluc.csv"
    df.write_csv(mine)
    b = open(mine).read().splitlines()
    Ny, Nz = P["Ny"], P["Nz"]
    assert b[0] == "z,y,u_fluc,v_fluc,w_fluc,T_fluc,rho_fluc" and len(b) == 1 + Ny * Nz
    yv, yc, dy = np.zeros(561), np.zeros(560), np.zeros(560)
    O.lib().orc_default_grid(C.c_int(560), C.c_double(P["d_i"]), O._d(yv), O._d(yc), O._d(dy))
    assert np.array_equal(yc[:Ny], P["yc"])
    ref = np.stack([o["fluc"][0], o["fluc"][1], o["fluc"][2], o["T"], o["rho"]]).reshape(5, -1)
    rms = np.sqrt((ref ** 2).mean(1))
    for n in range(0, Ny * Nz, 997):
        j, k = divmod(n, Nz)                           # one row per cell, j-major
        tb = b[1 + n].split(",")
        assert all(len(x.split(".")[1]) == 15 for x in tb)
        assert tb[0] == "%.15f" % (0.25 * (k * 0.000133 + (k + 1) * 0.000133 + k * 0.000133 + (k + 1) * 0.000133))
        assert tb[1] == "%.15f" % (0.25 * (yv[j] + yv[j] + yv[j + 1] + yv[j + 1]))
        for x, r, s in zip(tb[2:], ref[:, n], rms):
            assert abs(float(x) - r) <= TOL * max(abs(r), s) + 5e-16, (n, x, r)
    df.close()


# ---------------------------------------------------------------------------------------------
# edge cases: explicit (odd, zero, large) half-widths, awkward shapes, batch call
# ---------------------------------------------------------------------------------------------
def _explicit_plane(W, Ny, Nz, Ny_rows, Nz_rows):
    """row-uniform plane whose half-widths are SUPPLIED (dfb_config.N_y / N_z) instead of derived from geometry"""
    yc = (np.arange(Ny) + 0.5) * 1e-5
    N_y = np.stack([np.repeat(np.asarray(Ny_rows[f], dtype=np.int32)[:, None], Nz, axis=1) for f in range(3)])
    N_z = np.stack([np.repeat(np.asarray(Nz_rows[f], dtype=np.int32)[:, None], Nz, axis=1) for f in range(3)])
    return dict(name=f"explicit_{Ny}x{Nz}", Ny=Ny, Nz=Nz, d_i=W.D_I, U_e=W.U_E, yc=yc, dy=np.full(Ny, 1e-5), dz=np.full(Ny, 1e-5),
                rows=W.synthetic_rows(yc + 1e-4), scales=W._scales(W.D_I), explicit_N=True,
                N_y=N_y, N_z=N_z, Ny_max=[int(N_y[f].max()) for f in range(3)], Nz_max=[int(N_z[f].max()) for f in range(3)])


def _run_explicit(dfb, O, plane, seed, dts, variant=0):
    Ny, Nz = plane["Ny"], plane["Nz"]
    cfg = dfb.DFConfig.from_plane(plane, noise_mode=dfb.NOISE_INJECT, kernel_variant=variant)
    cfg.geom_per_row = 0                       # N arrays are per cell
    cfg.yc = cfg.dy = cfg.dz = None
    cfg.N_y, cfg.N_z = plane["N_y"], plane["N_z"]
    df = dfb.DIGITAL_FILTER(cfg)
    fo = np.zeros((3, Ny, Nz))
    for s, dt in enumerate([0.0] + list(dts)):
        rys = [O.noise_rys(seed, 0, f, s, Ny, plane["Ny_max"][f], Nz) for f in range(3)]
        hal = [O.noise_halo(seed, 0, f, s, Ny, plane["Nz_max"][f]) if plane["Nz_max"][f] else np.zeros((Ny, 0)) for f in range(3)]
        for f in range(3):
            df.set_noise(f, rys[f], hal[f] if plane["Nz_max"][f] else None)
        df.first_step() if s == 0 else df.filter(dt)
        df.fetch()
        o = O.step(plane, rys, hal, fo, dt, first_step=(s == 0))
        fo = o["filt_old"]
        for f, F in enumerate((df.u, df.v, df.w)):
            ok, r = normwise_close(F.fluc, o["fluc"][f], TOL)
            assert ok, (plane["name"], s, f, r)
        if s:
            assert normwise_close(df.T_fluc, o["T"], TOL)[0] and normwise_close(df.rho_fluc, o["rho"], TOL)[0]
    tuned = df.tuned
    df.close()
    return tuned


def test_explicit_odd_and_mixed_half_widths(dfb, O, W):
    rng = np.random.default_rng(5)
    Ny, Nz = 37, 530
    Nyr = [rng.integers(1, 40, Ny) for _ in range(3)]            # odd and even, changing every row
    Nzr = [rng.integers(1, 23, Ny) for _ in range(3)]
    plane = _explicit_plane(W, Ny, Nz, Nyr, Nzr)
    assert _run_explicit(dfb, O, plane, seed=12, dts=[3e-7])     # row-uniform -> tuned kernels, scalar z staging (odd N)


@pytest.mark.parametrize("ymode", [None, "2"], ids=["y-default", "y-run-forced"])
def test_large_half_widths_beyond_128(dfb, O, W, monkeypatch, ymode):
    """half-widths up to 300: the windows are too tall for two buffers of the run-recursive y-sweep, so by default the band-matrix
    kernels take the plane; forced (DFB_Y_MODE=2) the run form runs with ONE window buffer per CTA -- both against the oracle."""
    if ymode is not None:
        monkeypatch.setenv("DFB_Y_MODE", ymode)
    Ny, Nz = 24, 700
    Nyr = [np.full(Ny, 200), np.full(Ny, 96), np.linspace(20, 260, Ny).astype(int) // 2 * 2]
    Nzr = [np.full(Ny, 300), np.full(Ny, 2), np.full(Ny, 130)]
    plane = _explicit_plane(W, Ny, Nz, Nyr, Nzr)
    assert _run_explicit(dfb, O, plane, seed=13, dts=[3e-7])


@pytest.mark.parametrize("ymode", ["2", "1", "0"], ids=["y-run-recursive", "y-chunk-recursive", "y-dense"])
def test_G2_both_forms_of_the_y_sweep(dfb, O, W, monkeypatch, ymode):
    """The tuned y-sweep has three forms: run-recursive (ysweep_run_kernel, the default: every group of rows of one half-width
    through the exponential window -- short groups of <= 8 rows, long lock-step groups of up to min(32, 0.33 N) rows), and the
    band-matrix kernels kept for windows too tall for shared memory -- chunk-recursive (ysweep_rec_kernel) and dense.  Each forced
    in turn, on a boundary-layer profile (N_y changes every few rows: runs of every length, mixed leftovers) and on hand-made runs
    (lengths 1..40, N from 2 to 200 and N = 0, windows not aligned to the 8-row chunks; the third field one run of N = 128), all must pass
    the gate."""
    monkeypatch.setenv("DFB_Y_MODE", ymode)
    probe = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(W.plane_profile(200, 300, 96, 24), noise_mode=dfb.NOISE_INJECT))
    assert probe.info(10) == int(ymode)
    probe.close()
    worst = inject_and_step(dfb, O, W.plane_profile(200, 300, 96, 24), 0, seed=23, dts=[2e-7, 8e-7])
    assert max(worst.values()) < 1e-13, worst
    rng = np.random.default_rng(7)
    runs, Ns = [], [2, 8, 15, 16, 17, 18, 31, 40, 64, 66, 100, 128, 200]
    while sum(runs) < 330:
        runs.append(int(rng.integers(1, 41)))
    row_N = np.concatenate([np.full(r, Ns[int(rng.integers(0, len(Ns)))]) for r in runs])
    row_N = np.concatenate([row_N[:40], np.zeros(6, dtype=int), row_N[40:], [0]])     # and N = 0: a run of 6 rows, a lone last row
    Ny, Nz = len(row_N), 150
    plane = _explicit_plane(W, Ny, Nz, [row_N, row_N[::-1].copy(), np.full(Ny, 128)], [np.full(Ny, 4)] * 3)
    assert _run_explicit(dfb, O, plane, seed=24, dts=[3e-7])


@pytest.mark.parametrize("zk", ["8", "16"])
def test_recursive_z_sweep_every_window_geometry(dfb, O, W, monkeypatch, zk):
    """The recursive z-sweep has separate code for even / odd distance to the first tap, windows inside / beyond 64 lines, 64- and
    128-byte lines and partial last strips: one row per half-width covers them all, against the oracle."""
    monkeypatch.setenv("DFB_ZK", zk)
    monkeypatch.setenv("DFB_Z_MODE", "1")
    Ns = [1, 2, 3, 4, 7, 8, 9, 15, 16, 17, 24, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257, 300]
    Ny, Nz = len(Ns), 601                                          # 601: partial last strip, odd width
    Nzr = [np.array(Ns), np.array(Ns[::-1]), np.array(Ns)]
    Nyr = [np.full(Ny, 3), np.full(Ny, 2), np.full(Ny, 5)]
    plane = _explicit_plane(W, Ny, Nz, Nyr, Nzr)
    assert _run_explicit(dfb, O, plane, seed=19, dts=[2e-7, 5e-7])


@pytest.mark.parametrize("shape", [(3, 5), (9, 17), (8, 16), (65, 1)])
def test_tiny_and_awkward_shapes(dfb, O, W, shape):
    Ny, Nz = shape
    Nyr = [np.full(Ny, 2), np.full(Ny, 4), np.full(Ny, 2)]
    Nzr = [np.full(Ny, 2), np.full(Ny, 2), np.full(Ny, 4)]
    plane = _explicit_plane(W, Ny, Nz, Nyr, Nzr)
    _run_explicit(dfb, O, plane, seed=14, dts=[2e-7, 2e-7])


def test_filter_batch_matches_step_by_step(dfb, W):
    plane = W.plane_profile(40, 64, 8, 6)
    a = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=21))
    b = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=21), fetch=False)
    dts = np.array([1e-7, 2e-7, 3e-7, 1e-7])
    out = np.zeros((4, 5, 40, 64))
    b.filter_batch(dts, out)
    for s, dt in enumerate(dts):
        a.filter(float(dt))
        for i, ref in enumerate((a.u.fluc, a.v.fluc, a.w.fluc, a.T_fluc, a.rho_fluc)):
            assert np.array_equal(out[s, i], ref), (s, i)
    a.close(); b.close()


def test_timing_mode_does_not_change_results(dfb, W):
    plane = W.plane_profile(40, 64, 8, 6)
    a = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=22))
    b = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=22))
    b.set_timing(True)
    for _ in range(3):
        a.filter(1e-7); b.filter(1e-7)
    b.set_timing(False)
    a.filter(1e-7); b.filter(1e-7)
    assert np.array_equal(a.u.fluc, b.u.fluc) and np.array_equal(a.rho_fluc, b.rho_fluc)
    assert b.last_ms()["step"] > 0
    a.close(); b.close()


def test_G3_config1_default_plane_100_steps(dfb):
    """BASELINE.json configs[0]: the reference's own default plane (the tables its setup built from RST.dat + line.dat), u'/v'/w' over 100 filter(dt)
    steps with dt = 1e-5 (cpp-main.cpp:15).  Reynolds stresses averaged over the steps and the 400 spanwise cells against
    the target RST the setup interpolated from the DNS file.  Stated tolerance (n_eff ~ 100*400/13 ~ 3000 per row):
    diagonal terms median < 3 %, p95 < 8 %; the reference itself shows median 0.5 %, max 2-3 % (BASELINE.md section 2)."""
    P = default_plane()
    df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(P, seed=11), fetch=False)
    for f in range(3):                                       # the library derives the reference's half-widths from the stored geometry
        assert np.array_equal(df.half_widths(f, 0), P["N_y"][f]) and np.array_equal(df.half_widths(f, 1), P["N_z"][f])
    rows = df.rows()
    acc = np.zeros((4, df.Ny))
    for _ in range(100):
        df.filter(1e-5)
        u, v, w = df.get(dfb.U_FLUC), df.get(dfb.V_FLUC), df.get(dfb.W_FLUC)
        acc += np.stack([(u * u).mean(1), (v * v).mean(1), (w * w).mean(1), (u * v).mean(1)])
    acc /= 100
    ok_rows = rows[0] > 1e-6                                 # the wall row has R = 0 exactly
    for i, tgt in enumerate((rows[0], rows[2], rows[3])):
        rel = np.abs(acc[i][ok_rows] - tgt[ok_rows]) / tgt[ok_rows]
        assert np.median(rel) < 0.03 and np.percentile(rel, 95) < 0.08, (i, float(np.median(rel)), float(np.percentile(rel, 95)))
    df.close()


def test_N3_device_scatter_to_cfd_ghost_cells(dfb, W):
    """SURVEY 8f N3: the loop a US3D-style plugin runs over its inflow faces (ghost cell = mean + fluctuation,
    us3d_user.f90:88-113), on the device through dfb_scatter_to_cells, against numpy."""
    import torch
    plane = W.plane_profile(40, 96, 8, 6)
    df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=31))
    df.filter(1e-7)
    rng = np.random.default_rng(2)
    nfaces = 40 * 96
    face_cell = rng.permutation(nfaces).astype(np.int32)            # inflow face i looks at plane cell face_cell[i]
    ghost = (rng.permutation(3 * nfaces)[:nfaces]).astype(np.int32)  # ... and owns CFD cell ghost[i]
    u0 = rng.normal(869.1, 1.0, nfaces)
    u_cfd = rng.normal(0.0, 1.0, 3 * nfaces)
    t_cfd = u_cfd.copy()
    d_u, d_t = torch.from_numpy(u_cfd).cuda(), torch.from_numpy(t_cfd).cuda()
    pi, gi, mu = torch.from_numpy(face_cell).cuda(), torch.from_numpy(ghost).cuda(), torch.from_numpy(u0).cuda()
    df.scatter_to_cells(dfb.U_FLUC, pi, gi, d_u, mean=mu)             # u(ii) = u0 + u'
    df.scatter_to_cells(dfb.T_FLUC, pi, gi, d_t, mean=None, scale=2.0)   # t(ii) += 2 T'
    df.sync()
    exp_u = u_cfd.copy(); exp_u[ghost] = u0 + df.u.fluc.ravel()[face_cell]
    exp_t = t_cfd.copy(); exp_t[ghost] = t_cfd[ghost] + 2.0 * df.T_fluc.ravel()[face_cell]
    assert np.array_equal(d_u.cpu().numpy(), exp_u)
    assert np.allclose(d_t.cpu().numpy(), exp_t, rtol=0, atol=1e-15 * np.abs(exp_t).max())
    with pytest.raises(dfb.DfbError):
        df.scatter_to_cells(99, pi, gi, d_u)
    df.close()


def test_soak_tuned_against_simple_kernels_over_many_steps(dfb, W):
    """120 back-to-back steps in generate mode (look-ahead noise on the side stream, programmatic launches, work queues, u->v
    completion stamps all in play) of the tuned kernels against the one-thread-per-cell kernels on the same noise stream: a race
    anywhere in the tuned path would show up as a divergence (tools/soak.py runs the same at 1024x2048 for 400 steps)."""
    plane = W.plane_profile(160, 1300, 64, 64)
    a = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=99), fetch=False)
    b = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=99, kernel_variant=1), fetch=False)
    assert a.tuned and not b.tuned
    for s in range(120):
        a.filter(1e-7); b.filter(1e-7)
        if s % 40 == 39:
            for w in (dfb.U_FLUC, dfb.V_FLUC, dfb.W_FLUC, dfb.T_FLUC, dfb.RHO_FLUC):
                ok, r = normwise_close(a.get(w), b.get(w), TOL)
                assert ok, (s, w, r)
    a.close(); b.close()


def test_pipelined_filter_to_host_delivers_every_step(dfb, W):
    """dfb_filter_to_host_begin/_end (copy of step t under the compute of step t+1, two sets of host arrays) against the
    synchronous dfb_filter_to_host on a twin handle: same five fields for every step; a third outstanding begin is refused."""
    import ctypes as C
    plane = W.plane_profile(48, 200, 12, 10)
    a = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=41), fetch=False)
    b = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=41), fetch=False)
    L = dfb.lib()
    n = 48 * 200
    sets = [[np.zeros(n) for _ in range(5)] for _ in range(2)]
    ref = [np.zeros(n) for _ in range(5)]
    ptrs = lambda arrs: [x.ctypes.data_as(C.c_void_p) for x in arrs]
    dts = [1e-7, 2e-7, 3e-7, 1e-7, 2e-7]
    dfb._check(L.dfb_filter_to_host_begin(a._h, dts[0], *ptrs(sets[0])))
    for i in range(1, len(dts) + 1):
        if i < len(dts):
            dfb._check(L.dfb_filter_to_host_begin(a._h, dts[i], *ptrs(sets[i & 1])))
        if i == 1:
            assert L.dfb_filter_to_host_begin(a._h, 1e-7, *ptrs(sets[0])) != 0          # two are outstanding
        dfb._check(L.dfb_filter_to_host_end(a._h))                                       # step i-1 has arrived
        dfb._check(L.dfb_filter_to_host(b._h, dts[i - 1], *ptrs(ref)))
        for x, y in zip(sets[(i - 1) & 1], ref):
            assert np.array_equal(x, y), i
    assert L.dfb_filter_to_host_end(a._h) != 0                                           # nothing outstanding
    a.close(); b.close()


# ---------------------------------------------------------------------------------------------
# parity AT the benchmarked sizes (BASELINE.json configs 2, 3a, 3b, 4): the cost-model branches the headline takes
# (dense y-sweep with 128-column tiles over several CTA waves, recursive z-sweep with 16 outputs per lane over 4 strips x 1024
# rows, two CTAs per SM beside live noise CTAs) checked against the oracle itself, not only through properties.
# ---------------------------------------------------------------------------------------------
def _note_worst(name, worst):
    """worst normwise ratios of the at-size parity tests -> gpurun_out/parity_at_size.json (and the test log with -s)"""
    import json
    print("parity at size:", name, worst)
    out = os.path.join(os.path.dirname(GOLDEN), "..", "gpurun_out")
    if os.path.isdir(out):
        path = os.path.join(out, "parity_at_size.json")
        try:
            d = json.load(open(path))
        except Exception:
            d = {}
        d[name] = worst
        json.dump(d, open(path, "w"), indent=1, sort_keys=True)


@pytest.mark.parametrize("name", ["512x512_N32", "1024x2048_profile_N128", "1024x2048_saturated_N128"])
def test_G2_at_benchmarked_size_against_oracle(dfb, O, W, name):
    """constructor step + one filter(dt) of the tuned kernels with their default switches on the named BASELINE plane,
    every cell of every output against the oracle restatement (df.cpp:351-485) under identical injected noise."""
    plane = W.NAMED[name]()
    worst = inject_and_step(dfb, O, plane, 0, seed=31, dts=[DT_BENCH])
    _note_worst(name, worst)
    assert max(worst.values()) <= TOL


DT_BENCH = 1e-7          # bench.py's dt


def _oracle_window(O, plane, seed, plane_id, k_lo, k_hi, dts):
    """The oracle on the columns [k_lo, k_hi) of a plane too large to restate whole in a test: it is run on the sub-plane
    [k_lo - M, k_hi + M) (clipped; M = largest N_z), whose noise is the plane's own (addressed by global index); columns closer
    than M to a cut see wrong z-neighbours and are discarded, columns at a true plane edge get the true raw-noise halo.
    Yields dict(fluc[3], T, rho, filt_old[3]) restricted to [k_lo, k_hi) for the constructor step and every dt."""
    Ny, NzG = plane["Ny"], plane["Nz"]
    M = max(plane["Nz_max"])
    a, b = max(0, k_lo - M), min(NzG, k_hi + M)
    sub = dict(plane)
    sub.update(Nz=b - a, N_y=plane["N_y"][:, :, a:b], N_z=plane["N_z"][:, :, a:b])
    fo = np.zeros((3, Ny, b - a))
    for s, dt in enumerate([0.0] + list(dts)):
        rys = [O.noise_rys(seed, plane_id, f, s, Ny, plane["Ny_max"][f], NzG, a, b) for f in range(3)]
        hal = []
        for f in range(3):
            Mf = plane["Nz_max"][f]
            h = O.noise_halo(seed, plane_id, f, s, Ny, Mf) if (a == 0 or b == NzG) else np.zeros((Ny, 2 * Mf))
            if a != 0:
                h[:, :Mf] = 0.0
            if b != NzG:
                h[:, Mf:] = 0.0
            hal.append(h)
        o = O.step(sub, rys, hal, fo, dt, first_step=(s == 0))
        fo = o["filt_old"]
        sl = slice(k_lo - a, k_hi - a)
        yield dict(fluc=o["fluc"][:, :, sl], T=o["T"][:, sl], rho=o["rho"][:, sl], filt_old=o["filt_old"][:, :, sl])


@pytest.mark.parametrize("name", ["4096x8192_profile_N128"])
def test_config4_slabs_at_size_against_oracle_and_whole_plane(dfb, O, W, name):
    """BASELINE config 4 at its real size, generate mode: two spanwise slabs (cut where parallel.slab_bounds cuts) against
    (a) the oracle on 256-column windows -- the plane's left edge, the window straddling the cut between the slabs, the
    plane's right edge -- and (b) the single-GPU whole plane, bit for bit."""
    from digital_filtering_b200 import parallel
    plane = W.NAMED[name]()
    O.half_widths(plane)
    Ny, Nz = plane["Ny"], plane["Nz"]
    seed, dts = 77, [DT_BENCH]
    bounds = parallel.all_slab_bounds(Nz, 2)
    cut = bounds[0][1]
    windows = [(0, 256), (cut - 128, cut + 128), (Nz - 256, Nz)]
    ref = {w: list(_oracle_window(O, plane, seed, 0, w[0], w[1], dts)) for w in windows}
    sel = (dfb.U_FLUC, dfb.V_FLUC, dfb.W_FLUC, dfb.T_FLUC, dfb.RHO_FLUC)
    got = []
    for k0, k1 in bounds + [(0, Nz)]:
        df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=seed, k_begin=k0, k_end=k1), fetch=False)
        assert df.tuned
        per_step = [[df.get(w) for w in sel[:3]]]
        for dt in dts:
            df.filter(dt)
            per_step.append([df.get(w) for w in sel])
        got.append(per_step)
        df.close()
    slabs, whole = got[:2], got[2]
    # (b) slab == whole, bitwise, every field of every step
    for (k0, k1), per_step in zip(bounds, slabs):
        for s, fields in enumerate(per_step):
            for i, a in enumerate(fields):
                assert np.array_equal(a, whole[s][i][:, k0:k1]), (k0, k1, s, i)
    # (a) oracle windows, read from the slabs (stitched where the window straddles the cut)
    worst = 0.0
    for (lo, hi), steps in ref.items():
        for s, o in enumerate(steps):
            want = [o["fluc"][0], o["fluc"][1], o["fluc"][2]] + ([o["T"], o["rho"]] if s else [])
            for i, b in enumerate(want):
                a = np.concatenate([per_step[s][i][:, max(lo, k0) - k0:min(hi, k1) - k0] for (k0, k1), per_step in zip(bounds, slabs)
                                    if min(hi, k1) > max(lo, k0)], axis=1)
                ok, r = normwise_close(a, b, TOL)
                worst = max(worst, r)
                assert ok, (lo, hi, s, i, r)
    _note_worst(name, dict(windows=worst, slab_equals_whole="bitwise"))


def test_rewind_by_two_steps_is_bit_reproducible(dfb, W):
    """dfb_set_state to a step of the SAME parity as the look-ahead noise already in flight on the side stream (rolling back two
    steps): the regenerated noise must not race with that prefetch (both write the same buffer set)."""
    plane = W.plane_profile(160, 1300, 64, 64)
    a = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=17), fetch=False)
    b = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=17), fetch=False)
    for _ in range(3):
        a.filter(1e-7); b.filter(1e-7)
    fo, step = b.get_state()                    # step 4
    a.filter(1e-7); a.filter(1e-7)              # a is at step 6, noise of step 6 prefetching into set 0
    for rep in range(3):
        a.set_state(fo, step)                   # back to 4: same set as the prefetch
        a.filter(2e-7)
        if rep == 0:
            b.filter(2e-7)
        for w in (dfb.U_FLUC, dfb.V_FLUC, dfb.W_FLUC, dfb.RHO_FLUC):
            assert np.array_equal(a.get(w), b.get(w)), (rep, w)
        a.set_state(None, step + 2)             # filt_old3 = NULL: only the counter moves; prefetch for step 6 restarts
        a.filter(1e-7)
    a.close(); b.close()


# ---------------------------------------------------------------------------------------------
# BASELINE config 5: batched planes behind one handle; the remaining "next" rows (Tecplot / rms writers, face map)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(72, 530, 20, 16), (64, 130, 16, 12)])
def test_config5_batch_equals_independent_handles_bitwise(dfb, W, shape):
    """dfb_create_batch: P planes of one geometry advanced by ONE launch set per step (plane = extra tile / item coordinate) give,
    plane by plane, exactly what P single-plane handles with plane_id + p give -- every output field, several steps, checkpoint
    included."""
    plane = W.plane_profile(*shape)
    P = 5
    batch = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=9, plane_id=3), nplanes=P)
    singles = [dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=9, plane_id=3 + p), fetch=False) for p in range(P)]
    sel = (dfb.U_FLUC, dfb.V_FLUC, dfb.W_FLUC, dfb.T_FLUC, dfb.RHO_FLUC, dfb.U_FILT, dfb.V_FILT, dfb.W_FILT)
    # bit-identity holds between handles that run the same form of the y-sweep (a batch has P times the tiles and may take the
    # run form where a single plane would not; DFB_Y_MODE pins it)
    assert batch.info(10) == singles[0].info(10), (batch.info(10), singles[0].info(10))
    for s, dt in enumerate([None, 1e-7, 3e-7, 1e-7]):
        if dt is not None:
            batch.filter(dt)
            for d in singles:
                d.filter(dt)
        for p in range(P):
            for w in sel:
                assert np.array_equal(batch.get(w, plane=p), singles[p].get(w)), (s, p, w)
    fo, step = batch.get_state()
    assert fo.shape == (3, P, plane["Ny"], plane["Nz"]) and step == 4
    for p in range(P):
        assert np.array_equal(fo[:, p], singles[p].get_state()[0])
    # the five fields of all planes in one call: [P][Ny*Nz] per pointer
    import ctypes as C
    n = plane["Ny"] * plane["Nz"]
    host = [np.zeros((P, n)) for _ in range(5)]
    dfb._check(dfb.lib().dfb_filter_to_host(batch._h, 2e-7, *[h.ctypes.data_as(C.c_void_p) for h in host]))
    for p, d in enumerate(singles):
        d.filter(2e-7)
        for i, w in enumerate(sel[:5]):
            assert np.array_equal(host[i][p].reshape(plane["Ny"], plane["Nz"]), d.get(w)), (p, w)
    batch.close()
    for d in singles:
        d.close()


def test_config5_default_plane_batch_against_single_plane(dfb):
    """BASELINE config 5 proper: 8 planes of the reference's default geometry behind one handle.  The batch has 8 times the tiles
    and takes the run-recursive y-sweep on the row blocks where it pays (dfb_info 10 == 3), a single such plane stays on the band
    matrices (0): plane p of the batch and the single-plane handle with plane_id + p then agree to rounding (<= 1e-13 of the rms,
    far inside the 1e-12 gate each form passes against the oracle); bit for bit if they happen to run the same form."""
    P, p = 8, 5
    batch = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(default_plane(), seed=21, plane_id=2), fetch=False, nplanes=P)
    cfg1 = dfb.DFConfig.from_plane(default_plane(), seed=21, plane_id=2 + p)
    single = dfb.DIGITAL_FILTER(cfg1, fetch=False)
    same_form = batch.info(10) == single.info(10)
    for dt in (1e-5, 1e-5, 2e-5):
        batch.filter(dt); single.filter(dt)
    worst = 0.0
    for w in (dfb.U_FLUC, dfb.V_FLUC, dfb.W_FLUC, dfb.T_FLUC, dfb.RHO_FLUC):
        a, b = batch.get(w, plane=p), single.get(w)
        if same_form:
            assert np.array_equal(a, b), w
        ok, ratio = normwise_close(a, b, 1e-13)
        worst = max(worst, ratio)
        assert ok, (w, ratio)
    print("config 5 default plane: batch form %d, single form %d, worst normwise difference %.2e" % (batch.info(10), single.info(10), worst))
    batch.close(); single.close()


def test_config5_batch_statistics_per_plane(dfb, W):
    plane = W.plane_profile(40, 96, 8, 6)
    batch = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=4), nplanes=3)
    batch.stats_enable(True)
    acc = np.zeros((3, 6, 40, 96))
    for _ in range(4):
        batch.filter(3e-7)
        for p in range(3):
            f = [batch.get(w, plane=p) for w in (dfb.U_FLUC, dfb.V_FLUC, dfb.W_FLUC, dfb.T_FLUC, dfb.RHO_FLUC)]
            for i in range(5):
                acc[p, i] += f[i] * f[i]
            acc[p, 5] += f[0] * f[1]
    for p in range(3):
        for i in range(6):
            got, cnt = batch.stats(i, plane=p)
            assert cnt == 4 and np.array_equal(got, acc[p, i]), (p, i)
    batch.close()


@pytest.mark.parametrize("shape", [(40, 96, 8, 6), (24, 700, 8, 40)])
def test_N2_fused_statistics_every_path(dfb, W, shape):
    """the sums accumulated inside the z-sweep's epilogue (tuned kernels: coalesced strips, partial last strip, both lane widths)
    and by the separate kernel of the general path are the host accumulation of the fetched fields, bit for bit."""
    plane = W.plane_profile(*shape)
    for variant in (0, 1):
        df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=4, kernel_variant=variant))
        df.stats_enable(True)
        acc = np.zeros((6,) + df.u.fluc.shape)
        for _ in range(3):
            df.filter(3e-7)
            f = [df.u.fluc, df.v.fluc, df.w.fluc, df.T_fluc, df.rho_fluc]
            for i in range(5):
                acc[i] += f[i] * f[i]
            acc[5] += f[0] * f[1]
        for i in range(6):
            got, cnt = df.stats(i)
            assert cnt == 3 and np.array_equal(got, acc[i]), (variant, i)
        df.close()


def test_get_rms_and_its_csv(dfb, W, tmp_path):
    """get_rms / plot_rms (df.cpp:584-675): N steps of dt accumulated on the device, then the rms file in the reference's format."""
    plane = W.plane_profile(40, 96, 8, 6)
    df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=5))
    twin = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=5))
    path = tmp_path / "rms.csv"
    df.get_rms(nsteps=20, dt=1e-5, path=path)
    acc = np.zeros((5, 40, 96))
    for _ in range(20):
        twin.filter(1e-5)
        for i, a in enumerate((twin.u.fluc, twin.v.fluc, twin.w.fluc, twin.T_fluc, twin.rho_fluc)):
            acc[i] += a * a
    rms = np.sqrt(acc / 20)
    got, cnt = df.stats(0, rms=True)
    assert cnt == 20 and np.array_equal(got, rms[0])
    lines = open(path).read().splitlines()
    assert lines[0] == "z, y, u'_rms, v'_rms, w'_rms, T'_rms, rho'_rms " and len(lines) == 1 + 40 * 96
    vy, vz = df.table(12, n=41), df.table(13, n=97)
    for c in (0, 95, 96, 40 * 96 - 1):
        j, k = divmod(c, 96)
        want = ", ".join("%g" % x for x in (vz[k], vy[j], rms[0, j, k], rms[1, j, k], rms[2, j, k], rms[3, j, k], rms[4, j, k]))
        assert lines[1 + c] == want, (c, lines[1 + c], want)
    # later filter() calls do not add to the sums (get_rms is a self-contained driver)
    df.filter(1e-5)
    assert df.stats(0)[1] == 20
    df.close(); twin.close()


def test_N4_tecplot_block_writer(dfb, W, tmp_path):
    """write_tecplot (df.cpp:712-762): three header lines, vertex z and y blocks of (Ny+1)(Nz+1) values, cell-centred u', v', w' blocks."""
    plane = W.plane_profile(20, 36, 8, 6)
    df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=6))
    df.filter(1e-7)
    path = tmp_path / "fluc.dat"
    df.write_tecplot(path)
    lines = open(path).read().splitlines()
    assert lines[0] == 'VARIABLES = "z", "y", "u_fluc", "v_fluc", "w_fluc" '
    assert lines[1] == 'ZONE T="Flow Field", I=37, J=21, F=BLOCK' and lines[2] == "VARLOCATION=([3-5]=CELLCENTERED)"
    nv, nc = 21 * 37, 20 * 36
    assert len(lines) == 3 + 2 * nv + 3 * nc
    vy, vz = df.table(12, n=21), df.table(13, n=37)
    body = lines[3:]
    assert body[:37] == ["%g" % z for z in vz] and body[nv:nv + 37] == ["%g" % vy[0]] * 37 and body[2 * nv - 1] == "%g" % vy[20]
    for f, a in enumerate((df.u.fluc, df.v.fluc, df.w.fluc)):
        blk = body[2 * nv + f * nc:2 * nv + (f + 1) * nc]
        assert blk == ["%g" % x for x in a.ravel()], f
    df.close()


def test_N3_face_map_and_scatter_through_it(dfb, W):
    """face -> (j,k) map (the index a US3D-style plugin needs per inflow face, us3d_user.f90:85-114) on two slabs: every face is
    claimed by exactly one slab, lands in the cell that contains it, and the scatter through the map fills the ghost cells."""
    import torch
    plane = W.plane_profile(40, 96, 8, 6)
    rng = np.random.default_rng(3)
    whole = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=31))
    vy, vz = whole.table(12, n=41), whole.table(13, n=97)
    nf = 500
    jj, kk = rng.integers(0, 40, nf), rng.integers(0, 96, nf)
    yf = vy[jj] + (vy[jj + 1] - vy[jj]) * rng.uniform(0.05, 0.95, nf)
    zf = vz[kk] + (vz[kk + 1] - vz[kk]) * rng.uniform(0.05, 0.95, nf)
    assert np.array_equal(whole.face_map(yf, zf), jj * 96 + kk)
    whole.filter(1e-7)
    ghost = torch.zeros(nf, dtype=torch.float64, device="cuda")
    claimed = np.zeros(nf, dtype=int)
    for k0, k1 in [(0, 48), (48, 96)]:
        part = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=31, k_begin=k0, k_end=k1))
        part.filter(1e-7)
        m = part.face_map(yf, zf)
        mine = (kk >= k0) & (kk < k1)
        assert np.array_equal(m[mine], jj[mine] * (k1 - k0) + kk[mine] - k0) and np.all(m[~mine] == -1)
        claimed += (m >= 0)
        part.scatter_to_cells(dfb.U_FLUC, torch.from_numpy(m).cuda(), torch.arange(nf, dtype=torch.int32, device="cuda"), ghost,
                              mean=torch.zeros(nf, dtype=torch.float64, device="cuda"))
        part.sync()
        part.close()
    assert np.all(claimed == 1)
    assert np.array_equal(ghost.cpu().numpy(), whole.u.fluc[jj, kk])
    whole.close()


def test_G2_hybrid_y_sweep_run_blocks_and_band_matrices(dfb, O, W):
    """A plane whose half-widths are steady over most rows (run-recursive form pays) but change every row in a steep part (it does not):
    the y-sweep runs BOTH forms, each on its own row blocks (dfb_info 10 == 3) -- against the oracle, every output."""
    Ny, Nz = 320, 3400                                                  # wide enough for the run part to be worth a launch of its own
    steep = np.arange(40, 104, 1) * 2                                   # N = 80, 82, ..., 206: a new half-width every row
    row_N = np.concatenate([np.full(96, 40), steep, np.repeat(np.arange(100, 36, -4) * 2, 10)])[:Ny]
    plane = _explicit_plane(W, Ny, Nz, [row_N, np.full(Ny, 24), row_N[::-1].copy()], [np.full(Ny, 6)] * 3)
    cfg = dfb.DFConfig.from_plane(plane, noise_mode=dfb.NOISE_INJECT)
    cfg.geom_per_row = 0
    cfg.yc = cfg.dy = cfg.dz = None
    cfg.N_y, cfg.N_z = plane["N_y"], plane["N_z"]
    probe = dfb.DIGITAL_FILTER(cfg)
    assert probe.tuned and probe.info(10) == 3, probe.info(10)
    probe.close()
    assert _run_explicit(dfb, O, plane, seed=29, dts=[3e-7])
