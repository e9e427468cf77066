"""Spanwise-periodic planes (dfb_config.periodic_z = 1): the z filter wraps around the plane,
filt[j, k] = sum_i b_i * y_filtered[j, (k + i) mod Nz], for every field, row and column.

CPU: the struct layout, and the periodic restatement (periodic_step in tests/oracle_harness.py: the oracle's unchanged plain-C
stages recomposed with the wrap between the sweeps) against a direct circular convolution in numpy.  GPU (-m gpu): the library
against that oracle under identical noise, the noise contract (r_ys drawn as without periodic_z, no halo), rolled inputs (no seam),
interior columns unchanged, slabs, batches, errors, the config-4 gather."""
import ctypes
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, default_plane, normwise_close
from oracle_harness import Model, explicit_config, explicit_plane, periodic_step, run

TOL = 1e-12
gpu = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------
# fixtures / helpers local to this file
# ---------------------------------------------------------------------------------------------
def _ragged_half_widths(Ny, Nz, Nmax, seed):
    """per-cell half-widths that change from column to column (the general, non row-uniform path)"""
    rng = np.random.default_rng(seed)
    N_y = rng.integers(1, Nmax + 1, (3, Ny, Nz)).astype(np.int32)
    N_z = rng.integers(1, Nmax + 1, (3, Ny, Nz)).astype(np.int32)
    return N_y, N_z


def numpy_periodic_step(O, plane, rys, fo, dt, first_step):
    """the periodic step restated directly: y-filter per cell, circular z-filter (np.take(..., mode="wrap")), then
    correlate_fields / apply_RST_scaling / get_rho_T_fluc (df.cpp:408-485)"""
    Ny, Nz = plane["Ny"], plane["Nz"]
    filt = np.zeros((3, Ny, Nz))
    for f in range(3):
        Nym = plane["Ny_max"][f]
        yf = np.zeros((Ny, Nz))
        for N in np.unique(plane["N_y"][f]):
            b, acc = O.coeffs(int(N)), np.zeros((Ny, Nz))
            for i in range(-N, N + 1):
                acc = acc + b[N + i] * rys[f][Nym + i:Nym + i + Ny, :]
            m = plane["N_y"][f] == N
            yf[m] = acc[m]
        cols = np.arange(Nz)
        for N in np.unique(plane["N_z"][f]):
            b, acc = O.coeffs(int(N)), np.zeros((Ny, Nz))
            for i in range(-N, N + 1):
                acc = acc + b[N + i] * np.take(yf, cols + i, axis=1, mode="wrap")
            m = plane["N_z"][f] == N
            filt[f][m] = acc[m]
        if not first_step:
            alpha = np.exp(-3.141592654 * dt / plane["scales"][f][2])
            filt[f] = fo[f] * np.sqrt(alpha) + filt[f] * np.sqrt(1.0 - alpha)
    R11, R21, R22, R33, Us, Ts, rhos, Ms = (np.asarray(plane["rows"][i])[:, None] for i in range(8))
    b = np.where(R11 < 1e-10, 0.0, R21 / np.sqrt(np.where(R11 < 1e-10, 1.0, R11)))
    fluc = np.stack([np.sqrt(R11) * filt[0], b * filt[0] + np.sqrt(R22 - b * b) * filt[1], np.sqrt(R33) * filt[2]])
    t2 = -0.5 * (1.4 - 1) * Ms * Ms / Us * fluc[0]
    return dict(filt=filt, fluc=fluc, T=t2 * Ts, rho=-t2 * rhos)


def periodic_inject_and_step(dfb, O, plane, variant, seed, dts, explicit=False):
    """constructor step + len(dts) filter steps of a periodic handle in inject mode against the model (periodic_step) on the same
    counter-based r_ys; returns the worst normwise ratio per output"""
    kw = dict(noise_mode=dfb.NOISE_INJECT, kernel_variant=variant, periodic_z=1)
    if not explicit:
        O.half_widths(plane)
    df = dfb.DIGITAL_FILTER(explicit_config(dfb, plane, **kw) if explicit else dfb.DFConfig.from_plane(plane, **kw))
    assert df.periodic_z
    worst = run(df, Model(O, plane, seed, 0, periodic=True), dts)
    df.close()
    return worst


FIELDS = lambda d: (d.u.fluc, d.v.fluc, d.w.fluc, d.T_fluc, d.rho_fluc)


# ---------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------
def test_config_layout(dfb):
    """periodic_z lands in what was the struct's tail padding: size and struct_bytes unchanged, dfb_config_init leaves it 0"""
    assert ctypes.sizeof(dfb.dfb_config) == 200
    assert dfb.dfb_config.periodic_z.offset == 196 and dfb.dfb_config.kernel_variant.offset == 192
    c = dfb.dfb_config()
    c.periodic_z = 7
    assert dfb.lib().dfb_config_init(ctypes.byref(c)) == 0
    assert c.periodic_z == 0 and c.struct_bytes == 200
    assert dfb.DFConfig().periodic_z == 0


@pytest.mark.parametrize("case", ["odd_Nz", "Nz_max_eq_Nz", "ragged", "profile"])
def test_oracle_periodic_restatement_against_numpy(O, W, case):
    """periodic_step == a direct circular convolution over the y-filtered field, within 1e-12"""
    if case == "odd_Nz":
        plane = explicit_plane(W, 23, 37, [np.arange(23) % 5 + 1] * 3, [np.arange(23) % 7 + 2, np.full(23, 9), np.arange(23) % 3 + 1])
    elif case == "Nz_max_eq_Nz":
        plane = explicit_plane(W, 17, 20, [np.full(17, 3)] * 3, [np.full(17, 20), np.arange(17) % 20 + 1, np.full(17, 7)])
    elif case == "ragged":
        plane = explicit_plane(W, 19, 31, [np.ones(19, int)] * 3, [np.ones(19, int)] * 3)
        plane["N_y"], plane["N_z"] = _ragged_half_widths(19, 31, 9, seed=4)
        plane["Ny_max"] = [int(plane["N_y"][f].max()) for f in range(3)]
        plane["Nz_max"] = [int(plane["N_z"][f].max()) for f in range(3)]
    else:
        plane = O.half_widths(W.plane_profile(40, 36, 8, 6))
    Ny, Nz = plane["Ny"], plane["Nz"]
    fo = np.zeros((3, Ny, Nz))
    for s, dt in enumerate([0.0, 3e-7, 1e-6]):
        rys = [O.noise_rys(5, 0, f, s, Ny, plane["Ny_max"][f], Nz) for f in range(3)]
        o = periodic_step(O, plane, rys, fo, dt, first_step=(s == 0))
        n = numpy_periodic_step(O, plane, rys, fo, dt, s == 0)
        fo = o["filt_old"]
        for k in ("filt", "fluc") + (("T", "rho") if s else ()):
            ok, r = normwise_close(o[k], n[k], TOL)
            assert ok, (case, s, k, r)
        if s == 0:
            assert not o["T"].any()


def test_periodic_changes_only_the_edge_columns_in_the_oracle(O, W):
    """same noise, periodic (periodic_step) vs not (oracle.step, the reference's step bit for bit): columns whose z window stays
    inside the plane are bitwise equal, the others differ"""
    plane = O.half_widths(W.plane_profile(40, 64, 8, 6))
    Ny, Nz = 40, 64
    rys = [O.noise_rys(9, 0, f, 1, Ny, plane["Ny_max"][f], Nz) for f in range(3)]
    hal = [O.noise_halo(9, 0, f, 1, Ny, plane["Nz_max"][f]) for f in range(3)]
    a = O.step(plane, rys, hal, np.zeros((3, Ny, Nz)), 0.0, first_step=True)
    b = periodic_step(O, plane, rys, np.zeros((3, Ny, Nz)), 0.0, first_step=True)
    for f in range(3):
        M = plane["Nz_max"][f]
        assert np.array_equal(a["filt"][f][:, M:Nz - M], b["filt"][f][:, M:Nz - M])
        assert not np.array_equal(a["filt"][f][:, :M], b["filt"][f][:, :M])


# ---------------------------------------------------------------------------------------------
# GPU: noise contract (G1)
# ---------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("shape", [(40, 36, 8, 6), (33, 51, 6, 4), (64, 130, 16, 12)])
def test_G1_periodic_noise_bit_exact(dfb, O, W, shape):
    """r_ys is drawn exactly as without periodic_z; there is no halo: get_noise gives (r_ys, None), a halo pointer is refused"""
    plane = W.plane_profile(*shape)
    per = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=42, plane_id=9, periodic_z=1))
    ref = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=42, plane_id=9))
    Ny, Nz = plane["Ny"], plane["Nz"]
    for step in (0, 1, 7, 123456):
        per.generate_noise(step)
        ref.generate_noise(step)
        for f in range(3):
            r_ys, halo = per.get_noise(f)
            assert halo is None
            F = (per.u, per.v, per.w)[f]
            assert np.array_equal(r_ys, O.noise_rys(42, 9, f, step, Ny, F.Ny_max, Nz)), (step, f)
            assert np.array_equal(r_ys, ref.get_noise(f)[0]), (step, f)
    buf = np.zeros((Ny + 2 * per.u.Ny_max, Nz))
    hal = np.zeros((Ny, 2 * per.u.Nz_max))
    assert dfb.lib().dfb_get_noise(per._h, 0, buf.ctypes.data_as(dfb.c_dp), hal.ctypes.data_as(dfb.c_dp)) == dfb.ERR_ARG
    per.close(); ref.close()


# ---------------------------------------------------------------------------------------------
# GPU: filtered / scaled fields against the periodic oracle (G2)
# ---------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("variant", [0, 1], ids=["tuned", "simple"])
@pytest.mark.parametrize("shape", [(40, 36, 8, 6), (37, 45, 10, 4), (72, 530, 20, 16), (130, 1100, 40, 34)])
def test_G2_periodic_profile_planes(dfb, O, W, shape, variant):
    periodic_inject_and_step(dfb, O, W.plane_profile(*shape), variant, seed=5, dts=[2e-7, 9e-7])


@gpu
@pytest.mark.parametrize("variant", [0, 1], ids=["tuned", "simple"])
def test_G2_periodic_saturated_plane(dfb, O, W, variant):
    periodic_inject_and_step(dfb, O, W.plane_saturated(48, 600, 32), variant, seed=6, dts=[3e-7])


@gpu
def test_G2_periodic_ragged_per_cell_half_widths(dfb, O, W):
    """per-cell half-widths (the one-thread-per-cell path, whose y-sweep looks N_y up at the wrapped global column)"""
    Ny, Nz = 48, 64
    plane = explicit_plane(W, Ny, Nz, [np.ones(Ny, int)] * 3, [np.ones(Ny, int)] * 3)
    plane["N_y"], plane["N_z"] = _ragged_half_widths(Ny, Nz, 12, seed=3)
    plane["Ny_max"] = [int(plane["N_y"][f].max()) for f in range(3)]
    plane["Nz_max"] = [int(plane["N_z"][f].max()) for f in range(3)]
    periodic_inject_and_step(dfb, O, plane, 0, seed=8, dts=[4e-7], explicit=True)
    # and the geometry-derived ragged plane of the non-periodic suite
    periodic_inject_and_step(dfb, O, W.plane_ragged(48, 64, 12, seed=3), 0, seed=8, dts=[4e-7])


@gpu
@pytest.mark.parametrize("zmode", ["1", "0"], ids=["z-recursive", "z-direct"])
def test_G2_periodic_both_forms_of_the_z_sweep(dfb, O, W, monkeypatch, zmode):
    monkeypatch.setenv("DFB_Z_MODE", zmode)
    plane = W.plane_profile(72, 1100, 128, 128)
    worst = periodic_inject_and_step(dfb, O, plane, 0, seed=15, dts=[2e-7, 1e-6])
    assert max(worst.values()) < 1e-13, worst


@gpu
@pytest.mark.parametrize("ymode", ["2", "1", "0"], ids=["y-run-recursive", "y-chunk-recursive", "y-dense"])
def test_G2_periodic_every_form_of_the_y_sweep(dfb, O, W, monkeypatch, ymode):
    monkeypatch.setenv("DFB_Y_MODE", ymode)
    plane = W.plane_profile(200, 300, 96, 24)
    probe = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, noise_mode=dfb.NOISE_INJECT, periodic_z=1))
    assert probe.info(10) == int(ymode)
    probe.close()
    worst = periodic_inject_and_step(dfb, O, plane, 0, seed=23, dts=[2e-7, 8e-7])
    assert max(worst.values()) < 1e-13, worst


@gpu
def test_G2_periodic_stored_default_plane(dfb, O):
    """the reference's default 510x400 plane (mixed y forms in a batch, band matrices alone), periodic"""
    P = default_plane()
    P["name"] = "default"
    periodic_inject_and_step(dfb, O, P, 0, seed=20261018, dts=[1e-5])


@gpu
def test_periodic_generate_mode_equals_oracle_on_the_same_stream(dfb, O, W):
    """generate mode end to end: device noise + device filter == oracle noise + periodic oracle, for the whole plane and for
    slabs touching either edge (whose wrapped neighbour columns are regenerated locally)"""
    plane = O.half_widths(W.plane_profile(96, 200, 24, 10))
    for k in [(0, 200), (0, 64), (144, 200), (5, 50), (190, 200)]:
        df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=77, periodic_z=1, k_begin=k[0], k_end=k[1]), fetch=False)
        run(df, Model(O, plane, 77, 0, periodic=True), [1e-7, 1e-7, 3e-7], k=k)
        assert df.step == 4
        df.close()


# ---------------------------------------------------------------------------------------------
# GPU: at the benchmarked sizes
# ---------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", ["512x512_N32", "1024x2048_profile_N128", "1024x2048_saturated_N128"])
def test_G2_periodic_at_benchmarked_size_against_oracle(dfb, O, W, name):
    """every cell of every output of the tuned kernels with their default switches against the periodic oracle"""
    plane = W.NAMED[name]()
    worst = periodic_inject_and_step(dfb, O, plane, 0, seed=31, dts=[1e-7])
    print("periodic parity at size:", name, worst)
    assert max(worst.values()) <= TOL


# ---------------------------------------------------------------------------------------------
# GPU: no seam, interior unchanged
# ---------------------------------------------------------------------------------------------
def _inject_run(dfb, plane, rys, variant, steps=2):
    df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, noise_mode=dfb.NOISE_INJECT, kernel_variant=variant, periodic_z=1))
    out = []
    for s in range(steps):
        for f in range(3):
            df.set_noise(f, rys[s][f])
        df.first_step() if s == 0 else df.filter(3e-7)
        df.fetch()
        out.append([a.copy() for a in FIELDS(df)])
    df.close()
    return out


@gpu
@pytest.mark.parametrize("variant,shift,exact", [(0, 16, True), (0, 512, True), (0, 7, False), (1, 7, True), (1, 333, True)],
                         ids=["tuned-16", "tuned-512", "tuned-odd", "simple-7", "simple-333"])
def test_no_seam_rolled_noise_rolls_the_output(dfb, O, W, variant, shift, exact):
    """Noise rolled by `shift` columns gives the output rolled by `shift`: the plane has no seam.  Bitwise for the one-thread-
    per-cell kernels at any shift, and for the tuned kernels at multiples of 16 on a plane whose width is a multiple of 16 (the
    recursive z form evaluates 16-column lane blocks: a 16-column shift maps blocks onto blocks, as a slab cut on a multiple of
    16 does); within 1e-12 for the tuned kernels at any other shift.  1088 columns: several 512-column z strips."""
    plane = O.half_widths(W.plane_profile(64, 1088, 24, 48))
    Ny, Nz = 64, 1088
    rys = [[O.noise_rys(3, 0, f, s, Ny, plane["Ny_max"][f], Nz) for f in range(3)] for s in range(2)]
    rolled = [[np.roll(r, shift, axis=1) for r in rs] for rs in rys]
    a = _inject_run(dfb, plane, rys, variant)
    b = _inject_run(dfb, plane, rolled, variant)
    for s in range(2):
        for i, (x, y) in enumerate(zip(a[s], b[s])):
            want = np.roll(x, shift, axis=1)
            if exact:
                assert np.array_equal(y, want), (s, i)
            else:
                ok, r = normwise_close(y, want, TOL)
                assert ok, (s, i, r)


@gpu
def test_interior_columns_unchanged_at_the_headline_size(dfb, W):
    """same seed, generate mode, periodic vs not on the 1024x2048 profile plane: columns at least Nz_max + 32*16 + 16 from both
    edges are bitwise equal, the edge columns differ, and the y-sweep takes the same form in both modes"""
    plane = W.NAMED["1024x2048_profile_N128"]()
    a = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=1), fetch=False)
    b = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=1, periodic_z=1), fetch=False)
    assert a.info(10) == b.info(10) and a.info(7) == b.info(7) and (a.periodic_z, b.periodic_z) == (False, True)
    m = max(a.info(1, f) for f in range(3)) + 32 * 16 + 16
    for dt in (1e-7, 2e-7):
        a.filter(dt); b.filter(dt)
    for w in (dfb.U_FLUC, dfb.V_FLUC, dfb.W_FLUC, dfb.T_FLUC, dfb.RHO_FLUC):
        x, y = a.get(w), b.get(w)
        assert np.array_equal(x[:, m:2048 - m], y[:, m:2048 - m]), w
        assert not np.array_equal(x[:, :8], y[:, :8]) and not np.array_equal(x[:, -8:], y[:, -8:]), w
    a.close(); b.close()


# ---------------------------------------------------------------------------------------------
# GPU: slabs, batches
# ---------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("ymode", [None, "1"], ids=["y-default", "y-recursive"])
def test_periodic_slabs_reproduce_the_periodic_whole_plane(dfb, W, monkeypatch, ymode):
    """periodic slabs cut on multiples of 16 (both edge slabs, and one narrower than Nz_max) are the periodic whole plane bit for
    bit; cut anywhere else, within 1e-12"""
    if ymode is not None:
        monkeypatch.setenv("DFB_Y_MODE", ymode)
    plane = W.plane_profile(64, 700, 16, 24) if ymode is None else W.plane_profile(96, 700, 48, 24)
    whole = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=3, periodic_z=1))
    whole.filter(2e-7); whole.filter(2e-7)
    for k0, k1 in [(0, 160), (160, 176), (176, 400), (400, 700), (0, 700)]:
        part = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=3, periodic_z=1, k_begin=k0, k_end=k1))
        part.filter(2e-7); part.filter(2e-7)
        for a, b in zip(FIELDS(part), FIELDS(whole)):
            assert np.array_equal(a, b[:, k0:k1]), (k0, k1)
        part.close()
    for k0, k1 in [(150, 151), (151, 401), (400, 699), (699, 700), (3, 690)]:
        part = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=3, periodic_z=1, k_begin=k0, k_end=k1))
        part.filter(2e-7); part.filter(2e-7)
        for a, b in zip(FIELDS(part), FIELDS(whole)):
            ref = b[:, k0:k1]
            assert np.all(np.abs(a - ref) <= TOL * np.maximum(np.abs(ref), np.sqrt(np.mean(b * b)))), (k0, k1)
        part.close()
    whole.close()


def _batch_vs_singles(dfb, plane, P, plane_id, seed, dts, exact=True):
    batch = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=seed, plane_id=plane_id, periodic_z=1), nplanes=P)
    singles = [dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=seed, plane_id=plane_id + p, periodic_z=1), fetch=False)
               for p in range(P)]
    assert batch.periodic_z
    same_form = batch.info(10) == singles[0].info(10)
    worst = 0.0
    for dt in dts:
        batch.filter(dt)
        for d in singles:
            d.filter(dt)
    for p in range(P):
        for w in (dfb.U_FLUC, dfb.V_FLUC, dfb.W_FLUC, dfb.T_FLUC, dfb.RHO_FLUC, dfb.U_FILT, dfb.V_FILT, dfb.W_FILT):
            a, b = batch.get(w, plane=p), singles[p].get(w)
            if exact or same_form:
                assert np.array_equal(a, b), (p, w)
            ok, r = normwise_close(a, b, 1e-13)
            worst = max(worst, r)
            assert ok, (p, w, r)
    batch.close()
    for d in singles:
        d.close()
    return same_form, worst


@gpu
@pytest.mark.parametrize("shape", [(72, 530, 20, 16), (64, 130, 16, 12)])
def test_periodic_batch_equals_independent_handles_bitwise(dfb, W, shape):
    _batch_vs_singles(dfb, W.plane_profile(*shape), 5, 3, 9, [1e-7, 3e-7, 1e-7])


@gpu
@pytest.mark.parametrize("ymode", ["0", None], ids=["y-dense-pinned", "y-default"])
def test_periodic_default_plane_batch(dfb, monkeypatch, ymode):
    """8 periodic planes of the reference's default geometry behind one handle against single-plane periodic handles: bitwise when
    both run the same y-sweep form (pinned here with DFB_Y_MODE=0); by default a batch may take the run form where a single
    plane keeps the band matrices, and the two then agree to rounding (<= 1e-13), as without periodic_z"""
    if ymode is not None:
        monkeypatch.setenv("DFB_Y_MODE", ymode)
    same_form, worst = _batch_vs_singles(dfb, default_plane(), 8, 2, 21, [1e-5, 2e-5], exact=ymode is not None)
    print("periodic default-plane batch: same y form %s, worst normwise difference %.2e" % (same_form, worst))


# ---------------------------------------------------------------------------------------------
# GPU: errors and info
# ---------------------------------------------------------------------------------------------
@gpu
def test_periodic_errors_and_info(dfb, W):
    plane = W.plane_profile(40, 36, 8, 6)
    narrow = W.plane_profile(40, 16, 8, 24)                 # N_z of u up to 24 on a 16-column plane
    with pytest.raises(dfb.DfbError) as e:
        dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(narrow, periodic_z=1))
    assert e.value.code == dfb.ERR_ARG and "field u" in str(e.value) and "Nz_max" in str(e.value)
    dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(narrow)).close()          # fine without periodic_z
    with pytest.raises(dfb.DfbError) as e:
        dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, periodic_z=2))
    assert e.value.code == dfb.ERR_ARG and "periodic_z" in str(e.value)
    off = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane))
    on = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, noise_mode=dfb.NOISE_INJECT, periodic_z=1))
    assert off.info(13) == 0 and on.info(13) == 1
    r_ys = np.zeros((40 + 2 * on.u.Ny_max, 36))
    with pytest.raises(dfb.DfbError) as e:
        on.set_noise(0, r_ys, np.zeros((40, 2 * on.u.Nz_max)))
    assert e.value.code == dfb.ERR_ARG
    on.set_noise(0, r_ys, None)
    on.set_noise_ref_layout(1, np.zeros((40 + 2 * on.v.Ny_max, 36)), None)
    off.close(); on.close()


# ---------------------------------------------------------------------------------------------
# GPU: config 4 with periodic slabs (needs >= 2 GPUs)
# ---------------------------------------------------------------------------------------------
@gpu
def test_periodic_slab_gather_equals_the_periodic_whole_plane(dfb):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", str(port), os.path.join(ROOT, "tests", "periodic_slab_worker.py")],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "PERIODIC_SLAB_OK" in r.stdout, (r.stdout[-2000:], r.stderr[-3000:])
