"""Correlation statistics (dfb_corr_enable / dfb_corr_get / dfb_corr_integral_scales): per-row sums of lagged products of u', v', w'
along z, along y and in time, accumulated on the device.

CPU: the numpy checker of the sums, the normalisation and the integral-scale trapezoid against explicit loops; the exact expectation
of the filter (from the coefficient tables, the row constants and the blend) against a Monte-Carlo estimate from filtering white
noise in numpy; the Fortran bindings against the header; the C++ facade compiles.  GPU (-m gpu): the library's sums against numpy
on the fields it produced, at small and headline size; the statistics against the exact expectation; determinism; no side effects;
errors; the C++ facade."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT, default_plane, normwise_close
from oracle_harness import np_sums

gpu = pytest.mark.gpu
TOL = 1e-12
PI_BLEND = 3.141592654          # the blend's truncated pi (df.cpp:411)


# ---------------------------------------------------------------------------------------------
# numpy checker
# ---------------------------------------------------------------------------------------------
def np_normalize(S, pairs, d):
    Ny, n = S.shape
    R = np.full_like(S, np.nan)
    var = S[:, 0]
    with np.errstate(divide="ignore", invalid="ignore"):
        for j in range(Ny):
            for e in range(n):
                if d == 1:
                    if j + e < Ny and var[j] != 0 and var[j + e] != 0:
                        R[j, e] = S[j, e] / np.sqrt(var[j] * var[j + e])
                elif pairs[e] and pairs[0] and var[j] != 0:
                    R[j, e] = (S[j, e] / pairs[e]) / (var[j] / pairs[0])
    return R


def np_integral(R, x):
    """x(j, d) -> coordinate; trapezoid of row j up to the last lag before the first non-positive R"""
    out = np.full(R.shape[0], np.nan)
    for j in range(R.shape[0]):
        if not R[j, 0] > 0:
            continue
        acc, d = 0.0, 1
        while d < R.shape[1] and R[j, d] > 0:
            acc += 0.5 * (R[j, d - 1] + R[j, d]) * (x(j, d) - x(j, d - 1))
            d += 1
        out[j] = acc
    return out


def _loops(steps, L, periodic):
    """the definitions of include/dfb200.h, term by term"""
    Ny, Nz = steps[0].shape
    S = [np.zeros((Ny, L[d] + 1)) for d in range(3)]
    for s, f in enumerate(steps):
        for j in range(Ny):
            for k in range(Nz):
                for d in range(L[0] + 1):
                    if periodic or k + d < Nz:
                        S[0][j, d] += f[j, k] * f[j, (k + d) % Nz]
                for d in range(L[1] + 1):
                    if j + d < Ny:
                        S[1][j, d] += f[j, k] * f[j + d, k]
                for m in range(min(L[2], s) + 1):
                    S[2][j, m] += f[j, k] * steps[s - m][j, k]
    return S


@pytest.mark.parametrize("periodic", [False, True])
def test_numpy_checker_matches_the_definitions(periodic):
    rng = np.random.default_rng(3)
    steps = [rng.standard_normal((5, 7)) for _ in range(4)]
    L = (6, 4, 3)
    got = np_sums(steps, L, periodic)
    ref = _loops(steps, L, periodic)
    for d in range(3):
        assert np.allclose(got[d][0], ref[d], rtol=1e-13, atol=1e-13)
    assert list(got[0][1]) == [4 * (7 if periodic else 7 - d) for d in range(7)]
    assert list(got[2][1]) == [28, 21, 14, 7]
    # normalisation: z / t by the per-lag means, y by the two rows' variances; NaN beyond the plane and on zero rows
    steps[0][2] = steps[1][2] = steps[2][2] = steps[3][2] = 0.0
    got = np_sums(steps, L, periodic)
    Rz = np_normalize(*got[0], 0)
    assert Rz[0, 3] == pytest.approx((got[0][0][0, 3] / got[0][1][3]) / (got[0][0][0, 0] / got[0][1][0]), rel=1e-15)
    assert np.all(np.isnan(Rz[2])) and Rz[0, 0] == 1.0
    Ry = np_normalize(*got[1], 1)
    assert Ry[1, 2] == pytest.approx(got[1][0][1, 2] / np.sqrt(got[1][0][1, 0] * got[1][0][3, 0]), rel=1e-15)
    assert np.isnan(Ry[3, 2]) and np.isnan(Ry[1, 1]) and np.isnan(Ry[4, 1])
    # trapezoid: stops before the first non-positive value
    R = np.array([[1.0, 0.5, 0.25, -0.1, 0.3], [1.0, -0.2, 0.5, 0.5, 0.5], [np.nan] * 5])
    I = np_integral(R, lambda j, d: 2.0 * d)
    assert I[0] == pytest.approx(0.5 * (1.5 + 0.75) * 2.0) and I[1] == 0.0 and np.isnan(I[2])


# ---------------------------------------------------------------------------------------------
# exact expectation of the filter
# ---------------------------------------------------------------------------------------------
def _xcorr(b1, b2, d):
    """sum_i b1[i + d] b2[i] over the taps of both (centred: b[N + i], i = -N..N)"""
    N1, N2 = len(b1) // 2, len(b2) // 2
    i = np.arange(-N2, N2 + 1)
    ok = np.abs(i + d) <= N1
    return float(np.dot(b1[(i + d)[ok] + N1], b2[i[ok] + N2]))


def expected_rho(coef, Nyr, Nzr, rows, alpha, Nz, L, periodic=True):
    """Correlation coefficients the filter delivers in expectation, per field (u', v', w') and direction: {(field, dir): [Ny, L+1]}.
    Filtered white noise g(j, k) = sum_z bz_j[z] sum_y by_j[y] r(j + y, k + z), so cov_g((j,k), (j',k+d)) = Cy_g(j, j') Cz_g(j, j', d),
    the blend filt_s = sqrt(a) filt_{s-1} + sqrt(1-a) new_s multiplies it by a^(m/2) at m steps, and the Lund scaling mixes:
    u' = sqrt(R11) g_u, v' = b g_u + c g_v (b = R21/sqrt(R11), c = sqrt(R22 - b^2)), w' = sqrt(R33) g_w.
    coef(N) -> the 2N+1 coefficients; Nyr / Nzr [3][Ny]: half-widths per row; rows [8][Ny]; alpha[3] of the blend."""
    Ny = len(Nyr[0])
    Lz, Ly, Lt = L
    wraps = (-1, 0, 1) if periodic else (0,)

    def Cy(g, j, jp):
        return _xcorr(coef(int(Nyr[g][j])), coef(int(Nyr[g][jp])), jp - j)

    def Cz(g, j, jp, d):
        return sum(_xcorr(coef(int(Nzr[g][j])), coef(int(Nzr[g][jp])), d + w * Nz) for w in wraps)

    R11, R21, R22, R33 = (np.asarray(rows[i], dtype=np.float64) for i in range(4))
    b = np.where(R11 < 1e-10, 0.0, R21 / np.sqrt(np.where(R11 < 1e-10, 1.0, R11)))
    mix = [[(0, np.sqrt(R11))], [(0, b), (1, np.sqrt(R22 - b * b))], [(2, np.sqrt(R33))]]

    def cov(f, j, jp, d, m):
        return sum(w[j] * w[jp] * alpha[g] ** (m / 2.0) * Cy(g, j, jp) * Cz(g, j, jp, d) for g, w in mix[f])

    out = {}
    for f in range(3):
        v0 = np.array([cov(f, j, j, 0, 0) for j in range(Ny)])
        with np.errstate(divide="ignore", invalid="ignore"):
            if Lz:
                out[f, 0] = np.array([[cov(f, j, j, d, 0) for d in range(Lz + 1)] for j in range(Ny)]) / v0[:, None]
            if Ly:
                R = np.full((Ny, Ly + 1), np.nan)
                for j in range(Ny):
                    for d in range(min(Ly, Ny - 1 - j) + 1):
                        R[j, d] = cov(f, j, j + d, 0, 0) / np.sqrt(v0[j] * v0[j + d])
                out[f, 1] = R
            if Lt:
                out[f, 2] = np.array([[cov(f, j, j, 0, m) for m in range(Lt + 1)] for j in range(Ny)]) / v0[:, None]
        for k in list(out):
            if k[0] == f:
                out[k][v0 == 0] = np.nan
    return out


def sample_sigma(rho_z, rho_t, n):
    """standard error of a sample correlation from n products per row that are correlated along z and in time as rho_z, rho_t
    (one-sided, lag 0 first): sqrt(2 sum_z rho_z^2 sum_t rho_t^2 / n), sums over both signs of the lag (Bartlett's bound)"""
    two = lambda r: 2.0 * np.nansum(np.asarray(r) ** 2, axis=-1) - np.asarray(r)[..., 0] ** 2
    return np.sqrt(2.0 * two(rho_z) * two(rho_t) / n)


def _filter_numpy(coef, Nyr, Nzr, rng, Nz):
    """one filtered white-noise field per component: y filter per row, periodic z filter"""
    Ny = len(Nyr[0])
    out = []
    for g in range(3):
        M = int(max(Nyr[g]))
        r = rng.standard_normal((Ny + 2 * M, Nz))
        yf = np.stack([coef(int(Nyr[g][j])) @ r[j + M - Nyr[g][j]:j + M + Nyr[g][j] + 1] for j in range(Ny)])
        out.append(np.stack([sum(coef(int(Nzr[g][j]))[Nzr[g][j] + i] * np.roll(yf[j], -i) for i in range(-Nzr[g][j], Nzr[g][j] + 1))
                             for j in range(Ny)]))
    return out


def test_expected_correlation_matches_monte_carlo(O):
    """the expectation helper against correlations measured on white noise filtered in numpy with the oracle's coefficients:
    mixed half-widths between rows, the v' mixture, the blend"""
    rng = np.random.default_rng(11)
    Ny, Nz, S = 18, 48, 1500
    Nyr = [rng.integers(1, 5, Ny), rng.integers(1, 4, Ny), rng.integers(2, 5, Ny)]
    Nzr = [rng.integers(1, 5, Ny), rng.integers(2, 6, Ny), rng.integers(1, 3, Ny)]
    rows = np.zeros((8, Ny))
    rows[0], rows[1], rows[2], rows[3] = 1.0 + rng.random(Ny), -0.3 * rng.random(Ny), 1.0 + rng.random(Ny), 0.5 + rng.random(Ny)
    rows[0][0] = rows[1][0] = 0.0                               # a wall row: u' = 0
    alpha = [0.25, 0.5, 0.1]
    L = (10, 8, 4)
    cache = {}
    coef = lambda N: cache.setdefault(N, O.coeffs(N))
    R11, R21, R22, R33 = rows[:4]
    b = np.where(R11 < 1e-10, 0.0, R21 / np.sqrt(np.where(R11 < 1e-10, 1.0, R11)))
    g = _filter_numpy(coef, Nyr, Nzr, rng, Nz)
    steps = [[], [], []]
    for s in range(S):
        new = _filter_numpy(coef, Nyr, Nzr, rng, Nz)
        g = new if s == 0 else [np.sqrt(alpha[c]) * g[c] + np.sqrt(1 - alpha[c]) * new[c] for c in range(3)]
        fl = [np.sqrt(R11)[:, None] * g[0], b[:, None] * g[0] + np.sqrt(R22 - b * b)[:, None] * g[1], np.sqrt(R33)[:, None] * g[2]]
        for f in range(3):
            steps[f].append(fl[f])
    exp = expected_rho(coef, Nyr, Nzr, rows, alpha, Nz, L)
    for f in range(3):
        sums = np_sums(steps[f], L, periodic=True)
        sig = sample_sigma(exp[f, 0], exp[f, 2], Nz * S)
        for d in range(3):
            R = np_normalize(*sums[d], d)
            E = exp[f, d]
            assert np.array_equal(np.isnan(R), np.isnan(E)), (f, d)
            err = np.nanmax(np.abs(R - E) / sig[:, None])
            assert err < 6.0, (f, d, err)


# ---------------------------------------------------------------------------------------------
# bindings
# ---------------------------------------------------------------------------------------------
def test_fortran_corr_bindings_match_the_header():
    h = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "dfb200.h")).read(), flags=re.S)
    decl = {m.group(1): len([a for a in m.group(2).split(",") if a.strip()]) for m in re.finditer(r"\bint\s+(dfb_\w+)\s*\(([^)]*)\)\s*;", h)}
    f90 = open(os.path.join(ROOT, "fortran", "digital_filtering.f90")).read()
    found = re.findall(r"function\s+(\w+)\s*\(([^)]*)\)\s*bind\(C,\s*name='(dfb_corr_\w+)'\)", f90)
    assert {n for _, _, n in found} == {"dfb_corr_enable", "dfb_corr_get", "dfb_corr_integral_scales"}
    for fname, args, cname in found:
        assert fname == cname and cname in decl, cname
        assert len([a for a in args.split(",") if a.strip()]) == decl[cname], cname


CPP_PROG = r"""
#include <cmath>
#include <cstdio>
#include <vector>
#include "digital_filter.hpp"
int main(int argc, char** argv) {
    const int Ny = 40, Nz = 37;
    std::vector<double> buf(Ny * 3 + Ny * 8 + 9);
    FILE* fp = std::fopen(argv[1], "rb");
    if (!fp || std::fread(buf.data(), sizeof(double), buf.size(), fp) != buf.size()) return 2;
    std::fclose(fp);
    DFConfigEx c;
    c.honor_flow_config = true; c.base.d_i = 0.0013; c.base.U_e = 869.1;
    c.Ny = Ny; c.Nz = Nz; c.yc = buf.data(); c.dy = buf.data() + Ny; c.dz = buf.data() + 2 * Ny;
    c.rows = buf.data() + 3 * Ny; c.scales = buf.data() + 11 * Ny; c.seed = 5; c.fetch_every_step = false;
    DIGITAL_FILTER df(c);
    df.corr_enable(DFB_CORR_SUPPORT, DFB_CORR_SUPPORT, 3);
    for (int s = 0; s < 6; ++s) df.filter(1e-7);
    std::vector<double> R = df.corr(1, DFB_CORR_Y, false);
    std::vector<double> I = df.integral_scales(2, DFB_CORR_Z);
    std::printf("%zu %.17g %.17g %.17g\n", R.size(), R[0], R[R.size() / 2], I[Ny / 2]);
    return 0;
}
"""


def _cpp_build(tmp_path):
    src = tmp_path / "corr_main.cpp"
    src.write_text(CPP_PROG)
    libdir = os.path.join(ROOT, "digital-filtering_b200", "lib")
    exe = tmp_path / "corr_main"
    subprocess.run(["/usr/bin/g++", "-std=c++17", "-Wall", str(src), "-I" + os.path.join(ROOT, "include"), "-L" + libdir, "-ldfb200",
                    "-Wl,-rpath," + libdir, "-o", str(exe)], check=True, capture_output=True)
    return exe


def test_cpp_facade_with_corr_compiles(dfb, tmp_path):
    r = subprocess.run(["/usr/bin/g++", "-std=c++17", "-c", "-x", "c++", os.path.join(ROOT, "include", "digital_filter.hpp"),
                        "-I" + os.path.join(ROOT, "include"), "-o", str(tmp_path / "h.o")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert _cpp_build(tmp_path).exists()


# ---------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------
def _small_plane(W, Ny=40, Nz=37, N=8):
    return W.plane_profile(Ny, Nz, N, N)


def _run(dfb, cfg, lags, nsteps, dt=1e-7, nplanes=1):
    """handle with correlations on; u', v', w' of every plane after every accumulated step"""
    df = dfb.DIGITAL_FILTER(cfg, fetch=False, nplanes=nplanes)
    df.corr_enable(*lags)
    fields = [[[] for _ in range(3)] for _ in range(nplanes)]
    for _ in range(nsteps):
        df.filter(dt)
        for p in range(nplanes):
            for f in range(3):
                fields[p][f].append(df.get(f, plane=p).copy())
    return df, fields


def _check_exact(df, fields, periodic, plane=0):
    L = df.corr_lags
    worst = 0.0
    for f in range(3):
        ref = np_sums(fields[f], L, periodic)
        for d in range(3):
            if not L[d]:
                continue
            S, pairs, cnt = df.corr(f, d, normalized=False, plane=plane)
            ok, r = normwise_close(S, ref[d][0], TOL)
            assert ok, (f, d, r)
            worst = max(worst, r)
            assert np.array_equal(pairs, ref[d][1]) and cnt == len(fields[f]), (f, d)
            R = df.corr(f, d, plane=plane)[0]
            Rn = np_normalize(*ref[d], d)
            assert np.array_equal(np.isnan(R), np.isnan(Rn)) and normwise_close(np.nan_to_num(R), np.nan_to_num(Rn), 1e-11)[0]
    return worst


@gpu
@pytest.mark.parametrize("case", ["odd_nz", "periodic", "ragged_variant1", "limits", "lt_beyond_steps", "wide_full_lag"])
def test_exact_sums(dfb, W, O, case):
    plane = _small_plane(W)
    kw, lags, periodic, nsteps = {}, (dfb.DFB_CORR_SUPPORT, dfb.DFB_CORR_SUPPORT, 3), False, 5
    if case == "wide_full_lag":
        # two spanwise segments of <= 4096 columns, nine blocks of 512 lags staged one at a time, a split wall-normal sweep
        plane = W.plane_profile(16, 4500, 4, 4)
        lags, nsteps = (plane["Nz"] - 1, plane["Ny"] - 1, 0), 2
    elif case == "periodic":
        kw, periodic = dict(periodic_z=1), True
    elif case == "limits":
        lags = (plane["Nz"] - 1, plane["Ny"] - 1, 2)
    elif case == "lt_beyond_steps":
        lags, nsteps = (4, 0, 9), 4
    cfg = dfb.DFConfig.from_plane(plane, seed=7, **kw)
    if case == "ragged_variant1":
        rng = np.random.default_rng(2)
        cfg.geom_per_row = 0
        cfg.yc = cfg.dy = cfg.dz = None
        cfg.N_y = rng.integers(1, 7, (3, plane["Ny"], plane["Nz"])).astype(np.int32)
        cfg.N_z = rng.integers(1, 7, (3, plane["Ny"], plane["Nz"])).astype(np.int32)
        cfg.kernel_variant = 1
    df, fields = _run(dfb, cfg, lags, nsteps)
    if case == "ragged_variant1":
        assert not df.tuned
    if case == "limits":
        assert df.corr_lags == (plane["Nz"] - 1, plane["Ny"] - 1, 2)
    elif lags[0] == dfb.DFB_CORR_SUPPORT:
        assert df.corr_lags[0] == min(plane["Nz"] - 1, 2 * max(df.info(1, f) for f in range(3)))
        assert df.corr_lags[1] == min(plane["Ny"] - 1, 2 * max(df.info(0, f) for f in range(3)))
    _check_exact(df, fields[0], periodic)
    if case == "lt_beyond_steps":
        _, pairs, _ = df.corr(0, dfb.CORR_T)
        assert list(pairs[4:]) == [0] * 6 and np.all(np.isnan(df.corr(0, dfb.CORR_T)[0][:, 4:]))
    df.close()


@gpu
@pytest.mark.parametrize("which", ["small", "default_plane"])
def test_exact_sums_batch_and_bitwise_against_single_planes(dfb, W, which):
    """the default plane (400 columns, L_y = 424) splits the wall-normal sweep's columns and runs two blocks of lags: the split
    follows the plane's shape alone, so every plane of the batch adds its partial sums in the single plane's order"""
    plane = _small_plane(W) if which == "small" else default_plane()
    lags = (dfb.DFB_CORR_SUPPORT, dfb.DFB_CORR_SUPPORT, 3)
    df, fields = _run(dfb, dfb.DFConfig.from_plane(plane, seed=9, plane_id=2), lags, 4, nplanes=3)
    for p in range(3):
        _check_exact(df, fields[p], False, plane=p)
        single, _ = _run(dfb, dfb.DFConfig.from_plane(plane, seed=9, plane_id=2 + p), lags, 4)
        for f in range(3):
            for d in range(3):
                assert np.array_equal(df.corr(f, d, False, plane=p)[0], single.corr(f, d, False)[0]), (p, f, d)
        single.close()
    df.close()


@gpu
def test_exact_at_headline_size(dfb, W):
    plane = W.NAMED["1024x2048_profile_N128"]()
    df, fields = _run(dfb, dfb.DFConfig.from_plane(plane, seed=3), (dfb.DFB_CORR_SUPPORT, dfb.DFB_CORR_SUPPORT, 8), 3)
    assert df.corr_lags == (256, 256, 8)
    _check_exact(df, fields[0], False)
    yc, vz = df.table(8), df.table(13, n=plane["Nz"] + 1)
    wbar = (vz[-1] - vz[0]) / plane["Nz"]
    xs = {0: lambda j, d: d * wbar, 1: lambda j, d: yc[j + d] - yc[j], 2: lambda j, d: float(d)}
    for f in range(3):
        for d in range(3):
            I = df.integral_scales(f, d)
            Iref = np_integral(df.corr(f, d)[0], xs[d])
            assert np.array_equal(np.isnan(I), np.isnan(Iref))
            assert normwise_close(np.nan_to_num(I), np.nan_to_num(Iref), TOL)[0], (f, d)
    df.close()


@gpu
def test_statistics_match_the_exact_expectation(dfb, W):
    """a periodic row-uniform plane, a few hundred steps: the normalised correlations and their integral scales against the
    expectation computed from the library's own coefficient tables, half-widths and row constants"""
    plane = W.plane_profile(256, 1024, 16, 16)
    Lt_u = plane["scales"][0][2]
    dt = 2.0 * Lt_u * np.log(2.0) / PI_BLEND                   # exp(-pi dt / (2 Lt_u)) = 0.5
    S, L = 300, (40, 40, 8)
    df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=2024, periodic_z=1), fetch=False)
    df.corr_enable(*L)
    for _ in range(S):
        df.filter(dt)
    Nyr = [df.half_widths(f, 0)[:, 0] for f in range(3)]
    Nzr = [df.half_widths(f, 1)[:, 0] for f in range(3)]
    cache = {}
    coef = lambda N: cache.setdefault(N, df.table(11, N))
    Lt = df.table(10)
    alpha = [np.exp(-PI_BLEND * dt / Lt[f]) for f in range(3)]
    exp = expected_rho(coef, Nyr, Nzr, df.rows(), alpha, plane["Nz"], L)
    yc, vz = df.table(8), df.table(13, n=plane["Nz"] + 1)
    wbar = (vz[-1] - vz[0]) / plane["Nz"]
    xs = {0: lambda j, d: d * wbar, 1: lambda j, d: yc[j + d] - yc[j], 2: lambda j, d: float(d)}
    for f in range(3):
        sig = sample_sigma(exp[f, 0], exp[f, 2], plane["Nz"] * S)
        for d in range(3):
            R, _, cnt = df.corr(f, d)
            assert cnt == S
            E = exp[f, d]
            assert np.array_equal(np.isnan(R), np.isnan(E)), (f, d)
            err = np.nanmax(np.abs(R - E) / sig[:, None])
            assert err < 6.0, (f, d, err)
            # integral scales: both trapezoids run over lags where |R - E| <= 6 sigma, and E falls monotonically to 0
            I, Ie = df.integral_scales(f, d), np_integral(E, xs[d])
            for j in range(plane["Ny"]):
                if np.isnan(Ie[j]):
                    assert np.isnan(I[j])
                    continue
                dmax = min(1, plane["Ny"] - 1 - j) if d == 1 else 1
                while dmax < L[d] and (d != 1 or j + dmax + 1 < plane["Ny"]) and (R[j, dmax] > 0 or E[j, dmax] > 0):
                    dmax += 1
                assert abs(I[j] - Ie[j]) <= 6.0 * sig[j] * abs(xs[d](j, dmax)) + 1e-300, (f, d, j, I[j], Ie[j])
    df.close()


@gpu
def test_determinism_and_no_side_effects(dfb, W):
    plane = _small_plane(W, Ny=64, Nz=96, N=16)
    lags = (dfb.DFB_CORR_SUPPORT, dfb.DFB_CORR_SUPPORT, 4)
    outs = []
    for on in (True, True, False):
        df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=4), fetch=False)
        df.stats_enable()
        if on:
            df.corr_enable(*lags)
        for _ in range(6):
            df.filter(1e-7)
        o = dict(fields=[df.get(i).copy() for i in range(5)], stats=[df.stats(i)[0] for i in range(6)])
        if on:
            o["corr"] = [df.corr(f, d, False)[0] for f in range(3) for d in range(3)]
        outs.append(o)
        df.close()
    for a, b in zip(outs[0]["corr"], outs[1]["corr"]):
        assert np.array_equal(a, b)
    for k in ("fields", "stats"):
        for a, b in zip(outs[0][k], outs[2][k]):
            assert np.array_equal(a, b), k


@gpu
def test_set_state_empties_the_ring(dfb, W):
    plane = _small_plane(W)
    df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=6), fetch=False)
    df.corr_enable(0, 0, 3)
    assert df.corr_lags == (0, 0, 3)
    seen = []
    for _ in range(3):
        df.filter(1e-7)
        seen.append(df.get(0).copy())
    fo, step = df.get_state()
    df.set_state(fo, step)
    after = []
    for _ in range(2):
        df.filter(1e-7)
        after.append(df.get(0).copy())
    S, pairs, cnt = df.corr(0, dfb.CORR_T, normalized=False)
    Nz = plane["Nz"]
    assert cnt == 5 and list(pairs) == [5 * Nz, 3 * Nz, 1 * Nz, 0]
    a, b = np_sums(seen, (0, 0, 3))[2][0], np_sums(after, (0, 0, 3))[2][0]
    assert normwise_close(S, a + b, TOL)[0]
    df.corr_enable(on=False)                  # off: the sums stay, nothing more accumulates
    df.filter(1e-7)
    assert np.array_equal(df.corr(0, dfb.CORR_T, normalized=False)[0], S)
    df.corr_enable(0, 0, 3)                   # on again with the same lags: the ring comes back empty, the sums restart
    again = []
    for _ in range(2):
        df.filter(1e-7)
        again.append(df.get(0).copy())
    S, pairs, cnt = df.corr(0, dfb.CORR_T, normalized=False)
    assert cnt == 2 and list(pairs) == [2 * Nz, Nz, 0, 0]
    assert normwise_close(S, np_sums(again, (0, 0, 3))[2][0], TOL)[0]
    df.close()


@gpu
def test_errors(dfb, W):
    plane = _small_plane(W)
    df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=1), fetch=False)

    def status(fn, *a):
        with pytest.raises(dfb.DfbError) as e:
            fn(*a)
        return e.value.code, str(e.value)

    assert status(df.corr, 0, 0)[0] == dfb.ERR_STATE
    assert status(df.integral_scales, 0, 0)[0] == dfb.ERR_STATE
    for lags in [(plane["Nz"], 0, 0), (0, plane["Ny"], 0), (0, 0, 65), (-2, 0, 0), (0, 0, -1)]:
        code, msg = status(df.corr_enable, *lags)
        assert code == dfb.ERR_ARG and "lag" in msg, lags
    df.corr_enable(4, 4, 2)
    out = np.zeros((plane["Ny"], 5))
    L = dfb.lib()
    for args in [(0, 3, 0, 0), (0, -1, 0, 0), (0, 0, 3, 0), (1, 0, 0, 0)]:     # plane, field, dir
        rc = L.dfb_corr_get_plane(df._h, args[0], args[1], args[2], 1, out.ctypes.data_as(dfb.c_dp), None, None)
        assert rc == dfb.ERR_ARG and L.dfb_last_error(), args
    df.close()
    slab = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=1, k_begin=0, k_end=16), fetch=False)
    code, msg = status(slab.corr_enable, 4, 4, 0)
    assert code == dfb.ERR_ARG and "correlation statistics need the whole plane" in msg
    slab.close()


@gpu
def test_cpp_facade_runs(dfb, W, tmp_path):
    plane = _small_plane(W)
    blob = np.concatenate([plane["yc"], plane["dy"], plane["dz"], np.ravel(plane["rows"]), np.ravel(plane["scales"])])
    (tmp_path / "plane.bin").write_bytes(np.ascontiguousarray(blob, dtype=np.float64).tobytes())
    exe = _cpp_build(tmp_path)
    r = subprocess.run([str(exe), str(tmp_path / "plane.bin")], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    tok = r.stdout.split()
    df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=5), fetch=False)
    df.corr_enable(dfb.DFB_CORR_SUPPORT, dfb.DFB_CORR_SUPPORT, 3)
    for _ in range(6):
        df.filter(1e-7)
    R = df.corr(1, dfb.CORR_Y, normalized=False)[0].ravel()
    I = df.integral_scales(2, dfb.CORR_Z)
    assert int(tok[0]) == R.size
    assert [float(t) for t in tok[1:]] == [R[0], R[R.size // 2], I[plane["Ny"] // 2]]
    df.close()
