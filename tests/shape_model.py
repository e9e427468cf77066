"""A numpy restatement of the two spatial sweeps with any coefficient table, and the oracle's step rebuilt on it: the reference for
handles whose filter shape is not the oracle's exponential (dfb_set_filter_shape).  The sweeps are the oracle's orc_sweep_y /
orc_sweep_z (oracle/df_oracle.c) with the table as an argument, summed in the same order (taps i = -N..N); tests/test_filter_shape_host.py
pins them against the oracle's with the exponential table.  The rest of the step is the oracle's own, unchanged: orc_correlate,
orc_rst_scaling and orc_sra."""
import ctypes as C
import functools

import numpy as np

from oracle_harness import Model


@functools.lru_cache(maxsize=None)
def gauss_coef(N):
    """Klein, Sadiki & Janicka's kernel of half-width N (n = N / 2): exp(-pi i^2 / (2 n^2)) = exp(-2 pi i^2 / N^2), unit energy"""
    if N == 0:
        return np.ones(1)
    i = np.arange(-N, N + 1, dtype=np.float64)
    t = np.exp(-2.0 * np.pi * i * i / (float(N) * N))
    return t / np.sqrt(np.sum(t * t))


def _by_N(Nmap):
    """{N: (rows that have a cell with that N, mask of those cells within the rows)}"""
    out = {}
    for N in np.unique(Nmap):
        rows = np.nonzero((Nmap == N).any(axis=1))[0]
        out[int(N)] = (rows, Nmap[rows] == N)
    return out


def sweep_y(coef, N_y, Ny_max, r_ys):
    """r_ys [Ny + 2 Ny_max, Nz] -> the y-filtered plane [Ny, Nz]: out[j, k] = sum_i b_i r_ys[j + Ny_max + i, k], N = N_y[j, k]"""
    Ny, Nz = N_y.shape
    out = np.zeros((Ny, Nz))
    for N, (rows, mask) in _by_N(N_y).items():
        b = coef(N)
        acc = np.zeros((len(rows), Nz))
        for i in range(-N, N + 1):
            acc += b[i + N] * r_ys[rows + Ny_max + i]
        out[rows] = np.where(mask, acc, out[rows])
    return out


def sweep_z(coef, N_z, M, r_zs):
    """r_zs [Ny, Nz + 2 M] (interior at column M) -> filt [Ny, Nz]: filt[j, k] = sum_i b_i r_zs[j, M + k + i], N = N_z[j, k]"""
    Ny, Nz = N_z.shape
    out = np.zeros((Ny, Nz))
    for N, (rows, mask) in _by_N(N_z).items():
        b = coef(N)
        acc = np.zeros((len(rows), Nz))
        for i in range(-N, N + 1):
            acc += b[i + N] * r_zs[rows, M + i:M + i + Nz]
        out[rows] = np.where(mask, acc, out[rows])
    return out


def shape_step(O, plane, coef, rys, halos, fo, dt, first_step=False, periodic=False):
    """One step of the oracle (orc_step's order) with the sweeps above: y-sweep per field into r_zs (halo columns = raw noise, or for a
    periodic plane the y-filtered columns of the other edge), z-sweep, then orc_correlate, orc_rst_scaling and orc_sra.  Returns
    dict(filt, fluc, filt_old, T, rho) like oracle.step."""
    L, d = O.lib(), O._d
    Ny, Nz = plane["Ny"], plane["Nz"]
    Lt = np.asarray(plane["scales"], dtype=np.float64)[:, 2]
    rows = np.ascontiguousarray(plane["rows"], dtype=np.float64)
    fo = [np.array(fo[f], dtype=np.float64).reshape(Ny, Nz).copy() for f in range(3)]
    filt, fluc = [], [np.zeros((Ny, Nz)) for _ in range(3)]
    T, rho = np.zeros((Ny, Nz)), np.zeros((Ny, Nz))
    for f in range(3):
        M = int(plane["Nz_max"][f])
        N_y, N_z = np.asarray(plane["N_y"][f]), np.asarray(plane["N_z"][f])
        rz = np.zeros((Ny, Nz + 2 * M))
        rz[:, M:M + Nz] = sweep_y(coef, N_y, int(plane["Ny_max"][f]), np.asarray(rys[f], dtype=np.float64))
        if periodic:
            rz[:, :M] = rz[:, Nz:Nz + M]
            rz[:, Nz + M:] = rz[:, M:2 * M]
        else:
            rz[:, :M], rz[:, Nz + M:] = halos[f][:, :M], halos[f][:, M:]
        filt.append(np.ascontiguousarray(sweep_z(coef, N_z, M, rz)))
        if not first_step:
            L.orc_correlate(C.c_long(Ny * Nz), d(fo[f]), d(filt[f]), C.c_double(dt), C.c_double(float(Lt[f])))
    r = [np.ascontiguousarray(rows[k]) for k in range(8)]  # R11, R21, R22, R33, Us, Ts, rhos, Ms
    L.orc_rst_scaling(C.c_int(Ny), C.c_int(Nz), d(r[0]), d(r[1]), d(r[2]), d(r[3]), d(filt[0]), d(filt[1]), d(filt[2]),
                      d(fluc[0]), d(fluc[1]), d(fluc[2]), d(fo[0]), d(fo[1]), d(fo[2]))
    if not first_step:
        L.orc_sra(C.c_int(Ny), C.c_int(Nz), d(r[7]), d(r[4]), d(r[5]), d(r[6]), d(fluc[0]), d(T), d(rho))
    return dict(filt=np.stack(filt), fluc=np.stack(fluc), filt_old=np.stack(fo), T=T, rho=rho)


class ShapeModel(Model):
    """oracle_harness.Model whose steps are shape_step with the table `coef` (N -> b[2N+1])"""

    def __init__(self, O, plane, seed, plane_id, coef, nplanes=1, periodic=False):
        super().__init__(O, plane, seed, plane_id, nplanes, periodic)
        self.coef = coef

    def filter(self, dt, first=False):
        for p in range(self.P):
            rys = [self.noise(p, f, self.step)[0] for f in range(3)]
            hal = [self.noise(p, f, self.step)[1] for f in range(3)]
            o = shape_step(self.O, self.plane, self.coef, rys, hal, self.fo[p], dt, first, self.periodic)
            self.fo[p] = o["filt_old"]
            self.out[p, :3] = o["fluc"]
            if not first:
                self.out[p, 3], self.out[p, 4] = o["T"], o["rho"]
        if not first:
            self._accumulate()
        self.noise_step = self.step
        self.step += 1
