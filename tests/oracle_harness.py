"""What the tests that compare a handle with the oracle share: a host model of a handle (Model), the oracle's step for a
spanwise-periodic plane (periodic_step), the numpy checker of the correlation sums (np_sums), planes whose half-widths are supplied
(explicit_plane, explicit_config), and one driver and one gate: inject() hands an inject-mode handle the model's noise, check()
compares every output of a handle with the model at the 1e-12 normwise gate, run() steps both and checks after every step."""
import numpy as np

from conftest import normwise_close

TOL = 1e-12


def package():
    """the package, without loading the library (the dfb fixture loads it)"""
    import _dfb_import  # noqa: F401
    import digital_filtering_b200
    return digital_filtering_b200


# ---------------------------------------------------------------------------------------------
# the oracle's restatements
# ---------------------------------------------------------------------------------------------
def np_sums(steps, L, periodic=False):
    """steps: fields [Ny, Nz] of one (plane, field) after consecutive accumulated steps (the ring never emptied in between).
    Returns {dir: (S [Ny, L+1], pairs [L+1])} for the directions with L[dir] > 0."""
    Ny, Nz = steps[0].shape
    out = {}
    Lz, Ly, Lt = L
    if Lz:
        S = np.zeros((Ny, Lz + 1))
        for f in steps:
            for d in range(Lz + 1):
                S[:, d] += (f * np.roll(f, -d, axis=1)).sum(1) if periodic else (f[:, :Nz - d] * f[:, d:]).sum(1)
        out[0] = (S, np.array([len(steps) * (Nz if periodic else Nz - d) for d in range(Lz + 1)], dtype=np.int64))
    if Ly:
        S = np.zeros((Ny, Ly + 1))
        for f in steps:
            for d in range(Ly + 1):
                S[:Ny - d, d] += (f[:Ny - d] * f[d:]).sum(1)
        out[1] = (S, np.full(Ly + 1, len(steps) * Nz, dtype=np.int64))
    if Lt:
        S = np.zeros((Ny, Lt + 1))
        pairs = np.zeros(Lt + 1, dtype=np.int64)
        for s in range(len(steps)):
            for m in range(min(Lt, s) + 1):
                S[:, m] += (steps[s] * steps[s - m]).sum(1)
                pairs[m] += Nz
        out[2] = (S, pairs)
    return out


def periodic_step(O, plane, rys, fo, dt, first_step=False):
    """The oracle's step for a spanwise-periodic plane, which the reference does not have: the plain-C restatement's stages
    (oracle/df_oracle.c, unchanged) recomposed in orc_step's order -- orc_sweep_y per field, then the halo columns of r_zs set to
    the y-filtered columns of the other edge (r_zs[:, :M] = r_zs[:, Nz:Nz+M], r_zs[:, Nz+M:] = r_zs[:, M:2M]; needs M <= Nz),
    then the unchanged orc_sweep_z, orc_correlate, orc_rst_scaling and orc_sra.  Returns dict(filt, fluc, filt_old, T, rho, r_zs)
    like oracle.step."""
    import ctypes as C
    L, d, i = O.lib(), O._d, O._i
    Ny, Nz = plane["Ny"], plane["Nz"]
    Lt = np.asarray(plane["scales"], dtype=np.float64)[:, 2]
    rows = np.ascontiguousarray(plane["rows"], dtype=np.float64)
    fo = [np.array(fo[f], dtype=np.float64).reshape(Ny, Nz).copy() for f in range(3)]
    filt = [np.zeros((Ny, Nz)) for _ in range(3)]
    fluc = [np.zeros((Ny, Nz)) for _ in range(3)]
    T, rho = np.zeros((Ny, Nz)), np.zeros((Ny, Nz))
    rzs = []
    for f in range(3):
        M = int(plane["Nz_max"][f])
        assert M <= Nz, (f, M, Nz)
        N_y = np.ascontiguousarray(plane["N_y"][f], dtype=np.int32)
        N_z = np.ascontiguousarray(plane["N_z"][f], dtype=np.int32)
        ry = np.ascontiguousarray(rys[f], dtype=np.float64)
        rz = np.full((Ny, Nz + 2 * M), np.nan)
        L.orc_sweep_y(C.c_int(Ny), C.c_int(Nz), C.c_int(int(plane["Ny_max"][f])), C.c_int(M), i(N_y), d(ry), d(rz))
        rz[:, :M] = rz[:, Nz:Nz + M]                       # left of column 0: columns Nz-M .. Nz-1
        rz[:, Nz + M:] = rz[:, M:2 * M]                    # right of column Nz-1: columns 0 .. M-1
        L.orc_sweep_z(C.c_int(Ny), C.c_int(Nz), C.c_int(M), i(N_z), d(rz), d(filt[f]))
        if not first_step:
            L.orc_correlate(C.c_long(Ny * Nz), d(fo[f]), d(filt[f]), C.c_double(dt), C.c_double(float(Lt[f])))
        rzs.append(rz)
    r = [np.ascontiguousarray(rows[k]) for k in range(8)]  # R11, R21, R22, R33, Us, Ts, rhos, Ms
    L.orc_rst_scaling(C.c_int(Ny), C.c_int(Nz), d(r[0]), d(r[1]), d(r[2]), d(r[3]), d(filt[0]), d(filt[1]), d(filt[2]),
                      d(fluc[0]), d(fluc[1]), d(fluc[2]), d(fo[0]), d(fo[1]), d(fo[2]))
    if not first_step:
        L.orc_sra(C.c_int(Ny), C.c_int(Nz), d(r[7]), d(r[4]), d(r[5]), d(r[6]), d(fluc[0]), d(T), d(rho))
    return dict(filt=np.stack(filt), fluc=np.stack(fluc), filt_old=np.stack(fo), T=T, rho=rho, r_zs=rzs)


# ---------------------------------------------------------------------------------------------
# the host model of a handle
# ---------------------------------------------------------------------------------------------
class Model:
    """What a generate-mode handle holds, per plane p (noise stream group plane_id + p), and what each call does to it.  The
    semantics are the library's (include/dfb200.h):
      - a step consumes the noise of (seed, plane_id + p, field, counter), then the counter moves on by one;
      - a first step (the constructor's, dfb_first_step) does not blend and leaves T' / rho' untouched;
      - a first step is not accumulated by N2 or by the correlation statistics;
      - dfb_set_state keeps the N2 sums and empties the correlation ring (the next step follows the restored state, not the ring);
      - dfb_set_state(NULL, s) moves only the counter; with filt_old it replaces filt_old as well;
      - dfb_stats_enable(1) zeroes the N2 sums and their count, (0) stops accumulating and keeps them;
      - dfb_corr_enable(1, lags) zeroes the sums, the pair counts and the step count and empties the ring, (0) stops accumulating
        and keeps the sums readable;
      - dfb_generate_noise(k) changes nothing but which noise dfb_get_noise returns.
    After a step, fo holds its filt u, v, w (the oracle's filt_old is its filt)."""

    def __init__(self, O, plane, seed, plane_id, nplanes=1, periodic=False):
        self.O, self.plane, self.seed, self.plane_id, self.P, self.periodic = O, plane, seed, plane_id, nplanes, periodic
        self.Ny, self.Nz = plane["Ny"], plane["Nz"]
        self.step = 0
        self.fo = np.zeros((nplanes, 3, self.Ny, self.Nz))
        self.out = np.zeros((nplanes, 5, self.Ny, self.Nz))          # u', v', w', T', rho'
        self.noise_step = None                                      # the step whose noise dfb_get_noise returns
        self.stats = None                                           # [P][6][Ny][Nz]: u'^2, v'^2, w'^2, T'^2, rho'^2, u'v'
        self.stats_on, self.stats_count = False, 0
        self.lags = None                                            # correlation statistics: None before any enable
        self.corr_on = False
        self._noise = {}

    def noise(self, p, f, step):
        key = (p, f, step)
        if key not in self._noise:
            pl, O = self.plane, self.O
            rys = O.noise_rys(self.seed, self.plane_id + p, f, step, self.Ny, pl["Ny_max"][f], self.Nz)
            hal = None if self.periodic else O.noise_halo(self.seed, self.plane_id + p, f, step, self.Ny, pl["Nz_max"][f])
            self._noise[key] = (rys, hal)
        return self._noise[key]

    def filter(self, dt, first=False):
        for p in range(self.P):
            rys = [self.noise(p, f, self.step)[0] for f in range(3)]
            if self.periodic:
                o = periodic_step(self.O, self.plane, rys, self.fo[p], dt, first_step=first)
            else:
                o = self.O.step(self.plane, rys, [self.noise(p, f, self.step)[1] for f in range(3)], self.fo[p], dt, first_step=first)
            self.fo[p] = o["filt_old"]
            self.out[p, :3] = o["fluc"]
            if not first:                                           # a first step leaves T', rho' untouched
                self.out[p, 3], self.out[p, 4] = o["T"], o["rho"]
        if not first:                                               # ... and is not accumulated
            self._accumulate()
        self.noise_step = self.step
        self.step += 1

    def first_step(self):
        self.filter(0.0, first=True)

    def _accumulate(self):
        if self.stats_on:
            u, v = self.out[:, 0], self.out[:, 1]
            self.stats[:, :5] += self.out * self.out
            self.stats[:, 5] += u * v
            self.stats_count += 1
        if self.corr_on:
            Lz, Ly, Lt = self.lags
            M = min(Lt, len(self.ring))
            for p in range(self.P):
                for f in range(3):
                    x = self.out[p, f]
                    s = np_sums([x], (Lz, Ly, 0), self.periodic)
                    for d in (0, 1):
                        if d in s:
                            self.csum[d][p, f] += s[d][0]
                    if Lt:
                        for m in range(M + 1):
                            self.csum[2][p, f][:, m] += (x * (x if m == 0 else self.ring[-m][p, f])).sum(1)
            if Lt:
                self.tsteps[:M + 1] += 1
                self.ring = (self.ring + [self.out[:, :3].copy()])[-Lt:]
            self.corr_count += 1

    def set_state(self, fo, step):
        if fo is not None:
            self.fo = np.array(fo, dtype=np.float64).reshape(3, self.P, self.Ny, self.Nz).transpose(1, 0, 2, 3).copy()
        self.step = step
        if self.lags is not None:
            self.ring = []                                          # the N2 and correlation sums stay

    def stats_enable(self, on):
        if on:
            self.stats = np.zeros((self.P, 6, self.Ny, self.Nz))
            self.stats_count = 0
        self.stats_on = bool(on)

    def corr_enable(self, on, lags=None):
        if on:
            self.lags = tuple(lags)
            self.csum = {d: np.zeros((self.P, 3, self.Ny, lags[d] + 1)) for d in range(3) if lags[d]}
            self.corr_count, self.tsteps, self.ring = 0, np.zeros(lags[2] + 1, dtype=np.int64), []
        self.corr_on = bool(on)

    def generate_noise(self, k):
        self.noise_step = k

    def state_for_library(self):
        """filt_old in the layout dfb_set_state takes: [3][P][Ny][Nz] ([3][Ny][Nz] for one plane)"""
        fo = self.fo.transpose(1, 0, 2, 3)
        return np.ascontiguousarray(fo[:, 0] if self.P == 1 else fo)

    def pairs(self, d):
        Lz = self.lags[d]
        if d == 0:
            return np.array([self.corr_count * (self.Nz if self.periodic else self.Nz - e) for e in range(Lz + 1)], dtype=np.int64)
        if d == 1:
            return np.full(Lz + 1, self.corr_count * self.Nz, dtype=np.int64)
        return self.tsteps * self.Nz


# ---------------------------------------------------------------------------------------------
# planes whose half-widths are supplied
# ---------------------------------------------------------------------------------------------
def explicit_plane(W, Ny, Nz, Ny_rows, Nz_rows):
    """row-uniform plane whose half-widths are supplied per row (dfb_config.N_y / N_z) instead of derived from geometry"""
    yc = (np.arange(Ny) + 0.5) * 1e-5
    N_y = np.stack([np.repeat(np.asarray(Ny_rows[f], dtype=np.int32)[:, None], Nz, axis=1) for f in range(3)])
    N_z = np.stack([np.repeat(np.asarray(Nz_rows[f], dtype=np.int32)[:, None], Nz, axis=1) for f in range(3)])
    return dict(name=f"explicit_{Ny}x{Nz}", Ny=Ny, Nz=Nz, d_i=W.D_I, U_e=W.U_E, yc=yc, dy=np.full(Ny, 1e-5), dz=np.full(Ny, 1e-5),
                rows=W.synthetic_rows(yc + 1e-4), scales=W._scales(W.D_I), explicit_N=True,
                N_y=N_y, N_z=N_z, Ny_max=[int(N_y[f].max()) for f in range(3)], Nz_max=[int(N_z[f].max()) for f in range(3)])


def explicit_config(dfbm, plane, **kw):
    cfg = dfbm.DFConfig.from_plane(plane, **kw)
    cfg.geom_per_row = 0
    cfg.yc = cfg.dy = cfg.dz = None
    cfg.N_y, cfg.N_z = plane["N_y"], plane["N_z"]
    return cfg


# ---------------------------------------------------------------------------------------------
# the driver and the gate
# ---------------------------------------------------------------------------------------------
def inject(df, m):
    """hand an inject-mode handle the model's noise for the model's next step (plane 0); no halo for a periodic plane or a field
    with Nz_max = 0"""
    for f in range(3):
        rys, hal = m.noise(0, f, m.step)
        df.set_noise(f, rys, hal if m.plane["Nz_max"][f] else None)


# dfb_get_field selector of each output, in the order check() compares them, and the kind of output its worst ratio is kept under
OUTPUTS = ((5, "filt"), (6, "filt"), (7, "filt"), (0, "fluc"), (1, "fluc"), (2, "fluc"), (3, "T"), (4, "rho"))


def check(df, m, k=None, tol=TOL, worst=None):
    """Every output of every plane of handle df against model m at the normwise gate: u', v', w', T', rho' against m.out, filt u, v, w
    against m.fo.  An output the model holds at 0 (T', rho' after the constructor's step) must be exactly 0.  k = (k0, k1): df is a
    slab, compared with the model's columns [k0, k1).  Returns the worst ratio per kind of output (filt, fluc, T, rho), kept in
    `worst` across calls when given."""
    worst = {} if worst is None else worst
    cols = slice(None) if k is None else slice(k[0], k[1])
    for p in range(m.P):
        for which, kind in OUTPUTS:
            ref = (m.fo[p, which - 5] if which >= 5 else m.out[p, which])[:, cols]
            got = df.get(which, plane=p)
            ok, r = normwise_close(got, ref, tol)
            if not ref.any():
                ok = not got.any()
            worst[kind] = max(worst.get(kind, 0.0), r)
            assert ok, (m.plane.get("name"), "counter", m.step - 1, "plane", p, "output", which, r)
    return worst


def run(df, m, dts, k=None):
    """The constructor's step and one filter(dt) per dt on handle df and model m, check() after each step.  An inject-mode handle is
    handed the model's noise before every step and takes the first one through dfb_first_step.  Returns check()'s worst."""
    injected = df.noise_mode == package().NOISE_INJECT
    worst = {}
    for dt in [None] + list(dts):
        if injected:
            inject(df, m)
            df.first_step() if dt is None else df.filter(dt)
        elif dt is not None:
            df.filter(dt)
        m.first_step() if dt is None else m.filter(dt)
        check(df, m, k, worst=worst)
    return worst
