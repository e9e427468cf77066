"""oracle/oracle.py -- TEST INFRASTRUCTURE ONLY.

ctypes front-end to the two CPU checkers:
  * libdforacle.so      our plain-C restatement (df_oracle.c, pcg32_oracle.c, normal_oracle.c)
  * _ref/libdfref.so    the reference's own df.cpp compiled from /root/reference (ref_shim.cpp);
                        prebuilt here, travels to the GPU box, absent -> RefFilter unavailable.
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference / default-plane legs may
import this module.  The product (digital-filtering_b200/) never does.
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(HERE, "_ref")
REF_RUN = os.path.join(REF_DIR, "run")
REF_FILES = os.path.join(REF_DIR, "files")
RST_DAT = os.path.join(REF_FILES, "RST.dat")
LINE_DAT = os.path.join(REF_DIR, "line.dat")

c_dp = C.POINTER(C.c_double)
c_ip = C.POINTER(C.c_int)


def build(quiet=True):
    """make -C oracle (restatement always; _ref only when /root/reference is present)."""
    r = subprocess.run(["make", "-C", HERE, "all"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("oracle build failed:\n" + r.stdout + r.stderr)
    if not quiet:
        print(r.stdout)


_lib = None
_ref = None


def lib():
    global _lib
    if _lib is None:
        p = os.path.join(HERE, "libdforacle.so")
        if not os.path.exists(p):
            build()
        _lib = C.CDLL(p)
        _lib.orc_pcg32_kat_text.restype = C.c_int
    return _lib


def have_ref():
    return os.path.exists(os.path.join(REF_DIR, "libdfref.so")) and os.path.exists(RST_DAT) and os.path.exists(LINE_DAT)


def reflib():
    global _ref
    if _ref is None:
        if not have_ref():
            raise RuntimeError("oracle/_ref is not built (needs /root/reference at build time)")
        L = C.CDLL(os.path.join(REF_DIR, "libdfref.so"))
        L.ref_create.restype = C.c_void_p
        L.ref_create.argtypes = [C.c_char_p]
        L.ref_scalar.restype = C.c_double
        L.ref_field_scalar.restype = C.c_double
        L.ref_time_steps.restype = C.c_double
        L.ref_pcg32_distance.restype = C.c_uint64
        for fn in ("ref_get_vec", "ref_get_fvec", "ref_set_fvec", "ref_get_ivec"):
            getattr(L, fn).restype = C.c_long
        _ref = L
    return _ref


def _d(a):
    return a.ctypes.data_as(c_dp)


def _i(a):
    return a.ctypes.data_as(c_ip)


# ------------------------------------------------------------------------------------------------
# pcg32 + normals
# ------------------------------------------------------------------------------------------------
def pcg32_draw(seed, stream, delta, n, has_stream=True):
    out = np.zeros(n, dtype=np.uint32)
    lib().orc_pcg32_draw(C.c_uint64(seed), C.c_uint64(stream), C.c_int(int(has_stream)), C.c_uint64(delta),
                         C.c_int(n), out.ctypes.data_as(C.c_void_p))
    return out


def pcg32_state(seed, stream, has_stream=True):
    s, i = C.c_uint64(), C.c_uint64()
    lib().orc_pcg32_state(C.c_uint64(seed), C.c_uint64(stream), C.c_int(int(has_stream)), C.byref(s), C.byref(i))
    return s.value, i.value


def pcg32_kat_text(two_arg, rounds=5):
    buf = C.create_string_buffer(1 << 16)
    n = lib().orc_pcg32_kat_text(C.c_int(int(two_arg)), C.c_int(rounds), buf, C.c_int(len(buf)))
    return buf.raw[:n].decode()


def ref_pcg32_draw(seed, stream, delta, n, has_stream=True):
    out = np.zeros(n, dtype=np.uint32)
    reflib().ref_pcg32_draw(C.c_uint64(seed), C.c_uint64(stream), C.c_int(int(has_stream)), C.c_uint64(delta),
                            C.c_int(n), out.ctypes.data_as(C.c_void_p))
    return out


def normal_pair(o4):
    o = np.ascontiguousarray(o4, dtype=np.uint32)
    z = np.zeros(2)
    lib().orc_normal_pair(o.ctypes.data_as(C.c_void_p), _d(z))
    return z


def noise_elements(seed, stream, step, length, e0, n):
    out = np.zeros(n)
    lib().orc_noise_elements(C.c_uint64(seed), C.c_uint64(stream), C.c_uint64(step), C.c_uint64(length),
                             C.c_uint64(e0), C.c_uint64(n), _d(out))
    return out


def noise_rys(seed, plane, field, step, Ny, Ny_max, NzG, k0=0, k1=None):
    k1 = NzG if k1 is None else k1
    out = np.zeros((Ny + 2 * Ny_max, k1 - k0))
    lib().orc_noise_rys(C.c_uint64(seed), C.c_int(plane), C.c_int(field), C.c_uint64(step), C.c_int(Ny),
                        C.c_int(Ny_max), C.c_int(NzG), C.c_int(k0), C.c_int(k1), _d(out))
    return out


def noise_halo(seed, plane, field, step, Ny, Nz_max):
    out = np.zeros((Ny, 2 * Nz_max))
    lib().orc_noise_halo(C.c_uint64(seed), C.c_int(plane), C.c_int(field), C.c_uint64(step), C.c_int(Ny),
                         C.c_int(Nz_max), _d(out))
    return out


# ------------------------------------------------------------------------------------------------
# setup restatement
# ------------------------------------------------------------------------------------------------
def coeffs(N):
    b = np.zeros(2 * N + 1)
    lib().orc_coeffs(C.c_int(N), _d(b))
    return b


def linear_interpolate(y_data, f_data, y_new):
    y_data = np.ascontiguousarray(y_data, dtype=np.float64)
    f_data = np.ascontiguousarray(f_data, dtype=np.float64)
    y_new = np.ascontiguousarray(y_new, dtype=np.float64)
    out = np.zeros(len(y_new))
    lib().orc_linear_interpolate(C.c_int(len(y_data)), _d(y_data), _d(f_data), C.c_int(len(y_new)), _d(y_new), _d(out))
    return out


def half_widths(plane):
    """Fills plane['N_y'], ['N_z'] ([3,Ny,Nz] int32), ['Ny_max'], ['Nz_max'] (df.cpp:144-154,186-195)."""
    Ny, Nz = plane["Ny"], plane["Nz"]
    yc = np.ascontiguousarray(np.broadcast_to(np.asarray(plane["yc"], dtype=np.float64).reshape(Ny, -1), (Ny, Nz)))
    dy = np.ascontiguousarray(np.broadcast_to(np.asarray(plane["dy"], dtype=np.float64).reshape(Ny, -1), (Ny, Nz)))
    dz = np.ascontiguousarray(np.broadcast_to(np.asarray(plane["dz"], dtype=np.float64).reshape(-1, 1) if np.ndim(plane["dz"]) < 2 else plane["dz"], (Ny, Nz)))
    N_y = np.zeros((3, Ny, Nz), dtype=np.int32)
    N_z = np.zeros((3, Ny, Nz), dtype=np.int32)
    Ny_max, Nz_max = [], []
    for f in range(3):
        a, b = C.c_int(), C.c_int()
        lib().orc_half_widths(C.c_int(Ny), C.c_int(Nz), _d(yc), _d(dy), _d(dz), C.c_double(plane["d_i"]),
                              C.c_double(plane["scales"][f][0]), C.c_double(plane["scales"][f][1]),
                              _i(N_y[f]), _i(N_z[f]), C.byref(a), C.byref(b))
        Ny_max.append(a.value)
        Nz_max.append(b.value)
    plane.update(N_y=N_y, N_z=N_z, Ny_max=Ny_max, Nz_max=Nz_max)
    return plane


def _read_zone_file(path):
    """Both data files: one VARIABLES line, one 'ZONE ... i=N' line, then N rows (df.cpp:231-278,498-537)."""
    with open(path) as fh:
        fh.readline()
        zone = fh.readline()
        n = int(float(zone.split("i=")[1].split()[0]))
        rows = [[float(x) for x in ln.split()] for ln in fh if ln.strip()]
    return np.array(rows[:n])


DEFAULT_TABLES = os.path.join(os.path.dirname(HERE), "tests", "golden", "default_tables.npz")


def stored_default_plane(path=DEFAULT_TABLES):
    """The reference's default 510x400 plane as its own setup left it (tests/golden/default_tables.npz, written from the running
    reference object by tests/golden/make_golden.py): geometry, row tables, integral scales and half-widths, in the workload form
    DFConfig.from_plane takes.  d_i and the uniform spanwise spacing are the reference's constants (df.cpp:7-16)."""
    g = np.load(path)
    Ny, Nz = int(g["Ny"]), int(g["Nz"])
    return dict(name="reference_default_plane_510x400", Ny=Ny, Nz=Nz, d_i=0.0013, yc=g["yc"], dy=g["dy"], dz=np.full(Ny, 0.000133),
                rows=g["rows"], scales=g["scales"], N_y=np.repeat(g["N_y"][:, :, None], Nz, axis=2),
                N_z=np.repeat(g["N_z"][:, :, None], Nz, axis=2), Ny_max=[int(x) for x in g["Ny_max"]], Nz_max=[int(x) for x in g["Nz_max"]])


def default_plane(rst_path=RST_DAT, line_path=LINE_DAT):
    """Restatement of the constructor's setup for the reference's hard-coded case:
    df.cpp:7-16 (constants), read_grid 71-118, get_RST_in 220-330, read_line_file 487-553,
    integral scales 35-45."""
    d_i, U_e, mu, gcon = 0.0013, 869.1, 7.1212e-6, 287.0
    Ny0, Nz = 560, 400
    yv, yc, dy = np.zeros(Ny0 + 1), np.zeros(Ny0), np.zeros(Ny0)
    lib().orc_default_grid(C.c_int(Ny0), C.c_double(d_i), _d(yv), _d(yc), _d(dy))
    yc_d = yc / d_i
    rst = _read_zone_file(rst_path)
    yin_d = rst[:, 1].copy()
    Ny = 0
    while Ny < Ny0 and yc_d[Ny] <= yin_d[-1]:      # df.cpp:282-288
        Ny += 1
    yc, dy, yc_d = yc[:Ny].copy(), dy[:Ny].copy(), yc_d[:Ny].copy()
    line = _read_zone_file(line_path)
    y_file, rho_file, u_file, T_file, p_file = (line[:, c].copy() for c in (1, 4, 5, 8, 9))
    Us = linear_interpolate(y_file, u_file, yc)
    Ts = linear_interpolate(y_file, T_file, yc)
    rhos = linear_interpolate(y_file, rho_file, yc)
    Ms = Us / np.sqrt(1.4 * gcon * Ts)             # df.cpp:544
    tau_w = mu * (Us[1] - Us[0]) / (y_file[1] - y_file[0])   # df.cpp:547-549 (quirk 10)
    u_tau = np.sqrt(tau_w / rhos[0])
    R11_in = rst[:, 2] * rst[:, 2] * u_tau * u_tau # df.cpp:313-316
    R22_in = rst[:, 3] * rst[:, 3] * u_tau * u_tau
    R33_in = rst[:, 4] * rst[:, 4] * u_tau * u_tau
    R21_in = rst[:, 5] * u_tau * u_tau
    rows = np.stack([linear_interpolate(yin_d, R11_in, yc_d), linear_interpolate(yin_d, R21_in, yc_d),
                     linear_interpolate(yin_d, R22_in, yc_d), linear_interpolate(yin_d, R33_in, yc_d),
                     Us, Ts, rhos, Ms])
    d_v = d_i / 4500                                # df.cpp:326
    scales = [[150 * d_v, 0.4 * d_i, 0.8 * d_i / U_e],   # u  (Iz_inn, Iz_out, Lt)  df.cpp:35-37
              [75 * d_v, 0.3 * d_i, 0.3 * d_i / U_e],    # v  df.cpp:39-41
              [150 * d_v, 0.4 * d_i, 0.3 * d_i / U_e]]   # w  df.cpp:43-45
    plane = dict(Ny=Ny, Nz=Nz, d_i=d_i, yc=yc, dy=dy, dz=np.full(Ny, 0.000133), rows=rows,
                 scales=np.array(scales), u_tau=u_tau, tau_w=tau_w)
    return half_widths(plane)


# ------------------------------------------------------------------------------------------------
# hot path
# ------------------------------------------------------------------------------------------------
def make_rzs(halo, Ny, Nz, Nz_max, fill=np.nan):
    """r_zs in the reference's layout with the (dead) interior poisoned and the raw-noise halo
    columns in place (SURVEY quirk 1/4)."""
    rz = np.full((Ny, Nz + 2 * Nz_max), fill)
    rz[:, :Nz_max] = halo[:, :Nz_max]
    rz[:, Nz + Nz_max:] = halo[:, Nz_max:]
    return rz


def _pp(arrs, ctype):
    return (C.POINTER(ctype) * len(arrs))(*[a.ctypes.data_as(C.POINTER(ctype)) for a in arrs])


def step(plane, r_ys, halos, filt_old, dt, first_step=False):
    """One filter(dt) (df.cpp:449-461) on injected noise.  r_ys[f]: (Ny+2Ny_max[f], Nz); halos[f]:
    (Ny, 2*Nz_max[f]); filt_old: [3,Ny,Nz].  Returns dict(filt, fluc, filt_old, T, rho, r_zs)."""
    Ny, Nz = plane["Ny"], plane["Nz"]
    N_y = [np.ascontiguousarray(plane["N_y"][f]) for f in range(3)]
    N_z = [np.ascontiguousarray(plane["N_z"][f]) for f in range(3)]
    Ny_max = np.array(plane["Ny_max"], dtype=np.int32)
    Nz_max = np.array(plane["Nz_max"], dtype=np.int32)
    Lt = np.ascontiguousarray(np.asarray(plane["scales"])[:, 2], dtype=np.float64)
    rows = np.ascontiguousarray(plane["rows"], dtype=np.float64)
    rys = [np.ascontiguousarray(r_ys[f], dtype=np.float64) for f in range(3)]
    rzs = [make_rzs(np.asarray(halos[f]), Ny, Nz, int(Nz_max[f])) for f in range(3)]
    fo = [np.array(filt_old[f], dtype=np.float64).reshape(Ny, Nz).copy() for f in range(3)]
    filt = [np.zeros((Ny, Nz)) for _ in range(3)]
    fluc = [np.zeros((Ny, Nz)) for _ in range(3)]
    T, rho = np.zeros((Ny, Nz)), np.zeros((Ny, Nz))
    lib().orc_step(C.c_int(Ny), C.c_int(Nz), _pp(N_y, C.c_int), _pp(N_z, C.c_int), _i(Ny_max), _i(Nz_max),
                   _d(Lt), _d(rows), C.c_double(dt), C.c_int(int(first_step)),
                   _pp(rys, C.c_double), _pp(rzs, C.c_double), _pp(fo, C.c_double), _pp(filt, C.c_double),
                   _pp(fluc, C.c_double), _d(T), _d(rho))
    return dict(filt=np.stack(filt), fluc=np.stack(fluc), filt_old=np.stack(fo), T=T, rho=rho, r_zs=rzs)


# ------------------------------------------------------------------------------------------------
# the true reference object
# ------------------------------------------------------------------------------------------------
class RefFilter:
    """DIGITAL_FILTER from the reference's own df.cpp (oracle/_ref/libdfref.so)."""

    VEC = dict(R11=0, R21=1, R22=2, R33=3, Us=4, Ts=5, rhos=6, Ms=7, Ps=8, yline=9, ydline=10, yc=11, dy=12,
               dz=13, y=14, z=15, T_fluc=16, rho_fluc=17, yin_d=18, R11_in=19)
    FVEC = dict(by=0, bz=1, r_ys=2, r_zs=3, filt_old=4, filt=5, fluc=6)
    IVEC = dict(N_ys=0, N_zs=1, by_offsets=2, bz_offsets=3)

    def __init__(self):
        self.L = reflib()
        os.makedirs(REF_RUN, exist_ok=True)
        cwd = os.getcwd()
        try:
            self.h = C.c_void_p(self.L.ref_create(REF_RUN.encode()))
        finally:
            os.chdir(cwd)
        if not self.h:
            raise RuntimeError("reference constructor failed (data files missing under oracle/_ref?)")

    def close(self):
        if self.h:
            self.L.ref_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def dims(self):
        a, b = C.c_int(), C.c_int()
        self.L.ref_dims(self.h, C.byref(a), C.byref(b))
        return a.value, b.value

    def scalar(self, which):
        return self.L.ref_scalar(self.h, C.c_int(which))

    def field_scalar(self, f, which):
        return self.L.ref_field_scalar(self.h, C.c_int(f), C.c_int(which))

    def vec(self, name):
        n = self.L.ref_get_vec(self.h, C.c_int(self.VEC[name]), None, C.c_long(0))
        out = np.zeros(n)
        self.L.ref_get_vec(self.h, C.c_int(self.VEC[name]), _d(out), C.c_long(n))
        return out

    def fvec(self, f, name):
        n = self.L.ref_get_fvec(self.h, C.c_int(f), C.c_int(self.FVEC[name]), None, C.c_long(0))
        out = np.zeros(n)
        self.L.ref_get_fvec(self.h, C.c_int(f), C.c_int(self.FVEC[name]), _d(out), C.c_long(n))
        return out

    def set_fvec(self, f, name, a):
        a = np.ascontiguousarray(a, dtype=np.float64).ravel()
        r = self.L.ref_set_fvec(self.h, C.c_int(f), C.c_int(self.FVEC[name]), _d(a), C.c_long(a.size))
        if r != a.size:
            raise ValueError(f"size mismatch setting {name}: reference holds {-r}, got {a.size}")

    def ivec(self, f, name):
        n = self.L.ref_get_ivec(self.h, C.c_int(f), C.c_int(self.IVEC[name]), None, C.c_long(0))
        out = np.zeros(n, dtype=np.int32)
        self.L.ref_get_ivec(self.h, C.c_int(f), C.c_int(self.IVEC[name]), _i(out), C.c_long(n))
        return out

    def reshape(self, plane):
        """Synthetic shape: overwrite geometry + row tables, re-run the reference's own
        allocate_data_structures / calculate_filter_properties (SURVEY 8c)."""
        Ny, Nz = plane["Ny"], plane["Nz"]
        bc = lambda a: np.ascontiguousarray(np.broadcast_to(np.asarray(a, dtype=np.float64).reshape(Ny, -1), (Ny, Nz)))
        yc, dy, dz = bc(plane["yc"]), bc(plane["dy"]), bc(plane["dz"])
        rows = np.ascontiguousarray(plane["rows"], dtype=np.float64)
        scales = np.ascontiguousarray(plane["scales"], dtype=np.float64)
        self.L.ref_reshape(self.h, C.c_int(Ny), C.c_int(Nz), C.c_double(plane["d_i"]), _d(yc), _d(dy), _d(dz),
                           _d(rows), _d(scales))

    def plane(self):
        """The tables of the running reference object as a plane dict."""
        Ny, Nz = self.dims
        rows = np.stack([self.vec(k) for k in ("R11", "R21", "R22", "R33", "Us", "Ts", "rhos", "Ms")])
        scales = np.array([[self.field_scalar(f, 1), self.field_scalar(f, 2), self.field_scalar(f, 0)] for f in range(3)])
        n = Ny * Nz   # dz is not trimmed with the other geometry vectors (df.cpp:297-304)
        return dict(Ny=Ny, Nz=Nz, d_i=self.scalar(0), yc=self.vec("yc")[:n].reshape(Ny, Nz),
                    dy=self.vec("dy")[:n].reshape(Ny, Nz), dz=self.vec("dz")[:n].reshape(Ny, Nz), rows=rows, scales=scales,
                    N_y=np.stack([self.ivec(f, "N_ys").reshape(Ny, Nz) for f in range(3)]),
                    N_z=np.stack([self.ivec(f, "N_zs").reshape(Ny, Nz) for f in range(3)]),
                    Ny_max=[int(self.field_scalar(f, 3)) for f in range(3)],
                    Nz_max=[int(self.field_scalar(f, 4)) for f in range(3)])

    def inject(self, r_ys, halos, filt_old=None):
        Ny, Nz = self.dims
        for f in range(3):
            self.set_fvec(f, "r_ys", r_ys[f])
            self.set_fvec(f, "r_zs", make_rzs(np.asarray(halos[f]), Ny, Nz, int(self.field_scalar(f, 4))))
            if filt_old is not None:
                self.set_fvec(f, "filt_old", filt_old[f])

    def step_injected(self, dt):
        self.L.ref_step_injected(self.h, C.c_double(dt))

    def first_step_injected(self):
        self.L.ref_first_step_injected(self.h)

    def filter(self, dt):
        cwd = os.getcwd()
        os.chdir(REF_RUN)
        try:
            self.L.ref_filter(self.h, C.c_double(dt))
        finally:
            os.chdir(cwd)

    def outputs(self):
        Ny, Nz = self.dims
        return dict(filt=np.stack([self.fvec(f, "filt").reshape(Ny, Nz) for f in range(3)]),
                    fluc=np.stack([self.fvec(f, "fluc").reshape(Ny, Nz) for f in range(3)]),
                    filt_old=np.stack([self.fvec(f, "filt_old").reshape(Ny, Nz) for f in range(3)]),
                    T=self.vec("T_fluc").reshape(Ny, Nz), rho=self.vec("rho_fluc").reshape(Ny, Nz))

    def halos(self):
        """The raw-noise halo columns that survive a sweep (r_zs minus its interior)."""
        Ny, Nz = self.dims
        out = []
        for f in range(3):
            M = int(self.field_scalar(f, 4))
            rz = self.fvec(f, "r_zs").reshape(Ny, Nz + 2 * M)
            out.append(np.concatenate([rz[:, :M], rz[:, Nz + M:]], axis=1))
        return out

    def time_steps(self, dt, nsteps):
        st = np.zeros(5)
        tot = self.L.ref_time_steps(self.h, C.c_double(dt), C.c_int(nsteps), _d(st))
        return tot, st
