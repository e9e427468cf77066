"""digital_filtering_b200 -- host-side mirror of the reference's DIGITAL_FILTER interface over the C ABI.

The directory is named `digital-filtering_b200` (not importable as written); `_dfb_import.py` at the
repo root registers it as the module `digital_filtering_b200`.

The compute path is libdfb200.so (hand-written sm_100a CUDA, csrc/).  Nothing here computes:
this module only marshals arguments through ctypes, exactly like the C++ facade
(include/digital_filter.hpp) and the Fortran module (fortran/digital_filtering.f90) do.  If the
library is missing the import fails loudly; there is no Python / CPU fallback.

Reference surface mirrored (digital-filtering-c++/df/df.hpp):
    DFConfig                 df.hpp:38-49
    DIGITAL_FILTER(config)   df.hpp:89, df.cpp:4-66
    .filter(dt_input)        df.hpp:100, df.cpp:449-468
    .u/.v/.w (.fluc, .filt)  df.hpp:24-34, 87;  .T_fluc / .rho_fluc  df.hpp:59
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DFB_LIB") or os.path.join(_HERE, "lib", "libdfb200.so")   # DFB_LIB: development builds side by side

OK, ERR_ARG, ERR_IO, ERR_CUDA, ERR_STATE, ERR_INTERP = range(6)
U_FLUC, V_FLUC, W_FLUC, T_FLUC, RHO_FLUC, U_FILT, V_FILT, W_FILT = range(8)
NOISE_GENERATE, NOISE_INJECT = 0, 1
FILTER_EXPONENTIAL, FILTER_GAUSSIAN = 0, 1    # filter shapes (dfb_set_filter_shape)
FLUX_OFF, FLUX_MASS, FLUX_VOLUME = 0, 1, 2    # inflow flux correction modes (dfb_set_flux_correction)
CORR_Z, CORR_Y, CORR_T = 0, 1, 2        # correlation directions (dfb_corr_enable)
DFB_CORR_SUPPORT = CORR_SUPPORT = -1    # lag = the filter's whole support (z and y)
RESTART_STATE, RESTART_STATS, RESTART_CORR = 1, 2, 4   # sections of a restart file (dfb_save_restart)
MAP_POINT, MAP_AREA = 0, 1               # face maps (dfb_facemap_create): bilinear at the face centre / average over the face
MAP_WALL_ZERO = 1                        # point maps: linear to 0 at the wall below the first cell centre
FLUCS = (U_FLUC, V_FLUC, W_FLUC, T_FLUC, RHO_FLUC)
RESTART_INFO = ("version", "Ny", "Nz", "plane_id", "nplanes", "seed", "periodic_z", "noise_mode", "step", "sections", "records",
                "fingerprint", "Ny_max_u", "Ny_max_v", "Ny_max_w", "Nz_max_u", "Nz_max_v", "Nz_max_w", "tuned", "z_form", "y_form",
                "stats_count", "stats_on", "corr_lag_z", "corr_lag_y", "corr_lag_t", "corr_count", "corr_on", "ring_fields", "bytes")

c_dp = C.POINTER(C.c_double)
c_ip = C.POINTER(C.c_int)


class DfbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"dfb200 error {code}: {msg}")
        self.code = code


class dfb_config(C.Structure):
    """ctypes image of `struct dfb_config` (include/dfb200.h)."""
    _fields_ = [
        ("d_i", C.c_double), ("rho_e", C.c_double), ("U_e", C.c_double), ("mu_e", C.c_double),
        ("vel_file_offset", C.c_int), ("vel_file_N_values", C.c_int),
        ("grid_file", C.c_char_p), ("grid_file_len", C.c_int),
        ("vel_fluc_file", C.c_char_p), ("vel_fluc_file_len", C.c_int),
        ("struct_bytes", C.c_int), ("honor_flow_config", C.c_int),
        ("line_file", C.c_char_p), ("line_file_len", C.c_int),
        ("Ny", C.c_int), ("Nz", C.c_int), ("geom_per_row", C.c_int),
        ("yc", c_dp), ("dy", c_dp), ("dz", c_dp), ("rows", c_dp), ("scales", c_dp),
        ("N_y", c_ip), ("N_z", c_ip),
        ("seed", C.c_uint64), ("noise_mode", C.c_int), ("device", C.c_int), ("plane_id", C.c_int),
        ("k_begin", C.c_int), ("k_end", C.c_int), ("skip_first_step", C.c_int), ("kernel_variant", C.c_int),
        ("periodic_z", C.c_int),
    ]


_lib = None


def lib():
    """Loads libdfb200.so.  Missing library = hard error (no fallback of any kind)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(make -C digital-filtering_b200/csrc). There is no CPU fallback.")
        # libdfb200.so links libnccl.so.2 (config 4's hand-off).  If PyTorch's bundled NCCL is installed, bring that copy in first so that
        # the process holds ONE NCCL whichever of torch / this library is imported first (same soname: the loader would otherwise hand
        # torch the system copy, which may be older than the one it was built against).
        try:
            import importlib.util
            spec = importlib.util.find_spec("nvidia.nccl")
            if spec and spec.submodule_search_locations:
                cand = os.path.join(list(spec.submodule_search_locations)[0], "lib", "libnccl.so.2")
                if os.path.exists(cand):
                    C.CDLL(cand, mode=C.RTLD_GLOBAL)
        except Exception:
            pass
        L = C.CDLL(LIB_PATH)
        L.dfb_last_error.restype = C.c_char_p
        L.dfb_version.restype = C.c_char_p
        L.dfb_create.argtypes = [C.POINTER(dfb_config), C.POINTER(C.c_void_p)]
        L.dfb_create_batch.argtypes = [C.POINTER(dfb_config), C.c_int, C.POINTER(C.c_void_p)]
        L.dfb_num_planes.argtypes = [C.c_void_p, c_ip]
        L.dfb_get_field_plane.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int]
        L.dfb_device_ptr_plane.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.dfb_stats_get_plane.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, c_dp, C.POINTER(C.c_int64)]
        L.dfb_get_rms.argtypes = [C.c_void_p, C.c_int, C.c_double]
        L.dfb_write_rms_csv.argtypes = [C.c_void_p, C.c_char_p]
        L.dfb_write_tecplot.argtypes = [C.c_void_p, C.c_char_p]
        L.dfb_face_map.argtypes = [C.c_void_p, C.c_int, c_dp, c_dp, c_ip]
        L.dfb_comm_unique_id.argtypes = [C.c_void_p]
        L.dfb_comm_init.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        L.dfb_comm_info.argtypes = [C.c_void_p, c_ip, c_ip, c_ip]
        L.dfb_gather_begin.argtypes = [C.c_void_p, C.c_int]
        L.dfb_gather_end.argtypes = [C.c_void_p]
        L.dfb_gathered_ptr.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]
        L.dfb_gathered_to_host.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.dfb_gather_wire_bytes.argtypes = [C.c_void_p, C.POINTER(C.c_int64)]
        L.dfb_comm_destroy.argtypes = [C.c_void_p]
        L.dfb_comm_stream.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
        for name in ("dfb_destroy", "dfb_sync", "dfb_first_step"):
            getattr(L, name).argtypes = [C.c_void_p]
        L.dfb_dims.argtypes = [C.c_void_p, c_ip, c_ip]
        L.dfb_info.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int64)]
        L.dfb_get_table.argtypes = [C.c_void_p, C.c_int, C.c_int, c_dp, C.c_int]
        L.dfb_get_half_widths.argtypes = [C.c_void_p, C.c_int, C.c_int, c_ip]
        L.dfb_filter.argtypes = [C.c_void_p, C.c_double]
        L.dfb_scatter_to_cells.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p]
        L.dfb_filter_to_host.argtypes = [C.c_void_p, C.c_double] + [C.c_void_p] * 5
        L.dfb_filter_to_host_begin.argtypes = [C.c_void_p, C.c_double] + [C.c_void_p] * 5
        L.dfb_filter_to_host_end.argtypes = [C.c_void_p]
        L.dfb_filter_batch.argtypes = [C.c_void_p, C.c_int, c_dp, C.c_void_p]
        L.dfb_get_field.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        L.dfb_device_ptr.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]
        L.dfb_stream.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
        L.dfb_set_noise.argtypes = [C.c_void_p, C.c_int, c_dp, c_dp]
        L.dfb_set_noise_ref_layout.argtypes = [C.c_void_p, C.c_int, c_dp, c_dp]
        L.dfb_get_noise.argtypes = [C.c_void_p, C.c_int, c_dp, c_dp]
        L.dfb_generate_noise.argtypes = [C.c_void_p, C.c_int64]
        L.dfb_get_state.argtypes = [C.c_void_p, c_dp, C.POINTER(C.c_int64)]
        L.dfb_set_state.argtypes = [C.c_void_p, c_dp, C.c_int64]
        L.dfb_set_timing.argtypes = [C.c_void_p, C.c_int]
        L.dfb_last_ms.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_float)]
        L.dfb_measure_fp64_peak.argtypes = [C.c_int, c_dp, c_dp]
        L.dfb_stats_enable.argtypes = [C.c_void_p, C.c_int]
        L.dfb_stats_get.argtypes = [C.c_void_p, C.c_int, C.c_int, c_dp, C.POINTER(C.c_int64)]
        L.dfb_write_csv.argtypes = [C.c_void_p, C.c_char_p]
        L.dfb_corr_enable.argtypes = [C.c_void_p, C.c_int, c_ip]
        L.dfb_corr_get.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, c_dp, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        L.dfb_corr_get_plane.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, c_dp, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        L.dfb_corr_integral_scales.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, c_dp]
        L.dfb_save_restart.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
        L.dfb_load_restart.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
        L.dfb_restart_info.argtypes = [C.c_char_p, C.POINTER(C.c_int64), C.c_int]
        L.dfb_facemap_create.argtypes = [C.c_void_p, C.c_int, C.c_int, c_dp, c_dp, c_dp, c_dp, C.c_int, C.c_int, C.c_int, c_ip]
        L.dfb_facemap_served.argtypes = [C.c_void_p, C.c_int, c_ip]
        L.dfb_facemap_destroy.argtypes = [C.c_void_p, C.c_int]
        L.dfb_interp_to_cells.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_void_p), c_dp,
                                          C.POINTER(C.c_void_p), C.c_int]
        L.dfb_interp_to_host.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, c_dp]
        L.dfb_attach_stream.argtypes = [C.c_void_p, C.c_void_p]
        L.dfb_filter_dev.argtypes = [C.c_void_p, C.c_void_p]
        L.dfb_set_time_scales.argtypes = [C.c_void_p, c_dp]
        L.dfb_set_profiles.argtypes = [C.c_void_p, c_dp]
        L.dfb_time_scales_from_lengths.argtypes = [C.c_void_p, c_dp, C.c_double, c_dp]
        L.dfb_set_filter_shape.argtypes = [C.c_void_p, C.c_int]
        L.dfb_set_flux_correction.argtypes = [C.c_void_p, C.c_int]
        L.dfb_flux_info.argtypes = [C.c_void_p, C.c_int, c_dp]
        _lib = L
    return _lib


def _check(rc):
    if rc != OK:
        raise DfbError(rc, lib().dfb_last_error().decode(errors="replace"))


def _dptr(a):
    return a.ctypes.data_as(c_dp) if a is not None else None


def measure_fp64_peak(device=-1):
    """DFMA microbenchmark -> (TFLOP/s, implied SM MHz at 64 DFMA/clk/SM)."""
    t, m = C.c_double(), C.c_double()
    _check(lib().dfb_measure_fp64_peak(device, C.byref(t), C.byref(m)))
    return t.value, m.value


def restart_info(path):
    """Header of a restart file (dfb_restart_info; no handle, no device): a dict keyed by RESTART_INFO.  seed and fingerprint are
    unsigned 64-bit values."""
    out = (C.c_int64 * len(RESTART_INFO))()
    _check(lib().dfb_restart_info(os.fsencode(path), out, len(out)))
    d = dict(zip(RESTART_INFO, out))
    d["seed"] &= (1 << 64) - 1
    d["fingerprint"] &= (1 << 64) - 1
    return d


class DFConfig:
    """The reference's DFConfig (df.hpp:38-49) plus the extension fields of dfb_config.
    `dc_config` (the README's spelling, README.md:21) is an alias."""

    def __init__(self, **kw):
        self.d_i = self.rho_e = self.U_e = self.mu_e = 0.0
        self.vel_file_offset = self.vel_file_N_values = 0
        self.grid_file = ""
        self.vel_fluc_file = ""
        # extensions
        self.honor_flow_config = 0
        self.line_file = ""
        self.Ny = self.Nz = 0
        self.geom_per_row = 1
        self.yc = self.dy = self.dz = self.rows = self.scales = self.N_y = self.N_z = None
        self.seed = 0
        self.noise_mode = NOISE_GENERATE
        self.device = -1
        self.plane_id = 0
        self.k_begin = self.k_end = 0
        self.skip_first_step = 0
        self.kernel_variant = 0
        self.periodic_z = 0              # 1: spanwise-periodic plane (the z filter wraps around it; include/dfb200.h)
        self.filter_shape = FILTER_EXPONENTIAL   # FILTER_GAUSSIAN: Klein et al.'s kernel, which delivers the configured Iz / Iy
        for k, v in kw.items():
            if not hasattr(self, k):
                raise TypeError(f"DFConfig has no field {k!r}")
            setattr(self, k, v)

    @classmethod
    def from_plane(cls, plane, **kw):
        """Explicit-geometry config from a workload dict (workloads.py): Ny, Nz, d_i, yc, dy, dz, rows, scales
        [, N_y, N_z].  The half-widths are computed by the library from the geometry unless given."""
        c = cls(Ny=plane["Ny"], Nz=plane["Nz"], d_i=plane["d_i"], U_e=plane.get("U_e", 869.1), honor_flow_config=1,
                yc=plane["yc"], dy=plane["dy"], dz=plane["dz"], rows=plane["rows"], scales=plane["scales"],
                geom_per_row=1 if np.ndim(plane["yc"]) == 1 else 0)
        if plane.get("explicit_N"):
            c.N_y, c.N_z = plane["N_y"], plane["N_z"]
        for k, v in kw.items():
            setattr(c, k, v)
        return c


dc_config = DFConfig


def fill_config(c, config):
    """Fills the ctypes `dfb_config` c (initialised by dfb_config_init) from a DFConfig.  Returns the arrays c points into: keep
    them alive as long as c is used."""
    keep = []

    def arr(a, dtype):
        if a is None:
            return None
        a = np.ascontiguousarray(a, dtype=dtype)
        keep.append(a)
        return a

    c.d_i, c.rho_e, c.U_e, c.mu_e = config.d_i, config.rho_e, config.U_e, config.mu_e
    c.vel_file_offset, c.vel_file_N_values = config.vel_file_offset, config.vel_file_N_values
    c.grid_file = config.grid_file.encode() if config.grid_file else None
    c.vel_fluc_file = config.vel_fluc_file.encode() if config.vel_fluc_file else None
    c.line_file = config.line_file.encode() if config.line_file else None
    c.honor_flow_config = config.honor_flow_config
    c.Ny, c.Nz, c.geom_per_row = config.Ny, config.Nz, config.geom_per_row
    for name in ("yc", "dy", "dz", "rows", "scales"):
        a = arr(getattr(config, name), np.float64)
        setattr(c, name, _dptr(a))
    for name in ("N_y", "N_z"):
        a = arr(getattr(config, name), np.int32)
        setattr(c, name, a.ctypes.data_as(c_ip) if a is not None else None)
    c.seed, c.noise_mode, c.device, c.plane_id = config.seed, config.noise_mode, config.device, config.plane_id
    c.k_begin, c.k_end = config.k_begin, config.k_end
    c.skip_first_step, c.kernel_variant = config.skip_first_step, config.kernel_variant
    c.periodic_z = config.periodic_z
    return keep


def _mask(fields):
    m = 0
    for f in fields:
        if f not in FLUCS:
            raise ValueError(f"field {f!r} is not one of U_FLUC .. RHO_FLUC")
        m |= 1 << f
    return m


class FaceMap:
    """Interpolation of a handle's outputs onto a CFD code's inflow faces (dfb_facemap_create): made by DIGITAL_FILTER.facemap, alive
    until close() or the handle's close().  .served: 0/1 per face, 1 where this handle serves the face."""

    def __init__(self, owner, map_id, n):
        self._o, self.id, self.n = owner, map_id, n
        self.served = np.zeros(n, dtype=np.int32)
        _check(lib().dfb_facemap_served(owner._h, map_id, self.served.ctypes.data_as(c_ip)))

    def to_cells(self, dst, dst_index=None, mean=None, scale=None, fields=FLUCS, plane=0, stride=1):
        """dst[r][dst_index[i] * stride] = (mean[r][i] | dst's own value) + scale[r] * interpolated field fields[r], for each served
        face i, enqueued on the handle's stream.  dst, mean: sequences aligned with `fields` of CUDA float64 torch tensors on the
        handle's device (a mean entry may be None), dst_index an int32 CUDA tensor (None: face i -> i), scale a sequence of floats.
        The handle's stream (stream()) does not wait for other streams: finish writing the arrays first (torch.cuda.synchronize())."""
        fields = list(fields)
        d5, m5, s5 = (C.c_void_p * 5)(), (C.c_void_p * 5)(), (C.c_double * 5)(1, 1, 1, 1, 1)
        for r, f in enumerate(fields):
            d5[f] = dst[r].data_ptr()
            if mean is not None and mean[r] is not None:
                m5[f] = mean[r].data_ptr()
            if scale is not None:
                s5[f] = float(scale[r])
        _check(lib().dfb_interp_to_cells(self._o._h, self.id, plane, _mask(fields),
                                         C.c_void_p(dst_index.data_ptr()) if dst_index is not None else None, m5, s5, d5, int(stride)))

    def to_host(self, fields=FLUCS, plane=0, out=None):
        """[len(fields)][n] interpolated fluctuations (rows in increasing field order); only the served faces' entries are written"""
        fields = sorted(fields)
        out = np.zeros((len(fields), self.n)) if out is None else out
        assert out.dtype == np.float64 and out.flags.c_contiguous and out.shape == (len(fields), self.n)
        _check(lib().dfb_interp_to_host(self._o._h, self.id, plane, _mask(fields), _dptr(out)))
        return out

    def close(self):
        if self.id is not None and getattr(self._o, "_h", None):
            _check(lib().dfb_facemap_destroy(self._o._h, self.id))
        self.id = None


class FilterField:
    """Host view of one velocity component (df.hpp:24-34): .fluc and .filt, Ny x Nz, row-major j*Nz+k."""

    def __init__(self, owner, idx):
        self._o, self._i = owner, idx
        self.fluc = np.zeros((owner.Ny, owner.Nz))
        self.filt = np.zeros((owner.Ny, owner.Nz))

    @property
    def Ny_max(self):
        return self._o.info(0, self._i)

    @property
    def Nz_max(self):
        return self._o.info(1, self._i)

    @property
    def N_ys(self):
        return self._o.half_widths(self._i, 0)

    @property
    def N_zs(self):
        return self._o.half_widths(self._i, 1)


class DIGITAL_FILTER:
    """DIGITAL_FILTER (df.hpp:52-125) on one B200.  Construction = df.cpp:4-66 (setup + first step);
    filter(dt) = df.cpp:449-468 without the print and the CSV (SURVEY quirk 8)."""

    def __init__(self, config=None, fetch=True, nplanes=1):
        """nplanes > 1: a batch of independent planes of this geometry advanced by one launch set per step (dfb_create_batch,
        BASELINE config 5); plane p draws from stream group config.plane_id + p.  The host members then describe plane 0;
        get(which, plane=p) / device_ptr(which, plane=p) reach the others."""
        config = config or DFConfig()
        L = lib()
        c = dfb_config()
        _check(L.dfb_config_init(C.byref(c)))
        self._keep = fill_config(c, config)
        self._h = C.c_void_p()
        self.nplanes = int(nplanes)
        shaped = config.filter_shape != FILTER_EXPONENTIAL
        if shaped:
            c.skip_first_step = 1        # the shape is set before any step; the constructor's step follows below
        if self.nplanes == 1:
            _check(L.dfb_create(C.byref(c), C.byref(self._h)))
        else:
            _check(L.dfb_create_batch(C.byref(c), self.nplanes, C.byref(self._h)))
            fetch = False
        if shaped:
            try:
                self.set_filter_shape(config.filter_shape)
                if config.noise_mode == NOISE_GENERATE and not config.skip_first_step:
                    self.first_step()
            except Exception:
                self.close()
                raise
        ny, nz = C.c_int(), C.c_int()
        _check(L.dfb_dims(self._h, C.byref(ny), C.byref(nz)))
        self.Ny, self.Nz, self.n_cells = ny.value, nz.value, ny.value * nz.value
        self.noise_mode = config.noise_mode
        self._device = self.info(6)
        self.u, self.v, self.w = (FilterField(self, i) for i in range(3))
        self.T_fluc = np.zeros((self.Ny, self.Nz))
        self.rho_fluc = np.zeros((self.Ny, self.Nz))
        self.dt = 0.0
        self._fetch = fetch
        if fetch and config.noise_mode == NOISE_GENERATE and not config.skip_first_step:
            self.fetch()

    # ---- lifetime ----
    def close(self):
        if getattr(self, "_h", None):
            lib().dfb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- the reference's entry point ----
    def filter(self, dt_input):
        """One timestep.  With fetch=True (default) the five outputs land in .u.fluc, .v.fluc, .w.fluc,
        .T_fluc, .rho_fluc (host), like the reference's vectors; with fetch=False they stay on the device."""
        self.dt = float(dt_input)
        if self._fetch:
            _check(lib().dfb_filter_to_host(self._h, self.dt, self.u.fluc.ctypes.data, self.v.fluc.ctypes.data,
                                            self.w.fluc.ctypes.data, self.T_fluc.ctypes.data, self.rho_fluc.ctypes.data))
        else:
            _check(lib().dfb_filter(self._h, self.dt))

    def first_step(self):
        _check(lib().dfb_first_step(self._h))

    # ---- GPU-resident callers: steps on the caller's stream, dt in device memory, capturable (include/dfb200.h, dfb_attach_stream) ----
    def attach_stream(self, stream):
        """Every later call of this handle that enqueues device work goes on `stream` (a torch.cuda.Stream, or a raw cudaStream_t as an
        int), with the step's state in device memory, so that filter_dev() can be captured by torch.cuda.graph on that stream.  None
        detaches (synchronises, reads the step state back)."""
        if stream is not None and not isinstance(stream, int):
            stream = stream.cuda_stream
        _check(lib().dfb_attach_stream(self._h, C.c_void_p(stream) if stream else None))

    def filter_dev(self, dt):
        """One step with dt read from device memory when the step runs: dt is a 1-element CUDA float64 tensor on this handle's device,
        which must stay alive until the step has run (for a captured graph: as long as the graph is replayed).  The handle must be
        attached (attach_stream).  A dt that is not finite or < 0 voids the step; the next synchronising call raises DfbError(ERR_ARG)."""
        if not dt.is_cuda or dt.dtype.itemsize != 8 or not dt.dtype.is_floating_point or dt.numel() != 1:
            raise ValueError("dt must be a 1-element CUDA float64 tensor")
        _check(lib().dfb_filter_dev(self._h, C.c_void_p(dt.data_ptr())))

    # ---- filter shape (include/dfb200.h, dfb_set_filter_shape) ----
    def set_filter_shape(self, shape):
        """FILTER_EXPONENTIAL or FILTER_GAUSSIAN, on a handle that has not stepped (DFConfig(filter_shape=...) does this for you)"""
        _check(lib().dfb_set_filter_shape(self._h, int(shape)))

    @property
    def filter_shape(self):
        """FILTER_EXPONENTIAL or FILTER_GAUSSIAN (dfb_info 17)"""
        return self.info(17)

    # ---- inflow mass-flux correction (include/dfb200.h, dfb_set_flux_correction) ----
    def set_flux_correction(self, mode):
        """FLUX_OFF, FLUX_MASS or FLUX_VOLUME from the next step on: each step's plane-integrated first-order mass (or volume) flux of
        u' (and T', rho') is held at its mean; filt_old, v' and w' are untouched.  Whole planes and batches only (DfbError otherwise)."""
        _check(lib().dfb_set_flux_correction(self._h, int(mode)))

    @property
    def flux_correction(self):
        """FLUX_OFF, FLUX_MASS or FLUX_VOLUME (dfb_info 18)"""
        return self.info(18)

    def flux_info(self, plane=0):
        """(c, m', mean flux) of the last corrected step of `plane`: the subtracted multiple of sqrt(R11), the plane's first-order flux
        fluctuation before the correction, and sum A rhos Us (mass) or sum A Us (volume)"""
        out = np.zeros(3)
        _check(lib().dfb_flux_info(self._h, int(plane), _dptr(out)))
        return float(out[0]), float(out[1]), float(out[2])

    # ---- per-cell profiles (include/dfb200.h, dfb_set_profiles) ----
    def set_profiles(self, cells):
        """Per-cell R11, R21, R22, R33, Us, Ts, rhos, Ms from the next step on: cells = [8][Ny][Nz_global] for the whole plane, in the
        order of DFConfig rows (a slab uses its own columns, a batch the same table for every plane); None returns to the row tables.
        Refused (DfbError) for a value that is not finite or whose epilogue constant is not, while attached, with a communicator, or
        while a filter_to_host_begin / gather_begin is outstanding."""
        if cells is None:
            _check(lib().dfb_set_profiles(self._h, None))
            return
        a = np.ascontiguousarray(cells, dtype=np.float64)
        nzg = self.info(5)
        if a.shape != (8, self.Ny, nzg):
            raise ValueError("profiles must be [8][Ny][Nz_global] = [8][%d][%d], got %s" % (self.Ny, nzg, a.shape))
        _check(lib().dfb_set_profiles(self._h, _dptr(a)))

    @property
    def profiles(self):
        """the [8][Ny][Nz] profiles in use for this handle's columns (dfb_get_table 16), or None without per-cell profiles (dfb_info 19)"""
        if not self.info(19):
            return None
        return np.stack([self.table(16, q, self.Ny * self.Nz).reshape(self.Ny, self.Nz) for q in range(8)])

    # ---- per-row temporal scales (include/dfb200.h, dfb_set_time_scales) ----
    def set_time_scales(self, rows):
        """Lt per field and row for the temporal blend from the next step on: rows = [3][Ny] (u, v, w), finite and > 0; None returns to
        the config's scalar Lt.  Refused (DfbError) while attached or while a filter_to_host_begin / gather_begin is outstanding."""
        if rows is None:
            _check(lib().dfb_set_time_scales(self._h, None))
            return
        a = np.ascontiguousarray(rows, dtype=np.float64)
        if a.shape != (3, self.Ny):
            raise ValueError("time scales must be [3][Ny] = [3][%d], got %s" % (self.Ny, a.shape))
        _check(lib().dfb_set_time_scales(self._h, _dptr(a)))

    @property
    def time_scales(self):
        """the [3][Ny] time scales in use: the rows of set_time_scales, or the scalar Lt of each field repeated (dfb_get_table 14)"""
        return np.stack([self.table(14, f) for f in range(3)])

    def time_scales_from_lengths(self, Ix, u_min):
        """[3][Ny] time scales Ix_f(y_j) / max(Us_j, u_min) from streamwise lengths Ix = (inn_u, out_u, inn_v, out_v, inn_w, out_w),
        blended across the boundary layer like Iz (dfb_time_scales_from_lengths); host only, sets nothing"""
        ix = np.ascontiguousarray(Ix, dtype=np.float64)
        if ix.shape != (6,):
            raise ValueError("Ix must hold 6 lengths")
        out = np.zeros((3, self.Ny))
        _check(lib().dfb_time_scales_from_lengths(self._h, _dptr(ix), float(u_min), _dptr(out)))
        return out

    def filter_batch(self, dts, out=None):
        dts = np.ascontiguousarray(dts, dtype=np.float64)
        _check(lib().dfb_filter_batch(self._h, len(dts), _dptr(dts), out.ctypes.data if out is not None else None))

    # ---- data access ----
    def get(self, which, out=None, plane=0):
        out = np.zeros((self.Ny, self.Nz)) if out is None else out
        _check(lib().dfb_get_field_plane(self._h, plane, which, out.ctypes.data, 0))
        return out

    def get_to_device(self, which, device_ptr):
        _check(lib().dfb_get_field(self._h, which, C.c_void_p(device_ptr), 1))

    def device_ptr(self, which, plane=0):
        p = C.c_void_p()
        _check(lib().dfb_device_ptr_plane(self._h, plane, which, C.byref(p)))
        return p.value

    def device_tensor(self, which):
        """zero-copy torch view (Ny, Nz) of a device-resident field (for NCCL hand-offs)"""
        import torch

        class _View:
            pass

        v = _View()
        v.__cuda_array_interface__ = dict(shape=(self.Ny, self.Nz), typestr="<f8", data=(self.device_ptr(which), False),
                                          version=3, strides=None)
        return torch.as_tensor(v, device=torch.device("cuda", self._device))

    def scatter_to_cells(self, which, plane_index, dst_index, dst, mean=None, scale=1.0):
        """CFD hand-off on the device (dfb_scatter_to_cells): dst[dst_index[i]] = (mean[i] | dst[dst_index[i]]) + scale * field[plane_index[i]].
        Arguments are CUDA torch tensors (int32 indices, float64 values) on this handle's device."""
        n = int(plane_index.numel())
        _check(lib().dfb_scatter_to_cells(self._h, which, n, C.c_void_p(plane_index.data_ptr()), C.c_void_p(dst_index.data_ptr()),
                                          C.c_void_p(mean.data_ptr()) if mean is not None else None, C.c_double(scale), C.c_void_p(dst.data_ptr())))

    def stream(self):
        p = C.c_void_p()
        _check(lib().dfb_stream(self._h, C.byref(p)))
        return p.value

    def fetch(self):
        """Copy all outputs (and filt) to the host members."""
        for f, F in enumerate((self.u, self.v, self.w)):
            self.get(U_FLUC + f, F.fluc)
            self.get(U_FILT + f, F.filt)
        self.get(T_FLUC, self.T_fluc)
        self.get(RHO_FLUC, self.rho_fluc)
        return self

    def sync(self):
        _check(lib().dfb_sync(self._h))

    def info(self, what, field=0):
        v = C.c_int64()
        _check(lib().dfb_info(self._h, what, field, C.byref(v)))
        return v.value

    @property
    def step(self):
        return self.info(2)

    @property
    def tuned(self):
        return bool(self.info(3))

    @property
    def periodic_z(self):
        """True when the plane is spanwise-periodic (dfb_config.periodic_z; dfb_info 13)"""
        return bool(self.info(13))

    @property
    def taps_per_step(self):
        return self.info(4)

    def table(self, which, arg=0, n=None):
        n = n if n is not None else (3 if which == 10 else (2 * arg + 1 if which == 11 else self.Ny))   # 14: [Ny]
        out = np.zeros(n)
        _check(lib().dfb_get_table(self._h, which, arg, _dptr(out), n))
        return out

    def rows(self):
        return np.stack([self.table(i) for i in range(8)])

    def half_widths(self, field, direction):
        out = np.zeros((self.Ny, self.Nz), dtype=np.int32)
        _check(lib().dfb_get_half_widths(self._h, field, direction, out.ctypes.data_as(c_ip)))
        return out

    # ---- noise ----
    def set_noise(self, field, r_ys, halo=None):
        """r_ys (Ny + 2 Ny_max, Nz) and the r_zs halo (Ny, 2 Nz_max); a periodic plane takes r_ys alone (halo=None)."""
        r_ys = np.ascontiguousarray(r_ys, dtype=np.float64)
        halo = np.ascontiguousarray(halo, dtype=np.float64) if halo is not None else None
        _check(lib().dfb_set_noise(self._h, field, _dptr(r_ys), _dptr(halo)))

    def set_noise_ref_layout(self, field, r_ys, r_zs):
        r_ys = np.ascontiguousarray(r_ys, dtype=np.float64)
        r_zs = np.ascontiguousarray(r_zs, dtype=np.float64) if r_zs is not None else None
        _check(lib().dfb_set_noise_ref_layout(self._h, field, _dptr(r_ys), _dptr(r_zs)))

    def get_noise(self, field):
        """(r_ys, halo) of the last step's noise; (r_ys, None) on a periodic plane, which draws no halo."""
        F = (self.u, self.v, self.w)[field]
        r_ys = np.zeros((self.Ny + 2 * F.Ny_max, self.Nz))
        halo = None if self.periodic_z else np.zeros((self.Ny, 2 * F.Nz_max))
        _check(lib().dfb_get_noise(self._h, field, _dptr(r_ys), _dptr(halo)))
        return r_ys, halo

    def generate_noise(self, step):
        _check(lib().dfb_generate_noise(self._h, int(step)))

    # ---- checkpoint ----
    def get_state(self):
        fo = np.zeros((3, self.Ny, self.Nz)) if self.nplanes == 1 else np.zeros((3, self.nplanes, self.Ny, self.Nz))
        s = C.c_int64()
        _check(lib().dfb_get_state(self._h, _dptr(fo), C.byref(s)))
        return fo, s.value

    def set_state(self, filt_old, step):
        fo = np.ascontiguousarray(filt_old, dtype=np.float64) if filt_old is not None else None
        _check(lib().dfb_set_state(self._h, _dptr(fo), int(step)))

    # ---- restart files (include/dfb200.h, dfb_save_restart) ----
    @staticmethod
    def _restart_what(stats, corr):
        return RESTART_STATE | (RESTART_STATS if stats else 0) | (RESTART_CORR if corr else 0)

    def save_restart(self, path, stats=False, corr=False):
        """Write this handle's filter state and step counter (and the N2 sums with stats=True, the correlation statistics with
        corr=True) into the restart file `path`, in the plane's global layout.  Slabs of one plane (or of one batch) may save into one
        file; it is complete when every writer has returned."""
        _check(lib().dfb_save_restart(self._h, os.fsencode(path), self._restart_what(stats, corr)))

    def load_restart(self, path, stats=False, corr=False):
        """Resume from a restart file written by any decomposition of these planes: the next filter() produces the step the saved run
        would have produced next, bit for bit with the same kernel forms.  A refused load changes nothing."""
        _check(lib().dfb_load_restart(self._h, os.fsencode(path), self._restart_what(stats, corr)))

    # ---- N2 running statistics / N4 CSV (both opt-in; filter() itself never writes or accumulates) ----
    def stats_enable(self, on=True):
        _check(lib().dfb_stats_enable(self._h, int(on)))

    def stats(self, which, rms=False, plane=0):
        """which: 0 u'^2, 1 v'^2, 2 w'^2, 3 T'^2, 4 rho'^2, 5 u'v' (per-cell sums, or sqrt(sum/count) with rms=True).
        Returns (array, accumulated steps)."""
        out = np.zeros((self.Ny, self.Nz))
        cnt = C.c_int64()
        _check(lib().dfb_stats_get_plane(self._h, plane, which, int(rms), _dptr(out), C.byref(cnt)))
        return out, cnt.value

    def get_rms(self, nsteps=500, dt=1e-5, path=None):
        """get_rms (df.cpp:584-611): 500 steps of dt = 1e-5 with on-device accumulation; plot_rms's file when `path` is given."""
        _check(lib().dfb_get_rms(self._h, int(nsteps), float(dt)))
        if path is not None:
            _check(lib().dfb_write_rms_csv(self._h, str(path).encode()))

    # ---- correlation statistics (opt-in; include/dfb200.h, dfb_corr_enable) ----
    def corr_enable(self, z=DFB_CORR_SUPPORT, y=DFB_CORR_SUPPORT, t=0, on=True):
        """Accumulate per-row lagged products of u', v', w' after every step: lags z, y (0 = off, DFB_CORR_SUPPORT = the filter's
        whole support) and t (0..64 steps).  Zeroes the sums; on=False stops accumulating and keeps them readable."""
        lags = (C.c_int * 3)(int(z), int(y), int(t))
        _check(lib().dfb_corr_enable(self._h, int(on), lags))

    @property
    def corr_lags(self):
        """(L_z, L_y, L_t) of the correlation sums (dfb_info 14); 0 for a direction that is off"""
        return tuple(self.info(14, d) for d in range(3))

    def corr(self, field, dir, normalized=True, plane=0):
        """(array [Ny, L+1], pairs [L+1], accumulated steps) of field 0..2 (u', v', w') in direction CORR_Z / CORR_Y / CORR_T:
        correlation coefficients (normalized=True) or the raw sums"""
        n = self.corr_lags[dir] + 1
        out = np.zeros((self.Ny, n))
        pairs = np.zeros(n, dtype=np.int64)
        cnt = C.c_int64()
        _check(lib().dfb_corr_get_plane(self._h, plane, field, dir, int(normalized), _dptr(out),
                                        pairs.ctypes.data_as(C.POINTER(C.c_int64)), C.byref(cnt)))
        return out, pairs, cnt.value

    def integral_scales(self, field, dir, plane=0):
        """per-row integral scale of the normalised correlation up to its first non-positive lag: metres for z and y, steps for t"""
        out = np.zeros(self.Ny)
        _check(lib().dfb_corr_integral_scales(self._h, plane, field, dir, _dptr(out)))
        return out

    def write_csv(self, path):
        _check(lib().dfb_write_csv(self._h, str(path).encode()))

    def write_tecplot(self, path):
        _check(lib().dfb_write_tecplot(self._h, str(path).encode()))

    def face_map(self, yf, zf):
        """plane_index (j*Nz + k within this handle's slab, -1 outside it) of the cells containing the face centres (yf, zf)"""
        yf = np.ascontiguousarray(yf, dtype=np.float64)
        zf = np.ascontiguousarray(zf, dtype=np.float64)
        out = np.zeros(len(yf), dtype=np.int32)
        _check(lib().dfb_face_map(self._h, len(yf), _dptr(yf), _dptr(zf), out.ctypes.data_as(c_ip)))
        return out

    def facemap(self, yf, zf, hy=None, hz=None, own=None, wall_zero=False):
        """A face map for the faces centred at (yf, zf): bilinear at the centres, or with the extents hy, hz the average over each face
        rectangle.  own = (k_begin, k_end): the columns whose faces this handle serves (default its slab); wall_zero: a point map goes
        linearly to 0 at the wall below the first cell centre."""
        yf = np.ascontiguousarray(yf, dtype=np.float64)
        zf = np.ascontiguousarray(zf, dtype=np.float64)
        if (hy is None) != (hz is None):
            raise ValueError("give both hy and hz, or neither")
        kind = MAP_POINT if hy is None else MAP_AREA
        hy = None if hy is None else np.ascontiguousarray(hy, dtype=np.float64)
        hz = None if hz is None else np.ascontiguousarray(hz, dtype=np.float64)
        if any(a is not None and a.shape != yf.shape for a in (zf, hy, hz)) or yf.ndim != 1:
            raise ValueError("yf, zf (and hy, hz) must be 1-D arrays of one length")
        own = (0, 0) if own is None else own
        mid = C.c_int()
        _check(lib().dfb_facemap_create(self._h, kind, len(yf), _dptr(yf), _dptr(zf), _dptr(hy), _dptr(hz), int(own[0]), int(own[1]),
                                        MAP_WALL_ZERO if wall_zero else 0, C.byref(mid)))
        return FaceMap(self, mid.value, len(yf))

    # ---- config 4: this handle as one spanwise slab of a plane shared with the other ranks (NCCL inside the library) ----
    @staticmethod
    def comm_unique_id():
        """rank 0: the 128-byte NCCL id every rank passes to comm_init (ship it with the job's own means)"""
        buf = C.create_string_buffer(128)
        _check(lib().dfb_comm_unique_id(buf))
        return buf.raw

    def comm_init(self, ident, rank, world):
        _check(lib().dfb_comm_init(self._h, C.c_char_p(ident), int(rank), int(world)))
        self._NzG = self.info(5)

    def comm_bounds(self):
        r, w = C.c_int(), C.c_int()
        _check(lib().dfb_comm_info(self._h, C.byref(r), C.byref(w), None))
        b = np.zeros(2 * w.value, dtype=np.int32)
        _check(lib().dfb_comm_info(self._h, None, None, b.ctypes.data_as(c_ip)))
        return [(int(b[2 * i]), int(b[2 * i + 1])) for i in range(w.value)]

    def gather_begin(self, dst=0):
        _check(lib().dfb_gather_begin(self._h, int(dst)))

    def gather_end(self):
        _check(lib().dfb_gather_end(self._h))

    def gathered(self, which, out=None):
        """destination rank: host copy (Ny, Nz_global) of a gathered field"""
        out = np.zeros((self.Ny, self._NzG)) if out is None else out
        _check(lib().dfb_gathered_to_host(self._h, which, out.ctypes.data))
        return out

    def gathered_ptr(self, which):
        p = C.c_void_p()
        _check(lib().dfb_gathered_ptr(self._h, which, C.byref(p)))
        return p.value

    def comm_stream(self):
        p = C.c_void_p()
        _check(lib().dfb_comm_stream(self._h, C.byref(p)))
        return p.value

    def gather_wire_bytes(self):
        v = C.c_int64()
        _check(lib().dfb_gather_wire_bytes(self._h, C.byref(v)))
        return v.value

    # ---- timing ----
    def set_timing(self, on=True):
        _check(lib().dfb_set_timing(self._h, int(on)))

    def last_ms(self):
        out = []
        for s in range(4):
            v = C.c_float()
            _check(lib().dfb_last_ms(self._h, s, C.byref(v)))
            out.append(v.value)
        return dict(noise=out[0], ysweep=out[1], zsweep_epilogue=out[2], step=out[3])
