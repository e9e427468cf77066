// include/digital_filter.hpp -- the reference's C++ surface over the B200 library.
//
// Drop-in for digital-filtering-c++/df/df.hpp: the same names a caller uses
//     DFConfig config; DIGITAL_FILTER df(config); df.filter(dt);  df.u.fluc[j*Nz + k] ...
// (test/cpp-main.cpp:6-17), bound to the C ABI in dfb200.h.  Header-only; link with -ldfb200.
//
//   struct DFConfig          df.hpp:38-49   (field for field; `dc_config` = README.md:21's spelling)
//   struct FilterField       df.hpp:24-34   (the members a caller reads: fluc, filt, N_ys, N_zs, Ny_max, Nz_max, Lt)
//   class  DIGITAL_FILTER    df.hpp:52-125  (public u, v, w; DIGITAL_FILTER(DFConfig); filter(double))
//
// Differences a caller can observe, all deliberate:
//   * filter() neither prints "Filtering took ..." nor rewrites ../files/cpp_vel_fluc.csv every call
//     (df.cpp:462-467; SURVEY quirk 8);
//   * T_fluc / rho_fluc are private in the reference (df.hpp:59): read them through T_fluc() / rho_fluc();
//   * errors throw std::runtime_error with the library's message instead of printing to cerr and
//     carrying on half-initialised (df.cpp:225-228, 492-495);
//   * the per-stage public methods (generate_white_noise, filtering_sweeps, correlate_fields,
//     apply_RST_scaling, get_rho_T_fluc; df.hpp:96-101) do not exist: the stages are fused on the GPU.
//     get_rms() / plot_rms() / write_csv() / write_tecplot() (df.hpp:108-118) do: the reference's own driver calls get_rms()
//     (test/cpp-main.cpp:17), and that file compiles unchanged against include/df/df.hpp.
//   * the host vectors are page-locked (dfb_host_register) so that the five copies per filter() run at the PCIe rate;
//   * the noise is the counter-based pcg32 stream of include/dfb_rng_spec.h (seedable, reproducible)
//     instead of a random_device-seeded process-wide static (df.cpp:334).
#pragma once
#include <array>
#include <cstdint>
#include <cstdio>
#include <stdexcept>
#include <string>
#include <vector>
#include "dfb200.h"

typedef std::vector<double> Vector;

struct FilterField {
    Vector filt, fluc;                 // Ny*Nz, row-major j*Nz + k  (df.hpp:28)
    Vector rms_added, rms;             // df.hpp:27: filled by get_rms() (sums of squares on the device, df.cpp:571-582)
    std::vector<int> N_ys, N_zs;       // df.hpp:30
    double Lt = 0;                     // df.hpp:32
    int Nz_max = 0, Ny_max = 0;        // df.hpp:33
};

struct DFConfig {                      // df.hpp:38-49
    double d_i, rho_e, U_e, mu_e;
    int vel_file_offset, vel_file_N_values;
    std::string grid_file, vel_fluc_file;
};
typedef DFConfig dc_config;

// Everything the reference hard-codes (df.cpp:7-16, 73-74, 224) made configurable; defaults = the reference.
struct DFConfigEx {
    DFConfig base{0, 0, 0, 0, 0, 0, "", ""};
    bool honor_flow_config = false;    // take d_i, rho_e, U_e, mu_e from `base` (the Fortran behaviour, df.f90:80-87)
    std::string line_file;             // "" -> "../line.dat" (df.cpp:16)
    int Ny = 0, Nz = 0;                // 0,0 -> the reference's made-up grid (df.cpp:73-74)
    bool geom_per_row = true;
    const double *yc = nullptr, *dy = nullptr, *dz = nullptr, *rows = nullptr, *scales = nullptr;
    const int *N_y = nullptr, *N_z = nullptr;
    std::uint64_t seed = 0;
    int noise_mode = DFB_NOISE_GENERATE;
    int device = -1, plane_id = 0, k_begin = 0, k_end = 0;
    bool periodic_z = false;           // spanwise-periodic plane: the z filter wraps around it (LES/DNS inflow with periodic span)
    int filter_shape = DFB_FILTER_EXPONENTIAL;   // DFB_FILTER_GAUSSIAN: Klein et al.'s kernel, which delivers the configured Iz / Iy
    bool fetch_every_step = true;      // copy u', v', w', T', rho' into the host vectors after each filter()
};

// A face map of the CFD hand-off (dfb_facemap_create), from DIGITAL_FILTER::face_map_interp; destroyed with this object, which must
// not outlive its DIGITAL_FILTER.  fields: mask of 1 << DFB_U_FLUC .. 1 << DFB_RHO_FLUC.
class FaceMap {
  public:
    FaceMap(dfb_handle h, int id, int n) : h_(h), id_(id), n_(n), served_(n) {
        if (n > 0 && dfb_facemap_served(h_, id_, served_.data()) != DFB_OK) throw std::runtime_error(std::string("FaceMap: ") + dfb_last_error());
    }
    FaceMap(FaceMap&& o) noexcept : h_(o.h_), id_(o.id_), n_(o.n_), served_(std::move(o.served_)) { o.h_ = nullptr; }
    FaceMap(const FaceMap&) = delete;
    FaceMap& operator=(const FaceMap&) = delete;
    ~FaceMap() { if (h_) dfb_facemap_destroy(h_, id_); }
    const std::vector<int>& served() const { return served_; }   // 1 where this handle serves the face
    // device arrays: dst[f][dst_index[i] * stride] = (mean[f][i] | dst's own value) + scale[f] * interpolated field f
    void to_cells(int fields, const int* dst_index, const double* const mean[5], const double scale[5], double* const dst[5], int stride = 1,
                  int plane = 0) {
        check(dfb_interp_to_cells(h_, id_, plane, fields, dst_index, mean, scale, dst, stride));
    }
    // [nfields][n] interpolated fluctuations on the host (rows in increasing field order; unserved faces 0)
    std::vector<double> to_host(int fields = 31, int plane = 0) {
        int nf = 0;
        for (int f = 0; f < 5; ++f) nf += (fields >> f) & 1;
        std::vector<double> out((size_t)nf * n_, 0.0);
        check(dfb_interp_to_host(h_, id_, plane, fields, out.data()));
        return out;
    }

  private:
    dfb_handle h_;
    int id_, n_;
    std::vector<int> served_;
    static void check(int rc) {
        if (rc != DFB_OK) throw std::runtime_error(std::string("FaceMap: ") + dfb_last_error());
    }
};

class DIGITAL_FILTER {
  public:
    FilterField u, v, w;               // df.hpp:87

    // df.hpp:89 -- like the reference (df.cpp:7-16) this constructor IGNORES `config` and builds the
    // hard-coded default plane from ../files/RST.dat and ../line.dat.
    explicit DIGITAL_FILTER(DFConfig) { init(DFConfigEx()); }
    explicit DIGITAL_FILTER(const DFConfigEx& cfg) { init(cfg); }
    DIGITAL_FILTER(const DIGITAL_FILTER&) = delete;
    DIGITAL_FILTER& operator=(const DIGITAL_FILTER&) = delete;
    ~DIGITAL_FILTER() {
        for (void* p : pinned_) dfb_host_unregister(p);
        if (h_) dfb_destroy(h_);
    }

    // df.hpp:100, df.cpp:449-468.  dt_input must be finite and >= 0: otherwise check() throws (DFB_ERR_ARG) and nothing changes.
    void filter(double dt_input) {
        dt = dt_input;
        if (fetch_)
            check(dfb_filter_to_host(h_, dt, u.fluc.data(), v.fluc.data(), w.fluc.data(), T_fluc_.data(), rho_fluc_.data()));
        else
            check(dfb_filter(h_, dt));
    }
    // GPU-resident callers (dfb_attach_stream): every later step, dfb_interp_to_cells and copy goes on `stream` (a cudaStream_t;
    // nullptr detaches), with the step's state in device memory, so that filter_dev can be captured into the caller's CUDA graph
    void attach_stream(struct CUstream_st* stream) { check(dfb_attach_stream(h_, stream)); }
    // one step with dt read from device memory when it runs (the handle must be attached); the host vectors are not refreshed
    void filter_dev(const double* dt_dev) { check(dfb_filter_dev(h_, dt_dev)); }
    // per-row temporal scales (dfb_set_time_scales): Lt_rows = [3][Ny] (u, v, w rows), from the next step on; clear_time_scales
    // returns to the config's scalar Lt.  time_scales_from_lengths converts streamwise lengths Ix = {inn_u, out_u, inn_v, out_v,
    // inn_w, out_w}, blended across the boundary layer like Iz, with the plane's mean velocity: Lt = Ix(y) / max(U(y), u_min)
    void set_time_scales(const std::vector<double>& Lt_rows) {
        if (Lt_rows.size() != (size_t)3 * Ny) throw std::invalid_argument("set_time_scales: Lt_rows must hold 3 * Ny values");
        check(dfb_set_time_scales(h_, Lt_rows.data()));
    }
    void clear_time_scales() { check(dfb_set_time_scales(h_, nullptr)); }
    std::vector<double> time_scales_from_lengths(const double Ix[6], double u_min) const {
        std::vector<double> Lt_rows((size_t)3 * Ny);
        check(dfb_time_scales_from_lengths(h_, Ix, u_min, Lt_rows.data()));
        return Lt_rows;
    }
    // DFB_FILTER_EXPONENTIAL or DFB_FILTER_GAUSSIAN (DFConfigEx::filter_shape; dfb_info 17)
    int filter_shape() const {
        std::int64_t v = 0;
        check(dfb_info(h_, 17, 0, &v));
        return (int)v;
    }
    // inflow mass-flux correction (dfb_set_flux_correction): DFB_FLUX_OFF, DFB_FLUX_MASS or DFB_FLUX_VOLUME from the next step on;
    // flux_info(plane) = {c, m', mean flux} of the last corrected step of that plane
    void set_flux_correction(int mode) { check(dfb_set_flux_correction(h_, mode)); }
    int flux_correction() const {
        std::int64_t v = 0;
        check(dfb_info(h_, 18, 0, &v));
        return (int)v;
    }
    std::array<double, 3> flux_info(int plane = 0) const {
        std::array<double, 3> out{};
        check(dfb_flux_info(h_, plane, out.data()));
        return out;
    }
    // per-cell profiles (dfb_set_profiles): cells = [8][Ny][Nz of the whole plane], the quantities of DFConfig rows in their order, from
    // the next step on; clear_profiles returns to the row tables; profiles() tells whether they are in use (dfb_info 19)
    void set_profiles(const std::vector<double>& cells) {
        std::int64_t nzg = 0;
        check(dfb_info(h_, 5, 0, &nzg));
        if (cells.size() != (size_t)8 * Ny * (size_t)nzg) throw std::invalid_argument("set_profiles: cells must hold 8 * Ny * Nz values (the whole plane)");
        check(dfb_set_profiles(h_, cells.data()));
    }
    void clear_profiles() { check(dfb_set_profiles(h_, nullptr)); }
    bool profiles() const {
        std::int64_t v = 0;
        check(dfb_info(h_, 19, 0, &v));
        return v != 0;
    }
    // explicit fetch for fetch_every_step = false (also refreshes .filt)
    void fetch() {
        FilterField* F[3] = {&u, &v, &w};
        for (int f = 0; f < 3; ++f) {
            check(dfb_get_field(h_, DFB_U_FLUC + f, F[f]->fluc.data(), 0));
            check(dfb_get_field(h_, DFB_U_FILT + f, F[f]->filt.data(), 0));
        }
        check(dfb_get_field(h_, DFB_T_FLUC, T_fluc_.data(), 0));
        check(dfb_get_field(h_, DFB_RHO_FLUC, rho_fluc_.data(), 0));
    }
    // df.hpp:112, df.cpp:584-611 -- the reference's validation driver: 500 steps of dt = 1e-5 accumulating the squares of the five
    // fields (here: on the device, in the z-sweep's epilogue), then plot_rms().  This is the call test/cpp-main.cpp:17 makes.
    void get_rms() {
        dt = 1e-5;
        check(dfb_get_rms(h_, 500, dt));
        FilterField* F[3] = {&u, &v, &w};
        std::int64_t cnt = 0;
        for (int f = 0; f < 3; ++f) {
            F[f]->rms_added.assign(n_cells, 0.0); F[f]->rms.assign(n_cells, 0.0);
            check(dfb_stats_get(h_, f, 0, F[f]->rms_added.data(), &cnt));
            check(dfb_stats_get(h_, f, 1, F[f]->rms.data(), &cnt));
        }
        T_rms_.assign(n_cells, 0.0); rho_rms_.assign(n_cells, 0.0);
        check(dfb_stats_get(h_, 3, 1, T_rms_.data(), &cnt));
        check(dfb_stats_get(h_, 4, 1, rho_rms_.data(), &cnt));
        rms_counter = (int)cnt;
        fetch();                       // the fields of the last step, as the reference leaves them
        plot_rms();
    }
    // df.hpp:113, df.cpp:613-675: writes ../files/cpp_vel_fluc_rms.csv and says so
    void plot_rms() {
        const std::string filename = "../files/cpp_vel_fluc_rms.csv";
        check(dfb_write_rms_csv(h_, filename.c_str()));
        std::printf("Finished plotting to file: %s\n", filename.c_str());
    }
    void write_csv(const std::string& filename) { check(dfb_write_csv(h_, filename.c_str())); std::printf("CSV written to %s\n", filename.c_str()); }   // df.cpp:764-803
    void write_tecplot(const std::string& filename) { check(dfb_write_tecplot(h_, filename.c_str())); std::printf("Finished plotting.\n"); }           // df.cpp:712-762
    // correlation statistics (dfb_corr_enable): lags along z, y (0 = off, DFB_CORR_SUPPORT = the filter's support) and t (0..64 steps)
    void corr_enable(int lz, int ly, int lt) {
        const int lags[3] = {lz, ly, lt};
        check(dfb_corr_enable(h_, 1, lags));
    }
    // [Ny][L+1] of field 0..2 (u', v', w') in direction DFB_CORR_Z / _Y / _T: correlation coefficients, or the raw sums
    std::vector<double> corr(int field, int dir, bool normalized = true, int plane = 0) {
        std::int64_t L = 0;
        check(dfb_info(h_, 14, dir, &L));
        std::vector<double> R((size_t)Ny * (size_t)(L + 1));
        check(dfb_corr_get_plane(h_, plane, field, dir, normalized ? 1 : 0, R.data(), nullptr, nullptr));
        return R;
    }
    // per-row integral scale: metres for z and y, steps for t
    std::vector<double> integral_scales(int field, int dir, int plane = 0) {
        std::vector<double> L(Ny);
        check(dfb_corr_integral_scales(h_, plane, field, dir, L.data()));
        return L;
    }
    // restart files (dfb_save_restart / dfb_load_restart): what = DFB_RESTART_STATE [| DFB_RESTART_STATS | DFB_RESTART_CORR].  A load
    // resumes the saved run: the next filter() produces the step it would have produced next (the host vectors keep the last step's
    // outputs until then).  Slabs of one plane may save into one file; it is complete when every writer has returned.
    void save_restart(const std::string& path, int what = DFB_RESTART_STATE) { check(dfb_save_restart(h_, path.c_str(), what)); }
    void load_restart(const std::string& path, int what = DFB_RESTART_STATE) { check(dfb_load_restart(h_, path.c_str(), what)); }
    // face map at the face centres (yf, zf): bilinear (hy, hz empty) or the average over each face (extents hy, hz); own_begin,
    // own_end: the columns whose faces this handle serves (0, 0: its slab); flags: DFB_MAP_WALL_ZERO
    FaceMap face_map_interp(const std::vector<double>& yf, const std::vector<double>& zf, const std::vector<double>& hy = {},
                            const std::vector<double>& hz = {}, int own_begin = 0, int own_end = 0, int flags = 0) {
        const bool area = !hy.empty() || !hz.empty();
        if (zf.size() != yf.size() || (area && (hy.size() != yf.size() || hz.size() != yf.size())))
            throw std::runtime_error("DIGITAL_FILTER: yf, zf (and hy, hz) must have one length");
        int id = -1;
        check(dfb_facemap_create(h_, area ? DFB_MAP_AREA : DFB_MAP_POINT, (int)yf.size(), yf.data(), zf.data(), area ? hy.data() : nullptr,
                                 area ? hz.data() : nullptr, own_begin, own_end, flags, &id));
        return FaceMap(h_, id, (int)yf.size());
    }
    const Vector& T_rms() const { return T_rms_; }
    const Vector& rho_rms() const { return rho_rms_; }
    int rms_counter = 0;               // df.hpp:63

    const Vector& T_fluc() const { return T_fluc_; }
    const Vector& rho_fluc() const { return rho_fluc_; }
    int get_Ny() const { return Ny; }
    int get_Nz() const { return Nz; }
    dfb_handle handle() const { return h_; }
    double dt = 0;                     // df.hpp:64

  private:
    int Ny = 0, Nz = 0, n_cells = 0;   // df.hpp:56
    Vector rho_fluc_, T_fluc_;         // df.hpp:59
    Vector T_rms_, rho_rms_;           // df.hpp:84
    std::vector<void*> pinned_;
    dfb_handle h_ = nullptr;
    bool fetch_ = true;

    static void check(int rc) {
        if (rc != DFB_OK) throw std::runtime_error(std::string("DIGITAL_FILTER: ") + dfb_last_error());
    }
    void init(const DFConfigEx& c) {
        dfb_config k;
        dfb_config_init(&k);
        k.d_i = c.base.d_i; k.rho_e = c.base.rho_e; k.U_e = c.base.U_e; k.mu_e = c.base.mu_e;
        k.vel_file_offset = c.base.vel_file_offset; k.vel_file_N_values = c.base.vel_file_N_values;
        k.grid_file = c.base.grid_file.empty() ? nullptr : c.base.grid_file.c_str();
        k.vel_fluc_file = c.base.vel_fluc_file.empty() ? nullptr : c.base.vel_fluc_file.c_str();
        k.line_file = c.line_file.empty() ? nullptr : c.line_file.c_str();
        k.honor_flow_config = c.honor_flow_config;
        k.Ny = c.Ny; k.Nz = c.Nz; k.geom_per_row = c.geom_per_row;
        k.yc = c.yc; k.dy = c.dy; k.dz = c.dz; k.rows = c.rows; k.scales = c.scales; k.N_y = c.N_y; k.N_z = c.N_z;
        k.seed = c.seed; k.noise_mode = c.noise_mode; k.device = c.device; k.plane_id = c.plane_id;
        k.k_begin = c.k_begin; k.k_end = c.k_end; k.periodic_z = c.periodic_z ? 1 : 0;
        fetch_ = c.fetch_every_step;
        const bool shaped = c.filter_shape != DFB_FILTER_EXPONENTIAL;
        if (shaped) k.skip_first_step = 1;   // the shape is set before any step; the constructor's step follows
        check(dfb_create(&k, &h_));
        if (shaped) {
            if (dfb_set_filter_shape(h_, c.filter_shape) != DFB_OK ||
                (c.noise_mode == DFB_NOISE_GENERATE && dfb_first_step(h_) != DFB_OK)) {
                const std::string msg = std::string("DIGITAL_FILTER: ") + dfb_last_error();
                dfb_destroy(h_);
                h_ = nullptr;
                throw std::runtime_error(msg);
            }
        }
        check(dfb_dims(h_, &Ny, &Nz));
        n_cells = Ny * Nz;
        rho_fluc_.assign(n_cells, 0.0); T_fluc_.assign(n_cells, 0.0);
        FilterField* F[3] = {&u, &v, &w};
        double Lt[3];
        check(dfb_get_table(h_, 10, 0, Lt, 3));
        for (int f = 0; f < 3; ++f) {
            F[f]->filt.assign(n_cells, 0.0); F[f]->fluc.assign(n_cells, 0.0);
            F[f]->N_ys.assign(n_cells, 0); F[f]->N_zs.assign(n_cells, 0);
            check(dfb_get_half_widths(h_, f, 0, F[f]->N_ys.data()));
            check(dfb_get_half_widths(h_, f, 1, F[f]->N_zs.data()));
            std::int64_t v64 = 0;
            check(dfb_info(h_, 0, f, &v64)); F[f]->Ny_max = (int)v64;
            check(dfb_info(h_, 1, f, &v64)); F[f]->Nz_max = (int)v64;
            F[f]->Lt = Lt[f];
        }
        // page-lock what filter() copies into every step (a failure only costs speed: pageable copies still work)
        Vector* out[5] = {&u.fluc, &v.fluc, &w.fluc, &T_fluc_, &rho_fluc_};
        for (Vector* a : out)
            if (!a->empty() && dfb_host_register(a->data(), a->size() * sizeof(double)) == DFB_OK) pinned_.push_back(a->data());
        if (c.noise_mode == DFB_NOISE_GENERATE) fetch();   // the constructor's first step (df.cpp:57-62)
    }
};
