// csrc/capi.cu -- the C ABI declared in include/dfb200.h: handle lifetime, device layout, the step.
// Mirrors DIGITAL_FILTER's constructor (df.cpp:4-66) and filter(dt) (df.cpp:449-468).
// There is no CPU fallback: without an sm_100 device dfb_create fails with DFB_ERR_CUDA.
#include <algorithm>
#include <array>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <memory>
#include <string>
#include <vector>
#include <chrono>
#include <thread>
#include <nccl.h>
#include "dfb200.h"
#include "plan.hpp"
#include "noise.cuh"
#include "device.cuh"
#include "kernels.hpp"
#include "restart.hpp"
#include "facemap.hpp"

using namespace dfb;

namespace {

thread_local std::string g_last_error;

int fail(int code, const std::string& msg) {
    g_last_error = msg;
    return code;
}

#define CUDA_TRY(expr)                                                                              \
    do {                                                                                            \
        cudaError_t e__ = (expr);                                                                   \
        if (e__ != cudaSuccess)                                                                     \
            throw Error{DFB_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__)};         \
    } while (0)

// Device memory with one owner: everything allocated through it is freed when it is reset, destroyed or assigned over.
class DeviceMem {
public:
    DeviceMem() = default;
    DeviceMem(DeviceMem&& o) noexcept : ptrs_(std::move(o.ptrs_)) { o.ptrs_.clear(); }
    DeviceMem& operator=(DeviceMem&& o) noexcept {
        if (this != &o) { reset(); ptrs_ = std::move(o.ptrs_); o.ptrs_.clear(); }
        return *this;
    }
    ~DeviceMem() { reset(); }
    // frees everything; the first error of the frees
    cudaError_t reset() {
        cudaError_t first = cudaSuccess;
        for (void* p : ptrs_) {
            const cudaError_t e = cudaFree(p);
            if (first == cudaSuccess) first = e;
        }
        ptrs_.clear();
        return first;
    }
    template <class T>
    T* alloc(size_t n) {
        void* p = nullptr;
        CUDA_TRY(cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T)));
        ptrs_.push_back(p);
        return static_cast<T*>(p);
    }
    template <class T>
    T* zeroed(size_t n, cudaStream_t st) {
        T* p = alloc<T>(n);
        CUDA_TRY(cudaMemsetAsync(p, 0, std::max<size_t>(n, 1) * sizeof(T), st));
        return p;
    }
    template <class T>
    T* upload(const std::vector<T>& v, cudaStream_t st) {
        T* p = alloc<T>(v.size());
        if (!v.empty()) CUDA_TRY(cudaMemcpyAsync(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, st));
        return p;
    }

private:
    std::vector<void*> ptrs_;
};

// A face map on the device (dfb_facemap_create): the taps of facemap.hpp, and what dfb_interp_to_host needs to deliver the served faces
struct FaceMapDev {
    int kind = DFB_MAP_POINT, n = 0, n_served = 0;
    std::vector<int> served, faces;   // host: 0/1 per face; the served faces in order
    int* idx = nullptr;
    int* ptr = nullptr;               // DFB_MAP_AREA only
    int* slot = nullptr;              // face -> its row in stage; nullptr when every face is served (face i -> i)
    double* w = nullptr;
    double* stage = nullptr;          // [5][n_served], allocated by the first dfb_interp_to_host
    DeviceMem mem;
};

// What of the step's plan follows from the coefficients (build_sweeps): their device table, and the forms, work descriptions, tensor
// maps and grids of the sweeps for each buffer set b.  The plane's buffers and the noise tables follow from the half-widths alone and
// belong to the handle.
struct Sweeps {
    bool tuned = false;
    int y_form = 0;                           // 0 dense band matrices, 1 chunk-recursive, 2 run-recursive, 3 run + dense
    int n_tiles_dense = 0, n_tiles_rec = 0;   // y-sweep tiles: dense band-matrix tiles first, then recursive tiles
    YParams y[2]{};
    ZParams z[2]{};
    YMaps ymaps[2]{};
    YRMaps rmaps[2]{};                        // run-recursive y-sweep (the default form): tensor maps of r_ys with its box
    ZMaps zmaps[2]{};
    const int64_t* coef_ptr = nullptr;        // the coefficient table that PlaneDev::coef_ptr / coef_vals of both sets point at
    const double* coef_vals = nullptr;
    unsigned long long* tl = nullptr;         // development aid (DFB_TIMELINE): 64 steps x {noise, y, z} x {start, end}
    DeviceMem mem;

    // dfb_info 3, 7 and 10; the kernel forms a restart file records
    std::array<int, 3> forms() const { return {tuned ? 1 : 0, tuned ? z[0].zmode : 0, tuned ? y_form : -1}; }
};

}  // namespace

struct dfb_filter_s {
    Plan plan;
    int device = 0;
    int noise_mode = DFB_NOISE_GENERATE;
    uint64_t seed = 0;
    uint64_t fingerprint = 0;         // of the filter tables (restart.hpp): what a restart file must match
    int plane_id = 0;
    int nplanes = 1;                  // planes advanced together by this handle (dfb_create_batch): plane p draws from stream group plane_id + p
    int64_t step = 0;                 // steps completed (the constructor's first step counts as one)
    bool injected[3] = {false, false, false};
    cudaStream_t stream = nullptr;    // main stream (high priority): sweeps + epilogue
    cudaStream_t side = nullptr;      // low-priority stream: next step's noise, generated while this step filters
    cudaStream_t copy = nullptr;      // dfb_filter_to_host_begin/end: device-to-host copies of step t under the compute of step t+1
    // dfb_attach_stream: while attached, `stream` IS the caller's stream (every call that enqueues or synchronises uses it) and the
    // handle's own main stream waits in own_stream; the step's host state lives in the device record `rec`
    bool attached = false;
    cudaStream_t own_stream = nullptr;
    StepRecord* rec = nullptr;
    AdvanceParams adv{};              // what every attached step's advance launch takes (rec, time scales, seed, streams, pairs)
    double* stage[2] = {nullptr, nullptr};                 // staged copies of the five output fields
    cudaEvent_t ev_staged[2] = {nullptr, nullptr}, ev_copied[2] = {nullptr, nullptr};
    long long pipe_begun = 0, pipe_ended = 0;
    DeviceMem mem;                    // device memory that lives as long as the handle (dalloc, upload)
    // Two noise buffer sets (r_ys, r_zs): step s uses set s&1, so noise(s+1) can be written while
    // y(s)/z(s) still read set s&1.  D[b] differs from D[1-b] only in the r_ys / r_zs pointers.
    PlaneDev D[2]{};
    int64_t buf_step[2] = {-1, -1};   // which step's noise set b currently holds (or -1)
    int noise_view = 0;               // set holding the most recently consumed / generated noise
    cudaEvent_t ev_noise[2] = {nullptr, nullptr};   // noise into set b complete (either stream)
    cudaEvent_t ev_free[2] = {nullptr, nullptr};    // last readers of set b complete (main stream)
    Sweeps sw;                        // the sweeps of both sets and the coefficient table (build_sweeps)
    // noise
    NoiseParams np{};                 // geometry of the drawn arrays (fixed), their states (per step: fill_noise_params)
    uint64_t npairs[6] = {};          // pairs one step draws from each array's stream
    NoiseWindows nwin{};              // periodic_z: segment windows of the r_ys arrays whose extended rows wrap (else all nullptr)
    // N2: running statistics (opt-in)
    double* stats = nullptr;          // [P][6][Ny*W]: sum u'^2, v'^2, w'^2, T'^2, rho'^2, u'v'
    int64_t stats_count = 0;
    bool stats_on = false;
    // correlation statistics (opt-in, dfb_corr_enable): lagged products of u', v', w' along z, y and in time, after the z-sweep
    bool corr_on = false;
    bool corr_ready = false;          // sums allocated and readable (the first dfb_corr_enable(h, 1, ..) has succeeded)
    CorrParams corr{};                // lags, sums, scratch, ring
    int64_t corr_count = 0;           // accumulated steps
    std::vector<int64_t> corr_tsteps; // [L_t + 1]: accumulated steps that had an accumulated predecessor m steps back in the ring
    DeviceMem corr_sums;              // corr.sum: replaced when the lags change
    DeviceMem corr_work;              // corr.ring and corr.part: they exist only while accumulating
    // config 4: this handle as one spanwise slab of a plane shared with the other ranks of a job (dfb_comm_init)
    ncclComm_t comm = nullptr;
    int comm_rank = -1, comm_world = 0;
    std::vector<int> comm_bounds;     // [2*world]: k_begin, k_end of every rank
    cudaStream_t comm_stream = nullptr;   // NCCL transfers
    cudaStream_t asm_stream = nullptr;    // destination rank: assembly of a slab while the next one is on the wire
    cudaEvent_t ev_slab[16] = {};         // slab of rank r has landed (comm_stream)
    double* g_send = nullptr;         // staged u', v', w' of this slab: [3][Ny][W]
    double* g_recv = nullptr;         // dst rank: every rank's staged slab back to back, [rank][3][Ny][W_rank]
    double* g_plane = nullptr;        // dst rank: the assembled plane, [5][Ny][NzG]
    std::vector<size_t> g_recv_off;   // offsets (doubles) of the ranks' slabs in g_recv
    cudaEvent_t ev_gstaged = nullptr, ev_gdone = nullptr;
    // peer-to-peer transport of the hand-off (default; NCCL send/recv when CUDA IPC is not available between the ranks):
    // the destination's plane and every rank's flag block are mapped into the other ranks through CUDA IPC; a sender's copy
    // engine writes its slab straight into the plane's final layout over NVLink, flags (stream memory operations) order it
    int transport = 0;                // 0 none yet, 1 NCCL send/recv + assembly, 2 peer-to-peer copies
    unsigned long long* flags = nullptr;          // this rank's flag block: [r] = last gather whose slab of rank r has landed here; [32] = last gather this rank may write for
    unsigned long long* peer_flags[16] = {};      // the other ranks' flag blocks
    double* peer_plane = nullptr;     // the destination's g_plane as mapped here
    int peer_plane_of = -1;
    unsigned long long* seq_ring = nullptr;       // pinned host ring of gather sequence numbers (sources of the 8-byte flag copies)
    unsigned long long g_seq = 0;
    int g_dst = -1;
    int64_t g_begun = 0, g_ended = 0, g_bytes_wire = 0;
    bool g_after_first_only = false;  // the gathered step was the constructor's: T', rho' are zero (df.cpp:57-65)
    // face maps of the CFD hand-off (dfb_facemap_create): map id = index; a destroyed map leaves nullptr
    std::vector<std::unique_ptr<FaceMapDev>> facemaps;
    // per-row time scales (dfb_set_time_scales; the rows themselves are plan.Lt_rows): the blend constants {sa, sb} of every (field,
    // row) in device memory.  Host-driven steps: rows_tab holds those of dt = rows_dt, computed on the host and uploaded on the main
    // stream before a step whose dt differs (the z-sweeps that read the table are on that stream too, so one table serves both buffer
    // sets).  The uploads come from a ring of ROWS_SLOTS pinned slots: a slot is rewritten only after the event recorded behind its
    // last copy, so the host may run that many uploads ahead of the device.  Attached steps: step_advance_rows_kernel writes rows_att
    // from Lt_rows_dev.
    static constexpr int ROWS_SLOTS = 4;
    double* Lt_rows_dev = nullptr;    // [3][Ny]
    double2* rows_tab = nullptr;      // [3][Ny]
    double2* rows_att = nullptr;      // [3][Ny]
    double2* rows_host = nullptr;     // pinned, [ROWS_SLOTS][3][Ny]
    cudaEvent_t ev_rows[ROWS_SLOTS] = {};
    int rows_next = 0;
    double rows_dt = std::numeric_limits<double>::quiet_NaN();   // dt of rows_tab (NaN: none)
    // inflow mass-flux correction (dfb_set_flux_correction): the mode, the host tables of the mode last enabled (mode 0: never
    // enabled) and the device buffers, allocated by the first enable
    int flux_mode = DFB_FLUX_OFF;
    FluxTables flux_tab;
    FluxParams fx{};
    double* fx_wz = nullptr;          // [Ny][W] the per-cell weights of flux_tab (per-cell profiles), allocated by the first need
    // per-cell profiles (dfb_set_profiles; the quantities themselves are plan.cells): the epilogue's constants of this handle's cells,
    // [7][Ny][W], allocated by the first dfb_set_profiles
    double* prof_dev = nullptr;
    // timing
    bool timing = false;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    float last_ms[4] = {0, 0, 0, 0};

    void comm_release();              // ncclCommDestroy through the lazily loaded library (below)
    template <class T>
    T* dalloc(size_t n, bool zero = true) { return zero ? mem.zeroed<T>(n, stream) : mem.alloc<T>(n); }
    template <class T>
    T* upload(const std::vector<T>& v) { return mem.upload(v, stream); }
    ~dfb_filter_s() {
        cudaSetDevice(device);
        if (attached) { cudaStreamSynchronize(stream); stream = own_stream; }
        if (side) cudaStreamSynchronize(side);
        if (stream) cudaStreamSynchronize(stream);
        facemaps.clear();             // the device memory goes here, not after the last cudaGetLastError below
        sw = Sweeps{};
        corr_sums.reset();
        corr_work.reset();
        mem.reset();
        for (auto& e : ev) if (e) cudaEventDestroy(e);
        for (int b = 0; b < 2; ++b) { if (ev_noise[b]) cudaEventDestroy(ev_noise[b]); if (ev_free[b]) cudaEventDestroy(ev_free[b]); }
        for (int q = 0; q < 2; ++q) { if (ev_staged[q]) cudaEventDestroy(ev_staged[q]); if (ev_copied[q]) cudaEventDestroy(ev_copied[q]); }
        if (comm_stream) cudaStreamSynchronize(comm_stream);
        if (asm_stream) { cudaStreamSynchronize(asm_stream); cudaStreamDestroy(asm_stream); }
        for (auto& e : ev_slab) if (e) cudaEventDestroy(e);
        for (auto& pf : peer_flags) if (pf) cudaIpcCloseMemHandle(pf);
        if (peer_plane) cudaIpcCloseMemHandle(peer_plane);
        if (seq_ring) cudaFreeHost(seq_ring);
        if (rows_host) cudaFreeHost(rows_host);
        for (auto& e : ev_rows) if (e) cudaEventDestroy(e);
        if (ev_gstaged) cudaEventDestroy(ev_gstaged);
        if (ev_gdone) cudaEventDestroy(ev_gdone);
        comm_release();
        if (comm_stream) cudaStreamDestroy(comm_stream);
        if (copy) cudaStreamDestroy(copy);
        if (side) cudaStreamDestroy(side);
        if (stream) cudaStreamDestroy(stream);
        cudaGetLastError();               // nothing above is checked (a peer that has already gone makes its IPC mapping fail to close):
                                          // do not leave an error behind for the next call of this thread to trip over
    }
};

namespace {

// a driver entry point, reached through the runtime (the library does not link libcuda)
template <class Fn>
Fn driver_fn(const char* name) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    CUDA_TRY(cudaGetDriverEntryPoint(name, &p, cudaEnableDefault, &q));
    if (q != cudaDriverEntryPointSuccess || !p) throw Error{DFB_ERR_CUDA, std::string(name) + " not available"};
    return reinterpret_cast<Fn>(p);
}

typedef CUresult (*StreamWaitValue64Fn)(CUstream, CUdeviceptr, cuuint64_t, unsigned int);
StreamWaitValue64Fn stream_wait_value64() { static const auto fn = driver_fn<StreamWaitValue64Fn>("cuStreamWaitValue64"); return fn; }

void timeline_reset(unsigned long long* tl) {
    std::vector<unsigned long long> init(512, 0ull);
    for (int i = 0; i < 512; i += 2) init[i] = ~0ull;                  // starts: atomicMin
    CUDA_TRY(cudaMemcpy(tl, init.data(), 512 * sizeof(unsigned long long), cudaMemcpyHostToDevice));
}

// Tile queues of the run-recursive y-sweep (one per buffer set: {next tile, producers done}): at rest they hold the size of the
// persistent grid -- CTA b starts on tile b, the kernel puts the value back when its last producer has finished.  Written when the
// sweeps are built and again whenever the grid changes (dfb_comm_init leaving SMs free for NCCL); the stream is idle then.
void reset_run_queues(const dfb_filter_s& H, const Sweeps& sw) {
    if (!sw.y[0].rcounter) return;
    CUDA_TRY(cudaStreamSynchronize(H.stream));
    if (H.side) CUDA_TRY(cudaStreamSynchronize(H.side));
    for (int b = 0; b < 2; ++b) {
        const int grid = (int)std::min<long long>((long long)sw.y[b].n_rtiles * H.nplanes, (long long)sw.y[b].r_grid);
        const int init[2] = {grid, 0};
        CUDA_TRY(cudaMemcpy(sw.y[b].rcounter, init, sizeof(init), cudaMemcpyHostToDevice));
    }
}

// one TMA descriptor of an r_ys / r_zs array: float64, unit element strides, 256-byte L2 promotion, no out-of-bounds fill
void encode_map(CUtensorMap& m, double* base, cuuint32_t rank, const cuuint64_t* dims, const cuuint64_t* strides, const cuuint32_t* box,
                CUtensorMapSwizzle swizzle, const char* what) {
    static const auto encode_tiled = driver_fn<decltype(&cuTensorMapEncodeTiled)>("cuTensorMapEncodeTiled");
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    CUresult r = encode_tiled(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, rank, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle,
                                CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) throw Error{DFB_ERR_CUDA, std::string("cuTensorMapEncodeTiled") + what + " failed (" + std::to_string((int)r) + ")"};
}

std::optional<int> env_int(const char* name) { const char* e = std::getenv(name); return e ? std::optional<int>(std::atoi(e)) : std::nullopt; }

StepPlan plan_for_device(const dfb_filter_s& H, const Plan& P) {
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, H.device));
    return plan_step(P, H.nplanes, DeviceLimits{prop.multiProcessorCount, prop.sharedMemPerBlockOptin},
                     Overrides{env_int("DFB_Y_MODE"), env_int("DFB_Y_TK"), env_int("DFB_Y_COLGROUP"), env_int("DFB_ZK"), env_int("DFB_Z_MODE")});
}

Sweeps build_sweeps(const dfb_filter_s& H, const Plan& P, const StepPlan& S);

// Makes sw the handle's sweeps: both buffer sets read its coefficient table, and the memory of the sweeps it replaces is freed.
void install_sweeps(dfb_filter_s& H, Sweeps&& sw) {
    H.sw = std::move(sw);
    for (PlaneDev& D : H.D) { D.coef_ptr = H.sw.coef_ptr; D.coef_vals = H.sw.coef_vals; }
}

// Carries out the step's plan (stepplan.cpp) on the device: allocations, uploads, tensor maps, kernel attributes, occupancy.
void build_device(dfb_filter_s& H) {
    const Plan& P = H.plan;
    const int NP = H.nplanes, Ny = P.Ny, W = P.Nz();
    const StepPlan S = plan_for_device(H, P);
    PlaneDev& D = H.D[0];
    D = S.D;
    D.rowc = H.upload(S.rowc);
    D.T_fluc = H.dalloc<double>((size_t)NP * Ny * W);
    D.rho_fluc = H.dalloc<double>((size_t)NP * Ny * W);
    for (int f = 0; f < 3; ++f) {
        const FieldPlan& FP = P.f[f];
        FieldDev& F = D.f[f];
        F.r_ys = H.dalloc<double>(NP * F.ps_ys);
        F.r_zs = H.dalloc<double>(NP * F.ps_zs);
        F.filt_old = H.dalloc<double>((size_t)NP * Ny * W);
        F.fluc = H.dalloc<double>((size_t)NP * Ny * W);
        F.Ny_row = H.upload(FP.N_y_row);
        F.Nz_row = H.upload(FP.N_z_row);
        F.Ny_cell = FP.row_uniform ? nullptr : H.upload(FP.N_y);
        F.Nz_cell = FP.row_uniform ? nullptr : H.upload(FP.N_z);
    }
    H.D[1] = H.D[0];
    for (int f = 0; f < 3; ++f) {
        H.D[1].f[f].r_ys = H.dalloc<double>(NP * D.f[f].ps_ys);
        H.D[1].f[f].r_zs = H.dalloc<double>(NP * D.f[f].ps_zs);
    }
    install_sweeps(H, build_sweeps(H, P, S));

    H.np = S.np;
    for (int n = 0; n < H.np.n_arrays; ++n) {
        const NoiseTable& A = S.noise[n];
        H.np.a[n].seg_jump = H.upload(A.jump); H.np.a[n].seg_off = H.upload(A.off); H.np.a[n].seg_np = H.upload(A.np);
        H.nwin.seg_win[n] = A.win.empty() ? nullptr : H.upload(A.win);
        H.npairs[n] = A.npairs;
    }
    H.np.slot_jump = H.upload(S.slot_jump);
    CUDA_TRY(cudaStreamSynchronize(H.stream));
}

// What of the step's plan follows from the coefficients of P: their table, and the forms, work descriptions, tensor maps and grids of
// the sweeps.  The layout, the plane's buffers and the noise tables follow from the half-widths alone (build_device).  The handle is
// not changed, so that dfb_set_filter_shape can build new sweeps beside the old ones and install them only when this has succeeded.
Sweeps build_sweeps(const dfb_filter_s& H, const Plan& P, const StepPlan& S) {
    const int NP = H.nplanes, Ny = P.Ny;
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, H.device));
    Sweeps sw;
    DeviceMem& mem = sw.mem;
    sw.tuned = S.tuned;
    sw.coef_ptr = mem.upload(P.coef.ptr, H.stream);
    sw.coef_vals = mem.upload(P.coef.vals, H.stream);
    PlaneDev D[2] = {H.D[0], H.D[1]};                    // the buffer sets as the sweeps see them: with the new table
    for (PlaneDev& d : D) { d.coef_ptr = sw.coef_ptr; d.coef_vals = sw.coef_vals; }

    if (sw.tuned) {
        YParams& Y = sw.y[0];
        Y = S.yp;
        Y.yrec = mem.upload(S.yrec, H.stream); Y.ygc = mem.upload(S.ygc, H.stream);
        Y.resident_grid = env_int("DFB_Y_PERSIST").value_or(0);
        Y.groups = mem.upload(S.groups, H.stream); Y.tiles = mem.upload(S.tiles, H.stream); Y.cmat = mem.upload(S.cmat, H.stream);
        Y.D = D[0];
        Y.prof = mem.zeroed<unsigned long long>(8, H.stream);
        if (std::getenv("DFB_TIMELINE")) { sw.tl = mem.zeroed<unsigned long long>(512, H.stream); timeline_reset(sw.tl); }
        Y.debug = env_int("DFB_DEBUG_Y").value_or(0);
        sw.y_form = S.y_form; sw.n_tiles_dense = S.n_tiles_dense; sw.n_tiles_rec = S.n_tiles_rec;
        if (sw.y_form >= 2) {
            Y.rgroups = mem.upload(S.rgroups, H.stream); Y.rtiles = mem.upload(S.rtiles, H.stream);
            Y.rcounter = mem.alloc<int>(4);                 // tile queues, filled by reset_run_queues() below
            CUDA_TRY(ysweep_run_prepare((size_t)Y.r_smem));
        }
        sw.y[1] = Y; sw.y[1].D = D[1];
        if (sw.y[1].rcounter) sw.y[1].rcounter += 2;
        reset_run_queues(H, sw);
        CUDA_TRY(ysweep_prepare());
        ZParams& Z = sw.z[0];
        Z = S.zp;
        Z.D = D[0];
        Z.coef_pad = mem.upload(S.coef_pad, H.stream); Z.coef_pad_ptr = mem.upload(S.coef_pad_ptr, H.stream);
        Z.units = mem.upload(S.units, H.stream);
        Z.unit_par = S.unit_par.empty() ? nullptr : mem.upload(S.unit_par, H.stream);
        Z.counter = mem.zeroed<int>(2, H.stream);   // one work counter per buffer set: y(s+1) resets its own while z(s) still pulls from the other
        Z.debug = env_int("DFB_DEBUG_Z").value_or(0);
        Z.prof = mem.zeroed<unsigned long long>(4096, H.stream);
        int zb = 1;
        CUDA_TRY(zsweep_prepare(Z.zk, Z.zmode, (size_t)Z.smem_bytes, &zb));
        // The recursive form is bound by shared-memory traffic and latency, not by the fp64 pipe: two CTAs per SM run it as
        // fast as three would in the step as a whole, because the third's registers go to the next step's noise CTAs, which
        // then run beside the sweep instead of after it (measured: 0.168 vs 0.176 ms/step on 1024x2048 profile).
        if (Z.zmode == 1 && Z.zk == 16) zb = std::min(zb, 2);
        if (std::getenv("DFB_Z_BLOCKS_PER_SM")) zb = std::min(std::max(zb, 3), std::atoi(std::getenv("DFB_Z_BLOCKS_PER_SM")));
        Z.nblocks = std::max(1, std::min(std::max(zb, 1) * prop.multiProcessorCount, (Z.n_items * NP + 3) / 4));
        sw.y[0].zcounter = Z.counter; sw.y[1].zcounter = Z.counter + 1;
        sw.z[1] = Z; sw.z[1].D = D[1]; sw.z[1].counter = Z.counter + 1;
        for (int b = 0; b < 2; ++b)
            for (int f = 0; f < 3; ++f) {
                const FieldDev& F = D[b].f[f];
                const cuuint64_t ydims[2] = {(cuuint64_t)F.We, (cuuint64_t)F.rows_y * (cuuint64_t)NP};   // planes of a batch stacked along the rows
                const cuuint64_t ystrides[1] = {(cuuint64_t)F.pitch_y * sizeof(double)};
                const cuuint32_t ybox[2] = {(cuuint32_t)Y.tk, (cuuint32_t)Y_RC}, rbox[2] = {(cuuint32_t)YR_C, (cuuint32_t)YR_BOX};
                encode_map(sw.ymaps[b].m[f], F.r_ys, 2, ydims, ystrides, ybox, CU_TENSOR_MAP_SWIZZLE_NONE, "");
                if (sw.y_form >= 2) encode_map(sw.rmaps[b].m[f], F.r_ys, 2, ydims, ystrides, rbox, CU_TENSOR_MAP_SWIZZLE_NONE, " (y, run form)");
                const cuuint64_t zdims[3] = {(cuuint64_t)Z.zk, (cuuint64_t)(F.pitch_z / Z.zk), (cuuint64_t)Ny * (cuuint64_t)NP};
                const cuuint64_t zstrides[2] = {(cuuint64_t)Z.zk * 8, (cuuint64_t)F.pitch_z * sizeof(double)};
                const cuuint32_t zbox[3] = {(cuuint32_t)Z.zk, (cuuint32_t)Z.box_lines, 1u};
                encode_map(sw.zmaps[b].m[f], F.r_zs, 3, zdims, zstrides, zbox, Z.zk == 16 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, " (z)");
            }
    }
    return sw;
}

// Host-driven step with per-row time scales: the device table of blend constants for dt, uploaded on the main stream when it holds
// another dt (see dfb_filter_s::rows_tab).  Called before the step's first launch: nothing goes between its y- and z-sweep.
const double2* rows_for_step(dfb_filter_s& H, double dt) {
    if (H.rows_dt == dt) return H.rows_tab;
    const size_t n = H.plan.Lt_rows.size();
    const int slot = H.rows_next;
    H.rows_next = (H.rows_next + 1) % dfb_filter_s::ROWS_SLOTS;
    CUDA_TRY(cudaEventSynchronize(H.ev_rows[slot]));            // the copy that last read this slot has completed
    double2* src = H.rows_host + (size_t)slot * n;
    for (size_t i = 0; i < n; ++i) blend_consts(dt, H.plan.Lt_rows[i], src[i].x, src[i].y);
    CUDA_TRY(cudaMemcpyAsync(H.rows_tab, src, n * sizeof(double2), cudaMemcpyHostToDevice, H.stream));
    CUDA_TRY(cudaEventRecord(H.ev_rows[slot], H.stream));
    H.rows_dt = dt;
    return H.rows_tab;
}

void fill_noise_params(dfb_filter_s& H, int64_t step) { fill_noise_states(H.np, H.npairs, H.seed, H.plane_id, H.nplanes, step); }

void launch_noise_for(dfb_filter_s& H, int64_t step, int b, cudaStream_t st) {
    fill_noise_params(H, step);
    H.np.tl = H.sw.tl ? H.sw.tl + (step % 64) * 8 : nullptr;
    CUDA_TRY(launch_noise(H.np, H.nwin, H.D[b], st));
    CUDA_TRY(cudaEventRecord(H.ev_noise[b], st));
    H.buf_step[b] = step;
}

// The sweeps of one step on the main stream, after its noise: the y-sweep (band-matrix tiles, if any, first, then the run-recursive
// tiles: disjoint rows of r_zs), the z-sweep, the per-cell profiles' rescale, the flux correction and N2 where the z-sweep's epilogue
// does not accumulate it.  Buffer set b; rec: the step record of an attached step (nullptr host-driven); tl: the step's timeline slot
// (DFB_TIMELINE) or nullptr.
void enqueue_sweeps(dfb_filter_s& H, int b, const StepConsts& S, const double2* rows, const StepRecord* rec, unsigned long long* tl) {
    const Sweeps& sw = H.sw;
    const bool first = S.first_step != 0;
    const bool accumulate = H.stats_on && !first;                  // rms_add, df.cpp:606
    const bool flux = H.flux_mode != DFB_FLUX_OFF && !first;      // the constructor's step is never corrected
    const bool profiles = H.plan.cells != nullptr;
    const bool after = flux || profiles;                           // u', T', rho' change after the z-sweep: N2 from stats_kernel after them
    if (sw.tuned) {
        YParams Y = sw.y[b];
        Y.tl = tl ? tl + 2 : nullptr;
        Y.zcounter_init = 8 * sw.z[b].nblocks;                     // the z-sweep's warps (4 per CTA) start on two fixed items each
        if (sw.y_form != 2) CUDA_TRY(launch_ysweep_tma(sw.ymaps[b], Y, sw.n_tiles_dense, sw.n_tiles_rec, H.stream));
        if (sw.y_form >= 2) CUDA_TRY(launch_ysweep_run(sw.rmaps[b], Y, H.stream));
    } else {
        CUDA_TRY(launch_ysweep_simple(H.D[b], H.stream));
    }
    if (H.timing) CUDA_TRY(cudaEventRecord(H.ev[2], H.stream));
    if (sw.tuned) {
        ZParams Z = sw.z[b];
        Z.S = S;
        Z.rec = rec;
        Z.rows = rows;
        Z.tl = tl ? tl + 4 : nullptr;
        Z.stats = (accumulate && !after) ? H.stats : nullptr;      // N2 fused into the epilogue, unless u', T', rho' change after it
        CUDA_TRY(launch_zsweep_tuned(sw.zmaps[b], Z, H.stream));
    } else {
        CUDA_TRY(launch_zsweep_simple(H.D[b], S, rec, rows, H.stream));
    }
    if (profiles) CUDA_TRY(launch_profiles(H.D[0], H.prof_dev, first ? 1 : 0, rec, H.stream));
    if (flux) {
        const FluxCells cells{H.fx_wz, H.prof_dev};
        CUDA_TRY(launch_flux(H.fx, profiles ? &cells : nullptr, rec, H.stream));
    }
    if (accumulate && (!sw.tuned || after)) CUDA_TRY(launch_stats(H.D[0], H.stats, rec, H.stream));
}

// A step of a handle attached to a caller's stream (dfb_attach_stream): advance -> noise -> y-sweep(s) -> z-sweep (-> N2 for the
// one-thread-per-cell kernels), all on that stream, buffer set 0 only, the host's decisions taken on the device from the step record.
// No side stream, no event, no synchronisation, no allocation: the step can be captured into a CUDA graph, and each replay advances
// the generator by one step.  dt_dev == nullptr: dt and its blend constants are the host's (dfb_filter), bit for bit a host-driven step.
void run_step_attached(dfb_filter_s& H, double dt, const double* dt_dev, bool first) {
    CUDA_TRY(cudaSetDevice(H.device));
    const bool accumulate = H.stats_on && !first;
    AdvanceParams A = H.adv;
    A.dt_dev = dt_dev;
    A.dt = dt;
    if (!dt_dev)
        for (int f = 0; f < 3; ++f) blend_consts(dt, H.plan.f[f].Lt, A.sa[f], A.sb[f]);
    A.stats = accumulate ? 1 : 0;
    const double2* rows = (!first && !H.plan.Lt_rows.empty()) ? H.rows_att : nullptr;
    if (rows) { A.Lt_rows = H.Lt_rows_dev; A.rows = H.rows_att; A.n_rows = (int)H.plan.Lt_rows.size(); }
    CUDA_TRY(launch_advance(A, H.stream));
    NoiseParams np = H.np;
    np.rec = H.rec;
    np.tl = nullptr;
    CUDA_TRY(launch_noise(np, H.nwin, H.D[0], H.stream));
    H.buf_step[0] = H.buf_step[1] = -1;            // the sets hold no step the host knows of: host-driven steps after a detach draw anew
    H.noise_view = 0;
    StepConsts S{};
    S.first_step = first ? 1 : 0;
    enqueue_sweeps(H, 0, S, rows, H.rec, nullptr);
}

void run_step(dfb_filter_s& H, double dt, bool first) {
    if (H.attached) { run_step_attached(H, dt, nullptr, first); return; }
    CUDA_TRY(cudaSetDevice(H.device));
    const int b = (int)(H.step & 1);
    if (H.timing) CUDA_TRY(cudaEventRecord(H.ev[0], H.stream));
    const double2* rows = (!first && !H.plan.Lt_rows.empty()) ? rows_for_step(H, dt) : nullptr;
    if (H.noise_mode == DFB_NOISE_GENERATE) {
        // ev_noise[b] = the last noise launch into set b on EITHER stream: wait for it whether its result is the one this step
        // wants (prefetched) or not (after a dfb_set_state rewind the side stream's prefetch may still be writing set b)
        CUDA_TRY(cudaStreamWaitEvent(H.stream, H.ev_noise[b], 0));
        if (H.buf_step[b] != H.step) launch_noise_for(H, H.step, b, H.stream);
    } else if (!(H.injected[0] && H.injected[1] && H.injected[2])) {
        throw Error{DFB_ERR_STATE, "noise_mode = inject: dfb_set_noise must be called for u, v and w before every step"};
    }
    H.noise_view = b;
    if (H.timing) CUDA_TRY(cudaEventRecord(H.ev[1], H.stream));
    StepConsts S{};
    S.first_step = first ? 1 : 0;
    for (int f = 0; f < 3; ++f) blend_consts(dt, H.plan.f[f].Lt, S.sa[f], S.sb[f]);
    enqueue_sweeps(H, b, S, rows, nullptr, H.sw.tl ? H.sw.tl + (H.step % 64) * 8 : nullptr);
    if (H.stats_on && !first) H.stats_count += 1;
    if (H.corr_on && !first) {
        CorrParams& c = H.corr;
        if (c.L[0]) CUDA_TRY(launch_corr_z(c, H.stream));
        if (c.L[1]) CUDA_TRY(launch_corr_y(c, H.stream));
        if (c.L[2]) {
            const int M = (int)std::min<long long>(c.L[2], c.ring_count);
            CUDA_TRY(launch_corr_t(c, M, H.stream));
            for (int m = 0; m <= M; ++m) H.corr_tsteps[m] += 1;
            c.ring_count += 1;
        }
        H.corr_count += 1;
    }
    CUDA_TRY(cudaEventRecord(H.ev_free[b], H.stream));
    if (H.timing) CUDA_TRY(cudaEventRecord(H.ev[3], H.stream));
    H.step += 1;
    H.injected[0] = H.injected[1] = H.injected[2] = false;
    // The noise of the NEXT step depends on nothing but (seed, step): generate it now, on the
    // low-priority stream, into the other buffer set, while this step's sweeps own the fp64 pipe.
    if (H.noise_mode == DFB_NOISE_GENERATE && !H.timing) {
        const int nb = (int)(H.step & 1);
        CUDA_TRY(cudaStreamWaitEvent(H.side, H.ev_free[nb], 0));     // readers of that set (step-2... ) are done
        CUDA_TRY(cudaStreamWaitEvent(H.side, H.ev_noise[nb], 0));    // ... and so is its last writer: a dfb_generate_noise into it
                                                                       // on the main stream after that step would otherwise race this one
        launch_noise_for(H, H.step, nb, H.side);
    }
    if (H.timing) {
        CUDA_TRY(cudaEventSynchronize(H.ev[3]));
        for (int s = 0; s < 3; ++s) CUDA_TRY(cudaEventElapsedTime(&H.last_ms[s], H.ev[s], H.ev[s + 1]));
        CUDA_TRY(cudaEventElapsedTime(&H.last_ms[3], H.ev[0], H.ev[3]));
    }
}

const double* field_ptr0(const dfb_filter_s& H, int which) {
    switch (which) {
        case DFB_U_FLUC: return H.D[0].f[0].fluc;   case DFB_V_FLUC: return H.D[0].f[1].fluc;   case DFB_W_FLUC: return H.D[0].f[2].fluc;
        case DFB_T_FLUC: return H.D[0].T_fluc;      case DFB_RHO_FLUC: return H.D[0].rho_fluc;
        case DFB_U_FILT: return H.D[0].f[0].filt_old; case DFB_V_FILT: return H.D[0].f[1].filt_old; case DFB_W_FILT: return H.D[0].f[2].filt_old;
    }
    return nullptr;
}

// plane p of a batch: the dense arrays are [P][Ny*W]
const double* field_ptr(const dfb_filter_s& H, int which, int plane = 0) {
    const double* p = field_ptr0(H, which);
    return p ? p + (size_t)plane * H.D[0].ps_cells : nullptr;
}

// dt < 0 gives alpha = exp(-pi dt / Lt) > 1 and sqrt(1 - alpha) = NaN, a NaN dt NaN as well: either would turn every field, filt_old
// and the statistics into NaN for good.  Checked before a step enqueues anything, so a refused call leaves the handle as it was.
void check_dt(double dt) {
    if (std::isfinite(dt) && dt >= 0.0) return;
    char buf[64];
    std::snprintf(buf, sizeof(buf), "%g", dt);
    throw Error{DFB_ERR_ARG, std::string("dt must be finite and >= 0, got ") + buf};
}

const char* const VOID_STEP_MSG = "dt must be finite and >= 0: an attached step (dfb_filter_dev) read such a dt from device memory and was void";

std::string attached_msg(const char* call) { return std::string(call) + " is not available while the handle is attached to a stream (dfb_attach_stream)"; }
void refuse_attached(const dfb_filter_s& H, const char* call) { if (H.attached) throw Error{DFB_ERR_STATE, attached_msg(call)}; }

// Calls that change what a staged copy or a hand-off reads wait until neither is outstanding.  call: the message's prefix, or nullptr.
void refuse_outstanding(const dfb_filter_s& H, const char* call) {
    if (H.pipe_begun == H.pipe_ended && H.g_begun == H.g_ended) return;
    const std::string prefix = call ? std::string(call) + ": " : "";
    throw Error{DFB_ERR_STATE, prefix + "a dfb_filter_to_host_begin or dfb_gather_begin is outstanding: end it first"};
}

// Makes T the flux correction's tables: the device buffers on the first call, then the weights (steps enqueued before read the previous
// ones on this stream).
void install_flux(dfb_filter_s& H, FluxTables&& T) {
    CUDA_TRY(cudaSetDevice(H.device));
    FluxParams& F = H.fx;
    const int NP = H.nplanes, Ny = H.plan.Ny, W = H.plan.NzG;
    if (!F.out) {
        CUDA_TRY(flux_prepare());
        F.u = H.D[0].f[0].fluc; F.T = H.D[0].T_fluc; F.rho = H.D[0].rho_fluc; F.rowc = H.D[0].rowc;
        F.Ny = Ny; F.W = W; F.P = NP; F.ps_cells = H.D[0].ps_cells;
        F.wy = H.dalloc<double>(Ny, false);
        F.hz = H.upload(T.hz);
        F.part = H.dalloc<double>((size_t)NP * Ny, false);
        F.counter = H.dalloc<unsigned>(NP);
        F.out = H.dalloc<double2>(NP);
    }
    if (!T.wz.empty() && !H.fx_wz) H.fx_wz = H.dalloc<double>(T.wz.size(), false);
    CUDA_TRY(cudaMemcpyAsync(const_cast<double*>(F.wy), T.wy.data(), Ny * sizeof(double), cudaMemcpyHostToDevice, H.stream));
    if (!T.wz.empty()) CUDA_TRY(cudaMemcpyAsync(H.fx_wz, T.wz.data(), T.wz.size() * sizeof(double), cudaMemcpyHostToDevice, H.stream));
    CUDA_TRY(cudaStreamSynchronize(H.stream));
    F.D = T.D;
    H.flux_tab = std::move(T);
}

// Attached: waits for the caller's stream and reads the device step record back into the host's step counter and N2 count.  A void
// step since the last read is reported once, as DFB_ERR_ARG, and forgotten.  Host-driven: nothing.
void sync_record(dfb_filter_s& H) {
    if (!H.attached) return;
    CUDA_TRY(cudaSetDevice(H.device));
    StepRecord R;
    CUDA_TRY(cudaMemcpyAsync(&R, H.rec, sizeof(R), cudaMemcpyDeviceToHost, H.stream));
    CUDA_TRY(cudaStreamSynchronize(H.stream));
    H.step = R.step;
    H.stats_count = R.stats_count;
    if (R.void_seen) {
        static const int zero = 0;
        CUDA_TRY(cudaMemcpyAsync(&H.rec->void_seen, &zero, sizeof(zero), cudaMemcpyHostToDevice, H.stream));
        CUDA_TRY(cudaStreamSynchronize(H.stream));
        throw Error{DFB_ERR_ARG, VOID_STEP_MSG};
    }
}

// Writes the host's step counter and N2 count into the device step record (dfb_attach_stream, and dfb_set_state / dfb_load_restart
// while attached).  Its noise positions are those of the last step taken, which a void step's noise launch reproduces.
void push_record(dfb_filter_s& H) {
    StepRecord R{};
    R.step = H.step;
    R.stats_count = H.stats_count;
    NoiseParams np = H.np;
    fill_noise_states(np, H.npairs, H.seed, H.plane_id, H.nplanes, std::max<int64_t>(H.step - 1, 0));
    std::memcpy(R.pstate, np.pstate, sizeof(R.pstate));
    CUDA_TRY(cudaSetDevice(H.device));
    CUDA_TRY(cudaMemcpyAsync(H.rec, &R, sizeof(R), cudaMemcpyHostToDevice, H.stream));
    CUDA_TRY(cudaStreamSynchronize(H.stream));
}

// filt_old [3][P][Ny*W] (host; nullptr keeps it) and the step counter (dfb_set_state, dfb_load_restart)
void restore_state(dfb_filter_s& H, const double* filt_old3, int64_t step) {
    CUDA_TRY(cudaSetDevice(H.device));
    const size_t n = H.D[0].ps_cells * H.nplanes;
    if (filt_old3)
        for (int f = 0; f < 3; ++f)
            CUDA_TRY(cudaMemcpyAsync(H.D[0].f[f].filt_old, filt_old3 + f * n, n * 8, cudaMemcpyHostToDevice, H.stream));
    CUDA_TRY(cudaStreamSynchronize(H.stream));
    CUDA_TRY(cudaStreamSynchronize(H.side));      // a look-ahead noise launch for the old step counter may still be in flight
    if (step != H.step) H.buf_step[0] = H.buf_step[1] = -1;
    H.step = step;
    H.corr.ring_count = 0;       // the next step follows the restored state: no temporal pair reaches back across it
}

template <class Fn>
int guarded(Fn&& fn) {
    try {
        fn();
        return DFB_OK;
    } catch (const Error& e) {
        return fail(e.code, e.msg);
    } catch (const std::bad_alloc&) {
        return fail(DFB_ERR_ARG, "host allocation failed");
    } catch (const std::exception& e) {
        return fail(DFB_ERR_ARG, e.what());
    }
}

}  // namespace

extern "C" {

int dfb_config_init(dfb_config* cfg) {
    if (!cfg) return fail(DFB_ERR_ARG, "cfg is NULL");
    std::memset(cfg, 0, sizeof(*cfg));
    cfg->struct_bytes = (int)sizeof(dfb_config);
    cfg->grid_file_len = cfg->vel_fluc_file_len = cfg->line_file_len = -1;
    cfg->device = -1;
    return DFB_OK;
}

static int create_impl(const dfb_config* cfg, int nplanes, dfb_handle* out) {
    if (!cfg || !out) return fail(DFB_ERR_ARG, "cfg/out is NULL");
    *out = nullptr;
    if (nplanes < 1 || nplanes > DFB_MAXP) return fail(DFB_ERR_ARG, "nplanes must be 1.." + std::to_string(DFB_MAXP));
    if (cfg->struct_bytes != (int)sizeof(dfb_config))
        return fail(DFB_ERR_ARG, "dfb_config.struct_bytes does not match this library (call dfb_config_init first)");
    std::unique_ptr<dfb_filter_s> H(new dfb_filter_s());
    int rc = guarded([&] {
        int ndev = 0;
        cudaError_t e = cudaGetDeviceCount(&ndev);
        if (e != cudaSuccess || ndev == 0)
            throw Error{DFB_ERR_CUDA, std::string("no CUDA device (") + cudaGetErrorString(e) + "); this library has no CPU fallback"};
        int dev = cfg->device;
        if (dev < 0) CUDA_TRY(cudaGetDevice(&dev));
        if (dev >= ndev) throw Error{DFB_ERR_ARG, "device ordinal out of range"};
        cudaDeviceProp prop;
        CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
        if (prop.major != 10)
            throw Error{DFB_ERR_CUDA, std::string("device '") + prop.name + "' is sm_" + std::to_string(prop.major) + std::to_string(prop.minor) +
                                          "; the kernels are built for sm_100a only and there is no fallback"};
        H->device = dev;
        CUDA_TRY(cudaSetDevice(dev));
        if (cfg->noise_mode != DFB_NOISE_GENERATE && cfg->noise_mode != DFB_NOISE_INJECT) throw Error{DFB_ERR_ARG, "bad noise_mode"};
        H->noise_mode = cfg->noise_mode;
        H->seed = cfg->seed;
        H->plane_id = cfg->plane_id;
        H->nplanes = nplanes;
        if (nplanes > 1 && cfg->noise_mode != DFB_NOISE_GENERATE) throw Error{DFB_ERR_ARG, "a batch of planes generates its own noise (noise_mode = DFB_NOISE_GENERATE)"};
        build_plan(*cfg, H->plan);
        H->fingerprint = rst::fingerprint(H->plan);
        if (H->noise_mode == DFB_NOISE_INJECT && (H->plan.k0 != 0 || H->plan.k1 != H->plan.NzG))
            throw Error{DFB_ERR_ARG, "noise injection is defined on the whole plane (k_begin = k_end = 0)"};
        int prio_lo = 0, prio_hi = 0;
        CUDA_TRY(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        CUDA_TRY(cudaStreamCreateWithPriority(&H->stream, cudaStreamNonBlocking, prio_hi));
        CUDA_TRY(cudaStreamCreateWithPriority(&H->side, cudaStreamNonBlocking, prio_lo));
        for (auto& e2 : H->ev) CUDA_TRY(cudaEventCreate(&e2));
        for (int b = 0; b < 2; ++b) {
            CUDA_TRY(cudaEventCreateWithFlags(&H->ev_noise[b], cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&H->ev_free[b], cudaEventDisableTiming));
        }
        build_device(*H);
        // first step of the constructor, df.cpp:57-62 (generate mode only: in inject mode the
        // caller owns the noise and runs it through dfb_first_step semantics via dfb_filter after
        // dfb_set_noise; see dfb_set_state for a step counter of 0)
        if (H->noise_mode == DFB_NOISE_GENERATE && !cfg->skip_first_step) {
            run_step(*H, 0.0, true);
            CUDA_TRY(cudaStreamSynchronize(H->stream));
        }
    });
    if (rc != DFB_OK) return rc;
    *out = H.release();
    return DFB_OK;
}

int dfb_create(const dfb_config* cfg, dfb_handle* out) { return create_impl(cfg, 1, out); }
int dfb_create_batch(const dfb_config* cfg, int nplanes, dfb_handle* out) { return create_impl(cfg, nplanes, out); }

int dfb_num_planes(dfb_handle h, int* nplanes) {
    if (!h || !nplanes) return fail(DFB_ERR_ARG, "handle/nplanes is NULL");
    *nplanes = h->nplanes;
    return DFB_OK;
}

int dfb_destroy(dfb_handle h) {
    if (!h) return DFB_OK;
    delete h;
    return DFB_OK;
}

int dfb_dims(dfb_handle h, int* Ny, int* Nz) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    if (Ny) *Ny = h->plan.Ny;
    if (Nz) *Nz = h->plan.Nz();
    return DFB_OK;
}

int dfb_info(dfb_handle h, int what, int field, int64_t* out64) {
    if (!h || !out64) return fail(DFB_ERR_ARG, "handle/out is NULL");
    if (field < 0 || field > 2) return fail(DFB_ERR_ARG, "field must be 0..2");
    if (h->attached) {
        const int rc = guarded([&] { sync_record(*h); });
        if (rc != DFB_OK) return rc;
    }
    switch (what) {
        case 0: *out64 = h->plan.f[field].Ny_max; break;
        case 1: *out64 = h->plan.f[field].Nz_max; break;
        case 2: *out64 = h->step; break;
        case 3: *out64 = h->sw.forms()[0]; break;
        case 4: *out64 = h->plan.taps_per_step; break;
        case 5: *out64 = h->plan.NzG; break;
        case 6: *out64 = h->device; break;
        case 7: *out64 = h->sw.forms()[1]; break;
        case 8: *out64 = h->sw.tuned ? h->sw.n_tiles_rec : 0; break;
        case 9: *out64 = h->sw.tuned ? h->sw.n_tiles_dense : 0; break;
        case 10: *out64 = h->sw.forms()[2]; break;
        case 12: *out64 = h->transport; break;
        case 11: *out64 = h->sw.tuned ? h->sw.y[0].n_rtiles : 0; break;
        case 13: *out64 = h->plan.periodic ? 1 : 0; break;
        case 14: *out64 = h->corr_ready ? h->corr.L[field] : 0; break;
        case 15: *out64 = h->plan.Lt_rows.empty() ? 0 : 1; break;
        case 17: *out64 = h->plan.filter_shape; break;
        case 18: *out64 = h->flux_mode; break;
        case 19: *out64 = h->plan.cells ? 1 : 0; break;
        default: return fail(DFB_ERR_ARG, "unknown info selector");
    }
    return DFB_OK;
}

int dfb_get_table(dfb_handle h, int which, int arg, double* dst, int cap) {
    if (!h || !dst) return fail(DFB_ERR_ARG, "handle/dst is NULL");
    const Plan& P = h->plan;
    const double* src = nullptr;
    int n = 0;
    std::vector<double> tmp;
    if (which >= 0 && which < 8) { src = P.rows.data() + (size_t)which * P.Ny; n = P.Ny; }
    else if (which == 8) { src = P.yc_row.data(); n = P.Ny; }
    else if (which == 9) { src = P.dy_row.data(); n = P.Ny; }
    else if (which == 10) { tmp = {P.f[0].Lt, P.f[1].Lt, P.f[2].Lt}; src = tmp.data(); n = 3; }
    else if (which == 11) {
        if (arg < 0 || arg > P.coef.Nmax || P.coef.ptr[arg] < 0) return fail(DFB_ERR_ARG, "half-width not present in this plane");
        src = P.coef.vals.data() + P.coef.ptr[arg]; n = 2 * arg + 1;
    } else if (which == 12) { src = P.vert_y.data(); n = P.Ny + 1; }
    else if (which == 13) { src = P.vert_z.data(); n = P.NzG + 1; }
    else if (which == 14) {
        if (arg < 0 || arg > 2) return fail(DFB_ERR_ARG, "table 14: field must be 0..2");
        if (P.Lt_rows.empty()) { tmp.assign(P.Ny, P.f[arg].Lt); src = tmp.data(); }
        else src = P.Lt_rows.data() + (size_t)arg * P.Ny;
        n = P.Ny;
    } else if (which == 16) {
        if (arg < 0 || arg > 7) return fail(DFB_ERR_ARG, "table 16: quantity must be 0..7");
        n = P.Ny * P.Nz();
        if (P.cells) src = P.cells->data() + (size_t)arg * n;
        else {
            tmp.resize(n);
            for (int j = 0; j < P.Ny; ++j) std::fill_n(tmp.begin() + (size_t)j * P.Nz(), P.Nz(), P.rows[(size_t)arg * P.Ny + j]);
            src = tmp.data();
        }
    }
    else return fail(DFB_ERR_ARG, "unknown table selector");
    if (cap < n) return fail(DFB_ERR_ARG, "dst too small");
    std::memcpy(dst, src, sizeof(double) * n);
    return DFB_OK;
}

int dfb_get_half_widths(dfb_handle h, int field, int dir, int* dst) {
    if (!h || !dst || field < 0 || field > 2) return fail(DFB_ERR_ARG, "bad argument");
    const Plan& P = h->plan;
    const FieldPlan& F = P.f[field];
    for (int j = 0; j < P.Ny; ++j)
        for (int k = P.k0; k < P.k1; ++k) {
            int v = F.row_uniform ? (dir ? F.N_z_row[j] : F.N_y_row[j])
                                  : (dir ? F.N_z[(size_t)j * P.NzG + k] : F.N_y[(size_t)j * P.NzG + k]);
            dst[(size_t)j * P.Nz() + (k - P.k0)] = v;
        }
    return DFB_OK;
}

int dfb_filter(dfb_handle h, double dt) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    return guarded([&] { check_dt(dt); run_step(*h, dt, false); });
}

int dfb_first_step(dfb_handle h) {   // constructor semantics on demand (inject mode / after dfb_set_state(.., 0))
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    return guarded([&] { run_step(*h, 0.0, true); });
}

int dfb_get_field_plane(dfb_handle h, int plane, int which, double* dst, int dst_on_device) {
    if (!h || !dst) return fail(DFB_ERR_ARG, "handle/dst is NULL");
    if (plane < 0 || plane >= h->nplanes) return fail(DFB_ERR_ARG, "plane out of range");
    const double* src = field_ptr(*h, which, plane);
    if (!src) return fail(DFB_ERR_ARG, "unknown field selector");
    return guarded([&] {
        sync_record(*h);
        CUDA_TRY(cudaSetDevice(h->device));
        const size_t bytes = sizeof(double) * h->D[0].ps_cells;
        CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, dst_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->stream));
    });
}

int dfb_get_field(dfb_handle h, int which, double* dst, int dst_on_device) { return dfb_get_field_plane(h, 0, which, dst, dst_on_device); }

int dfb_filter_to_host(dfb_handle h, double dt, double* u, double* v, double* w, double* T, double* rho) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    return guarded([&] {
        check_dt(dt);
        sync_record(*h);
        run_step(*h, dt, false);
        const size_t bytes = sizeof(double) * h->D[0].ps_cells * h->nplanes;     // a batch delivers [P][Ny*Nz] per field
        double* dst[5] = {u, v, w, T, rho};
        for (int i = 0; i < 5; ++i)
            if (dst[i]) CUDA_TRY(cudaMemcpyAsync(dst[i], field_ptr(*h, i), bytes, cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->stream));
    });
}

int dfb_filter_to_host_begin(dfb_handle h, double dt, double* u, double* v, double* w, double* T, double* rho) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    return guarded([&] {
        refuse_attached(*h, "dfb_filter_to_host_begin");
        check_dt(dt);
        if (h->pipe_begun - h->pipe_ended >= 2) throw Error{DFB_ERR_STATE, "two dfb_filter_to_host_begin calls are already outstanding: call dfb_filter_to_host_end first"};
        CUDA_TRY(cudaSetDevice(h->device));
        const size_t n = h->D[0].ps_cells * h->nplanes, bytes = n * sizeof(double);
        const int p = (int)(h->pipe_begun & 1);
        if (!h->copy) {
            CUDA_TRY(cudaStreamCreateWithFlags(&h->copy, cudaStreamNonBlocking));
            for (int q = 0; q < 2; ++q) {
                h->stage[q] = h->dalloc<double>(5 * n, false);
                CUDA_TRY(cudaEventCreateWithFlags(&h->ev_staged[q], cudaEventDisableTiming));
                CUDA_TRY(cudaEventCreateWithFlags(&h->ev_copied[q], cudaEventDisableTiming));
            }
        }
        run_step(*h, dt, false);
        // stage the five fields (device to device, on the compute stream: the next step may then overwrite them), then copy the
        // staged set to the caller's arrays on the copy stream while the next step computes
        CUDA_TRY(cudaStreamWaitEvent(h->stream, h->ev_copied[p], 0));          // the copy that last read this staging set (a no-op before its first use)
        double* dst[5] = {u, v, w, T, rho};
        for (int i = 0; i < 5; ++i)
            if (dst[i]) CUDA_TRY(cudaMemcpyAsync(h->stage[p] + (size_t)i * n, field_ptr(*h, i), bytes, cudaMemcpyDeviceToDevice, h->stream));
        CUDA_TRY(cudaEventRecord(h->ev_staged[p], h->stream));
        CUDA_TRY(cudaStreamWaitEvent(h->copy, h->ev_staged[p], 0));
        for (int i = 0; i < 5; ++i)
            if (dst[i]) CUDA_TRY(cudaMemcpyAsync(dst[i], h->stage[p] + (size_t)i * n, bytes, cudaMemcpyDeviceToHost, h->copy));
        CUDA_TRY(cudaEventRecord(h->ev_copied[p], h->copy));
        h->pipe_begun += 1;
    });
}

int dfb_filter_to_host_end(dfb_handle h) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    return guarded([&] {
        refuse_attached(*h, "dfb_filter_to_host_end");
        if (h->pipe_ended >= h->pipe_begun) throw Error{DFB_ERR_STATE, "no dfb_filter_to_host_begin is outstanding"};
        CUDA_TRY(cudaEventSynchronize(h->ev_copied[(int)(h->pipe_ended & 1)]));
        h->pipe_ended += 1;
    });
}

int dfb_filter_batch(dfb_handle h, int nsteps, const double* dt, double* out) {
    if (!h || !dt || nsteps < 0) return fail(DFB_ERR_ARG, "bad argument");
    return guarded([&] {
        refuse_attached(*h, "dfb_filter_batch");
        for (int s = 0; s < nsteps; ++s) check_dt(dt[s]);            // the whole array before the first step
        const size_t n = h->D[0].ps_cells * h->nplanes;
        for (int s = 0; s < nsteps; ++s) {
            run_step(*h, dt[s], false);
            if (out)
                for (int i = 0; i < 5; ++i)
                    CUDA_TRY(cudaMemcpyAsync(out + ((size_t)s * 5 + i) * n, field_ptr(*h, i), n * sizeof(double),
                                             cudaMemcpyDeviceToHost, h->stream));
        }
        CUDA_TRY(cudaStreamSynchronize(h->stream));
    });
}

int dfb_device_ptr_plane(dfb_handle h, int plane, int which, void** ptr) {
    if (!h || !ptr) return fail(DFB_ERR_ARG, "handle/ptr is NULL");
    if (plane < 0 || plane >= h->nplanes) return fail(DFB_ERR_ARG, "plane out of range");
    const double* p = field_ptr(*h, which, plane);
    if (!p) return fail(DFB_ERR_ARG, "unknown field selector");
    *ptr = const_cast<double*>(p);
    return DFB_OK;
}
int dfb_device_ptr(dfb_handle h, int which, void** ptr) { return dfb_device_ptr_plane(h, 0, which, ptr); }

int dfb_scatter_to_cells(dfb_handle h, int which, int n, const int* plane_index, const int* dst_index, const double* mean, double scale,
                         double* dst) {
    if (!h || n < 0 || (n > 0 && (!plane_index || !dst_index || !dst))) return fail(DFB_ERR_ARG, "bad argument");
    const double* p = field_ptr(*h, which);
    if (!p) return fail(DFB_ERR_ARG, "unknown field selector");
    return guarded([&] {
        CUDA_TRY(cudaSetDevice(h->device));
        CUDA_TRY(launch_scatter(p, n, plane_index, dst_index, mean, scale, dst, h->stream));
    });
}

int dfb_stream(dfb_handle h, void** stream) {
    if (!h || !stream) return fail(DFB_ERR_ARG, "handle/stream is NULL");
    *stream = h->stream;
    return DFB_OK;
}

// page-lock / release a caller-owned host array so that the five copies of dfb_filter_to_host run at the PCIe rate
// (the facades call these for their own std::vector / allocatable storage)
int dfb_host_register(void* ptr, size_t bytes) {
    if (!ptr || bytes == 0) return fail(DFB_ERR_ARG, "bad argument");
    return guarded([&] { CUDA_TRY(cudaHostRegister(ptr, bytes, cudaHostRegisterPortable)); });
}
int dfb_host_unregister(void* ptr) {
    if (!ptr) return fail(DFB_ERR_ARG, "bad argument");
    return guarded([&] { CUDA_TRY(cudaHostUnregister(ptr)); });
}

int dfb_sync(dfb_handle h) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    return guarded([&] { CUDA_TRY(cudaSetDevice(h->device)); CUDA_TRY(cudaStreamSynchronize(h->stream)); sync_record(*h); });
}

int dfb_attach_stream(dfb_handle h, void* stream) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    return guarded([&] {
        if (!stream) {                                   // detach: the record back to the host, the handle's own stream again
            if (!h->attached) return;
            std::string void_msg;
            try { sync_record(*h); } catch (const Error& e) { if (e.code != DFB_ERR_ARG) throw; void_msg = e.msg; }
            h->stream = h->own_stream;
            h->own_stream = nullptr;
            h->attached = false;
            if (!void_msg.empty()) throw Error{DFB_ERR_ARG, void_msg};
            return;
        }
        if (h->attached) throw Error{DFB_ERR_STATE, "dfb_attach_stream: the handle is attached already (detach with stream = NULL first)"};
        if (h->noise_mode != DFB_NOISE_GENERATE) throw Error{DFB_ERR_STATE, "dfb_attach_stream: a handle in inject mode cannot be attached"};
        if (h->corr_on) throw Error{DFB_ERR_STATE, "dfb_attach_stream: correlation statistics are on (dfb_corr_enable(h, 0, NULL) first)"};
        if (h->timing) throw Error{DFB_ERR_STATE, "dfb_attach_stream: timing is on (dfb_set_timing(h, 0) first)"};
        refuse_outstanding(*h, "dfb_attach_stream");
        int dev = -1;
        CUDA_TRY(cudaStreamGetDevice(static_cast<cudaStream_t>(stream), &dev));
        if (dev != h->device)
            throw Error{DFB_ERR_ARG, "dfb_attach_stream: the stream belongs to device " + std::to_string(dev) + ", the handle to device " +
                                         std::to_string(h->device)};
        CUDA_TRY(cudaSetDevice(h->device));
        CUDA_TRY(attach_prepare());
        if (!h->rec) h->rec = h->dalloc<StepRecord>(1);
        CUDA_TRY(cudaStreamSynchronize(h->side));        // the look-ahead noise of the next host-driven step is not used
        AdvanceParams& A = h->adv;
        A = AdvanceParams{};
        A.rec = h->rec;
        for (int f = 0; f < 3; ++f) A.Lt[f] = h->plan.f[f].Lt;
        A.seed = h->seed;
        NoiseParams np = h->np;
        fill_noise_states(np, h->npairs, h->seed, h->plane_id, h->nplanes, 0);
        std::memcpy(A.pinc, np.pinc, sizeof(A.pinc));
        for (int n = 0; n < 6; ++n) A.npairs[n] = h->npairs[n];
        A.n_arrays = h->np.n_arrays;
        A.P = h->nplanes;
        push_record(*h);                                 // on the handle's own stream, which it also drains
        h->own_stream = h->stream;
        h->stream = static_cast<cudaStream_t>(stream);
        h->attached = true;
    });
}

int dfb_filter_dev(dfb_handle h, const double* dt_dev) {
    if (!h || !dt_dev) return fail(DFB_ERR_ARG, "handle/dt_dev is NULL");
    if (!h->attached) return fail(DFB_ERR_STATE, "dfb_filter_dev needs a stream attached with dfb_attach_stream");
    return guarded([&] { run_step_attached(*h, 0.0, dt_dev, false); });
}

int dfb_set_time_scales(dfb_handle h, const double* Lt_rows) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    if (h->attached) return fail(DFB_ERR_STATE, attached_msg("dfb_set_time_scales") + ": set the rows before attaching");
    return guarded([&] {
        refuse_outstanding(*h, "dfb_set_time_scales");
        Plan& P = h->plan;
        if (!Lt_rows) {
            P.Lt_rows.clear();
            h->fingerprint = rst::fingerprint(P);
            return;
        }
        check_time_scales(P, Lt_rows);
        const size_t n = (size_t)3 * P.Ny;
        CUDA_TRY(cudaSetDevice(h->device));
        if (!h->rows_host) {
            h->Lt_rows_dev = h->dalloc<double>(n, false);
            h->rows_tab = h->dalloc<double2>(n, false);
            h->rows_att = h->dalloc<double2>(n, false);
            for (auto& e : h->ev_rows) CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            CUDA_TRY(cudaHostAlloc(&h->rows_host, dfb_filter_s::ROWS_SLOTS * n * sizeof(double2), cudaHostAllocDefault));
        }
        // the attached steps' copy of the rows; the handle is not attached, so no step reads it now
        CUDA_TRY(cudaMemcpyAsync(h->Lt_rows_dev, Lt_rows, n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        P.Lt_rows.assign(Lt_rows, Lt_rows + n);
        h->rows_dt = std::numeric_limits<double>::quiet_NaN();    // the next step uploads the new rows' constants
        h->fingerprint = rst::fingerprint(P);
    });
}

int dfb_time_scales_from_lengths(dfb_handle h, const double Ix[6], double u_min, double* Lt_rows) {
    if (!h || !Ix || !Lt_rows) return fail(DFB_ERR_ARG, "handle/Ix/Lt_rows is NULL");
    return guarded([&] { time_scales_from_lengths(h->plan, Ix, u_min, Lt_rows); });
}

int dfb_set_filter_shape(dfb_handle h, int shape) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    if (shape != DFB_FILTER_EXPONENTIAL && shape != DFB_FILTER_GAUSSIAN)
        return fail(DFB_ERR_ARG, "unknown filter shape " + std::to_string(shape) + " (DFB_FILTER_EXPONENTIAL = 0, DFB_FILTER_GAUSSIAN = 1)");
    const char* why = nullptr;
    if (h->attached) why = "the handle is attached to a stream (dfb_attach_stream)";
    else if (h->step != 0) why = "the handle has stepped (create it with skip_first_step = 1, set the shape, then call dfb_first_step)";
    else if (h->comm) why = "the handle has a communicator (dfb_comm_init)";
    else if (h->stats_on) why = "N2 statistics are enabled (dfb_stats_enable)";
    else if (h->corr_on) why = "correlation statistics are enabled (dfb_corr_enable)";
    else if (!h->plan.Lt_rows.empty()) why = "per-row time scales are set (dfb_set_time_scales)";
    else if (std::any_of(h->facemaps.begin(), h->facemaps.end(), [](const auto& m) { return m != nullptr; }))
        why = "the handle has face maps (dfb_facemap_create)";
    else if (h->pipe_begun != h->pipe_ended) why = "a dfb_filter_to_host_begin is outstanding";
    if (why) return fail(DFB_ERR_STATE, std::string("dfb_set_filter_shape: ") + why);
    return guarded([&] {
        if (shape == h->plan.filter_shape) return;
        Plan P = h->plan;
        P.filter_shape = shape;
        build_coef_table(P);
        const StepPlan S = plan_for_device(*h, P);        // refusals (DFB_Y_MODE / DFB_Z_MODE against the shape) throw here
        CUDA_TRY(cudaSetDevice(h->device));
        Sweeps sw = build_sweeps(*h, P, S);               // beside the old sweeps: a failure leaves the handle as it was
        CUDA_TRY(cudaStreamSynchronize(h->stream));       // the new tables are uploaded, and nothing reads the old ones any more
        CUDA_TRY(cudaStreamSynchronize(h->side));
        install_sweeps(*h, std::move(sw));
        h->plan = std::move(P);
        h->fingerprint = rst::fingerprint(h->plan);
    });
}

int dfb_set_flux_correction(dfb_handle h, int mode) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    if (mode != DFB_FLUX_OFF && mode != DFB_FLUX_MASS && mode != DFB_FLUX_VOLUME)
        return fail(DFB_ERR_ARG, "unknown flux correction mode " + std::to_string(mode) + " (DFB_FLUX_OFF = 0, DFB_FLUX_MASS = 1, DFB_FLUX_VOLUME = 2)");
    if (h->attached) return fail(DFB_ERR_STATE, attached_msg("dfb_set_flux_correction") + ": set the mode before attaching");
    return guarded([&] {
        refuse_outstanding(*h, "dfb_set_flux_correction");
        if (mode == DFB_FLUX_OFF) { h->flux_mode = DFB_FLUX_OFF; return; }
        FluxTables T = flux_tables(h->plan, mode);          // refusals (slab, R11 = 0 everywhere) throw before anything changes
        install_flux(*h, std::move(T));
        h->flux_mode = mode;
    });
}

int dfb_set_profiles(dfb_handle h, const double* cells) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    if (h->attached) return fail(DFB_ERR_STATE, attached_msg("dfb_set_profiles") + ": set the profiles before attaching");
    if (h->comm)
        return fail(DFB_ERR_STATE, "dfb_set_profiles: the handle has a communicator (dfb_comm_init): the gathered plane is rebuilt with the row tables");
    return guarded([&] {
        refuse_outstanding(*h, "dfb_set_profiles");
        Plan P = h->plan;
        std::vector<double> pc;
        if (cells) {
            pc = profile_consts(P, cells);                  // refusals (DFB_ERR_ARG) throw before anything changes
            P.cells = std::make_shared<const std::vector<double>>(profile_columns(P, cells));
            P.cells_hash = rst::hash_f64(cells, (size_t)8 * P.Ny * P.NzG);
        } else {
            P.cells.reset();
            P.cells_hash = 0;
        }
        FluxTables T;
        if (h->flux_mode != DFB_FLUX_OFF) T = flux_tables(P, h->flux_mode);
        CUDA_TRY(cudaSetDevice(h->device));
        if (cells) {
            if (!h->prof_dev) {
                CUDA_TRY(profiles_prepare());
                h->prof_dev = h->dalloc<double>(pc.size(), false);
            }
            // steps enqueued before read the previous table on this stream
            CUDA_TRY(cudaMemcpyAsync(h->prof_dev, pc.data(), pc.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream));
            CUDA_TRY(cudaStreamSynchronize(h->stream));
        }
        h->plan = std::move(P);
        if (h->flux_mode != DFB_FLUX_OFF) install_flux(*h, std::move(T));
        h->fingerprint = rst::fingerprint(h->plan);
    });
}

int dfb_flux_info(dfb_handle h, int plane, double out[3]) {
    if (!h || !out) return fail(DFB_ERR_ARG, "handle/out is NULL");
    if (plane < 0 || plane >= h->nplanes) return fail(DFB_ERR_ARG, "plane out of range");
    if (!h->fx.out) return fail(DFB_ERR_STATE, "the flux correction was never enabled (dfb_set_flux_correction)");
    return guarded([&] {
        sync_record(*h);
        CUDA_TRY(cudaSetDevice(h->device));
        double2 r;
        CUDA_TRY(cudaMemcpyAsync(&r, h->fx.out + plane, sizeof(r), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        out[0] = r.x; out[1] = r.y; out[2] = h->flux_tab.mean;
    });
}

static int set_noise_impl(dfb_handle h, int field, const double* r_ys, const double* left, const double* right, size_t halo_pitch) {
    if (!h || !r_ys || field < 0 || field > 2) return fail(DFB_ERR_ARG, "bad argument");
    if (h->noise_mode != DFB_NOISE_INJECT) return fail(DFB_ERR_STATE, "handle was not created with noise_mode = DFB_NOISE_INJECT");
    if (h->nplanes != 1) return fail(DFB_ERR_STATE, "noise injection is defined for single-plane handles");
    if (h->plan.periodic && (left || right)) return fail(DFB_ERR_ARG, "periodic_z: the noise is r_ys alone, the r_zs halo must be NULL");
    return guarded([&] {
        CUDA_TRY(cudaSetDevice(h->device));
        const FieldDev& F = h->D[h->step & 1].f[field];      // the set the next step reads
        const int W = h->D[0].W, M = F.Nz_max;
        // the plane part sits at extended column -xk0 (0 unless periodic_z); a periodic plane's wrapped columns come from the same array
        CUDA_TRY(cudaMemcpy2DAsync(F.r_ys - F.xk0, (size_t)F.pitch_y * 8, r_ys, (size_t)W * 8, (size_t)W * 8, (size_t)F.rows_y,
                                   cudaMemcpyHostToDevice, h->stream));
        if (h->plan.periodic) {
            if (M > 0) {
                CUDA_TRY(cudaMemcpy2DAsync(F.r_ys, (size_t)F.pitch_y * 8, r_ys + (W - M), (size_t)W * 8, (size_t)M * 8, (size_t)F.rows_y,
                                           cudaMemcpyHostToDevice, h->stream));
                CUDA_TRY(cudaMemcpy2DAsync(F.r_ys + M + W, (size_t)F.pitch_y * 8, r_ys, (size_t)W * 8, (size_t)M * 8, (size_t)F.rows_y,
                                           cudaMemcpyHostToDevice, h->stream));
            }
        } else if (M > 0) {
            if (!left || !right) throw Error{DFB_ERR_ARG, "halo noise missing"};
            CUDA_TRY(cudaMemcpy2DAsync(F.r_zs + F.zoff, (size_t)F.pitch_z * 8, left, halo_pitch, (size_t)M * 8, (size_t)h->D[0].Ny,
                                       cudaMemcpyHostToDevice, h->stream));
            CUDA_TRY(cudaMemcpy2DAsync(F.r_zs + F.zoff + W + M, (size_t)F.pitch_z * 8, right, halo_pitch, (size_t)M * 8,
                                       (size_t)h->D[0].Ny, cudaMemcpyHostToDevice, h->stream));
        }
        CUDA_TRY(cudaStreamSynchronize(h->stream));   // the caller may reuse its buffers
        h->injected[field] = true;
    });
}

int dfb_set_noise(dfb_handle h, int field, const double* r_ys, const double* r_zs_halo) {
    if (!h || field < 0 || field > 2) return fail(DFB_ERR_ARG, "bad argument");
    const int M = h->D[0].f[field].Nz_max;
    return set_noise_impl(h, field, r_ys, r_zs_halo, r_zs_halo ? r_zs_halo + M : nullptr, (size_t)2 * M * 8);
}

int dfb_set_noise_ref_layout(dfb_handle h, int field, const double* r_ys, const double* r_zs) {
    if (!h || field < 0 || field > 2) return fail(DFB_ERR_ARG, "bad argument");
    const int M = h->D[0].f[field].Nz_max, W = h->D[0].W;
    if (h->plan.periodic) r_zs = nullptr;                  // periodic_z: nothing of r_zs is noise
    return set_noise_impl(h, field, r_ys, r_zs, r_zs ? r_zs + W + M : nullptr, (size_t)(W + 2 * M) * 8);
}

int dfb_get_noise(dfb_handle h, int field, double* r_ys, double* r_zs_halo) {
    if (!h || field < 0 || field > 2) return fail(DFB_ERR_ARG, "bad argument");
    if (h->plan.k0 != 0 || h->plan.k1 != h->plan.NzG) return fail(DFB_ERR_STATE, "dfb_get_noise is defined on whole-plane handles");
    if (h->plan.periodic && r_zs_halo) return fail(DFB_ERR_ARG, "periodic_z: there is no r_zs halo noise, r_zs_halo must be NULL");
    return guarded([&] {
        sync_record(*h);
        CUDA_TRY(cudaSetDevice(h->device));
        const FieldDev& F = h->D[h->noise_view].f[field];
        const int W = h->D[0].W, M = F.Nz_max;
        if (r_ys)
            CUDA_TRY(cudaMemcpy2DAsync(r_ys, (size_t)W * 8, F.r_ys - F.xk0, (size_t)F.pitch_y * 8, (size_t)W * 8, (size_t)F.rows_y,
                                       cudaMemcpyDeviceToHost, h->stream));
        if (r_zs_halo && M > 0) {
            CUDA_TRY(cudaMemcpy2DAsync(r_zs_halo, (size_t)2 * M * 8, F.r_zs + F.zoff, (size_t)F.pitch_z * 8, (size_t)M * 8,
                                       (size_t)h->D[0].Ny, cudaMemcpyDeviceToHost, h->stream));
            CUDA_TRY(cudaMemcpy2DAsync(r_zs_halo + M, (size_t)2 * M * 8, F.r_zs + F.zoff + W + M, (size_t)F.pitch_z * 8, (size_t)M * 8,
                                       (size_t)h->D[0].Ny, cudaMemcpyDeviceToHost, h->stream));
        }
        CUDA_TRY(cudaStreamSynchronize(h->stream));
    });
}

int dfb_generate_noise(dfb_handle h, int64_t step) {
    if (!h || step < 0) return fail(DFB_ERR_ARG, "bad argument");
    return guarded([&] {
        refuse_attached(*h, "dfb_generate_noise");
        CUDA_TRY(cudaSetDevice(h->device));
        const int b = (int)(step & 1);
        CUDA_TRY(cudaStreamWaitEvent(h->stream, h->ev_noise[b], 0));   // order after any prefetch into that set
        launch_noise_for(*h, step, b, h->stream);
        h->noise_view = b;
    });
}

int dfb_get_state(dfb_handle h, double* filt_old3, int64_t* step) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    return guarded([&] {
        sync_record(*h);
        CUDA_TRY(cudaSetDevice(h->device));
        const size_t n = h->D[0].ps_cells * h->nplanes;                 // [3][P][Ny*Nz]
        if (filt_old3)
            for (int f = 0; f < 3; ++f)
                CUDA_TRY(cudaMemcpyAsync(filt_old3 + f * n, h->D[0].f[f].filt_old, n * 8, cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        if (step) *step = h->step;
    });
}

int dfb_set_state(dfb_handle h, const double* filt_old3, int64_t step) {
    if (!h || step < 0) return fail(DFB_ERR_ARG, "bad argument");
    return guarded([&] {
        sync_record(*h);
        restore_state(*h, filt_old3, step);
        if (h->attached) push_record(*h);
    });
}

int dfb_set_timing(dfb_handle h, int on) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    if (on && h->attached) return fail(DFB_ERR_STATE, attached_msg("dfb_set_timing(h, 1)"));
    h->timing = on != 0;
    return DFB_OK;
}

int dfb_last_ms(dfb_handle h, int stage, float* ms) {
    if (!h || !ms || stage < 0 || stage > 3) return fail(DFB_ERR_ARG, "bad argument");
    *ms = h->last_ms[stage];
    return DFB_OK;
}

int dfb_measure_fp64_peak(int device, double* tflops, double* sm_mhz_est) {
    if (!tflops) return fail(DFB_ERR_ARG, "tflops is NULL");
    return guarded([&] {
        if (device >= 0) CUDA_TRY(cudaSetDevice(device));
        int dev = 0;
        CUDA_TRY(cudaGetDevice(&dev));
        cudaDeviceProp prop;
        CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
        const int blocks = prop.multiProcessorCount * 8;
        double* d = nullptr;
        CUDA_TRY(cudaMalloc(&d, sizeof(double) * (size_t)blocks * 256));
        cudaEvent_t a, b;
        CUDA_TRY(cudaEventCreate(&a)); CUDA_TRY(cudaEventCreate(&b));
        const int iters = 4096;
        float best = 1e30f;
        for (int rep = 0; rep < 6; ++rep) {
            CUDA_TRY(cudaEventRecord(a, 0));
            CUDA_TRY(launch_dfma_peak(d, blocks, iters, 0));
            CUDA_TRY(cudaEventRecord(b, 0));
            CUDA_TRY(cudaEventSynchronize(b));
            float ms = 0;
            CUDA_TRY(cudaEventElapsedTime(&ms, a, b));
            if (rep >= 2) best = std::min(best, ms);
        }
        const double fma = (double)blocks * 256.0 * iters * 64.0;
        *tflops = 2.0 * fma / (best * 1e-3) / 1e12;
        if (sm_mhz_est) *sm_mhz_est = fma / (best * 1e-3) / (prop.multiProcessorCount * 64.0) / 1e6;   // if 64 DFMA/clk/SM
        cudaEventDestroy(a); cudaEventDestroy(b); cudaFree(d);
    });
}

int dfb_stats_enable(dfb_handle h, int on) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    if (h->attached) return fail(DFB_ERR_STATE, attached_msg("dfb_stats_enable") + ": set N2 on or off before attaching");
    return guarded([&] {
        CUDA_TRY(cudaSetDevice(h->device));
        const size_t n = h->D[0].ps_cells * h->nplanes;
        if (on && !h->stats) h->stats = h->dalloc<double>(6 * n);
        if (on) { CUDA_TRY(cudaMemsetAsync(h->stats, 0, 6 * n * sizeof(double), h->stream)); h->stats_count = 0; }
        h->stats_on = on != 0;             // off: keep what was accumulated, stop accumulating
    });
}

int dfb_stats_get_plane(dfb_handle h, int plane, int which, int as_rms, double* dst, int64_t* count) {
    if (!h || which < 0 || which > 5) return fail(DFB_ERR_ARG, "bad argument");
    if (plane < 0 || plane >= h->nplanes) return fail(DFB_ERR_ARG, "plane out of range");
    if (!h->stats) return fail(DFB_ERR_STATE, "statistics are not enabled (dfb_stats_enable)");
    return guarded([&] {
        sync_record(*h);
        CUDA_TRY(cudaSetDevice(h->device));
        const size_t n = h->D[0].ps_cells;
        if (dst) {
            CUDA_TRY(cudaMemcpyAsync(dst, h->stats + ((size_t)plane * 6 + which) * n, n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
            CUDA_TRY(cudaStreamSynchronize(h->stream));
            if (as_rms && h->stats_count > 0 && which < 5)
                for (size_t i = 0; i < n; ++i) dst[i] = std::sqrt(dst[i] / (double)h->stats_count);   // plot_rms, df.cpp:615-620
        }
        if (count) *count = h->stats_count;
    });
}
int dfb_stats_get(dfb_handle h, int which, int as_rms, double* dst, int64_t* count) { return dfb_stats_get_plane(h, 0, which, as_rms, dst, count); }

// ---- correlation statistics (dfb_corr_enable / dfb_corr_get / dfb_corr_integral_scales) ----
int dfb_corr_enable(dfb_handle h, int on, const int lags[3]) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    if (h->attached) return fail(DFB_ERR_STATE, attached_msg("dfb_corr_enable"));
    if (!on) {                                                // the sums stay readable; the ring and the scratch go
        h->corr_on = false;
        return guarded([&] {
            CUDA_TRY(cudaSetDevice(h->device));
            CUDA_TRY(cudaStreamSynchronize(h->stream));
            h->corr.ring = h->corr.part = nullptr;
            CUDA_TRY(h->corr_work.reset());
        });
    }
    if (!lags) return fail(DFB_ERR_ARG, "lags is NULL");
    const Plan& P = h->plan;
    if (P.k0 != 0 || P.k1 != P.NzG) return fail(DFB_ERR_ARG, "correlation statistics need the whole plane");
    int L[3];
    const int extent[2] = {P.NzG, P.Ny};
    const char* name[3] = {"z", "y", "t"};
    for (int d = 0; d < 3; ++d) {
        if (lags[d] == DFB_CORR_SUPPORT) {
            if (d == DFB_CORR_T) return fail(DFB_ERR_ARG, "lag of direction t must be 0..64: DFB_CORR_SUPPORT is not defined for t");
            int sup = 0;
            for (int f = 0; f < 3; ++f) sup = std::max(sup, 2 * (d == DFB_CORR_Z ? P.f[f].Nz_max : P.f[f].Ny_max));
            L[d] = std::min(sup, extent[d] - 1);
        } else {
            const int hi = d == DFB_CORR_T ? 64 : extent[d] - 1;
            if (lags[d] < 0 || lags[d] > hi)
                return fail(DFB_ERR_ARG, std::string("lag of direction ") + name[d] + " must be 0.." + std::to_string(hi) +
                                             (d == DFB_CORR_T ? "" : " or DFB_CORR_SUPPORT") + ", got " + std::to_string(lags[d]));
            L[d] = lags[d];
        }
    }
    return guarded([&] {
        CUDA_TRY(cudaSetDevice(h->device));
        CorrParams& c = h->corr;
        const int NP = h->nplanes, Ny = P.Ny, W = P.NzG;
        const size_t rows = (size_t)NP * 3 * Ny;
        if (!h->corr_ready || L[0] != c.L[0] || L[1] != c.L[1] || L[2] != c.L[2]) {
            CUDA_TRY(cudaStreamSynchronize(h->stream));
            h->corr_sums.reset();
            h->corr_work.reset();
            h->corr_ready = false;
            h->corr_on = false;
            c = CorrParams{};
            for (int f = 0; f < 3; ++f) c.fluc[f] = h->D[0].f[f].fluc;
            c.P = NP; c.Ny = Ny; c.W = W; c.periodic = P.periodic ? 1 : 0;
            for (int d = 0; d < 3; ++d) {
                c.L[d] = L[d];
                if (L[d]) c.sum[d] = h->corr_sums.alloc<double>(rows * (L[d] + 1));
            }
            c.y_nsplit = c.y_split_cols = 1;
            if (L[1]) corr_y_split(Ny, W, &c.y_nsplit, &c.y_split_cols);
        }
        // the ring and the partial-sum scratch exist only while accumulating (on = 0 frees them)
        const size_t part = corr_part_doubles(NP, Ny, W, c.L[0], c.L[1], c.y_nsplit);
        if (part && !c.part) c.part = h->corr_work.alloc<double>(part);
        if (c.L[2] && !c.ring) c.ring = h->corr_work.alloc<double>((size_t)c.L[2] * rows * W);
        for (int d = 0; d < 3; ++d)
            if (c.sum[d]) CUDA_TRY(cudaMemsetAsync(c.sum[d], 0, rows * (c.L[d] + 1) * sizeof(double), h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        c.ring_count = 0;
        h->corr_count = 0;
        h->corr_tsteps.assign(c.L[2] + 1, 0);
        h->corr_ready = true;
        h->corr_on = true;
    });
}

namespace {

// the sums of one (plane, field, direction) on the host, [Ny][L+1], and the products per row behind each lag
void corr_fetch(dfb_filter_s& H, int plane, int field, int dir, std::vector<double>& S, std::vector<int64_t>& pairs) {
    const CorrParams& c = H.corr;
    const int Ny = c.Ny, nlag = c.L[dir] + 1;
    S.assign((size_t)Ny * nlag, 0.0);
    CUDA_TRY(cudaSetDevice(H.device));
    CUDA_TRY(cudaMemcpyAsync(S.data(), c.sum[dir] + ((size_t)plane * 3 + field) * Ny * nlag, S.size() * sizeof(double), cudaMemcpyDeviceToHost,
                             H.stream));
    CUDA_TRY(cudaStreamSynchronize(H.stream));
    pairs.assign(nlag, 0);
    for (int d = 0; d < nlag; ++d)
        pairs[d] = dir == DFB_CORR_Z ? H.corr_count * (c.periodic ? c.W : c.W - d)
                 : dir == DFB_CORR_Y ? H.corr_count * c.W
                                     : H.corr_tsteps[d] * c.W;
}

// correlation coefficients from the sums, in place
void corr_normalize(const CorrParams& c, int dir, std::vector<double>& S, const std::vector<int64_t>& pairs) {
    const int Ny = c.Ny, nlag = c.L[dir] + 1;
    const double nan = std::numeric_limits<double>::quiet_NaN();
    std::vector<double> var(Ny);
    for (int j = 0; j < Ny; ++j) var[j] = S[(size_t)j * nlag];
    for (int j = 0; j < Ny; ++j)
        for (int d = 0; d < nlag; ++d) {
            double& r = S[(size_t)j * nlag + d];
            if (dir == DFB_CORR_Y)
                r = (j + d >= Ny || var[j] == 0.0 || var[j + d] == 0.0) ? nan : r / std::sqrt(var[j] * var[j + d]);
            else
                r = (pairs[d] == 0 || pairs[0] == 0 || var[j] == 0.0) ? nan : (r / (double)pairs[d]) / (var[j] / (double)pairs[0]);
        }
}

int corr_check(dfb_handle h, int plane, int field, int dir) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    if (!h->corr_ready) return fail(DFB_ERR_STATE, "correlation statistics are not enabled (dfb_corr_enable)");
    if (plane < 0 || plane >= h->nplanes) return fail(DFB_ERR_ARG, "plane out of range");
    if (field < 0 || field > 2) return fail(DFB_ERR_ARG, "field must be 0..2 (u', v', w')");
    if (dir < 0 || dir > 2) return fail(DFB_ERR_ARG, "direction must be DFB_CORR_Z, DFB_CORR_Y or DFB_CORR_T");
    if (h->corr.L[dir] == 0) return fail(DFB_ERR_ARG, "that direction was enabled with lag 0 (off)");
    return DFB_OK;
}

}  // namespace

int dfb_corr_get_plane(dfb_handle h, int plane, int field, int dir, int normalized, double* dst, int64_t* pairs, int64_t* count) {
    const int rc = corr_check(h, plane, field, dir);
    if (rc != DFB_OK) return rc;
    return guarded([&] {
        std::vector<double> S;
        std::vector<int64_t> pr;
        corr_fetch(*h, plane, field, dir, S, pr);
        if (normalized) corr_normalize(h->corr, dir, S, pr);
        if (dst) std::memcpy(dst, S.data(), S.size() * sizeof(double));
        if (pairs) std::memcpy(pairs, pr.data(), pr.size() * sizeof(int64_t));
        if (count) *count = h->corr_count;
    });
}
int dfb_corr_get(dfb_handle h, int field, int dir, int normalized, double* dst, int64_t* pairs, int64_t* count) {
    return dfb_corr_get_plane(h, 0, field, dir, normalized, dst, pairs, count);
}

int dfb_corr_integral_scales(dfb_handle h, int plane, int field, int dir, double* dst) {
    const int rc = corr_check(h, plane, field, dir);
    if (rc != DFB_OK) return rc;
    if (!dst) return fail(DFB_ERR_ARG, "dst is NULL");
    return guarded([&] {
        std::vector<double> R;
        std::vector<int64_t> pr;
        corr_fetch(*h, plane, field, dir, R, pr);
        corr_normalize(h->corr, dir, R, pr);
        const Plan& P = h->plan;
        const int Ny = P.Ny, nlag = h->corr.L[dir] + 1;
        const double wbar = (P.vert_z[P.NzG] - P.vert_z[0]) / P.NzG;
        for (int j = 0; j < Ny; ++j) {
            const double* r = R.data() + (size_t)j * nlag;
            auto x = [&](int d) { return dir == DFB_CORR_Z ? d * wbar : dir == DFB_CORR_Y ? P.yc_row[j + d] - P.yc_row[j] : (double)d; };
            if (!(r[0] > 0.0)) { dst[j] = std::numeric_limits<double>::quiet_NaN(); continue; }
            double acc = 0.0;
            for (int d = 1; d < nlag && r[d] > 0.0; ++d) acc += 0.5 * (r[d - 1] + r[d]) * (x(d) - x(d - 1));
            dst[j] = acc;
        }
    });
}

// ---- restart files (restart.hpp: format, records and file I/O; here: what moves between the device and the file) ----
namespace {

int check_restart_call(dfb_handle h, const char* path, int& what) {
    if (!h || !path) return fail(DFB_ERR_ARG, "handle/path is NULL");
    if (what & ~(DFB_RESTART_STATE | DFB_RESTART_STATS | DFB_RESTART_CORR)) return fail(DFB_ERR_ARG, "what must be a combination of DFB_RESTART_STATE, _STATS and _CORR");
    what |= DFB_RESTART_STATE;
    if (const int rc = guarded([&] { refuse_outstanding(*h, nullptr); }); rc != DFB_OK) return rc;
    const Plan& P = h->plan;
    if ((what & DFB_RESTART_CORR) && (P.k0 != 0 || P.k1 != P.NzG)) return fail(DFB_ERR_ARG, "correlation statistics need the whole plane");
    return DFB_OK;
}

// The handle's sections as blocks of the file: host buffers in the device layout, [3][P][Ny][W], [P][6][Ny][W], [P][3][Ny][L_d+1] per
// direction, and n_ring ring fields [P][3][Ny][W] oldest first.  plane_ofs = this handle's first plane within the file.
struct RestartBuffers {
    std::vector<double> state, stats, sum[3], ring;
    std::vector<rst::Block> blocks;
};

void restart_buffers(const dfb_filter_s& H, const rst::Header& hd, int what, int plane_ofs, RestartBuffers& B) {
    const int NP = H.nplanes, Ny = H.plan.Ny, W = H.plan.Nz(), k0 = H.plan.k0;
    const size_t n = H.D[0].ps_cells;
    B.state.assign(3 * NP * n, 0.0);
    for (int f = 0; f < 3; ++f)
        for (int p = 0; p < NP; ++p) B.blocks.push_back({rst::SEC_STATE, f, p + plane_ofs, B.state.data() + ((size_t)f * NP + p) * n, Ny, W, k0});
    if (what & DFB_RESTART_STATS) {
        B.stats.assign(6 * NP * n, 0.0);
        for (int p = 0; p < NP; ++p)
            for (int s = 0; s < 6; ++s) B.blocks.push_back({rst::SEC_STATS, s, p + plane_ofs, B.stats.data() + ((size_t)p * 6 + s) * n, Ny, W, k0});
    }
    if (what & DFB_RESTART_CORR) {
        for (int d = 0; d < 3; ++d) {
            const int nl = hd.corr_L[d] + 1;
            if (!hd.corr_L[d]) continue;
            B.sum[d].assign((size_t)NP * 3 * Ny * nl, 0.0);
            for (int p = 0; p < NP; ++p)
                for (int f = 0; f < 3; ++f)
                    B.blocks.push_back({rst::SEC_CORR_Z + d, f, p + plane_ofs, B.sum[d].data() + ((size_t)p * 3 + f) * Ny * nl, Ny, nl, 0});
        }
        B.ring.assign((size_t)hd.n_ring * NP * 3 * n, 0.0);
        for (int i = 0; i < hd.n_ring; ++i)
            for (int p = 0; p < NP; ++p)
                for (int f = 0; f < 3; ++f)
                    B.blocks.push_back({rst::SEC_RING, i * 3 + f, p + plane_ofs, B.ring.data() + (((size_t)i * NP + p) * 3 + f) * n, Ny, W, 0});
    }
}

}  // namespace

int dfb_save_restart(dfb_handle h, const char* path, int what) {
    int rc = check_restart_call(h, path, what);
    if (rc != DFB_OK) return rc;
    if ((what & DFB_RESTART_STATS) && !h->stats) return fail(DFB_ERR_STATE, "DFB_RESTART_STATS: statistics were never enabled (dfb_stats_enable)");
    if ((what & DFB_RESTART_CORR) && !h->corr_ready) return fail(DFB_ERR_STATE, "DFB_RESTART_CORR: correlation statistics were never enabled (dfb_corr_enable)");
    return guarded([&] {
        sync_record(*h);
        const Plan& P = h->plan;
        const CorrParams& c = h->corr;
        rst::Header hd;
        hd.lib_version = dfb_version();
        hd.Ny = P.Ny; hd.NzG = P.NzG; hd.plane0 = h->plane_id; hd.nplanes = h->nplanes; hd.periodic = P.periodic ? 1 : 0;
        hd.noise_mode = h->noise_mode; hd.seed = h->seed; hd.step = h->step;
        for (int f = 0; f < 3; ++f) { hd.Ny_max[f] = P.f[f].Ny_max; hd.Nz_max[f] = P.f[f].Nz_max; hd.Lt[f] = P.f[f].Lt; }
        const std::array<int, 3> forms = h->sw.forms();
        std::copy(forms.begin(), forms.end(), hd.forms);
        hd.fingerprint = h->fingerprint;
        hd.filter_shape = P.filter_shape;
        hd.profiles = P.cells_hash;
        hd.sections = (uint32_t)what;
        if (what & DFB_RESTART_STATS) { hd.stats_count = h->stats_count; hd.stats_on = h->stats_on ? 1 : 0; }
        if (what & DFB_RESTART_CORR) {
            for (int d = 0; d < 3; ++d) hd.corr_L[d] = c.L[d];
            hd.corr_on = h->corr_on ? 1 : 0;
            hd.n_ring = (h->corr_on && c.ring) ? (int)std::min<long long>(c.L[2], c.ring_count) : 0;
            hd.corr_count = h->corr_count;
            for (int m = 0; m <= c.L[2]; ++m) hd.corr_tsteps[m] = h->corr_tsteps[m];
        }
        rst::layout(hd);
        RestartBuffers B;
        restart_buffers(*h, hd, what, 0, B);
        CUDA_TRY(cudaSetDevice(h->device));
        const size_t n = h->D[0].ps_cells * h->nplanes;
        for (int f = 0; f < 3; ++f)
            CUDA_TRY(cudaMemcpyAsync(B.state.data() + f * n, h->D[0].f[f].filt_old, n * 8, cudaMemcpyDeviceToHost, h->stream));
        if (what & DFB_RESTART_STATS) CUDA_TRY(cudaMemcpyAsync(B.stats.data(), h->stats, 6 * n * 8, cudaMemcpyDeviceToHost, h->stream));
        if (what & DFB_RESTART_CORR) {
            for (int d = 0; d < 3; ++d)
                if (c.L[d]) CUDA_TRY(cudaMemcpyAsync(B.sum[d].data(), c.sum[d], B.sum[d].size() * 8, cudaMemcpyDeviceToHost, h->stream));
            for (int i = 0; i < hd.n_ring; ++i) {                    // oldest first: slot (ring_count - n_ring + i) mod L_t
                const long long slot = (c.ring_count - hd.n_ring + i) % c.L[2];
                CUDA_TRY(cudaMemcpyAsync(B.ring.data() + (size_t)i * 3 * n, c.ring + (size_t)slot * 3 * n, 3 * n * 8, cudaMemcpyDeviceToHost, h->stream));
            }
        }
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        rst::save(path, hd, rst::Record{h->plane_id, h->nplanes, P.k0, P.k1, h->step, h->fingerprint}, B.blocks);
    });
}

int dfb_load_restart(dfb_handle h, const char* path, int what) {
    int rc = check_restart_call(h, path, what);
    if (rc != DFB_OK) return rc;
    return guarded([&] {
        sync_record(*h);
        // ---- everything is checked and read before the device is touched: a refused load leaves the handle as it was ----
        std::vector<rst::Record> recs;
        const rst::Header hd = rst::read_header(path, &recs);
        const Plan& P = h->plan;
        const int NP = h->nplanes;
        auto arg = [](const std::string& m) { return Error{DFB_ERR_ARG, m}; };
        if (hd.Ny != P.Ny || hd.NzG != P.NzG)
            throw arg("geometry differs: file Ny x Nz = " + std::to_string(hd.Ny) + " x " + std::to_string(hd.NzG) + ", handle " +
                      std::to_string(P.Ny) + " x " + std::to_string(P.NzG));
        if (hd.periodic != (P.periodic ? 1 : 0))
            throw arg("periodic_z differs: file " + std::to_string(hd.periodic) + ", handle " + std::to_string(P.periodic ? 1 : 0));
        if (hd.filter_shape != P.filter_shape) {
            static const char* const shape_name[2] = {"exponential", "Gaussian"};
            throw arg(std::string("filter shape differs: file ") + shape_name[hd.filter_shape] + ", handle " + shape_name[P.filter_shape] +
                      " (dfb_set_filter_shape)");
        }
        if (hd.profiles != P.cells_hash)
            throw arg(!P.cells_hash ? "the file was saved with per-cell profiles (dfb_set_profiles), the handle has none"
                      : !hd.profiles ? "the handle has per-cell profiles (dfb_set_profiles), the file was saved without them"
                                     : "the per-cell profiles (dfb_set_profiles) differ from the file's");
        if (hd.fingerprint != h->fingerprint) throw arg("the filter tables differ (half-widths, row tables or time scales)");
        if (h->noise_mode == DFB_NOISE_GENERATE && hd.seed != h->seed)
            throw arg("seed differs: file " + std::to_string(hd.seed) + ", handle " + std::to_string(h->seed));
        if (h->plane_id < hd.plane0 || h->plane_id + NP > hd.plane0 + hd.nplanes)
            throw arg("planes [" + std::to_string(h->plane_id) + ", " + std::to_string(h->plane_id + NP) + ") of this handle are not in the file's planes [" +
                      std::to_string(hd.plane0) + ", " + std::to_string(hd.plane0 + hd.nplanes) + ")");
        if ((what & DFB_RESTART_STATS) && !(hd.sections & DFB_RESTART_STATS)) throw arg("the file has no N2 statistics (saved without DFB_RESTART_STATS)");
        if ((what & DFB_RESTART_CORR) && !(hd.sections & DFB_RESTART_CORR)) throw arg("the file has no correlation statistics (saved without DFB_RESTART_CORR)");
        const std::string gap = rst::check_coverage(hd, recs, h->plane_id, h->plane_id + NP, P.k0, P.k1);
        if (!gap.empty()) throw Error{DFB_ERR_IO, std::string(path) + ": " + gap};
        RestartBuffers B;
        restart_buffers(*h, hd, what, h->plane_id - hd.plane0, B);
        rst::read_blocks(path, hd, B.blocks);

        // ---- the device ----
        restore_state(*h, B.state.data(), hd.step);
        const size_t n = h->D[0].ps_cells * NP;
        if (what & DFB_RESTART_STATS) {
            if (!h->stats) h->stats = h->dalloc<double>(6 * n, false);
            CUDA_TRY(cudaMemcpyAsync(h->stats, B.stats.data(), 6 * n * 8, cudaMemcpyHostToDevice, h->stream));
            h->stats_count = hd.stats_count;
            h->stats_on = hd.stats_on != 0;
        }
        if (what & DFB_RESTART_CORR) {
            if (dfb_corr_enable(h, 1, hd.corr_L) != DFB_OK) throw Error{DFB_ERR_CUDA, g_last_error};   // allocates, zeroes, empties the ring
            CorrParams& c = h->corr;
            for (int d = 0; d < 3; ++d)
                if (c.L[d]) CUDA_TRY(cudaMemcpyAsync(c.sum[d], B.sum[d].data(), B.sum[d].size() * 8, cudaMemcpyHostToDevice, h->stream));
            if (hd.n_ring) CUDA_TRY(cudaMemcpyAsync(c.ring, B.ring.data(), B.ring.size() * 8, cudaMemcpyHostToDevice, h->stream));   // slots 0..n_ring-1
            c.ring_count = hd.n_ring;
            h->corr_count = hd.corr_count;
            for (int m = 0; m <= c.L[2]; ++m) h->corr_tsteps[m] = hd.corr_tsteps[m];
            if (!hd.corr_on && dfb_corr_enable(h, 0, nullptr) != DFB_OK) throw Error{DFB_ERR_CUDA, g_last_error};
        }
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        if (h->attached) push_record(*h);
    });
}

int dfb_restart_info(const char* path, int64_t* out, int cap) {
    if (!path || cap < 0 || (cap > 0 && !out)) return fail(DFB_ERR_ARG, "bad argument");
    return guarded([&] {
        std::vector<rst::Record> recs;
        const rst::Header hd = rst::read_header(path, &recs);
        const std::vector<int64_t> v = rst::info_values(hd, (int)recs.size());
        std::copy(v.begin(), v.begin() + std::min<size_t>(v.size(), (size_t)cap), out);
    });
}

// write_csv (df.cpp:764-803), opt-in: header, fixed notation with 15 decimals, one row per cell
int dfb_write_csv(dfb_handle h, const char* path) {
    if (!h || !path) return fail(DFB_ERR_ARG, "bad argument");
    return guarded([&] {
        CUDA_TRY(cudaSetDevice(h->device));
        const int Ny = h->D[0].Ny, W = h->D[0].W;
        const size_t n = (size_t)Ny * W;
        std::vector<double> buf(5 * n);
        for (int i = 0; i < 5; ++i)
            CUDA_TRY(cudaMemcpyAsync(buf.data() + (size_t)i * n, field_ptr(*h, i), n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        FILE* fp = std::fopen(path, "w");
        if (!fp) throw Error{DFB_ERR_IO, std::string("Error: cannot open ") + path + " for writing. (df.cpp:766-769)"};
        std::fputs("z,y,u_fluc,v_fluc,w_fluc,T_fluc,rho_fluc\n", fp);
        for (int j = 0; j < Ny; ++j)
            for (int k = 0; k < W; ++k) {
                const size_t c = (size_t)j * W + k;
                std::fprintf(fp, "%.15f,%.15f,%.15f,%.15f,%.15f,%.15f,%.15f\n", h->plan.csv_zc[h->plan.k0 + k], h->plan.csv_yc[j],
                             buf[c], buf[n + c], buf[2 * n + c], buf[3 * n + c], buf[4 * n + c]);
            }
        std::fclose(fp);
    });
}

// write_tecplot (df.cpp:712-762), opt-in.  `file << double << endl` with the stream's default formatting == "%g\n".
int dfb_write_tecplot(dfb_handle h, const char* path) {
    if (!h || !path) return fail(DFB_ERR_ARG, "bad argument");
    return guarded([&] {
        CUDA_TRY(cudaSetDevice(h->device));
        const int Ny = h->D[0].Ny, W = h->D[0].W, k0 = h->plan.k0;
        const size_t n = (size_t)Ny * W;
        std::vector<double> buf(3 * n);
        for (int i = 0; i < 3; ++i)
            CUDA_TRY(cudaMemcpyAsync(buf.data() + (size_t)i * n, field_ptr(*h, i), n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        FILE* fp = std::fopen(path, "w");
        if (!fp) throw Error{DFB_ERR_IO, std::string("cannot open ") + path + " for writing"};
        std::fputs("VARIABLES = \"z\", \"y\", \"u_fluc\", \"v_fluc\", \"w_fluc\" \n", fp);                 // df.cpp:715
        std::fprintf(fp, "ZONE T=\"Flow Field\", I=%d, J=%d, F=BLOCK\n", W + 1, Ny + 1);                  // df.cpp:716
        std::fputs("VARLOCATION=([3-5]=CELLCENTERED)\n", fp);                                             // df.cpp:717
        for (int j = 0; j < Ny + 1; ++j) for (int k = 0; k < W + 1; ++k) std::fprintf(fp, "%g\n", h->plan.vert_z[k0 + k]);   // df.cpp:721-726
        for (int j = 0; j < Ny + 1; ++j) for (int k = 0; k < W + 1; ++k) std::fprintf(fp, "%g\n", h->plan.vert_y[j]);        // df.cpp:729-734
        for (int f = 0; f < 3; ++f)                                                                        // df.cpp:737-758
            for (size_t c = 0; c < n; ++c) std::fprintf(fp, "%g\n", buf[(size_t)f * n + c]);
        std::fclose(fp);
    });
}

// get_rms (df.cpp:584-611): reset the sums, `nsteps` steps with accumulation (on the device, in the z-sweep's epilogue)
int dfb_get_rms(dfb_handle h, int nsteps, double dt) {
    if (!h || nsteps < 0) return fail(DFB_ERR_ARG, "bad argument");
    if (h->attached) return fail(DFB_ERR_STATE, attached_msg("dfb_get_rms"));
    int rc = guarded([&] { check_dt(dt); });         // before dfb_stats_enable zeroes the sums
    if (rc != DFB_OK) return rc;
    rc = dfb_stats_enable(h, 1);
    if (rc != DFB_OK) return rc;
    return guarded([&] {
        for (int i = 0; i < nsteps; ++i) run_step(*h, dt, false);
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        h->stats_on = false;                 // the sums stay readable; later dfb_filter calls do not add to them
    });
}

// plot_rms (df.cpp:613-675)
int dfb_write_rms_csv(dfb_handle h, const char* path) {
    if (!h || !path) return fail(DFB_ERR_ARG, "bad argument");
    if (!h->stats) return fail(DFB_ERR_STATE, "statistics are not enabled (dfb_stats_enable / dfb_get_rms)");
    return guarded([&] {
        sync_record(*h);
        CUDA_TRY(cudaSetDevice(h->device));
        const int Ny = h->D[0].Ny, W = h->D[0].W, k0 = h->plan.k0;
        const size_t n = (size_t)Ny * W;
        std::vector<double> buf(5 * n);
        CUDA_TRY(cudaMemcpyAsync(buf.data(), h->stats, 5 * n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        const double cnt = (double)std::max<int64_t>(h->stats_count, 1);
        for (double& v : buf) v = std::sqrt(v / cnt);                                                      // df.cpp:615-621
        FILE* fp = std::fopen(path, "w");
        if (!fp) throw Error{DFB_ERR_IO, std::string("cannot open ") + path + " for writing"};
        std::fputs("z, y, u'_rms, v'_rms, w'_rms, T'_rms, rho'_rms \n", fp);                               // df.cpp:630
        for (int j = 0; j < Ny; ++j)
            for (int k = 0; k < W; ++k) {
                const size_t c = (size_t)j * W + k;
                std::fprintf(fp, "%g, %g, %g, %g, %g, %g, %g\n", h->plan.vert_z[k0 + k], h->plan.vert_y[j],           // df.cpp:633-639
                             buf[c], buf[n + c], buf[2 * n + c], buf[3 * n + c], buf[4 * n + c]);
            }
        std::fclose(fp);
    });
}

// N3: which cell of this handle's slab contains each face centre (us3d_user.f90:85-114 runs over faces; the map is built once)
int dfb_face_map(dfb_handle h, int n, const double* yf, const double* zf, int* plane_index) {
    if (!h || n < 0 || (n > 0 && (!yf || !zf || !plane_index))) return fail(DFB_ERR_ARG, "bad argument");
    const Plan& P = h->plan;
    const std::vector<double>& vy = P.vert_y;
    const std::vector<double>& vz = P.vert_z;
    const int Ny = P.Ny, NzG = P.NzG, W = P.Nz();
    for (int i = 0; i < n; ++i) {
        // cell j with vy[j] <= y < vy[j+1], clamped to the plane
        int j = (int)(std::upper_bound(vy.begin(), vy.end(), yf[i]) - vy.begin()) - 1;
        int k = (int)(std::upper_bound(vz.begin(), vz.end(), zf[i]) - vz.begin()) - 1;
        j = std::min(std::max(j, 0), Ny - 1);
        k = std::min(std::max(k, 0), NzG - 1);
        plane_index[i] = (k >= P.k0 && k < P.k1) ? j * W + (k - P.k0) : -1;
    }
    return DFB_OK;
}

}  // extern "C" (reopened below the face maps' helpers)

// ---- face maps: the taps are built on the host (facemap.cpp), summed on the device (interp_kernel) ----
namespace {

FaceMapDev& facemap_of(dfb_filter_s& H, int map_id) {
    if (map_id < 0 || map_id >= (int)H.facemaps.size() || !H.facemaps[map_id])
        throw Error{DFB_ERR_ARG, "no face map " + std::to_string(map_id) + " on this handle"};
    return *H.facemaps[map_id];
}

// the checks and arguments dfb_interp_to_cells and dfb_interp_to_host share
InterpArgs interp_args(dfb_filter_s& H, const FaceMapDev& F, int plane, int fields) {
    if (plane < 0 || plane >= H.nplanes) throw Error{DFB_ERR_ARG, "plane out of range"};
    if (fields <= 0 || (fields & ~31)) throw Error{DFB_ERR_ARG, "fields must be a non-empty mask of the bits 1 << DFB_U_FLUC .. 1 << DFB_RHO_FLUC"};
    InterpArgs a{};
    for (int f = 0; f < 5; ++f) { a.field[f] = (fields >> f) & 1 ? field_ptr(H, f, plane) : nullptr; a.scale[f] = 1.0; }
    a.n = F.n; a.fields = fields; a.stride = 1;
    a.idx = F.idx; a.w = F.w; a.ptr = F.ptr;
    return a;
}

}  // namespace

extern "C" {

int dfb_facemap_create(dfb_handle h, int kind, int n, const double* yf, const double* zf, const double* hy, const double* hz, int own_begin,
                       int own_end, int flags, int* map_id) {
    if (!h || !map_id) return fail(DFB_ERR_ARG, "handle/map_id is NULL");
    return guarded([&] {
        refuse_outstanding(*h, nullptr);
        const FaceMap M = build_face_map(h->plan, kind, n, yf, zf, hy, hz, own_begin, own_end, flags);
        CUDA_TRY(cudaSetDevice(h->device));
        auto F = std::make_unique<FaceMapDev>();
        F->kind = kind; F->n = n; F->n_served = M.n_served; F->served = M.served;
        for (int i = 0; i < n; ++i)
            if (M.served[i]) F->faces.push_back(i);
        F->idx = F->mem.upload(M.idx, h->stream);
        F->w = F->mem.upload(M.w, h->stream);
        if (kind == DFB_MAP_AREA) F->ptr = F->mem.upload(M.ptr, h->stream);
        if (M.n_served < n) {
            std::vector<int> slot(n, -1);
            for (int r = 0; r < M.n_served; ++r) slot[F->faces[r]] = r;
            F->slot = F->mem.upload(slot, h->stream);
        }
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        int id = 0;
        while (id < (int)h->facemaps.size() && h->facemaps[id]) ++id;
        if (id == (int)h->facemaps.size()) h->facemaps.emplace_back();
        h->facemaps[id] = std::move(F);
        *map_id = id;
    });
}

int dfb_facemap_served(dfb_handle h, int map_id, int* served) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    return guarded([&] {
        const FaceMapDev& F = facemap_of(*h, map_id);
        if (F.n > 0 && !served) throw Error{DFB_ERR_ARG, "served is NULL"};
        std::copy(F.served.begin(), F.served.end(), served);
    });
}

int dfb_facemap_destroy(dfb_handle h, int map_id) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    return guarded([&] {
        facemap_of(*h, map_id);
        CUDA_TRY(cudaSetDevice(h->device));
        CUDA_TRY(cudaStreamSynchronize(h->stream));        // an enqueued dfb_interp_to_cells may still read the taps
        h->facemaps[map_id].reset();
    });
}

int dfb_interp_to_cells(dfb_handle h, int map_id, int plane, int fields, const int* dst_index, const double* const mean[5],
                        const double scale[5], double* const dst[5], int stride) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    return guarded([&] {
        refuse_outstanding(*h, nullptr);
        const FaceMapDev& F = facemap_of(*h, map_id);
        InterpArgs a = interp_args(*h, F, plane, fields);
        if (stride < 1) throw Error{DFB_ERR_ARG, "stride must be >= 1"};
        if (F.n > 0 && !dst) throw Error{DFB_ERR_ARG, "dst is NULL"};
        for (int f = 0; f < 5; ++f) {
            if (!((fields >> f) & 1)) continue;
            if (F.n > 0 && !dst[f]) throw Error{DFB_ERR_ARG, "dst[" + std::to_string(f) + "] is NULL for a requested field"};
            a.dst[f] = F.n > 0 ? dst[f] : nullptr;
            a.mean[f] = mean ? mean[f] : nullptr;
            if (!a.mean[f]) a.add |= 1 << f;                    // dst's own value is the base
            if (scale) a.scale[f] = scale[f];
        }
        a.dst_index = dst_index;
        a.stride = stride;
        CUDA_TRY(cudaSetDevice(h->device));
        CUDA_TRY(launch_interp(a, h->stream));
    });
}

int dfb_interp_to_host(dfb_handle h, int map_id, int plane, int fields, double* out) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    return guarded([&] {
        refuse_outstanding(*h, nullptr);
        sync_record(*h);
        FaceMapDev& F = facemap_of(*h, map_id);
        InterpArgs a = interp_args(*h, F, plane, fields);
        if (F.n > 0 && !out) throw Error{DFB_ERR_ARG, "out is NULL"};
        CUDA_TRY(cudaSetDevice(h->device));
        const size_t ns = (size_t)F.n_served;
        if (!F.stage) F.stage = F.mem.alloc<double>(5 * ns);
        int nf = 0;
        for (int f = 0; f < 5; ++f)
            if ((fields >> f) & 1) a.dst[f] = F.stage + ns * nf++;
        a.dst_index = F.slot;
        CUDA_TRY(launch_interp(a, h->stream));
        if (ns == (size_t)F.n) {                                 // every face served: the staged rows are out's rows
            if (ns) CUDA_TRY(cudaMemcpyAsync(out, F.stage, nf * ns * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
            CUDA_TRY(cudaStreamSynchronize(h->stream));
        } else {                                                 // only the served faces' entries of out change
            std::vector<double> buf(nf * ns);
            if (ns) CUDA_TRY(cudaMemcpyAsync(buf.data(), F.stage, nf * ns * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
            CUDA_TRY(cudaStreamSynchronize(h->stream));
            for (int r = 0; r < nf; ++r)
                for (size_t s = 0; s < ns; ++s) out[(size_t)r * F.n + F.faces[s]] = buf[r * ns + s];
        }
    });
}

int dfb_debug_yprof(dfb_handle h, unsigned long long* out8) {
    if (!h || !out8) return fail(DFB_ERR_ARG, "bad argument");
    return guarded([&] {
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        if (!h->sw.y[0].prof) throw Error{DFB_ERR_STATE, "no profile buffer"};
        CUDA_TRY(cudaMemcpy(out8, h->sw.y[0].prof, 64, cudaMemcpyDeviceToHost));
        CUDA_TRY(cudaMemset(h->sw.y[0].prof, 0, 64));
    });
}

int dfb_debug_timeline(dfb_handle h, unsigned long long* out512) {
    // development aid: DFB_TIMELINE=1 at create; returns and clears 64 step slots x {noise, y, z, -} x {start, end} (ns)
    if (!h || !out512) return fail(DFB_ERR_ARG, "bad argument");
    return guarded([&] {
        if (!h->sw.tl) throw Error{DFB_ERR_STATE, "DFB_TIMELINE was not set when the handle was created"};
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->side));
        CUDA_TRY(cudaMemcpy(out512, h->sw.tl, 512 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        timeline_reset(h->sw.tl);
    });
}

int dfb_debug_zprof(dfb_handle h, unsigned long long* out8) {
    if (!h || !out8) return fail(DFB_ERR_ARG, "bad argument");
    return guarded([&] {
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        if (!h->sw.z[0].prof) throw Error{DFB_ERR_STATE, "no profile buffer"};
        CUDA_TRY(cudaMemcpy(out8, h->sw.z[0].prof, 1024, cudaMemcpyDeviceToHost));     // 128 counters
        CUDA_TRY(cudaMemset(h->sw.z[0].prof, 0, 1024));
    });
}

}  // extern "C" (the comm section below reopens it)

// =================================================================================================
// BASELINE config 4 -- one plane in spanwise slabs over the ranks of a job; NCCL only for the hand-off of the finished
// plane to the CFD rank (SURVEY 8e; README.md:55 "MPI support to distribute result"; us3d_user.f90:85-92).
// =================================================================================================
namespace {

// NCCL is a link-time dependency of libdfb200.so (libnccl.so.2: the system copy, or the one a host framework such as PyTorch
// has already loaded under the same soname)
struct NcclApi {
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = ncclGetUniqueId;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = ncclCommInitRank;
    ncclResult_t (*CommDestroy)(ncclComm_t) = ncclCommDestroy;
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = ncclSend;
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = ncclRecv;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = ncclAllGather;
    ncclResult_t (*GroupStart)() = ncclGroupStart;
    ncclResult_t (*GroupEnd)() = ncclGroupEnd;
    const char* (*GetErrorString)(ncclResult_t) = ncclGetErrorString;
};

NcclApi& nccl() {
    static NcclApi api;
    return api;
}

#define NCCL_TRY(expr)                                                                                   \
    do {                                                                                                 \
        ncclResult_t r__ = (expr);                                                                       \
        if (r__ != ncclSuccess) throw Error{DFB_ERR_CUDA, std::string(#expr) + ": " + nccl().GetErrorString(r__)};   \
    } while (0)

}  // namespace

void dfb_filter_s::comm_release() {
    if (comm) { try { nccl().CommDestroy(comm); } catch (...) {} comm = nullptr; }
}


namespace {

// Peer-to-peer hand-off of one step (transport 2).  seq = number of this gather (the same on every rank: the call is collective).
//   destination: tells every sender "the plane is free for gather seq" (8-byte copy into the sender's flag block), assembles its own
//                slab, then per sender waits -- a stream memory operation, no SM involved -- for "slab of gather seq landed" and
//                rebuilds T', rho' of that slab's columns from the u' that just arrived;
//   sender:      waits for "plane free", lets its copy engine write u', v', w' of its slab straight into the plane's final row-major
//                layout over NVLink (three strided 2-D copies: 24 bytes per cell on the wire, no SM, no staging on the far side),
//                then raises "slab landed" on the destination.
void gather_p2p(dfb_filter_s& H, int dst_rank, int first_only) {
    const int Ny = H.plan.Ny, NzG = H.plan.NzG, world = H.comm_world, me = H.comm_rank;
    const size_t n = H.D[0].ps_cells, np = (size_t)Ny * NzG;
    const int W = H.D[0].W, k0 = H.plan.k0;
    const bool dst = me == dst_rank;
    // (re)map the destination's plane: collective, only when the destination changes
    if (H.peer_plane_of != dst_rank) {
        struct Rec { cudaIpcMemHandle_t hd; int ok; int pad[3]; };
        Rec mine{};
        if (dst) mine.ok = cudaIpcGetMemHandle(&mine.hd, H.g_plane) == cudaSuccess ? 1 : 0;
        Rec* dr = reinterpret_cast<Rec*>(H.dalloc<unsigned char>(sizeof(Rec) * (size_t)(world + 1), false));
        CUDA_TRY(cudaMemcpyAsync(dr, &mine, sizeof(Rec), cudaMemcpyHostToDevice, H.comm_stream));
        NCCL_TRY(nccl().AllGather(dr, dr + 1, sizeof(Rec), ncclUint8, H.comm, H.comm_stream));
        std::vector<Rec> recs((size_t)world);
        CUDA_TRY(cudaMemcpyAsync(recs.data(), dr + 1, sizeof(Rec) * (size_t)world, cudaMemcpyDeviceToHost, H.comm_stream));
        CUDA_TRY(cudaStreamSynchronize(H.comm_stream));
        if (!recs[dst_rank].ok) throw Error{DFB_ERR_CUDA, "the destination rank could not export its plane through CUDA IPC"};
        if (H.peer_plane) { cudaIpcCloseMemHandle(H.peer_plane); H.peer_plane = nullptr; }
        if (!dst) {
            void* p = nullptr;
            CUDA_TRY(cudaIpcOpenMemHandle(&p, recs[dst_rank].hd, cudaIpcMemLazyEnablePeerAccess));
            H.peer_plane = static_cast<double*>(p);
        }
        H.peer_plane_of = dst_rank;
    }
    const unsigned long long seq = ++H.g_seq;
    unsigned long long* src = H.seq_ring + (seq % 64);      // pinned: the 8-byte flag copies below are truly asynchronous
    *src = seq;
    if (dst) {
        for (int r = 0; r < world; ++r)
            if (r != me) CUDA_TRY(cudaMemcpyAsync(H.peer_flags[r] + 32, src, 8, cudaMemcpyHostToDevice, H.asm_stream));   // "plane free for seq"
        // own slab: staged in g_recv (see dfb_gather_begin) -> plane, with T', rho'
        CUDA_TRY(launch_assemble(H.g_recv + H.g_recv_off[me], H.g_plane, H.D[0].rowc, Ny, NzG, k0, W, first_only, H.comm_stream));
        for (int r = 0; r < world; ++r) {
            if (r == me) continue;
            CUresult cr = stream_wait_value64()(H.comm_stream, (CUdeviceptr)(uintptr_t)(H.flags + r), seq, CU_STREAM_WAIT_VALUE_GEQ);
            if (cr != CUDA_SUCCESS) throw Error{DFB_ERR_CUDA, "cuStreamWaitValue64 failed (" + std::to_string((int)cr) + ")"};
            const int rk0 = H.comm_bounds[2 * r], rW = H.comm_bounds[2 * r + 1] - rk0;
            CUDA_TRY(launch_rebuild(H.g_plane, H.D[0].rowc, Ny, NzG, rk0, rW, first_only, H.comm_stream));
            H.g_bytes_wire += (int64_t)3 * Ny * rW * 8;
        }
    } else {
        CUresult cr = stream_wait_value64()(H.comm_stream, (CUdeviceptr)(uintptr_t)(H.flags + 32), seq, CU_STREAM_WAIT_VALUE_GEQ);
        if (cr != CUDA_SUCCESS) throw Error{DFB_ERR_CUDA, "cuStreamWaitValue64 failed (" + std::to_string((int)cr) + ")"};
        for (int f = 0; f < 3; ++f)
            CUDA_TRY(cudaMemcpy2DAsync(H.peer_plane + (size_t)f * np + k0, (size_t)NzG * 8, H.g_send + (size_t)f * n, (size_t)W * 8, (size_t)W * 8, (size_t)Ny,
                                       cudaMemcpyDeviceToDevice, H.comm_stream));
        CUDA_TRY(cudaMemcpyAsync(H.peer_flags[dst_rank] + me, src, 8, cudaMemcpyHostToDevice, H.comm_stream));             // "slab of rank me landed"
        H.g_bytes_wire = (int64_t)3 * n * 8;
    }
}

}  // namespace

extern "C" {

int dfb_comm_unique_id(void* id128) {
    if (!id128) return fail(DFB_ERR_ARG, "id128 is NULL");
    static_assert(sizeof(ncclUniqueId) == DFB_COMM_ID_BYTES, "ncclUniqueId is 128 bytes");
    return guarded([&] { NCCL_TRY(nccl().GetUniqueId(static_cast<ncclUniqueId*>(id128))); });
}

int dfb_comm_init(dfb_handle h, const void* id128, int rank, int world) {
    if (!h || !id128 || world < 1 || rank < 0 || rank >= world) return fail(DFB_ERR_ARG, "bad argument");
    if (h->comm) return fail(DFB_ERR_STATE, "dfb_comm_init was already called on this handle");
    if (h->attached) return fail(DFB_ERR_STATE, attached_msg("dfb_comm_init"));
    if (h->nplanes != 1) return fail(DFB_ERR_STATE, "slab communication is defined for single-plane handles");
    if (h->plan.cells)
        return fail(DFB_ERR_STATE, "dfb_comm_init: the handle has per-cell profiles (dfb_set_profiles): the gathered plane is rebuilt with the row tables");
    return guarded([&] {
        CUDA_TRY(cudaSetDevice(h->device));
        ncclUniqueId id;
        std::memcpy(&id, id128, sizeof(id));
        NCCL_TRY(nccl().CommInitRank(&h->comm, world, id, rank));
        h->comm_rank = rank; h->comm_world = world;
        if (world > 16) throw Error{DFB_ERR_ARG, "at most 16 ranks per plane"};
        // the transfer / assembly streams get the highest priority: their (small) kernels go first whenever an SM has room
        {
            int prio_lo = 0, prio_hi = 0;
            CUDA_TRY(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
            CUDA_TRY(cudaStreamCreateWithPriority(&h->comm_stream, cudaStreamNonBlocking, prio_hi));
            CUDA_TRY(cudaStreamCreateWithPriority(&h->asm_stream, cudaStreamNonBlocking, prio_hi));
            for (int r = 0; r < world; ++r) CUDA_TRY(cudaEventCreateWithFlags(&h->ev_slab[r], cudaEventDisableTiming));
        }
        CUDA_TRY(cudaEventCreateWithFlags(&h->ev_gstaged, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&h->ev_gdone, cudaEventDisableTiming));
        // every rank learns every rank's slab: one all-gather of (k_begin, k_end, Ny, Nz_global)
        int mine[4] = {h->plan.k0, h->plan.k1, h->plan.Ny, h->plan.NzG};
        int* d = h->dalloc<int>((size_t)4 * (world + 1), false);        // filled on comm_stream: no zeroing on the compute stream
        CUDA_TRY(cudaMemcpyAsync(d, mine, sizeof(mine), cudaMemcpyHostToDevice, h->comm_stream));
        NCCL_TRY(nccl().AllGather(d, d + 4, 4, ncclInt32, h->comm, h->comm_stream));
        std::vector<int> all((size_t)4 * world);
        CUDA_TRY(cudaMemcpyAsync(all.data(), d + 4, all.size() * sizeof(int), cudaMemcpyDeviceToHost, h->comm_stream));
        CUDA_TRY(cudaStreamSynchronize(h->comm_stream));
        h->comm_bounds.resize((size_t)2 * world);
        for (int r = 0; r < world; ++r) {
            if (all[4 * r + 2] != h->plan.Ny || all[4 * r + 3] != h->plan.NzG)
                throw Error{DFB_ERR_ARG, "the ranks of a slab job must describe the same plane (Ny, Nz differ on rank " + std::to_string(r) + ")"};
            h->comm_bounds[2 * r] = all[4 * r]; h->comm_bounds[2 * r + 1] = all[4 * r + 1];
        }
        for (int r = 0; r + 1 < world; ++r)
            if (h->comm_bounds[2 * r + 1] != h->comm_bounds[2 * r + 2])
                throw Error{DFB_ERR_ARG, "slabs must tile the plane in rank order (rank r's k_end = rank r+1's k_begin)"};
        if (h->comm_bounds[0] != 0 || h->comm_bounds[2 * world - 1] != h->plan.NzG)
            throw Error{DFB_ERR_ARG, "slabs must cover [0, Nz)"};
        h->g_send = h->dalloc<double>((size_t)3 * h->D[0].ps_cells, false);

        // ---- peer-to-peer transport: every rank exports a flag block through CUDA IPC; all ranks must succeed, else NCCL send/recv ----
        h->transport = 1;
        const char* tr = std::getenv("DFB_GATHER_TRANSPORT");
        if (world > 1 && !(tr && std::strcmp(tr, "nccl") == 0)) {
            struct Rec { cudaIpcMemHandle_t hd; int ok; int pad[3]; };
            static_assert(sizeof(Rec) % 8 == 0, "");
            Rec mine{};
            h->flags = h->dalloc<unsigned long long>(64);
            CUDA_TRY(cudaStreamSynchronize(h->stream));
            mine.ok = cudaIpcGetMemHandle(&mine.hd, h->flags) == cudaSuccess ? 1 : 0;
            if (mine.ok && cudaHostAlloc(reinterpret_cast<void**>(&h->seq_ring), 64 * sizeof(unsigned long long), cudaHostAllocPortable) != cudaSuccess) mine.ok = 0;
            cudaGetLastError();
            Rec* dr = reinterpret_cast<Rec*>(h->dalloc<unsigned char>(sizeof(Rec) * (size_t)(world + 1), false));
            CUDA_TRY(cudaMemcpyAsync(dr, &mine, sizeof(Rec), cudaMemcpyHostToDevice, h->comm_stream));
            NCCL_TRY(nccl().AllGather(dr, dr + 1, sizeof(Rec), ncclUint8, h->comm, h->comm_stream));
            std::vector<Rec> recs((size_t)world);
            CUDA_TRY(cudaMemcpyAsync(recs.data(), dr + 1, sizeof(Rec) * (size_t)world, cudaMemcpyDeviceToHost, h->comm_stream));
            CUDA_TRY(cudaStreamSynchronize(h->comm_stream));
            int ok = 1;
            for (int r = 0; r < world; ++r) ok &= recs[r].ok;
            for (int r = 0; ok && r < world; ++r) {
                if (r == rank) continue;
                void* p = nullptr;
                if (cudaIpcOpenMemHandle(&p, recs[r].hd, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { ok = 0; cudaGetLastError(); break; }
                h->peer_flags[r] = static_cast<unsigned long long*>(p);
            }
            // second round: did every rank manage to map every other rank?
            int* dok = h->dalloc<int>((size_t)world + 1, false);
            CUDA_TRY(cudaMemcpyAsync(dok, &ok, sizeof(int), cudaMemcpyHostToDevice, h->comm_stream));
            NCCL_TRY(nccl().AllGather(dok, dok + 1, 1, ncclInt32, h->comm, h->comm_stream));
            std::vector<int> oks((size_t)world);
            CUDA_TRY(cudaMemcpyAsync(oks.data(), dok + 1, sizeof(int) * (size_t)world, cudaMemcpyDeviceToHost, h->comm_stream));
            CUDA_TRY(cudaStreamSynchronize(h->comm_stream));
            for (int v : oks) ok &= v;
            if (ok) { h->transport = 2; (void)stream_wait_value64(); }
        }
        // The sweeps are persistent kernels that fill every SM (and all of its shared memory): an NCCL transfer kernel launched beside
        // them only starts at their kernel boundaries.  With the NCCL transport the persistent grids therefore leave a few SMs free
        // (DFB_COMM_SMS, default 8 of 148); the peer-to-peer transport moves the data with the copy engines and needs none.
        {
            cudaDeviceProp prop;
            CUDA_TRY(cudaGetDeviceProperties(&prop, h->device));
            const int reserve = std::getenv("DFB_COMM_SMS") ? std::atoi(std::getenv("DFB_COMM_SMS")) : (h->transport == 2 ? 0 : 8);
            const int sms = std::max(1, prop.multiProcessorCount - std::max(0, reserve));
            if (world > 1 && h->sw.tuned)
                for (int b = 0; b < 2; ++b) {
                    if (h->sw.y[b].r_grid > sms) h->sw.y[b].r_grid = sms;
                    const int per_sm = std::max(1, h->sw.z[b].nblocks / prop.multiProcessorCount);
                    if (h->sw.z[b].nblocks > per_sm * sms) h->sw.z[b].nblocks = per_sm * sms;
                }
            reset_run_queues(*h, h->sw);
        }
    });
}

int dfb_comm_info(dfb_handle h, int* rank, int* world, int* bounds) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    if (!h->comm) return fail(DFB_ERR_STATE, "dfb_comm_init has not been called");
    if (rank) *rank = h->comm_rank;
    if (world) *world = h->comm_world;
    if (bounds) std::memcpy(bounds, h->comm_bounds.data(), h->comm_bounds.size() * sizeof(int));
    return DFB_OK;
}

int dfb_gather_begin(dfb_handle h, int dst_rank) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    if (!h->comm) return fail(DFB_ERR_STATE, "dfb_comm_init has not been called");
    if (dst_rank < 0 || dst_rank >= h->comm_world) return fail(DFB_ERR_ARG, "dst_rank out of range");
    if (h->attached) return fail(DFB_ERR_STATE, attached_msg("dfb_gather_begin"));
    if (h->g_begun != h->g_ended) return fail(DFB_ERR_STATE, "a gather is already outstanding: call dfb_gather_end first");
    return guarded([&] {
        CUDA_TRY(cudaSetDevice(h->device));
        const int Ny = h->plan.Ny, NzG = h->plan.NzG, world = h->comm_world;
        const size_t n = h->D[0].ps_cells;
        const bool dst = h->comm_rank == dst_rank;
        if (dst && (!h->g_plane || h->g_dst != dst_rank)) {
            if (!h->g_plane) {
                h->g_plane = h->dalloc<double>((size_t)5 * Ny * NzG, false);
                h->g_recv = h->dalloc<double>((size_t)3 * Ny * NzG, false);
                h->g_recv_off.assign(world + 1, 0);
                for (int r = 0; r < world; ++r)
                    h->g_recv_off[r + 1] = h->g_recv_off[r] + (size_t)3 * Ny * (h->comm_bounds[2 * r + 1] - h->comm_bounds[2 * r]);
            }
        }
        h->g_dst = dst_rank;
        h->g_after_first_only = h->step <= 1;
        // stage u', v', w' of the step just enqueued (device to device, on the compute stream: the next step may overwrite the
        // fields as soon as this copy is done); the wire carries these 24 bytes per cell -- T', rho' are row-wise multiples of u'
        // (df.cpp:470-485) and are rebuilt on the destination
        double* stage = dst ? h->g_recv + h->g_recv_off[h->comm_rank] : h->g_send;
        CUDA_TRY(cudaStreamWaitEvent(h->stream, h->ev_gdone, 0));        // the previous gather has shipped / assembled the staging buffer
        for (int f = 0; f < 3; ++f)
            CUDA_TRY(cudaMemcpyAsync(stage + (size_t)f * n, field_ptr(*h, f), n * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
        CUDA_TRY(cudaEventRecord(h->ev_gstaged, h->stream));
        CUDA_TRY(cudaStreamWaitEvent(h->comm_stream, h->ev_gstaged, 0));
        h->g_bytes_wire = 0;
        const int first_only = h->g_after_first_only ? 1 : 0;
        if (h->transport == 2 && world > 1) {
            gather_p2p(*h, dst_rank, first_only);
        } else if (dst) {
            // [rank][3][Ny][W_rank] -> row-major planes u', v', w' + T', rho' rebuilt with the row constants (bitwise what the slabs
            // hold).  The slabs are received one after the other (each sender alone fills this GPU's NVLink ingress) and assembled
            // on a second stream as they land: the assembly of rank r runs under the transfer of rank r+1.
            auto assemble = [&](int r) {
                CUDA_TRY(cudaEventRecord(h->ev_slab[r], h->comm_stream));
                CUDA_TRY(cudaStreamWaitEvent(h->asm_stream, h->ev_slab[r], 0));
                CUDA_TRY(launch_assemble(h->g_recv + h->g_recv_off[r], h->g_plane, h->D[0].rowc, Ny, NzG, h->comm_bounds[2 * r],
                                         h->comm_bounds[2 * r + 1] - h->comm_bounds[2 * r], first_only, h->asm_stream));
            };
            assemble(h->comm_rank);                                        // this rank's own slab: staged above
            for (int r = 0; r < world; ++r) {
                if (r == dst_rank) continue;
                const size_t cnt = h->g_recv_off[r + 1] - h->g_recv_off[r];
                NCCL_TRY(nccl().Recv(h->g_recv + h->g_recv_off[r], cnt, ncclDouble, r, h->comm, h->comm_stream));
                h->g_bytes_wire += (int64_t)cnt * 8;
                assemble(r);
            }
            CUDA_TRY(cudaEventRecord(h->ev_slab[dst_rank], h->asm_stream));    // everything assembled
            CUDA_TRY(cudaStreamWaitEvent(h->comm_stream, h->ev_slab[dst_rank], 0));
        } else {
            NCCL_TRY(nccl().Send(h->g_send, 3 * n, ncclDouble, dst_rank, h->comm, h->comm_stream));
            h->g_bytes_wire = (int64_t)3 * n * 8;
        }
        CUDA_TRY(cudaEventRecord(h->ev_gdone, h->comm_stream));
        h->g_begun += 1;
    });
}

int dfb_gather_end(dfb_handle h) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    if (!h->comm) return fail(DFB_ERR_STATE, "dfb_comm_init has not been called");
    if (h->g_begun == h->g_ended) return fail(DFB_ERR_STATE, "no dfb_gather_begin is outstanding");
    if (h->attached) return fail(DFB_ERR_STATE, attached_msg("dfb_gather_end"));
    return guarded([&] {
        CUDA_TRY(cudaSetDevice(h->device));
        // bounded wait: a rank that died would otherwise leave this one blocked for ever on a flag that never comes
        const double limit = std::getenv("DFB_GATHER_TIMEOUT_S") ? std::atof(std::getenv("DFB_GATHER_TIMEOUT_S")) : 120.0;
        const auto t0 = std::chrono::steady_clock::now();
        for (;;) {
            cudaError_t q = cudaEventQuery(h->ev_gdone);
            if (q == cudaSuccess) break;
            if (q != cudaErrorNotReady) CUDA_TRY(q);
            if (std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() > limit)
                throw Error{DFB_ERR_STATE, "dfb_gather_end: the hand-off did not complete within the time limit (a rank of the job is missing?)"};
            std::this_thread::yield();
        }
        h->g_ended += 1;
    });
}

int dfb_gathered_ptr(dfb_handle h, int which, void** ptr) {
    if (!h || !ptr || which < 0 || which > 4) return fail(DFB_ERR_ARG, "bad argument");
    if (!h->g_plane) return fail(DFB_ERR_STATE, "this rank has not been the destination of a gather");
    *ptr = h->g_plane + (size_t)which * h->plan.Ny * h->plan.NzG;
    return DFB_OK;
}

int dfb_gathered_to_host(dfb_handle h, int which, double* dst) {
    if (!h || !dst || which < 0 || which > 4) return fail(DFB_ERR_ARG, "bad argument");
    if (!h->g_plane) return fail(DFB_ERR_STATE, "this rank has not been the destination of a gather");
    if (h->g_begun != h->g_ended) return fail(DFB_ERR_STATE, "a gather is outstanding: call dfb_gather_end first");
    return guarded([&] {
        CUDA_TRY(cudaSetDevice(h->device));
        const size_t n = (size_t)h->plan.Ny * h->plan.NzG;
        CUDA_TRY(cudaMemcpyAsync(dst, h->g_plane + (size_t)which * n, n * sizeof(double), cudaMemcpyDeviceToHost, h->comm_stream));
        CUDA_TRY(cudaStreamSynchronize(h->comm_stream));
    });
}

int dfb_comm_stream(dfb_handle h, void** stream) {
    if (!h || !stream) return fail(DFB_ERR_ARG, "bad argument");
    if (!h->comm) return fail(DFB_ERR_STATE, "dfb_comm_init has not been called");
    *stream = h->comm_stream;
    return DFB_OK;
}

int dfb_gather_wire_bytes(dfb_handle h, int64_t* bytes) {
    if (!h || !bytes) return fail(DFB_ERR_ARG, "bad argument");
    *bytes = h->g_bytes_wire;
    return DFB_OK;
}

int dfb_comm_destroy(dfb_handle h) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
    return guarded([&] {
        if (h->comm_stream) CUDA_TRY(cudaStreamSynchronize(h->comm_stream));
        h->comm_release();
        h->comm_rank = -1; h->comm_world = 0;
    });
}

}  // extern "C"

extern "C" {

const char* dfb_last_error(void) { return g_last_error.c_str(); }
const char* dfb_version(void) { return "dfb200 0.1 (sm_100a; rng spec v1)"; }

int dfb_create_f(const dfb_config* cfg, dfb_handle* out) { return dfb_create(cfg, out); }
int dfb_filter_f(const dfb_handle* h, const double* dt) { return (h && dt) ? dfb_filter(*h, *dt) : fail(DFB_ERR_ARG, "NULL argument"); }
int dfb_filter_to_host_f(const dfb_handle* h, const double* dt, double* u, double* v, double* w, double* T, double* rho) {
    return (h && dt) ? dfb_filter_to_host(*h, *dt, u, v, w, T, rho) : fail(DFB_ERR_ARG, "NULL argument");
}
int dfb_dims_f(const dfb_handle* h, int* Ny, int* Nz) { return h ? dfb_dims(*h, Ny, Nz) : fail(DFB_ERR_ARG, "NULL argument"); }
int dfb_create_batch_f(const dfb_config* cfg, const int* nplanes, dfb_handle* out) {
    return nplanes ? dfb_create_batch(cfg, *nplanes, out) : fail(DFB_ERR_ARG, "NULL argument");
}
int dfb_get_field_plane_f(const dfb_handle* h, const int* plane, const int* which, double* dst) {
    return (h && plane && which) ? dfb_get_field_plane(*h, *plane, *which, dst, 0) : fail(DFB_ERR_ARG, "NULL argument");
}
int dfb_comm_init_f(const dfb_handle* h, const void* id128, const int* rank, const int* world) {
    return (h && rank && world) ? dfb_comm_init(*h, id128, *rank, *world) : fail(DFB_ERR_ARG, "NULL argument");
}
int dfb_gather_begin_f(const dfb_handle* h, const int* dst_rank) { return (h && dst_rank) ? dfb_gather_begin(*h, *dst_rank) : fail(DFB_ERR_ARG, "NULL argument"); }
int dfb_gather_end_f(const dfb_handle* h) { return h ? dfb_gather_end(*h) : fail(DFB_ERR_ARG, "NULL argument"); }
int dfb_gathered_to_host_f(const dfb_handle* h, const int* which, double* dst) {
    return (h && which) ? dfb_gathered_to_host(*h, *which, dst) : fail(DFB_ERR_ARG, "NULL argument");
}
int dfb_face_map_f(const dfb_handle* h, const int* n, const double* yf, const double* zf, int* plane_index) {
    return (h && n) ? dfb_face_map(*h, *n, yf, zf, plane_index) : fail(DFB_ERR_ARG, "NULL argument");
}
static std::string fortran_path(const char* path, const int* len) { return (len && *len >= 0) ? std::string(path, (size_t)*len) : std::string(path); }
int dfb_save_restart_f(const dfb_handle* h, const char* path, const int* path_len, const int* what) {
    return (h && path && what) ? dfb_save_restart(*h, fortran_path(path, path_len).c_str(), *what) : fail(DFB_ERR_ARG, "NULL argument");
}
int dfb_load_restart_f(const dfb_handle* h, const char* path, const int* path_len, const int* what) {
    return (h && path && what) ? dfb_load_restart(*h, fortran_path(path, path_len).c_str(), *what) : fail(DFB_ERR_ARG, "NULL argument");
}
int dfb_facemap_create_f(const dfb_handle* h, const int* kind, const int* n, const double* yf, const double* zf, const double* hy,
                         const double* hz, const int* own_begin, const int* own_end, const int* flags, int* map_id) {
    return (h && kind && n && own_begin && own_end && flags)
               ? dfb_facemap_create(*h, *kind, *n, yf, zf, hy, hz, *own_begin, *own_end, *flags, map_id)
               : fail(DFB_ERR_ARG, "NULL argument");
}
int dfb_facemap_served_f(const dfb_handle* h, const int* map_id, int* served) {
    return (h && map_id) ? dfb_facemap_served(*h, *map_id, served) : fail(DFB_ERR_ARG, "NULL argument");
}
int dfb_facemap_destroy_f(const dfb_handle* h, const int* map_id) {
    return (h && map_id) ? dfb_facemap_destroy(*h, *map_id) : fail(DFB_ERR_ARG, "NULL argument");
}
int dfb_interp_to_host_f(const dfb_handle* h, const int* map_id, const int* plane, const int* fields, double* out) {
    return (h && map_id && plane && fields) ? dfb_interp_to_host(*h, *map_id, *plane, *fields, out) : fail(DFB_ERR_ARG, "NULL argument");
}
int dfb_interp_to_cells_f(const dfb_handle* h, const int* map_id, const int* plane, const int* fields, const int* dst_index,
                          const double* const mean[5], const double scale[5], double* const dst[5], const int* stride) {
    return (h && map_id && plane && fields && stride) ? dfb_interp_to_cells(*h, *map_id, *plane, *fields, dst_index, mean, scale, dst, *stride)
                                                      : fail(DFB_ERR_ARG, "NULL argument");
}
int dfb_attach_stream_f(const dfb_handle* h, void* const* stream) {
    return (h && stream) ? dfb_attach_stream(*h, *stream) : fail(DFB_ERR_ARG, "NULL argument");
}
int dfb_filter_dev_f(const dfb_handle* h, const double* const* dt_dev) {
    return (h && dt_dev) ? dfb_filter_dev(*h, *dt_dev) : fail(DFB_ERR_ARG, "NULL argument");
}
int dfb_set_time_scales_f(const dfb_handle* h, const double* const* Lt_rows) {
    return (h && Lt_rows) ? dfb_set_time_scales(*h, *Lt_rows) : fail(DFB_ERR_ARG, "NULL argument");
}
int dfb_time_scales_from_lengths_f(const dfb_handle* h, const double* Ix, const double* u_min, double* Lt_rows) {
    return (h && u_min) ? dfb_time_scales_from_lengths(*h, Ix, *u_min, Lt_rows) : fail(DFB_ERR_ARG, "NULL argument");
}
int dfb_set_filter_shape_f(const dfb_handle* h, const int* shape) {
    return (h && shape) ? dfb_set_filter_shape(*h, *shape) : fail(DFB_ERR_ARG, "NULL argument");
}
int dfb_set_flux_correction_f(const dfb_handle* h, const int* mode) {
    return (h && mode) ? dfb_set_flux_correction(*h, *mode) : fail(DFB_ERR_ARG, "NULL argument");
}
int dfb_set_profiles_f(const dfb_handle* h, const double* const* cells) {
    return (h && cells) ? dfb_set_profiles(*h, *cells) : fail(DFB_ERR_ARG, "NULL argument");
}
int dfb_flux_info_f(const dfb_handle* h, const int* plane, double* out) {
    return (h && plane) ? dfb_flux_info(*h, *plane, out) : fail(DFB_ERR_ARG, "NULL argument");
}
int dfb_destroy_f(dfb_handle* h) {
    if (!h) return DFB_OK;
    int rc = dfb_destroy(*h);
    *h = nullptr;
    return rc;
}

}  // extern "C"
