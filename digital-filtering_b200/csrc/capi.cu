// csrc/capi.cu -- the C ABI declared in include/dfb200.h: handle lifetime, device layout, the step.
// Mirrors DIGITAL_FILTER's constructor (df.cpp:4-66) and filter(dt) (df.cpp:449-468).
// There is no CPU fallback: without an sm_100 device dfb_create fails with DFB_ERR_CUDA.
#include <algorithm>
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

inline int round_up(int v, int m) { return (v + m - 1) / m * m; }

struct NoiseHost {            // one logical array of the noise contract
    int field, kind;
    uint64_t inc, state0, npairs;
    int n_seg;
    void *d_jump = nullptr, *d_off = nullptr, *d_np = nullptr, *d_win = nullptr;
};

}  // namespace

struct dfb_filter_s {
    Plan plan;
    int device = 0;
    int noise_mode = DFB_NOISE_GENERATE;
    int kernel_variant = 0;
    bool tuned = false;
    uint64_t seed = 0;
    int plane_id = 0;
    int nplanes = 1;                  // planes advanced together by this handle (dfb_create_batch): plane p draws from stream group plane_id + p
    int64_t step = 0;                 // steps completed (the constructor's first step counts as one)
    bool injected[3] = {false, false, false};
    cudaStream_t stream = nullptr;    // main stream (high priority): sweeps + epilogue
    cudaStream_t side = nullptr;      // low-priority stream: next step's noise, generated while this step filters
    cudaStream_t copy = nullptr;      // dfb_filter_to_host_begin/end: device-to-host copies of step t under the compute of step t+1
    double* stage[2] = {nullptr, nullptr};                 // staged copies of the five output fields
    cudaEvent_t ev_staged[2] = {nullptr, nullptr}, ev_copied[2] = {nullptr, nullptr};
    long long pipe_begun = 0, pipe_ended = 0;
    std::vector<void*> allocs;
    // Two noise buffer sets (r_ys, r_zs): step s uses set s&1, so noise(s+1) can be written while
    // y(s)/z(s) still read set s&1.  D[b] differs from D[1-b] only in the r_ys / r_zs pointers.
    PlaneDev D[2]{};
    bool overlap = true;
    int64_t buf_step[2] = {-1, -1};   // which step's noise set b currently holds (or -1)
    int64_t ybuf_step[2] = {-1, -1};  // which step's y-sweep result the r_zs interior of set b holds (or -1)
    bool y_ahead = false;             // optionally run the next step's y-sweep on the side stream too (measured: contention
                                      // with the z-sweep costs more than the filled tail gains; off by default)
    int noise_view = 0;               // set holding the most recently consumed / generated noise
    cudaEvent_t ev_noise[2] = {nullptr, nullptr};   // noise into set b complete (either stream)
    cudaEvent_t ev_free[2] = {nullptr, nullptr};    // last readers of set b complete (main stream)
    // tuned y-sweep
    YMaps maps[2]{};
    YParams yp[2]{};
    int n_items = 0;
    int n_tiles_dense = 0, n_tiles_rec = 0;   // y-sweep tiles: dense band-matrix tiles first, then recursive tiles
    YRMaps rmaps[2]{};                        // run-recursive y-sweep (the default form): tensor maps of r_ys with its box
    int y_form = 0;                           // 0 dense band matrices, 1 chunk-recursive (ysweep_rec_kernel), 2 run-recursive (ysweep_run_kernel)
    // tuned z-sweep
    ZParams zp[2]{};
    ZMaps zmaps[2]{};
    // noise
    std::vector<NoiseHost> noise;
    NoiseParams np{};
    NoiseWindows nwin{};              // periodic_z: segment windows of the r_ys arrays whose extended rows wrap (else all nullptr)
    unsigned long long* tl = nullptr; // development aid (DFB_TIMELINE): 64 steps x {noise, y, z} x {start, end}
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
    std::vector<void*> corr_mem;      // the sums: freed when the lags change and with the handle
                                      // (corr.ring and corr.part exist only while accumulating: corr_free_work)
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
    // timing
    bool timing = false;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    float last_ms[4] = {0, 0, 0, 0};

    void comm_release();              // ncclCommDestroy through the lazily loaded library (below)
    template <class T>
    T* dalloc(size_t n, bool zero = true) {
        void* p = nullptr;
        CUDA_TRY(cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T)));
        allocs.push_back(p);
        if (zero) CUDA_TRY(cudaMemsetAsync(p, 0, std::max<size_t>(n, 1) * sizeof(T), stream));
        return static_cast<T*>(p);
    }
    template <class T>
    T* upload(const std::vector<T>& v) {
        T* p = dalloc<T>(v.size(), false);
        if (!v.empty()) CUDA_TRY(cudaMemcpyAsync(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, stream));
        return p;
    }
    ~dfb_filter_s() {
        cudaSetDevice(device);
        if (side) cudaStreamSynchronize(side);
        if (stream) cudaStreamSynchronize(stream);
        for (void* p : allocs) cudaFree(p);
        for (void* p : corr_mem) cudaFree(p);
        cudaFree(corr.ring);
        cudaFree(corr.part);
        for (auto& e : ev) if (e) cudaEventDestroy(e);
        for (int b = 0; b < 2; ++b) { if (ev_noise[b]) cudaEventDestroy(ev_noise[b]); if (ev_free[b]) cudaEventDestroy(ev_free[b]); }
        for (int q = 0; q < 2; ++q) { if (ev_staged[q]) cudaEventDestroy(ev_staged[q]); if (ev_copied[q]) cudaEventDestroy(ev_copied[q]); }
        if (comm_stream) cudaStreamSynchronize(comm_stream);
        if (asm_stream) { cudaStreamSynchronize(asm_stream); cudaStreamDestroy(asm_stream); }
        for (auto& e : ev_slab) if (e) cudaEventDestroy(e);
        for (auto& pf : peer_flags) if (pf) cudaIpcCloseMemHandle(pf);
        if (peer_plane) cudaIpcCloseMemHandle(peer_plane);
        if (seq_ring) cudaFreeHost(seq_ring);
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

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        CUDA_TRY(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
        if (q != cudaDriverEntryPointSuccess || !p) throw Error{DFB_ERR_CUDA, "cuTensorMapEncodeTiled not available"};
        fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

typedef CUresult (*StreamWaitValue64Fn)(CUstream, CUdeviceptr, cuuint64_t, unsigned int);
StreamWaitValue64Fn stream_wait_value64() {
    static StreamWaitValue64Fn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        CUDA_TRY(cudaGetDriverEntryPoint("cuStreamWaitValue64", &p, cudaEnableDefault, &q));
        if (q != cudaDriverEntryPointSuccess || !p) throw Error{DFB_ERR_CUDA, "cuStreamWaitValue64 not available"};
        fn = reinterpret_cast<StreamWaitValue64Fn>(p);
    }
    return fn;
}

void timeline_reset(dfb_filter_s& H);

// Tile queues of the run-recursive y-sweep (one per buffer set: {next tile, producers done}): at rest they hold the size of the
// persistent grid -- CTA b starts on tile b, the kernel puts the value back when its last producer has finished.  Written here
// when the plan is built and again whenever the grid changes (dfb_comm_init leaving SMs free for NCCL); the stream is idle then.
void reset_run_queues(dfb_filter_s& H) {
    if (!H.yp[0].rcounter) return;
    CUDA_TRY(cudaStreamSynchronize(H.stream));
    if (H.side) CUDA_TRY(cudaStreamSynchronize(H.side));
    for (int b = 0; b < 2; ++b) {
        const int grid = (int)std::min<long long>((long long)H.yp[b].n_rtiles * H.nplanes, (long long)H.yp[b].r_grid);
        const int init[2] = {grid, 0};
        CUDA_TRY(cudaMemcpy(H.yp[b].rcounter, init, sizeof(init), cudaMemcpyHostToDevice));
    }
}

void build_device(dfb_filter_s& H) {
    const Plan& P = H.plan;
    PlaneDev& D = H.D[0];
    const int Ny = P.Ny, W = P.Nz(), NzG = P.NzG;
    D.Ny = Ny; D.W = W; D.NzG = NzG; D.k0 = P.k0;
    const int NP = H.nplanes;
    D.P = NP; D.ps_cells = (size_t)Ny * W;
    H.tuned = (H.kernel_variant == 0) && P.f[0].row_uniform && P.f[1].row_uniform && P.f[2].row_uniform;

    // ---- per-row epilogue constants, reference expressions (df.cpp:425-438, 474) ----
    std::vector<double> rowc((size_t)Ny * ROWC, 0.0);
    const double* R11 = P.rows.data(); const double* R21 = R11 + Ny; const double* R22 = R21 + Ny; const double* R33 = R22 + Ny;
    const double* Us = R33 + Ny; const double* Ts = Us + Ny; const double* rhos = Ts + Ny; const double* Ms = rhos + Ny;
    for (int j = 0; j < Ny; ++j) {
        double b = (R11[j] < 1e-10) ? 0.0 : R21[j] / std::sqrt(R11[j]);
        double* rc = &rowc[(size_t)j * ROWC];
        rc[0] = std::sqrt(R11[j]);
        rc[1] = b;
        rc[2] = std::sqrt(R22[j] - b * b);
        rc[3] = std::sqrt(R33[j]);
        rc[4] = -0.5 * (1.4 - 1) * Ms[j] * Ms[j] / Us[j];
        rc[5] = Ts[j];
        rc[6] = rhos[j];
    }
    D.rowc = H.upload(rowc);
    D.coef_ptr = H.upload(P.coef.ptr);
    D.coef_vals = H.upload(P.coef.vals);
    D.T_fluc = H.dalloc<double>((size_t)NP * Ny * W);
    D.rho_fluc = H.dalloc<double>((size_t)NP * Ny * W);

    int maxNz = 0;
    for (int f = 0; f < 3; ++f) {
        const FieldPlan& FP = P.f[f];
        FieldDev& F = D.f[f];
        F.Ny_max = FP.Ny_max; F.Nz_max = FP.Nz_max;
        maxNz = std::max(maxNz, FP.Nz_max);
        F.rows_y = Ny + 2 * FP.Ny_max;
        // periodic_z: the extended range is not clipped to the plane -- its columns beyond an edge are the plane's own columns,
        // wrapped (Nz_max <= NzG: at most once), y-filtered like the others, so that the z-sweep needs no change at all
        F.xk0 = P.periodic ? P.k0 - FP.Nz_max : std::max(0, P.k0 - FP.Nz_max);
        const int xk1 = P.periodic ? P.k1 + FP.Nz_max : std::min(NzG, P.k1 + FP.Nz_max);
        F.We = xk1 - F.xk0;
        F.pitch_y = round_up(F.We, 16);
        F.zoff = (16 - FP.Nz_max % 16) % 16;
        F.pitch_z = round_up(F.zoff + W + 2 * FP.Nz_max, 16) + 16;
        F.yshift = F.xk0 - P.k0 + FP.Nz_max;
        F.ps_ys = (size_t)F.rows_y * F.pitch_y;
        F.ps_zs = (size_t)Ny * F.pitch_z;
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

    // ---- tuned y-sweep: row groups, dense band matrices, work items, TMA maps ----
    if (H.tuned) {
        const int RC = ysweep_rc();
        std::vector<YGroup> groups;
        std::vector<YTile> tiles;
        std::vector<double> cmat;
        // ---- which rows go through the run-recursive form (ysweep_run_kernel), which through the band matrices ----
        // The run form evaluates a group of R rows (<= 8, or <= min(32, 0.33 N) for N >= 25) of ONE half-width N with 2(N+1) + 4R multiply-adds per column where the direct sum
        // spends R(2N+1): it pays in runs of equal N, not where N changes every row or two (a lone row costs its direct sum and
        // its window has to be staged whole).  Decided per block of 32 rows: run form where it executes less than half of the
        // direct sum's multiply-adds (and two of the block's windows fit in shared memory); the other rows keep the band matrices.
        // DFB_Y_MODE=2 forces the run form wherever a window fits at all, 0 / 1 force the band-matrix kernels (dense / chunk-recursive).
        const int ymode_env = std::getenv("DFB_Y_MODE") ? std::atoi(std::getenv("DFB_Y_MODE")) : -1;
        cudaDeviceProp yprop;
        CUDA_TRY(cudaGetDeviceProperties(&yprop, H.device));
        std::vector<char> run_row[3];
        std::vector<YRGroup> rg;
        std::vector<YRTile> rt;
        int r_wrows = 0, r_nbuf = 2;
        {
            constexpr int CB = 32;                                   // classification block
            std::vector<int> cheap[3];                               // band-matrix blocks whose rows are cheap in either form
            double band_cost = 0, all_cost = 0;                      // direct-sum multiply-adds per column: band-matrix blocks, all blocks
            bool band_convertible = true;                            // every band-matrix block could take the run form
            for (int f = 0; f < 3; ++f) {
                const std::vector<int>& Nr = P.f[f].N_y_row;
                run_row[f].assign(Ny, 0);
                if (ymode_env == 0 || ymode_env == 1) continue;
                for (int jb = 0; jb < Ny; jb += CB) {
                    const int je = std::min(Ny, jb + CB);
                    double c_run = 0, c_dense = 0;
                    for (int j = jb; j < je;) {
                        int R = 1;
                        const int cap = yr_group_cap(Nr[j]);
                        while (j + R < je && R < cap && Nr[j + R] == Nr[j]) ++R;
                        c_run += 2.0 * (Nr[j] + 1) + 4.0 * R;
                        for (int t = 0; t < R; ++t) c_dense += 2.0 * Nr[j + t] + 1.0;
                        j += R;
                    }
                    // ... and only where a 128-row block of such rows fits twice into shared memory (N up to ~150): taller windows force
                    // short blocks, which re-read their windows many times over (measured on the reference's default plane, N_y up to
                    // 212: 32-row blocks with 400-row windows made the y-sweep slower than the band matrices alone)
                    int Nm = 0, Nmin = 1 << 30;
                    for (int j = jb; j < je; ++j) { Nm = std::max(Nm, Nr[j]); Nmin = std::min(Nmin, Nr[j]); }
                    const bool roomy = ysweep_run_smem(round_up(128 + 2 * Nm, YR_BOX), 2) <= (size_t)yprop.sharedMemPerBlockOptin;
                    if (ymode_env == 2 || (c_run < 0.5 * c_dense && roomy)) std::fill(run_row[f].begin() + jb, run_row[f].begin() + je, 1);
                    else {
                        if (ymode_env < 0 && Nmin >= 1 && c_dense < 48.0 * (je - jb)) cheap[f].push_back(jb);
                        band_cost += c_dense;
                        band_convertible = band_convertible && roomy && Nmin >= 1;
                    }
                    all_cost += c_dense;
                }
            }
            // Blocks of small half-widths (N below ~24, near the wall) cost next to nothing in either form: where the plane runs the
            // run form anyway they join it, so that a plane is not split into two launches for their sake (1024x2048 profile:
            // 0.113 -> 0.109 ms/step)
            bool some_run = false;
            for (int f = 0; f < 3; ++f) some_run = some_run || std::count(run_row[f].begin(), run_row[f].end(), 1) > 0;
            if (some_run)
                for (int f = 0; f < 3; ++f)
                    for (int jb : cheap[f]) std::fill(run_row[f].begin() + jb, run_row[f].begin() + std::min(Ny, jb + CB), 1);
            // ... and so do the band-matrix blocks altogether when they are a small part of the plane's work (< 15 % of the direct
            // sum's multiply-adds) and all of them fit: the second launch costs more than the band matrices save on them
            // (1024x2048 profile, 64 of 1024 rows where N_y climbs from 20 to 118: 0.113 -> 0.109 ms/step as one launch)
            if (some_run && ymode_env < 0 && band_convertible && band_cost < 0.15 * all_cost)
                for (int f = 0; f < 3; ++f) run_row[f].assign(Ny, 1);
            // run plan over the run rows: maximal contiguous ranges chopped into blocks of RB rows; a block x 32 columns = one tile
            auto build = [&](int RB) {
                rg.clear(); rt.clear();
                int wmax = 0;
                for (int f = 0; f < 3; ++f) {
                    const FieldPlan& FP = P.f[f];
                    for (int ja = 0; ja < Ny;) {
                        if (!run_row[f][ja]) { ++ja; continue; }
                        int jz = ja;
                        while (jz < Ny && run_row[f][jz]) ++jz;                       // run range [ja, jz)
                        for (int jb = ja; jb < jz; jb += RB) {
                            const int je = std::min(jz, jb + RB);
                            std::vector<YRGroup> blk;
                            for (int j0 = jb; j0 < je;) {
                                const int N = FP.N_y_row[j0];
                                int R = 1;
                                const int cap = yr_group_cap(N);
                                while (j0 + R < je && R < cap && FP.N_y_row[j0 + R] == N) ++R;
                                YRGroup g{};
                                g.j0 = j0; g.nrows = R; g.N = N; g.pad = R > YJ ? 1 : 0;
                                if (N >= 1) {
                                    const long double a = (long double)std::exp(-2.0 * 3.14159265358979323846 * 1.0 / N);
                                    g.a = (double)a;
                                    g.a4 = (double)(a * a * a * a);
                                    g.naN1 = -(double)std::pow(a, (long double)(N + 1));
                                }
                                g.inv_s = *P.coef.centre(N);
                                blk.push_back(g);
                                j0 += R;
                            }
                            std::stable_sort(blk.begin(), blk.end(), [](const YRGroup& x, const YRGroup& y) { return 2 * x.N + 4 * x.nrows > 2 * y.N + 4 * y.nrows; });
                            YRTile t{};
                            t.field = f; t.g0 = (int)rg.size(); t.ngroups = (int)blk.size();
                            int lo = 1 << 30, hi = -1;
                            for (const YRGroup& g : blk) {
                                lo = std::min(lo, g.j0 + FP.Ny_max - g.N);
                                hi = std::max(hi, g.j0 + g.nrows - 1 + FP.Ny_max + g.N);
                            }
                            t.wlo = lo; t.wrows = hi - lo + 1;
                            wmax = std::max(wmax, round_up(t.wrows, YR_BOX));
                            rg.insert(rg.end(), blk.begin(), blk.end());
                            for (int c0 = 0; c0 < D.f[f].We; c0 += YR_C) { t.col0 = c0; rt.push_back(t); }
                        }
                        ja = jz;
                    }
                }
                return wmax;
            };
            const size_t smem_cap = (size_t)yprop.sharedMemPerBlockOptin;
            bool fits = false;
            for (int pass = 0; pass < 2 && !fits; ++pass) {
                for (int RB : {128, 64, 32}) {
                    r_wrows = build(RB); r_nbuf = 2;
                    if (rt.empty() || ysweep_run_smem(r_wrows, 2) <= smem_cap) { fits = true; break; }
                }
                if (fits) break;
                if (ymode_env == 2) {
                    // forced: one window buffer per CTA before giving a block up
                    for (int RB : {128, 64, 32}) {
                        r_wrows = build(RB); r_nbuf = 1;
                        if (ysweep_run_smem(r_wrows, 1) <= smem_cap) { fits = true; break; }
                    }
                    if (fits) break;
                }
                // blocks whose own window is too tall go back to the band matrices, then one more try
                const int nb = ymode_env == 2 ? 1 : 2;
                for (int f = 0; f < 3; ++f)
                    for (int jb = 0; jb < Ny; jb += CB) {
                        if (!run_row[f][jb]) continue;
                        const int je = std::min(Ny, jb + CB);
                        int Nm = 0;
                        for (int j = jb; j < je; ++j) Nm = std::max(Nm, P.f[f].N_y_row[j]);
                        if (ysweep_run_smem(round_up(CB + 2 * Nm, YR_BOX), nb) > smem_cap) std::fill(run_row[f].begin() + jb, run_row[f].begin() + je, 0);
                    }
            }
            if (!fits) { for (int f = 0; f < 3; ++f) run_row[f].assign(Ny, 0); rg.clear(); rt.clear(); }
        }
        bool any_run = !rt.empty(), any_band = false;
        for (int f = 0; f < 3; ++f) for (int j = 0; j < Ny; ++j) any_band = any_band || !run_row[f][j];
        // Both forms on one plane = two y-sweep launches per step; that only pays when the run-recursive part has enough tiles to
        // fill the machine a few times over (measured on the reference's default plane: alone 49.6 us per step against 42.5 with the
        // band matrices only; as a batch of 8 planes 20.8 us per plane-step against 23.8)
        // (counted on the WHOLE plane's width, so that every slab of a plane takes the decision the plane itself would take)
        long long run_tiles_plane = 0;
        for (const YRTile& t : rt) if (t.col0 == 0) run_tiles_plane += (NzG + YR_C - 1) / YR_C;
        if (any_run && any_band && ymode_env < 0 && run_tiles_plane * NP < 4ll * yprop.multiProcessorCount) {
            for (int f = 0; f < 3; ++f) run_row[f].assign(Ny, 0);
            rg.clear(); rt.clear();
            any_run = false;
        }
        // Row groups.  The reference's coefficients are b_i = a^|i| / s (df.cpp:168-177): a group whose rows all have the same
        // half-width N >= 16 is evaluated recursively (ysweep_rec_kernel: ~1 FMA per input row and column instead of 8); the
        // others keep the dense band matrix.  N_y changes every few rows on boundary-layer grids, so groups follow the runs of
        // equal N: whole groups of YJ rows out of a run, a tail of >= 4 rows as a short group, shorter leftovers merged into a
        // mixed (dense) group with their neighbours.  DFB_Y_MODE=0: fixed groups of YJ rows, all dense.
        constexpr int Y_REC_MIN_N = 16;
        // Recursive row groups (ysweep_rec_kernel) or not?  A group can only be recursive if all its rows share one N >= 16, so the
        // groups then follow the runs of equal N_y: more, shorter groups, each streaming its whole window.  Cost model in units of
        // 8-row chunks x columns: a dense chunk costs 256 FMAs per lane, a bulk chunk of a recursive group 32.  Measured: uniform
        // planes 0.223 -> 0.159 ms/step (model ratio 0.20), 4096x8192 boundary-layer profile 2.13 -> 2.05 (0.54), 1024x2048
        // boundary-layer profile 0.142 -> 0.153 (0.67: N_y changes every ~9 rows where it is large).  On when the ratio is below 0.6;
        // DFB_Y_MODE=1 / 0 forces it on / off.
        bool yrec_on;
        {
            double dense = 0, hybrid = 0;
            for (int f = 0; f < 3; ++f) {
                const std::vector<int>& Nr = P.f[f].N_y_row;
                const int Nmx = P.f[f].Ny_max;
                auto chunks = [&](int j0, int nr, int N) { return (j0 + nr - 1 + Nmx + N) / RC - (j0 + Nmx - N) / RC + 1; };
                for (int j0 = 0; j0 < Ny; j0 += YJ) {
                    const int nr = std::min(YJ, Ny - j0);
                    int N = 0;
                    for (int jj = 0; jj < nr; ++jj) N = std::max(N, Nr[j0 + jj]);
                    dense += 256.0 * chunks(j0, nr, N);
                }
                for (int j = 0; j < Ny;) {
                    int R = 1;
                    while (j + R < Ny && Nr[j + R] == Nr[j]) ++R;
                    const int N = Nr[j];
                    if (N >= Y_REC_MIN_N && R >= 4) {
                        const int nr = std::min(R, YJ), w0 = j + Nmx - N;
                        int nbulk = 0;
                        for (int c = w0 / RC; c <= (w0 + 2 * N + nr - 1) / RC; ++c) {
                            const int i0 = c * RC - w0;
                            if ((i0 >= nr - 1 && i0 + RC - 1 <= N - 1) || (i0 >= N + nr && i0 + RC - 1 <= 2 * N)) ++nbulk;
                        }
                        hybrid += 256.0 * (chunks(j, nr, N) - nbulk) + 32.0 * nbulk;
                        j += nr;
                    } else {
                        const int nr = std::min(std::min(R, YJ), Ny - j);          // (mixed groups merge leftovers: close enough)
                        hybrid += 256.0 * chunks(j, nr, N) * (R < 4 ? 0.5 : 1.0);
                        j += nr;
                    }
                }
            }
            yrec_on = !any_run && hybrid < 0.6 * dense;               // (rows the run form took are the ones this would have paid on)
            if (ymode_env >= 0) yrec_on = ymode_env == 1;
        }
        std::vector<char> yrec_need(P.coef.Nmax + 1, 0);
        std::vector<double> ygc(16, 0.0);     // recursive groups: 8 low-bulk + 8 high-bulk factors each; entry 0 = zeros (mixed groups)
        std::vector<YTile> tiles_dense, tiles_rec;
        // columns per dense tile: 64 instead of 128 when 128-column tiles would not even give every SM two CTAs (the reference's
        // default plane: 192 tiles of up to 57 chunks; y-sweep 0.036 -> 0.026 ms); recursive tiles always take 128
        int ytk = Y_TK;
        if (!yrec_on) {
            long long est = 0;
            for (int f = 0; f < 3; ++f) {
                const int nband = (int)std::count(run_row[f].begin(), run_row[f].end(), 0);
                est += (long long)((D.f[f].We + Y_TK - 1) / Y_TK) * (((nband + YJ - 1) / YJ + Y_G - 1) / Y_G);
            }
            int nymax = 0;
            for (int f = 0; f < 3; ++f) nymax = std::max(nymax, P.f[f].Ny_max);
            if (est * NP < 2 * 148 && nymax >= 64) ytk = 64;      // few, very long tiles (measured: 512x512 N <= 32 prefers 128); a batch has NP times as many
            if (const char* e = std::getenv("DFB_Y_TK")) ytk = std::atoi(e) == 64 ? 64 : Y_TK;
        }
        for (int f = 0; f < 3; ++f) {
            const FieldPlan& FP = P.f[f];
            std::vector<YGroup> gk[2];        // [0] dense (mixed half-widths or small N), [1] recursive, each in row order
            // (rows of the run-recursive form are skipped; a run of equal N ends where such rows begin)
            auto run_len = [&](int j) { int r = 1; while (j + r < Ny && !run_row[f][j + r] && FP.N_y_row[j + r] == FP.N_y_row[j]) ++r; return r; };
            for (int j0 = 0; j0 < Ny;) {
                if (run_row[f][j0]) { ++j0; continue; }
                YGroup g{};
                int nr;
                bool uniform = false;
                const int R = run_len(j0);
                if (yrec_on && FP.N_y_row[j0] >= Y_REC_MIN_N && R >= 4) { nr = std::min(R, YJ); uniform = true; }
                else {
                    // mixed group: up to YJ rows, but stop in front of a run long enough to be worth its own recursive groups
                    nr = 0;
                    while (nr < YJ && j0 + nr < Ny && !run_row[f][j0 + nr]) {
                        const int r2 = run_len(j0 + nr);
                        if (yrec_on && nr > 0 && FP.N_y_row[j0 + nr] >= Y_REC_MIN_N && r2 >= YJ) break;
                        nr += std::min(r2, YJ - nr);
                    }
                }
                g.field = f; g.j0 = j0; g.nrows = nr;
                g.Nmax = 0;
                for (int jj = 0; jj < g.nrows; ++jj) g.Nmax = std::max(g.Nmax, FP.N_y_row[j0 + jj]);
                // padded input rows touched: output row j0+jj, tap i -> row j0 + jj + Ny_max + i  (df.cpp:362,374)
                const int lo = j0 + FP.Ny_max - g.Nmax, hi = j0 + g.nrows - 1 + FP.Ny_max + g.Nmax;
                g.cstart = lo / RC;
                g.nchunks = hi / RC + 1 - g.cstart;
                g.rec = uniform ? 1 : 0;
                g.w0 = lo;
                // band matrix of the group (recursive groups only use the chunks at the ends of the window and around the output rows)
                g.cmat_off = (long long)cmat.size();
                cmat.resize(cmat.size() + (size_t)g.nchunks * RC * YJ, 0.0);
                {
                    double* cm = cmat.data() + g.cmat_off;
                    for (int jj = 0; jj < g.nrows; ++jj) {
                        const int N = FP.N_y_row[j0 + jj];
                        const double* b = P.coef.centre(N);
                        for (int i = -N; i <= N; ++i)
                            cm[(size_t)(j0 + jj + FP.Ny_max + i - g.cstart * RC) * YJ + jj] = b[i];
                    }
                }
                if (g.rec) {
                    // Bulk chunks: all 8 rows lie in EVERY output row's window and on one side of every centre, so their contribution
                    // to output t is one shared geometric sum times a per-row factor (<= 1):
                    //   low  bulk (window positions nrows-1 <= i <= N-1):  out_t += s^-1 a^(N+t-i_ll) * G,  G = sum a^(i_ll-i) x_i
                    //   high bulk (N+nrows <= i <= 2N):                    out_t += s^-1 a^(i_fh-N-t) * K,  K = sum a^(i-i_fh) x_i
                    // (i_ll / i_fh: last row of the last low / first row of the first high bulk chunk).  16 factors per group.
                    const int N = g.Nmax;
                    int i_ll = -1, i_fh = -1;
                    for (int c = g.cstart; c < g.cstart + g.nchunks; ++c) {
                        const int i0 = c * RC - g.w0;
                        if (i0 >= g.nrows - 1 && i0 + RC - 1 <= N - 1) i_ll = i0 + RC - 1;
                        if (i_fh < 0 && i0 >= N + g.nrows && i0 + RC - 1 <= 2 * N) i_fh = i0;
                    }
                    const long double a = (long double)std::exp(-2.0 * 3.14159265358979323846 * 1.0 / N);
                    const long double cn = (long double)*P.coef.centre(N);
                    g.gc_off = (int)(ygc.size() / 16);
                    ygc.resize(ygc.size() + 16, 0.0);
                    double* q = ygc.data() + (size_t)g.gc_off * 16;
                    for (int t = 0; t < g.nrows; ++t) {
                        q[t] = i_ll >= 0 ? (double)(cn * std::pow(a, (long double)(N + t - i_ll))) : 0.0;
                        q[8 + t] = i_fh >= 0 ? (double)(cn * std::pow(a, (long double)(i_fh - N - t))) : 0.0;
                    }
                    yrec_need[N] = 1;
                }
                gk[g.rec].push_back(g);
                j0 += nr;
            }
            // tiles: up to Y_G ADJACENT groups share one sample stream.  With recursive groups in play every tile goes through
            // ysweep_rec_kernel, which runs mixed groups entirely through its dense path (tiles of one kind only, built from
            // non-adjacent groups and launched as two kernels, measured slower: longer union windows, two tails)
            {
                const int first_group = (int)groups.size();
                std::vector<YGroup> all = gk[0];
                all.insert(all.end(), gk[1].begin(), gk[1].end());
                std::stable_sort(all.begin(), all.end(), [](const YGroup& a, const YGroup& b) { return a.j0 < b.j0; });
                groups.insert(groups.end(), all.begin(), all.end());
                const int ng = (int)all.size();
                for (int gb = 0; gb < ng;) {
                    YTile t{};
                    int cnt = 1;                                      // up to Y_G groups that are adjacent in the plane
                    while (cnt < Y_G && gb + cnt < ng && all[gb + cnt].j0 == all[gb + cnt - 1].j0 + all[gb + cnt - 1].nrows) ++cnt;
                    t.field = f; t.g0 = first_group + gb; t.ngroups = cnt;
                    t.cbegin = 1 << 30; t.cend = 0;
                    for (int w = 0; w < t.ngroups; ++w) {
                        const YGroup& g = groups[t.g0 + w];
                        t.cbegin = std::min(t.cbegin, g.cstart);
                        t.cend = std::max(t.cend, g.cstart + g.nchunks);
                    }
                    const int step = yrec_on ? Y_TK : ytk;
                    for (int c0 = 0; c0 < D.f[f].We; c0 += step) { t.col0 = c0; (yrec_on ? tiles_rec : tiles_dense).push_back(t); }
                    gb += cnt;
                }
            }
        }
        auto longest_first = [](const YTile& a, const YTile& b) { return (a.cend - a.cbegin) > (b.cend - b.cbegin); };
        std::stable_sort(tiles_dense.begin(), tiles_dense.end(), longest_first);
        std::stable_sort(tiles_rec.begin(), tiles_rec.end(), longest_first);
        H.n_tiles_dense = (int)tiles_dense.size();
        H.n_tiles_rec = (int)tiles_rec.size();
        tiles = tiles_dense;
        tiles.insert(tiles.end(), tiles_rec.begin(), tiles_rec.end());
        {
            // per half-width: a, -a^(N+1), 1/s, a^-1 .. a^-7, a^2, a^4, a^8
            std::vector<double> yrec((size_t)(P.coef.Nmax + 1) * 16, 0.0);
            for (int N = 1; N <= P.coef.Nmax; ++N) {
                if (!yrec_need[N]) continue;
                double* q = yrec.data() + (size_t)N * 16;
                const long double a = (long double)std::exp(-2.0 * 3.14159265358979323846 * 1.0 / N);
                q[0] = (double)a;
                q[1] = -(double)std::pow(a, (long double)(N + 1));
                q[2] = *P.coef.centre(N);
                for (int t = 1; t < 8; ++t) q[2 + t] = (double)std::pow(a, (long double)(-t));
                q[10] = (double)(a * a); q[11] = (double)std::pow(a, 4.0L); q[12] = (double)std::pow(a, 8.0L);
            }
            H.yp[0].yrec = H.upload(yrec);
            H.yp[0].ygc = H.upload(ygc);
        }
        H.yp[0].resident_grid = std::getenv("DFB_Y_PERSIST") ? std::atoi(std::getenv("DFB_Y_PERSIST")) : 0;
        H.yp[0].tk = ytk;
        H.yp[0].groups = H.upload(groups);
        H.yp[0].tiles = H.upload(tiles);
        H.yp[0].cmat = H.upload(cmat);
        H.yp[0].D = H.D[0];
        H.yp[0].prof = H.dalloc<unsigned long long>(8);
        if (std::getenv("DFB_TIMELINE")) { H.tl = H.dalloc<unsigned long long>(512); timeline_reset(H); }
        H.yp[0].debug = std::getenv("DFB_DEBUG_Y") ? std::atoi(std::getenv("DFB_DEBUG_Y")) : 0;
        // form of the y-sweep: 0 dense band matrices, 1 chunk-recursive band matrices, 2 run-recursive, 3 both (run form on the row
        // blocks where it pays, dense band matrices on the rest)
        H.y_form = any_run ? (any_band ? 3 : 2) : (yrec_on ? 1 : 0);
        if (any_run) {
            // most expensive tiles first; the persistent CTAs take them round-robin.  A tile's window overlaps those of the row blocks
            // above and below it (block + 2 N rows): while the sweep's whole input fits in L2 (126 MB) the re-reads are served from
            // there; a larger plane (4096x8192: 0.8 GB) is walked in groups of a few 32-column tiles -- every row block of every field
            // of the group, most expensive first, before the next group -- so that the overlapping rows are still in L2 when the
            // neighbouring block asks for them.  (The order of the tiles does not enter any cell's arithmetic.)
            auto cost = [&](const YRTile& t) { long long c = 0; for (int g = 0; g < t.ngroups; ++g) c += 2 * rg[t.g0 + g].N + 4 * rg[t.g0 + g].nrows + 8; return c; };
            size_t in_bytes = 0, coltile_bytes = 0;
            for (int f = 0; f < 3; ++f) {
                in_bytes += (size_t)NP * D.f[f].ps_ys * sizeof(double);
                coltile_bytes += (size_t)NP * D.f[f].rows_y * YR_C * sizeof(double);
            }
            int colgroup = 1 << 30;                                   // 32-column tiles per group: everything in one group
            if (in_bytes > ((size_t)96 << 20)) colgroup = (int)std::max<size_t>(1, ((size_t)16 << 20) / coltile_bytes);
            if (const char* e = std::getenv("DFB_Y_COLGROUP")) colgroup = std::max(1, std::atoi(e));
            std::stable_sort(rt.begin(), rt.end(), [&](const YRTile& x, const YRTile& y) {
                const int gx = x.col0 / YR_C / colgroup, gy = y.col0 / YR_C / colgroup;
                return gx != gy ? gx < gy : cost(x) > cost(y);
            });
            H.yp[0].rgroups = H.upload(rg);
            H.yp[0].rtiles = H.upload(rt);
            H.yp[0].n_rtiles = (int)rt.size();
            H.yp[0].r_wrows = r_wrows;
            H.yp[0].r_nbuf = r_nbuf;
            H.yp[0].r_smem = (int)ysweep_run_smem(r_wrows, r_nbuf);
            H.yp[0].r_grid = yprop.multiProcessorCount;
            H.yp[0].rcounter = H.dalloc<int>(4, false);          // tile queues, filled by reset_run_queues() below
            CUDA_TRY(ysweep_run_prepare((size_t)H.yp[0].r_smem));
        }
        H.yp[1] = H.yp[0];
        H.yp[1].D = H.D[1];
        if (H.yp[1].rcounter) H.yp[1].rcounter += 2;
        reset_run_queues(H);
        H.n_items = (int)tiles.size();
        for (int b = 0; b < 2; ++b)
        for (int f = 0; f < 3; ++f) {
            const FieldDev& F = H.D[b].f[f];
            cuuint64_t dims[2] = {(cuuint64_t)F.We, (cuuint64_t)F.rows_y * (cuuint64_t)NP};      // planes of a batch stacked along the rows
            cuuint64_t strides[1] = {(cuuint64_t)F.pitch_y * sizeof(double)};
            cuuint32_t box[2] = {(cuuint32_t)ytk, (cuuint32_t)RC};
            cuuint32_t estr[2] = {1u, 1u};
            CUresult r = encode_tiled()(&H.maps[b].m[f], CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, F.r_ys, dims, strides, box, estr,
                                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (r != CUDA_SUCCESS) throw Error{DFB_ERR_CUDA, "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")"};
        }
        if (H.y_form >= 2)
            for (int b = 0; b < 2; ++b)
                for (int f = 0; f < 3; ++f) {
                    const FieldDev& F = H.D[b].f[f];
                    cuuint64_t dims[2] = {(cuuint64_t)F.We, (cuuint64_t)F.rows_y * (cuuint64_t)NP};
                    cuuint64_t strides[1] = {(cuuint64_t)F.pitch_y * sizeof(double)};
                    cuuint32_t box[2] = {(cuuint32_t)YR_C, (cuuint32_t)YR_BOX};
                    cuuint32_t estr[2] = {1u, 1u};
                    CUresult r = encode_tiled()(&H.rmaps[b].m[f], CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, F.r_ys, dims, strides, box, estr,
                                                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                                CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
                    if (r != CUDA_SUCCESS) throw Error{DFB_ERR_CUDA, "cuTensorMapEncodeTiled (y, run form) failed (" + std::to_string((int)r) + ")"};
                }
        CUDA_TRY(ysweep_prepare());
        ZParams& Z = H.zp[0];
        Z.D = H.D[0];
        {
            // outputs per lane: 16 (fewest LDS per DFMA) unless the plane is narrower than one 512-column strip
            const char* zk_env = std::getenv("DFB_ZK");
            int nzmax_all = 0;
            for (int f = 0; f < 3; ++f) nzmax_all = std::max(nzmax_all, P.f[f].Nz_max);
            // by the PLANE's width and largest N_z (never the slab's): slabs then share the plane's lane blocking.  Short windows
            // (default reference plane: N_z <= 6) are latency-bound: 256-column units give twice as many of them (0.036 -> 0.017 ms).
            const int ZKc = zk_env ? std::atoi(zk_env) : ((P.NzG >= 384 && nzmax_all >= 24) ? 16 : 8);
            if (ZKc != 8 && ZKc != 16) throw Error{DFB_ERR_ARG, "DFB_ZK must be 8 or 16"};
            const int strip = 32 * ZKc;
            Z.zk = ZKc;
            // padded coefficient vectors: the staged window starts on a line boundary, d(N) columns before the first tap
            // (zoff + Nz_max is a multiple of 16 and strips start on multiples of 32*zk, so d = (-N) mod zk)
            std::vector<long long> pptr(P.coef.Nmax + 1, -1);
            std::vector<double> pvals;
            int maxlines = 0, maxcoef = 0;
            std::vector<char> need(P.coef.Nmax + 1, 0);
            for (int f = 0; f < 3; ++f) for (int v : P.f[f].N_z_row) need[v] = 1;
            for (int N = 0; N <= P.coef.Nmax; ++N) {
                if (!need[N]) continue;
                const int d = ((-N) % ZKc + ZKc) % ZKc;
                const int nchunk = 1 + (2 * N + d + ZKc - 1) / ZKc;
                const int clen = round_up((nchunk + 1) * ZKc, 16) + 16;     // + one 128-byte header line at the end (recursive form)
                pptr[N] = (long long)pvals.size();
                pvals.resize(pvals.size() + clen, 0.0);
                double* B = pvals.data() + pptr[N];
                const double* b = P.coef.vals.data() + P.coef.ptr[N];
                for (int t = 0; t <= 2 * N; ++t) B[t + ZKc + d] = b[t];
                if (N >= 1) {
                    // b_i = a^|i| / s with a = exp(-2 pi / N) (df.cpp:168-177): the header carries what the recursive
                    // evaluation needs: a, a^(N+1), 1/s, N, d.  a is the reference's own i = 1 weight: b_1 / b_0.
                    double* hdr = B + clen - 16;
                    const double a = std::exp(-2.0 * 3.14159265358979323846 * 1.0 / N);
                    hdr[0] = a;
                    hdr[1] = (double)std::pow((long double)a, (long double)(N + 1));
                    hdr[2] = b[N];                    // centre coefficient = 1 / s
                    hdr[3] = (double)N;
                    hdr[4] = (double)d;
                    for (int q = 1; q <= 4; ++q) hdr[4 + q] = (double)std::pow((long double)a, (long double)(1 << q));   // a^2, a^4, a^8, a^16
                }
                maxlines = std::max(maxlines, 32 + nchunk);          // lane 31 reads line 31 + ch, ch < nchunk
                maxcoef = std::max(maxcoef, clen);
            }
            Z.coef_pad = H.upload(pvals);
            Z.coef_pad_ptr = H.upload(pptr);
            Z.box_lines = maxlines;
            Z.box_bytes = maxlines * ZKc * 8;
            // Recursive evaluation of the truncated two-sided exponential (see the kernel) unless the slab starts or ends off a
            // 16-column boundary of the plane (its lane blocks would differ from the whole plane's: results would agree to
            // ~1e-14 but not bit for bit) or a row has N = 0.  DFB_Z_MODE=0 forces the direct Toeplitz form.
            {
                bool rec = (P.k0 % 16) == 0 && (P.k1 % 16 == 0 || P.k1 == P.NzG);
                for (int f = 0; f < 3; ++f) for (int v : P.f[f].N_z_row) rec = rec && v >= 1;
                const char* zm = std::getenv("DFB_Z_MODE");
                Z.zmode = zm ? std::atoi(zm) : (rec ? 1 : 0);
                if (Z.zmode == 1 && !rec) throw Error{DFB_ERR_ARG, "DFB_Z_MODE=1 needs slab boundaries on multiples of 16 columns and N_z >= 1"};
            }
            // what is staged after the window: the whole padded coefficient vector (direct form) or only its 128-byte header line
            const int tailcoef = Z.zmode == 1 ? 16 : maxcoef;
            Z.rc_off = Z.box_bytes + tailcoef * 8;                        // row constants: 64 bytes
            Z.fo_off = round_up(Z.rc_off + ROWC * 8, 128);                // staged strip of filt_old: 32 lines
            Z.unit_bytes = round_up(Z.fo_off + 32 * ZKc * 8, ZKc == 16 ? 1024 : 512);   // the swizzle pattern repeats every 1024 (512) bytes
            // per warp: two staging buffers + the u line buffer (32 lines); then mbarriers, item descriptors (2 x 2 x 8 ints per warp), alignment slack
            Z.smem_bytes = 4 * (2 * Z.unit_bytes + 32 * ZKc * 8) + 64 + 4 * 32 * 4 + 1024;
            if (maxlines > 256) throw Error{DFB_ERR_ARG, "z half-width too large for the staged window"};
            // Work items pulled from a counter by the persistent warps: per (row, strip) the pair of units (u, v) -- v' needs u's
            // blended field (df.cpp:437), which the u unit leaves in the warp's shared-memory line buffer for the v unit that
            // follows it -- and the unit w as an item of its own.
            std::vector<ZUnit> units;
            const int nstrips = (W + strip - 1) / strip;
            struct Item { int j, si, cost; };
            std::vector<Item> items;
            for (int j = 0; j < Ny; ++j)
                for (int si = 0; si < nstrips; ++si) items.push_back(Item{j, si, 0});
            auto make_unit = [&](const Item& it, int f) {
                const int N = P.f[f].N_z_row[it.j];
                const int d = ((-N) % ZKc + ZKc) % ZKc;
                const int clen = round_up((1 + (2 * N + d + ZKc - 1) / ZKc + 1) * ZKc, 16) + 16;
                ZUnit u{};
                u.j = it.j; u.f = f;
                u.nchunk = 1 + (2 * N + d + ZKc - 1) / ZKc;
                if (Z.zmode == 1) { u.cbytes = 16 * (int)sizeof(double); u.coff16 = (int)((pptr[N] + clen - 16) / 16); }
                else { u.cbytes = clen * (int)sizeof(double); u.coff16 = (int)(pptr[N] / 16); }
                const FieldDev& F = H.D[0].f[f];
                u.c0 = it.si * strip;
                u.line0 = (F.zoff + u.c0 + F.Nz_max - N) / ZKc;      // that column is d past a line boundary by construction
                return u;
            };
            // pairs (u, v) first, then the w units on their own: the tail of the queue is one unit long
            auto by_cost = [&](int fa, int fb) {
                std::vector<Item> v = items;
                for (Item& it : v) it.cost = P.f[fa].N_z_row[it.j] + (fb >= 0 ? P.f[fb].N_z_row[it.j] : 0);
                std::stable_sort(v.begin(), v.end(), [](const Item& a, const Item& b2) { return a.cost > b2.cost; });
                return v;
            };
            for (const Item& it : by_cost(0, 1)) { units.push_back(make_unit(it, 0)); units.push_back(make_unit(it, 1)); }
            for (const Item& it : by_cost(2, -1)) units.push_back(make_unit(it, 2));
            units.push_back(ZUnit{});                                // the last single item is fetched as 8 ints: nothing to pad, but keep the array non-empty-safe
            Z.units = H.upload(units);
            Z.unit_par = nullptr;
            if (Z.zmode == 1) {
                // one record per (row, field): the half-width's parameter line + the row's epilogue constants
                std::vector<double> par((size_t)Ny * 3 * (16 + ROWC), 0.0);
                for (int j = 0; j < Ny; ++j)
                    for (int f = 0; f < 3; ++f) {
                        const int N = P.f[f].N_z_row[j];
                        const int d = ((-N) % ZKc + ZKc) % ZKc;
                        const int clen = round_up((1 + (2 * N + d + ZKc - 1) / ZKc + 1) * ZKc, 16) + 16;
                        double* q = par.data() + ((size_t)j * 3 + f) * (16 + ROWC);
                        std::copy(pvals.begin() + pptr[N] + clen - 16, pvals.begin() + pptr[N] + clen, q);
                        std::copy(rowc.begin() + (size_t)j * ROWC, rowc.begin() + (size_t)(j + 1) * ROWC, q + 16);
                    }
                Z.unit_par = H.upload(par);
            }
            Z.n_uv = (int)items.size();
            Z.n_items = 2 * (int)items.size();
            Z.counter = H.dalloc<int>(2);        // one work counter per buffer set: y(s+1) resets its own while z(s) still pulls from the other
            Z.debug = std::getenv("DFB_DEBUG_Z") ? std::atoi(std::getenv("DFB_DEBUG_Z")) : 0;
            Z.prof = H.dalloc<unsigned long long>(4096);
            cudaDeviceProp prop;
            CUDA_TRY(cudaGetDeviceProperties(&prop, H.device));
            int zb = 1;
            CUDA_TRY(zsweep_prepare(Z.zk, Z.zmode, (size_t)Z.smem_bytes, &zb));
            // The recursive form is bound by shared-memory traffic and latency, not by the fp64 pipe: two CTAs per SM run it as
            // fast as three would in the step as a whole, because the third's registers go to the next step's noise CTAs, which
            // then run beside the sweep instead of after it (measured: 0.168 vs 0.176 ms/step on 1024x2048 profile).
            if (Z.zmode == 1 && Z.zk == 16) zb = std::min(zb, 2);
            if (std::getenv("DFB_Z_BLOCKS_PER_SM")) zb = std::min(std::max(zb, 3), std::atoi(std::getenv("DFB_Z_BLOCKS_PER_SM")));
            Z.nblocks = std::max(1, std::min(std::max(zb, 1) * prop.multiProcessorCount, (Z.n_items * NP + 3) / 4));
            Z.n_sm = prop.multiProcessorCount;
            H.yp[0].zcounter = Z.counter;
            H.yp[1].zcounter = Z.counter + 1;
            for (int b = 0; b < 2; ++b)
                for (int f = 0; f < 3; ++f) {
                    const FieldDev& F = H.D[b].f[f];
                    cuuint64_t dims[3] = {(cuuint64_t)Z.zk, (cuuint64_t)(F.pitch_z / Z.zk), (cuuint64_t)Ny * (cuuint64_t)NP};
                    cuuint64_t strides[2] = {(cuuint64_t)Z.zk * 8, (cuuint64_t)F.pitch_z * sizeof(double)};
                    cuuint32_t box[3] = {(cuuint32_t)Z.zk, (cuuint32_t)Z.box_lines, 1u};
                    cuuint32_t estr[3] = {1u, 1u, 1u};
                    CUresult r = encode_tiled()(&H.zmaps[b].m[f], CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, F.r_zs, dims, strides, box, estr,
                                                CU_TENSOR_MAP_INTERLEAVE_NONE, Z.zk == 16 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                                                CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
                    if (r != CUDA_SUCCESS) throw Error{DFB_ERR_CUDA, "cuTensorMapEncodeTiled (z) failed (" + std::to_string((int)r) + ")"};
                }
        }
        H.zp[1] = Z;
        H.zp[1].D = H.D[1];
        H.zp[1].counter = Z.counter + 1;
        
    }

    // ---- noise tables (include/dfb_rng_spec.h) ----
    int max_np = 1;
    for (int f = 0; f < 3; ++f) {
        const FieldDev& F = D.f[f];
        for (int kind = 0; kind < 2; ++kind) {
            NoiseHost A{};
            A.field = f; A.kind = kind;
            const uint64_t stream = (uint64_t)(((int64_t)H.plane_id * 3 + f) * 2 + kind);
            A.inc = (stream << 1) | 1u;
            A.state0 = pcg_lcg(H.seed + A.inc, A.inc);
            std::vector<Jump> jumps;
            std::vector<int> offv;         // r_ys: extended column of the segment's first pair (its first column, or one less); halo: 0
            std::vector<int> npv;
            std::vector<int4> winv;        // periodic_z, extended rows that wrap: {padded row, first, end extended column} per piece
            if (kind == 0) {
                A.npairs = ((uint64_t)F.rows_y * (uint64_t)NzG + 1u) / 2u;
                const int xk1 = F.xk0 + F.We;
                const bool wraps = F.xk0 < 0 || xk1 > NzG;   // periodic_z only
                for (int r = 0; r < F.rows_y; ++r) {
                    // the row's extended range as contiguous pieces of the stream: global columns [g0, g1) at extended column x0
                    // (left of the plane: its last columns; the plane part; right of it: its first columns)
                    const int pieces[3][3] = {{NzG + F.xk0, NzG, 0},
                                              {std::max(F.xk0, 0), std::min(xk1, NzG), std::max(F.xk0, 0) - F.xk0},
                                              {0, xk1 - NzG, NzG - F.xk0}};
                    for (const auto& pc : pieces) {
                        if (pc[1] <= pc[0]) continue;
                        const long long ea = (long long)r * NzG + pc[0], eb = (long long)r * NzG + pc[1] - 1;
                        const long long qa = ea >> 1, qb = eb >> 1;
                        offv.push_back((int)(2 * qa - ea) + pc[2]); npv.push_back((int)(qb - qa + 1));
                        jumps.push_back(pcg_jump(4u * (uint64_t)qa, 1u));
                        if (wraps) winv.push_back(make_int4(r, pc[2], pc[2] + pc[1] - pc[0], 0));
                    }
                }
                if (wraps && offv.size() > 65535u) throw Error{DFB_ERR_ARG, "periodic_z: too many padded rows for the noise kernel's grid"};
            } else if (!P.periodic) {      // periodic_z: the z filter reads no raw noise, array 1 is not drawn
                const int M = F.Nz_max;
                A.npairs = (uint64_t)Ny * (uint64_t)M;
                const bool touches = (P.k0 - M < 0) || (P.k1 + M > NzG);
                if (M > 0 && touches)
                    for (int j = 0; j < Ny; ++j) {
                        offv.push_back(0); npv.push_back(M);
                        jumps.push_back(pcg_jump(4u * (uint64_t)j * (uint64_t)M, 1u));
                    }
            }
            A.n_seg = (int)offv.size();
            for (int v : npv) max_np = std::max(max_np, v);
            if (A.n_seg) {
                A.d_jump = H.upload(jumps); A.d_off = H.upload(offv); A.d_np = H.upload(npv);
                if (!winv.empty()) A.d_win = H.upload(winv);
            }
            H.noise.push_back(A);
        }
    }
    std::vector<Jump> slot(max_np);
    for (int t = 0; t < max_np; ++t) slot[t] = pcg_jump(4u * (uint64_t)t, 1u);
    H.np.slot_jump = H.upload(slot);
    H.np.max_np = max_np;
    H.np.stride = pcg_jump(4u * (uint64_t)noise_stride_pairs(), 1u);
    H.np.chunks = (max_np + noise_threads() - 1) / noise_threads();
    CUDA_TRY(cudaStreamSynchronize(H.stream));
}

void fill_noise_params(dfb_filter_s& H, int64_t step) {
    int n = 0;
    for (const NoiseHost& A : H.noise) {
        if (!A.n_seg) continue;
        NoiseArray& a = H.np.a[n];
        a.seg_jump = A.d_jump; a.seg_off = static_cast<const int*>(A.d_off); a.seg_np = static_cast<const int*>(A.d_np);
        H.nwin.seg_win[n] = static_cast<const int4*>(A.d_win);
        a.n_seg = A.n_seg; a.kind = A.kind; a.field = A.field;
        for (int p = 0; p < H.nplanes; ++p) {
            // stream ((plane*3 + field)*2 + array) of include/dfb_rng_spec.h; plane p of a batch is plane_id + p
            const uint64_t stream = (uint64_t)((((int64_t)H.plane_id + p) * 3 + A.field) * 2 + A.kind);
            const uint64_t inc = (stream << 1) | 1u;
            const uint64_t state0 = pcg_lcg(H.seed + inc, inc);
            const Jump j = pcg_jump(4u * ((uint64_t)step * A.npairs), inc);
            H.np.pstate[p][n] = j.A * state0 + j.C;
            H.np.pinc[p][n] = inc;
        }
        ++n;
    }
    H.np.n_arrays = n;
}

void timeline_reset(dfb_filter_s& H) {
    std::vector<unsigned long long> init(512, 0ull);
    for (int i = 0; i < 512; i += 2) init[i] = ~0ull;                  // starts: atomicMin
    CUDA_TRY(cudaMemcpy(H.tl, init.data(), 512 * sizeof(unsigned long long), cudaMemcpyHostToDevice));
}

void launch_noise_for(dfb_filter_s& H, int64_t step, int b, cudaStream_t st) {
    H.ybuf_step[b] = -1;                 // new noise invalidates whatever y-sweep result the set held
    fill_noise_params(H, step);
    H.np.tl = H.tl ? H.tl + (step % 64) * 8 : nullptr;
    CUDA_TRY(launch_noise(H.np, H.nwin, H.D[b], st));
    CUDA_TRY(cudaEventRecord(H.ev_noise[b], st));
    H.buf_step[b] = step;
}

void run_step(dfb_filter_s& H, double dt, bool first) {
    CUDA_TRY(cudaSetDevice(H.device));
    const int b = (int)(H.step & 1);
    if (H.timing) CUDA_TRY(cudaEventRecord(H.ev[0], H.stream));
    if (H.noise_mode == DFB_NOISE_GENERATE) {
        // ev_noise[b] = the last noise launch into set b on EITHER stream: wait for it whether its result is the one this step
        // wants (prefetched) or not (after a dfb_set_state rewind the side stream's prefetch may still be writing set b)
        CUDA_TRY(cudaStreamWaitEvent(H.stream, H.ev_noise[b], 0));
        if (H.buf_step[b] != H.step) launch_noise_for(H, H.step, b, H.stream);
    } else if (!(H.injected[0] && H.injected[1] && H.injected[2])) {
        throw Error{DFB_ERR_STATE, "noise_mode = inject: dfb_set_noise must be called for u, v and w before every step"};
    }
    H.noise_view = b;
    if (H.tl) { H.yp[b].tl = H.tl + (H.step % 64) * 8 + 2; H.zp[b].tl = H.tl + (H.step % 64) * 8 + 4; }
    if (H.timing) CUDA_TRY(cudaEventRecord(H.ev[1], H.stream));
    if (H.noise_mode == DFB_NOISE_GENERATE && H.ybuf_step[b] == H.step) {
        // this step's y-sweep already ran (or is running) on the side stream; ev_noise[b] above covers it
    } else if (H.tuned) {
        // band-matrix tiles (if any) first, then the run-recursive tiles: disjoint rows of r_zs
        H.yp[b].zcounter_init = 8 * H.zp[b].nblocks;               // the z-sweep's warps (4 per CTA) start on two fixed items each
        if (H.y_form != 2) CUDA_TRY(launch_ysweep_tma(H.maps[b], H.yp[b], H.n_tiles_dense, H.n_tiles_rec, H.stream));
        if (H.y_form >= 2) CUDA_TRY(launch_ysweep_run(H.rmaps[b], H.yp[b], H.stream));
    }
    else CUDA_TRY(launch_ysweep_simple(H.D[b], H.stream));
    if (H.timing) CUDA_TRY(cudaEventRecord(H.ev[2], H.stream));
    StepConsts S{};
    S.first_step = first ? 1 : 0;
    for (int f = 0; f < 3; ++f) {
        const double pi = 3.141592654;                             // df.cpp:411 (SURVEY quirk 2)
        const double alpha = std::exp(-pi * dt / H.plan.f[f].Lt);  // df.cpp:412
        S.sa[f] = std::sqrt(alpha);                                // df.cpp:415
        S.sb[f] = std::sqrt(1.0 - alpha);
    }
    const bool accumulate = H.stats_on && !first;                  // rms_add, df.cpp:606
    if (H.tuned) {
        H.zp[b].S = S;
        H.zp[b].stats = accumulate ? H.stats : nullptr;            // N2 fused into the epilogue
        CUDA_TRY(launch_zsweep_tuned(H.zmaps[b], H.zp[b], H.stream));
    } else {
        CUDA_TRY(launch_zsweep_simple(H.D[b], S, H.stream));
        if (accumulate) CUDA_TRY(launch_stats(H.D[0], H.stats, H.stream));
    }
    if (accumulate) H.stats_count += 1;
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
    if (H.noise_mode == DFB_NOISE_GENERATE && H.overlap && !H.timing) {
        const int nb = (int)(H.step & 1);
        CUDA_TRY(cudaStreamWaitEvent(H.side, H.ev_free[nb], 0));     // readers of that set (step-2... ) are done
        CUDA_TRY(cudaStreamWaitEvent(H.side, H.ev_noise[nb], 0));    // ... and so is its last writer: a dfb_generate_noise into it
                                                                       // on the main stream after that step would otherwise race this one
        launch_noise_for(H, H.step, nb, H.side);
        // ... and so does its y-sweep (it reads only that noise and writes only that set's r_zs interior): it
        // becomes resident as this step's z-sweep CTAs retire and keeps the fp64 pipe busy through the tail.
        if (H.tuned && H.y_ahead) {
            H.yp[nb].zcounter_init = 8 * H.zp[nb].nblocks;
            if (H.y_form != 2) CUDA_TRY(launch_ysweep_tma(H.maps[nb], H.yp[nb], H.n_tiles_dense, H.n_tiles_rec, H.side));
            if (H.y_form >= 2) CUDA_TRY(launch_ysweep_run(H.rmaps[nb], H.yp[nb], H.side));
            CUDA_TRY(cudaEventRecord(H.ev_noise[nb], H.side));      // "set nb is ready" now means noise + y-sweep
            H.ybuf_step[nb] = H.step;
        }
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
        H->y_ahead = std::getenv("DFB_Y_AHEAD") != nullptr;
        H->kernel_variant = cfg->kernel_variant;
        H->seed = cfg->seed;
        H->plane_id = cfg->plane_id;
        H->nplanes = nplanes;
        if (nplanes > 1 && cfg->noise_mode != DFB_NOISE_GENERATE) throw Error{DFB_ERR_ARG, "a batch of planes generates its own noise (noise_mode = DFB_NOISE_GENERATE)"};
        build_plan(*cfg, H->plan);
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
    switch (what) {
        case 0: *out64 = h->plan.f[field].Ny_max; break;
        case 1: *out64 = h->plan.f[field].Nz_max; break;
        case 2: *out64 = h->step; break;
        case 3: *out64 = h->tuned ? 1 : 0; break;
        case 4: *out64 = h->plan.taps_per_step; break;
        case 5: *out64 = h->plan.NzG; break;
        case 6: *out64 = h->device; break;
        case 7: *out64 = h->tuned ? h->zp[0].zmode : 0; break;
        case 8: *out64 = h->tuned ? h->n_tiles_rec : 0; break;
        case 9: *out64 = h->tuned ? h->n_tiles_dense : 0; break;
        case 10: *out64 = h->tuned ? h->y_form : -1; break;
        case 12: *out64 = h->transport; break;
        case 11: *out64 = h->tuned ? h->yp[0].n_rtiles : 0; break;
        case 13: *out64 = h->plan.periodic ? 1 : 0; break;
        case 14: *out64 = h->corr_ready ? h->corr.L[field] : 0; break;
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
        if (h->pipe_ended >= h->pipe_begun) throw Error{DFB_ERR_STATE, "no dfb_filter_to_host_begin is outstanding"};
        CUDA_TRY(cudaEventSynchronize(h->ev_copied[(int)(h->pipe_ended & 1)]));
        h->pipe_ended += 1;
    });
}

int dfb_filter_batch(dfb_handle h, int nsteps, const double* dt, double* out) {
    if (!h || !dt || nsteps < 0) return fail(DFB_ERR_ARG, "bad argument");
    return guarded([&] {
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
    return guarded([&] { CUDA_TRY(cudaSetDevice(h->device)); CUDA_TRY(cudaStreamSynchronize(h->stream)); });
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
        CUDA_TRY(cudaSetDevice(h->device));
        const size_t n = h->D[0].ps_cells * h->nplanes;
        if (filt_old3)
            for (int f = 0; f < 3; ++f)
                CUDA_TRY(cudaMemcpyAsync(h->D[0].f[f].filt_old, filt_old3 + f * n, n * 8, cudaMemcpyHostToDevice, h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->side));      // a look-ahead noise launch for the old step counter may still be in flight
        if (step != h->step) { h->buf_step[0] = h->buf_step[1] = -1; h->ybuf_step[0] = h->ybuf_step[1] = -1; }
        h->step = step;
        h->corr.ring_count = 0;       // the next step follows the restored state: no temporal pair reaches back across it
    });
}

int dfb_set_timing(dfb_handle h, int on) {
    if (!h) return fail(DFB_ERR_ARG, "handle is NULL");
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
    if (!on) {                                                // the sums stay readable; the ring and the scratch go
        h->corr_on = false;
        return guarded([&] {
            CUDA_TRY(cudaSetDevice(h->device));
            CUDA_TRY(cudaStreamSynchronize(h->stream));
            CUDA_TRY(cudaFree(h->corr.ring));
            CUDA_TRY(cudaFree(h->corr.part));
            h->corr.ring = h->corr.part = nullptr;
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
        auto alloc = [&](size_t n) {
            void* q = nullptr;
            CUDA_TRY(cudaMalloc(&q, std::max<size_t>(n, 1) * sizeof(double)));
            return static_cast<double*>(q);
        };
        if (!h->corr_ready || L[0] != c.L[0] || L[1] != c.L[1] || L[2] != c.L[2]) {
            CUDA_TRY(cudaStreamSynchronize(h->stream));
            for (void* q : h->corr_mem) cudaFree(q);
            h->corr_mem.clear();
            cudaFree(c.ring);
            cudaFree(c.part);
            h->corr_ready = false;
            h->corr_on = false;
            c = CorrParams{};
            for (int f = 0; f < 3; ++f) c.fluc[f] = h->D[0].f[f].fluc;
            c.P = NP; c.Ny = Ny; c.W = W; c.periodic = P.periodic ? 1 : 0;
            for (int d = 0; d < 3; ++d) {
                c.L[d] = L[d];
                if (L[d]) { c.sum[d] = alloc(rows * (L[d] + 1)); h->corr_mem.push_back(c.sum[d]); }
            }
            c.y_nsplit = c.y_split_cols = 1;
            if (L[1]) corr_y_split(Ny, W, &c.y_nsplit, &c.y_split_cols);
        }
        // the ring and the partial-sum scratch exist only while accumulating (on = 0 frees them)
        const size_t part = corr_part_doubles(NP, Ny, W, c.L[0], c.L[1], c.y_nsplit);
        if (part && !c.part) c.part = alloc(part);
        if (c.L[2] && !c.ring) c.ring = alloc((size_t)c.L[2] * rows * W);
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

int dfb_debug_yprof(dfb_handle h, unsigned long long* out8) {
    if (!h || !out8) return fail(DFB_ERR_ARG, "bad argument");
    return guarded([&] {
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        if (!h->yp[0].prof) throw Error{DFB_ERR_STATE, "no profile buffer"};
        CUDA_TRY(cudaMemcpy(out8, h->yp[0].prof, 64, cudaMemcpyDeviceToHost));
        CUDA_TRY(cudaMemset(h->yp[0].prof, 0, 64));
    });
}

int dfb_debug_timeline(dfb_handle h, unsigned long long* out512) {
    // development aid: DFB_TIMELINE=1 at create; returns and clears 64 step slots x {noise, y, z, -} x {start, end} (ns)
    if (!h || !out512) return fail(DFB_ERR_ARG, "bad argument");
    return guarded([&] {
        if (!h->tl) throw Error{DFB_ERR_STATE, "DFB_TIMELINE was not set when the handle was created"};
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->side));
        CUDA_TRY(cudaMemcpy(out512, h->tl, 512 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        timeline_reset(*h);
    });
}

int dfb_debug_zprof(dfb_handle h, unsigned long long* out8) {
    if (!h || !out8) return fail(DFB_ERR_ARG, "bad argument");
    return guarded([&] {
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        if (!h->zp[0].prof) throw Error{DFB_ERR_STATE, "no profile buffer"};
        CUDA_TRY(cudaMemcpy(out8, h->zp[0].prof, 1024, cudaMemcpyDeviceToHost));     // 128 counters
        CUDA_TRY(cudaMemset(h->zp[0].prof, 0, 1024));
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
    if (h->nplanes != 1) return fail(DFB_ERR_STATE, "slab communication is defined for single-plane handles");
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
            if (world > 1 && h->tuned)
                for (int b = 0; b < 2; ++b) {
                    if (h->yp[b].r_grid > sms) h->yp[b].r_grid = sms;
                    const int per_sm = std::max(1, h->zp[b].nblocks / prop.multiProcessorCount);
                    if (h->zp[b].nblocks > per_sm * sms) h->zp[b].nblocks = per_sm * sms;
                }
            reset_run_queues(*h);
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
int dfb_destroy_f(dfb_handle* h) {
    if (!h) return DFB_OK;
    int rc = dfb_destroy(*h);
    *h = nullptr;
    return rc;
}

}  // extern "C"
