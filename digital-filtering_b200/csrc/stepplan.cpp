// csrc/stepplan.cpp -- the step's plan: device layout, the work descriptions of the tuned y- and z-sweeps and the noise tables,
// decided on the host from the plan and the device's limits alone.  No CUDA call, no environment: capi.cu uploads the result.
#include <algorithm>
#include <cmath>
#include "plan.hpp"
#include "noise.cuh"

namespace dfb {

namespace {

inline int round_up(int v, int m) { return (v + m - 1) / m * m; }

// The run-recursive and chunk-recursive y forms and the recursive z form evaluate the two-sided exponential by its sliding recursion;
// a Gaussian has none, so a Gaussian plane runs the direct forms, which read the coefficient table and nothing else.
Error shape_refusal(const char* what) {
    return Error{DFB_ERR_ARG, std::string(what) + " evaluates the exponential filter recursively: the filter shape is Gaussian "
                                                  "(DFB_FILTER_GAUSSIAN), which runs the direct forms only"};
}

// ratio of neighbouring coefficients, b_i = a^|i| / s (df.cpp:168-177)
inline long double exp_ratio(int N) { return (long double)std::exp(-2.0 * 3.14159265358979323846 * 1.0 / N); }

// padded coefficient vector of half-width N in the z-sweep with zk outputs per lane: the staged window starts on a line boundary,
// d(N) columns before the first tap (zoff + Nz_max is a multiple of 16 and strips start on multiples of 32*zk, so d = (-N) mod zk)
struct ZPad { int d, nchunk, clen; };
ZPad zpad(int N, int zk) {
    const int d = ((-N) % zk + zk) % zk;
    const int nchunk = 1 + (2 * N + d + zk - 1) / zk;
    return {d, nchunk, round_up((nchunk + 1) * zk, 16) + 16};     // + one 128-byte header line at the end (recursive form)
}

void plan_y(const Plan& P, int NP, const DeviceLimits& dev, const Overrides& ovr, StepPlan& S) {
    const PlaneDev& D = S.D;
    const int Ny = P.Ny, NzG = P.NzG;
    // ---- which rows go through the run-recursive form (ysweep_run_kernel), which through the band matrices ----
    // The run form evaluates a group of R rows (<= 8, or <= min(32, 0.33 N) for N >= 25) of ONE half-width N with 2(N+1) + 4R multiply-adds per column where the direct sum
    // spends R(2N+1): it pays in runs of equal N, not where N changes every row or two (a lone row costs its direct sum and
    // its window has to be staged whole).  Decided per block of 32 rows: run form where it executes less than half of the
    // direct sum's multiply-adds (and two of the block's windows fit in shared memory); the other rows keep the band matrices.
    // DFB_Y_MODE=2 forces the run form wherever a window fits at all, 0 / 1 force the band-matrix kernels (dense / chunk-recursive).
    // a Gaussian plane: dense band matrices on every block (as DFB_Y_MODE=0)
    if (P.filter_shape == DFB_FILTER_GAUSSIAN && (ovr.y_mode == 1 || ovr.y_mode == 2))
        throw shape_refusal(ovr.y_mode == 1 ? "DFB_Y_MODE=1 (chunk-recursive y-sweep)" : "DFB_Y_MODE=2 (run-recursive y-sweep)");
    const int ymode_env = P.filter_shape == DFB_FILTER_GAUSSIAN ? 0 : ovr.y_mode.value_or(-1);
    std::vector<char> run_row[3];
    std::vector<YRGroup>& rg = S.rgroups;
    std::vector<YRTile>& rt = S.rtiles;
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
                const bool roomy = ysweep_run_smem(round_up(128 + 2 * Nm, YR_BOX), 2) <= dev.smem_optin;
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
                                const long double a = exp_ratio(N);
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
        const size_t smem_cap = dev.smem_optin;
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
    if (any_run && any_band && ymode_env < 0 && run_tiles_plane * NP < 4ll * dev.sms) {
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
            auto chunks = [&](int j0, int nr, int N) { return (j0 + nr - 1 + Nmx + N) / Y_RC - (j0 + Nmx - N) / Y_RC + 1; };
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
                    for (int c = w0 / Y_RC; c <= (w0 + 2 * N + nr - 1) / Y_RC; ++c) {
                        const int i0 = c * Y_RC - w0;
                        if ((i0 >= nr - 1 && i0 + Y_RC - 1 <= N - 1) || (i0 >= N + nr && i0 + Y_RC - 1 <= 2 * N)) ++nbulk;
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
    std::vector<double>& ygc = S.ygc;
    ygc.assign(16, 0.0);                  // recursive groups: 8 low-bulk + 8 high-bulk factors each; entry 0 = zeros (mixed groups)
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
        if (ovr.y_tk) ytk = *ovr.y_tk == 64 ? 64 : Y_TK;
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
            g.cstart = lo / Y_RC;
            g.nchunks = hi / Y_RC + 1 - g.cstart;
            g.rec = uniform ? 1 : 0;
            g.w0 = lo;
            // band matrix of the group (recursive groups only use the chunks at the ends of the window and around the output rows)
            g.cmat_off = (long long)S.cmat.size();
            S.cmat.resize(S.cmat.size() + (size_t)g.nchunks * Y_RC * YJ, 0.0);
            {
                double* cm = S.cmat.data() + g.cmat_off;
                for (int jj = 0; jj < g.nrows; ++jj) {
                    const int N = FP.N_y_row[j0 + jj];
                    const double* b = P.coef.centre(N);
                    for (int i = -N; i <= N; ++i)
                        cm[(size_t)(j0 + jj + FP.Ny_max + i - g.cstart * Y_RC) * YJ + jj] = b[i];
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
                    const int i0 = c * Y_RC - g.w0;
                    if (i0 >= g.nrows - 1 && i0 + Y_RC - 1 <= N - 1) i_ll = i0 + Y_RC - 1;
                    if (i_fh < 0 && i0 >= N + g.nrows && i0 + Y_RC - 1 <= 2 * N) i_fh = i0;
                }
                const long double a = exp_ratio(N);
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
            const int first_group = (int)S.groups.size();
            std::vector<YGroup> all = gk[0];
            all.insert(all.end(), gk[1].begin(), gk[1].end());
            std::stable_sort(all.begin(), all.end(), [](const YGroup& a, const YGroup& b) { return a.j0 < b.j0; });
            S.groups.insert(S.groups.end(), all.begin(), all.end());
            const int ng = (int)all.size();
            for (int gb = 0; gb < ng;) {
                YTile t{};
                int cnt = 1;                                      // up to Y_G groups that are adjacent in the plane
                while (cnt < Y_G && gb + cnt < ng && all[gb + cnt].j0 == all[gb + cnt - 1].j0 + all[gb + cnt - 1].nrows) ++cnt;
                t.field = f; t.g0 = first_group + gb; t.ngroups = cnt;
                t.cbegin = 1 << 30; t.cend = 0;
                for (int w = 0; w < t.ngroups; ++w) {
                    const YGroup& g = S.groups[t.g0 + w];
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
    S.n_tiles_dense = (int)tiles_dense.size();
    S.n_tiles_rec = (int)tiles_rec.size();
    S.tiles = tiles_dense;
    S.tiles.insert(S.tiles.end(), tiles_rec.begin(), tiles_rec.end());
    // per half-width: a, -a^(N+1), 1/s, a^-1 .. a^-7, a^2, a^4, a^8
    S.yrec.assign((size_t)(P.coef.Nmax + 1) * 16, 0.0);
    for (int N = 1; N <= P.coef.Nmax; ++N) {
        if (!yrec_need[N]) continue;
        double* q = S.yrec.data() + (size_t)N * 16;
        const long double a = exp_ratio(N);
        q[0] = (double)a;
        q[1] = -(double)std::pow(a, (long double)(N + 1));
        q[2] = *P.coef.centre(N);
        for (int t = 1; t < 8; ++t) q[2 + t] = (double)std::pow(a, (long double)(-t));
        q[10] = (double)(a * a); q[11] = (double)std::pow(a, 4.0L); q[12] = (double)std::pow(a, 8.0L);
    }
    S.yp.tk = ytk;
    // form of the y-sweep: 0 dense band matrices, 1 chunk-recursive band matrices, 2 run-recursive, 3 both (run form on the row
    // blocks where it pays, dense band matrices on the rest)
    S.y_form = any_run ? (any_band ? 3 : 2) : (yrec_on ? 1 : 0);
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
        if (ovr.y_colgroup) colgroup = std::max(1, *ovr.y_colgroup);
        std::stable_sort(rt.begin(), rt.end(), [&](const YRTile& x, const YRTile& y) {
            const int gx = x.col0 / YR_C / colgroup, gy = y.col0 / YR_C / colgroup;
            return gx != gy ? gx < gy : cost(x) > cost(y);
        });
        S.yp.n_rtiles = (int)rt.size();
        S.yp.r_wrows = r_wrows;
        S.yp.r_nbuf = r_nbuf;
        S.yp.r_smem = (int)ysweep_run_smem(r_wrows, r_nbuf);
        S.yp.r_grid = dev.sms;
    }
}

// Plans the tuned z-sweep; false when its staged window does not fit (more than 256 lines, the largest box of a tensor map, or
// more shared memory than one block may opt in to): the handle then runs the general kernels.  Whether it fits follows from the
// half-widths and the lane blocking alone, so slabs on 16-column boundaries decide as their plane does.  A window that does not
// fit under a forced DFB_ZK or DFB_Z_MODE is an error.
bool plan_z(const Plan& P, const DeviceLimits& dev, const Overrides& ovr, StepPlan& S) {
    ZParams& Z = S.zp;
    const int Ny = P.Ny, W = P.Nz();
    // outputs per lane: 16 (fewest LDS per DFMA) unless the plane is narrower than one 512-column strip
    int nzmax_all = 0;
    for (int f = 0; f < 3; ++f) nzmax_all = std::max(nzmax_all, P.f[f].Nz_max);
    // by the PLANE's width and largest N_z (never the slab's): slabs then share the plane's lane blocking.  Short windows
    // (default reference plane: N_z <= 6) are latency-bound: 256-column units give twice as many of them (0.036 -> 0.017 ms).
    const int ZKc = ovr.zk ? *ovr.zk : ((P.NzG >= 384 && nzmax_all >= 24) ? 16 : 8);
    if (ZKc != 8 && ZKc != 16) throw Error{DFB_ERR_ARG, "DFB_ZK must be 8 or 16"};
    const int strip = 32 * ZKc;
    Z.zk = ZKc;
    std::vector<long long>& pptr = S.coef_pad_ptr;
    std::vector<double>& pvals = S.coef_pad;
    pptr.assign(P.coef.Nmax + 1, -1);
    int maxlines = 0, maxcoef = 0;
    std::vector<char> need(P.coef.Nmax + 1, 0);
    for (int f = 0; f < 3; ++f) for (int v : P.f[f].N_z_row) need[v] = 1;
    for (int N = 0; N <= P.coef.Nmax; ++N) {
        if (!need[N]) continue;
        const ZPad zp = zpad(N, ZKc);
        pptr[N] = (long long)pvals.size();
        pvals.resize(pvals.size() + zp.clen, 0.0);
        double* B = pvals.data() + pptr[N];
        const double* b = P.coef.vals.data() + P.coef.ptr[N];
        for (int t = 0; t <= 2 * N; ++t) B[t + ZKc + zp.d] = b[t];
        if (N >= 1 && P.filter_shape == DFB_FILTER_EXPONENTIAL) {
            // b_i = a^|i| / s with a = exp(-2 pi / N) (df.cpp:168-177): the header carries what the recursive
            // evaluation needs: a, a^(N+1), 1/s, N, d.  a is the reference's own i = 1 weight: b_1 / b_0.
            double* hdr = B + zp.clen - 16;
            const double a = (double)exp_ratio(N);
            hdr[0] = a;
            hdr[1] = (double)std::pow((long double)a, (long double)(N + 1));
            hdr[2] = b[N];                    // centre coefficient = 1 / s
            hdr[3] = (double)N;
            hdr[4] = (double)zp.d;
            for (int q = 1; q <= 4; ++q) hdr[4 + q] = (double)std::pow((long double)a, (long double)(1 << q));   // a^2, a^4, a^8, a^16
        }
        maxlines = std::max(maxlines, 32 + zp.nchunk);          // lane 31 reads line 31 + ch, ch < nchunk
        maxcoef = std::max(maxcoef, zp.clen);
    }
    Z.box_lines = maxlines;
    Z.box_bytes = maxlines * ZKc * 8;
    // Recursive evaluation of the truncated two-sided exponential (see the kernel) unless the slab starts or ends off a
    // 16-column boundary of the plane (its lane blocks would differ from the whole plane's: results would agree to
    // ~1e-14 but not bit for bit), a row has N = 0, or the filter shape is Gaussian.  DFB_Z_MODE=0 forces the direct Toeplitz form.
    {
        if (P.filter_shape == DFB_FILTER_GAUSSIAN && ovr.z_mode == 1) throw shape_refusal("DFB_Z_MODE=1 (recursive z-sweep)");
        bool rec = P.filter_shape == DFB_FILTER_EXPONENTIAL && (P.k0 % 16) == 0 && (P.k1 % 16 == 0 || P.k1 == P.NzG);
        for (int f = 0; f < 3; ++f) for (int v : P.f[f].N_z_row) rec = rec && v >= 1;
        Z.zmode = ovr.z_mode ? *ovr.z_mode : (rec ? 1 : 0);
        if (Z.zmode == 1 && !rec) throw Error{DFB_ERR_ARG, "DFB_Z_MODE=1 needs slab boundaries on multiples of 16 columns and N_z >= 1"};
    }
    // what is staged after the window: the whole padded coefficient vector (direct form) or only its 128-byte header line
    const int tailcoef = Z.zmode == 1 ? 16 : maxcoef;
    Z.rc_off = Z.box_bytes + tailcoef * 8;                        // row constants: 64 bytes
    Z.fo_off = round_up(Z.rc_off + ROWC * 8, 128);                // staged strip of filt_old: 32 lines
    Z.unit_bytes = round_up(Z.fo_off + 32 * ZKc * 8, ZKc == 16 ? 1024 : 512);   // the swizzle pattern repeats every 1024 (512) bytes
    // per warp: two staging buffers + the u line buffer (32 lines); then mbarriers, item descriptors (2 x 2 x 8 ints per warp), alignment slack
    Z.smem_bytes = 4 * (2 * Z.unit_bytes + 32 * ZKc * 8) + 64 + 4 * 32 * 4 + 1024;
    if (maxlines > 256 || (size_t)Z.smem_bytes > dev.smem_optin) {
        if (!ovr.zk && !ovr.z_mode) return false;
        throw Error{DFB_ERR_ARG, "z half-width too large for the tuned z-sweep under DFB_ZK / DFB_Z_MODE: its staged window needs " +
                                 std::to_string(maxlines) + " lines (at most 256) and " + std::to_string(Z.smem_bytes) +
                                 " bytes of shared memory, the device allows " + std::to_string(dev.smem_optin)};
    }
    // Work items pulled from a counter by the persistent warps: per (row, strip) the pair of units (u, v) -- v' needs u's
    // blended field (df.cpp:437), which the u unit leaves in the warp's shared-memory line buffer for the v unit that
    // follows it -- and the unit w as an item of its own.
    std::vector<ZUnit>& units = S.units;
    const int nstrips = (W + strip - 1) / strip;
    struct Item { int j, si, cost; };
    std::vector<Item> items;
    for (int j = 0; j < Ny; ++j)
        for (int si = 0; si < nstrips; ++si) items.push_back(Item{j, si, 0});
    auto make_unit = [&](const Item& it, int f) {
        const int N = P.f[f].N_z_row[it.j];
        const ZPad zp = zpad(N, ZKc);
        ZUnit u{};
        u.j = it.j; u.f = f;
        u.nchunk = zp.nchunk;
        if (Z.zmode == 1) { u.cbytes = 16 * (int)sizeof(double); u.coff16 = (int)((pptr[N] + zp.clen - 16) / 16); }
        else { u.cbytes = zp.clen * (int)sizeof(double); u.coff16 = (int)(pptr[N] / 16); }
        const FieldDev& F = S.D.f[f];
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
    if (Z.zmode == 1) {
        // one record per (row, field): the half-width's parameter line + the row's epilogue constants
        S.unit_par.assign((size_t)Ny * 3 * (16 + ROWC), 0.0);
        for (int j = 0; j < Ny; ++j)
            for (int f = 0; f < 3; ++f) {
                const int N = P.f[f].N_z_row[j];
                const int clen = zpad(N, ZKc).clen;
                double* q = S.unit_par.data() + ((size_t)j * 3 + f) * (16 + ROWC);
                std::copy(pvals.begin() + pptr[N] + clen - 16, pvals.begin() + pptr[N] + clen, q);
                std::copy(S.rowc.begin() + (size_t)j * ROWC, S.rowc.begin() + (size_t)(j + 1) * ROWC, q + 16);
            }
    }
    Z.n_uv = (int)items.size();
    Z.n_items = 2 * (int)items.size();
    return true;
}

// ---- noise tables (include/dfb_rng_spec.h) ----
void plan_noise(const Plan& P, StepPlan& S) {
    const int Ny = P.Ny, NzG = P.NzG;
    int max_np = 1;
    for (int f = 0; f < 3; ++f) {
        const FieldDev& F = S.D.f[f];
        for (int kind = 0; kind < 2; ++kind) {
            NoiseTable A{};
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
                        A.off.push_back((int)(2 * qa - ea) + pc[2]); A.np.push_back((int)(qb - qa + 1));
                        A.jump.push_back(pcg_jump(4u * (uint64_t)qa, 1u));
                        if (wraps) A.win.push_back(make_int4(r, pc[2], pc[2] + pc[1] - pc[0], 0));
                    }
                }
                if (wraps && A.off.size() > 65535u) throw Error{DFB_ERR_ARG, "periodic_z: too many padded rows for the noise kernel's grid"};
            } else if (!P.periodic) {      // periodic_z: the z filter reads no raw noise, array 1 is not drawn
                const int M = F.Nz_max;
                A.npairs = (uint64_t)Ny * (uint64_t)M;
                const bool touches = (P.k0 - M < 0) || (P.k1 + M > NzG);
                if (M > 0 && touches)
                    for (int j = 0; j < Ny; ++j) {
                        A.off.push_back(0); A.np.push_back(M);
                        A.jump.push_back(pcg_jump(4u * (uint64_t)j * (uint64_t)M, 1u));
                    }
            }
            for (int v : A.np) max_np = std::max(max_np, v);
            if (A.off.empty()) continue;                 // a halo that no window reaches is not drawn
            NoiseArray& a = S.np.a[S.np.n_arrays++];
            a.n_seg = (int)A.off.size(); a.kind = kind; a.field = f;
            S.noise.push_back(std::move(A));
        }
    }
    S.slot_jump.resize(max_np);
    for (int t = 0; t < max_np; ++t) S.slot_jump[t] = pcg_jump(4u * (uint64_t)t, 1u);
    S.np.max_np = max_np;
    S.np.stride = pcg_jump(4u * (uint64_t)NOISE_THREADS, 1u);      // the 4*NOISE_THREADS draws between two pairs of one thread
    S.np.chunks = (max_np + NOISE_THREADS * NOISE_PAIRS - 1) / (NOISE_THREADS * NOISE_PAIRS);
}

}  // namespace

StepPlan plan_step(const Plan& P, int NP, const DeviceLimits& dev, const Overrides& ovr) {
    StepPlan S;
    PlaneDev& D = S.D;
    const int Ny = P.Ny, W = P.Nz(), NzG = P.NzG;
    D.Ny = Ny; D.W = W; D.NzG = NzG; D.k0 = P.k0;
    D.P = NP; D.ps_cells = (size_t)Ny * W;
    S.tuned = (P.kernel_variant == 0) && P.f[0].row_uniform && P.f[1].row_uniform && P.f[2].row_uniform;

    // ---- per-row epilogue constants, reference expressions (df.cpp:425-438, 474) ----
    S.rowc.assign((size_t)Ny * ROWC, 0.0);
    for (int j = 0; j < Ny; ++j) {
        double q[8];
        for (int i = 0; i < 8; ++i) q[i] = P.rows[(size_t)i * Ny + j];
        epilogue_consts(q, &S.rowc[(size_t)j * ROWC]);
    }
    for (int f = 0; f < 3; ++f) {
        const FieldPlan& FP = P.f[f];
        FieldDev& F = D.f[f];
        F.Ny_max = FP.Ny_max; F.Nz_max = FP.Nz_max;
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
    }
    if (S.tuned && !plan_z(P, dev, ovr, S)) {
        S.tuned = false;
        S.zp = ZParams{}; S.coef_pad.clear(); S.coef_pad_ptr.clear();
    }
    if (S.tuned) plan_y(P, NP, dev, ovr, S);
    plan_noise(P, S);
    return S;
}

void fill_noise_states(NoiseParams& np, const uint64_t* npairs, uint64_t seed, int plane_id, int nplanes, int64_t step) {
    for (int n = 0; n < np.n_arrays; ++n)
        for (int p = 0; p < nplanes; ++p) {
            const uint64_t inc = noise_inc((int64_t)plane_id + p, np.a[n].field, np.a[n].kind);
            np.pstate[p][n] = noise_step_state(seed, inc, step, npairs[n]);
            np.pinc[p][n] = inc;
        }
}

}  // namespace dfb
