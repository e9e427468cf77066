// csrc/facemap.cpp -- face maps of the CFD hand-off (facemap.hpp).  No CUDA call: the taps are host arrays the caller uploads.
//
// DFB_MAP_POINT: bilinear interpolation at the face centre between the cell centres write_csv prints (Plan::csv_yc, csv_zc).
// DFB_MAP_AREA:  the average over the face rectangle of the cells [vert_y[j], vert_y[j+1]) x [vert_z[k], vert_z[k+1]).
#include "facemap.hpp"
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <limits>
#include <map>
#include <string>
#include <utility>

namespace dfb {

namespace {

Error arg(const std::string& m) { return Error{DFB_ERR_ARG, m}; }

std::string face_str(int i, double y, double z) {
    char b[96];
    std::snprintf(b, sizeof(b), "face %d at (y, z) = (%.9g, %.9g)", i, y, z);
    return b;
}

// cell of v (vertices, increasing) holding x, clamped to [0, N): dfb_face_map's rule
int cell_of(const std::vector<double>& v, double x) {
    const int N = (int)v.size() - 1;
    const int c = (int)(std::upper_bound(v.begin(), v.end(), x) - v.begin()) - 1;
    return std::min(std::max(c, 0), N - 1);
}

bool increasing(const std::vector<double>& v) {
    for (size_t i = 1; i < v.size(); ++i)
        if (!(v[i] > v[i - 1])) return false;
    return true;
}

// Linear weights between the nodes x[0..N) (increasing) at p, clamped beyond the end nodes: up to two (node, weight) pairs
// (node, 1 - s), (node + 1, s).  The second weight is 0 when p sits on or beyond a node.
void lin(const std::vector<double>& x, double p, int c[2], double t[2]) {
    const int N = (int)x.size();
    if (p <= x[0]) { c[0] = c[1] = 0; t[0] = 1; t[1] = 0; return; }
    if (p >= x[N - 1]) { c[0] = c[1] = N - 1; t[0] = 1; t[1] = 0; return; }
    const int j = (int)(std::upper_bound(x.begin(), x.end(), p) - x.begin()) - 1;   // x[j] <= p < x[j+1]
    const double s = (p - x[j]) / (x[j + 1] - x[j]);
    c[0] = j; c[1] = j + 1; t[0] = 1 - s; t[1] = s;
}

// Lengths of the overlaps of [lo, hi) with the cells [v[c], v[c+1]) of the vertices v; open_ends: the first cell reaches down to
// -inf and the last up to +inf (a part of the interval outside the plane counts toward the nearest edge cell).
void overlaps(const std::vector<double>& v, double lo, double hi, bool open_ends, std::vector<std::pair<int, double>>& out) {
    const int N = (int)v.size() - 1;
    const int first = cell_of(v, lo);
    const int last = std::min(std::max((int)(std::lower_bound(v.begin(), v.end(), hi) - v.begin()) - 1, 0), N - 1);
    for (int c = first; c <= last; ++c) {
        const double a = (open_ends && c == 0) ? lo : std::max(lo, v[c]);
        const double b = (open_ends && c == N - 1) ? hi : std::min(hi, v[c + 1]);
        if (b > a) out.push_back({c, b - a});
    }
}

// A face edge within rounding of a vertex is put on it, so that a face computed from a cell's vertices is exactly that cell
double snap(const std::vector<double>& v, double x, double extent) {
    const double tol = 1e-9 * extent + 8 * DBL_EPSILON * std::fabs(x);
    const auto it = std::lower_bound(v.begin(), v.end(), x);
    if (it != v.end() && *it - x <= tol) return *it;
    if (it != v.begin() && x - *(it - 1) <= tol) return *(it - 1);
    return x;
}

}  // namespace

FaceMap build_face_map(const Plan& P, int kind, int n, const double* yf, const double* zf, const double* hy, const double* hz,
                       int own0, int own1, int flags) {
    if (kind != DFB_MAP_POINT && kind != DFB_MAP_AREA) throw arg("kind must be DFB_MAP_POINT or DFB_MAP_AREA");
    if (flags & ~DFB_MAP_WALL_ZERO) throw arg("flags must be 0 or DFB_MAP_WALL_ZERO");
    if ((flags & DFB_MAP_WALL_ZERO) && kind != DFB_MAP_POINT) throw arg("DFB_MAP_WALL_ZERO applies to DFB_MAP_POINT maps only");
    if (n < 0) throw arg("n must be >= 0");
    if (n > 0 && (!yf || !zf)) throw arg("yf / zf is NULL");
    if (kind == DFB_MAP_AREA && n > 0 && (!hy || !hz)) throw arg("a DFB_MAP_AREA map needs the face extents hy and hz");
    if (kind == DFB_MAP_POINT && (hy || hz)) throw arg("a DFB_MAP_POINT map takes no face extents (hy, hz must be NULL)");
    if (own0 == 0 && own1 == 0) { own0 = P.k0; own1 = P.k1; }
    if (own0 < P.k0 || own1 > P.k1 || own0 >= own1)
        throw arg("own columns [" + std::to_string(own0) + ", " + std::to_string(own1) + ") must be a non-empty part of this handle's slab [" +
                  std::to_string(P.k0) + ", " + std::to_string(P.k1) + ")");
    const std::vector<double>&yc = P.csv_yc, &zc = P.csv_zc, &vy = P.vert_y, &vz = P.vert_z;
    if (kind == DFB_MAP_POINT && !increasing(yc)) throw arg("a DFB_MAP_POINT map needs increasing cell-centre heights (dfb_config.yc)");
    if (kind == DFB_MAP_AREA && !increasing(vy)) throw arg("a DFB_MAP_AREA map needs cells that do not overlap in y (dfb_config.yc, dy)");
    const int NzG = P.NzG, W = P.Nz();
    const double Lz = vz[NzG] - vz[0];

    FaceMap M;
    M.kind = kind; M.flags = flags; M.n = n;
    M.served.assign(n, 0);
    if (kind == DFB_MAP_POINT) { M.idx.assign((size_t)n * 4, -1); M.w.assign((size_t)n * 4, 0.0); }
    else M.ptr.assign((size_t)n + 1, 0);

    std::vector<int> tj, tk;          // taps of one face: global row, column, weight
    std::vector<double> tw;
    std::vector<std::pair<int, double>> oy, oz;
    for (int i = 0; i < n; ++i) {
        const double y = yf[i], z = zf[i];
        if (!std::isfinite(y) || !std::isfinite(z)) throw arg(face_str(i, y, z) + ": the coordinates must be finite");
        if (kind == DFB_MAP_AREA && !(std::isfinite(hy[i]) && std::isfinite(hz[i]) && hy[i] > 0 && hz[i] > 0))
            throw arg(face_str(i, y, z) + ": the extents hy, hz must be finite and > 0");
        const int jo = cell_of(vy, y), ko = cell_of(vz, z);     // the cell holding the centre decides who serves the face
        if (ko < own0 || ko >= own1) {
            if (kind == DFB_MAP_AREA) M.ptr[i + 1] = M.ptr[i];
            continue;
        }
        tj.clear(); tk.clear(); tw.clear();
        if (kind == DFB_MAP_POINT) {
            int r[2], c[2];
            double ty[2], tz[2];
            if ((flags & DFB_MAP_WALL_ZERO) && y < yc[0]) {      // linear to 0 at the wall vert_y[0], 0 below it
                r[0] = r[1] = 0;
                ty[0] = y <= vy[0] ? 0.0 : (y - vy[0]) / (yc[0] - vy[0]);
                ty[1] = 0;
            } else {
                lin(yc, y, r, ty);
            }
            if (P.periodic) {                                       // z wraps: column NzG-1 neighbours column 0
                double p = z;
                if (p < vz[0] || p >= vz[NzG]) p -= std::floor((p - vz[0]) / Lz) * Lz;
                if (p < zc[0] || p >= zc[NzG - 1]) {
                    const double left = p < zc[0] ? zc[NzG - 1] - Lz : zc[NzG - 1];
                    const double right = p < zc[0] ? zc[0] : zc[0] + Lz;
                    const double s = (p - left) / (right - left);
                    c[0] = NzG - 1; c[1] = 0; tz[0] = 1 - s; tz[1] = s;
                } else {
                    lin(zc, p, c, tz);
                }
            } else {
                lin(zc, z, c, tz);
            }
            for (int a = 0; a < 2; ++a)
                for (int b = 0; b < 2; ++b) {
                    tj.push_back(r[a]); tk.push_back(c[b]); tw.push_back(ty[a] * tz[b]);
                }
        } else {
            double ylo = y - 0.5 * hy[i], yhi = y + 0.5 * hy[i], zlo = z - 0.5 * hz[i], zhi = z + 0.5 * hz[i];
            ylo = snap(vy, ylo, hy[i]); yhi = snap(vy, yhi, hy[i]); zlo = snap(vz, zlo, hz[i]); zhi = snap(vz, zhi, hz[i]);
            oy.clear(); oz.clear();
            overlaps(vy, ylo, yhi, true, oy);
            if (P.periodic) {                                       // the pieces of [zlo, zhi) in each period, wrapped onto the plane
                if (hz[i] > Lz) throw arg(face_str(i, y, z) + ": an area face is wider than the spanwise-periodic plane");
                std::vector<std::pair<int, double>> piece;
                std::map<int, double> acc;
                const long long m0 = (long long)std::floor((zlo - vz[0]) / Lz), m1 = (long long)std::floor((zhi - vz[0]) / Lz);
                for (long long m = m0; m <= m1; ++m) {
                    const double a = std::max(zlo - m * Lz, vz[0]), b = std::min(zhi - m * Lz, vz[NzG]);
                    if (!(b > a)) continue;
                    piece.clear();
                    overlaps(vz, a, b, false, piece);
                    for (auto& q : piece) acc[q.first] += q.second;
                }
                oz.assign(acc.begin(), acc.end());
            } else {
                overlaps(vz, zlo, zhi, true, oz);
            }
            // weight = overlap area / face area, the face's extents taken as the sums of its overlaps: the weights sum to 1 to
            // rounding whatever the rounding of yf -+ hy/2, and a face equal to a cell gets weight 1 exactly
            double sy = 0, sz = 0;
            for (auto& a : oy) sy += a.second;
            for (auto& b : oz) sz += b.second;
            for (auto& a : oy)
                for (auto& b : oz) {
                    tj.push_back(a.first); tk.push_back(b.first); tw.push_back((a.second / sy) * (b.second / sz));
                }
        }
        // every column a tap of nonzero weight reads must be computed by this handle
        int kmin = NzG, kmax = -1;
        bool bad = false;
        for (size_t t = 0; t < tw.size(); ++t)
            if (tw[t] != 0.0) {
                kmin = std::min(kmin, tk[t]); kmax = std::max(kmax, tk[t]);
                bad |= tk[t] < P.k0 || tk[t] >= P.k1;
            }
        if (bad) {
            const bool seam = P.periodic && kmin == 0 && kmax == NzG - 1 && NzG > 2;
            throw arg(face_str(i, y, z) + " needs columns " + std::to_string(kmin) + ".." + std::to_string(kmax) +
                      (seam ? " (across the periodic seam)" : "") + ", but this handle computes [" + std::to_string(P.k0) + ", " +
                      std::to_string(P.k1) + "): create the slab 16 columns wider on each side (k_begin - 16, k_end + 16) and pass its "
                      "unwidened columns as own_begin, own_end");
        }
        M.served[i] = 1;
        M.n_served += 1;
        const int own_cell = jo * W + (ko - P.k0);
        if (kind == DFB_MAP_POINT) {
            for (int t = 0; t < 4; ++t) {
                M.idx[(size_t)i * 4 + t] = tw[t] != 0.0 ? tj[t] * W + (tk[t] - P.k0) : own_cell;
                M.w[(size_t)i * 4 + t] = tw[t];
            }
        } else {
            for (size_t t = 0; t < tw.size(); ++t)
                if (tw[t] != 0.0) { M.idx.push_back(tj[t] * W + (tk[t] - P.k0)); M.w.push_back(tw[t]); }
            if (M.idx.size() > (size_t)std::numeric_limits<int>::max()) throw arg("more than 2^31 - 1 taps in one map");
            M.ptr[i + 1] = (int)M.idx.size();
        }
    }
    return M;
}

}  // namespace dfb
