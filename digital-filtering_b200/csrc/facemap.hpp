// csrc/facemap.hpp -- face maps of the CFD hand-off (dfb_facemap_create): for each face of a CFD code's inflow boundary, a fixed list
// of (plane cell, weight) taps that dfb_interp_to_cells / dfb_interp_to_host sum on the device.  Host code only (no CUDA call), so
// that tests/test_facemap_host.py checks it through a g++ shim.
#pragma once
#include <vector>
#include "plan.hpp"

namespace dfb {

struct FaceMap {
    int kind = DFB_MAP_POINT, flags = 0, n = 0;
    int n_served = 0;
    std::vector<int> served;          // [n] 0/1
    // DFB_MAP_POINT: 4 taps per face, idx / w [n][4] (an unserved face has idx[4i] = -1).  A tap of weight 0 repeats the face's
    //                first cell, so that it reads nothing the other taps do not.
    // DFB_MAP_AREA:  CSR, taps of face i at [ptr[i], ptr[i+1]) (an unserved face has none).
    // idx is the cell j*W + (k - k0) of the handle's slab; the weights come from the plane's global tables alone, so every slab
    // and every plane of a batch computes the same doubles in the same order.
    std::vector<int> ptr, idx;
    std::vector<double> w;
};

// Builds a map for the handle whose plan is P, serving the faces whose centre lies in a cell of the columns [own0, own1) (0,0: the
// slab [k0, k1)).  hy, hz: face extents (DFB_MAP_AREA only, else nullptr).  Throws dfb::Error (DFB_ERR_ARG) naming the face.
FaceMap build_face_map(const Plan& P, int kind, int n, const double* yf, const double* zf, const double* hy, const double* hz,
                       int own0, int own1, int flags);

}  // namespace dfb
