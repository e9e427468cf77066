// tests/filter_shape_fp_shim.cpp -- the restart fingerprint (csrc/restart.cpp) of the plan dfb_create builds from cfg, in either filter
// shape, for tests/test_filter_shape_host.py.  Linked against no CUDA library; a refusal returns its code with err = "code msg".
#include <cstdio>
#include "restart.hpp"

using namespace dfb;

extern "C" {

int fs_fingerprint(const dfb_config* cfg, int shape, uint64_t* fp, char* err, int errlen) {
    try {
        Plan P;
        build_plan(*cfg, P);
        P.filter_shape = shape;
        build_coef_table(P);
        *fp = rst::fingerprint(P);
        return 0;
    } catch (const Error& e) {
        std::snprintf(err, (size_t)errlen, "%d %s", e.code, e.msg.c_str());
        return e.code;
    }
}

}  // extern "C"
