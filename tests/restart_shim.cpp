// tests/restart_shim.cpp -- C entry points over the restart file's host code (csrc/restart.cpp) for tests/test_restart_format.py.
// Linked with restart.cpp and csrc/setup.cpp alone, against no CUDA library: that it links at all shows the format makes no CUDA call.
// A header travels as the int64 values of dfb_restart_info (include/dfb200.h), in that order; its Lt[3], corr_tsteps[65] and library
// version travel beside it.
#include <cstdio>
#include <cstring>
#include <string>
#include "restart.hpp"

using namespace dfb;

namespace {

rst::Header header_from(const int64_t* v, const double* Lt, const int64_t* tsteps, const char* version) {
    rst::Header h;
    h.lib_version = version ? version : "";
    h.Ny = (int32_t)v[1]; h.NzG = (int32_t)v[2]; h.plane0 = (int32_t)v[3]; h.nplanes = (int32_t)v[4]; h.seed = (uint64_t)v[5];
    h.periodic = (int32_t)v[6]; h.noise_mode = (int32_t)v[7]; h.step = v[8]; h.sections = (uint32_t)v[9]; h.fingerprint = (uint64_t)v[11];
    for (int f = 0; f < 3; ++f) { h.Ny_max[f] = (int32_t)v[12 + f]; h.Nz_max[f] = (int32_t)v[15 + f]; h.forms[f] = (int32_t)v[18 + f]; }
    h.stats_count = v[21]; h.stats_on = (int32_t)v[22];
    for (int d = 0; d < 3; ++d) h.corr_L[d] = (int32_t)v[23 + d];
    h.corr_count = v[26]; h.corr_on = (int32_t)v[27]; h.n_ring = (int32_t)v[28];
    for (int f = 0; f < 3; ++f) h.Lt[f] = Lt ? Lt[f] : 0.0;
    for (int m = 0; m <= rst::MAX_LT; ++m) h.corr_tsteps[m] = tsteps ? tsteps[m] : 0;
    rst::layout(h);
    return h;
}

std::vector<rst::Record> records_from(int n, const int64_t* r) {
    std::vector<rst::Record> recs(n);
    for (int i = 0; i < n; ++i) {
        const int64_t* x = r + 6 * i;
        recs[i] = rst::Record{(int32_t)x[0], (int32_t)x[1], (int32_t)x[2], (int32_t)x[3], x[4], (uint64_t)x[5]};
    }
    return recs;
}

int failed(const Error& e, char* err, int errlen) {
    std::snprintf(err, (size_t)errlen, "%d %s", e.code, e.msg.c_str());
    return e.code;
}

}  // namespace

extern "C" {

// fingerprint of the plan dfb_create would build from cfg; 0 with err = "code msg" on a refused config
uint64_t rs_fingerprint(const dfb_config* cfg, char* err, int errlen) {
    try {
        Plan P;
        build_plan(*cfg, P);
        return rst::fingerprint(P);
    } catch (const Error& e) {
        failed(e, err, errlen);
        return 0;
    }
}

// encode -> decode of a header: out = its dfb_restart_info values, Lt_out, tsteps_out, version_out (64 bytes)
int rs_roundtrip(const int64_t* v, const double* Lt, const int64_t* tsteps, const char* version, int64_t* out, double* Lt_out,
                 int64_t* tsteps_out, char* version_out, char* err, int errlen) {
    try {
        std::vector<unsigned char> b(rst::HEADER_BYTES);
        rst::encode_header(header_from(v, Lt, tsteps, version), b.data());
        const rst::Header h = rst::decode_header(b.data());
        const std::vector<int64_t> vals = rst::info_values(h, (int)v[10]);
        std::memcpy(out, vals.data(), vals.size() * sizeof(int64_t));
        for (int f = 0; f < 3; ++f) Lt_out[f] = h.Lt[f];
        for (int m = 0; m <= rst::MAX_LT; ++m) tsteps_out[m] = h.corr_tsteps[m];
        std::snprintf(version_out, 64, "%s", h.lib_version.c_str());
        return 0;
    } catch (const Error& e) {
        return failed(e, err, errlen);
    }
}

long long rs_offset(const int64_t* v, int section, int comp, int plane, int j, int k) {
    return (long long)rst::segment_offset(header_from(v, nullptr, nullptr, nullptr), section, comp, plane, j, k);
}

long long rs_file_bytes(const int64_t* v) { return (long long)header_from(v, nullptr, nullptr, nullptr).file_bytes; }

// records [n][6] = plane0, nplanes, k0, k1, step, fingerprint; 0 = covered, 1 = msg holds the reason
int rs_coverage(const int64_t* v, int n, const int64_t* recs, int p0, int p1, int k0, int k1, char* msg, int msglen) {
    const std::string m = rst::check_coverage(header_from(v, nullptr, nullptr, nullptr), records_from(n, recs), p0, p1, k0, k1);
    std::snprintf(msg, (size_t)msglen, "%s", m.c_str());
    return m.empty() ? 0 : 1;
}

// one writer's save: record[6] as above; blocks [nb][6] = section, comp, plane, nrows, width, k0, with their rows back to back in data
int rs_save(const char* path, const int64_t* v, const int64_t* record, int nb, const int* blocks, double* data, char* err, int errlen) {
    try {
        const rst::Header h = header_from(v, nullptr, nullptr, "restart shim");
        std::vector<rst::Block> B;
        size_t at = 0;
        for (int i = 0; i < nb; ++i) {
            const int* b = blocks + 6 * i;
            B.push_back(rst::Block{b[0], b[1], b[2], data + at, b[3], b[4], b[5]});
            at += (size_t)b[3] * b[4];
        }
        rst::save(path, h, records_from(1, record)[0], B);
        return 0;
    } catch (const Error& e) {
        return failed(e, err, errlen);
    }
}

// header values (dfb_restart_info order) and records [cap][6] of a file; returns the record count, or -code with err
int rs_read(const char* path, int64_t* out, int64_t* recs, int cap, char* err, int errlen) {
    try {
        std::vector<rst::Record> R;
        const rst::Header h = rst::read_header(path, &R);
        const std::vector<int64_t> vals = rst::info_values(h, (int)R.size());
        std::memcpy(out, vals.data(), vals.size() * sizeof(int64_t));
        for (int i = 0; i < (int)R.size() && i < cap; ++i) {
            const int64_t x[6] = {R[i].plane0, R[i].nplanes, R[i].k0, R[i].k1, R[i].step, (int64_t)R[i].fingerprint};
            std::memcpy(recs + 6 * i, x, sizeof(x));
        }
        return (int)R.size();
    } catch (const Error& e) {
        return -failed(e, err, errlen);
    }
}

}  // extern "C"
