// csrc/restart.cpp -- the restart file: header, fingerprint, writer records and file I/O (restart.hpp).  No CUDA call.
#include "restart.hpp"

#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <cerrno>
#include <cstring>

namespace dfb {
namespace rst {

namespace {

const char MAGIC[8] = {'D', 'F', 'B', 'R', 'S', 'T', 'R', 'T'};

Error io(const std::string& msg) { return Error{DFB_ERR_IO, msg}; }

// explicit little-endian encoding, whatever the host's byte order
struct Out {
    unsigned char* p;
    size_t at = 0;
    void u32(uint32_t v) { for (int i = 0; i < 4; ++i) p[at++] = (unsigned char)(v >> (8 * i)); }
    void u64(uint64_t v) { for (int i = 0; i < 8; ++i) p[at++] = (unsigned char)(v >> (8 * i)); }
    void i32(int32_t v) { u32((uint32_t)v); }
    void i64(int64_t v) { u64((uint64_t)v); }
    void f64(double v) { uint64_t b; std::memcpy(&b, &v, 8); u64(b); }
    void bytes(const void* s, size_t n) { std::memcpy(p + at, s, n); at += n; }
};
struct In {
    const unsigned char* p;
    size_t at = 0;
    uint32_t u32() { uint32_t v = 0; for (int i = 0; i < 4; ++i) v |= (uint32_t)p[at++] << (8 * i); return v; }
    uint64_t u64() { uint64_t v = 0; for (int i = 0; i < 8; ++i) v |= (uint64_t)p[at++] << (8 * i); return v; }
    int32_t i32() { return (int32_t)u32(); }
    int64_t i64() { return (int64_t)u64(); }
    double f64() { uint64_t b = u64(); double v; std::memcpy(&v, &b, 8); return v; }
};

// 64-bit hash of a canonical sequence of 64-bit words (each value widened to one word, doubles by their bits)
struct Hash {
    uint64_t h = 0xcbf29ce484222325ull;
    void word(uint64_t w) {
        h ^= w;
        h *= 0x9e3779b97f4a7c15ull;
        h ^= h >> 31;
    }
    void f64(double v) { uint64_t b; std::memcpy(&b, &v, 8); word(b); }
    void ints(const std::vector<int>& v) { word(v.size()); for (int x : v) word((uint64_t)(int64_t)x); }
};

int64_t row_width(const Header& h, int section) {
    return section >= SEC_CORR_Z && section <= SEC_CORR_T ? h.corr_L[section - SEC_CORR_Z] + 1 : h.NzG;
}

struct Fd {
    int fd = -1;
    ~Fd() { if (fd >= 0) ::close(fd); }
};

void lock(int fd, short type, const char* path) {
    struct flock l;
    std::memset(&l, 0, sizeof(l));
    l.l_type = type;
    l.l_whence = SEEK_SET;
    l.l_start = 0;
    l.l_len = DATA_AT;                      // the header and the record table
    while (fcntl(fd, F_OFD_SETLKW, &l) != 0)
        if (errno != EINTR) throw io(std::string("cannot lock ") + path + ": " + std::strerror(errno));
}

void pwrite_all(int fd, const void* buf, size_t n, int64_t at, const char* path) {
    const char* p = static_cast<const char*>(buf);
    while (n) {
        const ssize_t w = ::pwrite(fd, p, n, (off_t)at);
        if (w < 0 && errno == EINTR) continue;
        if (w <= 0) throw io(std::string("cannot write ") + path + ": " + std::strerror(errno));
        p += w; n -= (size_t)w; at += w;
    }
}

// false on a short read (end of file)
bool pread_all(int fd, void* buf, size_t n, int64_t at, const char* path) {
    char* p = static_cast<char*>(buf);
    while (n) {
        const ssize_t r = ::pread(fd, p, n, (off_t)at);
        if (r < 0 && errno == EINTR) continue;
        if (r < 0) throw io(std::string("cannot read ") + path + ": " + std::strerror(errno));
        if (r == 0) return false;
        p += r; n -= (size_t)r; at += r;
    }
    return true;
}

std::vector<unsigned char> encode_records(const std::vector<Record>& recs) {
    std::vector<unsigned char> b(8 + (size_t)MAX_RECORDS * RECORD_BYTES, 0);
    Out o{b.data()};
    o.u32((uint32_t)recs.size()); o.u32(0);
    for (const Record& r : recs) {
        const size_t at = o.at;
        o.i32(r.plane0); o.i32(r.nplanes); o.i32(r.k0); o.i32(r.k1); o.i64(r.step); o.u64(r.fingerprint);
        o.at = at + RECORD_BYTES;
    }
    return b;
}

std::vector<Record> decode_records(const unsigned char* b) {
    In in{b};
    const uint32_t n = in.u32();
    in.u32();
    if (n > (uint32_t)MAX_RECORDS) throw io("corrupt writer record table (" + std::to_string(n) + " records)");
    std::vector<Record> recs(n);
    for (Record& r : recs) {
        const size_t at = in.at;
        r.plane0 = in.i32(); r.nplanes = in.i32(); r.k0 = in.i32(); r.k1 = in.i32(); r.step = in.i64(); r.fingerprint = in.u64();
        in.at = at + RECORD_BYTES;
    }
    return recs;
}

// the header's bytes without the last writer's kernel forms: equal for every writer of one checkpoint
std::vector<unsigned char> identity(Header h) {
    h.forms[0] = h.forms[1] = h.forms[2] = 0;
    std::vector<unsigned char> b(HEADER_BYTES);
    encode_header(h, b.data());
    return b;
}

std::string range(int a, int b) { return "[" + std::to_string(a) + ", " + std::to_string(b) + ")"; }

}  // namespace

uint64_t fingerprint(const Plan& P) {
    Hash H;
    H.word((uint64_t)P.Ny); H.word((uint64_t)P.NzG); H.word(P.periodic ? 1 : 0);
    for (int f = 0; f < 3; ++f) {
        const FieldPlan& F = P.f[f];
        H.word(F.row_uniform ? 1 : 0);
        if (F.row_uniform) { H.ints(F.N_y_row); H.ints(F.N_z_row); }
        else { H.ints(F.N_y); H.ints(F.N_z); }
        H.f64(F.Lt);
    }
    H.word(P.rows.size());
    for (double v : P.rows) H.f64(v);
    if (!P.Lt_rows.empty()) {                    // per-row time scales: hashed only when set, so a handle without them keeps its fingerprint
        H.word(0x4c745f726f7773ull);             // "Lt_rows"
        H.word(P.Lt_rows.size());
        for (double v : P.Lt_rows) H.f64(v);
    }
    if (P.filter_shape != DFB_FILTER_EXPONENTIAL) {   // hashed only when Gaussian, so an exponential handle keeps its fingerprint
        H.word(0x67617573736961ull);             // "gaussia"
        H.word((uint64_t)P.filter_shape);
    }
    if (P.cells_hash) {                          // per-cell profiles: hashed only when set, so a handle without them keeps its fingerprint
        H.word(0x70726f66696c6573ull);           // "profiles"
        H.word(P.cells_hash);
    }
    return H.h;
}

uint64_t hash_f64(const double* v, size_t n) {
    Hash H;
    H.word(n);
    for (size_t i = 0; i < n; ++i) H.f64(v[i]);
    return H.h;
}

void layout(Header& h) {
    const int64_t plane = (int64_t)h.Ny * h.NzG * 8;
    int64_t at = DATA_AT;
    for (int s = 0; s < N_SECTIONS; ++s) h.off[s] = 0;
    h.off[SEC_STATE] = at; at += 3 * h.nplanes * plane;
    if (h.sections & DFB_RESTART_STATS) { h.off[SEC_STATS] = at; at += 6 * h.nplanes * plane; }
    if (h.sections & DFB_RESTART_CORR) {
        for (int d = 0; d < 3; ++d)
            if (h.corr_L[d]) { h.off[SEC_CORR_Z + d] = at; at += (int64_t)h.nplanes * 3 * h.Ny * (h.corr_L[d] + 1) * 8; }
        if (h.n_ring) { h.off[SEC_RING] = at; at += (int64_t)h.n_ring * h.nplanes * 3 * plane; }
    }
    h.file_bytes = at;
}

void encode_header(const Header& h, unsigned char* out) {
    std::memset(out, 0, HEADER_BYTES);
    Out o{out};
    o.bytes(MAGIC, 8);
    o.u32(VERSION); o.u32(HEADER_BYTES);
    char lv[64] = {};
    std::strncpy(lv, h.lib_version.c_str(), 63);
    o.bytes(lv, 64);
    o.i32(h.Ny); o.i32(h.NzG); o.i32(h.plane0); o.i32(h.nplanes); o.i32(h.periodic); o.i32(h.noise_mode);
    o.u64(h.seed); o.i64(h.step);
    for (int f = 0; f < 3; ++f) { o.i32(h.Ny_max[f]); o.i32(h.Nz_max[f]); o.f64(h.Lt[f]); }
    for (int i = 0; i < 3; ++i) o.i32(h.forms[i]);
    o.u64(h.fingerprint); o.u32(h.sections);
    o.i64(h.stats_count); o.i32(h.stats_on);
    for (int d = 0; d < 3; ++d) o.i32(h.corr_L[d]);
    o.i32(h.corr_on); o.i32(h.n_ring); o.i64(h.corr_count);
    for (int m = 0; m <= MAX_LT; ++m) o.i64(h.corr_tsteps[m]);
    for (int s = 0; s < N_SECTIONS; ++s) o.i64(h.off[s]);
    o.i64(h.file_bytes);
    o.i32(h.filter_shape);
    o.u64(h.profiles);
}

Header decode_header(const unsigned char* in_) {
    In in{in_};
    if (std::memcmp(in_, MAGIC, 8) != 0) throw io("not a restart file of this library (bad magic)");
    in.at = 8;
    const uint32_t version = in.u32();
    if (version != VERSION) throw io("restart file format version " + std::to_string(version) + ", this library reads version " + std::to_string(VERSION));
    if (in.u32() != (uint32_t)HEADER_BYTES) throw io("corrupt restart header (size field)");
    Header h;
    char lv[65] = {};
    std::memcpy(lv, in_ + in.at, 64); in.at += 64;
    h.lib_version = lv;
    h.Ny = in.i32(); h.NzG = in.i32(); h.plane0 = in.i32(); h.nplanes = in.i32(); h.periodic = in.i32(); h.noise_mode = in.i32();
    h.seed = in.u64(); h.step = in.i64();
    for (int f = 0; f < 3; ++f) { h.Ny_max[f] = in.i32(); h.Nz_max[f] = in.i32(); h.Lt[f] = in.f64(); }
    for (int i = 0; i < 3; ++i) h.forms[i] = in.i32();
    h.fingerprint = in.u64(); h.sections = in.u32();
    h.stats_count = in.i64(); h.stats_on = in.i32();
    for (int d = 0; d < 3; ++d) h.corr_L[d] = in.i32();
    h.corr_on = in.i32(); h.n_ring = in.i32(); h.corr_count = in.i64();
    for (int m = 0; m <= MAX_LT; ++m) h.corr_tsteps[m] = in.i64();
    int64_t off[N_SECTIONS];
    for (int s = 0; s < N_SECTIONS; ++s) off[s] = in.i64();
    const int64_t bytes = in.i64();
    h.filter_shape = in.i32();
    h.profiles = in.u64();
    if (h.Ny <= 0 || h.NzG <= 0 || h.nplanes <= 0 || h.nplanes > DFB_MAXP || h.corr_L[2] < 0 || h.corr_L[2] > MAX_LT || h.n_ring < 0 ||
        h.n_ring > h.corr_L[2] || h.filter_shape < 0 || h.filter_shape > DFB_FILTER_GAUSSIAN || h.corr_L[0] < 0 || h.corr_L[0] >= h.NzG || h.corr_L[1] < 0 || h.corr_L[1] >= h.Ny)
        throw io("corrupt restart header (sizes)");
    layout(h);
    if (bytes != h.file_bytes || std::memcmp(off, h.off, sizeof(off)) != 0) throw io("corrupt restart header (section offsets)");
    return h;
}

std::vector<int64_t> info_values(const Header& h, int n_records) {
    std::vector<int64_t> v = {(int64_t)VERSION, h.Ny, h.NzG, h.plane0, h.nplanes, (int64_t)h.seed, h.periodic, h.noise_mode, h.step,
                              (int64_t)h.sections, n_records, (int64_t)h.fingerprint};
    for (int f = 0; f < 3; ++f) v.push_back(h.Ny_max[f]);
    for (int f = 0; f < 3; ++f) v.push_back(h.Nz_max[f]);
    for (int i = 0; i < 3; ++i) v.push_back(h.forms[i]);
    v.push_back(h.stats_count); v.push_back(h.stats_on);
    for (int d = 0; d < 3; ++d) v.push_back(h.corr_L[d]);
    v.push_back(h.corr_count); v.push_back(h.corr_on); v.push_back(h.n_ring); v.push_back(h.file_bytes);
    return v;
}

int64_t segment_offset(const Header& h, int section, int comp, int plane, int j, int k) {
    const int64_t P = h.nplanes, Ny = h.Ny, w = row_width(h, section);
    int64_t row = 0;
    switch (section) {
        case SEC_STATE: row = ((int64_t)comp * P + plane) * Ny + j; break;
        case SEC_STATS: row = ((int64_t)plane * 6 + comp) * Ny + j; break;
        case SEC_RING: row = ((((int64_t)(comp / 3)) * P + plane) * 3 + comp % 3) * Ny + j; break;
        default: row = ((int64_t)plane * 3 + comp) * Ny + j; break;
    }
    return h.off[section] + (row * w + k) * 8;
}

std::string check_coverage(const Header& h, const std::vector<Record>& recs, int p0, int p1, int k0, int k1) {
    for (int p = p0; p < p1; ++p) {
        std::vector<std::pair<int, int>> cov;
        for (const Record& r : recs) {
            if (p < r.plane0 || p >= r.plane0 + r.nplanes || r.k1 <= k0 || r.k0 >= k1) continue;
            if (r.step != h.step || r.fingerprint != h.fingerprint)
                return "stale writer record for columns " + range(r.k0, r.k1) + " of planes " + range(r.plane0, r.plane0 + r.nplanes) + ": " +
                       (r.step != h.step ? "step " + std::to_string(r.step) + ", the header's is " + std::to_string(h.step)
                                         : std::string("its fingerprint differs from the header's"));
            cov.push_back({r.k0, r.k1});
        }
        std::sort(cov.begin(), cov.end());
        int at = k0;
        for (const auto& c : cov) {
            if (c.first > at) break;
            at = std::max(at, c.second);
        }
        if (at < k1) {
            int end = k1;
            for (const auto& c : cov) if (c.first > at) { end = std::min(end, c.first); break; }
            return "no writer record covers columns " + range(at, end) + " of plane " + std::to_string(p) +
                   " (a writer of this checkpoint did not finish its save, or the file belongs to another checkpoint)";
        }
    }
    return "";
}

void save(const char* path, const Header& h, const Record& mine, const std::vector<Block>& blocks) {
    Fd f;
    f.fd = ::open(path, O_RDWR | O_CREAT | O_CLOEXEC, 0644);
    if (f.fd < 0) throw io(std::string("cannot open ") + path + " for writing: " + std::strerror(errno));
    std::vector<unsigned char> head(HEADER_BYTES), table(8 + (size_t)MAX_RECORDS * RECORD_BYTES);
    const std::vector<unsigned char> me = identity(h);
    // the record table of the file as it stands, if it belongs to this checkpoint (same step, same identity); else empty
    auto current_records = [&]() -> std::vector<Record> {
        if (!pread_all(f.fd, head.data(), head.size(), 0, path) || !pread_all(f.fd, table.data(), table.size(), RECORDS_AT, path)) return {};
        try {
            if (identity(decode_header(head.data())) != me) return {};
            return decode_records(table.data());
        } catch (const Error&) {
            return {};
        }
    };
    lock(f.fd, F_WRLCK, path);
    try {
        const std::vector<Record> recs = current_records();
        std::vector<unsigned char> out(HEADER_BYTES);
        encode_header(h, out.data());
        pwrite_all(f.fd, out.data(), out.size(), 0, path);
        const std::vector<unsigned char> t = encode_records(recs);
        pwrite_all(f.fd, t.data(), t.size(), RECORDS_AT, path);
        if (::ftruncate(f.fd, (off_t)h.file_bytes) != 0) throw io(std::string("cannot size ") + path + ": " + std::strerror(errno));
    } catch (...) {
        lock(f.fd, F_UNLCK, path);
        throw;
    }
    lock(f.fd, F_UNLCK, path);

    for (const Block& b : blocks) {
        const int64_t w = row_width(h, b.section);
        if (b.k0 == 0 && b.width == w) {          // whole rows: one contiguous range
            pwrite_all(f.fd, b.rows, (size_t)b.nrows * b.width * 8, segment_offset(h, b.section, b.comp, b.plane, 0, 0), path);
        } else {
            for (int j = 0; j < b.nrows; ++j)
                pwrite_all(f.fd, b.rows + (size_t)j * b.width, (size_t)b.width * 8, segment_offset(h, b.section, b.comp, b.plane, j, b.k0), path);
        }
    }

    lock(f.fd, F_WRLCK, path);
    try {
        if (!pread_all(f.fd, head.data(), head.size(), 0, path) || identity(decode_header(head.data())) != me)
            throw io(std::string("another writer replaced the header of ") + path + " during this save (writers of one file must save the same step)");
        std::vector<Record> recs = current_records();
        auto same = [&](const Record& r) { return r.plane0 == mine.plane0 && r.nplanes == mine.nplanes && r.k0 == mine.k0 && r.k1 == mine.k1; };
        recs.erase(std::remove_if(recs.begin(), recs.end(), same), recs.end());
        if ((int)recs.size() >= MAX_RECORDS) throw io(std::string("the writer record table of ") + path + " is full (64 writers)");
        recs.push_back(mine);
        const std::vector<unsigned char> t = encode_records(recs);
        pwrite_all(f.fd, t.data(), t.size(), RECORDS_AT, path);
    } catch (...) {
        lock(f.fd, F_UNLCK, path);
        throw;
    }
    lock(f.fd, F_UNLCK, path);
}

Header read_header(const char* path, std::vector<Record>* recs) {
    Fd f;
    f.fd = ::open(path, O_RDONLY | O_CLOEXEC);
    if (f.fd < 0) throw io(std::string("cannot open ") + path + ": " + std::strerror(errno));
    std::vector<unsigned char> head(HEADER_BYTES), table(8 + (size_t)MAX_RECORDS * RECORD_BYTES);
    if (!pread_all(f.fd, head.data(), head.size(), 0, path)) throw io(std::string(path) + " is too short for a restart header");
    const Header h = decode_header(head.data());
    struct stat st;
    if (fstat(f.fd, &st) != 0) throw io(std::string("cannot stat ") + path + ": " + std::strerror(errno));
    if ((int64_t)st.st_size != h.file_bytes)
        throw io(std::string(path) + " has " + std::to_string((long long)st.st_size) + " bytes, its header describes " + std::to_string(h.file_bytes) +
                 " (truncated or still being written)");
    if (recs) {
        if (!pread_all(f.fd, table.data(), table.size(), RECORDS_AT, path)) throw io(std::string(path) + " is too short for its record table");
        *recs = decode_records(table.data());
    }
    return h;
}

void read_blocks(const char* path, const Header& h, const std::vector<Block>& blocks) {
    Fd f;
    f.fd = ::open(path, O_RDONLY | O_CLOEXEC);
    if (f.fd < 0) throw io(std::string("cannot open ") + path + ": " + std::strerror(errno));
    for (const Block& b : blocks) {
        const int64_t w = row_width(h, b.section);
        bool ok = true;
        if (b.k0 == 0 && b.width == w)
            ok = pread_all(f.fd, b.rows, (size_t)b.nrows * b.width * 8, segment_offset(h, b.section, b.comp, b.plane, 0, 0), path);
        else
            for (int j = 0; ok && j < b.nrows; ++j)
                ok = pread_all(f.fd, b.rows + (size_t)j * b.width, (size_t)b.width * 8, segment_offset(h, b.section, b.comp, b.plane, j, b.k0), path);
        if (!ok) throw io(std::string(path) + " ended inside a section (truncated)");
    }
}

}  // namespace rst
}  // namespace dfb
