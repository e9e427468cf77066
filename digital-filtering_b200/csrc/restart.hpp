// csrc/restart.hpp -- the restart file (dfb_save_restart / dfb_load_restart / dfb_restart_info): format, fingerprint, writer records
// and file I/O.  Host code only, no CUDA call (tests/restart_shim.cpp drives it with g++ alone).
//
// File layout, every integer little-endian with the width given, every double an IEEE-754 binary64 in little-endian byte order:
//   [0, 4096)      header (encode_header): magic "DFBRSTRT", format version, library version, geometry, plane range, seed, step,
//                  per-field Ny_max / Nz_max / Lt, the kernel forms of the last writer, the fingerprint, sections and their scalars
//   [4096, 7176)   writer records: u32 count, u32 0, then 64 x 48 bytes {i32 plane0, i32 nplanes, i32 k0, i32 k1, i64 step, u64 fp, 16 x 0}
//   [8192, ...)    sections, each in the plane's GLOBAL layout (any decomposition writes and reads it):
//                  state     filt_old         [3][P][Ny][NzG]
//                  stats     N2 sums          [P][6][Ny][NzG]                      (DFB_RESTART_STATS)
//                  corr z/y/t sums            [P][3][Ny][L_d + 1] for each d with L_d > 0  (DFB_RESTART_CORR)
//                  ring      temporal ring    [n_ring][P][3][Ny][NzG], oldest first         (DFB_RESTART_CORR)
#pragma once
#include <cstdint>
#include <string>
#include <vector>
#include "plan.hpp"

namespace dfb {
namespace rst {

constexpr uint32_t VERSION = 1;
constexpr int HEADER_BYTES = 4096;
constexpr int MAX_RECORDS = 64;
constexpr int RECORD_BYTES = 48;
constexpr int64_t RECORDS_AT = HEADER_BYTES;
constexpr int64_t DATA_AT = 8192;                 // RECORDS_AT + 8 + MAX_RECORDS * RECORD_BYTES, rounded up to 4096
constexpr int MAX_LT = 64;                        // dfb_corr_enable's largest temporal lag
constexpr int INFO_VALUES = 30;                   // dfb_restart_info

enum Section { SEC_STATE = 0, SEC_STATS = 1, SEC_CORR_Z = 2, SEC_CORR_Y = 3, SEC_CORR_T = 4, SEC_RING = 5, N_SECTIONS = 6 };

struct Header {
    std::string lib_version;                      // at most 63 bytes are stored
    int32_t Ny = 0, NzG = 0, plane0 = 0, nplanes = 0, periodic = 0, noise_mode = 0;
    uint64_t seed = 0;
    int64_t step = 0;
    int32_t Ny_max[3] = {}, Nz_max[3] = {};
    double Lt[3] = {};
    int32_t forms[3] = {};                        // dfb_info 3, 7 and 10 of the last writer (not part of the file's identity)
    uint64_t fingerprint = 0;
    uint32_t sections = 0;                        // DFB_RESTART_STATE | _STATS | _CORR
    int64_t stats_count = 0;
    int32_t stats_on = 0;
    int32_t corr_L[3] = {};                       // lags z, y, t
    int32_t corr_on = 0, n_ring = 0;              // n_ring: fields in the ring section (min(L_t, ring_count) while accumulating, else 0)
    int64_t corr_count = 0;
    int64_t corr_tsteps[MAX_LT + 1] = {};
    int32_t filter_shape = 0;                     // DFB_FILTER_*; stored after file_bytes, so files written before it read 0 (exponential)
    uint64_t profiles = 0;                        // Plan::cells_hash (0: no per-cell profiles); stored after filter_shape, older files read 0
    // derived by layout(): byte offset of each section (0 when absent) and the file's size
    int64_t off[N_SECTIONS] = {};
    int64_t file_bytes = 0;
};

struct Record {
    int32_t plane0 = 0, nplanes = 0, k0 = 0, k1 = 0;
    int64_t step = 0;
    uint64_t fingerprint = 0;
};

// Everything that decides the numbers of the next steps besides the seed and the plane range: Ny, NzG, periodic_z, the whole-plane
// half-width tables of each field (per row when row-uniform, per cell otherwise), Lt of each field and the [8][Ny] row tables,
// the per-row time scales when set, the filter shape when it is Gaussian, and the hash of the per-cell profiles when set.
uint64_t fingerprint(const Plan& P);
// the hash fingerprint() uses, of n doubles by their bits (Plan::cells_hash of a whole-plane profile table)
uint64_t hash_f64(const double* v, size_t n);

void layout(Header& h);                                       // fills off[] and file_bytes from the sizes and sections
void encode_header(const Header& h, unsigned char* out);      // HEADER_BYTES bytes
Header decode_header(const unsigned char* in);                // throws Error{DFB_ERR_IO} on a foreign file or another format version
std::vector<int64_t> info_values(const Header& h, int n_records);   // the INFO_VALUES values of dfb_restart_info, in its order

// byte offset of element (plane, j, k) of component `comp` of a section: comp = field (state, corr sums), statistic 0..5 (stats),
// i * 3 + field for ring entry i; k is the column (NzG-wide rows) or the lag (corr sums)
int64_t segment_offset(const Header& h, int section, int comp, int plane, int j, int k);

// "" when the records that carry the header's step and fingerprint cover columns [k0, k1) of planes [p0, p1) (global plane ids) and
// no record over that region is stale; else the message, naming the missing or stale column range
std::string check_coverage(const Header& h, const std::vector<Record>& recs, int p0, int p1, int k0, int k1);

// rows of one (section, comp, plane) block in host memory: `nrows` rows of `width` doubles, row j at rows + j * width, written to /
// read from columns [k0, k0 + width) of the section's row j
struct Block {
    int section, comp, plane;
    double* rows;
    int nrows, width, k0;
};

// A writer's save: under an open-file-description lock on the header, clears the record table when it belongs to another step or
// another file identity, writes the header and sizes the file; writes its blocks; then adds `mine` under the lock.  Throws Error.
void save(const char* path, const Header& h, const Record& mine, const std::vector<Block>& blocks);
// header and records of a file; throws Error{DFB_ERR_IO} for a missing, short or foreign file
Header read_header(const char* path, std::vector<Record>* recs);
void read_blocks(const char* path, const Header& h, const std::vector<Block>& blocks);

}  // namespace rst
}  // namespace dfb
