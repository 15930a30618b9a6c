// Test-only CPU emulation of the distance kernels (csrc/distance.cu): csrc/cube_distance.cuh compiled as plain
// C++, driven the way the kernels drive it -- the level-by-level table build, one lookup / solve per row.
// Never linked into the product library.
#include <cstdint>
#include <cstring>

#include "../../rubiks_cube_solver_b200/csrc/cube_distance.cuh"

namespace {
void row_words(const uint8_t* rows, long long i, uint32_t* row) { std::memcpy(row, rows + 24 * i, 24); }
}  // namespace

extern "C" {

long long emul_dist2_entries() { return kDist2Entries; }

// rank of every row, -1 where the row is not reachable
void emul_dist2_rank(const uint8_t* rows, long long n, long long* out)
{
    for (long long i = 0; i < n; ++i) {
        uint32_t row[6];
        row_words(rows, i, row);
        bool ok;
        const uint64_t w = dist2_from_row(row, ok);
        out[i] = ok ? (long long)dist2_rank(w) : -1;
    }
}

// number of ranks r with rank(unrank(r)) != r
long long emul_dist2_roundtrip_failures()
{
    long long bad = 0;
    for (uint32_t r = 0; r < kDist2Entries; ++r) bad += dist2_rank(dist2_unrank(r)) != r;
    return bad;
}

// launch_distance_build2: memset to 255, rank 0 = 0, then levels 0 .. kDist2Max - 1 over the table's words
void emul_dist2_build(uint8_t* table)
{
    std::memset(table, CUBE_DISTANCE_UNREACHABLE, kDist2Entries);
    table[0] = 0;
    for (uint32_t d = 0; d < (uint32_t)kDist2Max; ++d)
        for (uint32_t i = 0; i < kDist2Entries / 4; ++i) {
            uint32_t v;
            std::memcpy(&v, table + 4 * i, 4);
            for (int k = 0; k < 4; ++k)
                if (((v >> (8 * k)) & 0xffu) == d) dist2_expand(table, 4u * i + (uint32_t)k, d);
        }
}

void emul_dist2_lookup(const uint8_t* table, const uint8_t* rows, long long n, uint8_t* out)
{
    for (long long i = 0; i < n; ++i) {
        uint32_t row[6];
        row_words(rows, i, row);
        out[i] = (uint8_t)dist2_lookup(table, row);
    }
}

void emul_dist2_solve(const uint8_t* table, const uint8_t* rows, long long n, uint8_t* actions, uint8_t* length)
{
    for (long long i = 0; i < n; ++i) {
        uint32_t row[6];
        row_words(rows, i, row);
        length[i] = (uint8_t)dist2_solve(table, row, actions + kDist2Max * i);
    }
}

}  // extern "C"
