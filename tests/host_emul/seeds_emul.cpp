// Test-only CPU emulation of K0 (csrc/seeds.cu): csrc/cube_seeds.cuh compiled as plain C++, one row per seed
// the way the kernel's threads draw them, fast path and slow path alike.  Never linked into the product library.
#include <cstdint>

#include "../../rubiks_cube_solver_b200/csrc/cube_seeds.cuh"

namespace {
struct HostRow {
    uint8_t *p, *end;
    bool full() const { return p >= end; }
    void put(uint32_t v) { *p++ = (uint8_t)v; }
};
}  // namespace

extern "C" {

// moves[i, :] = RandomState(seeds[i]).randint(A, size=depth); returns the number of rows that took the slow path
long long emul_moves_from_seeds(int cube_size, const uint32_t* seeds, long long n, int depth, uint8_t* moves)
{
    const uint32_t max_value = cube_size == 3 ? 11u : 5u, mask = seed_mask(max_value);
    long long slow = 0;
    for (long long i = 0; i < n; ++i) {
        uint8_t* row = moves + i * depth;
        slow += seed_row(seeds[i], max_value, mask, HostRow{row, row + depth}) ? 1 : 0;
    }
    return slow;
}

}  // extern "C"
