// Test-only CPU emulation of the pattern kernels (csrc/pattern.cu): csrc/cube_pattern.cuh compiled as plain C++,
// driven the way the kernels drive it -- the level-by-level build of a section, one bound / solve per row -- plus a
// check that a built section is a BFS distance table.  Never linked into the product library.
#include <cstdint>
#include <cstring>
#include <thread>
#include <vector>

#include "../../rubiks_cube_solver_b200/csrc/cube_pattern.cuh"

extern "C" {

long long emul_pat3_bytes() { return kPat3Bytes; }
long long emul_pat3_offset(int section) { return kPat3Offset[section]; }
long long emul_pat3_entries(int section) { return kPat3Entries[section]; }

// ranks [n, 3] of every row (corners, edges A, edges B) and reachable [n]
void emul_pat3_rank(const uint8_t* rows, long long n, long long* ranks, uint8_t* reachable)
{
    for (long long i = 0; i < n; ++i) {
        bool ok;
        const Pat3 s = pat3_from_row(rows + 54 * i, ok);
        reachable[i] = ok;
        for (int k = 0; k < 3; ++k) ranks[3 * i + k] = pat3_rank(k, s);
    }
}

// ranks [n, 12, 3] of the 12 children of every row, turned as cubies
void emul_pat3_child_ranks(const uint8_t* rows, long long n, long long* ranks)
{
    for (long long i = 0; i < n; ++i) {
        bool ok;
        const Pat3 s = pat3_from_row(rows + 54 * i, ok);
        for (int a = 0; a < 12; ++a) {
            const Pat3 c = pat3_turn(s, a);
            for (int k = 0; k < 3; ++k) ranks[36 * i + 3 * a + k] = pat3_rank(k, c);
        }
    }
}

// number of ranks r of a section with rank(unrank(r)) != r, over r = lo, lo + step, ...
long long emul_pat3_roundtrip_failures(int section, long long step)
{
    long long bad = 0;
    for (long long r = 0; r < (long long)kPat3Entries[section]; r += step)
        bad += pat3_rank(section, pat3_unrank(section, (uint32_t)r)) != (uint32_t)r;
    return bad;
}

// launch_pattern_build3 for one section: memset to 255, rank 0 = 0, then levels 0 .. max - 1 over its words
void emul_pat3_build(uint8_t* tables, int section)
{
    uint8_t* t = tables + kPat3Offset[section];
    const uint32_t entries = kPat3Entries[section];
    std::memset(t, CUBE_DISTANCE_UNREACHABLE, entries);
    t[0] = 0;
    for (uint32_t d = 0; d < (uint32_t)kPat3Levels[section]; ++d)
        for (uint32_t i = 0; i < entries / 4; ++i) {
            uint32_t v;
            std::memcpy(&v, t + 4 * i, 4);
            for (int k = 0; k < 4; ++k)
                if (((v >> (8 * k)) & 0xffu) == d) pat3_expand(t, section, 4u * i + (uint32_t)k, d);
        }
}

// Ranks of a section that break the characterisation of a BFS distance table: the value is 0 exactly at rank 0, no
// rank is left at 255, neighbours differ by at most 1 (by exactly 1 for the corners: a quarter turn is an odd
// corner permutation), and every nonzero rank has a neighbour one level closer.  Read-only: threaded over ranks.
long long emul_pat3_check(const uint8_t* tables, int section, int threads)
{
    const uint8_t* t = tables + kPat3Offset[section];
    const uint32_t entries = kPat3Entries[section];
    std::vector<long long> bad(threads, 0);
    std::vector<std::thread> pool;
    for (int w = 0; w < threads; ++w)
        pool.emplace_back([&, w] {
            const uint32_t lo = (uint32_t)((uint64_t)entries * w / threads), hi = (uint32_t)((uint64_t)entries * (w + 1) / threads);
            for (uint32_t r = lo; r < hi; ++r) {
                const uint32_t v = t[r];
                bool wrong = (v == 0) != (r == 0) || v == CUBE_DISTANCE_UNREACHABLE, closer = false;
                const Pat3 s = pat3_unrank(section, r);
                for (int a = 0; a < 12; ++a) {
                    const uint32_t u = t[pat3_rank(section, pat3_turn(s, a))];
                    const uint32_t diff = u > v ? u - v : v - u;
                    wrong |= diff > 1 || (section == 0 && diff != 1);
                    closer |= u + 1 == v;
                }
                bad[w] += wrong || (v != 0 && !closer);
            }
        });
    long long total = 0;
    for (int w = 0; w < threads; ++w) {
        pool[w].join();
        total += bad[w];
    }
    return total;
}

void emul_pat3_bound(const uint8_t* tables, const uint8_t* rows, long long n, uint8_t* bound, uint8_t* parts)
{
    for (long long i = 0; i < n; ++i) {
        uint32_t p[3];
        bound[i] = (uint8_t)pat3_row_bound(tables, rows + 54 * i, p);
        for (int k = 0; k < 3; ++k) parts[3 * i + k] = (uint8_t)p[k];
    }
}

void emul_pat3_solve(const uint8_t* tables, const uint8_t* rows, long long n, int max_length, long long max_nodes,
                     uint8_t* actions, uint8_t* length, uint8_t* lower, long long* nodes)
{
    for (long long i = 0; i < n; ++i) {
        const Pat3Solve r = pat3_solve(tables, rows + 54 * i, max_length, max_nodes, actions + (long long)max_length * i);
        length[i] = (uint8_t)r.length;
        lower[i] = (uint8_t)r.lower;
        nodes[i] = r.nodes;
    }
}

}  // extern "C"
