// 3x3x3 pattern databases: rank / unrank / turn of the exact encoding's cubies and the per-state bodies of the
// pattern kernels (pattern.cu) -- the level-synchronous build of the three tables, the admissible bound and the
// bounded IDA* solve.  Device code under nvcc, plain C++ under a host compiler, so that the test-only emulation
// harness (tests/host_emul/pattern_emul.cpp) runs exactly this code on the CPU.
//
// Cubies (include/cube_b200.h): byte q = piece | ori << 4 of corner slot q = 0..7 (CORNER_DEFS_EXACT) and of edge
// slot q = 0..11 (the shipped edge table), the pairs cube_encode(3, ..., CUBE_ENCODING_EXACT) builds its columns from.
// Sections of the table buffer, one byte per rank:
//   corners   Lehmer(p_0..p_7) * 2187 + sum_{q<7} o_q * 3^(6-q)                     (o_7 is implied)
//   edges A   pieces k = 0..5: r = r * (12 - k) + #{free slots below the slot of piece k}, then r * 64 + the six
//             flips in base 2 (piece 0 the most significant)
//   edges B   the same for pieces 6..11, slots relabelled s -> (s - 6) mod 12
// The solved cube is rank 0 in every section.
#pragma once
#include "cube_common.cuh"

#if defined(__CUDACC__)
#define PAT3_FN __device__ __forceinline__     // the tables below are __device__ arrays under nvcc
#else
#define PAT3_FN inline
#endif

constexpr uint32_t kPat3Corners = 88179840u;                       // 8! * 3^7
constexpr uint32_t kPat3Edges = 42577920u;                         // 12! / 6! * 2^6
constexpr uint32_t kPat3Offset[3] = {0u, kPat3Corners, kPat3Corners + kPat3Edges};
constexpr uint32_t kPat3Entries[3] = {kPat3Corners, kPat3Edges, kPat3Edges};
constexpr uint32_t kPat3Bytes = kPat3Corners + 2u * kPat3Edges;     // 173 335 680
constexpr int kPat3Levels[3] = {CUBE_PATTERN_MAX_CORNERS, CUBE_PATTERN_MAX_EDGES, CUBE_PATTERN_MAX_EDGES};
static_assert(kPat3Corners % 16 == 0 && kPat3Edges % 16 == 0, "sections start on 16 bytes and are read as words");

struct Pat3 {
    uint64_t c;      // corner slots 0..7, one byte each
    uint64_t e;      // edge slots 0..7
    uint32_t e8;     // edge slots 8..11
};

PAT3_FN uint32_t pat3_popc(uint32_t x)
{
#if defined(__CUDA_ARCH__)
    return __popc(x);
#else
    return (uint32_t)__builtin_popcount(x);
#endif
}

PAT3_FN uint32_t pat3_fact(int k) { return k == 7 ? 5040u : k == 6 ? 720u : k == 5 ? 120u : k == 4 ? 24u : k == 3 ? 6u : k == 2 ? 2u : 1u; }

PAT3_FN uint32_t pat3_edge(const Pat3& s, uint32_t q)
{
    return q < 8u ? (uint32_t)(s.e >> (8u * q)) & 0xffu : (s.e8 >> (8u * (q - 8u))) & 0xffu;
}

PAT3_FN Pat3 pat3_solved()
{
    return Pat3{0x0706050403020100ull, 0x0706050403020100ull, 0x0b0a0908u};
}

// face turn a < 12 (the action order of cube_env.py:24-28) through kPatMove3 (gen_tables.py PAT_MOVE_3)
PAT3_FN uint64_t pat3_turn_corners(uint64_t c, int a)
{
    uint64_t out = 0;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const uint32_t m = kPatMove3[20 * a + q], b = (uint32_t)(c >> (8u * (m & 15u))) & 0xffu;
        uint32_t o = (b >> 4) + (m >> 4);
        o -= o >= 3u ? 3u : 0u;
        out |= (uint64_t)((b & 15u) | o << 4) << (8 * q);
    }
    return out;
}

PAT3_FN void pat3_turn_edges(const Pat3& s, int a, Pat3& out)
{
    out.e = 0;
    out.e8 = 0;
#pragma unroll
    for (int q = 0; q < 12; ++q) {
        const uint32_t m = kPatMove3[20 * a + 8 + q], b = pat3_edge(s, m & 15u) ^ (m & 0x10u);
        if (q < 8) out.e |= (uint64_t)b << (8 * q);
        else out.e8 |= b << (8 * (q - 8));
    }
}

PAT3_FN Pat3 pat3_turn(const Pat3& s, int a)
{
    Pat3 out;
    out.c = pat3_turn_corners(s.c, a);
    pat3_turn_edges(s, a, out);
    return out;
}

// corner rank; parity = parity of the corner permutation (every quarter turn flips it)
PAT3_FN uint32_t pat3_corner_rank(uint64_t c, uint32_t& parity)
{
    uint32_t L = 0, T = 0, later = 0, inv = 0;
#pragma unroll
    for (int i = 7; i >= 0; --i) {
        const uint32_t p = (uint32_t)(c >> (8 * i)) & 15u, smaller = pat3_popc(later & ((1u << p) - 1u));
        L += smaller * pat3_fact(7 - i);
        inv += smaller;
        later |= 1u << p;
    }
#pragma unroll
    for (int i = 0; i < 7; ++i) T = T * 3u + ((uint32_t)(c >> (8 * i + 4)) & 15u);
    parity = inv & 1u;
    return L * 2187u + T;
}

// rank of edge section base / 6 + 1 (base 0: pieces 0..5, base 6: pieces 6..11 with slots relabelled)
PAT3_FN uint32_t pat3_edge_rank(const Pat3& s, uint32_t base)
{
    uint64_t pos = 0;                                                // 4 bits per tracked piece: its slot
    uint32_t flips = 0;
#pragma unroll
    for (uint32_t q = 0; q < 12; ++q) {
        const uint32_t b = pat3_edge(s, q), k = (b & 15u) - base;   // wraps for pieces below base
        if (k < 6u) {
            const uint32_t slot = q >= base ? q - base : q + 12u - base;
            pos |= (uint64_t)slot << (4u * k);
            flips |= ((b >> 4) & 1u) << (5u - k);
        }
    }
    uint32_t r = 0, used = 0;
#pragma unroll
    for (uint32_t k = 0; k < 6; ++k) {
        const uint32_t sl = (uint32_t)(pos >> (4u * k)) & 15u;
        r = r * (12u - k) + sl - pat3_popc(used & ((1u << sl) - 1u));
        used |= 1u << sl;
    }
    return r * 64u + flips;
}

PAT3_FN uint32_t pat3_rank(int section, const Pat3& s)
{
    uint32_t parity;
    return section == 0 ? pat3_corner_rank(s.c, parity) : pat3_edge_rank(s, section == 1 ? 0u : 6u);
}

// A cube whose section `section` has rank r.  Corners: the edges are solved.  Edges: the corners are solved and
// the slots of the six untracked edges hold 0x0f, which no rank reads.
PAT3_FN Pat3 pat3_unrank(int section, uint32_t r)
{
    Pat3 s = pat3_solved();
    if (section == 0) {
        uint32_t L = r / 2187u, T = r - 2187u * L, ori[8], sum = 0;
#pragma unroll
        for (int i = 6; i >= 0; --i) {
            ori[i] = T % 3u;
            T /= 3u;
            sum += ori[i];
        }
        ori[7] = (3u - sum % 3u) % 3u;
        uint32_t used = 0;
        s.c = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const uint32_t f = pat3_fact(7 - i), d = L / f;
            L -= d * f;
            uint32_t p = 0, seen = 0;                              // the d-th piece not placed yet
#pragma unroll
            for (uint32_t v = 0; v < 8; ++v) {
                const uint32_t free_v = ((used >> v) & 1u) ^ 1u;
                if (free_v && seen == d) p = v;
                seen += free_v;
            }
            used |= 1u << p;
            s.c |= (uint64_t)(p | ori[i] << 4) << (8 * i);
        }
        return s;
    }
    const uint32_t base = section == 1 ? 0u : 6u;
    uint32_t flips = r & 63u, digit[6];
    r >>= 6;
#pragma unroll
    for (int k = 5; k >= 0; --k) {
        digit[k] = r % (12u - (uint32_t)k);
        r /= 12u - (uint32_t)k;
    }
    s.e = 0x0f0f0f0f0f0f0f0full;
    s.e8 = 0x0f0f0f0fu;
    uint32_t used = 0;
#pragma unroll
    for (uint32_t k = 0; k < 6; ++k) {
        uint32_t sl = 0, seen = 0;                                  // the digit-th slot not taken yet
#pragma unroll
        for (uint32_t v = 0; v < 12; ++v) {
            const uint32_t free_v = ((used >> v) & 1u) ^ 1u;
            if (free_v && seen == digit[k]) sl = v;
            seen += free_v;
        }
        used |= 1u << sl;
        const uint32_t q = sl + base < 12u ? sl + base : sl + base - 12u;
        const uint32_t b = (base + k) | ((flips >> (5u - k)) & 1u) << 4;
        if (q < 8u) s.e = (s.e & ~(0xffull << (8u * q))) | (uint64_t)b << (8u * q);
        else s.e8 = (s.e8 & ~(0xffu << (8u * (q - 8u)))) | b << (8u * (q - 8u));
    }
    return s;
}

// Cubies of a 54-byte sticker row.  `reachable` is set exactly when the row is a state reachable from solved: the
// six centres are in place, every slot shows the colours of its (piece, ori), the corners and the edges are each a
// permutation, the twists sum to 0 mod 3, the flips to 0 mod 2, and the two permutations have the same parity.
PAT3_FN Pat3 pat3_from_row(const uint8_t* row, bool& reachable)
{
    Pat3 s{0, 0, 0};
    uint32_t cseen = 0, eseen = 0, twist = 0, flip = 0, cinv = 0, einv = 0;
    bool same = true;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const uint32_t w = kHashDef3x[q];
        const uint32_t a = row[w & 0xffu], b = row[(w >> 8) & 0xffu], c = row[(w >> 16) & 0xffu];
        const uint32_t h = a + 2u * b + 10u * c;
        const uint32_t col = kCornerCol3x[h < 128u ? h : 0u];      // a colour >= 6 never matches: any entry will do
        const uint32_t p = col / 3u, o = col - 3u * p;
        same &= (a | b << 8 | c << 16) == kCornerHome3x[col];
        cseen |= 1u << p;
        twist += o;
        s.c |= (uint64_t)(p | o << 4) << (8 * q);
    }
#pragma unroll
    for (int q = 0; q < 12; ++q) {
        const uint32_t w = kHashDef3x[8 + q];
        const uint32_t a = row[w & 0xffu], b = row[(w >> 8) & 0xffu];
        const uint32_t h = a + 10u * b;
        const uint32_t col = kEdgeCol3[h < 128u ? h : 0u];
        const uint32_t p = col >> 1, o = col & 1u;
        same &= (a | b << 8) == kEdgeHome3[col];
        eseen |= 1u << p;
        flip += o;
        if (q < 8) s.e |= (uint64_t)(p | o << 4) << (8 * q);
        else s.e8 |= (p | o << 4) << (8 * (q - 8));
    }
#pragma unroll
    for (int f = 0; f < 6; ++f) same &= row[9 * f + 4] == (uint8_t)f;
    uint32_t later = 0;
#pragma unroll
    for (int i = 7; i >= 0; --i) {
        const uint32_t p = (uint32_t)(s.c >> (8 * i)) & 15u;
        cinv += pat3_popc(later & ((1u << p) - 1u));
        later |= 1u << p;
    }
    later = 0;
#pragma unroll
    for (int i = 11; i >= 0; --i) {
        const uint32_t p = pat3_edge(s, (uint32_t)i) & 15u;
        einv += pat3_popc(later & ((1u << p) - 1u));
        later |= 1u << p;
    }
    reachable = same && cseen == 0xffu && eseen == 0xfffu && twist % 3u == 0u && (flip & 1u) == 0u &&
                ((cinv ^ einv) & 1u) == 0u;
    return s;
}

// table reads of the bound / solve kernels (the tables are read-only there)
PAT3_FN uint32_t pat3_load(const uint8_t* tables, uint32_t r)
{
#if defined(__CUDA_ARCH__)
    return __ldg(tables + r);
#else
    return tables[r];
#endif
}

// One state of BFS level d of a section: its unvisited neighbours get d + 1.  Concurrent threads may store the
// same byte; they all store d + 1.
PAT3_FN void pat3_expand(uint8_t* section_table, int section, uint32_t r, uint32_t d)
{
    const Pat3 s = pat3_unrank(section, r);
#pragma unroll 1
    for (int a = 0; a < 12; ++a) {
        Pat3 t;
        if (section == 0) t.c = pat3_turn_corners(s.c, a);
        else pat3_turn_edges(s, a, t);
        const uint32_t c = pat3_rank(section, t);
        if (section_table[c] == CUBE_DISTANCE_UNREACHABLE) section_table[c] = (uint8_t)(d + 1u);
    }
}

// max of the three section values, plus 1 when its parity differs from the corner permutation's: every quarter
// turn is a 4-cycle of corners, so a state's distance has that parity.  An admissible quarter-turn lower bound.
PAT3_FN uint32_t pat3_bound(const uint8_t* tables, const Pat3& s, uint32_t* parts)
{
    uint32_t parity;
    const uint32_t hc = pat3_load(tables, pat3_corner_rank(s.c, parity));
    const uint32_t ha = pat3_load(tables + kPat3Corners, pat3_edge_rank(s, 0u));
    const uint32_t hb = pat3_load(tables + kPat3Corners + kPat3Edges, pat3_edge_rank(s, 6u));
    parts[0] = hc;
    parts[1] = ha;
    parts[2] = hb;
    uint32_t h = hc > ha ? hc : ha;
    h = h > hb ? h : hb;
    return h + ((h ^ parity) & 1u);
}

// bound of a sticker row, CUBE_DISTANCE_UNREACHABLE (and parts of 255) for an unreachable row
PAT3_FN uint32_t pat3_row_bound(const uint8_t* tables, const uint8_t* row, uint32_t* parts)
{
    bool ok;
    const Pat3 s = pat3_from_row(row, ok);
    if (!ok) {
        parts[0] = parts[1] = parts[2] = CUBE_DISTANCE_UNREACHABLE;
        return CUBE_DISTANCE_UNREACHABLE;
    }
    return pat3_bound(tables, s, parts);
}

// Canonical quarter-turn sequences: no a ^ 1 right after a; a face twice in a row only as two equal clockwise turns,
// never three times; after a turn of face f no turn of the opposite face f' < f (faces U F R D B L = a >> 1, the
// opposite of f is f +- 3).  Every state has an optimal solution among them.
PAT3_FN bool pat3_canonical(const uint8_t* path, uint32_t g, uint32_t a)
{
    if (g == 0) return true;
    const uint32_t p = path[g - 1], f = a >> 1, pf = p >> 1;
    if (f == pf) return a == p && (a & 1u) == 0u && (g < 2 || (uint32_t)(path[g - 2] >> 1) != f);
    return f + 3u != pf;
}

struct Pat3Solve {
    uint32_t length, lower;        // CUBE_DISTANCE_UNREACHABLE where not proven / unreachable
    long long nodes;               // child states generated (each costs a bound)
};

// IDA* from a sticker row: thresholds from the bound in steps of 2 up to max_length; children in increasing action
// index among the canonical sequences; a child whose g + bound exceeds the threshold is cut.  actions[0, max_length)
// = the first solution found in that order, padded with CUBE_NOOP.  length = its length (optimal) or 255 when none
// was proven: the row is unreachable, every threshold up to max_length completed without one (then lower >
// max_length), or the next child would have been generated past max_nodes.  lower = the best proven lower bound:
// the bound, then t + 2 after each completed threshold t, the length once solved; 255 for an unreachable row.
PAT3_FN Pat3Solve pat3_solve(const uint8_t* tables, const uint8_t* row, int max_length, long long max_nodes,
                             uint8_t* actions)
{
    Pat3Solve res{CUBE_DISTANCE_UNREACHABLE, CUBE_DISTANCE_UNREACHABLE, 0};
    for (int k = 0; k < max_length; ++k) actions[k] = CUBE_NOOP;
    bool ok;
    const Pat3 root = pat3_from_row(row, ok);
    if (!ok) return res;
    uint32_t parts[3];
    const uint32_t h0 = pat3_bound(tables, root, parts);
    res.lower = h0;
    if (h0 == 0) {
        res.length = 0;
        return res;
    }
    uint8_t path[CUBE_SOLVE_BOUNDED_MAX_LENGTH];
    for (uint32_t t = h0; t <= (uint32_t)max_length; t += 2) {
        Pat3 s = root;
        uint32_t g = 0, a = 0;
        for (;;) {
            if (a < 12u) {
                if (!pat3_canonical(path, g, a)) {
                    ++a;
                    continue;
                }
                if (res.nodes == max_nodes) return res;               // budget spent: lower stays proven
                ++res.nodes;
                const Pat3 c = pat3_turn(s, (int)a);
                const uint32_t gc = g + 1;
                uint32_t parity;
                const uint32_t hc = pat3_load(tables, pat3_corner_rank(c.c, parity));
                if (gc + hc <= t) {                                   // the corners alone cut most children
                    const uint32_t ha = pat3_load(tables + kPat3Corners, pat3_edge_rank(c, 0u));
                    const uint32_t hb = pat3_load(tables + kPat3Corners + kPat3Edges, pat3_edge_rank(c, 6u));
                    uint32_t h = hc > ha ? hc : ha;
                    h = h > hb ? h : hb;
                    h += (h ^ parity) & 1u;
                    if (gc + h <= t) {
                        path[g] = (uint8_t)a;
                        if (h == 0) {                                 // solved (every section at rank 0)
                            for (uint32_t k = 0; k < gc; ++k) actions[k] = path[k];
                            res.length = res.lower = gc;
                            return res;
                        }
                        s = c;
                        g = gc;
                        a = 0;
                        continue;
                    }
                }
                ++a;
            } else {
                if (g == 0) break;                                    // threshold t completed without a solution
                --g;
                a = path[g];
                s = pat3_turn(s, (int)(a ^ 1u));
                ++a;
            }
        }
        res.lower = t + 2;
    }
    return res;
}
