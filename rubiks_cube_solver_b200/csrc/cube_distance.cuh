// Exact 2x2x2 distance table: rank / unrank / turn of py222's cubies and the per-state bodies of the
// distance kernels (distance.cu).  Device code under nvcc, plain C++ under a host compiler, so that the
// test-only emulation harness (tests/host_emul/) runs exactly this code on the CPU.
//
// Layout (include/cube_b200.h): (p_i, o_i) = py222 getOP of slot i = 0..6,
//   rank = L * 729 + T,   L = sum_i #{j > i : p_j < p_i} * (6 - i)!,   T = sum_{i < 6} o_i * 3^(5 - i);
// o_6 is implied (the orientations of a reachable state sum to 0 mod 3).  Rank 0 is the solved cube.
#pragma once
#include "cube_common.cuh"

#if defined(__CUDACC__)
#define DIST2_FN __device__ __forceinline__     // the tables below are __device__ arrays under nvcc
#else
#define DIST2_FN inline
#endif

constexpr uint32_t kDist2Entries = 3674160u;   // 7! * 3^6
constexpr int kDist2Max = CUBE_DISTANCE_MAX_2;  // quarter-turn diameter of the 2x2x2

// Cubie word: byte q = cubelet | ori << 4 of slot q = 0..6 (kPieceCode2's format).
DIST2_FN uint32_t dist2_byte(uint64_t w, int q) { return (uint32_t)(w >> (8 * q)) & 0xffu; }

DIST2_FN uint32_t dist2_fact(int k) { return k == 6 ? 720u : k == 5 ? 120u : k == 4 ? 24u : k == 3 ? 6u : k == 2 ? 2u : 1u; }

DIST2_FN uint32_t dist2_rank(uint64_t w)
{
    uint32_t L = 0, T = 0;
#pragma unroll
    for (int i = 0; i < 7; ++i) {
        const uint32_t p = dist2_byte(w, i) & 15u;
        uint32_t smaller = 0;
#pragma unroll
        for (int j = i + 1; j < 7; ++j) smaller += (dist2_byte(w, j) & 15u) < p ? 1u : 0u;
        L += smaller * dist2_fact(6 - i);
        if (i < 6) T = T * 3u + (dist2_byte(w, i) >> 4);
    }
    return L * 729u + T;
}

DIST2_FN uint64_t dist2_unrank(uint32_t r)
{
    uint32_t L = r / 729u, T = r - 729u * L, ori[7], sum = 0;
#pragma unroll
    for (int i = 5; i >= 0; --i) {
        ori[i] = T % 3u;
        T /= 3u;
        sum += ori[i];
    }
    ori[6] = (3u - sum % 3u) % 3u;
    uint32_t used = 0;
    uint64_t w = 0;
#pragma unroll
    for (int i = 0; i < 7; ++i) {
        const uint32_t f = dist2_fact(6 - i), d = L / f;
        L -= d * f;
        uint32_t p = 0, seen = 0;                                  // the d-th cubelet not placed yet
#pragma unroll
        for (uint32_t v = 0; v < 7; ++v) {
            const uint32_t free_v = ((used >> v) & 1u) ^ 1u;
            if (free_v && seen == d) p = v;
            seen += free_v;
        }
        used |= 1u << p;
        w |= (uint64_t)(p | ori[i] << 4) << (8 * i);
    }
    return w;
}

// face turn a < 6 (the action order of cube_env.py:24-28)
DIST2_FN uint64_t dist2_turn(uint64_t w, int a)
{
    uint64_t out = 0;
#pragma unroll
    for (int q = 0; q < 7; ++q) {
        const uint32_t m = kDistMove2[7 * a + q], b = dist2_byte(w, (int)(m & 15u));
        uint32_t o = (b >> 4) + (m >> 4);
        o -= o >= 3u ? 3u : 0u;
        out |= (uint64_t)((b & 15u) | o << 4) << (8 * q);
    }
    return out;
}

DIST2_FN uint32_t dist2_sticker(const uint32_t* row, int s) { return (row[s >> 2] >> (8 * (s & 3))) & 0xffu; }

// py222 getOP of every slot of a sticker row (24 bytes as six little-endian words).  `reachable` is set
// exactly when the row rebuilt from its rank is the row: the rebuilt stickers match, the cubelets are a
// permutation and the orientations sum to 0 mod 3.  Colours >= 6, hashes outside py222's table, swapped
// stickers and a twisted corner all fail it.
DIST2_FN uint64_t dist2_from_row(const uint32_t* row, bool& reachable)
{
    uint64_t w = 0;
    uint32_t seen = 0, osum = 0;
    bool same = true;
#pragma unroll
    for (int q = 0; q < 7; ++q) {
        const uint32_t a = dist2_sticker(row, cube_piece_def2(q, 0)), b = dist2_sticker(row, cube_piece_def2(q, 1)),
                       c = dist2_sticker(row, cube_piece_def2(q, 2));
        const uint32_t h = a + 2u * b + 10u * c;
        const uint32_t code = kPieceCode2[h < 128u ? h : 0u];   // a colour >= 6 never rebuilds: any entry will do
        const uint32_t p = code & 15u, o = code >> 4;
        same &= (a | b << 8 | c << 16) == kCubieColours2[3u * p + o];
        seen |= 1u << p;
        osum += o;
        w |= (uint64_t)code << (8 * q);
    }
    same &= dist2_sticker(row, 14) == 3u && dist2_sticker(row, 18) == 4u && dist2_sticker(row, 23) == 5u;
    reachable = same && seen == 0x7fu && osum % 3u == 0u;
    return w;
}

// table reads of the lookup / solve kernels (the table is read-only there)
DIST2_FN uint32_t dist2_load(const uint8_t* table, uint32_t r)
{
#if defined(__CUDA_ARCH__)
    return __ldg(table + r);
#else
    return table[r];
#endif
}

// One state of BFS level d: its unvisited neighbours get d + 1.  Concurrent threads may store the same byte;
// they all store d + 1.
DIST2_FN void dist2_expand(uint8_t* table, uint32_t r, uint32_t d)
{
    const uint64_t w = dist2_unrank(r);
#pragma unroll
    for (int a = 0; a < 6; ++a) {
        const uint32_t c = dist2_rank(dist2_turn(w, a));
        if (table[c] == CUBE_DISTANCE_UNREACHABLE) table[c] = (uint8_t)(d + 1u);
    }
}

DIST2_FN uint32_t dist2_lookup(const uint8_t* table, const uint32_t* row)
{
    bool ok;
    const uint64_t w = dist2_from_row(row, ok);
    return ok ? dist2_load(table, dist2_rank(w)) : (uint32_t)CUBE_DISTANCE_UNREACHABLE;
}

// Optimal solution of one row: at every step the lowest action index whose child is one level closer.
// actions[0, kDist2Max) = the solution padded with CUBE_NOOP; returns its length, CUBE_DISTANCE_UNREACHABLE
// for an unreachable row.  The walk stops after kDist2Max steps or where no child is closer (only a buffer
// that is not a distance table can do that).
DIST2_FN uint32_t dist2_solve(const uint8_t* table, const uint32_t* row, uint8_t* actions)
{
    bool ok;
    uint64_t w = dist2_from_row(row, ok);
    for (int k = 0; k < kDist2Max; ++k) actions[k] = CUBE_NOOP;
    if (!ok) return CUBE_DISTANCE_UNREACHABLE;
    uint32_t d = dist2_load(table, dist2_rank(w)), len = 0;
    while (d > 0 && len < (uint32_t)kDist2Max) {
        uint32_t cd[6];
#pragma unroll
        for (int a = 0; a < 6; ++a) cd[a] = dist2_load(table, dist2_rank(dist2_turn(w, a)));   // six loads in flight
        int best = -1;
#pragma unroll
        for (int a = 5; a >= 0; --a) best = cd[a] + 1u == d ? a : best;
        if (best < 0) break;
        actions[len++] = (uint8_t)best;
        w = dist2_turn(w, best);
        --d;
    }
    return len;
}
