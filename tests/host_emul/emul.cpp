// Test-only CPU emulation of the kernels' per-thread code (csrc/cube_threads.cuh compiled as
// plain C++): runs the exact byte-permute / table / shared-memory-image arithmetic of the CUDA
// kernels tile by tile, so index and selector bugs surface in the CPU test-suite, before a GPU
// is involved.  Never linked into the product library.
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../rubiks_cube_solver_b200/csrc/cube_threads.cuh"

namespace {
constexpr int kTile = 256;
inline int round16(int x) { return (x + 15) & ~15; }

template <int SIZE>
void scramble_t(const uint8_t* moves, long long n, int depth, uint8_t* out, uint8_t* solved)
{
    using G = CubeGeom<SIZE>;
    const uint32_t* tbl = SIZE == 3 ? kMoveWords3 : kMoveWords2;
    const uint32_t* clut = SIZE == 3 ? kCornerColour3 : kCornerColour2;
    std::vector<uint8_t> s_moves(round16(kTile * depth) + 32), s_out(round16(kTile * G::S));
    for (long long base = 0; base < n; base += kTile) {
        const int cnt = (int)((n - base) < kTile ? (n - base) : kTile);
        std::memset(s_moves.data(), 0xee, s_moves.size());
        std::memcpy(s_moves.data(), moves + base * depth, (size_t)cnt * depth);
        for (int tid = 0; tid < cnt; ++tid) {
            CubieState st;
            cubie_init(st);
            scramble_run_staged<SIZE>(st, tid, depth, s_moves.data(), tbl);
            solved[base + tid] = scramble_finish<SIZE>(st, tid, clut, kEdgeColour3, s_out.data());
        }
        std::memcpy(out + base * G::S, s_out.data(), (size_t)cnt * G::S);
    }
}

// K1p: persistent pair-table kernel, one tile of 32 * NS rows at a time with the kernel's lane -> row map
// (rows beyond the last whole tile are left untouched: the library hands them to the tile-per-CTA kernel)
// K1p sliced (depth > 320): the kernel's staging arithmetic -- per row and slice a copy from the 16-byte
// boundary below the piece into a 272-byte slot, the piece starting (row * depth) & 15 bytes in -- and the slice
// runner that takes the shift out in registers and carries the state over.  `moves` must be readable 16 bytes
// past its end (the kernel never stages the last tile for that reason; the emulation stages all of them).
template <int SIZE>
void scramble_sliced_t(const uint8_t* moves, long long n, int depth, uint8_t* out, uint8_t* solved, const uint8_t* last,
                       int kSlice)
{
    using G = CubeGeom<SIZE>;
    const int kStride = ((kSlice + 32) / 16) % 2 ? kSlice + 32 : kSlice + 48;        // slice_stride() of scramble.cu
    const uint32_t* clut = SIZE == 3 ? kCornerColour3 : kCornerColour2;
    std::vector<uint8_t> tbl(65792 + 256, 0xa5);
    uint8_t* s_ptbl_mem = tbl.data() + ((16 - (reinterpret_cast<uintptr_t>(tbl.data()) & 15)) & 15);
    for (int t = 0; t < 96; ++t) pair_table_fill<SIZE>(s_ptbl_mem, t, 96);
    const PairTableHost s_ptbl{s_ptbl_mem};
    std::vector<uint8_t> buf(64 * kStride + 32), s_out(64 * G::S);
    uint8_t* s_moves = buf.data() + ((16 - (reinterpret_cast<uintptr_t>(buf.data()) & 15)) & 15);
    const int n_slices = (depth + kSlice - 1) / kSlice;
    for (long long tile = 0; tile * 64 + 64 <= n; ++tile) {
        std::vector<CubieState> st(64);
        for (auto& c : st) cubie_init(c);
        for (int s = 0; s < n_slices; ++s) {
            const int len = depth - s * kSlice < kSlice ? depth - s * kSlice : kSlice;
            std::memset(s_moves, 0xee, 64 * kStride);
            for (int row = 0; row < 64; ++row) {
                const long long g = (tile * 64 + row) * depth + (long long)s * kSlice;
                const uint32_t shift = (uint32_t)(((long long)row * depth) & 15);
                std::memcpy(s_moves + row * kStride, moves + (g & ~15LL), (shift + len + 15) & ~15u);
            }
            for (int lane = 0; lane < 32; ++lane) {
                const int rows[2] = {lane, lane + 32};
                CubieState two[2] = {st[rows[0]], st[rows[1]]};
                const uint32_t base[2] = {(uint32_t)(rows[0] * kStride), (uint32_t)(rows[1] * kStride)};
                const uint32_t shift[2] = {(uint32_t)(((long long)rows[0] * depth) & 15), (uint32_t)(((long long)rows[1] * depth) & 15)};
                scramble_pairs_run_units<SIZE, 2>(two, base, shift, len, s_moves, s_ptbl, pair_lanereg<SIZE>(lane, s_ptbl), pair_roff2(lane));
                st[rows[0]] = two[0]; st[rows[1]] = two[1];
            }
        }
        for (int lane = 0; lane < 32; ++lane)
            for (int k = 0; k < 2; ++k) {
                const int row = lane + 32 * k;
                if (last) scramble_pairs_last<SIZE>(st[row], last[tile * 64 + row], s_ptbl, pair_lanereg<SIZE>(lane, s_ptbl), pair_roff2(lane));
                solved[tile * 64 + row] = scramble_pairs_finish<SIZE>(st[row], row, ColourLutHost{clut, kEdgeColourSlot3}, s_out.data());
            }
        std::memcpy(out + tile * 64 * G::S, s_out.data(), (size_t)64 * G::S);
    }
}

// K1x: all prefixes of every scramble, a tile of 8 cubes at a time with the kernel's tile image and its
// four-lanes-per-cube split of the levels
template <int SIZE>
void prefixes_t(const uint8_t* moves, long long n, int depth, uint8_t* out, uint8_t* solved)
{
    using G = CubeGeom<SIZE>;
    constexpr int kSplit = 4, kCubes = 32 / kSplit;
    const uint32_t* tbl = SIZE == 3 ? kMoveWords3 : kMoveWords2;
    const uint32_t* clut = SIZE == 3 ? kCornerColour3 : kCornerColour2;
    std::vector<uint8_t> img((size_t)kCubes * depth * G::S + 16);
    for (long long cube0 = 0; cube0 < n; cube0 += kCubes) {
        const int cnt = (int)((n - cube0) < kCubes ? (n - cube0) : kCubes);
        std::memset(img.data(), 0xee, img.size());
        for (int lane = 0; lane < 32; ++lane) {
            const int cube = lane % kCubes, part = lane / kCubes;
            const int k_begin = part * depth / kSplit, k_end = (part + 1) * depth / kSplit;
            if (cube < cnt && k_begin < k_end)
                prefix_walk<SIZE>(moves + (cube0 + cube) * depth, depth, cube * depth, tbl, clut, kEdgeColour3, img.data(),
                                  solved + (cube0 + cube) * depth, k_begin, k_end);
        }
        std::memcpy(out + cube0 * depth * G::S, img.data(), (size_t)cnt * depth * G::S);
    }
}

template <int SIZE, int NS>
void scramble_pairs_t(const uint8_t* moves, long long n, int depth, uint8_t* out, uint8_t* solved, bool fixed, bool priv,
                      const uint8_t* last = nullptr)
{
    using G = CubeGeom<SIZE>;
    constexpr int T = 32 * NS;
    const uint32_t* clut = SIZE == 3 ? kCornerColour3 : kCornerColour2;
    std::vector<uint8_t> tbl(65792 + 256, 0xa5);
    uint8_t* s_ptbl_mem = tbl.data() + ((16 - (reinterpret_cast<uintptr_t>(tbl.data()) & 15)) & 15);
    for (int t = 0; t < 96; ++t) pair_table_fill<SIZE>(s_ptbl_mem, t, 96);
    std::vector<uint8_t> s_moves(T * depth + 16), s_out(T * G::S);
    std::vector<uint8_t> s_priv(T * depth + 16);
    for (long long base = 0; base + T <= n; base += T) {
        std::memset(s_moves.data(), 0xee, s_moves.size());
        std::memcpy(s_moves.data(), moves + base * depth, (size_t)T * depth);
        if (priv) {                                                  // the copy engine's 128-byte swizzle
            std::memset(s_priv.data(), 0xee, s_priv.size());
            for (int f = 0; f < T * depth; f += 16)
                std::memcpy(s_priv.data() + cube_swz128((uint32_t)f), moves + base * depth + f, 16);
        }
        uint32_t ok[NS] = {};
        for (int lane = 0; lane < 32; ++lane) {                      // one lane = NS rows in lockstep
            int rows[NS];
            CubieState st[NS];
            for (int k = 0; k < NS; ++k) {
                rows[k] = (SIZE == 3) ? 64 * (k >> 1) + 2 * lane + (k & 1) : lane + 32 * k;
                cubie_init(st[k]);
            }
            const PairTableHost s_ptbl{s_ptbl_mem};
            const uint32_t lr = pair_lanereg<SIZE>(lane, s_ptbl);
            if constexpr (SIZE == 2 || NS == 2) {
                if (priv) scramble_pairs_run_swizzled<SIZE, NS>(st, s_priv.data(), lane, depth, s_ptbl, lr, pair_roff2(lane));
            }
            if (priv) {}
            else if (fixed && depth == 30) scramble_pairs_run<SIZE, 30, NS>(st, rows, depth, s_moves.data(), s_ptbl, lr, pair_roff2(lane));
            else if (fixed && depth == 20) scramble_pairs_run<SIZE, 20, NS>(st, rows, depth, s_moves.data(), s_ptbl, lr, pair_roff2(lane));
            else if (fixed && depth == 43) scramble_pairs_run<SIZE, 43, NS>(st, rows, depth, s_moves.data(), s_ptbl, lr, pair_roff2(lane));
            else scramble_pairs_run<SIZE, 0, NS>(st, rows, depth, s_moves.data(), s_ptbl, lr, pair_roff2(lane));
            if (last)
                for (int k = 0; k < NS; ++k) scramble_pairs_last<SIZE>(st[k], last[base + rows[k]], s_ptbl, lr, pair_roff2(lane));
            for (int k = 0; k < NS; ++k)
                ok[k] |= (uint32_t)scramble_pairs_finish<SIZE>(st[k], rows[k], ColourLutHost{clut, kEdgeColourSlot3}, s_out.data()) << lane;
        }
        if (SIZE == 3) {
            for (int k = 0; k < T / 4; ++k) {                        // the kernel's verdict exchange
                const int h = 2 * (k >> 4);
                const uint32_t w = pair_solved_word<SIZE>(ok[h % NS], ok[(h + 1) % NS], k & 15);
                std::memcpy(solved + base + 4 * k, &w, 4);
            }
        } else {
            for (int k = 0; k < NS; ++k)
                for (int lane = 0; lane < 32; ++lane) solved[base + 32 * k + lane] = (ok[k] >> lane) & 1u;
        }
        std::memcpy(out + base * G::S, s_out.data(), (size_t)T * G::S);
    }
}

template <int SIZE>
void walk_t(const uint8_t* in, const uint8_t* moves, long long n, int depth, uint8_t* out, uint8_t* solved)
{
    using G = CubeGeom<SIZE>;
    const uint32_t* cyc = SIZE == 3 ? kCycles3 : kCycles2;
    for (long long i = 0; i < n; ++i) {
        alignas(4) uint8_t row[56];
        std::memcpy(row, in + i * G::S, G::S);
        for (int k = 0; k < depth; ++k) walk_turn<SIZE>(row, moves[i * depth + k] & 0xfu, cyc);
        solved[i] = row_solved<SIZE>(row);
        std::memcpy(out + i * G::S, row, G::S);
    }
}

// K2p: lane-private layout, 64-row tiles, the kernel's two passes per lane
template <int SIZE>
void walk_private_t(const uint8_t* in, const uint8_t* moves, long long n, int depth, uint8_t* out, uint8_t* solved)
{
    using G = CubeGeom<SIZE>;
    constexpr int W = WalkImage<SIZE>::W;
    const uint32_t* cyc = SIZE == 3 ? kCycles3 : kCycles2;
    std::vector<uint32_t> ent(2 * G::NCYC * CUBE_MOVE_ROWS * 2);
    for (int i = 0; i < 2 * G::NCYC * CUBE_MOVE_ROWS; ++i) {
        const int shift = (i >= G::NCYC * CUBE_MOVE_ROWS) ? 2 : 0;
        walk_cycle_entry(cyc[i - (shift ? G::NCYC * CUBE_MOVE_ROWS : 0)], shift, ent.data() + 2 * i);
    }
    std::vector<uint32_t> tile32(64 * G::S / 4 + 4), scratch32(32 * W);
    uint8_t* tile = reinterpret_cast<uint8_t*>(tile32.data());
    uint8_t* scratch = reinterpret_cast<uint8_t*>(scratch32.data());
    for (long long base = 0; base + 64 <= n; base += 64) {
        std::memcpy(tile, in + base * G::S, (size_t)64 * G::S);
        uint32_t mask[2] = {0, 0};
        for (int pass = 0; pass < 2; ++pass)
            for (int lane = 0; lane < 32; ++lane) {
                const int row = (SIZE == 3) ? 2 * lane + pass : lane + 32 * pass;
                const int shift = (pass && SIZE == 3) ? 2 : 0;
                uint32_t* img_p = reinterpret_cast<uint32_t*>(tile + G::S * row - shift);
                uint32_t w[W];
                for (int j = 0; j < W; ++j) w[j] = img_p[j];
                uint8_t* lane_base = scratch + 4 * lane;
                if (SIZE == 3) {
                    for (int j = 0; j < W; ++j) reinterpret_cast<uint32_t*>(lane_base)[32 * j] = w[j];
                    const uint32_t* e = ent.data() + (shift ? 2 * G::NCYC * CUBE_MOVE_ROWS : 0);
                    for (int k = 0; k < depth; ++k)
                        walk_turn_private<SIZE>(lane_base, e, moves[(base + row) * depth + k] & 0xfu);
                    for (int j = 0; j < W; ++j) w[j] = reinterpret_cast<const uint32_t*>(lane_base)[32 * j];
                } else {
                    for (int k = 0; k < depth; ++k) walk_turn_registers2(w, moves[(base + row) * depth + k] & 0xfu);
                }
                const bool ok = shift ? image_solved<SIZE, (SIZE == 3 ? 2 : 0)>(w) : image_solved<SIZE, 0>(w);
                mask[pass] |= (uint32_t)ok << lane;
                for (int j = 0; j < W; ++j) img_p[j] = w[j];
            }
        std::memcpy(out + base * G::S, tile, (size_t)64 * G::S);
        for (int k = 0; k < 16; ++k) {
            const uint32_t v = pair_solved_word<SIZE>(mask[0], mask[1], k);
            std::memcpy(solved + base + 4 * k, &v, 4);
        }
    }
}

template <int SIZE, int DTYPE>
void expand_t(const uint8_t* states, long long n, uint8_t* children, uint8_t* child_oh, uint8_t* parent_oh,
              uint8_t* solved)
{
    using G = CubeGeom<SIZE>;
    constexpr int S = G::S, A = G::A, R = G::R, C = G::C, ES = OneHot<DTYPE>::ESIZE, P = (SIZE == 3) ? 16 : 64;
    const uint8_t* gather = SIZE == 3 ? kGather3 : kGather2;
    const int gstride = SIZE == 3 ? 56 : 24;
    const uint32_t* def = SIZE == 3 ? kHashDef3 : kHashDef2;
    const uint8_t* lut0 = SIZE == 3 ? kCornerCol3 : kPieceCode2;
    const uint8_t* lut1 = kEdgeCol3;
    std::vector<uint8_t> s_child(P * A * S), colc(P * A * R + 4), colp(P * R + 4);
    for (long long base = 0; base < n; base += P) {
        const int cnt = (int)((n - base) < P ? (n - base) : P), rows = cnt * A;
        const uint8_t* s_par = states + base * S;
        std::memset(colc.data(), 255, colc.size());
        std::memset(colp.data(), 255, colp.size());
        for (int r = 0; r < rows; ++r)
            for (int i = 0; i < S; ++i) s_child[r * S + i] = s_par[(r / A) * S + gather[(r % A) * gstride + i]];
        for (int it = 0; it < (rows + cnt) * R; ++it) {
            const int r = it / R, slot = it % R;
            const bool is_child = r < rows;
            const int rr = is_child ? r : r - rows;
            const uint8_t* row = is_child ? &s_child[rr * S] : s_par + rr * S;
            uint8_t* colrow = is_child ? &colc[rr * R] : &colp[rr * R];
            const uint32_t code = onehot_code<SIZE>(row, slot, def, lut0, lut1);
            if (SIZE == 3) colrow[slot] = (uint8_t)code;
            else colrow[code & 0xfu] = (uint8_t)(3 * slot + (code >> 4));
        }
        for (int r = 0; r < rows; ++r) solved[base * A + r] = stickers_solved<SIZE>(&s_child[r * S]);
        if (children) std::memcpy(children + base * A * S, s_child.data(), (size_t)rows * S);
        // 2x2x2: a column byte left at 255 means some row names a cubelet twice (any_unset_column of expand.cu)
        bool literal = false;
        for (int i = 0; SIZE == 2 && i < rows * R; ++i) literal |= colc[i] == 255;
        for (int i = 0; SIZE == 2 && i < cnt * R; ++i) literal |= colp[i] == 255;
        for (int pass = 0; pass < 2; ++pass) {
            uint8_t* dst = pass == 0 ? child_oh : parent_oh;
            if (!dst) continue;
            const int nr = pass == 0 ? rows : cnt;
            const uint8_t* col = pass == 0 ? colc.data() : colp.data();
            const uint8_t* src = pass == 0 ? s_child.data() : s_par;
            dst += base * (pass == 0 ? A : 1) * (long long)(G::D * ES);
            if ((nr * G::D * ES) % 16 == 0 && !literal) {
                const int n_vec = nr * R * C / OneHot<DTYPE>::V;
                for (int v = 0; v < n_vec; ++v) {
                    uint32_t w[4];
                    onehot_vector<DTYPE, C>(v, col, nr * R, w);
                    std::memcpy(dst + 16 * (long long)v, w, 16);
                }
            } else {
                for (int e = 0; e < nr * G::D; ++e) {
                    const int seg = e / C;
                    const bool one = (SIZE == 2 && literal)
                                         ? onehot2_element(src + (seg / R) * S, seg % R, e % C, def, lut0)
                                         : col[seg] == e % C;
                    if (DTYPE == 0) reinterpret_cast<uint16_t*>(dst)[e] = one ? 0x3f80 : 0;
                    else if (DTYPE == 1) reinterpret_cast<uint32_t*>(dst)[e] = one ? 0x3f800000u : 0u;
                    else dst[e] = one ? 1 : 0;
                }
            }
        }
    }
}
}  // namespace

extern "C" {
void emul_scramble(int size, const uint8_t* moves, long long n, int depth, uint8_t* out, uint8_t* solved)
{
    if (size == 3) scramble_t<3>(moves, n, depth, out, solved); else scramble_t<2>(moves, n, depth, out, solved);
}
// fixed & 3 == 1: use the compile-time-depth instantiation when one exists (30, 20; 43 only here, to
// exercise the unrolled fold schedule); == 2: the swizzled move tile (depth % 8 == 0 for 3x3x3,
// % 16 == 0 for 2x2x2); fixed & 4: four instances per lane, 128-row tiles (2x2x2 only)
void emul_scramble_pairs(int size, const uint8_t* moves, long long n, int depth, uint8_t* out, uint8_t* solved, int fixed)
{
    const bool fix = (fixed & 3) == 1, swz = (fixed & 3) == 2;
    if (size == 3) scramble_pairs_t<3, 2>(moves, n, depth, out, solved, fix, swz);
    else if (fixed & 4) scramble_pairs_t<2, 4>(moves, n, depth, out, solved, fix, swz);
    else scramble_pairs_t<2, 2>(moves, n, depth, out, solved, fix, swz);
}
// cube_scramble_step through the pair kernel: the walk, then one more face turn from `last` (whole tiles only)
void emul_scramble_step_pairs(int size, const uint8_t* moves, const uint8_t* last, long long n, int depth, uint8_t* out,
                              uint8_t* solved, int fixed)
{
    const bool fix = (fixed & 3) == 1, swz = (fixed & 3) == 2;
    if (size == 3) scramble_pairs_t<3, 2>(moves, n, depth, out, solved, fix, swz, last);
    else if (fixed & 4) scramble_pairs_t<2, 4>(moves, n, depth, out, solved, fix, swz, last);
    else scramble_pairs_t<2, 2>(moves, n, depth, out, solved, fix, swz, last);
}
// K1p sliced (deep scrambles; `last` may be null); `moves` readable 16 bytes past its end
void emul_scramble_sliced(int size, const uint8_t* moves, const uint8_t* last, long long n, int depth, uint8_t* out, uint8_t* solved,
                          int slice)
{
    if (size == 3) scramble_sliced_t<3>(moves, n, depth, out, solved, last, slice);
    else scramble_sliced_t<2>(moves, n, depth, out, solved, last, slice);
}
// cube_scramble_prefixes: out [n, depth, S] cube-major, solved [n, depth]
void emul_prefixes(int size, const uint8_t* moves, long long n, int depth, uint8_t* out, uint8_t* solved)
{
    if (size == 3) prefixes_t<3>(moves, n, depth, out, solved); else prefixes_t<2>(moves, n, depth, out, solved);
}
void emul_walk(int size, const uint8_t* in, const uint8_t* moves, long long n, int depth, uint8_t* out,
               uint8_t* solved)
{
    if (size == 3) walk_t<3>(in, moves, n, depth, out, solved); else walk_t<2>(in, moves, n, depth, out, solved);
}
void emul_walk_private(int size, const uint8_t* in, const uint8_t* moves, long long n, int depth, uint8_t* out,
                       uint8_t* solved)
{
    if (size == 3) walk_private_t<3>(in, moves, n, depth, out, solved);
    else walk_private_t<2>(in, moves, n, depth, out, solved);
}
void emul_expand(int size, int dtype, const uint8_t* states, long long n, uint8_t* children, uint8_t* child_oh,
                 uint8_t* parent_oh, uint8_t* solved)
{
#define CASE(SZ, DT) if (size == SZ && dtype == DT) return expand_t<SZ, DT>(states, n, children, child_oh, parent_oh, solved);
    CASE(3, 0) CASE(3, 1) CASE(3, 2) CASE(2, 0) CASE(2, 1) CASE(2, 2)
#undef CASE
}
}
