// Per-thread bodies of the cube kernels, host+device (CUBE_HD) so that the test-only
// emulation harness (tests/host_emul/) can run exactly this code on the CPU.
#pragma once
#include <cstdlib>
#include "cube_common.cuh"

// ---- K1: fused scramble -------------------------------------------------------------------
template <int SIZE>
CUBE_HD void scramble_apply_word(CubieState& st, const uint32_t* s_tbl, uint32_t w)
{
    // byte offsets of the four table rows: (m & 15) * 4 per byte (rows 12..15 are identity),
    // then one byte-extract per move
    const uint32_t w4 = (w * 4u) & 0x3c3c3c3cu;
#pragma unroll
    for (int k = 0; k < 4; ++k) cubie_move_at<SIZE>(st, s_tbl, cube_prmt(w4, 0u, 0x4440u + k));
}

// moves of the tile are a flat byte image in s_moves (row `tid` at byte tid*depth, any alignment)
template <int SIZE>
CUBE_HD void scramble_run_staged(CubieState& st, int tid, int depth, const uint8_t* s_moves, const uint32_t* s_tbl)
{
    const uint32_t* mw = reinterpret_cast<const uint32_t*>(s_moves);
    const uint32_t r = (uint32_t)tid * (uint32_t)depth;
    const uint32_t wi = r >> 2, sh = (r & 3u) << 3;
    const int nfull = depth >> 2, tail = depth & 3;
    uint32_t lo = mw[wi];
#pragma unroll 2
    for (int j = 0; j < nfull; ++j) {
        const uint32_t hi = mw[wi + j + 1];             // may run <= 4 bytes past the row (tile is padded)
        const uint32_t w = cube_funnel_r(lo, hi, sh);
        lo = hi;
        scramble_apply_word<SIZE>(st, s_tbl, w);
        st.c0 = cubie_fold_twist(st.c0);                 // every 4 turns, see cubie_fold_twist
        st.c1 = cubie_fold_twist(st.c1);
    }
    if (tail) {                                          // last 1..3 moves (uniform over the grid)
        const uint32_t w = cube_funnel_r(lo, mw[wi + nfull + 1], sh);
        const uint32_t w4 = (w * 4u) & 0x3c3c3c3cu;
        for (int k = 0; k < tail; ++k) cubie_move_at<SIZE>(st, s_tbl, cube_prmt(w4, 0u, 0x4440u + k));
    }
}

// reduce, judge, expand to stickers and store the row into the shared output tile
template <int SIZE>
CUBE_HD bool scramble_finish(CubieState& st, int tid, const uint32_t* s_clut, const uint32_t* s_elut, uint8_t* s_out)
{
    st.c0 = cubie_reduce_twist(st.c0);
    st.c1 = cubie_reduce_twist(st.c1);
    const bool ok = cubie_is_identity<SIZE>(st);
    uint32_t words[CubeGeom<SIZE>::WORDS];
    cubie_to_stickers<SIZE>(st, s_clut, s_elut, words);
    if (SIZE == 3) {
        // 54-byte rows: odd rows start 2 bytes off a word boundary -> shift by selector, no branch
        const uint32_t odd = (uint32_t)tid & 1u;
        const uint32_t sel = odd ? 0x5432u : 0x3210u;
        uint8_t* rowp = s_out + 54 * tid;
        uint32_t* wbase = reinterpret_cast<uint32_t*>(rowp + 2 * odd);
#pragma unroll
        for (int j = 0; j < 13; ++j) wbase[j] = cube_prmt(words[j], words[j + 1], sel);
        *reinterpret_cast<uint16_t*>(rowp + (odd ? 0 : 52)) = (uint16_t)(odd ? words[0] : words[13]);
    } else {
        // 24-byte rows as three 8-byte stores: a half-warp's 16 rows hit 16 distinct bank pairs
        uint64_t* rowp = reinterpret_cast<uint64_t*>(s_out + 24 * tid);
#pragma unroll
        for (int j = 0; j < 3; ++j) rowp[j] = (uint64_t)words[2 * j] | ((uint64_t)words[2 * j + 1] << 32);
    }
    return ok;
}


// ---- K1x: every prefix of one scramble (cube_scramble_prefixes) ---------------------------------
// `my` = the cube's depth move bytes; row0 = index of its first row in the tile image s_img (rows are the
// tile's output block: cube-major, depth rows per cube).  The caller's lane produces the levels [k_begin, k_end)
// only -- a cube's levels are split over several lanes, each of which first fast-forwards through the moves
// before its share (a move is ~12 instructions, finishing a level ~100) -- and returns the number of solved
// prefixes among them; flags (or null) receives the done flag of every produced level.  The running state stays
// lazy (twist fields folded every 4 moves like the fused scramble); each level is finished on a copy.
template <int SIZE>
CUBE_HD unsigned prefix_walk(const uint8_t* my, int depth, int row0, const uint32_t* s_tbl, const uint32_t* s_clut,
                             const uint32_t* s_elut, uint8_t* s_img, uint8_t* flags, int k_begin, int k_end)
{
    CubieState st;
    cubie_init(st);
    unsigned n_solved = 0;
    (void)depth;
    // fast-forward (trip counts differ between the lanes of a warp, but the body is a dozen instructions) ...
    for (int k = 0; k < k_begin; ++k) {
        cubie_move<SIZE>(st, s_tbl, (uint32_t)my[k] & 0xfu);
        if ((k & 3) == 3) { st.c0 = cubie_fold_twist(st.c0); st.c1 = cubie_fold_twist(st.c1); }
    }
    // ... then the lane's own levels, which the lanes of a warp produce in lockstep (their shares differ by <= 1)
    for (int k = k_begin; k < k_end; ++k) {
        cubie_move<SIZE>(st, s_tbl, (uint32_t)my[k] & 0xfu);
        if ((k & 3) == 3) { st.c0 = cubie_fold_twist(st.c0); st.c1 = cubie_fold_twist(st.c1); }
        CubieState now = st;
        const bool ok = scramble_finish<SIZE>(now, row0 + k, s_clut, s_elut, s_img);
        n_solved += ok ? 1u : 0u;
        if (flags) flags[k] = ok ? 1 : 0;
    }
    return n_solved;
}

// ---- K1p: fused scramble, two moves per table row --------------------------------------------
// The pair table lives in shared memory as TWO arrays of 128-byte rows (the second kPairSecond bytes behind
// the first), every vector replicated once per lane slot: 3x3x3 rows are the two 16-byte vectors P and Q x 8
// slots each; 2x2x2 rows are (selectors, T0) as 8 bytes x 16 slots and T1 as 4 bytes x 32 slots.  A lane only
// ever reads its own slot, so the 128- / 64- / 32-bit loads of a quarter / half / whole warp touch disjoint
// banks whatever rows the lanes ask for: no bank conflicts by construction.
// `lanereg` = the address of the lane's slot in row 0 of the first array; the address of a pair's row is then
// ONE byte dot product with the word that carries the pair indices in bytes 1 and 3 (weight 128 on the wanted
// byte, `lanereg` as the accumulator): IDP.4A issues on the FMA pipe, which idles while PRMT / LOP3 keep the
// ALU pipe busy.  (Until round 2 the rows were 256 bytes and the address a PRMT of the pair byte over the slot
// byte: one more instruction on the binding pipe per pair.)
constexpr int kPairSecond = CUBE_PAIR_ROWS * 128;

template <int HALF>
CUBE_HD uint32_t pair_addr(uint32_t y, uint32_t lanereg)        // HALF 0: the pair in byte 1 of y, 1: in byte 3
{
    return cube_dp4a(y, HALF ? 0x80000000u : 0x00008000u, lanereg);
}

struct CubeVec4 { uint32_t x, y, z, w; };

CUBE_HD CubeVec4 cube_ld128(const uint8_t* p)
{
#if defined(__CUDA_ARCH__)
    const uint4 v = *reinterpret_cast<const uint4*>(p);
    return CubeVec4{v.x, v.y, v.z, v.w};
#else
    CubeVec4 v;
    if (reinterpret_cast<uintptr_t>(p) & 15) abort();    // the device's 128-bit load would fault
    const uint32_t* q = reinterpret_cast<const uint32_t*>(p);
    v.x = q[0]; v.y = q[1]; v.z = q[2]; v.w = q[3];
    return v;
#endif
}

// Where the pair table is read from.  Host (test emulation): a plain pointer, addresses relative to it.
// Device: absolute 32-bit shared-window addresses (`lanereg` includes the table's).
struct PairTableHost {
    const uint8_t* base;
    CUBE_HD uint32_t origin() const { return 0u; }
    CUBE_HD CubeVec4 ld(uint32_t addr, int off) const { return cube_ld128(base + addr + off); }
    CUBE_HD void ld64(uint32_t addr, uint32_t& x, uint32_t& y) const
    {
        const uint32_t* q = reinterpret_cast<const uint32_t*>(base + addr);
        x = q[0]; y = q[1];
    }
    CUBE_HD uint32_t ld32(uint32_t addr) const { return *reinterpret_cast<const uint32_t*>(base + addr); }
};
#if defined(__CUDACC__)
struct PairTableShared {
    uint32_t origin_;                                   // shared-window address of the table
    __device__ __forceinline__ uint32_t origin() const { return origin_; }
    __device__ __forceinline__ CubeVec4 ld(uint32_t addr, int off) const
    {
        CubeVec4 v;
        if (off == 0)
            asm("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
        else
            asm("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4+%5];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr), "n"(kPairSecond));
        return v;
    }
    __device__ __forceinline__ void ld64(uint32_t addr, uint32_t& x, uint32_t& y) const
    {
        asm("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(x), "=r"(y) : "r"(addr));
    }
    __device__ __forceinline__ uint32_t ld32(uint32_t addr) const
    {
        uint32_t v;
        asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
        return v;
    }
};
#endif

// Colour LUT access of the finishing pass.  Host: pointers.  Device: "base + 4 * cubie byte q" is ONE
// dot-product instruction (weights 4 << 8q, accumulator = the LUT's shared-window address): byte
// extraction, scaling and address arithmetic on the FMA pipe instead of PRMT + shift on the ALU pipe.
// Edges have one 32-entry LUT PER SLOT (kEdgeColourSlot3: bytes 2, 3 carry the centre colours of the slot's
// faces for the row assembly); the slot's LUT is an immediate offset of the load.
struct ColourLutHost {
    const uint32_t* c;
    const uint32_t* e;                                  // [12][32]
    // x = four cubie bytes; entry of byte q
    CUBE_HD uint32_t corner(uint32_t x, int q) const { return cube_lut_at(c, cube_dp4a(x, 4u << (8 * q), 0u)); }
    template <int SLOT> CUBE_HD uint32_t edge(uint32_t x) const
    {
        return cube_lut_at(e + 32 * SLOT, cube_dp4a(x, 4u << (8 * (SLOT & 3)), 0u));
    }
};
#if defined(__CUDACC__)
struct ColourLutShared {
    uint32_t cbase, ebase;                              // shared-window addresses
    static __device__ __forceinline__ uint32_t lds32(uint32_t addr)
    {
        uint32_t v;
        asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
        return v;
    }
    __device__ __forceinline__ uint32_t corner(uint32_t x, int q) const { return lds32(cube_dp4a(x, 4u << (8 * q), cbase)); }
    template <int SLOT> __device__ __forceinline__ uint32_t edge(uint32_t x) const
    {
        uint32_t v;
        asm("ld.shared.u32 %0, [%1+%2];" : "=r"(v) : "r"(cube_dp4a(x, 4u << (8 * (SLOT & 3)), ebase)), "n"(128 * SLOT));
        return v;
    }
};
#endif

template <int SIZE, class TBL>
CUBE_HD uint32_t pair_lanereg(int lane, const TBL& tbl)
{
    return tbl.origin() + (SIZE == 3 ? (uint32_t)(lane & 7) << 4 : (uint32_t)(lane & 15) << 3);
}

// 2x2x2: the lane's T1 slot (32 x 4 bytes per row of the second array) relative to its (selectors, T0) slot
CUBE_HD uint32_t pair_roff2(int lane)
{
    return (uint32_t)kPairSecond + (uint32_t)lane * 4u - ((uint32_t)(lane & 15) << 3);
}

// fill the shared-memory image from kPairWords{3,2}; thread `t` of `nthreads`
template <int SIZE>
CUBE_HD void pair_table_fill(uint8_t* s_ptbl, int t, int nthreads)
{
    for (int i = t; i < CUBE_PAIR_ROWS * 16; i += nthreads) {
        const int row = i >> 4, slot = i & 15;
        if (SIZE == 3) {
            const uint32_t* v = kPairWords3 + (row * 2 + (slot >> 3)) * 4;       // slots 0..7: P, 8..15: Q
            uint32_t* d = reinterpret_cast<uint32_t*>(s_ptbl + (slot >> 3) * kPairSecond + row * 128 + (slot & 7) * 16);
            d[0] = v[0]; d[1] = v[1]; d[2] = v[2]; d[3] = v[3];
        } else {
            const uint32_t* v = kPairWords2 + row * 4;
            uint32_t* d = reinterpret_cast<uint32_t*>(s_ptbl + row * 128);
            uint32_t* d1 = reinterpret_cast<uint32_t*>(s_ptbl + kPairSecond + row * 128);
            d[2 * slot] = v[0]; d[2 * slot + 1] = v[1];
            d1[2 * slot] = v[2]; d1[2 * slot + 1] = v[2];
        }
    }
}

// two face turns: one row of the pair table (gen_tables.py pair_words_3 / pair_words_2)
template <int SIZE, class TBL>
CUBE_HD void pair_apply(CubieState& s, const TBL& tbl, uint32_t addr, uint32_t roff)
{
    if (SIZE == 3) {
        const CubeVec4 P = tbl.ld(addr, 0);
        const uint32_t n0 = cube_prmt(s.c0, s.c1, P.x) + P.y;
        const uint32_t n1 = cube_prmt(s.c0, s.c1, cube_hi16(P.x)) + P.z;
        s.c0 = n0; s.c1 = n1;
        const CubeVec4 Q = tbl.ld(addr, kPairSecond);
        const uint32_t t0 = cube_prmt(s.e1, s.e2, Q.x);
        const uint32_t t1 = cube_prmt(s.e0, s.e2, Q.y);
        const uint32_t t2 = cube_prmt(s.e0, s.e1, Q.z);
        const uint32_t m0 = cube_prmt(s.e0, t0, cube_hi16(Q.x)) ^ (P.w & 0x10101010u);
        const uint32_t m1 = cube_prmt(s.e1, t1, cube_hi16(Q.y)) ^ Q.w;
        const uint32_t m2 = cube_prmt(s.e2, t2, cube_hi16(Q.z)) ^ (P.w & 0x20202020u);
        s.e0 = m0; s.e1 = m1; s.e2 = m2;
    } else {
        uint32_t sel, t0w;
        tbl.ld64(addr, sel, t0w);
        const uint32_t t1w = tbl.ld32(addr + roff);
        const uint32_t n0 = cube_prmt(s.c0, s.c1, sel) + t0w;
        const uint32_t n1 = cube_prmt(s.c0, s.c1, cube_hi16(sel)) + t1w;
        s.c0 = n0; s.c1 = n1;
    }
}

// Moves of the tile are a flat byte image (row `row` at byte row*depth, any alignment; readable
// up to 8 bytes past the last row).  A pair adds at most 2 to a twist field, so 15 pairs
// (depth <= 30) never need a fold; the generic path folds after every complete group of 5 words
// (10 pairs: <= 10 + 20 stays below 32).  DEPTH > 0 fixes the depth at compile time (straight-line code for
// the reference's default scramble depth, config.yaml:7 sample_scramble_count = 30, and
// BASELINE config 2's depth 20); DEPTH == 0 takes it from `depth_rt`.
// Byte shift of instance k's move stream relative to the word grid when it is the same for every
// lane (compile-time depth, the kernel's lane -> row maps: 3x3x3 rows 2l + k, 2x2x2 rows l + 32k);
// -1 = depends on the lane.
template <int SIZE, int DEPTH>
CUBE_HD constexpr int pair_static_shift(int k)
{
    return DEPTH <= 0 ? -1
         : SIZE == 3 ? ((2 * DEPTH) % 4 == 0 ? ((k * DEPTH) % 4) * 8 : -1)
                     : (DEPTH % 4 == 0 ? 0 : -1);
}

// pair rows (bytes 1 and 3) of the next four moves: (move word) * 269.  With a static shift
// the funnel shift (ALU pipe) is folded into multiply-adds (FMA pipe):
//   shift 0: lo * 269;   shift 16: (lo >> 16) * 269 + hi * (269 << 16)   (mod 2^32, like the product)
template <int SSH>
CUBE_HD uint32_t pair_rows_word(uint32_t lo, uint32_t hi, uint32_t sh)
{
    constexpr uint32_t K = (uint32_t)(CUBE_PAIR_BASE + 256);
    if (SSH == 0) return lo * K;
    if (SSH == 16) return hi * (K << 16) + cube_hi16(lo) * K;
    return cube_funnel_r(lo, hi, sh) * K;
}

template <int SIZE, int DEPTH, int NS, class TBL>
CUBE_HD void scramble_pairs_run(CubieState (&st)[NS], const int (&rows)[NS], int depth_rt, const uint8_t* s_moves,
                                const TBL& tbl, uint32_t lanereg, uint32_t roff)
{
    // NS instances per lane advance in lockstep (independent dependency chains for the scheduler)
    const int depth = DEPTH > 0 ? DEPTH : depth_rt;
    const uint32_t* mw = reinterpret_cast<const uint32_t*>(s_moves);
    const int nfull = depth >> 2, tail = depth & 3;
    uint32_t wi[NS], sh[NS], lo[NS];
#pragma unroll
    for (int k = 0; k < NS; ++k) {
        const uint32_t r = (uint32_t)rows[k] * (uint32_t)depth;
        wi[k] = r >> 2; sh[k] = (r & 3u) << 3;
        lo[k] = mw[wi[k]];
    }
    auto word = [&](int j) {
        uint32_t y[NS];
        static_assert(NS == 1 || NS % 2 == 0, "instances come in pairs");
        if (SIZE == 3 || NS <= 2) {
            // 3x3x3: instances 2h, 2h+1 are the rows 2l, 2l+1 of the h-th 64 rows of the tile; 64 rows are a
            // whole number of words for an even depth, so the static shift depends on the row's parity only
            {
                constexpr int s0 = (NS >= 2) ? pair_static_shift<SIZE, DEPTH>(0) : -1;
#pragma unroll
                for (int h = 0; h < NS; h += 2) {
                    const uint32_t hi = (s0 == 0) ? 0u : mw[wi[h] + j + 1];
                    y[h] = pair_rows_word<s0>(lo[h], hi, sh[h]);              // bytes 1, 3 = pair rows
                    lo[h] = (s0 == 0) ? mw[wi[h] + j + 1] : hi;
                }
            }
            if (NS >= 2) {
                constexpr int s1 = pair_static_shift<SIZE, DEPTH>(1);
#pragma unroll
                for (int h = 1; h < NS; h += 2) {
                    const uint32_t hi = (s1 == 0) ? 0u : mw[wi[h] + j + 1];
                    y[h] = pair_rows_word<s1>(lo[h], hi, sh[h]);
                    lo[h] = (s1 == 0) ? mw[wi[h] + j + 1] : hi;
                }
            }
        } else {
            constexpr int s = pair_static_shift<2, DEPTH>(0);                       // 2x2x2: the same for every row
#pragma unroll
            for (int k = 0; k < NS; ++k) {
                const uint32_t hi = (s == 0) ? 0u : mw[wi[k] + j + 1];
                y[k] = pair_rows_word<s>(lo[k], hi, sh[k]);
                lo[k] = (s == 0) ? mw[wi[k] + j + 1] : hi;
            }
        }
#pragma unroll
        for (int k = 0; k < NS; ++k) pair_apply<SIZE>(st[k], tbl, pair_addr<0>(y[k], lanereg), roff);
#pragma unroll
        for (int k = 0; k < NS; ++k) pair_apply<SIZE>(st[k], tbl, pair_addr<1>(y[k], lanereg), roff);
    };
    auto fold = [&]() {
#pragma unroll
        for (int k = 0; k < NS; ++k) {
            st[k].c0 = cubie_fold_twist(st[k].c0);
            st[k].c1 = cubie_fold_twist(st[k].c1);
        }
    };
    if (DEPTH > 0) {
#pragma unroll
        for (int j = 0; j < DEPTH / 4; ++j) {
            word(j);
            if (DEPTH > 30 && (j % 5 == 4 || j == DEPTH / 4 - 1)) fold();
        }
    } else {
        // groups of five words (ten pairs: a field grows by <= 20), each followed by a fold (<= 31 -> <= 10);
        // the <= 4 words left over and the tail add <= 16 + 4 on top of <= 10: no further fold needed
        int j = 0;
        for (; j + 5 <= nfull; j += 5) {
            word(j); word(j + 1); word(j + 2); word(j + 3); word(j + 4);
            fold();
        }
        for (; j < nfull; ++j) word(j);
    }
    if (tail) {                                          // last 1..3 moves, padded with the no-move index
        const uint32_t keep = (1u << (8 * tail)) - 1u;
        uint32_t y[NS];
#pragma unroll
        for (int k = 0; k < NS; ++k) {
            const uint32_t w = (cube_funnel_r(lo[k], mw[wi[k] + nfull + 1], sh[k]) & keep) | (0x0c0c0c0cu & ~keep);
            y[k] = w * (uint32_t)(CUBE_PAIR_BASE + 256);
        }
#pragma unroll
        for (int k = 0; k < NS; ++k) pair_apply<SIZE>(st[k], tbl, pair_addr<0>(y[k], lanereg), roff);
        if (tail == 3) {
#pragma unroll
            for (int k = 0; k < NS; ++k) pair_apply<SIZE>(st[k], tbl, pair_addr<1>(y[k], lanereg), roff);
        }
    }
}

// A SLICE of a deep scramble (depth > 320, scramble_sliced_kernel): `len` moves per instance, applied to a state
// that is carried over from the previous slice.  Instance k's bytes start shift[k] (0..15) bytes into the 16-byte
// aligned slot at offset base[k] of s_moves (the slot was filled from the 16-byte boundary below the piece).  The
// moves are read sixteen bytes at a time with 128-bit loads -- 32-bit loads would bank-conflict 4- to 8-fold,
// because slots can only be 16-byte aligned -- and the per-row byte shift is taken out in registers: a two-level
// word select on (shift >> 2) and a funnel shift by (shift & 3) bytes.  A fold first (the previous slice may have
// left a twist field at 26), then one after every unit (a unit adds <= 16 to <= 10); the <= 15 moves left add <= 16.
template <int SIZE, int NS, class TBL>
CUBE_HD void scramble_pairs_run_units(CubieState (&st)[NS], const uint32_t (&base)[NS], const uint32_t (&shift)[NS], int len,
                                      const uint8_t* s_moves, const TBL& tbl, uint32_t lanereg, uint32_t roff)
{
    constexpr uint32_t K = (uint32_t)(CUBE_PAIR_BASE + 256);
    auto fold = [&]() {
#pragma unroll
        for (int k = 0; k < NS; ++k) {
            st[k].c0 = cubie_fold_twist(st[k].c0);
            st[k].c1 = cubie_fold_twist(st[k].c1);
        }
    };
    auto word = [&](const uint32_t (&w)[NS], bool second) {
        uint32_t y[NS];
#pragma unroll
        for (int k = 0; k < NS; ++k) y[k] = w[k] * K;
#pragma unroll
        for (int k = 0; k < NS; ++k) pair_apply<SIZE>(st[k], tbl, pair_addr<0>(y[k], lanereg), roff);
        if (second) {
#pragma unroll
            for (int k = 0; k < NS; ++k) pair_apply<SIZE>(st[k], tbl, pair_addr<1>(y[k], lanereg), roff);
        }
    };
    // the 16 move bytes that start `shift` bytes into the unit pair (a, b), as four words
    auto aligned = [&](const CubeVec4& a, const CubeVec4& b, uint32_t sh, uint32_t (&o)[4]) {
        const bool q0 = (sh & 4u) != 0, q1 = (sh & 8u) != 0;
        const uint32_t c[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        uint32_t e[7], d[5];
#pragma unroll
        for (int j = 0; j < 7; ++j) e[j] = q0 ? c[j + 1] : c[j];
#pragma unroll
        for (int j = 0; j < 5; ++j) d[j] = q1 ? e[j + 2] : e[j];
        const uint32_t r = (sh & 3u) << 3;
#pragma unroll
        for (int j = 0; j < 4; ++j) o[j] = cube_funnel_r(d[j], d[j + 1], r);
    };
    fold();
    CubeVec4 cur[NS];
#pragma unroll
    for (int k = 0; k < NS; ++k) cur[k] = cube_ld128(s_moves + base[k]);
    int g = 0;
    for (; g + 16 <= len; g += 16) {
        CubeVec4 nxt[NS];
        uint32_t m[NS][4], w[NS];
#pragma unroll
        for (int k = 0; k < NS; ++k) {
            nxt[k] = cube_ld128(s_moves + base[k] + g + 16);
            aligned(cur[k], nxt[k], shift[k], m[k]);
            cur[k] = nxt[k];
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
#pragma unroll
            for (int k = 0; k < NS; ++k) w[k] = m[k][j];
            word(w, true);
        }
        fold();
    }
    const int rem = len - g;                             // 0..15 moves left (the same for every instance)
    if (rem) {
        uint32_t m[NS][4], w[NS];
#pragma unroll
        for (int k = 0; k < NS; ++k) {
            const CubeVec4 nxt = cube_ld128(s_moves + base[k] + g + 16);
            aligned(cur[k], nxt, shift[k], m[k]);
        }
        const int nwords = rem >> 2, tail = rem & 3;
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            if (j < nwords) {
#pragma unroll
                for (int k = 0; k < NS; ++k) w[k] = m[k][j];
                word(w, true);
            }
        }
        if (tail) {                                      // last 1..3 moves, padded with the no-move index
            const uint32_t keep = (1u << (8 * tail)) - 1u;
#pragma unroll
            for (int k = 0; k < NS; ++k) {
                const uint32_t t = nwords == 0 ? m[k][0] : nwords == 1 ? m[k][1] : nwords == 2 ? m[k][2] : m[k][3];
                w[k] = (t & keep) | (0x0c0c0c0cu & ~keep);
            }
            word(w, tail == 3);
        }
    }
}

// cube_scramble_step: one more face turn after the walk -- the pair row (action, no move).  The fold first:
// the walk may leave a twist field at 30, and a turn adds up to 2.
template <int SIZE, class TBL>
CUBE_HD void scramble_pairs_last(CubieState& st, uint32_t action, const TBL& tbl, uint32_t lanereg, uint32_t roff)
{
    st.c0 = cubie_fold_twist(st.c0);
    st.c1 = cubie_fold_twist(st.c1);
    const uint32_t y = (action | 0x0c0c0c00u) * (uint32_t)(CUBE_PAIR_BASE + 256);
    pair_apply<SIZE>(st, tbl, pair_addr<0>(y, lanereg), roff);
}

// Swizzled move tile.  In the flat tile image a lane's move words are `rows * depth` bytes apart: when
// that stride shares a large power of two with the 32 banks (depth 32: 16 words, depth 64: 32 words) every
// move-word load of the warp serialises 16- or 32-fold.  For depths that are multiples of 8 (3x3x3) / 16
// (2x2x2) the kernel stages the tile with ONE 2-D tensor copy whose shared-memory side uses the copy
// engine's 128-byte swizzle: the 16-byte unit at flat offset f lands at f ^ (((f >> 7) & 7) << 4).  The
// moves are then read sixteen at a time with 128-bit loads; the eight lanes of a quarter warp, 2*depth
// bytes apart, fall into (nearly always) eight different bank groups.  `tile` is the buffer (1024-byte
// aligned in the shared window), `lane` the lane: 3x3x3 rows 2l, 2l+1 are the contiguous slice at
// lane * 2 * depth, 2x2x2 rows l + 32k sit at (lane + 32k) * depth.  A group of four words
// adds <= 16 to a twist field and the fold after it leaves <= 10, so a field never exceeds 26.
CUBE_HD uint32_t cube_swz128(uint32_t f) { return f ^ ((f >> 3) & 0x70u); }

template <int SIZE, int NS, class TBL>
CUBE_HD void scramble_pairs_run_swizzled(CubieState (&st)[NS], const uint8_t* tile, int lane, int depth, const TBL& tbl,
                                         uint32_t lanereg, uint32_t roff)
{
    constexpr uint32_t K = (uint32_t)(CUBE_PAIR_BASE + 256);
    static_assert(SIZE == 2 || NS == 2, "3x3x3: two rows per lane");
    auto word = [&](const uint32_t (&w)[NS]) {
        uint32_t y[NS];
#pragma unroll
        for (int k = 0; k < NS; ++k) y[k] = w[k] * K;
#pragma unroll
        for (int k = 0; k < NS; ++k) pair_apply<SIZE>(st[k], tbl, pair_addr<0>(y[k], lanereg), roff);
#pragma unroll
        for (int k = 0; k < NS; ++k) pair_apply<SIZE>(st[k], tbl, pair_addr<1>(y[k], lanereg), roff);
    };
    auto fold = [&]() {
#pragma unroll
        for (int k = 0; k < NS; ++k) {
            st[k].c0 = cubie_fold_twist(st[k].c0);
            st[k].c1 = cubie_fold_twist(st[k].c1);
        }
    };
    auto unit = [&](uint32_t f) { return cube_ld128(tile + cube_swz128(f)); };
    if (SIZE == 3 && (depth & 8)) {
        // depth = 16a + 8: row 1 starts in the middle of 16-byte unit a of the lane's slice.  Row 0's words
        // 4g..4g+3 are unit g; row 1's are the upper half of unit a+g and the lower half of unit a+g+1
        // (carried over in `p`).
        const int a = depth >> 4;
        const uint32_t f0 = (uint32_t)(lane * 2 * depth);
        CubeVec4 p = unit(f0 + 16 * a);
        const uint32_t last0[2] = {p.x, p.y};
        auto word2 = [&](uint32_t w0, uint32_t w1) {
            uint32_t w[NS];
            w[0] = w0; w[NS - 1] = w1;
            word(w);
        };
        for (int g = 0; g < a; ++g) {
            const CubeVec4 v = unit(f0 + 16 * g), q = unit(f0 + 16 * (a + g + 1));
            word2(v.x, p.z);
            word2(v.y, p.w);
            word2(v.z, q.x);
            word2(v.w, q.y);
            p = q;
            fold();
        }
        word2(last0[0], p.z);
        word2(last0[1], p.w);
        return;
    }
    uint32_t f[NS];
#pragma unroll
    for (int k = 0; k < NS; ++k) f[k] = (uint32_t)((SIZE == 3 ? 2 * lane + k : lane + 32 * k) * depth);
    for (int g = 0; g < depth; g += 16) {                // rows 16-byte aligned (depth % 16 == 0)
        CubeVec4 v[NS];
#pragma unroll
        for (int k = 0; k < NS; ++k) v[k] = unit(f[k] + g);
        uint32_t w[NS];
#pragma unroll
        for (int k = 0; k < NS; ++k) w[k] = v[k].x;
        word(w);
#pragma unroll
        for (int k = 0; k < NS; ++k) w[k] = v[k].y;
        word(w);
#pragma unroll
        for (int k = 0; k < NS; ++k) w[k] = v[k].z;
        word(w);
#pragma unroll
        for (int k = 0; k < NS; ++k) w[k] = v[k].w;
        word(w);
        fold();
    }
}

CUBE_HD uint32_t cube_shr1(uint32_t x)          // x >> 1 on the FMA pipe
{
#if defined(__CUDA_ARCH__)
    uint32_t r;
    asm("mul.hi.u32 %0, %1, 2147483648;" : "=r"(r) : "r"(x));
    return r;
#else
    return x >> 1;
#endif
}

// edge byte piece | a << 4 | b << 5  ->  piece | (a ^ b) << 4: every (piece, flip) then has ONE
// entry in the 32-entry colour LUT, one entry per bank, so the lookups never conflict
CUBE_HD uint32_t cubie_canonical_flip(uint32_t e)
{
    return ((cube_shr1(e) & 0x10101010u) ^ e) & 0x1f1f1f1fu;
}

// reduce, judge, expand to stickers and store the row into a 64-row shared output tile.
// 3x3x3: `row`'s parity must be uniform over the warp (odd rows sit two bytes off the word grid
// and use the pre-shifted assembly), so the two warps of a pair take the even and the odd rows.
template <int SIZE, class LUT>
CUBE_HD bool scramble_pairs_finish(CubieState& st, int row, const LUT& lut, uint8_t* s_out)
{
    st.c0 = cubie_reduce_twist(st.c0);
    st.c1 = cubie_reduce_twist(st.c1);
    bool ok = (st.c0 == 0x03020100u) & (st.c1 == 0x07060504u);
    uint32_t L[20];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        L[q] = lut.corner(st.c0, q);
        L[4 + q] = lut.corner(st.c1, q);
    }
    if (SIZE == 3) {
        const uint32_t f0 = cubie_canonical_flip(st.e0), f1 = cubie_canonical_flip(st.e1), f2 = cubie_canonical_flip(st.e2);
        ok = ok && ((f0 == 0x03020100u) & (f1 == 0x07060504u) & (f2 == 0x0b0a0908u));
        L[8] = lut.template edge<0>(f0);   L[9] = lut.template edge<1>(f0);   L[10] = lut.template edge<2>(f0);  L[11] = lut.template edge<3>(f0);
        L[12] = lut.template edge<4>(f1);  L[13] = lut.template edge<5>(f1);  L[14] = lut.template edge<6>(f1);  L[15] = lut.template edge<7>(f1);
        L[16] = lut.template edge<8>(f2);  L[17] = lut.template edge<9>(f2);  L[18] = lut.template edge<10>(f2); L[19] = lut.template edge<11>(f2);
        uint32_t w[13], h;
        uint8_t* rowp = s_out + 54 * row;
        if (row & 1) {
            cube_assemble3_odd(L, w, &h);
            *reinterpret_cast<uint16_t*>(rowp) = (uint16_t)h;
            uint32_t* wb = reinterpret_cast<uint32_t*>(rowp + 2);
#pragma unroll
            for (int j = 0; j < 13; ++j) wb[j] = w[j];
        } else {
            cube_assemble3_even(L, w, &h);
            uint32_t* wb = reinterpret_cast<uint32_t*>(rowp);
#pragma unroll
            for (int j = 0; j < 13; ++j) wb[j] = w[j];
            *reinterpret_cast<uint16_t*>(rowp + 52) = (uint16_t)h;
        }
    } else {
        uint32_t w[6];
        cube_assemble2(L, w);
        uint64_t* rowp = reinterpret_cast<uint64_t*>(s_out + 24 * row);
#pragma unroll
        for (int j = 0; j < 3; ++j) rowp[j] = (uint64_t)w[2 * j] | ((uint64_t)w[2 * j + 1] << 32);
    }
    return ok;
}

// verdicts of a 64-row tile from the warp ballots of its two passes (m0 = first, m1 = second).
// 3x3x3: row 2l+p is bit l of m_p; 2x2x2: row l+32p is bit l of m_p.
template <int SIZE>
CUBE_HD uint32_t pair_row_bit(uint32_t m0, uint32_t m1, int row)
{
    if (SIZE == 3) return (((row & 1) ? m1 : m0) >> (row >> 1)) & 1u;
    return (((row & 32) ? m1 : m0) >> (row & 31)) & 1u;
}

template <int SIZE>
CUBE_HD uint32_t pair_solved_word(uint32_t m0, uint32_t m1, int k)          // solved bytes of rows 4k .. 4k+3
{
    return pair_row_bit<SIZE>(m0, m1, 4 * k) | pair_row_bit<SIZE>(m0, m1, 4 * k + 1) << 8 |
           pair_row_bit<SIZE>(m0, m1, 4 * k + 2) << 16 | pair_row_bit<SIZE>(m0, m1, 4 * k + 3) << 24;
}

// ---- K2: one face turn of a sticker row in shared memory ------------------------------------
template <int SIZE>
CUBE_HD void walk_turn(uint8_t* row, uint32_t m, const uint32_t* s_cyc)
{
#pragma unroll
    for (int c = 0; c < CubeGeom<SIZE>::NCYC; ++c) {
        const uint32_t w = s_cyc[c * CUBE_MOVE_ROWS + m];
        const uint32_t a = w & 0xffu, b = (w >> 8) & 0xffu, cc = (w >> 16) & 0xffu, d = w >> 24;
        const uint8_t vb = row[b], vc = row[cc], vd = row[d], va = row[a];
        row[a] = vb; row[b] = vc; row[cc] = vd; row[d] = va;
    }
}

// face uniformity of a 2-byte-aligned row: s[i] == s[i-1] for every i that does not start a face
template <int SIZE>
CUBE_HD bool row_solved(const uint8_t* row)
{
    constexpr int S = CubeGeom<SIZE>::S, K = S / 6;
    const uint16_t* h = reinterpret_cast<const uint16_t*>(row);
    uint32_t diff = 0;
    uint32_t prev = 0;
#pragma unroll
    for (int i = 0; i < S / 2; ++i) {
        const uint32_t cur = h[i];
        const uint32_t b0 = cur & 0xffu, b1 = cur >> 8;
        if ((2 * i) % K != 0) diff |= b0 ^ prev;
        if ((2 * i + 1) % K != 0) diff |= b1 ^ b0;
        prev = b1;
    }
    return diff == 0;
}


// ---- K2p: moves on resident rows in a lane-private working layout ------------------------------
// A lane keeps its row as an IMAGE of whole words: 2x2x2 the 6 words of the row; 3x3x3 the 14
// words that cover the 54-byte row on the word grid -- even rows start on a word (image byte k =
// sticker k, the last two bytes belong to the next row), odd rows two bytes later (image byte k =
// sticker k - 2, the first two bytes belong to the previous row).  The face turn itself is a byte
// gather at data-dependent offsets, so the image is parked in a scratch area where image word j
// of lane l sits at word 32 j + l: every byte a lane touches is in the lane's own bank, whatever
// the move, and the 4-cycles cost exactly one wavefront per access.
template <int SIZE> struct WalkImage { static constexpr int W = (SIZE == 3) ? 14 : 6; };

CUBE_HD uint32_t walk_private_off(int k) { return (uint32_t)((k >> 2) * 128 + (k & 3)); }

// 8-byte table entry of one sticker 4-cycle (bytes a, b, c, d of kCycles*) for an image that starts
// `shift` bytes before sticker 0: the four scratch offsets, 16 bits each
CUBE_HD void walk_cycle_entry(uint32_t cw, int shift, uint32_t* e)
{
    const int a = (int)(cw & 0xffu) + shift, b = (int)((cw >> 8) & 0xffu) + shift;
    const int c = (int)((cw >> 16) & 0xffu) + shift, d = (int)(cw >> 24) + shift;
    e[0] = walk_private_off(a) | walk_private_off(b) << 16;
    e[1] = walk_private_off(c) | walk_private_off(d) << 16;
}

// one face turn of the lane's image; lane_base = scratch + 4 * lane, ent = [cycle][16 moves][2]
template <int SIZE>
CUBE_HD void walk_turn_private(uint8_t* lane_base, const uint32_t* ent, uint32_t m)
{
#pragma unroll
    for (int c = 0; c < CubeGeom<SIZE>::NCYC; ++c) {
        const uint32_t w0 = ent[(c * CUBE_MOVE_ROWS + m) * 2], w1 = ent[(c * CUBE_MOVE_ROWS + m) * 2 + 1];
        const uint32_t a = w0 & 0xffffu, b = cube_hi16(w0), cc = w1 & 0xffffu, d = cube_hi16(w1);
        const uint8_t vb = lane_base[b], vc = lane_base[cc], vd = lane_base[d], va = lane_base[a];
        lane_base[a] = vb; lane_base[b] = vc; lane_base[cc] = vd; lane_base[d] = va;
    }
}

// 2x2x2: the row is six registers and every child is a compile-time byte gather (<= 6 PRMT,
// gen_tables.py cube_child2), so the turn stays in registers: all six children are formed and the
// lane's own is kept by predicated selects -- no shared-memory traffic at all, no divergence.
template <int A>
CUBE_HD void walk_select_child2(const uint32_t* p, uint32_t m, uint32_t* out)
{
    uint32_t c[6];
    cube_child2<A>(p, c);
#pragma unroll
    for (int j = 0; j < 6; ++j) out[j] = (m == (uint32_t)A) ? c[j] : out[j];
}

CUBE_HD void walk_turn_registers2(uint32_t* w, uint32_t m)            // m >= 6: no move
{
    uint32_t out[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) out[j] = w[j];
    walk_select_child2<0>(w, m, out);
    walk_select_child2<1>(w, m, out);
    walk_select_child2<2>(w, m, out);
    walk_select_child2<3>(w, m, out);
    walk_select_child2<4>(w, m, out);
    walk_select_child2<5>(w, m, out);
#pragma unroll
    for (int j = 0; j < 6; ++j) w[j] = out[j];
}

// face uniformity (py333.py:229-233 / py222 isSolved) of an image held in registers: every sticker
// that does not start a face equals its predecessor.  SHIFT = image byte of sticker 0 (0 or 2).
template <int SIZE, int SHIFT>
CUBE_HD bool image_solved(const uint32_t* w)
{
    constexpr int S = CubeGeom<SIZE>::S, K = S / 6, W = WalkImage<SIZE>::W;
    uint32_t acc = 0;
#pragma unroll
    for (int j = 0; j < W; ++j) {
        uint32_t mask = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int i = 4 * j + k - SHIFT;              // sticker index of image byte 4j+k
            if (i >= 1 && i < S && (i % K) != 0) mask |= 0xffu << (8 * k);
        }
        if (mask) {
            const uint32_t prev = (j == 0) ? (w[0] << 8) : ((w[j] << 8) | (w[j - 1] >> 24));
            acc |= (w[j] ^ prev) & mask;
        }
    }
    return acc == 0;
}

// ---- K3: one-hot columns and vectors ----------------------------------------------------------
template <int DTYPE> struct OneHot;      // V = elements per 16-byte vector
template <> struct OneHot<0> { static constexpr int V = 8, ESIZE = 2; };   // bf16
template <> struct OneHot<1> { static constexpr int V = 4, ESIZE = 4; };   // f32
template <> struct OneHot<2> { static constexpr int V = 16, ESIZE = 1; };  // u8

// 16 bytes with element `p` set to 1
template <int DTYPE>
CUBE_HD void onehot_set(uint32_t* w, int p)
{
    if (DTYPE == 0) {
        const uint32_t v = (p & 1) ? 0x3f800000u : 0x00003f80u;
#pragma unroll
        for (int q = 0; q < 4; ++q) w[q] |= ((p >> 1) == q) ? v : 0u;
    } else if (DTYPE == 1) {
#pragma unroll
        for (int q = 0; q < 4; ++q) w[q] |= (p == q) ? 0x3f800000u : 0u;
    } else {
        const uint32_t v = 1u << (8 * (p & 3));
#pragma unroll
        for (int q = 0; q < 4; ++q) w[q] |= ((p >> 2) == q) ? v : 0u;
    }
}

// The 16-byte vector that starts `off` elements into segment `seg` of a stream of one-hot
// segments of width C; col[s] = position of the 1 in segment s (255 = none).  One byte per segment
// holds the one-hot rows of real states; a 2x2x2 row that names a cubelet twice needs two 1s in a
// segment and is written element by element (onehot2_element).  A vector touches at
// most two segments (V <= C).  Branch-free: onehot_set ignores positions outside [0, V), and a
// 255 column always lands outside; col[] must be readable one entry past the last segment.
template <int DTYPE, int C>
CUBE_HD void onehot_vector_at(int seg, int off, const uint8_t* col, uint32_t* w)
{
    w[0] = w[1] = w[2] = w[3] = 0u;
    onehot_set<DTYPE>(w, (int)col[seg] - off);
    if (C % OneHot<DTYPE>::V != 0) onehot_set<DTYPE>(w, C - off + (int)col[seg + 1]);   // segments straddle vectors
}

// vector number v of the stream
template <int DTYPE, int C>
CUBE_HD void onehot_vector(int v, const uint8_t* col, int n_seg, uint32_t* w)
{
    (void)n_seg;
    const int e0 = v * OneHot<DTYPE>::V;
    const int seg = e0 / C;
    onehot_vector_at<DTYPE, C>(seg, e0 - seg * C, col, w);
}

// column of the 1 for one (row, slot): 3x3x3 returns the column, 2x2x2 returns cubelet | ori << 4 of the
// cubelet at position `slot` (cubelet <= 6 for every byte content: the table holds no other value)
template <int SIZE>
CUBE_HD uint32_t onehot_code(const uint8_t* row, int slot, const uint32_t* s_def, const uint8_t* s_lut0,
                             const uint8_t* s_lut1)
{
    const uint32_t d = s_def[slot];
    const uint32_t a = row[d & 0xffu], b = row[(d >> 8) & 0xffu], c = row[(d >> 16) & 0xffu];
    if (SIZE == 3 && slot >= 8) return s_lut1[(a + 10u * b) & 127u];
    return s_lut0[(a + 2u * b + 10u * c) & 127u];
}

// 2x2x2 one-hot element (cubelet `cubelet`, column `col`) of a sticker row, the reference's loop read literally
// (cube_env.py:141-147: state[cubelet][3 * position + ori] = 1 for every position): 1 exactly when position
// col / 3 holds that cubelet at orientation col % 3.  A row that names a cubelet twice has two 1s in that
// cubelet's one-hot row and none in the missing cubelet's; a per-cubelet column byte cannot say that.
CUBE_HD bool onehot2_element(const uint8_t* row, int cubelet, int col, const uint32_t* s_def, const uint8_t* s_lut0)
{
    const int pos = col / 3;
    return onehot_code<2>(row, pos, s_def, s_lut0, s_lut0) == (uint32_t)(cubelet | (col - 3 * pos) << 4);
}

// 2x2x2: the lowest column set in cubelet `cubelet`'s one-hot row (what argmax gives), 255 for a row without a 1
CUBE_HD uint32_t onehot2_first_column(const uint8_t* row, int cubelet, const uint32_t* s_def, const uint8_t* s_lut0)
{
    uint32_t col = 255u;
    for (int pos = 6; pos >= 0; --pos) {
        const uint32_t code = onehot_code<2>(row, pos, s_def, s_lut0, s_lut0);
        if ((int)(code & 0xfu) == cubelet) col = 3u * pos + (code >> 4);
    }
    return col;
}
