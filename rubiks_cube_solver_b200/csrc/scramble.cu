// K1 -- fused scramble from the solved cube (sm_100a).
//
// Replaces the reference's per-cube Python loop  init_state(); for a in seq: step(a)
// (cube_env.py:62-67 reset, :187-191 get_random_samples) for a whole batch: every
// thread owns one instance, keeps the cube as five registers of cubie bytes and
// applies the whole move sequence with PRMT byte permutes driven by per-move
// selector words in shared memory (see gen_tables.py) -- no branch on the move and
// no intermediate state in HBM.  The final state is expanded to the reference's
// sticker row (identical to chaining s[moveDefs[m]], py333.py:220-222), the
// face-uniformity verdict (py333.py:229-233) and the +-1 reward (cube_env.py:89-104).
//
// HBM traffic per instance: depth (moves in) + S (stickers out) + 1 + 4 bytes.
// One CTA handles one tile of 256 instances.  The tile's move bytes arrive in
// shared memory through one 1-D bulk asynchronous copy (TMA, mbarrier-signalled) and
// its sticker rows leave through one bulk store, so neither costs LSU wavefronts or
// address arithmetic (rows are 54 / 24 bytes: per-thread global stores would touch a
// different sector per lane).  Several CTAs per SM overlap load, compute and store.
// The kernel is bound by the ALU pipe (PRMT/LOP3) and the shared-memory pipe (six
// table words per move), not by HBM -- see DESIGN.md.
#include <cstring>
#include <cuda.h>
#include <cuda_runtime.h>
#include "cube_bulk.cuh"
#include "cube_kernels.h"
#include "cube_launch.cuh"
#include "cube_sched.cuh"
#include "cube_threads.cuh"

namespace {

#ifndef CUBE_SCRAMBLE_MIN_BLOCKS
#define CUBE_SCRAMBLE_MIN_BLOCKS 6      // 40 registers/thread, no spills; 6 CTAs x 8 warps per SM
#endif
constexpr int kTile = 256;              // instances per tile == threads per CTA
constexpr int kMaxStagedDepth = 160;    // deeper sequences are read straight from global

__host__ __device__ constexpr int round16(int x) { return (x + 15) & ~15; }

template <int SIZE>
struct ScrambleSmem {                   // carve-up of the dynamic shared memory
    using G = CubeGeom<SIZE>;
    static constexpr int kTable = 0;
    static constexpr int kCornerLut = kTable + G::MW * CUBE_MOVE_ROWS * 4;
    static constexpr int kEdgeLut = kCornerLut + 32 * 4;
    static constexpr int kBarrier = kEdgeLut + 64 * 4;
    static constexpr int kFlags = kBarrier + 16;          // one solved byte per row of the tile
    static constexpr int kOut = round16(kFlags + kTile);
    static constexpr int kMoves = kOut + round16(kTile * G::S);
    __host__ __device__ static constexpr int bytes(int depth, bool staged)
    {
        return kMoves + (staged ? round16(kTile * depth) + 32 : 0);
    }
};

template <int SIZE>
__device__ __forceinline__ void load_tables(uint8_t* smem, int tid)
{
    using L = ScrambleSmem<SIZE>;
    uint32_t* s_tbl = reinterpret_cast<uint32_t*>(smem + L::kTable);
    uint32_t* s_clut = reinterpret_cast<uint32_t*>(smem + L::kCornerLut);
    uint32_t* s_elut = reinterpret_cast<uint32_t*>(smem + L::kEdgeLut);
    if (tid < CubeGeom<SIZE>::MW * CUBE_MOVE_ROWS) s_tbl[tid] = (SIZE == 3) ? kMoveWords3[tid] : kMoveWords2[tid];
    if (tid >= 128 && tid < 160) s_clut[tid - 128] = (SIZE == 3) ? kCornerColour3[tid - 128] : kCornerColour2[tid - 128];
    if (tid >= 160 && tid < 224) s_elut[tid - 160] = (SIZE == 3) ? kEdgeColour3[tid - 160] : 0u;
}

// one tile per CTA; move bytes staged in shared memory.  FULL: every tile of the grid has 256
// rows (bulk copies); !FULL: the single ragged tile at the end of a batch (plain copies).
// `tile0` is the index of the first tile this launch handles.
template <int SIZE, bool FULL>
__global__ void __launch_bounds__(kTile, CUBE_SCRAMBLE_MIN_BLOCKS)
scramble_tile_kernel(const uint8_t* __restrict__ moves, long long n, long long tile0, int depth,
                     uint8_t* __restrict__ out, uint8_t* __restrict__ solved, float* __restrict__ reward,
                     unsigned long long* __restrict__ counters, const uint8_t* __restrict__ last)
{
    using G = CubeGeom<SIZE>;
    using L = ScrambleSmem<SIZE>;
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t* s_tbl = reinterpret_cast<const uint32_t*>(smem + L::kTable);
    const uint32_t* s_clut = reinterpret_cast<const uint32_t*>(smem + L::kCornerLut);
    const uint32_t* s_elut = reinterpret_cast<const uint32_t*>(smem + L::kEdgeLut);
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(smem + L::kBarrier);
    uint8_t* s_flags = smem + L::kFlags;
    uint8_t* s_out = smem + L::kOut;
    uint8_t* s_moves = smem + L::kMoves;

    const int tid = threadIdx.x;
    // Row of the tile this thread computes.  3x3x3 rows are 54 bytes = 13.5 words, so rows of
    // different parity sit differently on the word grid: warps 0-3 take the even rows, warps 4-7
    // the odd ones.  Within a warp consecutive lanes are then 27 words apart (odd), which makes
    // every per-lane shared-memory access of the row (14 stores) and of the moves (60-byte
    // stride at depth 30) bank-conflict free, and the row's alignment is warp-uniform.
    const int row = (SIZE == 3) ? 2 * (((tid >> 5) & 3) * 32 + (tid & 31)) + (tid >> 7) : tid;
    const long long base = (tile0 + blockIdx.x) * kTile;
    const int cnt = FULL ? kTile : (int)(n - base);       // bulk copies need 16-byte multiples: full tiles only
    constexpr bool full = FULL;
    const uint32_t move_bytes = (uint32_t)(kTile * depth);

    if (full && depth > 0 && tid == 0) {
        bulk::mbar_init(s_bar, 1);
        bulk::mbar_expect_tx(s_bar, move_bytes);
        bulk::load(s_moves, moves + base * depth, move_bytes, s_bar);
    }
    load_tables<SIZE>(smem, tid);
    if (!full) {                                          // ragged last tile: plain copies
        const long long byte0 = base * depth;
        const int nbytes = cnt * depth;
        for (int i = tid; i < nbytes; i += kTile) s_moves[i] = moves[byte0 + i];
    }
    __syncthreads();                                      // tables + barrier init visible to every thread
    if (full && depth > 0) bulk::mbar_wait(s_bar, 0);

    bool ok = false;
    if (row < cnt) {
        CubieState st;
        cubie_init(st);
        scramble_run_staged<SIZE>(st, row, depth, s_moves, s_tbl);
        if (last) {                                       // cube_scramble_step: one more face turn per instance
            st.c0 = cubie_fold_twist(st.c0); st.c1 = cubie_fold_twist(st.c1);
            cubie_move<SIZE>(st, s_tbl, (uint32_t)__ldg(last + base + row) & 0xfu);
        }
        ok = scramble_finish<SIZE>(st, row, s_clut, s_elut, s_out);
        s_flags[row] = ok ? 1 : 0;
    }
    const unsigned bal = __ballot_sync(0xffffffffu, ok);
    if ((tid & 31) == 0 && bal && counters) atomicAdd(&counters[0], (unsigned long long)__popc(bal));
    if (blockIdx.x == 0 && tid == 0 && counters) atomicAdd(&counters[1], (unsigned long long)(FULL ? (long long)gridDim.x * kTile : (long long)cnt));

    if (full) bulk::fence_smem_writes();                  // rows written above -> visible to the copy engine
    __syncthreads();
    if (full) {
        if (tid == 0) {
            bulk::store(out + base * G::S, s_out, (uint32_t)(kTile * G::S));
            bulk::commit();
        }
    } else {
        const long long byte0 = base * G::S;
        const int nbytes = cnt * G::S;
        for (int i = tid; i < nbytes; i += kTile) out[byte0 + i] = s_out[i];
    }
    if (tid < cnt) {                                      // verdicts leave in row order, coalesced
        const bool row_ok = s_flags[tid] != 0;
        if (solved) solved[base + tid] = row_ok ? 1 : 0;
        if (reward) reward[base + tid] = row_ok ? 1.0f : -1.0f;
    }
    if (full && tid == 0) bulk::wait_read_all();          // shared memory must outlive the copy's reads
}


// ---- K1p: persistent pair-table kernel (the default for depth 1..kMaxPairDepth) ----------------
// One CTA per SM; every WARP owns a private pipeline over tiles of 64 (or 128) instances and never
// synchronises with another warp after the prologue.  The tile's move bytes arrive by one bulk copy
// (double-buffered: tile i+1 is in flight while tile i is computed) -- a flat 1-D copy, or a 2-D tensor
// copy with the 128-byte swizzle for the depths whose flat image bank-conflicts (DEPTH < 0); each lane
// walks TWO (2x2x2, shallow: FOUR) instances in lockstep through the PAIR table (one conflict-free
// 2 x 128-bit row per two moves, see cube_threads.cuh) -- rows 2l and 2l+1 for 3x3x3, so that each
// finishing pass writes rows of one parity (54-byte rows alternate between word-aligned and two bytes
// off); the sticker rows are assembled in the warp's output tile and leave by one bulk store, the
// verdicts straight from the lanes' own flags.  The 43 KB table is loaded once per CTA.  Tiles of 64
// rows keep every bulk copy a multiple of 16 bytes for any depth.
constexpr int kMaxPairDepth = 320;       // four warps' double-buffered move tiles still fit
constexpr int kPairTableBytes = CUBE_PAIR_ROWS * 256;
// kNS instances per lane in lockstep = tiles of 32 * kNS rows.  2x2x2 (two state registers per instance)
// walks four: the per-tile work (claim, staging, barrier, stores, verdict words) is ~150 instructions per
// lane, a quarter of that kernel's instruction count with two.
// (Chosen for shallow sequences only: the 128-row tiles of a deep one leave room for too few warps.
// 3x3x3 with four instances per lane and 12 warps was measured: depth 30 -1.6 %, depth 20 +2 %, depth 10
// +4 % -- that kernel is bound by the shared-memory pipe, not by instruction issue; not instantiated.
// 2x2x2 with eight per lane (256-row tiles, 8 warps): depth 20 -10 %.)
template <int SIZE, int NS> struct PairCfg;
template <> struct PairCfg<3, 2> { static constexpr int kMaxWarps = 24; };    // 768 threads: 85 registers each
template <> struct PairCfg<2, 2> { static constexpr int kMaxWarps = 32; };
template <> struct PairCfg<2, 4> { static constexpr int kMaxWarps = 20; };    // 640 threads: 102 registers each
constexpr int kMinWarpsFour = 16;         // 2x2x2 walks four instances per lane when at least this many warps fit

template <int SIZE, int NS>
struct PairSmem {
    using G = CubeGeom<SIZE>;
    static constexpr int kPairTile = 32 * NS;
    static constexpr int kTable = 0;                                  // + up to 255 bytes: 256-byte aligned in the window
    static constexpr int kCornerLut = kPairTableBytes + 256;          // (relative to the aligned table start: + 0)
    static constexpr int kEdgeLut = kCornerLut + 256;                 // 3x3x3: one 32-entry LUT per edge slot (1 536 bytes)
    static constexpr int kPerWarp = (kEdgeLut + (SIZE == 3 ? 1536 : 256) + 1023) / 1024 * 1024;   // swizzled move tiles: 1 KB boundaries
    static constexpr int kOutBytes = kPairTile * G::S;                // 3456 / 3072: multiples of 16
    // flat tile image (+16: the last row's word loads run past it), or the swizzled tile (`swz`: the copy
    // engine's 128-byte swizzle wants 1024-byte aligned buffers)
    __host__ __device__ static constexpr int round1k(int x) { return (x + 1023) & ~1023; }
    __host__ __device__ static constexpr int move_stride(int depth, bool swz = false)
    {
        return swz ? round1k(kPairTile * depth) : kPairTile * depth + 16;
    }
    __host__ __device__ static constexpr int moves_at(bool swz = false) { return swz ? round1k(16 + kOutBytes) : 16 + kOutBytes; }
    __host__ __device__ static constexpr int per_warp(int depth, bool swz = false)
    {
        return moves_at(swz) + 2 * move_stride(depth, swz);
    }
    // never below 65 792 + 256 bytes: a garbage move byte (> 12) makes a garbage pair row (<= 255) whose
    // two vectors must still be inside the CTA's allocation (169 * 128 + 255 * 128 + 128 = 54 400 would do)
    __host__ __device__ static constexpr int bytes(int depth, int warps, bool priv = false)
    {
        return kPerWarp + warps * per_warp(depth, priv) < 66048 ? 66048 : kPerWarp + warps * per_warp(depth, priv);
    }
};

// MODE 1: the common call -- solved and reward arrays present, no trailing action -- with the per-tile null
// checks and the action fetch compiled out (~18 of a tile's ~1 080 instructions); MODE 2: the same with the
// trailing action of cube_scramble_step; MODE 0: any combination, decided at run time
template <int SIZE, int DEPTH, int NS, int MODE>
__global__ void __launch_bounds__(PairCfg<SIZE, NS>::kMaxWarps * 32, 1)
scramble_pairs_kernel(const uint8_t* __restrict__ moves, int n_tiles, int depth_rt, uint8_t* __restrict__ out,
                      uint8_t* __restrict__ solved, float* __restrict__ reward, unsigned long long* __restrict__ counters,
                      sched::Slot* slot, int tail_div, const __grid_constant__ CUtensorMap move_map,
                      const uint8_t* __restrict__ last)
{
    using L = PairSmem<SIZE, NS>;
    constexpr int kPairTile = L::kPairTile;
    extern __shared__ __align__(128) uint8_t smem_raw[];
    const int depth = DEPTH > 0 ? DEPTH : depth_rt;
    // DEPTH < 0: any depth that is a multiple of 8 (3x3x3) / 16 (2x2x2), staged as a swizzled tile through
    // `move_map` (see scramble_pairs_run_swizzled): the flat image bank-conflicts at those depths
    constexpr bool kPriv = DEPTH < 0;
    constexpr uint32_t kAlign = kPriv ? 1024u : 256u;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // everything is laid out from a 256-byte boundary of the shared window (table rows on 128-byte boundaries)
    const uint32_t window = bulk::smem_addr(smem_raw);
    uint8_t* smem = smem_raw + ((kAlign - (window & (kAlign - 1u))) & (kAlign - 1u));
    uint8_t* s_ptbl = smem + L::kTable;
    const PairTableShared tbl{bulk::smem_addr(s_ptbl)};
    uint32_t* s_clut = reinterpret_cast<uint32_t*>(smem + L::kCornerLut);
    uint32_t* s_elut = reinterpret_cast<uint32_t*>(smem + L::kEdgeLut);
    uint8_t* mine = smem + L::kPerWarp + warp * L::per_warp(depth, kPriv);
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(mine);             // [2] mbarriers
    uint8_t* s_out = mine + 16;                                       // [kOutBytes]
    uint8_t* s_moves = mine + L::moves_at(kPriv);                     // [2][move_stride]
    const int mstride = L::move_stride(depth, kPriv);
    const uint32_t move_bytes = (uint32_t)(kPairTile * depth);
    // stage tile `t`'s move bytes in buffer `b` (warp-uniform arguments): one 1-D bulk copy for the flat
    // image, one 2-D tensor copy (rows of 128 bytes, 128-byte swizzle) for the swizzled tile
    auto stage = [&](int t, int b) {
        if (bulk::elect_one()) {
            bulk::mbar_expect_tx(&s_bar[b], move_bytes);
            if (!kPriv) bulk::load(s_moves + b * mstride, moves + (long long)t * move_bytes, move_bytes, &s_bar[b]);
            else bulk::load_tile_2d(s_moves + b * mstride, &move_map, 0, t * (kPairTile * depth >> 7), &s_bar[b]);
        }
    };

    // Programmatic dependent launch: the NEXT kernel of the stream may start as soon as SM resources free
    // up; its prologue below touches only constant tables and shared memory, and it waits for this grid
    // to complete (griddepcontrol.wait) before its first global access.
    asm volatile("griddepcontrol.launch_dependents;");
    pair_table_fill<SIZE>(s_ptbl, tid, blockDim.x);
    if (tid < 32) s_clut[tid] = (SIZE == 3) ? kCornerColour3[tid] : kCornerColour2[tid];
    if (SIZE == 3) for (int i = tid; i < 12 * 32; i += blockDim.x) s_elut[i] = kEdgeColourSlot3[i];   // canonical flips: 32 entries per slot
    if (lane == 0) { bulk::mbar_init(&s_bar[0], 1); bulk::mbar_init(&s_bar[1], 1); }
    // the warp's first two tiles (its static share starts at its global warp index) are hinted into L2 while the
    // previous grid of the stream drains: after the wait 3 552 warps fetch their first tile at once, and a tile
    // of moves that comes from L2 is there in half the time (a hint only: the bytes are READ after the wait).
    // Measured with per-warp %globaltimer stamps (tools/k1p_timeline.py): wait over -> first tile landed
    // 2.4 -> 1.1-1.7 us; with the scheduler's one-round-trip exhaustion check +0.9 % at 8 Mi x depth 30.
    // (One tile per claim instead of two in the dynamic tail: the same +0.9 % without the hint, +0.6 % with it.)
    if (lane == 0 && depth > 0) {
        const int total = (int)gridDim.x * (int)(blockDim.x >> 5);
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int t = (int)blockIdx.x * (int)(blockDim.x >> 5) + warp + k * total;
            if (t < n_tiles) bulk::prefetch_l2(moves + (long long)t * move_bytes, move_bytes);
        }
    }
    __syncthreads();
    asm volatile("griddepcontrol.wait;" ::: "memory");                // everything earlier in the stream is complete

    // tiles are claimed dynamically (cube_sched.cuh): `tile` is being computed, `next` is in flight
    sched::WarpTiles tiles;
    tiles.init(slot, n_tiles, (int)(blockDim.x >> 5), warp, lane, tail_div);
    int tile = tiles.pop(lane);
    if (tile < n_tiles) stage(tile, 0);
    int rows[NS];
#pragma unroll
    for (int k = 0; k < NS; ++k) rows[k] = (SIZE == 3) ? 64 * (k >> 1) + 2 * lane + (k & 1) : lane + 32 * k;
    const uint32_t lanereg = pair_lanereg<SIZE>(lane, tbl), roff = pair_roff2(lane);
    const ColourLutShared lut{bulk::smem_addr(s_clut), bulk::smem_addr(s_elut)};
    unsigned n_solved = 0;
    const bool has_last = MODE == 2 || (MODE == 0 && last != nullptr);
    const bool has_solved = MODE != 0 || solved != nullptr, has_reward = MODE != 0 || reward != nullptr;
    for (int it = 0; tile < n_tiles; ++it) {
        const int buf = it & 1;
        const int next = tiles.pop(lane);
        if (next < n_tiles) stage(next, buf ^ 1);                     // prefetch the next tile's moves
        // cube_scramble_step: the trailing action of every instance (rows 2l, 2l+1 are neighbours: one 16-bit load;
        // 2x2x2 rows l + 32k: 32 consecutive bytes per load), fetched before the walk so its latency is hidden
        uint32_t last_w[NS];
        if (has_last) {
            if (SIZE == 3) {
#pragma unroll
                for (int h = 0; h < NS; h += 2) {
                    const uint32_t v = *reinterpret_cast<const uint16_t*>(last + (long long)tile * kPairTile + 32 * h + 2 * lane);
                    last_w[h] = v & 0xffu; last_w[h + 1] = v >> 8;
                }
            } else {
#pragma unroll
                for (int k = 0; k < NS; ++k) last_w[k] = last[(long long)tile * kPairTile + 32 * k + lane];
            }
        }
        bulk::mbar_wait(&s_bar[buf], (uint32_t)(it >> 1) & 1u);

        CubieState st[NS];
#pragma unroll
        for (int k = 0; k < NS; ++k) cubie_init(st[k]);
        if constexpr (kPriv) scramble_pairs_run_swizzled<SIZE, NS>(st, s_moves + buf * mstride, lane, depth, tbl, lanereg, roff);
        else scramble_pairs_run<SIZE, (DEPTH > 0 ? DEPTH : 0), NS>(st, rows, depth, s_moves + buf * mstride, tbl, lanereg, roff);
        if (has_last) {                                               // cube_scramble_step: one more face turn
#pragma unroll
            for (int k = 0; k < NS; ++k) scramble_pairs_last<SIZE>(st[k], last_w[k], tbl, lanereg, roff);
        }
        if (bulk::elect_one()) bulk::wait_read_all();                 // the previous store has released the out tile (elect.sync picks the same lane every time)
        __syncwarp();
        bool ok[NS];
#pragma unroll
        for (int k = 0; k < NS; ++k) {
            ok[k] = scramble_pairs_finish<SIZE>(st[k], rows[k], lut, s_out);
            n_solved += ok[k] ? 1u : 0u;                              // per lane; summed over the warp after the last tile
        }

        bulk::fence_smem_writes();                                    // rows -> visible to the copy engine
        __syncwarp();
        if (bulk::elect_one()) {
            bulk::store(out + (long long)tile * L::kOutBytes, s_out, (uint32_t)L::kOutBytes);
            bulk::commit();
        }
        // verdicts leave coalesced, straight from the lane's own flags: one solved byte and one reward per row
        if (SIZE == 3) {                                              // rows 2l, 2l+1 of every 64 are neighbours
#pragma unroll
            for (int h = 0; h < NS; h += 2) {
                const long long r0 = (long long)tile * kPairTile + 32 * h + 2 * lane;
                if (has_solved) *reinterpret_cast<uint16_t*>(solved + r0) = (uint16_t)((ok[h] ? 1u : 0u) | (ok[h + 1] ? 0x100u : 0u));
                if (has_reward) *reinterpret_cast<float2*>(reward + r0) = make_float2(ok[h] ? 1.0f : -1.0f, ok[h + 1] ? 1.0f : -1.0f);
            }
        } else {                                                      // rows l + 32k: 32 in a row per store
#pragma unroll
            for (int k = 0; k < NS; ++k) {
                if (has_solved) solved[(long long)tile * kPairTile + 32 * k + lane] = ok[k] ? 1 : 0;
                if (has_reward) reward[(long long)tile * kPairTile + 32 * k + lane] = ok[k] ? 1.0f : -1.0f;
            }
        }
        tile = next;
    }
    n_solved = __reduce_add_sync(0xffffffffu, n_solved);
    if (lane == 0 && n_solved && counters) atomicAdd(&counters[0], (unsigned long long)n_solved);
    if (blockIdx.x == 0 && tid == 0 && counters) atomicAdd(&counters[1], (unsigned long long)n_tiles * kPairTile);
    __syncwarp();
    if (bulk::elect_one()) bulk::wait_read_all();                     // shared memory must outlive the copies' reads
    __syncthreads();
    sched::release(slot);
}

// ---- K1p, sliced: sequences deeper than kMaxPairDepth (test.py scrambles 1 000 deep, test.py:44) -------------
// A tile's move bytes no longer fit in a warp's buffers, so they arrive in SLICES of kSlice moves per row while
// the cubie state stays in registers from slice to slice.  A slice of a tile is 64 pieces of the row-major move
// array, `depth` bytes apart and at any byte alignment: every lane fetches the pieces of its two rows (lane and
// lane + 32) with two small bulk copies from the 16-byte boundary below each piece (the piece then starts
// (row * depth) & 15 bytes into its slot: the same shift in every slice, because kSlice is a multiple of 16; the
// slice runner takes it out in registers) and announces their bytes on the buffer's mbarrier (32 arrivals).
// Slots are 17 x 16 bytes apart, so the 128-bit move loads of a quarter warp fall into eight different bank
// groups.  Double-buffered across slices AND tiles.
// (Tried on the way: 32-bit move loads at the per-row shift -- slots can only be 16-byte aligned, so they conflict
// 8-fold: 0.96e12 tr/s at depth 1000; byte-coordinate copies through a 1-D tensor map, which would land every
// piece aligned -- tensor copies want 128-byte aligned destinations, which brings the conflicts back.)
// Slice length: moves per row and slice, a multiple of 16; a row's slot is slice + 32 bytes (shift <= 15, the
// runner reads one unit ahead) and must be an ODD number of 16-byte units.  112 moves (144-byte slots) let 8
// warps' double buffers fit; 240 (272-byte slots: 4 warps, one per scheduler) issued at 0.42 of a scheduler's
// rate, single-warp latency-bound: 0.98e12 tr/s at depth 1000 (CUBE_SLICE=240 for A/B runs).
constexpr int kSliceDefault = 112;
__host__ __device__ constexpr int slice_stride(int slice) { return ((slice + 32) / 16) % 2 ? slice + 32 : slice + 48; }

template <int SIZE>
struct SlicedSmem {
    using G = CubeGeom<SIZE>;
    static constexpr int kOutBytes = 64 * G::S;
    static constexpr int kMovesAt = 16 + kOutBytes;                   // after the two mbarriers and the out tile
    __host__ __device__ static constexpr int per_warp(int slice) { return kMovesAt + 2 * 64 * slice_stride(slice); }
    static constexpr int kFixed = PairSmem<SIZE, 2>::kPerWarp;        // pair table + colour LUTs, as in K1p
    __host__ __device__ static constexpr int bytes(int warps, int slice) { return kFixed + warps * per_warp(slice); }
};

template <int SIZE>
__global__ void __launch_bounds__(8 * 32, 1)
scramble_sliced_kernel(const uint8_t* __restrict__ moves, int n_tiles, int depth, uint8_t* __restrict__ out,
                       uint8_t* __restrict__ solved, float* __restrict__ reward, unsigned long long* __restrict__ counters,
                       const uint8_t* __restrict__ last, int kSlice)
{
    using L = SlicedSmem<SIZE>;
    using P = PairSmem<SIZE, 2>;
    extern __shared__ __align__(128) uint8_t smem_raw[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, warps = (int)(blockDim.x >> 5);
    const uint32_t window = bulk::smem_addr(smem_raw);
    uint8_t* smem = smem_raw + ((256u - (window & 255u)) & 255u);     // the pair table on a 256-byte boundary
    uint8_t* s_ptbl = smem + P::kTable;
    const PairTableShared tbl{bulk::smem_addr(s_ptbl)};
    uint32_t* s_clut = reinterpret_cast<uint32_t*>(smem + P::kCornerLut);
    uint32_t* s_elut = reinterpret_cast<uint32_t*>(smem + P::kEdgeLut);
    const int kSliceStride = slice_stride(kSlice);
    uint8_t* mine = smem + L::kFixed + warp * L::per_warp(kSlice);
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(mine);              // [2]: 32 arrivals each
    uint8_t* s_out = mine + 16;
    uint8_t* s_moves = mine + L::kMovesAt;                            // [2][64][kSliceStride]

    pair_table_fill<SIZE>(s_ptbl, tid, blockDim.x);
    if (tid < 32) s_clut[tid] = (SIZE == 3) ? kCornerColour3[tid] : kCornerColour2[tid];
    if (SIZE == 3) for (int i = tid; i < 12 * 32; i += blockDim.x) s_elut[i] = kEdgeColourSlot3[i];
    if (lane == 0) { bulk::mbar_init(&s_bar[0], 32); bulk::mbar_init(&s_bar[1], 32); }
    __syncthreads();

    const int n_slices = (depth + kSlice - 1) / kSlice;
    const int rows[2] = {lane, lane + 32};
    const uint32_t shift[2] = {(uint32_t)(((long long)rows[0] * depth) & 15), (uint32_t)(((long long)rows[1] * depth) & 15)};
    // the lane's two pieces of slice `s` of tile `t` into buffer `b`: from the 16-byte boundary below the piece to
    // the one above its end (never past the move array: the last whole tile is left to the caller)
    auto stage = [&](int t, int s, int b) {
        const int len = depth - s * kSlice < kSlice ? depth - s * kSlice : kSlice;
        uint32_t bytes[2];
#pragma unroll
        for (int k = 0; k < 2; ++k) bytes[k] = (shift[k] + (uint32_t)len + 15u) & ~15u;
        bulk::mbar_expect_tx(&s_bar[b], bytes[0] + bytes[1]);
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const long long g = ((long long)t * 64 + rows[k]) * depth + (long long)s * kSlice;
            bulk::load(s_moves + (b * 64 + rows[k]) * kSliceStride, moves + (g & ~15LL), bytes[k], &s_bar[b]);
        }
    };
    const uint32_t lanereg = pair_lanereg<SIZE>(lane, tbl), roff = pair_roff2(lane);
    const ColourLutShared lut{bulk::smem_addr(s_clut), bulk::smem_addr(s_elut)};
    unsigned n_solved = 0;
    const int stride = (int)gridDim.x * warps;
    int tile = (int)blockIdx.x * warps + warp;
    if (tile < n_tiles) stage(tile, 0, 0);
    for (unsigned it = 0; tile < n_tiles; tile += stride) {
        CubieState st[2];
        cubie_init(st[0]);
        cubie_init(st[1]);
        for (int s = 0; s < n_slices; ++s, ++it) {
            const int buf = (int)(it & 1u);
            __syncwarp();                                             // every lane is done with the other buffer
            if (s + 1 < n_slices) stage(tile, s + 1, buf ^ 1);
            else if (tile + stride < n_tiles) stage(tile + stride, 0, buf ^ 1);
            bulk::mbar_wait(&s_bar[buf], (it >> 1) & 1u);
            const int len = depth - s * kSlice < kSlice ? depth - s * kSlice : kSlice;
            const uint32_t base[2] = {(uint32_t)((buf * 64 + rows[0]) * kSliceStride), (uint32_t)((buf * 64 + rows[1]) * kSliceStride)};
            scramble_pairs_run_units<SIZE, 2>(st, base, shift, len, s_moves, tbl, lanereg, roff);
        }
        if (last) {
#pragma unroll
            for (int k = 0; k < 2; ++k)
                scramble_pairs_last<SIZE>(st[k], (uint32_t)__ldg(last + (long long)tile * 64 + rows[k]), tbl, lanereg, roff);
        }
        if (lane == 0) bulk::wait_read_all();                         // the previous store has released the out tile
        __syncwarp();
        bool ok[2];
#pragma unroll
        for (int k = 0; k < 2; ++k) {                                 // rows lane, lane + 32: both parities in a pass (3x3x3:
            ok[k] = scramble_pairs_finish<SIZE>(st[k], rows[k], lut, s_out);   // two half-masked store sequences, noise here)
            n_solved += ok[k] ? 1u : 0u;
        }
        bulk::fence_smem_writes();
        __syncwarp();
        if (lane == 0) {
            bulk::store(out + (long long)tile * L::kOutBytes, s_out, (uint32_t)L::kOutBytes);
            bulk::commit();
        }
#pragma unroll
        for (int k = 0; k < 2; ++k) {                                 // 32 consecutive bytes / floats per store
            if (solved) solved[(long long)tile * 64 + rows[k]] = ok[k] ? 1 : 0;
            if (reward) reward[(long long)tile * 64 + rows[k]] = ok[k] ? 1.0f : -1.0f;
        }
    }
    n_solved = __reduce_add_sync(0xffffffffu, n_solved);
    if (lane == 0 && n_solved && counters) atomicAdd(&counters[0], (unsigned long long)n_solved);
    if (blockIdx.x == 0 && tid == 0 && counters) atomicAdd(&counters[1], (unsigned long long)n_tiles * 64);
    if (lane == 0) bulk::wait_read_all();
}

// Whole tiles of a deep batch through the sliced kernel; the LAST whole tile is left to the caller (a piece's
// copy may run up to 15 bytes past its row: never past the move array when a tile follows).  Returns the number
// of instances handled (0: not applicable) or -cudaError.
template <int SIZE>
long long launch_sliced(const uint8_t* moves, long long n, int depth, uint8_t* out, uint8_t* solved, float* reward,
                        unsigned long long* counters, cudaStream_t stream, const uint8_t* last)
{
    using L = SlicedSmem<SIZE>;
    long long n_tiles = n / 64 - 1;
    if (n_tiles < 1) return 0;
    if (n_tiles > 0x3fffffff) n_tiles = 0x3fffffff;
    static const int slice = [] {
        const int v = cube::env_int("CUBE_SLICE", kSliceDefault);
        return (v >= 16 && v <= 240 && v % 16 == 0) ? v : kSliceDefault;
    }();
    int warps = cube::warps_that_fit(256 + L::kFixed, L::per_warp(slice), 8);
    if (warps >= 4) warps &= ~3;                                      // the same number on every scheduler
    if (warps < 1) return 0;
    const int smem = L::bytes(warps, slice) + 256 < 66048 + 256 ? 66048 + 256 : L::bytes(warps, slice) + 256;
    auto kern = scramble_sliced_kernel<SIZE>;
    cudaError_t e = cube::raise_smem_limit(kern, smem);
    if (e != cudaSuccess) return -(long long)e;
    kern<<<cube::persistent_grid(n_tiles, warps), warps * 32, smem, stream>>>(moves, (int)n_tiles, depth, out, solved, reward,
                                                                            counters, last, slice);
    e = cudaGetLastError();
    if (e != cudaSuccess) return -(long long)e;
    return n_tiles * 64;
}

// deep sequences (depth > kMaxStagedDepth): persistent CTAs, moves read straight from global
template <int SIZE>
__global__ void __launch_bounds__(kTile, 4)
scramble_deep_kernel(const uint8_t* __restrict__ moves, long long n, int depth, uint8_t* __restrict__ out,
                     uint8_t* __restrict__ solved, float* __restrict__ reward,
                     unsigned long long* __restrict__ counters, const uint8_t* __restrict__ last)
{
    using G = CubeGeom<SIZE>;
    using L = ScrambleSmem<SIZE>;
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t* s_tbl = reinterpret_cast<const uint32_t*>(smem + L::kTable);
    const uint32_t* s_clut = reinterpret_cast<const uint32_t*>(smem + L::kCornerLut);
    const uint32_t* s_elut = reinterpret_cast<const uint32_t*>(smem + L::kEdgeLut);
    uint8_t* s_out = smem + L::kOut;
    const int tid = threadIdx.x;
    load_tables<SIZE>(smem, tid);

    const long long n_tiles = (n + kTile - 1) / kTile;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long base = tile * kTile;
        const int cnt = (int)((n - base) < (long long)kTile ? (n - base) : (long long)kTile);
        __syncthreads();            // tables visible; previous tile's copy-out finished
        bool ok = false;
        if (tid < cnt) {
            CubieState st;
            cubie_init(st);
            const uint8_t* row = moves + (base + tid) * depth;
            for (int k = 0; k < depth; ++k) {
                cubie_move<SIZE>(st, s_tbl, (uint32_t)__ldg(row + k) & 0xfu);
                if ((k & 3) == 3) { st.c0 = cubie_fold_twist(st.c0); st.c1 = cubie_fold_twist(st.c1); }
            }
            if (last) {
                st.c0 = cubie_fold_twist(st.c0); st.c1 = cubie_fold_twist(st.c1);
                cubie_move<SIZE>(st, s_tbl, (uint32_t)__ldg(last + base + tid) & 0xfu);
            }
            ok = scramble_finish<SIZE>(st, tid, s_clut, s_elut, s_out);
            if (solved) solved[base + tid] = ok ? 1 : 0;
            if (reward) reward[base + tid] = ok ? 1.0f : -1.0f;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, ok);
        if ((tid & 31) == 0 && bal && counters) atomicAdd(&counters[0], (unsigned long long)__popc(bal));
        __syncthreads();
        const long long byte0 = base * G::S;               // multiple of 16
        const int nbytes = cnt * G::S;
        const int nvec = nbytes >> 4;
        int4* dst = reinterpret_cast<int4*>(out + byte0);
        for (int i = tid; i < nvec; i += kTile) __stcs(dst + i, reinterpret_cast<const int4*>(s_out)[i]);
        for (int i = (nvec << 4) + tid; i < nbytes; i += kTile) out[byte0 + i] = s_out[i];
    }
    if (blockIdx.x == 0 && tid == 0 && counters) atomicAdd(&counters[1], (unsigned long long)n);
}

template <int SIZE>
int launch_classic(const uint8_t* moves, long long n, int depth, uint8_t* out, uint8_t* solved, float* reward,
                   unsigned long long* counters, cudaStream_t stream, const uint8_t* last)
{
    const bool staged = depth <= kMaxStagedDepth;
    const int smem = ScrambleSmem<SIZE>::bytes(depth, staged);
    const long long n_tiles = (n + kTile - 1) / kTile;
    if (staged) {
        auto kern_full = scramble_tile_kernel<SIZE, true>;
        auto kern_tail = scramble_tile_kernel<SIZE, false>;
        cudaError_t e = cube::raise_smem_limit(kern_full, smem);
        if (e == cudaSuccess) e = cube::raise_smem_limit(kern_tail, smem);
        if (e != cudaSuccess) return (int)e;
        cube::prefer_max_shared(kern_full);
        const long long full_tiles = n / kTile;
        if (full_tiles > 0)
            kern_full<<<(unsigned)full_tiles, kTile, smem, stream>>>(moves, n, 0, depth, out, solved, reward, counters, last);
        if (full_tiles < n_tiles)
            kern_tail<<<1, kTile, smem, stream>>>(moves, n, full_tiles, depth, out, solved, reward, counters, last);
    } else {
        auto kern = scramble_deep_kernel<SIZE>;
        int per_sm = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kTile, smem) != cudaSuccess || per_sm < 1)
            per_sm = 1;
        long long grid = (long long)cube::sm_count() * per_sm;
        if (grid > n_tiles) grid = n_tiles;
        kern<<<(unsigned)grid, kTile, smem, stream>>>(moves, n, depth, out, solved, reward, counters, last);
    }
    return (int)cudaGetLastError();
}

// Tensor map of a move array for the swizzled tiles of K1p: the bytes as rows of 128, a box = one tile of
// 64 / 128 move rows (`tile_rows` = tile * depth / 128 rows of 128 bytes), 128-byte swizzle on the shared-memory side.  The encoder is a
// driver entry point, fetched through the runtime so that the library does not link libcuda.
using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

bool encode_move_map(CUtensorMap* map, const uint8_t* moves, long long n_tiles, int tile_rows)
{
    static const EncodeTiledFn encode = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            p = nullptr;
        (void)cudaGetLastError();
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    if (!encode) return false;
    const cuuint64_t dims[2] = {128, (cuuint64_t)(n_tiles * tile_rows)};
    const cuuint64_t strides[1] = {128};
    const cuuint32_t box[2] = {128, (cuuint32_t)tile_rows};
    const cuuint32_t elem[2] = {1, 1};
    return encode(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<uint8_t*>(moves), dims, strides, box, elem,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// K1p on the whole tiles of a batch with NS instances per lane.  Returns the number of instances handled
// (a multiple of 32 * NS; 0 = not applicable: fewer than `min_warps` warps fit, too few rows), or -cudaError.
template <int SIZE, int NS>
long long launch_pairs(const uint8_t* moves, long long n, int depth, uint8_t* out, uint8_t* solved, float* reward,
                       unsigned long long* counters, cudaStream_t stream, int min_warps, const uint8_t* last)
{
    using L = PairSmem<SIZE, NS>;
    constexpr int kPairTile = L::kPairTile;
    if (n < kPairTile) return 0;
    // depths whose flat row stride bank-conflicts on the move words are staged as swizzled tiles
    static const bool swz_ok = cube::env_flag("CUBE_PAIR_SWIZZLE", true);
    static_assert(L::kPerWarp % 1024 == 0, "the per-warp areas of the swizzled variant start on 1 KB");
    long long n_tiles = n / kPairTile;
    if (n_tiles > 0x3fffffff) n_tiles = 0x3fffffff;                   // 32-bit tile counters; the caller handles the rest
    const int tile_rows = kPairTile * depth / 128;                    // of the tensor map, when swizzled
    constexpr bool kCanSwizzle = SIZE == 2 || NS == 2;                // 3x3x3 with four instances per lane: flat only
    bool priv = kCanSwizzle && swz_ok && depth % (SIZE == 3 ? 8 : 16) == 0 && n_tiles * tile_rows < 0x7fffffffLL;
    auto warps_for = [&](bool p) {                                    // the same number on every scheduler
        return cube::warps_that_fit((p ? 1024 : 256) + L::kPerWarp, L::per_warp(depth, p), PairCfg<SIZE, NS>::kMaxWarps) & ~3;
    };
    if (warps_for(priv) < min_warps) return 0;
    alignas(64) CUtensorMap move_map;
    memset(&move_map, 0, sizeof(move_map));
    if (priv && !encode_move_map(&move_map, moves, n_tiles, tile_rows)) priv = false;
    const int slack = priv ? 1024 : 256;                              // alignment of the carve-up in the window
    const int warps = warps_for(priv);
    if (warps < min_warps) return 0;
    const int smem = L::bytes(depth, warps, priv) + slack;
    // straight-line specialisations: the reference's default depth (config.yaml:7) and BASELINE config 2's
    // (2x2x2 with four instances per lane is 7 % SLOWER with the action fetch unconditional -- 0.151 against 0.141 ms
    // for 16 Mi x 20 -- so its trailing-action calls keep the run-time checks)
    constexpr int kM2 = SIZE == 3 ? 2 : 0;
    const int mode = (solved && reward) ? (last ? kM2 : 1) : 0;
    const int variant = depth == 30 ? 1 : depth == 20 ? 2 : priv ? 3 : 0;
    using Kern = decltype(&scramble_pairs_kernel<SIZE, 0, NS, 0>);
    constexpr int kSwz = kCanSwizzle ? -1 : 0;
    static const Kern kerns[3][4] = {
        {scramble_pairs_kernel<SIZE, 0, NS, 0>, scramble_pairs_kernel<SIZE, 30, NS, 0>, scramble_pairs_kernel<SIZE, 20, NS, 0>, scramble_pairs_kernel<SIZE, kSwz, NS, 0>},
        {scramble_pairs_kernel<SIZE, 0, NS, 1>, scramble_pairs_kernel<SIZE, 30, NS, 1>, scramble_pairs_kernel<SIZE, 20, NS, 1>, scramble_pairs_kernel<SIZE, kSwz, NS, 1>},
        {scramble_pairs_kernel<SIZE, 0, NS, kM2>, scramble_pairs_kernel<SIZE, 30, NS, kM2>, scramble_pairs_kernel<SIZE, 20, NS, kM2>, scramble_pairs_kernel<SIZE, kSwz, NS, kM2>}};
    const Kern kern = kerns[mode][variant];
    cudaError_t e = cube::raise_smem_limit(kern, smem);
    if (e != cudaSuccess) return -(long long)e;
    sched::Slot* slot = sched::claim_slot();
    if (!slot) return -(long long)cudaErrorUnknown;
    e = cube::launch_pdl(kern, cube::persistent_grid(n_tiles, warps), warps * 32, smem, stream, moves, (int)n_tiles, depth,
                         out, solved, reward, counters, slot, sched::tail_div(), move_map, last);
    if (e != cudaSuccess) return -(long long)e;
    return n_tiles * kPairTile;
}

template <int SIZE>
int launch_one(const uint8_t* moves, long long n, int depth, uint8_t* out, uint8_t* solved, float* reward,
               unsigned long long* counters, cudaStream_t stream, const uint8_t* last)
{
    using G = CubeGeom<SIZE>;
    long long done = 0;
    static const bool classic = cube::env_flag("CUBE_SCRAMBLE_CLASSIC", false);     // A/B switches for profiling
    static const bool four_ok = cube::env_flag("CUBE_PAIR_FOUR", true);
    static const bool sliced_ok = cube::env_flag("CUBE_PAIR_SLICED", true);
    // K1p writes the verdicts of rows 2l, 2l+1 as one 16-bit / float2 word: a sliced solved / reward buffer
    // that is not aligned like that takes the byte-wise tile kernel
    const bool aligned = ((reinterpret_cast<uintptr_t>(solved) & 1u) | (reinterpret_cast<uintptr_t>(reward) & 7u) |
                          (reinterpret_cast<uintptr_t>(last) & 1u)) == 0;
    if (depth >= 1 && depth <= kMaxPairDepth && aligned && !classic) {
        if (SIZE == 2 && four_ok)
            done = launch_pairs<2, 4>(moves, n, depth, out, solved, reward, counters, stream, kMinWarpsFour, last);
        if (done == 0) done = launch_pairs<SIZE, 2>(moves, n, depth, out, solved, reward, counters, stream, 4, last);
        if (done < 0) return (int)-done;
    }
    if (depth > kMaxPairDepth && aligned && sliced_ok && !classic) {
        done = launch_sliced<SIZE>(moves, n, depth, out, solved, reward, counters, stream, last);
        if (done < 0) return (int)-done;
    }
    if (done == n) return 0;
    return launch_classic<SIZE>(moves + done * depth, n - done, depth, out + done * G::S, solved ? solved + done : nullptr,
                                reward ? reward + done : nullptr, counters, stream, last ? last + done : nullptr);
}

}  // namespace

namespace cube {

int launch_scramble(int size, const uint8_t* moves, long long n, int depth, uint8_t* states_out,
                    uint8_t* solved, float* reward, unsigned long long* counters, cudaStream_t stream, const uint8_t* last)
{
    if (n == 0) return 0;
    if (size == 3) return launch_one<3>(moves, n, depth, states_out, solved, reward, counters, stream, last);
    return launch_one<2>(moves, n, depth, states_out, solved, reward, counters, stream, last);
}

}  // namespace cube
