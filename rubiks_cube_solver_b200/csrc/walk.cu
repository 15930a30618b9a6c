// K2 -- moves applied to resident sticker rows (sm_100a): the reference's
// CubeEnv.step (cube_env.py:71-111) for a batch, for ANY byte content of the
// rows: new[i] = old[moveDefs[a][i]] (py333.py:220-222; py222 doMove), then
// face uniformity (py333.py:229-233) and the +-1 reward (cube_env.py:89-104).
//
// One CTA turns one tile of 256 rows.  The tile comes in through one 1-D bulk
// asynchronous copy (TMA) and leaves through one bulk store; in between each
// thread turns its own row in place in shared memory -- a face turn is five
// (3x3x3) or three (2x2x2) sticker 4-cycles whose byte offsets come from a
// [cycle][move] table, so there is no branch on the move.  3x3x3 rows are 13.5
// words, so even rows go to warps 0-3 and odd rows to warps 4-7: lanes of a warp
// are then 27 words apart and row-relative accesses spread over all 32 banks.
// depth = 1 is `step`; depth > 1 walks several moves without leaving shared
// memory; depth = 0 with no output is `cube_solved`.
// HBM traffic per instance: 2*S + depth + 1 + 4 bytes.
#include <cuda_runtime.h>
#include "cube_bulk.cuh"
#include "cube_kernels.h"
#include "cube_launch.cuh"
#include "cube_sched.cuh"
#include "cube_threads.cuh"

namespace {

constexpr int kTile = 256;

__host__ __device__ constexpr int round16(int x) { return (x + 15) & ~15; }

// FULL: all tiles of the launch have 256 rows (bulk copies); !FULL: the ragged last tile.
template <int SIZE, bool FULL>
__global__ void __launch_bounds__(kTile, 6)
walk_tile_kernel(const uint8_t* in, const uint8_t* __restrict__ moves, long long n, long long tile0, int depth,
                 uint8_t* out, uint8_t* __restrict__ solved, float* __restrict__ reward,
                 unsigned long long* __restrict__ counters)
{
    using G = CubeGeom<SIZE>;
    __shared__ __align__(128) uint8_t s_rows[round16(kTile * G::S)];
    __shared__ uint32_t s_cyc[G::NCYC * CUBE_MOVE_ROWS];
    __shared__ uint8_t s_flags[kTile];
    __shared__ __align__(8) uint64_t s_bar;

    const int tid = threadIdx.x;
    const int row = (SIZE == 3) ? 2 * (((tid >> 5) & 3) * 32 + (tid & 31)) + (tid >> 7) : tid;
    const long long base = (tile0 + blockIdx.x) * kTile;
    const int cnt = FULL ? kTile : (int)(n - base);
    constexpr uint32_t kTileBytes = kTile * G::S;

    if (FULL && tid == 0) {
        bulk::mbar_init(&s_bar, 1);
        bulk::mbar_expect_tx(&s_bar, kTileBytes);
        bulk::load(s_rows, in + base * G::S, kTileBytes, &s_bar);
    }
    if (tid < G::NCYC * CUBE_MOVE_ROWS) s_cyc[tid] = (SIZE == 3) ? kCycles3[tid] : kCycles2[tid];
    if (!FULL) {
        const long long byte0 = base * G::S;
        for (int i = tid; i < cnt * G::S; i += kTile) s_rows[i] = in[byte0 + i];
    }
    // the moves of this thread's row, fetched while the tile is in flight (depth 1: one byte)
    uint32_t first_move = CUBE_NOOP_MOVE;
    const uint8_t* mrow = moves + (base + row) * depth;
    if (row < cnt && depth > 0) first_move = (uint32_t)__ldcs(mrow) & 0xfu;
    __syncthreads();
    if (FULL) bulk::mbar_wait(&s_bar, 0);

    bool ok = false;
    if (row < cnt) {
        uint8_t* r = s_rows + G::S * row;
        if (depth > 0) walk_turn<SIZE>(r, first_move, s_cyc);
        for (int k = 1; k < depth; ++k) walk_turn<SIZE>(r, (uint32_t)__ldcs(mrow + k) & 0xfu, s_cyc);
        ok = row_solved<SIZE>(r);
        s_flags[row] = ok ? 1 : 0;
    }
    const unsigned bal = __ballot_sync(0xffffffffu, ok);
    if ((tid & 31) == 0 && bal && counters) atomicAdd(&counters[0], (unsigned long long)__popc(bal));
    if (blockIdx.x == 0 && tid == 0 && counters)
        atomicAdd(&counters[1], (unsigned long long)(FULL ? (long long)gridDim.x * kTile : (long long)cnt));

    if (FULL && out) bulk::fence_smem_writes();
    __syncthreads();
    if (out) {
        if (FULL) {
            if (tid == 0) {
                bulk::store(out + base * G::S, s_rows, kTileBytes);
                bulk::commit();
            }
        } else {
            const long long byte0 = base * G::S;
            for (int i = tid; i < cnt * G::S; i += kTile) out[byte0 + i] = s_rows[i];
        }
    }
    if (tid < cnt) {
        const bool row_ok = s_flags[tid] != 0;
        if (solved) solved[base + tid] = row_ok ? 1 : 0;
        if (reward) reward[base + tid] = row_ok ? 1.0f : -1.0f;
    }
    if (FULL && out && tid == 0) bulk::wait_read_all();
}


// ---- K2p: persistent lane-private kernel (depth >= 1 with an output, the step / walk hot path) ----
// One CTA per SM, every warp owns a private pipeline over tiles of 64 rows (the same shape as the
// scramble kernel K1p): rows + move bytes of tile i+1 arrive by bulk copies while tile i is turned;
// per pass (even rows, then odd rows: 54-byte rows alternate between word-aligned and two bytes
// off, and a pass must have one alignment) each lane lifts its row out of the packed tile into
// registers (stride 27 words: conflict-free), parks it in the lane-private scratch layout
// (cube_threads.cuh), applies the 4-cycles there (one wavefront per byte access, whatever the
// moves), judges face uniformity in registers and writes the row back in place; the tile then
// leaves by one bulk store.  Replaces byte gathers on the packed tile, which bank-conflicted ~3x.
constexpr int kRowsPerTile = 64;
constexpr int kMaxWalkWarps = 24;         // measured: 32 warps on the 2x2x2 step (58 registers) are 2 % slower, the kernel sits at the HBM limit
constexpr int kMaxPrivateDepth = 64;

template <int SIZE>
struct WalkSmem {
    using G = CubeGeom<SIZE>;
    static constexpr int kEntries = 0;                                // [2 shifts][NCYC][16][2] words
    static constexpr int kPerWarp = 2 * G::NCYC * CUBE_MOVE_ROWS * 8;
    static constexpr int kTileBytes = kRowsPerTile * G::S;            // 3456 / 1536
    static constexpr int kScratch = 32 * WalkImage<SIZE>::W * 4;
    __host__ __device__ static constexpr int move_stride(int depth) { return kRowsPerTile * depth + 16; }
    __host__ __device__ static constexpr int per_warp(int depth)
    {
        return 16 + 2 * (kTileBytes + 16) + kScratch + 2 * move_stride(depth);
    }
    __host__ __device__ static constexpr int bytes(int depth, int warps) { return kPerWarp + warps * per_warp(depth); }
};

template <int SIZE>
__global__ void __launch_bounds__(kMaxWalkWarps * 32, 1)
walk_private_kernel(const uint8_t* in, const uint8_t* __restrict__ moves, int n_tiles, int depth, uint8_t* out,
                    uint8_t* __restrict__ solved, float* __restrict__ reward, unsigned long long* __restrict__ counters,
                    sched::Slot* slot, int tail_div)
{
    using G = CubeGeom<SIZE>;
    using L = WalkSmem<SIZE>;
    constexpr int W = WalkImage<SIZE>::W;
    extern __shared__ __align__(128) uint8_t smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t* s_ent = reinterpret_cast<uint32_t*>(smem + L::kEntries);
    uint8_t* mine = smem + L::kPerWarp + warp * L::per_warp(depth);
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(mine);             // [2]
    uint8_t* s_tile = mine + 16;                                      // [2][kTileBytes + 16]
    uint8_t* s_scratch = s_tile + 2 * (L::kTileBytes + 16);           // lane-private layout
    uint8_t* s_moves = s_scratch + L::kScratch;                       // [2][move_stride]
    const int mstride = L::move_stride(depth);
    const uint32_t move_bytes = (uint32_t)(kRowsPerTile * depth);

    asm volatile("griddepcontrol.launch_dependents;");                 // programmatic dependent launch, see scramble.cu
    for (int i = tid; i < 2 * G::NCYC * CUBE_MOVE_ROWS; i += blockDim.x) {
        const int shift = (i >= G::NCYC * CUBE_MOVE_ROWS) ? 2 : 0;
        const int cm = i - (shift ? G::NCYC * CUBE_MOVE_ROWS : 0);
        walk_cycle_entry((SIZE == 3) ? kCycles3[cm] : kCycles2[cm], shift, s_ent + 2 * i);
    }
    if (lane == 0) { bulk::mbar_init(&s_bar[0], 1); bulk::mbar_init(&s_bar[1], 1); }
    __syncthreads();
    asm volatile("griddepcontrol.wait;" ::: "memory");                // everything earlier in the stream is complete

    // tiles are claimed dynamically (cube_sched.cuh): `tile` is being turned, `next` is in flight
    sched::WarpTiles tiles;
    tiles.init(slot, n_tiles, (int)(blockDim.x >> 5), warp, lane, tail_div);
    int tile = tiles.pop(lane);
    if (lane == 0 && tile < n_tiles) {
        bulk::mbar_expect_tx(&s_bar[0], (uint32_t)L::kTileBytes + move_bytes);
        bulk::load(s_tile, in + (long long)tile * L::kTileBytes, (uint32_t)L::kTileBytes, &s_bar[0]);
        bulk::load(s_moves, moves + (long long)tile * move_bytes, move_bytes, &s_bar[0]);
    }
    uint8_t* lane_base = s_scratch + 4 * lane;
    unsigned n_solved = 0;

    for (int it = 0; tile < n_tiles; ++it) {
        const int buf = it & 1;
        const int next = tiles.pop(lane);
        if (lane == 0) {
            bulk::wait_read_all();                                    // the previous tile's store has left its buffer
            if (next < n_tiles) {                                     // ... which the next tile now fills
                bulk::mbar_expect_tx(&s_bar[buf ^ 1], (uint32_t)L::kTileBytes + move_bytes);
                bulk::load(s_tile + (buf ^ 1) * (L::kTileBytes + 16), in + (long long)next * L::kTileBytes,
                           (uint32_t)L::kTileBytes, &s_bar[buf ^ 1]);
                bulk::load(s_moves + (buf ^ 1) * mstride, moves + (long long)next * move_bytes, move_bytes, &s_bar[buf ^ 1]);
            }
        }
        bulk::mbar_wait(&s_bar[buf], (uint32_t)(it >> 1) & 1u);
        uint8_t* tile_p = s_tile + buf * (L::kTileBytes + 16);
        const uint8_t* moves_p = s_moves + buf * mstride;

        unsigned mask[2];
#pragma unroll
        for (int pass = 0; pass < 2; ++pass) {
            const int row = (SIZE == 3) ? 2 * lane + pass : lane + 32 * pass;
            constexpr int kShiftOdd = (SIZE == 3) ? 2 : 0;
            const int shift = pass ? kShiftOdd : 0;
            uint32_t* img_p = reinterpret_cast<uint32_t*>(tile_p + G::S * row - shift);
            uint32_t w[W];
            if (SIZE == 3) {
#pragma unroll
                for (int j = 0; j < W; ++j) w[j] = img_p[j];
            } else {                                                  // 24-byte rows: 8-byte accesses are conflict-free
                const uint2* q = reinterpret_cast<const uint2*>(img_p);
#pragma unroll
                for (int j = 0; j < 3; ++j) { const uint2 v = q[j]; w[2 * j] = v.x; w[2 * j + 1] = v.y; }
            }
            const uint8_t* mrow = moves_p + row * depth;
            if (SIZE == 3) {
#pragma unroll
                for (int j = 0; j < W; ++j) reinterpret_cast<uint32_t*>(lane_base)[32 * j] = w[j];
                const uint32_t* ent = s_ent + (shift ? 2 * G::NCYC * CUBE_MOVE_ROWS : 0);
                for (int k = 0; k < depth; ++k) walk_turn_private<SIZE>(lane_base, ent, (uint32_t)mrow[k] & 0xfu);
#pragma unroll
                for (int j = 0; j < W; ++j) w[j] = reinterpret_cast<const uint32_t*>(lane_base)[32 * j];
            } else {
                for (int k = 0; k < depth; ++k) walk_turn_registers2(w, (uint32_t)mrow[k] & 0xfu);
            }
            const bool ok = (pass && SIZE == 3) ? image_solved<SIZE, kShiftOdd>(w) : image_solved<SIZE, 0>(w);
            mask[pass] = __ballot_sync(0xffffffffu, ok);
            if (SIZE == 3) {
#pragma unroll
                for (int j = 0; j < W; ++j) img_p[j] = w[j];
            } else {
                uint2* q = reinterpret_cast<uint2*>(img_p);
#pragma unroll
                for (int j = 0; j < 3; ++j) q[j] = make_uint2(w[2 * j], w[2 * j + 1]);
            }
        }
        n_solved += (unsigned)(__popc(mask[0]) + __popc(mask[1]));

        bulk::fence_smem_writes();
        __syncwarp();
        if (lane == 0) {
            bulk::store(out + (long long)tile * L::kTileBytes, tile_p, (uint32_t)L::kTileBytes);
            bulk::commit();
        }
        if (solved && lane < 16)
            reinterpret_cast<uint32_t*>(solved + (long long)tile * kRowsPerTile)[lane] = pair_solved_word<SIZE>(mask[0], mask[1], lane);
        if (reward) {
            float2 v;
            v.x = pair_row_bit<SIZE>(mask[0], mask[1], 2 * lane) ? 1.0f : -1.0f;
            v.y = pair_row_bit<SIZE>(mask[0], mask[1], 2 * lane + 1) ? 1.0f : -1.0f;
            reinterpret_cast<float2*>(reward + (long long)tile * kRowsPerTile)[lane] = v;
        }
        tile = next;
    }
    if (lane == 0 && n_solved && counters) atomicAdd(&counters[0], (unsigned long long)n_solved);
    if (blockIdx.x == 0 && tid == 0 && counters) atomicAdd(&counters[1], (unsigned long long)n_tiles * kRowsPerTile);
    if (lane == 0) bulk::wait_read_all();
    __syncthreads();
    sched::release(slot);
}

// out-of-range action scan (the reference raises IndexError, cube_env.py:86,96)
__global__ void __launch_bounds__(256)
validate_kernel(const uint8_t* __restrict__ actions, long long count, unsigned n_actions,
                unsigned long long* __restrict__ counters)
{
    unsigned bad = 0;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long nvec = count >> 4;
    const uint4* v = reinterpret_cast<const uint4*>(actions);
    const uint32_t k = (0x80u - n_actions) * 0x01010101u;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += stride) {
        const uint4 q = __ldcs(v + i);
        const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int j = 0; j < 4; ++j)
            bad += __popc((((w[j] & 0x7f7f7f7fu) + k) | w[j]) & 0x80808080u);
    }
    for (long long i = (nvec << 4) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride)
        bad += actions[i] >= n_actions;
    for (int o = 16; o > 0; o >>= 1) bad += __shfl_xor_sync(0xffffffffu, bad, o);
    if ((threadIdx.x & 31) == 0 && bad) atomicAdd(&counters[2], (unsigned long long)bad);
}

template <int SIZE>
int launch_classic(const uint8_t* in, const uint8_t* moves, long long n, int depth, uint8_t* out, uint8_t* solved,
                   float* reward, unsigned long long* counters, cudaStream_t stream)
{
    cube::prefer_max_shared(walk_tile_kernel<SIZE, true>);
    const long long full_tiles = n / kTile;
    if (full_tiles > 0)
        walk_tile_kernel<SIZE, true><<<(unsigned)full_tiles, kTile, 0, stream>>>(in, moves, n, 0, depth, out, solved,
                                                                               reward, counters);
    if (full_tiles * kTile < n)
        walk_tile_kernel<SIZE, false><<<1, kTile, 0, stream>>>(in, moves, n, full_tiles, depth, out, solved, reward,
                                                              counters);
    return (int)cudaGetLastError();
}

template <int SIZE>
int launch_tiles(const uint8_t* in, const uint8_t* moves, long long n, int depth, uint8_t* out, uint8_t* solved,
                 float* reward, unsigned long long* counters, cudaStream_t stream)
{
    using L = WalkSmem<SIZE>;
    using G = CubeGeom<SIZE>;
    long long done = 0;
    static const bool classic = cube::env_flag("CUBE_WALK_CLASSIC", false);        // A/B switch for profiling
    // K2p stages the move bytes by bulk copies (16-byte aligned source) and writes the verdicts as 32-bit /
    // float2 words; a caller's sliced tensor (actions_all[t] of a [T, N] array, a view into a larger solved /
    // reward buffer) need not be aligned like that: such calls take the byte-wise tile kernel below
    const bool aligned = ((reinterpret_cast<uintptr_t>(moves) & 15u) | (reinterpret_cast<uintptr_t>(solved) & 3u) |
                          (reinterpret_cast<uintptr_t>(reward) & 7u)) == 0;
    if (depth >= 1 && depth <= kMaxPrivateDepth && out && n >= kRowsPerTile && aligned && !classic) {
        const int warps = cube::warps_that_fit(L::kPerWarp, L::per_warp(depth), kMaxWalkWarps) & ~3;
        if (warps >= 8) {
            long long n_tiles = n / kRowsPerTile;
            if (n_tiles > 0x3fffffff) n_tiles = 0x3fffffff;
            const int smem = L::bytes(depth, warps);
            auto kern = walk_private_kernel<SIZE>;
            cudaError_t e = cube::raise_smem_limit(kern, smem);
            if (e != cudaSuccess) return (int)e;
            sched::Slot* slot = sched::claim_slot();
            if (!slot) return (int)cudaErrorUnknown;
            e = cube::launch_pdl(kern, cube::persistent_grid(n_tiles, warps), warps * 32, smem, stream, in, moves, (int)n_tiles,
                                 depth, out, solved, reward, counters, slot, sched::tail_div());
            if (e != cudaSuccess) return (int)e;
            done = n_tiles * kRowsPerTile;
        }
    }
    if (done == n) return 0;
    return launch_classic<SIZE>(in + done * G::S, moves ? moves + done * depth : nullptr, n - done, depth,
                                out ? out + done * G::S : nullptr, solved ? solved + done : nullptr,
                                reward ? reward + done : nullptr, counters, stream);
}

}  // namespace

namespace cube {

int launch_walk(int size, const uint8_t* states_in, const uint8_t* moves, long long n, int depth,
                uint8_t* states_out, uint8_t* solved, float* reward, unsigned long long* counters,
                cudaStream_t stream)
{
    if (n == 0) return 0;
    if (size == 3) return launch_tiles<3>(states_in, moves, n, depth, states_out, solved, reward, counters, stream);
    return launch_tiles<2>(states_in, moves, n, depth, states_out, solved, reward, counters, stream);
}

int launch_solved(int size, const uint8_t* states, long long n, uint8_t* solved, float* reward,
                  unsigned long long* counters, cudaStream_t stream)
{
    if (n == 0) return 0;
    if (size == 3) return launch_tiles<3>(states, nullptr, n, 0, nullptr, solved, reward, counters, stream);
    return launch_tiles<2>(states, nullptr, n, 0, nullptr, solved, reward, counters, stream);
}

int launch_validate(int size, const uint8_t* actions, long long count, unsigned long long* counters,
                    cudaStream_t stream)
{
    if (count == 0) return 0;
    long long blocks = (count / 16 + 255) / 256;
    const long long cap = (long long)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    validate_kernel<<<(unsigned)blocks, 256, 0, stream>>>(actions, count, size == 3 ? 12u : 6u, counters);
    return (int)cudaGetLastError();
}

}  // namespace cube
