// K1x -- every prefix of every scramble in ONE launch, cube-major (sm_100a).
//
// The reference's get_random_samples (cube_env.py:187-194) emits a sample after EVERY move of every
// scramble: the parents of an ADI batch are all scramble prefixes, appended cube by cube, depth by
// depth.  This kernel writes exactly that array:
//     states_out[i, k, :] = the sticker row after moves[i, 0..k]        (k = 0 .. depth-1)
// A warp owns a tile of 8 cubes = one contiguous block of 8 * depth sticker rows of the output, and
// FOUR lanes share a cube: lane (part, cube) walks the cube with the fused-scramble arithmetic (five
// registers of cubie bytes, one PRMT table row per move, cube_common.cuh), fast-forwards through the
// moves before its quarter of the levels (a move is ~12 instructions) and expands every level of its
// quarter to a sticker row (~100 instructions) in a shared-memory image of the tile's output block; the
// finished block leaves by one bulk store (TMA), so the 54-byte rows cost no uncoalesced global stores.
// (The first version gave a lane a whole cube and a warp 32 cubes: a 52 KB image per warp at depth 30,
// 4 warps per SM, 30 dependent levels per lane: 0.095 ms for config 4's parents, occupancy 6 %.)  Replaces one cube_walk launch
// per depth level plus the step-major -> cube-major transposes of round 1 (adi.py).
// HBM traffic per cube: depth (moves in) + depth * (S + 1) bytes out.
#include <cuda_runtime.h>
#include "cube_bulk.cuh"
#include "cube_kernels.h"
#include "cube_launch.cuh"
#include "cube_threads.cuh"

namespace {

constexpr int kSplit = 4;                          // lanes per cube: the levels of a cube are split four ways
constexpr int kCubesPerTile = 32 / kSplit;
constexpr int kMaxWarps = 16;

template <int SIZE>
struct PrefixSmem {
    using G = CubeGeom<SIZE>;
    static constexpr int kTable = 0;                                   // [MW][16] move words
    static constexpr int kCornerLut = kTable + G::MW * CUBE_MOVE_ROWS * 4;
    static constexpr int kEdgeLut = kCornerLut + 32 * 4;
    static constexpr int kPerWarp = (kEdgeLut + 64 * 4 + 127) & ~127;
    __host__ __device__ static constexpr int image_bytes(int depth) { return (kCubesPerTile * depth * G::S + 15) & ~15; }
    __host__ __device__ static constexpr int moves_bytes(int depth) { return (kCubesPerTile * depth + 15 + 16) & ~15; }
    __host__ __device__ static constexpr int per_warp(int depth) { return image_bytes(depth) + moves_bytes(depth); }
    __host__ __device__ static constexpr int bytes(int depth, int warps) { return kPerWarp + warps * per_warp(depth); }
};

template <int SIZE>
__global__ void __launch_bounds__(kMaxWarps * 32, 1)
prefix_kernel(const uint8_t* __restrict__ moves, long long n, int depth, uint8_t* __restrict__ out,
              uint8_t* __restrict__ solved, unsigned long long* __restrict__ counters)
{
    using G = CubeGeom<SIZE>;
    using L = PrefixSmem<SIZE>;
    extern __shared__ __align__(128) uint8_t smem[];
    uint32_t* s_tbl = reinterpret_cast<uint32_t*>(smem + L::kTable);
    uint32_t* s_clut = reinterpret_cast<uint32_t*>(smem + L::kCornerLut);
    uint32_t* s_elut = reinterpret_cast<uint32_t*>(smem + L::kEdgeLut);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, warps = (int)(blockDim.x >> 5);
    uint8_t* s_img = smem + L::kPerWarp + warp * L::per_warp(depth);
    uint8_t* s_mv = s_img + L::image_bytes(depth);

    for (int i = tid; i < G::MW * CUBE_MOVE_ROWS; i += blockDim.x) s_tbl[i] = (SIZE == 3) ? kMoveWords3[i] : kMoveWords2[i];
    for (int i = tid; i < 32; i += blockDim.x) s_clut[i] = (SIZE == 3) ? kCornerColour3[i] : kCornerColour2[i];
    for (int i = tid; i < 64; i += blockDim.x) s_elut[i] = (SIZE == 3) ? kEdgeColour3[i] : 0u;
    __syncthreads();

    const long long n_tiles = (n + kCubesPerTile - 1) / kCubesPerTile;
    const long long row_bytes = (long long)depth * G::S;                // one cube's block of the output
    unsigned n_solved = 0;
    for (long long tile = (long long)blockIdx.x * warps + warp; tile < n_tiles; tile += (long long)gridDim.x * warps) {
        const long long cube0 = tile * kCubesPerTile;
        const int cnt = (n - cube0) < kCubesPerTile ? (int)(n - cube0) : kCubesPerTile;
        // the tile's move bytes: 8 * depth contiguous bytes, word-aligned (cube0 is a multiple of 8)
        const uint8_t* mv_g = moves + cube0 * depth;
        const int mv_bytes = cnt * depth;
        {
            const uint32_t* src = reinterpret_cast<const uint32_t*>(mv_g);
            uint32_t* dst = reinterpret_cast<uint32_t*>(s_mv);
            const int nw = mv_bytes >> 2;
            for (int i = lane; i < nw; i += 32) dst[i] = __ldcs(src + i);
            for (int i = (nw << 2) + lane; i < mv_bytes; i += 32) s_mv[i] = mv_g[i];
        }
        if (lane == 0) bulk::wait_read_all();                           // the previous tile's store has read the image
        __syncwarp();
        {
            const int cube = lane % kCubesPerTile, part = lane / kCubesPerTile;
            const int k_begin = part * depth / kSplit, k_end = (part + 1) * depth / kSplit;
            if (cube < cnt && k_begin < k_end)
                n_solved += prefix_walk<SIZE>(s_mv + cube * depth, depth, cube * depth, s_tbl, s_clut, s_elut, s_img,
                                              solved ? solved + (cube0 + cube) * depth : nullptr, k_begin, k_end);
        }
        bulk::fence_smem_writes();
        __syncwarp();
        uint8_t* dst_g = out + cube0 * row_bytes;
        // a whole tile leaves by one bulk store when its block is a multiple of 16 bytes (8 * S is: any depth
        // for 2x2x2; 8 * 54 = 432 = 27 * 16 for 3x3x3)
        if (cnt == kCubesPerTile) {
            if (lane == 0) {
                bulk::store(dst_g, s_img, (uint32_t)(kCubesPerTile * depth * G::S));
                bulk::commit();
            }
        } else {                                                        // ragged last tile: plain copies
            const long long nb = (long long)cnt * row_bytes;
            const int nw = (int)(nb >> 2);
            for (int i = lane; i < nw; i += 32) reinterpret_cast<uint32_t*>(dst_g)[i] = reinterpret_cast<const uint32_t*>(s_img)[i];
            for (long long i = ((long long)nw << 2) + lane; i < nb; i += 32) dst_g[i] = s_img[i];
        }
    }
    n_solved = __reduce_add_sync(0xffffffffu, n_solved);
    if (lane == 0 && n_solved && counters) atomicAdd(&counters[0], (unsigned long long)n_solved);
    if (blockIdx.x == 0 && tid == 0 && counters) atomicAdd(&counters[1], (unsigned long long)n * (unsigned long long)depth);
    if (lane == 0) bulk::wait_read_all();                               // shared memory must outlive the copies' reads
}

template <int SIZE>
int launch_one(const uint8_t* moves, long long n, int depth, uint8_t* out, uint8_t* solved, unsigned long long* counters,
               cudaStream_t stream)
{
    using L = PrefixSmem<SIZE>;
    const int warps = cube::warps_that_fit(L::kPerWarp, L::per_warp(depth), kMaxWarps);
    if (warps < 1) return CUBE_ERR_ARG;                                 // depth too large for one tile image
    const int smem = L::bytes(depth, warps);
    auto kern = prefix_kernel<SIZE>;
    const cudaError_t e = cube::raise_smem_limit(kern, smem);
    if (e != cudaSuccess) return (int)e;
    const long long n_tiles = (n + kCubesPerTile - 1) / kCubesPerTile;
    long long grid = (n_tiles + warps - 1) / warps;
    if (grid > cube::sm_count()) grid = cube::sm_count();
    kern<<<(unsigned)grid, warps * 32, smem, stream>>>(moves, n, depth, out, solved, counters);
    return (int)cudaGetLastError();
}

}  // namespace

namespace cube {

int prefix_max_depth(int size)
{
    const int per_level = kCubesPerTile * (size == 3 ? 54 : 24) + kCubesPerTile;
    return (cube::kSmemPerBlock - (size == 3 ? PrefixSmem<3>::kPerWarp : PrefixSmem<2>::kPerWarp) - 32) / per_level;
}

int launch_prefixes(int size, const uint8_t* moves, long long n, int depth, uint8_t* states_out, uint8_t* solved,
                    unsigned long long* counters, cudaStream_t stream)
{
    if (n == 0 || depth == 0) return 0;
    if (size == 3) return launch_one<3>(moves, n, depth, states_out, solved, counters, stream);
    return launch_one<2>(moves, n, depth, states_out, solved, counters, stream);
}

}  // namespace cube
