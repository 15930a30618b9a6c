// Exact 2x2x2 distances (include/cube_b200.h cube_distance_*): the table of every state's quarter-turn distance,
// built on the device by a level-synchronous breadth-first search over ranks, and two row kernels on top of it --
// the lookup (one table load per row) and the optimal solve (a walk down the table).  The per-state code is in
// cube_distance.cuh, shared with the CPU emulation of the tests.
#include <cuda_runtime.h>
#include "cube_distance.cuh"
#include "cube_kernels.h"

namespace {

constexpr int kThreads = 256;
constexpr uint32_t kTableWords = kDist2Entries / 4;                // 3 674 160 is a multiple of 16
static_assert(kDist2Entries % 16 == 0, "the level kernel reads the table as words");

// Level d: every rank at distance d marks its unvisited neighbours d + 1.  The table is read with plain loads:
// other threads of the same launch write d + 1 into it, which is never mistaken for d.
__global__ void __launch_bounds__(kThreads)
dist2_level_kernel(uint8_t* table, uint32_t d)
{
    const uint32_t i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= kTableWords) return;
    const uint32_t v = reinterpret_cast<const uint32_t*>(table)[i];
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (((v >> (8 * k)) & 0xffu) == d) dist2_expand(table, 4u * i + (uint32_t)k, d);
}

__device__ __forceinline__ void dist2_row_words(const uint8_t* states, long long i, uint32_t* row)
{
    const uint2* p = reinterpret_cast<const uint2*>(states + 24 * i);  // 16-byte aligned base: rows on 8 bytes
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const uint2 v = __ldcs(p + j);
        row[2 * j] = v.x;
        row[2 * j + 1] = v.y;
    }
}

__global__ void __launch_bounds__(kThreads)
dist2_lookup_kernel(const uint8_t* __restrict__ table, const uint8_t* __restrict__ states, long long n,
                    uint8_t* __restrict__ distance)
{
    const long long i = (long long)blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    uint32_t row[6];
    dist2_row_words(states, i, row);
    distance[i] = (uint8_t)dist2_lookup(table, row);
}

// one thread per row; the block's [rows, 14] action bytes are staged in shared memory and leave coalesced
constexpr int kSolveThreads = 128;

__global__ void __launch_bounds__(kSolveThreads)
dist2_solve_kernel(const uint8_t* __restrict__ table, const uint8_t* __restrict__ states, long long n,
                   uint8_t* __restrict__ actions, uint8_t* __restrict__ length)
{
    __shared__ uint8_t s_act[kSolveThreads * kDist2Max];
    const long long base = (long long)blockIdx.x * kSolveThreads;
    const long long i = base + threadIdx.x;
    if (i < n) {
        uint32_t row[6];
        dist2_row_words(states, i, row);
        length[i] = (uint8_t)dist2_solve(table, row, s_act + kDist2Max * threadIdx.x);
    }
    __syncthreads();
    const int cnt = (int)((n - base) < (long long)kSolveThreads ? (n - base) : (long long)kSolveThreads);
    uint8_t* dst = actions + base * kDist2Max;
    for (int k = threadIdx.x; k < cnt * kDist2Max; k += kSolveThreads) dst[k] = s_act[k];
}

}  // namespace

namespace cube {

int launch_distance_build2(uint8_t* table, cudaStream_t stream)
{
    cudaError_t e = cudaMemsetAsync(table, CUBE_DISTANCE_UNREACHABLE, kDist2Entries, stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(table, 0, 1, stream);                 // the solved cube: rank 0
    if (e != cudaSuccess) return (int)e;
    // every state is at most kDist2Max turns from solved: levels 0 .. kDist2Max - 1 reach them all
    const unsigned blocks = (kTableWords + kThreads - 1) / kThreads;
    for (uint32_t d = 0; d < (uint32_t)kDist2Max; ++d) dist2_level_kernel<<<blocks, kThreads, 0, stream>>>(table, d);
    return (int)cudaGetLastError();
}

int launch_distance2(const uint8_t* table, const uint8_t* states, long long n, uint8_t* distance, cudaStream_t stream)
{
    if (n == 0) return 0;
    dist2_lookup_kernel<<<(unsigned)((n + kThreads - 1) / kThreads), kThreads, 0, stream>>>(table, states, n, distance);
    return (int)cudaGetLastError();
}

int launch_solve_optimal2(const uint8_t* table, const uint8_t* states, long long n, uint8_t* actions, uint8_t* length,
                          cudaStream_t stream)
{
    if (n == 0) return 0;
    dist2_solve_kernel<<<(unsigned)((n + kSolveThreads - 1) / kSolveThreads), kSolveThreads, 0, stream>>>(
        table, states, n, actions, length);
    return (int)cudaGetLastError();
}

}  // namespace cube
