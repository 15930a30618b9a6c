// 3x3x3 pattern databases (include/cube_b200.h cube_pattern_* / cube_distance_bound / cube_solve_bounded): the
// corner and the two 6-edge tables, built on the device by a level-synchronous breadth-first search over ranks, and
// two row kernels on top of them -- the admissible bound (three table loads per row) and the bounded IDA* solve
// (one thread per row).  The per-state code is in cube_pattern.cuh, shared with the CPU emulation of the tests.
#include <cuda_runtime.h>
#include "cube_pattern.cuh"
#include "cube_kernels.h"

namespace {

constexpr int kThreads = 256;

// Level d of section SECTION: every rank at distance d marks its unvisited neighbours d + 1.  The table is read with
// plain loads: other threads of the same launch write d + 1 into it, which is never mistaken for d, and a rank
// marked d + 1 during the launch is expanded by the next one -- so the result does not depend on the order.
template <int SECTION>
__global__ void __launch_bounds__(kThreads)
pat3_level_kernel(uint8_t* table, uint32_t words, uint32_t d)
{
    const uint32_t i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= words) return;
    const uint32_t v = reinterpret_cast<const uint32_t*>(table)[i];
#pragma unroll 1
    for (int k = 0; k < 4; ++k)
        if (((v >> (8 * k)) & 0xffu) == d) pat3_expand(table, SECTION, 4u * i + (uint32_t)k, d);
}

// The block's sticker rows (54 bytes each) are staged in shared memory with 16-byte loads: the row base is 16-byte
// aligned and every block starts a multiple of 16 bytes into it.
constexpr int kRowBytes = 54;

template <int ROWS>
__device__ __forceinline__ void pat3_stage_rows(const uint8_t* states, long long base, int cnt, uint8_t* s_rows)
{
    static_assert(ROWS * kRowBytes % 16 == 0, "a block's rows must span whole 16-byte vectors");
    const uint8_t* src = states + base * kRowBytes;
    const int bytes = cnt * kRowBytes, vecs = bytes >> 4;
    for (int k = threadIdx.x; k < vecs; k += blockDim.x)
        reinterpret_cast<uint4*>(s_rows)[k] = __ldcs(reinterpret_cast<const uint4*>(src) + k);
    for (int k = 16 * vecs + threadIdx.x; k < bytes; k += blockDim.x) s_rows[k] = src[k];
    __syncthreads();
}

constexpr int kBoundThreads = 128;

__global__ void __launch_bounds__(kBoundThreads)
pat3_bound_kernel(const uint8_t* __restrict__ tables, const uint8_t* __restrict__ states, long long n,
                  uint8_t* __restrict__ bound, uint8_t* __restrict__ parts)
{
    __shared__ __align__(16) uint8_t s_rows[kBoundThreads * kRowBytes];
    const long long base = (long long)blockIdx.x * kBoundThreads;
    const int cnt = (int)((n - base) < (long long)kBoundThreads ? (n - base) : (long long)kBoundThreads);
    pat3_stage_rows<kBoundThreads>(states, base, cnt, s_rows);
    if ((int)threadIdx.x >= cnt) return;
    const long long i = base + threadIdx.x;
    uint32_t p[3];
    bound[i] = (uint8_t)pat3_row_bound(tables, s_rows + kRowBytes * threadIdx.x, p);
    if (parts) {
        parts[3 * i] = (uint8_t)p[0];
        parts[3 * i + 1] = (uint8_t)p[1];
        parts[3 * i + 2] = (uint8_t)p[2];
    }
}

// one thread per row: a row's search runs from its first threshold to its last in one thread
constexpr int kSolveThreads = 64;

__global__ void __launch_bounds__(kSolveThreads)
pat3_solve_kernel(const uint8_t* __restrict__ tables, const uint8_t* __restrict__ states, long long n, int max_length,
                  long long max_nodes, uint8_t* __restrict__ actions, uint8_t* __restrict__ length,
                  uint8_t* __restrict__ lower, long long* __restrict__ nodes)
{
    __shared__ __align__(16) uint8_t s_rows[kSolveThreads * kRowBytes];
    const long long base = (long long)blockIdx.x * kSolveThreads;
    const int cnt = (int)((n - base) < (long long)kSolveThreads ? (n - base) : (long long)kSolveThreads);
    pat3_stage_rows<kSolveThreads>(states, base, cnt, s_rows);
    if ((int)threadIdx.x >= cnt) return;
    const long long i = base + threadIdx.x;
    const Pat3Solve r = pat3_solve(tables, s_rows + kRowBytes * threadIdx.x, max_length, max_nodes,
                                   actions + (long long)max_length * i);
    length[i] = (uint8_t)r.length;
    lower[i] = (uint8_t)r.lower;
    if (nodes) nodes[i] = r.nodes;
}

template <int SECTION>
void pat3_build_section(uint8_t* tables, cudaStream_t stream)
{
    uint8_t* table = tables + kPat3Offset[SECTION];
    const uint32_t words = kPat3Entries[SECTION] / 4;
    const unsigned blocks = (words + kThreads - 1) / kThreads;
    // every state of the section is at most kPat3Levels turns from solved: levels 0 .. max - 1 reach them all
    for (uint32_t d = 0; d < (uint32_t)kPat3Levels[SECTION]; ++d)
        pat3_level_kernel<SECTION><<<blocks, kThreads, 0, stream>>>(table, words, d);
}

}  // namespace

namespace cube {

int launch_pattern_build3(uint8_t* tables, cudaStream_t stream)
{
    cudaError_t e = cudaMemsetAsync(tables, CUBE_DISTANCE_UNREACHABLE, kPat3Bytes, stream);
    for (int s = 0; s < 3 && e == cudaSuccess; ++s) e = cudaMemsetAsync(tables + kPat3Offset[s], 0, 1, stream);   // rank 0
    if (e != cudaSuccess) return (int)e;
    pat3_build_section<0>(tables, stream);
    pat3_build_section<1>(tables, stream);
    pat3_build_section<2>(tables, stream);
    return (int)cudaGetLastError();
}

int launch_distance_bound3(const uint8_t* tables, const uint8_t* states, long long n, uint8_t* bound, uint8_t* parts,
                           cudaStream_t stream)
{
    if (n == 0) return 0;
    pat3_bound_kernel<<<(unsigned)((n + kBoundThreads - 1) / kBoundThreads), kBoundThreads, 0, stream>>>(
        tables, states, n, bound, parts);
    return (int)cudaGetLastError();
}

int launch_solve_bounded3(const uint8_t* tables, const uint8_t* states, long long n, int max_length, long long max_nodes,
                          uint8_t* actions, uint8_t* length, uint8_t* lower, long long* nodes, cudaStream_t stream)
{
    if (n == 0) return 0;
    pat3_solve_kernel<<<(unsigned)((n + kSolveThreads - 1) / kSolveThreads), kSolveThreads, 0, stream>>>(
        tables, states, n, max_length, max_nodes, actions, length, lower, nodes);
    return (int)cudaGetLastError();
}

}  // namespace cube
