// K0 -- identically seeded scrambles on the device (sm_100a): the move indices the reference draws in
//   reset(seed, k):  np.random.seed(seed); np.random.randint(A, size=k)          cube_env.py:62-65
// i.e. np.random.RandomState(seed).randint(A, size=k), for n seeds at once, so that seeded batches
// (config 1: seeds 0..1023; validation: seed = 10 * cube, train.py:180) need no host RNG and no
// upload of move bytes.  The per-seed draw -- a one-word-recurrence fast path for the first 227 raw
// outputs and an exact slow path for the rare row that needs more -- is csrc/cube_seeds.cuh; a row that
// took the slow path is counted in counters[3].
#include <cuda_runtime.h>
#include "cube_kernels.h"
#include "../../include/cube_b200.h"
#include "cube_seeds.cuh"

namespace {

constexpr int kSeedThreads = 128;

// a row of the CTA's shared-memory staging area as a 32-bit shared-window address that only ever advances: the
// generic pointer form made the compiler rebuild the window base (S2R) for every accepted draw
struct SharedRow {
    uint32_t p, end;
    __device__ __forceinline__ bool full() const { return p >= end; }
    __device__ __forceinline__ void put(uint32_t v)
    {
        asm volatile("st.shared.u8 [%0], %1;" ::"r"(p), "r"(v) : "memory");
        ++p;
    }
};

__global__ void __launch_bounds__(kSeedThreads)
seeded_moves_kernel(const uint32_t* __restrict__ seeds, long long n, int depth, uint32_t max_value, uint32_t mask,
                    uint8_t* __restrict__ moves, unsigned long long* __restrict__ counters)
{
    // the CTA's 128 rows are staged in shared memory and leave as one coalesced stream: per-thread byte
    // stores to rows `depth` bytes apart cost one partial L2 sector write per lane and move
    extern __shared__ __align__(16) uint8_t s_rows[];
    const int tid = threadIdx.x;
    const long long base = (long long)blockIdx.x * kSeedThreads;
    const long long i = base + tid;
    if (i < n) {
        const uint32_t p = (uint32_t)__cvta_generic_to_shared(s_rows) + (uint32_t)(tid * depth);
        if (seed_row(seeds[i], max_value, mask, SharedRow{p, p + (uint32_t)depth}) && counters)
            atomicAdd(&counters[3], 1ull);
    }
    __syncthreads();
    const long long rows = (n - base) < (long long)kSeedThreads ? (n - base) : (long long)kSeedThreads;
    const int nbytes = (int)rows * depth;
    uint8_t* dst = moves + base * depth;                                         // 128 * depth: a multiple of 16
    const int nvec = nbytes >> 4;
    for (int v = tid; v < nvec; v += kSeedThreads)
        reinterpret_cast<int4*>(dst)[v] = reinterpret_cast<const int4*>(s_rows)[v];
    for (int k = (nvec << 4) + tid; k < nbytes; k += kSeedThreads) dst[k] = s_rows[k];
}

}  // namespace

namespace cube {

int launch_seeded_moves(int size, const uint32_t* seeds, long long n, int depth, uint8_t* moves,
                        unsigned long long* counters, cudaStream_t stream)
{
    if (n == 0 || depth == 0) return 0;
    const uint32_t max_value = size == 3 ? 11u : 5u;
    const uint32_t mask = seed_mask(max_value);
    const long long blocks = (n + kSeedThreads - 1) / kSeedThreads;
    seeded_moves_kernel<<<(unsigned)blocks, kSeedThreads, (size_t)kSeedThreads * depth, stream>>>(seeds, n, depth, max_value,
                                                                                                   mask, moves, counters);
    return (int)cudaGetLastError();
}

}  // namespace cube
