// Host-buffer front end of the fused scramble: the end-to-end path a caller with NumPy /
// pinned host arrays uses (bench.py's `e2e` figure).  The batch is cut into chunks that
// rotate over a few stages, each with its own stream and device buffers, so the H2D copy of
// chunk c+1, the kernel of chunk c and the D2H copy of chunk c-1 overlap (the two copy
// engines run in opposite directions at the same time).  All device memory is owned by
// the handle; the per-call entry point allocates nothing.
#include <cuda_runtime.h>
#include <sys/mman.h>
#include <cstring>
#include <map>
#include <mutex>
#include <new>

#include "../../include/cube_b200.h"
#include "cube_common.cuh"
#include "cube_kernels.h"

struct cube_pipeline {
    int cube_size, depth, n_stages;
    long long chunk;                 // instances per chunk (multiple of 256)
    cudaStream_t stream[4];
    uint8_t* d_moves[4];
    uint32_t* d_seeds[4];            // cube_pipeline_reset_host: the chunk's seeds (4 bytes per instance instead of `depth`)
    uint8_t* d_states[4];
    uint8_t* d_solved[4];
    float* d_reward[4];
    unsigned long long* d_counters;  // [n_stages][4]
    unsigned long long* h_counters;  // pinned mirror
};

namespace {

void destroy(cube_pipeline* p)
{
    if (!p) return;
    for (int s = 0; s < p->n_stages; ++s) {
        if (p->d_moves[s]) cudaFree(p->d_moves[s]);
        if (p->d_seeds[s]) cudaFree(p->d_seeds[s]);
        if (p->d_states[s]) cudaFree(p->d_states[s]);
        if (p->d_solved[s]) cudaFree(p->d_solved[s]);
        if (p->d_reward[s]) cudaFree(p->d_reward[s]);
        if (p->stream[s]) cudaStreamDestroy(p->stream[s]);
    }
    if (p->d_counters) cudaFree(p->d_counters);
    if (p->h_counters) cudaFreeHost(p->h_counters);
    delete p;
}

}  // namespace

extern "C" {

int cube_pipeline_create(int cube_size, int depth, int64_t chunk_instances, int n_stages, cube_pipeline** out)
{
    if (cube_size != 2 && cube_size != 3) return CUBE_ERR_SIZE;
    if (!out || depth < 0 || chunk_instances < 1 || n_stages < 1 || n_stages > 4) return CUBE_ERR_ARG;
    cube_pipeline* p = new (std::nothrow) cube_pipeline();
    if (!p) return (int)cudaErrorMemoryAllocation;
    p->cube_size = cube_size;
    p->depth = depth;
    p->n_stages = n_stages;
    p->chunk = (chunk_instances + 255) / 256 * 256;
    const size_t S = cube_size == 3 ? 54 : 24;
    cudaError_t e = cudaSuccess;
    for (int s = 0; s < n_stages && e == cudaSuccess; ++s) {
        e = cudaStreamCreateWithFlags(&p->stream[s], cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaMalloc(&p->d_moves[s], (size_t)p->chunk * (depth > 0 ? depth : 1));
        if (e == cudaSuccess) e = cudaMalloc(&p->d_seeds[s], (size_t)p->chunk * sizeof(uint32_t));
        if (e == cudaSuccess) e = cudaMalloc(&p->d_states[s], (size_t)p->chunk * S);
        if (e == cudaSuccess) e = cudaMalloc(&p->d_solved[s], (size_t)p->chunk);
        if (e == cudaSuccess) e = cudaMalloc(&p->d_reward[s], (size_t)p->chunk * sizeof(float));
    }
    if (e == cudaSuccess) e = cudaMalloc(&p->d_counters, sizeof(unsigned long long) * 4 * n_stages);
    if (e == cudaSuccess) e = cudaMallocHost(&p->h_counters, sizeof(unsigned long long) * 4 * n_stages);
    if (e != cudaSuccess) {
        destroy(p);
        return (int)e;
    }
    *out = p;
    return 0;
}

int cube_pipeline_destroy(cube_pipeline* p)
{
    destroy(p);
    return 0;
}

}  // extern "C"

namespace {

// the chunk loop shared by the two front ends: `seeds_host` != nullptr draws the moves on the device (K0)
int run_host(cube_pipeline* p, const uint8_t* moves_host, const uint32_t* seeds_host, int64_t n, uint8_t* states_out_host,
             uint8_t* solved_host, float* reward_host, int64_t* solved_count)
{
    const size_t S = p->cube_size == 3 ? 54 : 24;
    cudaError_t e = cudaMemsetAsync(p->d_counters, 0, sizeof(unsigned long long) * 4 * p->n_stages, p->stream[0]);
    if (e == cudaSuccess) e = cudaStreamSynchronize(p->stream[0]);
    int rc = 0;
    long long c = 0;
    for (long long off = 0; off < n && e == cudaSuccess && rc == 0; off += p->chunk, ++c) {
        const int s = (int)(c % p->n_stages);
        const long long cnt = (n - off) < p->chunk ? (n - off) : p->chunk;
        cudaStream_t st = p->stream[s];
        if (seeds_host) {
            e = cudaMemcpyAsync(p->d_seeds[s], seeds_host + off, (size_t)cnt * sizeof(uint32_t), cudaMemcpyHostToDevice, st);
            if (e != cudaSuccess) break;
            rc = cube::launch_seeded_moves(p->cube_size, p->d_seeds[s], cnt, p->depth, p->d_moves[s],
                                           p->d_counters + 4 * s, st);
            if (rc) break;
        } else if (p->depth > 0) {
            e = cudaMemcpyAsync(p->d_moves[s], moves_host + off * p->depth, (size_t)cnt * p->depth,
                                cudaMemcpyHostToDevice, st);
            if (e != cudaSuccess) break;
        }
        rc = cube::launch_scramble(p->cube_size, p->d_moves[s], cnt, p->depth, p->d_states[s],
                                   solved_host ? p->d_solved[s] : nullptr, reward_host ? p->d_reward[s] : nullptr,
                                   p->d_counters + 4 * s, st);
        if (rc) break;
        e = cudaMemcpyAsync(states_out_host + off * S, p->d_states[s], (size_t)cnt * S, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess && solved_host)
            e = cudaMemcpyAsync(solved_host + off, p->d_solved[s], (size_t)cnt, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess && reward_host)
            e = cudaMemcpyAsync(reward_host + off, p->d_reward[s], (size_t)cnt * sizeof(float),
                                cudaMemcpyDeviceToHost, st);
    }
    for (int s = 0; s < p->n_stages; ++s) {
        cudaError_t e2 = cudaStreamSynchronize(p->stream[s]);
        if (e == cudaSuccess) e = e2;
    }
    if (rc) return rc;
    if (e != cudaSuccess) return (int)e;
    e = cudaMemcpy(p->h_counters, p->d_counters, sizeof(unsigned long long) * 4 * p->n_stages, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return (int)e;
    long long total = 0;
    for (int s = 0; s < p->n_stages; ++s) total += (long long)p->h_counters[4 * s];
    if (solved_count) *solved_count = total;
    return 0;
}

}  // namespace

extern "C" {

// moves_host [n, depth]; states_out_host [n, S]; solved_host [n] / reward_host [n] may be NULL.
// Blocks until the host buffers are filled.  Host buffers should be page-locked for the
// copies to overlap; pageable memory works but serialises.
int cube_pipeline_scramble_host(cube_pipeline* p, const uint8_t* moves_host, int64_t n, uint8_t* states_out_host,
                                uint8_t* solved_host, float* reward_host, int64_t* solved_count)
{
    if (!p || n < 0 || (n > 0 && (!states_out_host || (p->depth > 0 && !moves_host)))) return CUBE_ERR_ARG;
    return run_host(p, moves_host, nullptr, n, states_out_host, solved_host, reward_host, solved_count);
}

// Batched reset(seed, k) (cube_env.py:50-69) for host arrays: 4 bytes per instance go to the device, the moves
// np.random.RandomState(seed).randint(A, size=depth) are drawn there (K0) and scrambled (K1p).
int cube_pipeline_reset_host(cube_pipeline* p, const uint32_t* seeds_host, int64_t n, uint8_t* states_out_host,
                             uint8_t* solved_host, float* reward_host, int64_t* solved_count)
{
    if (!p || n < 0 || p->depth < 1 || p->depth > 128 || (n > 0 && (!states_out_host || !seeds_host))) return CUBE_ERR_ARG;
    return run_host(p, nullptr, seeds_host, n, states_out_host, solved_host, reward_host, solved_count);
}

}  // extern "C"

// ---- page-locked host buffers on huge pages ---------------------------------------------------------
// cudaMallocHost / pin_memory give 4 KiB pages.  With one process per GPU all copying at once, the DMA
// engines' address translations (IOMMU / ATS in a virtual machine) are one more shared resource; a buffer
// that sits on 2 MiB transparent huge pages needs 512 times fewer of them.  The buffer is 2 MiB-aligned,
// advised MADV_HUGEPAGE, touched (so the pages exist before they are locked) and then registered.
namespace {
std::mutex g_host_mu;
std::map<void*, std::pair<void*, size_t>> g_host_maps;      // aligned pointer -> (mapping base, mapping length)
constexpr size_t kHuge = 2u << 20;
}  // namespace

extern "C" {

int cube_host_alloc(int64_t bytes, void** out)
{
    if (!out || bytes <= 0) return CUBE_ERR_ARG;
    const size_t len = ((size_t)bytes + kHuge - 1) / kHuge * kHuge;
    void* base = mmap(nullptr, len + kHuge, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
    if (base == MAP_FAILED) return (int)cudaErrorMemoryAllocation;
    void* p = reinterpret_cast<void*>((reinterpret_cast<uintptr_t>(base) + kHuge - 1) / kHuge * kHuge);
    (void)madvise(p, len, MADV_HUGEPAGE);                    // best effort: THP may be disabled on the host
    memset(p, 0, len);
    const cudaError_t e = cudaHostRegister(p, len, cudaHostRegisterPortable);
    if (e != cudaSuccess) {
        munmap(base, len + kHuge);
        return (int)e;
    }
    std::lock_guard<std::mutex> lock(g_host_mu);
    g_host_maps[p] = std::make_pair(base, len + kHuge);
    *out = p;
    return 0;
}

int cube_host_free(void* p)
{
    std::pair<void*, size_t> m;
    {
        std::lock_guard<std::mutex> lock(g_host_mu);
        auto it = g_host_maps.find(p);
        if (it == g_host_maps.end()) return CUBE_ERR_ARG;
        m = it->second;
        g_host_maps.erase(it);
    }
    cudaHostUnregister(p);
    munmap(m.first, m.second);
    return 0;
}

}  // extern "C"
