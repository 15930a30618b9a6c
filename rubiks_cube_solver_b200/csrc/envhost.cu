// Single-cube host front end: what the reference's per-cube callers do through the drop-in CubeEnv
// (cube_env.py:56-111: reset, step, get_obs -- train.py:155, :186-191, mcts.py:80, test.py:123).
//
// One call = one cube, host buffers in and out, ONE launch, ONE stream synchronisation and NO copy calls:
// the handle owns a page of mapped pinned memory that the kernel reads and writes directly over PCIe
// (sticker row and moves in; sticker row, solved flag and the uint8 one-hot out).  Round 2: step, reset and
// encode are each ONE launch of a dedicated single-CTA kernel (`env_cube_kernel`: the moves applied as
// sticker gathers in shared memory, the verdict, the one-hot rows assembled in shared memory and written back
// with 16-byte stores) -- round 1 went through the batch kernels (a 12-child expansion of which the host kept
// one child: 6.4 KB over PCIe per step; reset and encode were two launches).  The torch-level path (upload,
// two kernels, three downloads with their synchronisations) took ~120 us per step; the reference's own NumPy
// step takes ~25 us on the same host.
#include <atomic>
#include <cstring>
#include <cuda_runtime.h>
#include <new>

#include "../../include/cube_b200.h"
#include "cube_threads.cuh"
#include "cube_kernels.h"
#include "cube_launch.cuh"

struct cube_env_host {
    int cube_size, max_depth;
    uint8_t* pin;        // mapped pinned page, laid out below
    uint8_t* dev;        // the same page as the device sees it
    int off_moves, off_out, off_solved, off_onehot, bytes;
    int off_flag;        // completion flag of the last launch (the kernel writes `seq` there when it is done)
    uint32_t seq;
    int off_children, off_child_onehot, off_child_solved;            // [A, S], [A, D] uint8, [A]
};

namespace {

inline int round16(int x) { return (x + 15) & ~15; }

const bool g_spin = cube::env_flag("CUBE_ENV_SPIN", true);     // A/B switch

// One cube: `depth` moves (indices >= A are no-ops, like the batch kernels' identity rows) applied to the row at
// `in` (or to the solved cube when in == nullptr), then the verdict and the uint8 one-hot rows.  All pointers are
// in the handle's mapped pinned page.  64 threads: one per sticker for the gathers, one per one-hot row.
template <int SIZE>
__global__ void __launch_bounds__(64)
env_cube_kernel(const uint8_t* in, const uint8_t* moves, int depth, uint8_t* out_row, uint8_t* solved, uint8_t* onehot,
                volatile uint32_t* done_flag, uint32_t seq)
{
    using G = CubeGeom<SIZE>;
    constexpr int S = G::S, A = G::A, R = G::R, C = G::C, D = G::D, GS = (SIZE == 3) ? 56 : 24;
    __shared__ uint8_t s_row[2][64];
    __shared__ uint8_t s_col[R + 4];
    __shared__ __align__(16) uint8_t s_oh[(D + 15) & ~15];
    __shared__ uint8_t s_moves[64];
    const int t = threadIdx.x;
    if (t < S) s_row[0][t] = in ? in[t] : (uint8_t)(t / (S / 6));
    int cur = 0;
    for (int k0 = 0; k0 < depth; k0 += 64) {                          // the moves arrive 64 at a time
        __syncthreads();
        if (k0 + t < depth) s_moves[t] = moves[k0 + t];
        __syncthreads();
        const int cnt = depth - k0 < 64 ? depth - k0 : 64;
        for (int k = 0; k < cnt; ++k) {
            const uint32_t m = s_moves[k];
            if (t < S) s_row[cur ^ 1][t] = s_row[cur][m < (uint32_t)A ? ((SIZE == 3) ? kGather3 : kGather2)[m * GS + t] : t];
            cur ^= 1;
            __syncthreads();
        }
    }
    __syncthreads();
    const uint8_t* row = s_row[cur];
    if (out_row && t < S) out_row[t] = row[t];
    if (solved && t == 0) *solved = stickers_solved<SIZE>(row) ? 1 : 0;
    if (onehot) {
        for (int i = t; i < (int)sizeof(s_oh) / 4; i += 64) reinterpret_cast<uint32_t*>(s_oh)[i] = 0u;
        __syncthreads();
        if (t < R) {
            const uint32_t code = onehot_code<SIZE>(row, t, (SIZE == 3) ? kHashDef3 : kHashDef2,
                                                    (SIZE == 3) ? kCornerCol3 : kPieceCode2, kEdgeCol3);
            if (SIZE == 3) s_col[t] = (uint8_t)code;
            // one 1 per position, as the reference's loop sets it (cube_env.py:145-147): a row that names a cubelet
            // twice gets two 1s in that cubelet's one-hot row
            else s_oh[(code & 0xfu) * C + 3 * t + (code >> 4)] = 1;
        }
        __syncthreads();
        if (SIZE == 3 && t < R && s_col[t] < C) s_oh[t * C + s_col[t]] = 1;
        __syncthreads();
        for (int i = t; i < D / 16; i += 64) reinterpret_cast<int4*>(onehot)[i] = reinterpret_cast<const int4*>(s_oh)[i];
        for (int i = (D / 16) * 16 + t; i < D; i += 64) onehot[i] = s_oh[i];
    }
    // completion flag in the page: the host polls it instead of paying the driver's synchronisation path
    __threadfence_system();
    __syncthreads();
    if (t == 0) *done_flag = seq;
}

int launch_env_cube(int size, const uint8_t* in, const uint8_t* moves, int depth, uint8_t* out_row, uint8_t* solved,
                    uint8_t* onehot, volatile uint32_t* done_flag, uint32_t seq, cudaStream_t stream)
{
    if (size == 3) env_cube_kernel<3><<<1, 64, 0, stream>>>(in, moves, depth, out_row, solved, onehot, done_flag, seq);
    else env_cube_kernel<2><<<1, 64, 0, stream>>>(in, moves, depth, out_row, solved, onehot, done_flag, seq);
    return (int)cudaGetLastError();
}

}  // namespace

extern "C" {

int cube_env_host_create(int cube_size, int max_depth, cube_env_host** out)
{
    if (cube_size != 2 && cube_size != 3) return CUBE_ERR_SIZE;
    if (!out || max_depth < 1 || max_depth > 4096) return CUBE_ERR_ARG;
    cube_env_host* h = new (std::nothrow) cube_env_host();
    if (!h) return (int)cudaErrorMemoryAllocation;
    const int S = cube_size == 3 ? 54 : 24, D = cube_size == 3 ? 480 : 147;
    h->cube_size = cube_size;
    h->max_depth = max_depth;
    h->off_moves = round16(S);
    h->off_out = h->off_moves + round16(max_depth);
    h->off_solved = h->off_out + round16(S);
    h->off_onehot = h->off_solved + 16;
    const int A = cube_size == 3 ? 12 : 6;
    h->off_children = h->off_onehot + round16(D);
    h->off_child_onehot = h->off_children + round16(A * S);
    h->off_child_solved = h->off_child_onehot + round16(A * D);
    h->off_flag = h->off_child_solved + 16;
    h->bytes = h->off_flag + 16;
    h->seq = 0;
    void* p = nullptr;
    cudaError_t e = cudaHostAlloc(&p, (size_t)h->bytes, cudaHostAllocMapped | cudaHostAllocPortable);
    if (e != cudaSuccess) { delete h; return (int)e; }
    h->pin = static_cast<uint8_t*>(p);
    memset(h->pin, 0, (size_t)h->bytes);
    void* d = nullptr;
    e = cudaHostGetDevicePointer(&d, p, 0);
    if (e != cudaSuccess) { cudaFreeHost(p); delete h; return (int)e; }
    h->dev = static_cast<uint8_t*>(d);
    *out = h;
    return CUBE_OK;
}

int cube_env_host_destroy(cube_env_host* h)
{
    if (!h) return CUBE_OK;
    if (h->pin) cudaFreeHost(h->pin);
    delete h;
    return CUBE_OK;
}

// one launch, one synchronisation, then the results out of the page
static int run_one(cube_env_host* h, bool from_row, int depth, uint8_t* stickers_out_host, uint8_t* onehot_u8_host,
                   int* solved_host, cudaStream_t stream)
{
    const int S = h->cube_size == 3 ? 54 : 24, D = h->cube_size == 3 ? 480 : 147;
    const uint32_t seq = ++h->seq;
    volatile uint32_t* flag = reinterpret_cast<volatile uint32_t*>(h->pin + h->off_flag);
    const int rc = launch_env_cube(h->cube_size, from_row ? h->dev : nullptr, h->dev + h->off_moves, depth,
                                   stickers_out_host ? h->dev + h->off_out : nullptr, solved_host ? h->dev + h->off_solved : nullptr,
                                   onehot_u8_host ? h->dev + h->off_onehot : nullptr,
                                   reinterpret_cast<volatile uint32_t*>(h->dev + h->off_flag), seq, stream);
    if (rc) return rc;
    // The kernel's last act is to write `seq` into the page (after a system-wide fence): a short spin on it sees
    // the result a few microseconds before cudaStreamSynchronize would return.  A kernel that never gets there
    // (a fault, a stream blocked by other work) falls through to the synchronisation, which also reports errors.
    bool seen = false;
    if (g_spin) {
        for (int i = 0; i < 20000 && !(seen = (*flag == seq)); ++i) {
#if defined(__x86_64__)
            __builtin_ia32_pause();
#endif
        }
    }
    if (!seen) {
        const cudaError_t e = cudaStreamSynchronize(stream);
        if (e != cudaSuccess) return (int)e;
    }
    std::atomic_thread_fence(std::memory_order_acquire);
    if (stickers_out_host) memcpy(stickers_out_host, h->pin + h->off_out, (size_t)S);
    if (onehot_u8_host) memcpy(onehot_u8_host, h->pin + h->off_onehot, (size_t)D);
    if (solved_host) *solved_host = h->pin[h->off_solved] != 0;
    return CUBE_OK;
}

int cube_env_host_step(cube_env_host* h, const uint8_t* stickers_host, int action, uint8_t* stickers_out_host,
                       uint8_t* onehot_u8_host, int* solved_host, void* stream)
{
    if (!h || !stickers_host || action < 0 || action > 255) return CUBE_ERR_ARG;
    memcpy(h->pin, stickers_host, (size_t)(h->cube_size == 3 ? 54 : 24));
    h->pin[h->off_moves] = (uint8_t)action;                           // A..255: no move, like CUBE_NOOP
    return run_one(h, true, 1, stickers_out_host, onehot_u8_host, solved_host, (cudaStream_t)stream);
}

int cube_env_host_scramble(cube_env_host* h, const uint8_t* moves_host, int depth, uint8_t* stickers_out_host,
                           uint8_t* onehot_u8_host, int* solved_host, void* stream)
{
    if (!h || depth < 0 || depth > h->max_depth || (depth > 0 && !moves_host)) return CUBE_ERR_ARG;
    if (depth > 0) memcpy(h->pin + h->off_moves, moves_host, (size_t)depth);
    return run_one(h, false, depth, stickers_out_host, onehot_u8_host, solved_host, (cudaStream_t)stream);
}

int cube_env_host_encode(cube_env_host* h, const uint8_t* stickers_host, uint8_t* onehot_u8_host, void* stream)
{
    if (!h || !stickers_host || !onehot_u8_host) return CUBE_ERR_ARG;
    memcpy(h->pin, stickers_host, (size_t)(h->cube_size == 3 ? 54 : 24));
    return run_one(h, true, 0, nullptr, onehot_u8_host, nullptr, (cudaStream_t)stream);
}

}  // extern "C"
