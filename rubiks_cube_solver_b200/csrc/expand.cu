// K3 -- ADI-style expansion and one-hot encoding (sm_100a).
//
// For every parent state: all A children in action order (cube_env.py:212-238),
// each child's one-hot network input (sim_state_to_state cube_env.py:132-152 ->
// getOP_3 py333.py:224-227 + pos_to_state_3 :235-246 for 3x3x3; py222 getOP and the
// loop at cube_env.py:141-147 for 2x2x2), its face-uniformity verdict (py333.py:229-233)
// and reward, written straight into the [N, A, D] batch the value/policy net
// consumes (bf16 by default; 1.0 is exact).  Optionally also the children's sticker
// rows (the MCTS leaf expansion, mcts.py:96-101) and the parent's own one-hot
// (mcts.py:92, `cube_encode`).
//
// The kernel is an HBM write stream: 2*D*A bytes per parent against S bytes read.
// A tile of 16 parents is staged in shared memory, its children are gathered in
// shared memory, every (row, slot) hash is reduced to one byte (the column of
// the single 1), and then all threads emit the one-hot rows as fully coalesced
// 16-byte streaming stores, deciding per vector which of its elements is 1.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include "cube_threads.cuh"
#include "cube_kernels.h"
#include "cube_launch.cuh"

namespace {

constexpr int kThreads = 256;
// parents per tile; a multiple of 16 keeps every stream 16-byte aligned.  2x2x2 parents are
// small (6 children of 24 bytes), so a tile takes 64 of them to keep all 256 threads busy.
template <int SIZE> struct ExpandTile { static constexpr int kParents = (SIZE == 3) ? 16 : 64; };

__host__ __device__ constexpr int round16(int x) { return (x + 15) & ~15; }

// Emit `n_seg` one-hot segments of width C (element stream = n_seg * C elements) starting at
// byte offset 0 of `dst`; col[s] = position of the 1 inside segment s, 255 = none.
// The stream length in bytes must be a multiple of 16.
template <int DTYPE, int C>
__device__ __forceinline__ void emit_onehot(uint8_t* __restrict__ dst, const uint8_t* col, int n_seg, int tid)
{
    constexpr int V = OneHot<DTYPE>::V;
    constexpr int kSegStep = (kThreads * V) / C, kOffStep = (kThreads * V) % C;   // advance per iteration
    const int n_vec = n_seg * C / V;
    int4* out = reinterpret_cast<int4*>(dst);
    int seg = (tid * V) / C;
    int off = tid * V - seg * C;
    for (int v = tid; v < n_vec; v += kThreads) {
        uint32_t w[4];
        onehot_vector_at<DTYPE, C>(seg, off, col, w);
        __stcs(out + v, make_int4((int)w[0], (int)w[1], (int)w[2], (int)w[3]));
        seg += kSegStep;
        off += kOffStep;
        if (off >= C) { off -= C; ++seg; }
    }
}

template <int SIZE, int DTYPE>
__global__ void __launch_bounds__(kThreads, 6)
expand_kernel(const uint8_t* __restrict__ states, long long n, uint8_t* __restrict__ children,
              uint8_t* __restrict__ child_onehot, uint8_t* __restrict__ parent_onehot,
              uint8_t* __restrict__ solved, float* __restrict__ reward,
              unsigned long long* __restrict__ counters, uint8_t* __restrict__ child_codes,
              uint8_t* __restrict__ parent_codes, int exact)
{
    using G = CubeGeom<SIZE>;
    constexpr int S = G::S, A = G::A, R = G::R, C = G::C;
    constexpr int ESIZE = OneHot<DTYPE>::ESIZE;
    constexpr int KEY = (R + 3) & ~3;                     // bytes of a code row: the R column indices, zero-padded to words
    constexpr int kParents = ExpandTile<SIZE>::kParents;
    constexpr int kRows = kParents * A;

    __shared__ __align__(16) uint8_t s_par[round16(kParents * S)];
    __shared__ __align__(16) uint8_t s_child[round16(kRows * S)];
    __shared__ uint8_t s_colc[kRows * R + 4];
    __shared__ uint8_t s_colp[kParents * R + 4];
    __shared__ uint8_t s_gather[A * S];
    __shared__ uint32_t s_def[R];
    __shared__ uint8_t s_lut[3][128];
    __shared__ unsigned int s_solved_count;

    const int tid = threadIdx.x;
    for (int i = tid; i < A * S; i += kThreads) {
        const int a = i / S, k = i - a * S;
        s_gather[i] = (SIZE == 3) ? kGather3[a * 56 + k] : kGather2[a * 24 + k];
    }
    // `exact`: the opt-in exact 3x3x3 encoding (un-mirrored slot 6, every corner rotation assigned); the
    // default is the reference's table as shipped.  2x2x2 has one encoding (py222's is a bijection).
    if (tid < R) s_def[tid] = (SIZE == 3) ? (exact ? kHashDef3x[tid] : kHashDef3[tid]) : kHashDef2[tid];
    if (tid < 128) {
        s_lut[0][tid] = (SIZE == 3) ? (exact ? kCornerCol3x[tid] : kCornerCol3[tid]) : kPieceCode2[tid];
        s_lut[1][tid] = (SIZE == 3) ? kEdgeCol3[tid] : 0;
    }
    if (tid == 0) s_solved_count = 0;
    const bool need_children = children || child_onehot || solved || reward || counters || child_codes;
    const bool need_parent_cols = parent_onehot || parent_codes;

    const long long n_tiles = (n + kParents - 1) / kParents;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long base = tile * kParents;
        const int cnt = (int)((n - base) < (long long)kParents ? (n - base) : (long long)kParents);
        const int rows = cnt * A;
        __syncthreads();
        {   // parents in (coalesced)
            const long long byte0 = base * S;              // multiple of 16
            const int nbytes = cnt * S;
            const int nvec = nbytes >> 4;
            const int4* src = reinterpret_cast<const int4*>(states + byte0);
            for (int i = tid; i < nvec; i += kThreads) reinterpret_cast<int4*>(s_par)[i] = __ldcs(src + i);
            for (int i = (nvec << 4) + tid; i < nbytes; i += kThreads) s_par[i] = states[byte0 + i];
        }
        if (SIZE == 2) {
            for (int i = tid; i < kRows * R; i += kThreads) s_colc[i] = 255;
            for (int i = tid; i < kParents * R; i += kThreads) s_colp[i] = 255;
        }
        __syncthreads();

        if (need_children) {
            // children[p][a][i] = parent[p][moveDefs[a][i]]: one sticker per lane, 64 (3x3x3) or 32
            // (2x2x2) lanes per row, so 4 / 8 rows are in flight
            constexpr int kLanes = (S > 32) ? 64 : 32;
            const int lane = tid & (kLanes - 1);
            if (lane < S) {
                for (int r = tid / kLanes; r < rows; r += kThreads / kLanes) {
                    const int p = r / A, a = r - p * A;
                    s_child[r * S + lane] = s_par[p * S + s_gather[a * S + lane]];
                }
            }
        }
        __syncthreads();

        // one-hot columns: child rows, then parent rows
        const int n_items = (need_children ? rows : 0) + (need_parent_cols ? cnt : 0);
        for (int it = tid; it < n_items * R; it += kThreads) {
            const int r = it / R, slot = it - r * R;
            const bool is_child = need_children && r < rows;
            const int rr = is_child ? r : r - (need_children ? rows : 0);
            const uint8_t* row = is_child ? s_child + rr * S : s_par + rr * S;
            uint8_t* colrow = is_child ? s_colc + rr * R : s_colp + rr * R;
            const uint32_t code = onehot_code<SIZE>(row, slot, s_def, s_lut[0], s_lut[1]);
            if (SIZE == 3) colrow[slot] = (uint8_t)code;
            else colrow[code & 0xfu] = (uint8_t)(3 * slot + (code >> 4));            // cube_env.py:145-147
        }

        // verdicts of the children
        if (need_children) {
            for (int r0 = 0; r0 < rows; r0 += kThreads) {     // warp-uniform trip count
                const int r = r0 + tid;
                bool ok = false;
                if (r < rows) {
                    ok = stickers_solved<SIZE>(s_child + r * S);
                    if (solved) solved[base * A + r] = ok ? 1 : 0;
                    if (reward) reward[base * A + r] = ok ? 1.0f : -1.0f;
                }
                const unsigned bal = __ballot_sync(0xffffffffu, ok);
                if ((tid & 31) == 0 && bal) atomicAdd(&s_solved_count, (unsigned)__popc(bal));
            }
        }
        __syncthreads();

        if (children) {
            const long long byte0 = base * A * S;          // multiple of 16 (kParents = 16)
            const int nbytes = rows * S;
            const int nvec = nbytes >> 4;
            int4* dst = reinterpret_cast<int4*>(children + byte0);
            for (int i = tid; i < nvec; i += kThreads) __stcs(dst + i, reinterpret_cast<const int4*>(s_child)[i]);
            for (int i = (nvec << 4) + tid; i < nbytes; i += kThreads) children[byte0 + i] = s_child[i];
        }
        // compact codes: the column of the single 1 of every one-hot row (what argmax over the row gives; a
        // 2x2x2 row without a 1 reads 0 like argmax), KEY bytes per state
        if (child_codes) {
            uint8_t* dst = child_codes + base * A * KEY;
            for (int i = tid; i < rows * KEY; i += kThreads) {
                const int r = i / KEY, k = i - r * KEY;
                const uint8_t c = k < R ? s_colc[r * R + k] : (uint8_t)0;
                dst[i] = c == 255 ? (uint8_t)0 : c;
            }
        }
        if (parent_codes) {
            uint8_t* dst = parent_codes + base * KEY;
            for (int i = tid; i < cnt * KEY; i += kThreads) {
                const int r = i / KEY, k = i - r * KEY;
                const uint8_t c = k < R ? s_colp[r * R + k] : (uint8_t)0;
                dst[i] = c == 255 ? (uint8_t)0 : c;
            }
        }
        if (child_onehot) {
            uint8_t* dst = child_onehot + base * A * (long long)(G::D * ESIZE);
            if ((rows * G::D * ESIZE) % 16 == 0) {
                emit_onehot<DTYPE, C>(dst, s_colc, rows * R, tid);
            } else {                                        // ragged last tile: element-wise
                for (int e = tid; e < rows * G::D; e += kThreads) {
                    const int seg = e / C, off = e - seg * C;
                    const bool one = s_colc[seg] == off;
                    if (DTYPE == 0) reinterpret_cast<uint16_t*>(dst)[e] = one ? 0x3f80 : 0;
                    else if (DTYPE == 1) reinterpret_cast<uint32_t*>(dst)[e] = one ? 0x3f800000u : 0u;
                    else dst[e] = one ? 1 : 0;
                }
            }
        }
        if (parent_onehot) {
            uint8_t* dst = parent_onehot + base * (long long)(G::D * ESIZE);
            if ((cnt * G::D * ESIZE) % 16 == 0) {
                emit_onehot<DTYPE, C>(dst, s_colp, cnt * R, tid);
            } else {
                for (int e = tid; e < cnt * G::D; e += kThreads) {
                    const int seg = e / C, off = e - seg * C;
                    const bool one = s_colp[seg] == off;
                    if (DTYPE == 0) reinterpret_cast<uint16_t*>(dst)[e] = one ? 0x3f80 : 0;
                    else if (DTYPE == 1) reinterpret_cast<uint32_t*>(dst)[e] = one ? 0x3f800000u : 0u;
                    else dst[e] = one ? 1 : 0;
                }
            }
        }
    }
    __syncthreads();
    if (tid == 0 && counters) {
        if (s_solved_count) atomicAdd(&counters[0], (unsigned long long)s_solved_count);
        if (blockIdx.x == 0) atomicAdd(&counters[1], (unsigned long long)n * A);
    }
}

// encode only (`cube_encode`, sim_state_to_state cube_env.py:132-152): no children to build, so a
// tile is 128 rows -- enough output (123 KB for 3x3x3 bf16) per CTA to amortise the table loads
constexpr int kEncodeRows = 128;

template <int SIZE, int DTYPE>
__global__ void __launch_bounds__(kThreads, 6)
encode_kernel(const uint8_t* __restrict__ states, long long n, uint8_t* __restrict__ onehot, int exact)
{
    using G = CubeGeom<SIZE>;
    constexpr int S = G::S, R = G::R, C = G::C, ESIZE = OneHot<DTYPE>::ESIZE;
    __shared__ __align__(16) uint8_t s_rows[round16(kEncodeRows * S)];
    __shared__ uint8_t s_col[kEncodeRows * R + 4];
    __shared__ uint32_t s_def[R];
    __shared__ uint8_t s_lut[2][128];

    const int tid = threadIdx.x;
    if (tid < R) s_def[tid] = (SIZE == 3) ? (exact ? kHashDef3x[tid] : kHashDef3[tid]) : kHashDef2[tid];
    if (tid < 128) {
        s_lut[0][tid] = (SIZE == 3) ? (exact ? kCornerCol3x[tid] : kCornerCol3[tid]) : kPieceCode2[tid];
        s_lut[1][tid] = (SIZE == 3) ? kEdgeCol3[tid] : 0;
    }
    const long long base = (long long)blockIdx.x * kEncodeRows;
    const int cnt = (int)((n - base) < (long long)kEncodeRows ? (n - base) : (long long)kEncodeRows);
    {
        const long long byte0 = base * S;                  // multiple of 16
        const int nbytes = cnt * S;
        const int nvec = nbytes >> 4;
        const int4* src = reinterpret_cast<const int4*>(states + byte0);
        for (int i = tid; i < nvec; i += kThreads) reinterpret_cast<int4*>(s_rows)[i] = __ldcs(src + i);
        for (int i = (nvec << 4) + tid; i < nbytes; i += kThreads) s_rows[i] = states[byte0 + i];
    }
    if (SIZE == 2) for (int i = tid; i < kEncodeRows * R; i += kThreads) s_col[i] = 255;
    __syncthreads();
    for (int it = tid; it < cnt * R; it += kThreads) {
        const int r = it / R, slot = it - r * R;
        const uint32_t code = onehot_code<SIZE>(s_rows + r * S, slot, s_def, s_lut[0], s_lut[1]);
        if (SIZE == 3) s_col[it] = (uint8_t)code;
        else s_col[r * R + (code & 0xfu)] = (uint8_t)(3 * slot + (code >> 4));
    }
    __syncthreads();
    uint8_t* dst = onehot + base * (long long)(G::D * ESIZE);
    if ((cnt * G::D * ESIZE) % 16 == 0) {
        emit_onehot<DTYPE, C>(dst, s_col, cnt * R, tid);
    } else {
        for (int e = tid; e < cnt * G::D; e += kThreads) {
            const int seg = e / C, off = e - seg * C;
            const bool one = s_col[seg] == off;
            if (DTYPE == 0) reinterpret_cast<uint16_t*>(dst)[e] = one ? 0x3f80 : 0;
            else if (DTYPE == 1) reinterpret_cast<uint32_t*>(dst)[e] = one ? 0x3f800000u : 0u;
            else dst[e] = one ? 1 : 0;
        }
    }
}

template <int SIZE, int DTYPE>
int launch_one(const uint8_t* states, long long n, uint8_t* children, void* child_onehot, void* parent_onehot,
               uint8_t* solved, float* reward, unsigned long long* counters, cudaStream_t stream,
               uint8_t* child_codes = nullptr, uint8_t* parent_codes = nullptr, int exact = 0)
{
    if (!children && !child_onehot && !solved && !reward && !counters && !child_codes && !parent_codes) {
        if (!parent_onehot) return 0;
        const long long tiles = (n + kEncodeRows - 1) / kEncodeRows;
        encode_kernel<SIZE, DTYPE><<<(unsigned)tiles, kThreads, 0, stream>>>(states, n, (uint8_t*)parent_onehot, exact);
        return (int)cudaGetLastError();
    }
    auto kern = expand_kernel<SIZE, DTYPE>;
    constexpr int kParents = ExpandTile<SIZE>::kParents;
    const long long n_tiles = (n + kParents - 1) / kParents;
    // one tile per CTA (the in-kernel tile loop only runs more than once for gigantic batches):
    // the phases of a tile are separated by barriers, so overlap comes from having many CTAs
    // per SM in different phases, scheduled by the hardware
    const long long grid = n_tiles < 0x7fffffffLL ? n_tiles : 0x7fffffffLL;
    cube::prefer_max_shared(kern);
    kern<<<(unsigned)grid, kThreads, 0, stream>>>(states, n, children, (uint8_t*)child_onehot,
                                                  (uint8_t*)parent_onehot, solved, reward, counters, child_codes,
                                                  parent_codes, exact);
    return (int)cudaGetLastError();
}

}  // namespace

namespace cube {

int launch_expand(int size, const uint8_t* states, long long n, uint8_t* children, void* child_onehot,
                  void* parent_onehot, int dtype, uint8_t* solved, float* reward,
                  unsigned long long* counters, cudaStream_t stream, int encoding)
{
    if (n == 0) return 0;
    const int exact = (size == 3 && encoding == CUBE_ENCODING_EXACT) ? 1 : 0;
    // 2x2x2: whole tiles of parents through a dedicated kernel, the remainder through the generic kernel below.
    // The ADI shape takes the image kernel K3c (f32: the generic kernel already streams at the HBM peak, 1.03
    // measured; K3c with 8 parents per CTA reached 0.98), the MCTS leaf shape (BASELINE config 5) the
    // register-resident kernel.
    long long done = 0;
    if (size == 2 && child_onehot && dtype != 1)
        done = launch_leaf2_children(states, n, children, child_onehot, parent_onehot, dtype, solved, reward, counters,
                                     stream);
    else if (size == 2 && !child_onehot && (children || parent_onehot))
        done = launch_leaf2(states, n, children, parent_onehot, dtype, solved, reward, counters, stream);
    if (done < 0) return (int)-done;
    if (done == n) return 0;
    if (done > 0) {                                          // the generic kernel takes the parents after the tiles
        using G = CubeGeom<2>;
        const long long es = dtype == 0 ? 2 : (dtype == 1 ? 4 : 1);
        auto skip = [done](auto* p, long long per_parent) { return p ? p + done * per_parent : p; };
        states += done * G::S;
        n -= done;
        children = skip(children, G::A * G::S);
        child_onehot = skip(static_cast<uint8_t*>(child_onehot), G::A * G::D * es);
        parent_onehot = skip(static_cast<uint8_t*>(parent_onehot), G::D * es);
        solved = skip(solved, G::A);
        reward = skip(reward, G::A);
    }
#define CUBE_EXPAND_CASE(SZ, DT)                                                                         \
    if (size == SZ && dtype == DT)                                                                       \
        return launch_one<SZ, DT>(states, n, children, child_onehot, parent_onehot, solved, reward,      \
                                  counters, stream, nullptr, nullptr, exact);
    CUBE_EXPAND_CASE(3, 0) CUBE_EXPAND_CASE(3, 1) CUBE_EXPAND_CASE(3, 2)
    CUBE_EXPAND_CASE(2, 0) CUBE_EXPAND_CASE(2, 1) CUBE_EXPAND_CASE(2, 2)
#undef CUBE_EXPAND_CASE
    return CUBE_ERR_ARG;
}

// expansion with compact codes instead of the children's one-hot rows (the MCTS tree's keys): always the
// generic kernel, whose column bytes ARE the codes
int launch_expand_codes(int size, const uint8_t* states, long long n, uint8_t* children, uint8_t* child_codes,
                        uint8_t* parent_codes, void* parent_onehot, int dtype, uint8_t* solved, float* reward,
                        unsigned long long* counters, cudaStream_t stream, int encoding)
{
    if (n == 0) return 0;
    const int exact = (size == 3 && encoding == CUBE_ENCODING_EXACT) ? 1 : 0;
#define CUBE_EXPAND_CASE(SZ, DT)                                                                         \
    if (size == SZ && dtype == DT)                                                                       \
        return launch_one<SZ, DT>(states, n, children, nullptr, parent_onehot, solved, reward, counters,  \
                                  stream, child_codes, parent_codes, exact);
    CUBE_EXPAND_CASE(3, 0) CUBE_EXPAND_CASE(3, 1) CUBE_EXPAND_CASE(3, 2)
    CUBE_EXPAND_CASE(2, 0) CUBE_EXPAND_CASE(2, 1) CUBE_EXPAND_CASE(2, 2)
#undef CUBE_EXPAND_CASE
    return CUBE_ERR_ARG;
}

}  // namespace cube
