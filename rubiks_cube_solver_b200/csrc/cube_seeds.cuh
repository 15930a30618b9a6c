// K0's per-seed draw: the move indices reset(seed, k) draws (cube_env.py:62-65),
//   np.random.seed(seed); np.random.randint(A, size=k)  ==  np.random.RandomState(seed).randint(A, size=k),
// one row per thread.  Device code under nvcc (seeds.cu), plain C++ under a host compiler, so that the test-only
// emulation harness (tests/host_emul/seeds_emul.cpp) runs exactly this code on the CPU.
//
// NumPy's legacy generator is MT19937 seeded by init_genrand (mt[0] = seed, mt[j] = 1812433253 *
// (mt[j-1] ^ mt[j-1] >> 30) + j) and randint(A) draws 32-bit outputs, masks them with the smallest
// 2^b - 1 >= A - 1 and rejects values > A - 1 (numpy/random/_bounded_integers: masked rejection).
//
// Fast path: output i < 227 of a freshly seeded generator only needs mt[i], mt[i+1] and mt[i+397] of the SEED
// state, and those follow from a one-word recurrence -- so a thread keeps two running words (one at i, one 397
// ahead) and never materialises the 624-word state.  With acceptance 3/4 (A = 12) or 6/8 (A = 6), 227 raw draws
// hold fewer than 128 accepted values for about one seed in 3e9: among all 2^32 seeds, 2103926524 and 3830291768
// for randint(12) and 3969546545 for randint(6).
// Slow path (seed_row_slow): a row still short after 227 draws materialises the seed state, runs the full twist
// and goes on drawing from output 227 exactly as NumPy does (twisting again after output 623).  It is a separate,
// never-inlined function so that the fast path keeps its registers and instructions; its 2.5 KB state array is
// local memory that only such rows touch.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define SEED_FN __device__ __forceinline__
#define SEED_COLD_FN __device__ __noinline__
#else
#define SEED_FN inline
#define SEED_COLD_FN inline
#endif

constexpr int kSeedFastDraws = 227;            // outputs of the first twist that need no materialised state
constexpr int kMtWords = 624;
constexpr int kMtShift = 397;

// randint(A)'s rejection mask: the smallest 2^b - 1 >= max_value (= A - 1)
inline uint32_t seed_mask(uint32_t max_value)
{
    uint32_t mask = max_value;
    mask |= mask >> 1; mask |= mask >> 2; mask |= mask >> 4; mask |= mask >> 8; mask |= mask >> 16;
    return mask;
}

// x >> K on the FMA pipe (IMAD.HI) instead of the ALU pipe (SHF): the recurrence and the tempering are
// shift / xor / multiply chains.  Measured: 8 Mi seeds x depth 30 take 1.3 ms either way (3 390 warp
// instructions per 32 seeds, ALU pipe 63 %, issue 59 %, `math_pipe_throttle` and `dispatch_stall` on top:
// profiles/r01_k0_seeded_moves_ncu_summary.json) -- the 397 sequential seed-state steps and ~50 draw
// iterations of ~35 instructions are what the generator costs (1.22 ms after the row stores stopped
// rebuilding their address per draw); the fused scramble behind it takes 0.18 ms.
template <int K>
SEED_FN uint32_t shr(uint32_t x)
{
#if defined(__CUDA_ARCH__)
    return __umulhi(x, 1u << (32 - K));
#else
    return x >> K;
#endif
}

SEED_FN uint32_t mt_next_seed_word(uint32_t prev, uint32_t j)
{
    return 1812433253u * (prev ^ shr<30>(prev)) + j;
}

// new mt[i] from mt[i], mt[i+1] and mt[i+397]
SEED_FN uint32_t mt_twist_word(uint32_t cur, uint32_t next, uint32_t far)
{
    const uint32_t y = (cur & 0x80000000u) | (next & 0x7fffffffu);
    return far ^ shr<1>(y) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
}

SEED_FN uint32_t mt_temper(uint32_t v)
{
    v ^= shr<11>(v);
    v ^= (v << 7) & 0x9d2c5680u;
    v ^= (v << 15) & 0xefc60000u;
    v ^= shr<18>(v);
    return v;
}

#if defined(__CUDACC__)
// j as a constant-bank operand of the multiply-add (IMAD r, g, M, c[j]): with the loop index in a register
// an unrolled step needs an extra ALU add for "+ j"
struct SeedIndex { uint32_t v[400]; };
constexpr SeedIndex make_seed_index()
{
    SeedIndex t{};
    for (int j = 0; j < 400; ++j) t.v[j] = (uint32_t)j;
    return t;
}
__constant__ SeedIndex kSeedIndex = make_seed_index();
#define SEED_INDEX(j) kSeedIndex.v[j]
#else
#define SEED_INDEX(j) ((uint32_t)(j))
#endif

// the full twist, in place and in MT19937's order: words past 226 read the new values of words 0..226
SEED_FN void mt_twist(uint32_t* mt)
{
    for (int k = 0; k < kMtWords; ++k) {
        const int k1 = k + 1 < kMtWords ? k + 1 : 0, kf = k + kMtShift < kMtWords ? k + kMtShift : k + kMtShift - kMtWords;
        mt[k] = mt_twist_word(mt[k], mt[k1], mt[kf]);
    }
}

// The rest of a row whose first 227 draws fell short: `row` continues where the fast path stopped.
// Row: full() -- the row has `depth` entries; put(v) -- append one.
template <class Row>
SEED_COLD_FN void seed_row_slow(uint32_t seed, uint32_t max_value, uint32_t mask, Row row)
{
    uint32_t mt[kMtWords];
    mt[0] = seed;
    for (int j = 1; j < kMtWords; ++j) mt[j] = mt_next_seed_word(mt[j - 1], (uint32_t)j);
    mt_twist(mt);                                        // a freshly seeded generator twists before its first output
    for (int pos = kSeedFastDraws; !row.full(); ++pos) {
        if (pos == kMtWords) {
            mt_twist(mt);
            pos = 0;
        }
        const uint32_t val = mt_temper(mt[pos]) & mask;
        if (val <= max_value) row.put(val);
    }
}

// One row: randint(max_value + 1, size=depth) of `seed` into `row`.  Returns whether the slow path ran.
template <class Row>
SEED_FN bool seed_row(uint32_t seed, uint32_t max_value, uint32_t mask, Row row)
{
    uint32_t z = seed;
#pragma unroll
    for (int j = 1; j <= kMtShift; ++j) z = mt_next_seed_word(z, SEED_INDEX(j));   // mt[397]: 3 instructions per step
    uint32_t x = seed, xn = mt_next_seed_word(seed, 1), idx = 0;                  // mt[0], mt[1]
    while (!row.full() && idx < kSeedFastDraws) {
        const uint32_t v = mt_temper(mt_twist_word(x, xn, z));                   // output idx of the first twist
        ++idx;
        x = xn;
        xn = mt_next_seed_word(xn, idx + 1);
        z = mt_next_seed_word(z, idx + kMtShift);                                 // only used while idx + 397 <= 623
        const uint32_t val = v & mask;
        if (val <= max_value) row.put(val);
    }
    if (row.full()) return false;
    seed_row_slow(seed, max_value, mask, row);
    return true;
}
