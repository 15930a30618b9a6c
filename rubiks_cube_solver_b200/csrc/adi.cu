// K4 -- ADI target assembly (sm_100a): the tail of get_target_value (cube_env.py:239-252) for a
// batch of parents whose children were produced by cube_expand and valued by the caller's net.
//   first solved child a  ->  (target_value, target_policy) = (1.0, a)            cube_env.py:217-220
//   otherwise                 value_a = V(child_a) + (-1.0)   in float32          cube_env.py:243
//                             (target_value, target_policy) = max / first argmax  cube_env.py:244-245
//   error = |V(state) - target_value| * scramble_count ** (-temperature)  in float64 (cube_env.py:247-251)
// The weight k ** (-T) is looked up in a table the HOST computes (k = 0 .. table_len-1): Python's
// float power is the C library's pow, CUDA's pow is not correctly rounded, and the replay buffer's
// priorities are compared bit for bit in the parity tests.
// One thread per parent; the A child values are read as 16-byte vectors (A*4 = 48 / 24 bytes).
#include <cuda_runtime.h>
#include "cube_kernels.h"
#include "cube_launch.cuh"

namespace {

template <int A>
__global__ void __launch_bounds__(256)
adi_targets_kernel(const float* __restrict__ child_values, const uint8_t* __restrict__ child_solved,
                   const float* __restrict__ parent_values, const int* __restrict__ scramble_count,
                   const double* __restrict__ weight, int table_len, long long n, float* __restrict__ target_value,
                   int* __restrict__ target_policy, double* __restrict__ error)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        float v[A];
        if (A == 12) {
            const float4* p = reinterpret_cast<const float4*>(child_values + i * A);      // 48-byte rows: 16-byte aligned
#pragma unroll
            for (int j = 0; j < 3; ++j) { const float4 q = __ldcs(p + j); v[4 * j] = q.x; v[4 * j + 1] = q.y; v[4 * j + 2] = q.z; v[4 * j + 3] = q.w; }
        } else {
            const float2* p = reinterpret_cast<const float2*>(child_values + i * A);      // 24-byte rows: 8-byte aligned
#pragma unroll
            for (int j = 0; j < A / 2; ++j) { const float2 q = __ldcs(p + j); v[2 * j] = q.x; v[2 * j + 1] = q.y; }
        }
        int first_solved = A;
#pragma unroll
        for (int a = A - 1; a >= 0; --a) first_solved = child_solved[i * A + a] ? a : first_solved;
        float best = __fadd_rn(v[0], -1.0f);
        int arg = 0;
#pragma unroll
        for (int a = 1; a < A; ++a) {
            const float x = __fadd_rn(v[a], -1.0f);
            if (x > best) { best = x; arg = a; }                     // strict: the first maximum wins (torch.max)
        }
        if (first_solved < A) { best = 1.0f; arg = first_solved; }
        const int k = scramble_count[i];
        const double w = (k >= 0 && k < table_len) ? weight[k] : 0.0;
        target_value[i] = best;
        target_policy[i] = arg;
        error[i] = fabs((double)parent_values[i] - (double)best) * w;
    }
}

}  // namespace

namespace cube {

int launch_adi_targets(int size, const float* child_values, const uint8_t* child_solved, const float* parent_values,
                       const int* scramble_count, const double* weight, int table_len, long long n,
                       float* target_value, int* target_policy, double* error, cudaStream_t stream)
{
    if (n == 0) return 0;
    long long blocks = (n + 255) / 256;
    const long long cap = (long long)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    if (size == 3)
        adi_targets_kernel<12><<<(unsigned)blocks, 256, 0, stream>>>(child_values, child_solved, parent_values,
                                                                    scramble_count, weight, table_len, n, target_value,
                                                                    target_policy, error);
    else
        adi_targets_kernel<6><<<(unsigned)blocks, 256, 0, stream>>>(child_values, child_solved, parent_values,
                                                                   scramble_count, weight, table_len, n, target_value,
                                                                   target_policy, error);
    return (int)cudaGetLastError();
}

}  // namespace cube
