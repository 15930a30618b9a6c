// Internal launchers behind the C ABI (include/cube_b200.h).  All pointers are
// device pointers, already validated by abi.cu; every launcher returns 0 or a
// cudaError_t and never synchronises.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "../../include/cube_b200.h"

// counters layout (uint64[4], device): [0] += solved outputs, [1] += outputs written,
// [2] += out-of-range actions seen by cube_validate_actions, [3] += seeded rows that took the slow path of
// cube_moves_from_seeds
namespace cube {

// `last` (n action bytes or null): one more face turn per instance after the `depth` moves (cube_scramble_step)
int launch_scramble(int size, const uint8_t* moves, long long n, int depth, uint8_t* states_out,
                    uint8_t* solved, float* reward, unsigned long long* counters, cudaStream_t stream,
                    const uint8_t* last = nullptr);

// every prefix of every scramble, cube-major: states_out[i, k, :] = row after moves[i, 0..k]; solved [n, depth] or null.
// depth <= prefix_max_depth(size) (one tile image of 32 cubes must fit in shared memory), else CUBE_ERR_ARG
int launch_prefixes(int size, const uint8_t* moves, long long n, int depth, uint8_t* states_out, uint8_t* solved,
                    unsigned long long* counters, cudaStream_t stream);
int prefix_max_depth(int size);

// depth moves applied to resident sticker rows (depth = 1: the reference's step)
int launch_walk(int size, const uint8_t* states_in, const uint8_t* moves, long long n, int depth,
                uint8_t* states_out, uint8_t* solved, float* reward, unsigned long long* counters,
                cudaStream_t stream);

int launch_solved(int size, const uint8_t* states, long long n, uint8_t* solved, float* reward,
                  unsigned long long* counters, cudaStream_t stream);

// dtype: 0 = bf16, 1 = f32, 2 = u8.  Any of children / child_onehot / parent_onehot / solved /
// reward may be null.
int launch_expand(int size, const uint8_t* states, long long n, uint8_t* children, void* child_onehot,
                  void* parent_onehot, int dtype, uint8_t* solved, float* reward,
                  unsigned long long* counters, cudaStream_t stream, int encoding = CUBE_ENCODING_REFERENCE);

// the same expansion with compact codes (column of the 1 of every one-hot row, (R + 3) & ~3 bytes per state,
// zero-padded) for the children and / or the parents instead of the children's one-hot rows
int launch_expand_codes(int size, const uint8_t* states, long long n, uint8_t* children, uint8_t* child_codes,
                        uint8_t* parent_codes, void* parent_onehot, int dtype, uint8_t* solved, float* reward,
                        unsigned long long* counters, cudaStream_t stream, int encoding = CUBE_ENCODING_REFERENCE);

int launch_validate(int size, const uint8_t* actions, long long count, unsigned long long* counters,
                    cudaStream_t stream);

// 2x2x2 leaf expansion (children + parent one-hot, no child one-hot): handles the leading
// multiple-of-tile parents and returns how many, or -cudaError
long long launch_leaf2(const uint8_t* states, long long n, uint8_t* children, void* parent_onehot, int dtype,
                       uint8_t* solved, float* reward, unsigned long long* counters, cudaStream_t stream);

// moves[i, :] = np.random.RandomState(seeds[i]).randint(A, size=depth) (cube_env.py:62-65); depth <= 128
int launch_seeded_moves(int size, const uint32_t* seeds, long long n, int depth, uint8_t* moves,
                        unsigned long long* counters, cudaStream_t stream);

// ADI targets (cube_env.py:239-252) from child values / solved flags; weight[k] = k ** (-temperature)
int launch_adi_targets(int size, const float* child_values, const uint8_t* child_solved, const float* parent_values,
                       const int* scramble_count, const double* weight, int table_len, long long n,
                       float* target_value, int* target_policy, double* error, cudaStream_t stream);

// the same with the children's one-hot rows (the 2x2x2 ADI shape): leading whole tiles, or -cudaError
long long launch_leaf2_children(const uint8_t* states, long long n, uint8_t* children, void* child_onehot,
                                void* parent_onehot, int dtype, uint8_t* solved, float* reward,
                                unsigned long long* counters, cudaStream_t stream);

// batched MCTS (mcts.py:17-154): traverse all trees to their leaves / insert the expanded leaves,
// back-propagate and test for solved children
int launch_mcts_traverse(int size, const cube_mcts_tree_t& t, float cpuct, int virtual_loss, cudaStream_t stream);
int launch_mcts_update(int size, const cube_mcts_tree_t& t, const uint8_t* leaf_key, const uint8_t* child_key_new,
                       const uint8_t* child_done_new, const float* value, const float* policy, float value_min,
                       int sim_index, int8_t* actions_out, int* n_actions, int* n_sims, int* n_active, cudaStream_t stream);

int launch_decode2(const void* onehot, int dtype, long long n, uint8_t* out, cudaStream_t stream);
// 3x3x3 one-hot rows in the EXACT encoding -> sticker rows
int launch_decode3_exact(const void* onehot, int dtype, long long n, uint8_t* out, cudaStream_t stream);

// exact 2x2x2 distances (distance.cu, layout in cube_distance.cuh): the BFS table build (memsets and one launch
// per level), the lookup and the optimal solve
int launch_distance_build2(uint8_t* table, cudaStream_t stream);
int launch_distance2(const uint8_t* table, const uint8_t* states, long long n, uint8_t* distance, cudaStream_t stream);
int launch_solve_optimal2(const uint8_t* table, const uint8_t* states, long long n, uint8_t* actions, uint8_t* length,
                          cudaStream_t stream);

// 3x3x3 pattern databases (pattern.cu, layout in cube_pattern.cuh): the BFS build of the three sections (memsets and
// one launch per level), the bound and the bounded IDA* solve
int launch_pattern_build3(uint8_t* tables, cudaStream_t stream);
int launch_distance_bound3(const uint8_t* tables, const uint8_t* states, long long n, uint8_t* bound, uint8_t* parts,
                           cudaStream_t stream);
int launch_solve_bounded3(const uint8_t* tables, const uint8_t* states, long long n, int max_length, long long max_nodes,
                          uint8_t* actions, uint8_t* length, uint8_t* lower, long long* nodes, cudaStream_t stream);

// one-shot SUM all-reduce of int64 values over peer-mapped exchange buffers (peer.cu)
size_t peer_buffer_bytes(int cap);
int launch_peer_allreduce_i64(int world, int rank, const uint64_t* peer_bufs, long long* values, int n, int cap,
                              unsigned epoch, cudaStream_t stream);

}  // namespace cube
