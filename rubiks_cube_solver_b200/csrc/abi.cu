// extern "C" boundary of libcube_b200.so: argument checks, then the launchers.
// See include/cube_b200.h for the contract of every entry point.
#include <cstdio>
#include <initializer_list>
#include <cuda_runtime.h>

#include "../../include/cube_b200.h"
#include "cube_common.cuh"
#include "cube_distance.cuh"
#include "cube_kernels.h"
#include "cube_launch.cuh"

namespace {

thread_local char t_err[256] = "";

int fail(int code, const char* what)
{
    if (code > 0)
        snprintf(t_err, sizeof(t_err), "%s: CUDA error %d (%s)", what, code, cudaGetErrorString((cudaError_t)code));
    else
        snprintf(t_err, sizeof(t_err), "%s: %s", what,
                 code == CUBE_ERR_SIZE ? "cube_size must be 2 or 3"
                 : code == CUBE_ERR_ARG ? "bad argument (null pointer, negative count or unknown dtype)"
                 : code == CUBE_ERR_ALIGN ? "misaligned device pointer (sticker, move and one-hot arrays: 16 bytes; "
                                            "float / int32: 4; float64: 8; MCTS tree store: see cube_mcts_tree_t)"
                 : code == CUBE_ERR_ACTION ? "action index out of range" : "error");
    return code;
}

inline bool misaligned(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) != 0; }
inline bool misaligned4(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 3u) != 0; }   // float / int32 arrays
inline bool misaligned8(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 7u) != 0; }   // float64 arrays

#define CUBE_CHECK_SIZE(fn) if (cube_size != 2 && cube_size != 3) return fail(CUBE_ERR_SIZE, fn)

// the exact distance table exists for the 2x2x2 only
int fail_distance_size(const char* what)
{
    snprintf(t_err, sizeof(t_err), "%s: exact distances exist for cube_size 2 only", what);
    return CUBE_ERR_SIZE;
}
#define CUBE_DONE(fn, rc) do { int rc_ = (rc); return rc_ ? fail(rc_, fn) : 0; } while (0)

// the tree store of cube_mcts_traverse / cube_mcts_update (include/cube_b200.h): CUBE_ERR_ARG for bad sizes and, with
// trees, for any NULL pointer but sim_counter; CUBE_ERR_ALIGN for a pointer the kernels load as a vector or a word
int mcts_tree_check(int cube_size, const cube_mcts_tree_t* t)
{
    if (!t || t->n_trees < 0 || t->n_slots < 1 || t->n_slots > 255 || t->path_cap < 1 || t->rand_cap < 1)
        return CUBE_ERR_ARG;
    if (t->n_trees == 0) return CUBE_OK;
    if (!t->node_key || !t->child_key || !t->child_done || !t->P || !t->W || !t->N || !t->L || !t->n_nodes ||
        !t->active || !t->root_state || !t->root_key || !t->rand_table || !t->rand_ptr || !t->path_node ||
        !t->path_action || !t->path_len || !t->leaf_state || !t->flags || !t->child_slot)
        return CUBE_ERR_ARG;
    const uintptr_t row = cube_size == 3 ? 15u : 7u;                  // int4 / int2 rows of N, P, W, L
    for (const void* p : {(const void*)t->P, (const void*)t->W, (const void*)t->N, (const void*)t->L})
        if (reinterpret_cast<uintptr_t>(p) & row) return CUBE_ERR_ALIGN;
    if (reinterpret_cast<uintptr_t>(t->child_slot) & 1u) return CUBE_ERR_ALIGN;
    for (const void* p : {(const void*)t->node_key, (const void*)t->child_key, (const void*)t->root_key,
                          (const void*)t->root_state, (const void*)t->leaf_state, (const void*)t->path_node,
                          (const void*)t->path_action, (const void*)t->n_nodes, (const void*)t->rand_ptr,
                          (const void*)t->path_len, (const void*)t->flags, (const void*)t->sim_counter})
        if (misaligned4(p)) return CUBE_ERR_ALIGN;
    return CUBE_OK;
}

}  // namespace

extern "C" {

int cube_abi_version(void) { return CUBE_ABI_VERSION; }

const char* cube_last_error(void) { return t_err; }

int cube_sm_count(void) { return cube::sm_count(); }

int cube_set_reserved_sms(int n)
{
    if (n < 0) return fail(CUBE_ERR_ARG, "cube_set_reserved_sms");
    cube::set_reserved_sms(n);
    return CUBE_OK;
}

int cube_scramble(int cube_size, const uint8_t* moves, int64_t n, int depth, uint8_t* states_out,
                  uint8_t* solved, float* reward, uint64_t* counters, void* stream)
{
    CUBE_CHECK_SIZE("cube_scramble");
    if (n < 0 || depth < 0 || (n > 0 && (!states_out || (depth > 0 && !moves)))) return fail(CUBE_ERR_ARG, "cube_scramble");
    if (misaligned(moves) || misaligned(states_out) || misaligned4(reward)) return fail(CUBE_ERR_ALIGN, "cube_scramble");
    CUBE_DONE("cube_scramble", cube::launch_scramble(cube_size, moves, n, depth, states_out, solved, reward,
                                                     (unsigned long long*)counters, (cudaStream_t)stream));
}

int cube_scramble_step(int cube_size, const uint8_t* moves, const uint8_t* actions, int64_t n, int depth,
                       uint8_t* states_out, uint8_t* solved, float* reward, uint64_t* counters, void* stream)
{
    CUBE_CHECK_SIZE("cube_scramble_step");
    if (n < 0 || depth < 0 || (n > 0 && (!states_out || !actions || (depth > 0 && !moves))))
        return fail(CUBE_ERR_ARG, "cube_scramble_step");
    if (misaligned(moves) || misaligned(states_out) || misaligned4(reward)) return fail(CUBE_ERR_ALIGN, "cube_scramble_step");
    CUBE_DONE("cube_scramble_step", cube::launch_scramble(cube_size, moves, n, depth, states_out, solved, reward,
                                                          (unsigned long long*)counters, (cudaStream_t)stream, actions));
}

int cube_scramble_prefixes_max_depth(int cube_size)
{
    CUBE_CHECK_SIZE("cube_scramble_prefixes_max_depth");
    return cube::prefix_max_depth(cube_size);
}

int cube_scramble_prefixes(int cube_size, const uint8_t* moves, int64_t n, int depth, uint8_t* states_out,
                           uint8_t* solved, uint64_t* counters, void* stream)
{
    CUBE_CHECK_SIZE("cube_scramble_prefixes");
    if (n < 0 || depth < 0 || depth > cube::prefix_max_depth(cube_size) || (n > 0 && depth > 0 && (!moves || !states_out)))
        return fail(CUBE_ERR_ARG, "cube_scramble_prefixes");
    if (misaligned(moves) || misaligned(states_out)) return fail(CUBE_ERR_ALIGN, "cube_scramble_prefixes");
    CUBE_DONE("cube_scramble_prefixes", cube::launch_prefixes(cube_size, moves, n, depth, states_out, solved,
                                                              (unsigned long long*)counters, (cudaStream_t)stream));
}

int cube_step(int cube_size, uint8_t* states, const uint8_t* actions, int64_t n, uint8_t* solved,
              float* reward, uint64_t* counters, void* stream)
{
    CUBE_CHECK_SIZE("cube_step");
    if (n < 0 || (n > 0 && (!states || !actions))) return fail(CUBE_ERR_ARG, "cube_step");
    if (misaligned(states) || misaligned4(reward)) return fail(CUBE_ERR_ALIGN, "cube_step");
    CUBE_DONE("cube_step", cube::launch_walk(cube_size, states, actions, n, 1, states, solved, reward,
                                             (unsigned long long*)counters, (cudaStream_t)stream));
}

int cube_walk(int cube_size, const uint8_t* states_in, const uint8_t* moves, int64_t n, int depth,
              uint8_t* states_out, uint8_t* solved, float* reward, uint64_t* counters, void* stream)
{
    CUBE_CHECK_SIZE("cube_walk");
    if (n < 0 || depth < 0 || (n > 0 && (!states_in || !states_out || (depth > 0 && !moves))))
        return fail(CUBE_ERR_ARG, "cube_walk");
    if (misaligned(states_in) || misaligned(states_out) || misaligned4(reward)) return fail(CUBE_ERR_ALIGN, "cube_walk");
    CUBE_DONE("cube_walk", cube::launch_walk(cube_size, states_in, moves, n, depth, states_out, solved, reward,
                                             (unsigned long long*)counters, (cudaStream_t)stream));
}

int cube_solved(int cube_size, const uint8_t* states, int64_t n, uint8_t* solved, float* reward,
                uint64_t* counters, void* stream)
{
    CUBE_CHECK_SIZE("cube_solved");
    if (n < 0 || (n > 0 && !states)) return fail(CUBE_ERR_ARG, "cube_solved");
    if (misaligned(states) || misaligned4(reward)) return fail(CUBE_ERR_ALIGN, "cube_solved");
    CUBE_DONE("cube_solved", cube::launch_solved(cube_size, states, n, solved, reward,
                                                 (unsigned long long*)counters, (cudaStream_t)stream));
}

int cube_moves_from_seeds(int cube_size, const uint32_t* seeds, int64_t n, int depth, uint8_t* moves_out,
                          uint64_t* counters, void* stream)
{
    CUBE_CHECK_SIZE("cube_moves_from_seeds");
    if (n < 0 || depth < 0 || depth > 128 || (n > 0 && depth > 0 && (!seeds || !moves_out)))
        return fail(CUBE_ERR_ARG, "cube_moves_from_seeds");
    CUBE_DONE("cube_moves_from_seeds", cube::launch_seeded_moves(cube_size, seeds, n, depth, moves_out,
                                                                (unsigned long long*)counters, (cudaStream_t)stream));
}

int cube_mcts_traverse(int cube_size, const cube_mcts_tree_t* tree, float cpuct, int virtual_loss, void* stream)
{
    CUBE_CHECK_SIZE("cube_mcts_traverse");
    if (const int rc = mcts_tree_check(cube_size, tree)) return fail(rc, "cube_mcts_traverse");
    CUBE_DONE("cube_mcts_traverse", cube::launch_mcts_traverse(cube_size, *tree, cpuct, virtual_loss, (cudaStream_t)stream));
}

int cube_mcts_update(int cube_size, const cube_mcts_tree_t* tree, const uint8_t* leaf_key, const uint8_t* child_key_new,
                     const uint8_t* child_done_new, const float* value, const float* policy, float value_min,
                     int sim_index, int8_t* actions_out, int32_t* n_actions, int32_t* n_sims, int32_t* n_active, void* stream)
{
    CUBE_CHECK_SIZE("cube_mcts_update");
    if (const int rc = mcts_tree_check(cube_size, tree)) return fail(rc, "cube_mcts_update");
    if (tree->n_trees > 0 && (!leaf_key || !child_key_new || !child_done_new || !value || !policy || !actions_out ||
                              !n_actions || !n_sims))
        return fail(CUBE_ERR_ARG, "cube_mcts_update");
    if (misaligned4(leaf_key) || misaligned4(child_key_new) || misaligned4(value) || misaligned4(policy) ||
        misaligned4(n_actions) || misaligned4(n_sims) || misaligned4(n_active))
        return fail(CUBE_ERR_ALIGN, "cube_mcts_update");
    CUBE_DONE("cube_mcts_update", cube::launch_mcts_update(cube_size, *tree, leaf_key, child_key_new, child_done_new, value,
                                                           policy, value_min, sim_index, actions_out, n_actions, n_sims, n_active,
                                                           (cudaStream_t)stream));
}

int cube_adi_targets(int cube_size, const float* child_values, const uint8_t* child_solved, const float* parent_values,
                     const int32_t* scramble_count, const double* weight, int table_len, int64_t n,
                     float* target_value, int32_t* target_policy, double* error, void* stream)
{
    CUBE_CHECK_SIZE("cube_adi_targets");
    if (n < 0 || table_len < 0 || (n > 0 && (!child_values || !child_solved || !parent_values || !scramble_count ||
                                             !weight || !target_value || !target_policy || !error)))
        return fail(CUBE_ERR_ARG, "cube_adi_targets");
    if (misaligned(child_values) || misaligned4(parent_values) || misaligned4(scramble_count) || misaligned8(weight) ||
        misaligned4(target_value) || misaligned4(target_policy) || misaligned8(error))
        return fail(CUBE_ERR_ALIGN, "cube_adi_targets");
    CUBE_DONE("cube_adi_targets", cube::launch_adi_targets(cube_size, child_values, child_solved, parent_values,
                                                           scramble_count, weight, table_len, n, target_value,
                                                           target_policy, error, (cudaStream_t)stream));
}

int cube_encode(int cube_size, const uint8_t* states, int64_t n, void* onehot, int dtype, int encoding, void* stream)
{
    CUBE_CHECK_SIZE("cube_encode");
    if (n < 0 || dtype < 0 || dtype > 2 || encoding < 0 || encoding > 1 || (n > 0 && (!states || !onehot)))
        return fail(CUBE_ERR_ARG, "cube_encode");
    if (misaligned(states) || misaligned(onehot)) return fail(CUBE_ERR_ALIGN, "cube_encode");
    CUBE_DONE("cube_encode", cube::launch_expand(cube_size, states, n, nullptr, nullptr, onehot, dtype, nullptr,
                                                 nullptr, nullptr, (cudaStream_t)stream, encoding));
}

int cube_expand(int cube_size, const uint8_t* states, int64_t n, uint8_t* children, void* child_onehot,
                void* parent_onehot, int dtype, int encoding, uint8_t* solved, float* reward, uint64_t* counters,
                void* stream)
{
    CUBE_CHECK_SIZE("cube_expand");
    if (n < 0 || dtype < 0 || dtype > 2 || encoding < 0 || encoding > 1 || (n > 0 && !states))
        return fail(CUBE_ERR_ARG, "cube_expand");
    if (misaligned(states) || misaligned(children) || misaligned(child_onehot) || misaligned(parent_onehot) ||
        misaligned4(reward))
        return fail(CUBE_ERR_ALIGN, "cube_expand");
    CUBE_DONE("cube_expand", cube::launch_expand(cube_size, states, n, children, child_onehot, parent_onehot, dtype,
                                                 solved, reward, (unsigned long long*)counters,
                                                 (cudaStream_t)stream, encoding));
}

int cube_expand_codes(int cube_size, const uint8_t* states, int64_t n, uint8_t* children, uint8_t* child_codes,
                      uint8_t* parent_codes, void* parent_onehot, int dtype, int encoding, uint8_t* solved, float* reward,
                      uint64_t* counters, void* stream)
{
    CUBE_CHECK_SIZE("cube_expand_codes");
    if (n < 0 || dtype < 0 || dtype > 2 || encoding < 0 || encoding > 1 || (n > 0 && !states))
        return fail(CUBE_ERR_ARG, "cube_expand_codes");
    if (misaligned(states) || misaligned(children) || misaligned(parent_onehot) || misaligned4(reward))
        return fail(CUBE_ERR_ALIGN, "cube_expand_codes");
    CUBE_DONE("cube_expand_codes", cube::launch_expand_codes(cube_size, states, n, children, child_codes, parent_codes,
                                                             parent_onehot, dtype, solved, reward,
                                                             (unsigned long long*)counters, (cudaStream_t)stream, encoding));
}

int cube_decode(int cube_size, const void* onehot, int dtype, int encoding, int64_t n, uint8_t* states_out, void* stream)
{
    CUBE_CHECK_SIZE("cube_decode");
    if (n < 0 || dtype < 0 || dtype > 2 || encoding < 0 || encoding > 1 || (n > 0 && (!onehot || !states_out)))
        return fail(CUBE_ERR_ARG, "cube_decode");
    if (cube_size == 3 && encoding != CUBE_ENCODING_EXACT)
        return fail(CUBE_ERR_SIZE, "cube_decode (the reference's 3x3x3 encoding is lossy: NotImplemented there too; use CUBE_ENCODING_EXACT)");
    if (misaligned(onehot) || misaligned(states_out)) return fail(CUBE_ERR_ALIGN, "cube_decode");
    if (cube_size == 3)
        CUBE_DONE("cube_decode", cube::launch_decode3_exact(onehot, dtype, n, states_out, (cudaStream_t)stream));
    CUBE_DONE("cube_decode", cube::launch_decode2(onehot, dtype, n, states_out, (cudaStream_t)stream));
}

int64_t cube_peer_buffer_bytes(int capacity)
{
    if (capacity < 1) return fail(CUBE_ERR_ARG, "cube_peer_buffer_bytes");
    return (int64_t)cube::peer_buffer_bytes(capacity);
}

int cube_peer_allreduce_i64(int world, int rank, const uint64_t* peer_buffers, int64_t* values, int n, int capacity,
                            uint32_t epoch, void* stream)
{
    if (world < 1 || world > CUBE_PEER_MAX_RANKS || rank < 0 || rank >= world || n < 0 || capacity < 1 || n > capacity ||
        epoch == 0 || !peer_buffers || (n > 0 && !values))
        return fail(CUBE_ERR_ARG, "cube_peer_allreduce_i64");
    for (int p = 0; p < world; ++p)
        if (!peer_buffers[p] || (peer_buffers[p] & 127u)) return fail(CUBE_ERR_ALIGN, "cube_peer_allreduce_i64");
    if (reinterpret_cast<uintptr_t>(values) & 7u) return fail(CUBE_ERR_ALIGN, "cube_peer_allreduce_i64");
    if (n == 0) return CUBE_OK;
    CUBE_DONE("cube_peer_allreduce_i64", cube::launch_peer_allreduce_i64(world, rank, peer_buffers, (long long*)values, n,
                                                                         capacity, epoch, (cudaStream_t)stream));
}

int cube_validate_actions(int cube_size, const uint8_t* actions, int64_t count, uint64_t* counters, void* stream)
{
    CUBE_CHECK_SIZE("cube_validate_actions");
    if (count < 0 || !counters || (count > 0 && !actions)) return fail(CUBE_ERR_ARG, "cube_validate_actions");
    if (misaligned(actions)) return fail(CUBE_ERR_ALIGN, "cube_validate_actions");
    CUBE_DONE("cube_validate_actions", cube::launch_validate(cube_size, actions, count,
                                                             (unsigned long long*)counters, (cudaStream_t)stream));
}

int64_t cube_distance_table_entries(int cube_size)
{
    if (cube_size != 2) return fail_distance_size("cube_distance_table_entries");
    return (int64_t)kDist2Entries;
}

int cube_distance_table_build(int cube_size, uint8_t* table, void* stream)
{
    if (cube_size != 2) return fail_distance_size("cube_distance_table_build");
    if (!table) return fail(CUBE_ERR_ARG, "cube_distance_table_build");
    if (misaligned(table)) return fail(CUBE_ERR_ALIGN, "cube_distance_table_build");
    CUBE_DONE("cube_distance_table_build", cube::launch_distance_build2(table, (cudaStream_t)stream));
}

int cube_distance(int cube_size, const uint8_t* table, const uint8_t* states, int64_t n, uint8_t* distance,
                  void* stream)
{
    if (cube_size != 2) return fail_distance_size("cube_distance");
    if (!table || !states || n < 0 || (n > 0 && !distance)) return fail(CUBE_ERR_ARG, "cube_distance");
    if (misaligned(table) || misaligned(states)) return fail(CUBE_ERR_ALIGN, "cube_distance");
    CUBE_DONE("cube_distance", cube::launch_distance2(table, states, n, distance, (cudaStream_t)stream));
}

int cube_solve_optimal(int cube_size, const uint8_t* table, const uint8_t* states, int64_t n, uint8_t* actions_out,
                       uint8_t* length, void* stream)
{
    if (cube_size != 2) return fail_distance_size("cube_solve_optimal");
    if (!table || !states || n < 0 || (n > 0 && (!actions_out || !length))) return fail(CUBE_ERR_ARG, "cube_solve_optimal");
    if (misaligned(table) || misaligned(states)) return fail(CUBE_ERR_ALIGN, "cube_solve_optimal");
    CUBE_DONE("cube_solve_optimal", cube::launch_solve_optimal2(table, states, n, actions_out, length,
                                                                (cudaStream_t)stream));
}

}  // extern "C"
