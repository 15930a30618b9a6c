/* cube_b200.h -- C ABI of the B200-native batched cube simulator (libcube_b200.so).
 *
 * This is the drop-in boundary for the reference's rollout / training-data hot
 * path.  The reference is pure Python (no FFI of its own); each entry point below
 * names the reference code whose batched equivalent it computes, and
 * INTEGRATION.md shows the ctypes binding a maintainer of the reference adds.
 * Paths are relative to the reference tree (SUNGBEOMCHOI/Rubiks-Cube-Solver).
 *
 * Conventions
 *   - cube_size is 2 (2x2x2: S=24 stickers, A=6 actions, one-hot 7x21=147) or
 *     3 (3x3x3: S=54, A=12, one-hot 20x24=480); anything else -> CUBE_ERR_SIZE
 *     (the reference raises NotImplementedError, cube_env.py:43-44).
 *   - sticker rows are uint8 colours 0..5 in the reference's sticker order
 *     (py333.py:3-19; py222), row-major [n, S]; actions are uint8 indices in the
 *     order of cube_env.py:24-28.
 *   - every pointer is a DEVICE pointer unless the name ends in _host; arrays
 *     are contiguous.  Sticker rows, one-hot buffers and cube_scramble's move
 *     array must start on a 16-byte boundary, float / int32 arrays on their
 *     natural 4 bytes, float64 arrays on 8 (CUBE_ERR_ALIGN otherwise); action / move bytes of
 *     cube_step / cube_walk and the solved flags may start anywhere (a sliced
 *     buffer that is not 16- / 8- / 4-byte aligned takes a byte-wise kernel).
 *   - calls are asynchronous on `stream` (a cudaStream_t, may be NULL), never
 *     allocate, never synchronise, keep no state between calls and are
 *     re-entrant (the persistent kernels' tile counters come from a ring of 1 024
 *     slots per device: fewer than that many launches may be RUNNING at once).  Return value: 0, a negative CUBE_ERR_*, or a positive
 *     cudaError_t.  cube_last_error() describes the last non-zero return of
 *     the calling thread.
 *   - action indices are NOT range-checked on the hot path: indices A..12 are
 *     no-ops (12 = CUBE_NOOP, the padding index for ragged batches); indices
 *     13..255 are memory-safe but give unspecified states.  Call
 *     cube_validate_actions when the reference's IndexError (cube_env.py:86,96)
 *     must be reproduced.
 *   - counters, when non-NULL, is uint64[4] on the device and is only ever
 *     ADDED to: [0] += outputs that are solved, [1] += outputs produced,
 *     [2] += out-of-range actions (cube_validate_actions), [3] += seeded rows that needed
 *     more than 227 raw draws (cube_moves_from_seeds; such rows are exact, see there).
 *     Rewards are +1.0f / -1.0f, so a reward total is 2*[0] - [1] exactly.
 */
#ifndef CUBE_B200_H
#define CUBE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CUBE_ABI_VERSION 2   /* 2: cube_mcts_tree_t memo fields, cube_mcts_update n_active, new entry points */

#define CUBE_OK 0
#define CUBE_ERR_SIZE (-1)
#define CUBE_ERR_ARG (-2)
#define CUBE_ERR_ALIGN (-3)
#define CUBE_ERR_ACTION (-4)

#define CUBE_NOOP 12 /* action index that leaves the cube unchanged (both sizes) */

#define CUBE_DTYPE_BF16 0
#define CUBE_DTYPE_F32 1
#define CUBE_DTYPE_U8 2

/* One-hot encodings of a 3x3x3 state ([20, 24]: row = slot, corners 3 * piece + ori, edges 2 * piece + ori).
 * REFERENCE is the reference's table as shipped (py333.py:140-198): its corner part is lossy -- row 6 of
 * corner_pieceDefs is mirrored and 21 reachable hashes are unassigned -- and it is what a model trained
 * with the reference expects; it is the default everywhere and bit-exact against the reference.
 * EXACT is an opt-in bijection with the same layout: slot 6 read the right way round, every rotation of
 * every corner assigned (piece, ori) <- np.roll(home colours, ori) like py222; edges are unchanged.  Only
 * EXACT can be decoded (cube_decode).  2x2x2 has a single encoding (py222's, already exact): both values
 * mean the same there. */
#define CUBE_ENCODING_REFERENCE 0
#define CUBE_ENCODING_EXACT 1

int cube_abi_version(void);
const char* cube_last_error(void);

/* number of SMs of the current device (grid sizing is done inside the library) */
int cube_sm_count(void);

/* The persistent kernels (cube_scramble, cube_step, cube_walk) run one CTA per SM and fill it
 * (registers, shared memory).  A kernel of another stream that must make progress WHILE they run --
 * NCCL's all-reduce of the counters in a multi-GPU job -- would otherwise wait for a CTA to retire.
 * n SMs are left free for such kernels (default 0, or the CUBE_RESERVED_SMS environment variable).
 * Measured on 2 x B200 with the 32-byte counter all-reduce per step: no gain (99 % weak-scaling
 * efficiency either way), so nothing sets it by default. */
int cube_set_reserved_sms(int n);

/* Multi-GPU: the path's only collective -- the SUM of the solved / produced counters over the ranks of ONE box
 * (SURVEY.md 8e; the reference is single-process, its counterpart is the `solved` tally of a test loop,
 * test.py:52-60) -- as a one-shot all-reduce over NVLink peer memory: one small kernel per rank stores its values
 * into its slot of EVERY rank's exchange buffer, raises a flag there and sums all slots of its own buffer once
 * every flag has arrived (csrc/peer.cu).  Every rank gets the same totals, in place.
 *   peer_buffers [world]  uint64  host  device addresses, valid on THIS device, of all ranks' exchange
 *                                        buffers in rank order (own buffer included; e.g. torch symmetric memory's
 *                                        buffer_ptrs), each cube_peer_buffer_bytes(capacity) bytes, 128-byte
 *                                        aligned, zero-filled before the first call
 *   values       [n]      int64   device in/out, n <= capacity (the same n and capacity on every rank)
 *   epoch                 uint32         call number: 1 for the first call on a set of buffers, then 2, 3, ...
 *                                        -- the same on every rank (nothing is ever reset; slots alternate with
 *                                        the epoch's parity, so consecutive calls may overlap across ranks)
 * All ranks must make the call (it waits for every rank's flag: a missing rank hangs the kernel, like any
 * collective); world <= CUBE_PEER_MAX_RANKS.  Measured against ncclAllReduce of the same 640 bytes: DESIGN.md 6. */
#define CUBE_PEER_MAX_RANKS 8
int64_t cube_peer_buffer_bytes(int capacity);
int cube_peer_allreduce_i64(int world, int rank, const uint64_t* peer_buffers, int64_t* values, int n, int capacity,
                            uint32_t epoch, void* stream);

/* Identically seeded scrambles -- the move indices reset(seed, k) draws (cube_env.py:62-65):
 *   moves_out[i, :] = np.random.RandomState(seeds[i]).randint(A, size=depth)      (bit for bit)
 * generated on the device (MT19937 seeded by init_genrand, masked rejection sampling like NumPy's
 * legacy randint).  A shorter reset(seed, k') is the first k' entries of the row.
 *   seeds      [n]        uint32   in   (the reference's integer seeds, < 2^32)
 *   moves_out  [n, depth] uint8    out  depth <= 128
 * A row is drawn from the first 227 raw outputs of its generator without materialising its state; a row
 * those leave short (about one seed in 3e9 at depth 128: 2103926524 and 3830291768 for the 3x3x3,
 * 3969546545 for the 2x2x2) continues from the full 624-word state, exactly as NumPy does, and
 * counters[3] += 1 for it. */
int cube_moves_from_seeds(int cube_size, const uint32_t* seeds, int64_t n, int depth, uint8_t* moves_out,
                          uint64_t* counters, void* stream);

/* Fused scramble from the solved cube -- reset()'s loop `init_state(); for a in
 * action_sequence: step(a)` (cube_env.py:61-67) and the per-cube loop of
 * get_random_samples (cube_env.py:187-191), for n instances at once.
 *   moves      [n, depth] uint8     in
 *   states_out [n, S]     uint8     out  final sticker rows (== chaining doMove_3, py333.py:220-222)
 *   solved     [n]        uint8     out  or NULL   isSolved_3 (py333.py:229-233) of the final row
 *   reward     [n]        float32   out  or NULL   +1.0 / -1.0 (cube_env.py:89-104)
 * depth >= 0 (depth 0 returns solved cubes). */
int cube_scramble(int cube_size, const uint8_t* moves, int64_t n, int depth, uint8_t* states_out,
                  uint8_t* solved, float* reward, uint64_t* counters, void* stream);

/* Scramble, then one step, fused -- `state = env.reset(seed, k); env.step(a)` (cube_env.py:50-111) for n
 * instances in one launch: the `depth` moves and then actions[i] are applied in registers, only the final
 * sticker row, its done flag and its reward are written (BASELINE configs[2] read literally: "scramble + step").
 *   actions [n] uint8 in; everything else as cube_scramble.  Equals cube_scramble on [moves | actions]. */
int cube_scramble_step(int cube_size, const uint8_t* moves, const uint8_t* actions, int64_t n, int depth,
                       uint8_t* states_out, uint8_t* solved, float* reward, uint64_t* counters, void* stream);

/* Every prefix of every scramble, in ONE launch -- the parents of an ADI batch: get_random_samples
 * (cube_env.py:187-194) emits a sample after EVERY move of every cube, cube by cube.
 *   moves      [n, depth]    uint8  in
 *   states_out [n, depth, S] uint8  out  states_out[i, k] = sticker row after moves[i, 0..k]  (cube-major:
 *                                        the order in which the reference appends to its replay buffer)
 *   solved     [n, depth]    uint8  out or NULL  isSolved of every prefix
 * counters[0] += solved prefixes, [1] += n * depth.  depth <= cube_scramble_prefixes_max_depth(cube_size)
 * (526 / 1159: a tile of 8 cubes x depth rows is staged in shared memory), else CUBE_ERR_ARG. */
int cube_scramble_prefixes(int cube_size, const uint8_t* moves, int64_t n, int depth, uint8_t* states_out,
                           uint8_t* solved, uint64_t* counters, void* stream);
int cube_scramble_prefixes_max_depth(int cube_size);

/* One transition on resident states -- CubeEnv.step (cube_env.py:71-111):
 * states[i] <- states[i][moveDefs[actions[i]]], then solved / reward.  In place. */
int cube_step(int cube_size, uint8_t* states, const uint8_t* actions, int64_t n, uint8_t* solved,
              float* reward, uint64_t* counters, void* stream);

/* `depth` transitions per instance starting from given sticker rows (any byte
 * content); states_out may alias states_in.  moves is [n, depth]. */
int cube_walk(int cube_size, const uint8_t* states_in, const uint8_t* moves, int64_t n, int depth,
              uint8_t* states_out, uint8_t* solved, float* reward, uint64_t* counters, void* stream);

/* isSolved_3 / isSolved (py333.py:229-233) and the reward of resident rows. */
int cube_solved(int cube_size, const uint8_t* states, int64_t n, uint8_t* solved, float* reward,
                uint64_t* counters, void* stream);

/* sim_state_to_state (cube_env.py:132-152): one-hot network input of each row,
 * [n, 20, 24] or [n, 7, 21] elements of `dtype` (bf16 / f32 / u8), exactly one 1
 * per one-hot row for the rows of real states; `encoding` = CUBE_ENCODING_REFERENCE (3x3x3 corners through the
 * reference's table as shipped) or CUBE_ENCODING_EXACT.  A 2x2x2 row that names a cubelet twice gets what the
 * reference's loop gives it (cube_env.py:141-147): two 1s in that cubelet's one-hot row, none in the missing
 * cubelet's. */
int cube_encode(int cube_size, const uint8_t* states, int64_t n, void* onehot, int dtype, int encoding, void* stream);

/* ADI / MCTS expansion -- the child loop of get_target_value (cube_env.py:212-238)
 * and of MCTS.expand (mcts.py:96-101) for n parents at once, children in action order.
 *   children      [n, A, S]   uint8    or NULL   child sticker rows
 *   child_onehot  [n, A, D]   dtype    or NULL   network input of every child
 *   parent_onehot [n, D]      dtype    or NULL   network input of the parent (mcts.py:92)
 *   solved        [n, A]      uint8    or NULL   done flag of every child
 *   reward        [n, A]      float32  or NULL
 * The reference stops at the first solved child (cube_env.py:217-220); here all A
 * children are produced and `solved` lets the caller apply that override. */
int cube_expand(int cube_size, const uint8_t* states, int64_t n, uint8_t* children, void* child_onehot,
                void* parent_onehot, int dtype, int encoding, uint8_t* solved, float* reward, uint64_t* counters,
                void* stream);

/* ADI target assembly -- the tail of get_target_value (cube_env.py:239-252) for n parents whose
 * children came from cube_expand and were valued by the caller's network:
 *   child_values   [n, A] float32  in   V(child_a)
 *   child_solved   [n, A] uint8    in   cube_expand's `solved`
 *   parent_values  [n]    float32  in   V(state)
 *   scramble_count [n]    int32    in   depth k of every parent (cube_env.py:190-192)
 *   weight         [table_len] float64 in  weight[k] = k ** (-temperature), computed by the HOST so the
 *                                       priorities match Python's float power bit for bit
 *   target_value   [n]    float32  out  1.0 at the first solved child, else max_a(V(child_a) + (-1.0))
 *   target_policy  [n]    int32    out  that child (the first maximum wins, like torch.max)
 *   error          [n]    float64  out  |V(state) - target_value| * weight[scramble_count] */
int cube_adi_targets(int cube_size, const float* child_values, const uint8_t* child_solved,
                     const float* parent_values, const int32_t* scramble_count, const double* weight,
                     int table_len, int64_t n, float* target_value, int32_t* target_policy, double* error,
                     void* stream);

/* ---- batched MCTS tree store (mcts.py:17-154) --------------------------------------------------
 * B independent trees, one per cube, each a slab of n_slots node slots (one simulation adds at most
 * one node: n_slots = numMCTSSim + 1 <= 255).  A node is children_and_data[key] of the reference
 * (mcts.py:103-110): key = the observation, here the one-hot rows' column indices (KEY = 20 bytes for
 * 3x3x3, 8 for 2x2x2: 7 indices + one zero byte), children keys, P, W, N, L and done flags.  All
 * members are DEVICE pointers owned by the caller; A = 12 / 6, S = 54 / 24.
 * When n_trees > 0, every pointer except sim_counter must be non-NULL (else CUBE_ERR_ARG), and the kernels'
 * vector loads need (else CUBE_ERR_ALIGN; both checked before any launch):
 *   P, W, N, L                                      16 bytes (3x3x3: 48-byte rows) / 8 bytes (2x2x2: 24-byte rows)
 *   child_slot                                      2 bytes
 *   node_key, child_key, root_key, root_state,
 *   leaf_state, path_node, path_action              4 bytes (read and written as 32-bit words)
 *   n_nodes, rand_ptr, path_len, flags, sim_counter 4 bytes
 * The same holds for cube_mcts_update's leaf_key and child_key_new (4 bytes) and its value, policy, n_actions,
 * n_sims and n_active (4 bytes; only n_active may be NULL). */
typedef struct cube_mcts_tree {
    int32_t n_trees, n_slots, path_cap, rand_cap; /* B, M, capacity of one traversal path, draws per tree */
    uint8_t* node_key;                    /* [B, M, KEY]     key of every expanded node                  */
    uint8_t* child_key;                   /* [B, M, A, KEY]  keys of its children (mcts.py:96-101)       */
    uint8_t* child_done;                  /* [B, M, A]       is_solved of its children                   */
    float* P;                             /* [B, M, A]       policy (mcts.py:92)                         */
    float* W;                             /* [B, M, A]       max-backed-up value, starts at value_min    */
    int32_t* N;                           /* [B, M, A]       visit counts                                */
    int32_t* L;                           /* [B, M, A]       virtual loss                                */
    int32_t* n_nodes;                     /* [B]             expanded nodes so far                       */
    uint8_t* active;                      /* [B]             0 once the tree has returned a solution     */
    const uint8_t* root_state;            /* [B, S]          sticker rows of the roots                   */
    const uint8_t* root_key;              /* [B, KEY]                                                    */
    const uint8_t* rand_table;            /* [B, rand_cap]   pre-drawn random actions (mcts.py:69-70; a node
                                           *                  revisited inside one traversal draws again) */
    int32_t* rand_ptr;                    /* [B]             draws used so far                           */
    uint8_t* path_node;                   /* [B, path_cap]   out: node slots of the last traversal       */
    uint8_t* path_action;                 /* [B, path_cap]   out: actions of the last traversal          */
    int32_t* path_len;                    /* [B]             out                                         */
    uint8_t* leaf_state;                  /* [B, S]          out: sticker row of the leaf that was reached */
    int32_t* flags;                       /* [1]  |= 1 path_cap exceeded, 2 rand_table exhausted, 4 n_slots exceeded,
                                           *            8 rand_table holds an action >= A (taken as 0)           */
    /* the dict lookup `key in children_and_data` (mcts.py:57), resolved eagerly by cube_mcts_update */
    uint8_t* child_slot;                  /* [B, M, A]       slot of the child's node, 255 = the child is not in the tree
                                           *                  (library scratch: start it at 255)                          */
    int32_t* sim_counter;                 /* [1] or NULL     device-side simulation index: every cube_mcts_traverse adds 1 (start
                                           *                  it at -1) and cube_mcts_update uses it INSTEAD of its sim_index
                                           *                  argument -- lets a caller replay one captured simulation (CUDA graph) */
} cube_mcts_tree_t;

/* MCTS.traverse (mcts.py:52-81) for every active tree: from the root to the first key that is not in
 * the tree; fills path_*, leaf_state; adds virtual_loss to L along the way. */
int cube_mcts_traverse(int cube_size, const cube_mcts_tree_t* tree, float cpuct, int virtual_loss, void* stream);

/* The rest of MCTS.train for every active tree (mcts.py:38-50): store the expanded leaf
 * (leaf_key [B, KEY], child_key_new [B, A, KEY], child_done_new [B, A] from cube_expand; value [B],
 * policy [B, A] from the network; W = value_min, N = L = 0), back-propagate along the path
 * (W = max(W, value), L -= 150, N += 1: mcts.py:122-129) and, if a child of the new leaf is solved,
 * write path actions + that child to actions_out [B, path_cap + 1] (int8), n_actions [B],
 * n_sims [B] = sim_index + 1 and clear `active`.  n_active (int32 [number of simulations] on the device, or
 * NULL): n_active[sim_index] += trees that are still searching after this simulation, so a caller can stop
 * early without reading `active` back. */
int cube_mcts_update(int cube_size, const cube_mcts_tree_t* tree, const uint8_t* leaf_key,
                     const uint8_t* child_key_new, const uint8_t* child_done_new, const float* value,
                     const float* policy, float value_min, int sim_index, int8_t* actions_out,
                     int32_t* n_actions, int32_t* n_sims, int32_t* n_active, void* stream);

/* cube_expand with COMPACT CODES instead of the children's one-hot rows: code[row] = the column of the
 * first 1 of that one-hot row, 0 for a row without a 1 (what argmax over the row gives), KEY = (R + 3) & ~3 bytes per state
 * (8 / 20), zero-padded.  The batched MCTS keys its tree nodes with them (the reference keys its dict with
 * np.array2string of the observation, mcts.py:57,105: equal observations <=> equal codes).
 *   child_codes   [n, A, KEY] uint8  out or NULL
 *   parent_codes  [n, KEY]    uint8  out or NULL
 *   parent_onehot [n, R, C]   dtype  out or NULL     children / solved / reward / counters as in cube_expand */
int cube_expand_codes(int cube_size, const uint8_t* states, int64_t n, uint8_t* children, uint8_t* child_codes,
                      uint8_t* parent_codes, void* parent_onehot, int dtype, int encoding, uint8_t* solved, float* reward,
                      uint64_t* counters, void* stream);

/* state_to_sim_state (cube_env.py:154-175 + py222 getStickers): one-hot [n, 7, 21] of
 * `dtype` -> sticker rows [n, 24].  For cube_size 3 the reference raises NotImplementedError
 * (cube_env.py:171-172: its corner encoding cannot be inverted) and so does CUBE_ENCODING_REFERENCE here
 * (CUBE_ERR_SIZE); with CUBE_ENCODING_EXACT one-hot [n, 20, 24] -> sticker rows [n, 54]. */
int cube_decode(int cube_size, const void* onehot, int dtype, int encoding, int64_t n, uint8_t* states_out, void* stream);

/* counters[2] += number of entries of actions[0..count) that are >= A. */
int cube_validate_actions(int cube_size, const uint8_t* actions, int64_t count, uint64_t* counters,
                          void* stream);

/* ---- exact 2x2x2 distances ----------------------------------------------------------------------
 * The reference measures a solver by its solve percentage alone (test.py:103-158, train.py:167-198); the
 * DeepCube line of work compares solution lengths with optimal ones.  The 2x2x2 of the reference (U, U', F,
 * F', R, R', the DBL corner fixed) has 7! * 3^6 = 3 674 160 states, none more than 14 quarter turns from
 * solved, so a table of every state's distance fits in 3.7 MB (resident in L2).
 *
 * Table layout: one uint8 distance per rank.  With (p_i, o_i) = py222 getOP of slot i = 0..6 (the pairs the
 * 2x2x2 one-hot encoding is built from):
 *     rank = L * 729 + T,   L = sum_{i=0..6} #{j > i : p_j < p_i} * (6 - i)!,   T = sum_{i=0..5} o_i * 3^(5 - i)
 * o_6 is implied: the orientations of a reachable state sum to 0 mod 3.  The solved cube is rank 0.  A sticker
 * row is REACHABLE exactly when the row rebuilt from its rank is the row; any other content (colours >= 6,
 * hashes outside py222's table, two stickers swapped, a twisted corner) has distance CUBE_DISTANCE_UNREACHABLE.
 * cube_size 3 returns CUBE_ERR_SIZE (its 4.3e19 states are out of reach).  A NULL table or states pointer, or
 * n < 0, returns CUBE_ERR_ARG.  The table and sticker rows start on 16-byte boundaries; the byte outputs may start
 * anywhere. */
#define CUBE_DISTANCE_UNREACHABLE 255
#define CUBE_DISTANCE_MAX_2 14

/* number of table entries: 3 674 160 for cube_size 2 */
int64_t cube_distance_table_entries(int cube_size);

/* Fill table [cube_distance_table_entries] uint8 (caller-owned) with the distance of every rank: a
 * level-synchronous breadth-first search from the solved cube, one launch per level. */
int cube_distance_table_build(int cube_size, uint8_t* table, void* stream);

/* distance [n] uint8 out: table[rank(states[i])], or CUBE_DISTANCE_UNREACHABLE.  states [n, 24] uint8. */
int cube_distance(int cube_size, const uint8_t* table, const uint8_t* states, int64_t n, uint8_t* distance,
                  void* stream);

/* An optimal solution of every row, walking down the table: at every step the LOWEST action index whose child
 * is one level closer.
 *   actions_out [n, CUBE_DISTANCE_MAX_2] uint8  out  the solution, padded with CUBE_NOOP (cube_walk of the
 *                                                     row with it ends solved for every reachable row)
 *   length      [n]                     uint8  out  the solution's length = the distance (0 for a solved
 *                                                     row); CUBE_DISTANCE_UNREACHABLE and only NOOPs for an
 *                                                     unreachable row */
int cube_solve_optimal(int cube_size, const uint8_t* table, const uint8_t* states, int64_t n, uint8_t* actions_out,
                       uint8_t* length, void* stream);

/* ---- host-buffer front end (end-to-end path) ------------------------------------------
 * For callers that hold NumPy / host arrays, as every caller of the reference does
 * (train.py:155, :186; test.py:123).  A pipeline handle owns a few stages of device
 * buffers and streams; cube_pipeline_scramble_host cuts the batch into chunks and
 * overlaps the host->device copy of the moves, the fused scramble kernel and the
 * device->host copy of the results.  It blocks until the host buffers are filled.
 * Page-locked host buffers are needed for the overlap (pageable ones still work).
 * The handle is bound to the device that was current at creation. */
typedef struct cube_pipeline cube_pipeline_t;

int cube_pipeline_create(int cube_size, int depth, int64_t chunk_instances, int n_stages /* 1..4 */,
                         cube_pipeline_t** out);
int cube_pipeline_destroy(cube_pipeline_t* p);

/*   moves_host      [n, depth] uint8   in
 *   states_out_host [n, S]     uint8   out
 *   solved_host     [n]        uint8   out or NULL
 *   reward_host     [n]        float32 out or NULL
 *   solved_count               int64   out or NULL  (number of solved final states) */
int cube_pipeline_scramble_host(cube_pipeline_t* p, const uint8_t* moves_host, int64_t n,
                                uint8_t* states_out_host, uint8_t* solved_host, float* reward_host,
                                int64_t* solved_count);

/* Batched reset(seed, k) (cube_env.py:50-69) for host arrays: only 4 bytes per instance cross the bus on the
 * way in -- the moves np.random.RandomState(seed).randint(A, size=depth) are drawn on the device
 * (cube_moves_from_seeds) and scrambled there.  The handle's depth must be 1..128.
 *   seeds_host [n] uint32 in; the outputs as in cube_pipeline_scramble_host (solved_host / reward_host may be
 *   NULL: the reward is +1 where solved, -1 elsewhere, so a caller that wants it can derive it). */
int cube_pipeline_reset_host(cube_pipeline_t* p, const uint32_t* seeds_host, int64_t n, uint8_t* states_out_host,
                             uint8_t* solved_host, float* reward_host, int64_t* solved_count);

/* Page-locked host buffer on transparent huge pages: 2 MiB-aligned, MADV_HUGEPAGE, touched, then
 * cudaHostRegister'ed (portable).  For the host arrays of cube_pipeline_*: with one process per GPU copying
 * at once, 2 MiB pages need 512 times fewer DMA address translations than cudaMallocHost's 4 KiB pages. */
int cube_host_alloc(int64_t bytes, void** out);
int cube_host_free(void* p);

/* ---- single-cube host front end (the drop-in CubeEnv's per-call path) ---------------------
 * The reference's callers drive ONE cube per call (env.reset / env.step / get_obs:
 * cube_env.py:56-111, used by train.py:155,186-191, mcts.py:80, test.py:123).  A handle owns a
 * page of mapped pinned memory that the kernel reads and writes directly, so a call is ONE launch
 * of a one-cube kernel plus a wait for its completion word (polled in the page; cudaStreamSynchronize
 * as the fallback), with no copy calls: ~20 us instead of ~120 us through device tensors.  Blocking; all buffers are HOST buffers; any out pointer may be NULL.
 * A handle is bound to the device current at creation and must not be used by two threads at once.
 *   stickers_host      [S]   uint8  in
 *   stickers_out_host  [S]   uint8  out
 *   onehot_u8_host     [D]   uint8  out  (the observation as 0/1 bytes, D = 147 / 480)
 *   solved_host              int    out  (1 = solved: done, reward +1; else -1) */
typedef struct cube_env_host cube_env_host_t;

int cube_env_host_create(int cube_size, int max_depth, cube_env_host_t** out);
int cube_env_host_destroy(cube_env_host_t* h);
/* step (cube_env.py:71-111): one face turn of the given cube */
int cube_env_host_step(cube_env_host_t* h, const uint8_t* stickers_host, int action, uint8_t* stickers_out_host,
                       uint8_t* onehot_u8_host, int* solved_host, void* stream);
/* reset (cube_env.py:56-69): `depth` <= max_depth moves applied to the solved cube */
int cube_env_host_scramble(cube_env_host_t* h, const uint8_t* moves_host, int depth, uint8_t* stickers_out_host,
                           uint8_t* onehot_u8_host, int* solved_host, void* stream);
/* sim_state_to_state / get_obs (cube_env.py:113-147) */
int cube_env_host_encode(cube_env_host_t* h, const uint8_t* stickers_host, uint8_t* onehot_u8_host, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CUBE_B200_H */
