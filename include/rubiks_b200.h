/*
 * rubiks_b200.h -- C ABI of librubiks_b200.so, the B200 (sm_100a) implementation of the
 * cube-dynamics hot path of peleiden/rl-rubiks.
 *
 * This is the drop-in boundary (SURVEY.md 8b): every entry point replaces one function (or one
 * fused group of functions) of the reference's `librubiks.cube` module API or of the hot part of
 * `Train.ADI_traindata` / `AStar.expand_batch` / `BFS.search`.  The citation after each
 * declaration is the reference file:line it replaces (paths relative to the reference root).
 *
 * Conventions
 *   - Plain C types only.  `rb_*` entry points take DEVICE pointers owned by the caller (e.g. the
 *     storage of a torch CUDA tensor) plus the CUDA stream to launch on (`rb_stream_t` is a
 *     `cudaStream_t`; 0 = legacy default stream).  They never allocate, free or synchronise.
 *     `rbh_*` entry points take HOST pointers, do their own staging + copies and return when the
 *     result is in the caller's host buffer.
 *   - Return value: RB_OK or an RB_ERR_* code; `rb_last_error()` gives a message for the calling
 *     thread.  The reference has no error API (IndexError from numpy on bad input); the Python
 *     mirror turns RB_ERR_RANGE into IndexError and everything else into RuntimeError.
 *   - rep: RB_REP_2024 = the 20x24 representation (state = int8[20], one-hot width 480);
 *     RB_REP_686 = the 6x8x6 representation (state = int8[6][8][6], one-hot width 288).
 *   - Action index a in [0,12) <-> (face = a / 2, direction = 1 - a % 2)   (librubiks/cube/cube.py:33-35).
 *     Where a function takes `faces` and `dirs`, `dirs` may be NULL: `faces` then holds action indices.
 *   - All state tensors are contiguous, row-major, in the reference's own layout.
 */
#ifndef RUBIKS_B200_H
#define RUBIKS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RB_OK              0
#define RB_ERR_BAD_ARG     1   /* null pointer, negative size, unknown rep / reward method */
#define RB_ERR_CUDA        2   /* a CUDA runtime call or launch failed */
#define RB_ERR_RANGE       3   /* rb_check_* found a face/dir/state value out of range */
#define RB_ERR_CAPACITY    4   /* hash set full / output buffer too small */

#define RB_REP_2024        0
#define RB_REP_686         1

#define RB_REWARD_PAPER      0  /* librubiks/train.py:292-296, 318-325 */
#define RB_REWARD_LAPANFIX   1
#define RB_REWARD_SCHULTZFIX 2
#define RB_REWARD_REWARD0    3

typedef void* rb_stream_t;      /* cudaStream_t */

/* ---- library ------------------------------------------------------------------------------ */
int         rb_version(void);
const char* rb_last_error(void);
/* Number of kernels this library has launched in the calling process (for bench accounting). */
int64_t     rb_launch_count(void);

/* ---- tables (librubiks/cube/maps.py:107-145 get_tensor_map; cube.py:311-326 constants) ------ */
/* Host-side copies of the tables the kernels stage in shared memory, for inspection/tests.
 * delta: int8[2][6][2][24] exactly as get_tensor_map returns it; lut: uint8[12][2][24] direct
 * form lut[a][kind][s] = s + delta[dir(a)][face(a)][kind][s]; perm686: uint8[12][48] gather
 * table new[slot] = old[perm[a][slot]] over the 48 sticker slots (slot = face*8 + ring index). */
int rb_get_delta_maps(int8_t* delta);
int rb_get_lut2024(uint8_t* lut);
int rb_get_perm686(uint8_t* perm);
/* The fused 2-move table of the fast scramble kernel (csrc/rb_scramble_macro.cuh): uint32[13*13][5], row index
 * a0 + 13 a1 (action 12 = identity), derived from the 20x24 LUT.  For inspection / CPU emulation tests. */
int rb_get_macro_table(uint32_t* rows);
/* The fused 3-move table of the same kernel's 3-moves-per-row variant: uint32[12*12*12][5], row index a0 + 12 a1 + 144 a2. */
int rb_get_macro3_table(uint32_t* rows);
/* The deduplicated form of that table the kernel stages in shared memory: elems uint32[1080][4], the distinct 16-byte parts
 * (selector words) of the rows; remap uint32[2372][2] = {twist|flip word, element index}.  remap index a0 + 12 a1 + 144 a2
 * (4-bit actions, up to 2355) stands for the row of the INVERSE moves (a0 ^ 1, a1 ^ 1, a2 ^ 1), invalid indices for element 0
 * with no twist or flip; index 2356 + a (a < 16) for the single inverse move a ^ 1 (a >= 12: element 0 again). */
int rb_get_macro3_dedup(uint32_t* elems, uint32_t* remap);
/* Sticker view used to render a 6x8x6 state from the 20x24 state of the same move sequence (fast 6x8x6 scramble):
 * corner_home uint8[8][3], corner_dst uint8[8][24][3], edge_home uint8[12][2], edge_dst uint8[12][24][2]: sticker k of a
 * cubie sits in 6x8x6 slot *_home[c][k] when solved and in slot *_dst[c][v][k] when the cubie's 20x24 value is v.
 * Derived by running both representations' tables side by side (cube.py:244-263 vs 330-361). */
int rb_get_stickers686(uint8_t* corner_home, uint8_t* corner_dst, uint8_t* edge_home, uint8_t* edge_dst);
/* get_solved (cube.py:58-83): writes int8[20] or int8[288] to a HOST buffer. */
int rb_get_solved(int rep, int8_t* state);

/* ---- single-step dynamics ---------------------------------------------------------------- */
/* multi_rotate (cube.py:49-52, 257-263, 349-361): out[i] = move(faces[i], dirs[i]) on states[i]. */
int rb_multi_rotate(int rep, const int8_t* states, const uint8_t* faces, const uint8_t* dirs,
                    int8_t* out, int64_t n, rb_stream_t stream);
/* multi_is_solved (cube.py:85-89): flags[i] = 1 iff states[i] equals the solved state. */
int rb_multi_is_solved(int rep, const int8_t* states, uint8_t* flags, int64_t n, rb_stream_t stream);
/* as_oh (cube.py:130-133, 265-277, 363-369): f32 [n][480] or [n][288], every element written. */
int rb_as_oh(int rep, const int8_t* states, float* oh, int64_t n, rb_stream_t stream);
/* as_correct (cube.py:135-137, 371-380): 6x8x6 only; oh f32 [n][288] -> f32 [n][6][8] of +-1. */
int rb_as_correct_686(const float* oh, float* out, int64_t n, rb_stream_t stream);
/* 12-neighbour expansion (cube.py:142-147 repeat_state + :179-184 iter_actions + multi_rotate, as used
 * at train.py:285 and agents.py:277-281): child i*12+a = action a on states[i].  Any of the three
 * outputs may be NULL: children int8 [12n][*shape], children_oh f32 [12n][W], solved uint8 [12n]. */
int rb_expand12(int rep, const int8_t* states, int8_t* children, float* children_oh,
                uint8_t* solved, int64_t n, rb_stream_t stream);
/* Range check used by the Python mirror to reproduce the reference's IndexError: returns
 * RB_ERR_RANGE if any face >= 6, dir >= 2 (or action >= 12 when dirs is NULL) or, for
 * RB_REP_2024 with states != NULL, any state value outside [0,24).  Synchronises the stream. */
int rb_check_range(int rep, const int8_t* states, int64_t n_states, const uint8_t* faces,
                   const uint8_t* dirs, int64_t n_actions, int32_t* scratch_dev, rb_stream_t stream);

/* ---- scramblers -------------------------------------------------------------------------- */
/* scramble (cube.py:206-216) for n cubes at once: applies `depth` host-drawn moves to each cube,
 * starting from `start` (int8 [n][*shape]) or from solved when start is NULL; writes the final states.
 * Action of cube i at move m is actions[i*stride_cube + m*stride_move] (action index, 0..11), so
 * both [n][depth] (stride_cube = depth, stride_move = 1) and [depth][n] layouts are accepted. */
int rb_scramble(int rep, const uint8_t* actions, int64_t stride_cube, int64_t stride_move,
                const int8_t* start, int8_t* out, int64_t n, int32_t depth, rb_stream_t stream);
/* sequence_scrambler (cube.py:218-234) with the random draw supplied by the caller:
 * faces/dirs uint8 [depth][games] (the reference's draw shape; dirs NULL => faces are action indices).
 * Emits every state of every game, game-major/depth-minor; with_solved != 0 emits the solved state
 * first and applies only rows 0..depth-2.  states int8 [games*depth][*shape], oh f32 [games*depth][W],
 * solved uint8 [games*depth]; each may be NULL. */
int rb_sequence_scramble(int rep, const uint8_t* faces, const uint8_t* dirs, int32_t games, int32_t depth,
                         int32_t with_solved, int8_t* states, float* oh, uint8_t* solved, rb_stream_t stream);

/* scramble with the random draw made ON the device (cube.py:206-211 for n cubes: `depth` moves per cube, every move uniform over
 * the 12 actions; SURVEY 8d C2 "generate on device from the same counter-based stream").  Cube i uses subsequence
 * first_cube + i of the Philox4x32-10 stream keyed by `seed` (csrc/rb_scramble_seeded.cuh defines word -> moves), so the result
 * for a cube does not depend on how the cubes are split over calls, streams or GPUs.  No action bytes are read: 20 (288) B per
 * cube leave the chip.  start: optional start states as for rb_scramble. */
int rb_scramble_seeded(int rep, uint64_t seed, uint64_t first_cube, const int8_t* start, int8_t* out, int64_t n,
                       int32_t depth, rb_stream_t stream);
/* The same stream written out as action indices, uint8 [n][depth]: what rb_scramble_seeded applied to cube i.  (Parity of the
 * seeded path = these bytes replayed through the reference's own rotate loop.) */
int rb_seeded_actions(uint64_t seed, uint64_t first_cube, uint8_t* actions, int64_t n, int32_t depth, rb_stream_t stream);
/* Packed actions: two moves per byte, p = a(2k) + 13 * a(2k+1), a second digit of 12 = "no move" (last byte of an odd-depth
 * row) -- the row index of the 2-move table (rb_get_macro_table).  packed uint8 [n][(depth + 1) / 2] -> actions uint8 [n][depth].
 * Halves the host->device bytes of a host-drawn scramble (rbh_scramble_packed). */
int rb_unpack_actions(const uint8_t* packed, uint8_t* actions, int64_t n, int32_t depth, rb_stream_t stream);

/* The same cube in the other representation (the two are isomorphic: cube.py:149-173 maps both to the 6x3x3 sticker view).
 * rb_as686: int8 [n][20] -> int8 [n][6][8][6].  rb_as2024: int8 [n][6][8][6] -> int8 [n][20]; ok (uint8 [n], may be NULL) is
 * cleared for rows that are not a reachable cube (their values are 255).  The batched A* keeps its stored states in the
 * 20-byte form whatever the caller's representation and renders 6x8x6 rows only for the value net's input. */
int rb_as686(const int8_t* states2024, int8_t* states686, int64_t n, rb_stream_t stream);
int rb_as2024(const int8_t* states686, int8_t* states2024, uint8_t* ok, int64_t n, rb_stream_t stream);

/* ---- ADI training batch (librubiks/train.py:256-339) --------------------------------------- */
/* Fused generator, train.py:277-296 in one launch: sequence scramble -> 12 children of every state ->
 * one-hot of states and of children -> solved flags of both.  n = games*depth.
 * Outputs (NULL to skip): states int8 [n][*shape]; oh_states f32 [n][W]; children int8 [12n][*shape];
 * children_oh f32 [12n][W]; solved_states uint8 [n]; solved_children uint8 [12n]. */
int rb_adi_generate(int rep, const uint8_t* faces, const uint8_t* dirs, int32_t games, int32_t depth,
                    int32_t with_solved, int8_t* states, float* oh_states, int8_t* children,
                    float* children_oh, uint8_t* solved_states, uint8_t* solved_children, rb_stream_t stream);

/* ---- bfloat16 one-hot variants ----------------------------------------------------------------
 * Same functions with the one-hot emitted as bfloat16 (raw bits in uint16_t; 0.0 and 1.0 -- and every int8 value of a
 * 6x8x6 state -- are exact in bf16, so the rows equal the f32 rows converted): half the HBM write traffic of the
 * write-bound emitters and the input dtype of a bf16 tensor-core forward of the value/policy net (model.py:131-141).
 * The reference emits f32 (cube.py:273-276, 368); these are an opt-in of the Python mirror (`as_oh(states, dtype=...)`,
 * `ADIGenerator(oh_dtype=...)`). */
int rb_as_oh_bf16(int rep, const int8_t* states, uint16_t* oh, int64_t n, rb_stream_t stream);
int rb_expand12_bf16(int rep, const int8_t* states, int8_t* children, uint16_t* children_oh,
                     uint8_t* solved, int64_t n, rb_stream_t stream);
int rb_sequence_scramble_bf16(int rep, const uint8_t* faces, const uint8_t* dirs, int32_t games, int32_t depth,
                              int32_t with_solved, int8_t* states, uint16_t* oh, uint8_t* solved, rb_stream_t stream);
int rb_adi_generate_bf16(int rep, const uint8_t* faces, const uint8_t* dirs, int32_t games, int32_t depth,
                         int32_t with_solved, int8_t* states, uint16_t* oh_states, int8_t* children,
                         uint16_t* children_oh, uint8_t* solved_states, uint8_t* solved_children, rb_stream_t stream);
/* Target assembly, train.py:292-296 + 313-325: values f32 [12n] are the net's outputs for the children;
 * rewards (+1 / 0 with reward0 for a solved child, -1 otherwise) are added in f32, the row argmax takes the
 * FIRST maximum (NaN counts as maximum, as torch.argmax), lapanfix zeroes targets of solved states,
 * schultzfix zeroes rows 0, depth, 2*depth, ...  policy int64 [n], value f32 [n]. */
int rb_adi_targets(const float* values, const uint8_t* solved_children, const uint8_t* solved_states,
                   int64_t n, int32_t depth, int32_t reward_method, int64_t* policy, float* value,
                   rb_stream_t stream);
/* rb_adi_targets and rb_adi_loss_weights in one launch (n = games*depth): train.py:313-333. */
int rb_adi_targets_weights(const float* values, const uint8_t* solved_children, const uint8_t* solved_states,
                           int32_t games, int32_t depth, int32_t reward_method, double alpha, double ws,
                           int64_t* policy, float* value, float* loss_weights, rb_stream_t stream);
/* Loss weights, train.py:329-333, evaluated in f64 and rounded to f32 like the reference:
 * ((1-alpha) w/ws + alpha/N)(ws+N), w = 1/(1 + i % depth), N = games*depth.  `ws` is the f64 sum of w the
 * caller obtained the reference's way (numpy pairwise sum; rb_adi_weight_sum restates it). */
double rb_adi_weight_sum(int32_t games, int32_t depth);
int rb_adi_loss_weights(float* out, int32_t games, int32_t depth, double alpha, double ws, rb_stream_t stream);

/* ---- search frontier: seen-set on the packed state (agents.py:103-121, 286-306, 517-526, 605-609) --- */
/* Open-addressing hash set keyed on the packed state, 128 bit: 20x24 -> 20 cubies x 5 bit = 100 bit;
 * 6x8x6 -> the 8 sticker colours of each face as a base-6 number (6^8 < 2^21), 6 x 21 = 126 bit, injective on
 * valid one-hot states (the only ones a cube can reach).
 * The table lives in caller-owned device memory of rb_hashset_bytes(capacity) bytes (32 per slot), 32-byte aligned; capacity
 * must be a power of two <= 2^30 (RB_ERR_CAPACITY above that).  The set maps state -> index (int32, 1-based in insertion order
 * like the reference's `indices` dict; 0 = absent).
 * Overflow: a batch that finds the table full cannot report it through the return value (nothing synchronises); it sets
 * *count_dev (and *n_new_dev) to -1, which every later batch on that counter preserves, and gives the dropped items index -1.
 * Keep the load factor <= 1/2 (the Python mirror grows the table with rb_hashset_rehash before a batch could exceed it). */
int64_t rb_hashset_bytes(int64_t capacity);
int rb_hashset_clear(void* table, int64_t capacity, rb_stream_t stream);
/* Growth: clears `dst` (dst_capacity >= src_capacity) and re-inserts every (state key, index) pair of `src`. */
int rb_hashset_rehash(void* src, int64_t src_capacity, void* dst, int64_t dst_capacity, rb_stream_t stream);
/* Batch insert with the reference's order semantics (agents.py:286-306): for states[0..n) in order,
 * seen[i] = state was in the set before this call; first[i] = i is the first occurrence of its state in this
 * batch; index[i] = index of the state after the call, new states (first & ~seen) numbered count+1, count+2, ...
 * in batch order.  `count_dev` (int32 on device) holds the set size and is updated; no host sync.
 * scratch: caller-owned device buffer of rb_hashset_scratch_bytes(n) bytes. */
int64_t rb_hashset_scratch_bytes(int64_t n);
int rb_hashset_insert_unique(int rep, void* table, int64_t capacity, const int8_t* states, int64_t n,
                             int32_t* count_dev, uint8_t* seen, uint8_t* first, int32_t* index,
                             void* scratch, rb_stream_t stream);
/* Lookup only (agents.py:606-607 `_complete_graph`): index[i] or 0 when absent.  scratch: as for insert
 * (needed for RB_REP_686 only; may be NULL for RB_REP_2024). */
int rb_hashset_lookup(int rep, const void* table, int64_t capacity, const int8_t* states, int64_t n,
                      int32_t* index, void* scratch, rb_stream_t stream);
/* One layer of breadth-first search (BFS.search agents.py:96-123 made layer-synchronous; the frontier part of
 * AStar.expand_batch agents.py:272-307): expands frontier[0..n) to 12n children, inserts them with
 * rb_hashset_insert_unique semantics and compacts the new ones, in batch order, to
 * next_frontier (int8 [<=12n][*shape]) with their parent position and action (parent int32, action uint8;
 * NULL to skip) and solved flag.  n_new_dev (int32, device) receives the number of new states. */
int rb_frontier_expand(int rep, void* table, int64_t capacity, const int8_t* frontier, int64_t n,
                       int32_t* count_dev, int8_t* next_frontier, int32_t* parent, uint8_t* action,
                       uint8_t* solved, uint8_t* seen, uint8_t* first, int32_t* index, int32_t* n_new_dev,
                       void* scratch, rb_stream_t stream);
/* The same with the frontier's size on the DEVICE: frontier holds *n_dev (<= n_max) states; buffers and scratch are sized for
 * n_max.  Lets a caller enqueue consecutive layers (n_dev of layer d+1 = n_new_dev of layer d) without a host round trip while
 * the upper bound 12^d is small.  20x24 representation; no per-item seen / first / index outputs. */
int rb_frontier_expand_dev(int rep, void* table, int64_t capacity, const int8_t* frontier, int64_t n_max, const int32_t* n_dev,
                           int32_t* count_dev, int8_t* next_frontier, int32_t* parent, uint8_t* action, uint8_t* solved,
                           int32_t* n_new_dev, void* scratch, rb_stream_t stream);
/* `layers` consecutive rb_frontier_expand_dev calls enqueued by one host call: layer d reads its frontier from buf_a (d even) or
 * buf_b (d odd) and writes the next one into the other; sizes_dev[0] = n0 on entry, sizes_dev[d + 1] receives the number of new
 * states of layer d.  Buffers hold n0 * 12^layers states, scratch is rb_frontier_scratch_bytes(rep, n0 * 12^(layers-1)). */
int rb_frontier_expand_chain(int rep, void* table, int64_t capacity, int8_t* buf_a, int8_t* buf_b, int64_t n0, int32_t layers,
                             int32_t* sizes_dev, int32_t* count_dev, void* scratch, rb_stream_t stream);
int64_t rb_frontier_scratch_bytes(int rep, int64_t n);

/* ---- batched weighted A* on the device (agents.py:221-367 for K cubes at once; 20x24 representation) -----------------
 * K independent searches advance in lockstep.  Every buffer is caller-owned device memory; [K][M] arrays are indexed by the
 * reference's state index (1-based, 0 unused), M >= max_states + 1.  One step of all searches =
 *   rb_astar_expand  (pop the <= N cheapest open states per search in heapq order, expand, dedup, number and store the new
 *                     states, append them to one contiguous batch for the value net)
 *   [caller: one-hot + value net on new_states[0 .. *n_new_total)]
 *   rb_astar_commit  (costs lambda*G - value into the open list, the two relaxation passes, bookkeeping).
 * A search stops when it generated the solved state (won[s] = 1, solved_index[s]) or when count[s] + 12 N > max_states. */
typedef struct rb_astar_view {
	int32_t K, M, N;              /* searches, rows per search, expansions per step (N <= 1024) */
	int8_t*  states;              /* [K][M][20] */
	double*  G;                   /* [K][M] path cost upper bound */
	int32_t* parents;             /* [K][M] */
	uint8_t* parent_actions;      /* [K][M] */
	double*  cost;                /* [K][M] the (cost, index) heap entry of a state, valid while in_open */
	uint8_t* in_open;             /* [K][M] */
	int32_t* count;               /* [K] states stored (= len(agent)) */
	int32_t* n_sel;               /* [K] parents popped in the running step */
	int32_t* sel;                 /* [K][N] their indices, ascending (cost, index) */
	uint8_t* won;                 /* [K] */
	int32_t* solved_index;        /* [K] */
	void*    table;               /* shared seen-set, rb_hashset_bytes(capacity) bytes, cleared with rb_hashset_clear */
	int64_t  capacity;            /* power of two, >= 2 K M (checked: RB_ERR_CAPACITY below that) */
	void*    scratch;             /* rb_astar_scratch_bytes(K, N) bytes */
} rb_astar_view;
int64_t rb_astar_scratch_bytes(int32_t K, int32_t N);
/* roots int8 [K][20]: state 1 of every search (a solved root marks the search won at once, agents.py:230). */
int rb_astar_init(const rb_astar_view* v, const int8_t* roots, rb_stream_t stream);
/* new_states int8 [K*12N][20], new_search / new_index int32 [K*12N]; n_new_total, n_active: int32 on the device. */
int rb_astar_expand(const rb_astar_view* v, int64_t max_states, int8_t* new_states, int32_t* new_search,
                    int32_t* new_index, int32_t* n_new_total, int32_t* n_active, rb_stream_t stream);
/* values f32 [*n_new_total]: the value net's output for new_states, in order. */
int rb_astar_commit(const rb_astar_view* v, const float* values, double lambda, const int32_t* new_search,
                    const int32_t* new_index, const int32_t* n_new_total, rb_stream_t stream);

/* ---- batched breadth-first search on the device (BFS.search agents.py:96-123 for K cubes at once; 20x24 representation) ---
 * K independent searches advance in lockstep.  Every buffer is caller-owned device memory; [K][M] arrays are indexed by the
 * reference's state index (1-based in discovery order, 0 unused), M >= max_states + 1.  The FIFO of a search is its stored
 * states: a step pops the next min(N, count - head + 1) of them, tests the budget `len(states) < max_states` before every
 * pop (agents.py:104), dedups the children against the search's own states, numbers the new ones in (parent, action) order
 * and stops the search at the first solved new child under a popped parent (not recorded, agents.py:112-118).  States
 * numbered >= max_states are never popped and are not stored.  A search that runs out of budget stops unsolved. */
typedef struct rb_bfs_view {
	int32_t K, M, N;              /* searches (<= 65535), rows per search, pops per search and step */
	int8_t*  states;              /* [K][M][20] */
	int32_t* parents;             /* [K][M] FIFO index of the state's parent (agents.py:117) */
	uint8_t* parent_actions;      /* [K][M] */
	int32_t* count;               /* [K] states recorded (= len(agent); 0 for a solved start) */
	int32_t* head;                /* [K] FIFO index of the next pop */
	uint8_t* won;                 /* [K] */
	uint8_t* done;                /* [K] */
	int32_t* solved_parent;       /* [K] FIFO index of the solved child's parent (0: solved start) */
	uint8_t* solved_action;       /* [K] action from that parent to the solved child */
	void*    table;               /* shared seen-set, rb_hashset_bytes(capacity) bytes, cleared with rb_hashset_clear */
	int64_t  capacity;            /* power of two, >= 2 K (M + 12 N) (checked: RB_ERR_CAPACITY below that) */
	void*    scratch;             /* rb_bfs_scratch_bytes(K, N) bytes */
} rb_bfs_view;
/* agents.py:96-123: scratch bytes of a view with K searches and N pops per step. */
int64_t rb_bfs_scratch_bytes(int32_t K, int32_t N);
/* agents.py:99-103: roots int8 [K][20] become state 1 of every search (a solved root: found, len 0). */
int rb_bfs_init(const rb_bfs_view* v, const int8_t* roots, rb_stream_t stream);
/* agents.py:104-121, one step of every search: up to N pops each.  n_active (int32, device) receives the number of searches
 * still running after the step; it is the one value a caller reads per step. */
int rb_bfs_step(const rb_bfs_view* v, int64_t max_states, int32_t* n_active, rb_stream_t stream);
/* agents.py:112-116: action queue of every search, uint8 [K][L]; lengths int32 [K] (0 when not found or solved at the start,
 * -1 when the queue is longer than L). */
int rb_bfs_paths(const rb_bfs_view* v, uint8_t* queues, int32_t* lengths, int32_t L, rb_stream_t stream);

/* ---- host-buffer entry points (end-to-end: H2D + kernels + D2H inside the call) --------------- */
/* rb_scramble on host buffers; actions uint8 [n][depth] (cube-major), out int8 [n][*shape].  Copies are
 * chunked and double-buffered on internal streams; pinned host memory makes them asynchronous. */
int rbh_scramble(int rep, const uint8_t* actions, int8_t* out, int64_t n, int32_t depth);
/* rbh_scramble with packed actions (see rb_unpack_actions): half the bytes over PCIe. */
int rbh_scramble_packed(int rep, const uint8_t* packed, int8_t* out, int64_t n, int32_t depth);
/* rb_scramble_seeded into a host buffer: nothing but the seed goes to the device, 20 (288) B per cube come back. */
int rbh_scramble_seeded(int rep, uint64_t seed, uint64_t first_cube, int8_t* out, int64_t n, int32_t depth);
/* multi_rotate on host buffers (the reference's own call shape: numpy in, numpy out). */
int rbh_multi_rotate(int rep, const int8_t* states, const uint8_t* faces, const uint8_t* dirs,
                     int8_t* out, int64_t n);
/* Pinned host buffers for the rbh_* calls (optional: any host pointer works, pinned ones copy asynchronously).  huge != 0 asks
 * for transparent huge pages before pinning.  NULL on failure (rb_last_error). */
void* rbh_host_alloc(int64_t bytes, int huge);
int   rbh_host_free(void* ptr, int64_t bytes);
/* Release cached device staging buffers held by the rbh_* entry points. */
int rbh_release(void);

#ifdef __cplusplus
}
#endif
#endif /* RUBIKS_B200_H */
