// librubiks_b200.so -- C ABI (include/rubiks_b200.h) over the sm_100a kernels.  Single translation unit.
#include <sys/mman.h>
#include "rb_common.cuh"
#include "rb_tables.cuh"
#include "rb_cube2024.cuh"
#include "rb_scramble_macro.cuh"
#include "rb_scramble_seeded.cuh"
#include "rb_cube686.cuh"
#include "rb_adi.cuh"
#include "rb_frontier.cuh"
#include "rb_search.cuh"
#include "rb_astar.cuh"
#include "rb_bfs.cuh"
#include "rb_host.cuh"

#define RB_INIT()                                   \
	do {                                            \
		int rc_ = rbt::ensure_device();             \
		if (rc_ != RB_OK) return rc_;               \
	} while (0)

static inline bool aligned(const void* p, uintptr_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; }
static inline cudaStream_t S(rb_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }
static inline bool rep_ok(int rep) { return rep == RB_REP_2024 || rep == RB_REP_686; }

extern "C" {

int rb_version(void) { return 100; }
const char* rb_last_error(void) { return g_rb_err; }
int64_t rb_launch_count(void) { return g_rb_launches.load(); }

int rb_get_delta_maps(int8_t* delta) {
	RB_REQUIRE(delta, "null output");
	memcpy(delta, rbt::host().delta, sizeof(rbt::host().delta));
	return RB_OK;
}
int rb_get_lut2024(uint8_t* lut) {
	RB_REQUIRE(lut, "null output");
	memcpy(lut, rbt::host().lut, sizeof(rbt::host().lut));
	return RB_OK;
}
int rb_get_perm686(uint8_t* perm) {
	RB_REQUIRE(perm, "null output");
	memcpy(perm, rbt::host().perm686, sizeof(rbt::host().perm686));
	return RB_OK;
}
int rb_get_macro_table(uint32_t* rows) {
	RB_REQUIRE(rows, "null output");
	const rbs::Host& h = rbs::host();
	if (!h.ok) return rb_fail(RB_ERR_BAD_ARG, "macro-move tables: a host check failed (twist additivity or the deduplicated 3-move table)%s%s");
	memcpy(rows, h.rows, sizeof(uint32_t) * rbs::kRows * rbs::kRowWords);
	return RB_OK;
}
int rb_get_macro3_table(uint32_t* rows) {
	RB_REQUIRE(rows, "null output");
	const rbs::Host& h = rbs::host();
	if (!h.ok) return rb_fail(RB_ERR_BAD_ARG, "macro-move tables: a host check failed (twist additivity or the deduplicated 3-move table)%s%s");
	memcpy(rows, h.rows3, sizeof(uint32_t) * rbs::kRows3 * rbs::kRowWords);
	return RB_OK;
}
int rb_get_macro3_dedup(uint32_t* elems, uint32_t* remap) {
	RB_REQUIRE(elems && remap, "null output");
	const rbs::Host& h = rbs::host();
	if (!h.ok) return rb_fail(RB_ERR_BAD_ARG, "macro-move tables: a host check failed (twist additivity or the deduplicated 3-move table)%s%s");
	memcpy(elems, h.elems3, sizeof(h.elems3));
	memcpy(remap, h.remap3, sizeof(h.remap3));
	return RB_OK;
}
int rb_get_stickers686(uint8_t* corner_home, uint8_t* corner_dst, uint8_t* edge_home, uint8_t* edge_dst) {
	RB_REQUIRE(corner_home && corner_dst && edge_home && edge_dst, "null output");
	const rbt::Tables& t = rbt::host();
	if (!t.stickers_ok) return rb_fail(RB_ERR_BAD_ARG, "sticker tables: the 20x24 and 6x8x6 move tables disagree%s%s");
	memcpy(corner_home, t.corner_home, sizeof(t.corner_home));
	memcpy(corner_dst, t.corner_dst, sizeof(t.corner_dst));
	memcpy(edge_home, t.edge_home, sizeof(t.edge_home));
	memcpy(edge_dst, t.edge_dst, sizeof(t.edge_dst));
	return RB_OK;
}
int rb_get_solved(int rep, int8_t* state) {
	RB_REQUIRE(state && rep_ok(rep), "bad argument");
	if (rep == RB_REP_2024) memcpy(state, rbt::host().solved2024, 20);
	else memcpy(state, rbt::host().solved686, 288);
	return RB_OK;
}

int rb_multi_rotate(int rep, const int8_t* states, const uint8_t* faces, const uint8_t* dirs, int8_t* out,
                    int64_t n, rb_stream_t stream) {
	RB_REQUIRE(rep_ok(rep) && n >= 0, "bad rep or size");
	if (n == 0) return RB_OK;
	RB_REQUIRE(states && faces && out, "null pointer");
	RB_INIT();
	if (rep == RB_REP_2024) {
		if (aligned(states, 4) && aligned(out, 4))
			rb2024::k_multi_rotate<<<rb_grid(n, 256, 5), rb2024::kThreads, 0, S(stream)>>>(states, faces, dirs, out, n);
		else
			rb2024::k_multi_rotate_any<<<rb_grid(n, rb2024::kTile, 2), rb2024::kThreads, 0, S(stream)>>>(states, faces, dirs, out, n);
		RB_LAUNCHED("multi_rotate_2024");
	} else {
		RB_REQUIRE(aligned(states, 4) && aligned(out, 4), "6x8x6 states must be 4-byte aligned");
		rb686::k_multi_rotate<<<rb_grid(n, rb686::kMrStates * rb686::kWarps, 5), rb686::kThreads, 0, S(stream)>>>(states, faces, dirs, out, n);
		RB_LAUNCHED("multi_rotate_686");
	}
	return RB_OK;
}

int rb_multi_is_solved(int rep, const int8_t* states, uint8_t* flags, int64_t n, rb_stream_t stream) {
	RB_REQUIRE(rep_ok(rep) && n >= 0, "bad rep or size");
	if (n == 0) return RB_OK;
	RB_REQUIRE(states && flags, "null pointer");
	RB_INIT();
	if (rep == RB_REP_2024) {
		if (aligned(states, 4))
			rb2024::k_is_solved<<<rb_grid(n, 256, 8), rb2024::kThreads, 0, S(stream)>>>(states, flags, n);
		else
			rb2024::k_is_solved_any<<<rb_grid(n, rb2024::kTile, 2), rb2024::kThreads, 0, S(stream)>>>(states, flags, n);
		RB_LAUNCHED("is_solved_2024");
	} else {
		RB_REQUIRE(aligned(states, 4), "6x8x6 states must be 4-byte aligned");
		rb686::k_is_solved<<<rb_grid(n, 4 * rb686::kWarps, 8), rb686::kThreads, 0, S(stream)>>>(states, flags, n);
		RB_LAUNCHED("is_solved_686");
	}
	return RB_OK;
}

// OH = float (the reference's one-hot dtype) or rb_bf16 (raw bfloat16 bits: the same 0/1 values, half the bytes)
extern "C++" {
template <typename OH>
static int as_oh_impl(int rep, const int8_t* states, OH* oh, int64_t n, rb_stream_t stream) {
	RB_REQUIRE(rep_ok(rep) && n >= 0, "bad rep or size");
	if (n == 0) return RB_OK;
	RB_REQUIRE(states && oh, "null pointer");
	RB_REQUIRE(aligned(oh, 16), "one-hot output must be 16-byte aligned");
	RB_INIT();
	const int64_t esz = sizeof(OH);
	if (rep == RB_REP_2024) {
		if (aligned(states, 4))
			rb2024::k_as_oh<OH><<<rb_grid(n, rb2024::kThreads, kGridUncapped), rb2024::kThreads, 0, S(stream)>>>(states, oh, n, rb_store_policy(n * 480 * esz));
		else
			rb2024::k_as_oh_any<OH><<<rb_grid(n, 8, kGridUncapped), rb2024::kThreads, 0, S(stream)>>>(states, oh, n, rb_store_policy(n * 480 * esz));
		RB_LAUNCHED("as_oh_2024");
	} else {
		RB_REQUIRE(aligned(states, 4), "6x8x6 states must be 4-byte aligned");
		rb686::k_as_oh<OH><<<rb_grid(n * 72, rb686::kThreads * 8, kGridUncapped), rb686::kThreads, 0, S(stream)>>>(states, oh, n * 72, rb_store_policy(n * 288 * esz));
		RB_LAUNCHED("as_oh_686");
	}
	return RB_OK;
}
}  // extern "C++"
int rb_as_oh(int rep, const int8_t* states, float* oh, int64_t n, rb_stream_t stream) { return as_oh_impl<float>(rep, states, oh, n, stream); }
int rb_as_oh_bf16(int rep, const int8_t* states, uint16_t* oh, int64_t n, rb_stream_t stream) { return as_oh_impl<uint16_t>(rep, states, oh, n, stream); }

int rb_as_correct_686(const float* oh, float* out, int64_t n, rb_stream_t stream) {
	RB_REQUIRE(n >= 0, "bad size");
	if (n == 0) return RB_OK;
	RB_REQUIRE(oh && out && aligned(oh, 8), "null or misaligned pointer");
	RB_INIT();
	rb686::k_as_correct<<<rb_grid(n * 48, rb686::kThreads, 8), rb686::kThreads, 0, S(stream)>>>(oh, out, n * 48);
	RB_LAUNCHED("as_correct_686");
	return RB_OK;
}

extern "C++" {
template <typename OH>
static int expand12_impl(int rep, const int8_t* states, int8_t* children, OH* children_oh, uint8_t* solved, int64_t n,
                         rb_stream_t stream) {
	const int64_t esz = sizeof(OH);
	RB_REQUIRE(rep_ok(rep) && n >= 0, "bad rep or size");
	if (n == 0) return RB_OK;
	RB_REQUIRE(states && (children || children_oh || solved), "null pointer");
	RB_REQUIRE(aligned(children_oh, 16), "one-hot output must be 16-byte aligned");
	RB_INIT();
	if (rep == RB_REP_2024) {
		if (!children_oh && aligned(states, 4) && aligned(children, 16) && aligned(solved, 4))
			rb2024::k_expand12_states<<<rb_grid(n, rb2024::kExpThreads, kGridUncapped), rb2024::kExpThreads, 0, S(stream)>>>(states, children, solved, n, rb_store_policy(n * 240));
		else
			rb2024::k_expand12<OH><<<rb_grid(n, 8, kGridUncapped), rb2024::kThreads, 0, S(stream)>>>(states, children, children_oh, solved, n,
			                                                                                 rb_store_policy(children_oh ? n * 12 * 480 * esz : n * 240));
		RB_LAUNCHED("expand12_2024");
	} else {
		RB_REQUIRE(aligned(states, 16) && aligned(children, 16), "6x8x6 states must be 16-byte aligned");
		if (!children_oh && !solved)
			rb686::k_expand12_states<<<rb_grid(n, rb686::kWarps, 32), rb686::kThreads, 0, S(stream)>>>(states, children, n);
		else
			rb686::k_expand12<OH><<<rb_grid(n, rb686::kWarps, kGridUncapped), rb686::kThreads, 0, S(stream)>>>(states, children, children_oh, solved, n,
			                                                                                     rb_store_policy(n * 12 * (children_oh ? 288 * (esz + 1) : 288)));
		RB_LAUNCHED("expand12_686");
	}
	return RB_OK;
}
}  // extern "C++"
int rb_expand12(int rep, const int8_t* states, int8_t* children, float* children_oh, uint8_t* solved, int64_t n, rb_stream_t stream) {
	return expand12_impl<float>(rep, states, children, children_oh, solved, n, stream);
}
int rb_expand12_bf16(int rep, const int8_t* states, int8_t* children, uint16_t* children_oh, uint8_t* solved, int64_t n, rb_stream_t stream) {
	return expand12_impl<uint16_t>(rep, states, children, children_oh, solved, n, stream);
}

// The rbs:: scramble kernels leave each cube's net 20x24 state at pitch 20, or parked at the head of its 6x8x6 output row; the
// start state then goes in front of it (20x24: k_compose) or is rendered through it (6x8x6: one gather of its sticker records).
static int scramble_pitch(int rep) { return rep == RB_REP_2024 ? 20 : rb686::kStateBytes; }
static int scramble_finish(int rep, const int8_t* start, int8_t* out, int64_t n, cudaStream_t st) {
	if (rep == RB_REP_2024) {
		if (!start) return RB_OK;
		rb2024::k_compose<<<rb_grid(n, 8, 8), rb2024::kThreads, 0, st>>>(out, start, n);   // start, then the sequence
		RB_LAUNCHED("compose_2024");
		return RB_OK;
	}
	rb686::k_render_from2024<<<rb_grid((n + 31) / 32, rb686::kWarps, 8), rb686::kThreads, 0, st>>>(out, start, n);
	RB_LAUNCHED("render_686");
	return RB_OK;
}

int rb_scramble(int rep, const uint8_t* actions, int64_t stride_cube, int64_t stride_move, const int8_t* start,
                int8_t* out, int64_t n, int32_t depth, rb_stream_t stream) {
	RB_REQUIRE(rep_ok(rep) && n >= 0 && depth >= 0, "bad rep or size");
	if (n == 0) return RB_OK;
	RB_REQUIRE(out && (actions || depth == 0), "null pointer");
	RB_INIT();
	if (rep != RB_REP_2024) RB_REQUIRE(aligned(out, 16) && aligned(start, 16), "6x8x6 states must be 16-byte aligned");
	if (depth > 0 && start != out && (rep == RB_REP_2024 || rbt::host().stickers_ok)) {
		// slot-major macro-move kernels: cube-major actions [n][depth], or move-major [depth][n] -- the reference's draw shape
		// (cube.py:226-227) -- by 2-D tensor copies and in-register transposes
		const bool cube_major = stride_move == 1 && stride_cube == depth && aligned(actions, 16) && rbs::warps_for(n, depth) > 0;
		if (cube_major || (stride_cube == 1 && stride_move == n && rbs::can_transposed(actions, n, depth) && rbs::quads_for(n, depth) > 0)) {
			const int rc = cube_major ? rbs::launch(actions, out, n, depth, S(stream), scramble_pitch(rep))
			                          : rbs::launch_mm(actions, out, n, depth, S(stream), scramble_pitch(rep));
			return rc != RB_OK ? rc : scramble_finish(rep, start, out, n, S(stream));
		}
	}
	if (rep == RB_REP_2024) {
		rb2024::k_scramble<<<rb_grid(n, rb2024::kThreads, 8), rb2024::kThreads, 0, S(stream)>>>(
			actions, stride_cube, stride_move, start, out, n, depth);
		RB_LAUNCHED("scramble_2024");
	} else {
		rb686::k_scramble<<<rb_grid(n, rb686::kWarps, 6), rb686::kThreads, 0, S(stream)>>>(
			actions, stride_cube, stride_move, start, out, n, depth);
		RB_LAUNCHED("scramble_686");
	}
	return RB_OK;
}

static int sequence_chunk(int64_t games, int depth, int units_per_sm) {
	// (game, chunk of positions) units per SM -- a unit replays its game's prefix to reach its chunk, so finer units balance the
	// grid better but replay more.  Measured (profiles/r2g_grid_sweep.txt): the 20x24 ADI generator (13 one-hot rows = 25 kB of
	// stores per position against at most `depth` byte lookups per lane of replay) wants one position per unit (1024 per SM;
	// 1000 x 25: 0.117 -> 0.111 ms, 7500 x 30 with bf16 rows 0.498 -> 0.461 ms); the 20x24 sequence with one one-hot row per position
	// 256 per SM (7500 x 30: 0.084 -> 0.074 ms; 1024 per SM: 0.096 ms); everything else 64.  RB_SEQ_UNITS_PER_SM overrides the ADI value.
	int64_t target_units = (int64_t)RB_NUM_SMS * units_per_sm;
	int64_t chunks_per_game = (target_units + games - 1) / games;
	if (chunks_per_game < 1) chunks_per_game = 1;
	if (chunks_per_game > depth) chunks_per_game = depth;
	return (int)((depth + chunks_per_game - 1) / chunks_per_game);
}
static int sequence_units_per_sm(int rep, bool with_children, bool with_oh) {
	static const int adi_per_sm = [] { const char* e = getenv("RB_SEQ_UNITS_PER_SM"); const int v = e ? atoi(e) : 1024; return v > 0 ? v : 1024; }();
	if (rep != RB_REP_2024) return 64;
	return with_children ? adi_per_sm : (with_oh ? 256 : 64);
}

extern "C++" {
template <typename OH>
static int launch_sequence(int rep, bool with_children, const uint8_t* faces, const uint8_t* dirs, int32_t games,
                           int32_t depth, int32_t with_solved, int8_t* states, OH* oh, uint8_t* solved_states,
                           int8_t* children, OH* children_oh, uint8_t* solved_children, rb_stream_t stream) {
	const int64_t esz = sizeof(OH);
	RB_REQUIRE(rep_ok(rep) && games >= 0 && depth >= 0, "bad rep or size");
	if (games == 0 || depth == 0) return RB_OK;
	RB_REQUIRE(faces || (depth == 1 && with_solved), "null action pointer");
	RB_REQUIRE(aligned(oh, 16) && aligned(children_oh, 16), "one-hot outputs must be 16-byte aligned");
	RB_INIT();
	const int ws = with_solved ? 1 : 0;
	const int chunk = sequence_chunk(games, depth, sequence_units_per_sm(rep, with_children, oh != nullptr));
	const int64_t units = (int64_t)games * ((depth + chunk - 1) / chunk);
	const int64_t rows = (int64_t)games * depth * (with_children ? 13 : 1);
	const int pol = rb_store_policy(rows * (rep == RB_REP_2024 ? ((oh || children_oh) ? 480 * esz : 20) : ((oh || children_oh) ? 288 * (esz + 1) : 288)));
	if (rep == RB_REP_2024 && !with_children && !oh && aligned(states, 4)) {
		// states / flags only: thread per game, register LUT, staged coalesced output
		rb2024::k_sequence_states<<<rb_grid(games, rb2024::kThreads, 24), rb2024::kThreads, 0, S(stream)>>>(faces, dirs, games, depth, ws,
		                                                                                             states, solved_states);
		RB_LAUNCHED("sequence_states_2024");
	} else if (rep == RB_REP_2024) {
		const int grid = rb_grid(units, 8, kGridUncapped);
		if (with_children)
			rb2024::k_sequence<true, OH><<<grid, rb2024::kThreads, 0, S(stream)>>>(faces, dirs, games, depth, ws, chunk, states, oh,
			                                                                   solved_states, children, children_oh, solved_children, pol);
		else
			rb2024::k_sequence<false, OH><<<grid, rb2024::kThreads, 0, S(stream)>>>(faces, dirs, games, depth, ws, chunk, states, oh,
			                                                                    solved_states, nullptr, (OH*)nullptr, nullptr, pol);
		RB_LAUNCHED("sequence_2024");
	} else {
		RB_REQUIRE(aligned(states, 16) && aligned(children, 16), "6x8x6 states must be 16-byte aligned");
		const int grid = rb_grid(units, rb686::kWarps, 6);
		if (with_children)
			rb686::k_sequence<true, OH><<<grid, rb686::kThreads, 0, S(stream)>>>(faces, dirs, games, depth, ws, chunk, states, oh,
			                                                                  solved_states, children, children_oh, solved_children, pol);
		else
			rb686::k_sequence<false, OH><<<grid, rb686::kThreads, 0, S(stream)>>>(faces, dirs, games, depth, ws, chunk, states, oh,
			                                                                   solved_states, nullptr, (OH*)nullptr, nullptr, pol);
		RB_LAUNCHED("sequence_686");
	}
	return RB_OK;
}
}  // extern "C++"

int rb_sequence_scramble(int rep, const uint8_t* faces, const uint8_t* dirs, int32_t games, int32_t depth,
                         int32_t with_solved, int8_t* states, float* oh, uint8_t* solved, rb_stream_t stream) {
	return launch_sequence<float>(rep, false, faces, dirs, games, depth, with_solved, states, oh, solved, nullptr, nullptr, nullptr, stream);
}
int rb_sequence_scramble_bf16(int rep, const uint8_t* faces, const uint8_t* dirs, int32_t games, int32_t depth,
                              int32_t with_solved, int8_t* states, uint16_t* oh, uint8_t* solved, rb_stream_t stream) {
	return launch_sequence<uint16_t>(rep, false, faces, dirs, games, depth, with_solved, states, oh, solved, nullptr, nullptr, nullptr, stream);
}

int rb_adi_generate(int rep, const uint8_t* faces, const uint8_t* dirs, int32_t games, int32_t depth, int32_t with_solved,
                    int8_t* states, float* oh_states, int8_t* children, float* children_oh, uint8_t* solved_states,
                    uint8_t* solved_children, rb_stream_t stream) {
	return launch_sequence<float>(rep, true, faces, dirs, games, depth, with_solved, states, oh_states, solved_states, children,
	                              children_oh, solved_children, stream);
}
int rb_adi_generate_bf16(int rep, const uint8_t* faces, const uint8_t* dirs, int32_t games, int32_t depth, int32_t with_solved,
                         int8_t* states, uint16_t* oh_states, int8_t* children, uint16_t* children_oh, uint8_t* solved_states,
                         uint8_t* solved_children, rb_stream_t stream) {
	return launch_sequence<uint16_t>(rep, true, faces, dirs, games, depth, with_solved, states, oh_states, solved_states, children,
	                                 children_oh, solved_children, stream);
}

static int adi_targets_impl(const float* values, const uint8_t* solved_children, const uint8_t* solved_states, int64_t n,
                            int32_t depth, int32_t reward_method, int64_t* policy, float* value, float* weights, double alpha,
                            double ws, rb_stream_t stream) {
	RB_REQUIRE(n >= 0 && depth > 0, "bad size");
	RB_REQUIRE(reward_method >= RB_REWARD_PAPER && reward_method <= RB_REWARD_REWARD0, "unknown reward method");
	if (n == 0) return RB_OK;
	RB_REQUIRE(values && solved_children && policy && value, "null pointer");
	RB_REQUIRE(reward_method != RB_REWARD_LAPANFIX || solved_states, "lapanfix needs solved_states");
	RB_REQUIRE(aligned(values, 16) && aligned(solved_children, 4), "values must be 16-byte and flags 4-byte aligned");
	rbadi::k_targets<<<rb_grid(n, rbadi::kThreads, 8), rbadi::kThreads, 0, S(stream)>>>(values, solved_children, solved_states, n,
	                                                                             depth, reward_method, policy, value, weights, alpha, ws);
	RB_LAUNCHED("adi_targets");
	return RB_OK;
}

int rb_adi_targets(const float* values, const uint8_t* solved_children, const uint8_t* solved_states, int64_t n,
                   int32_t depth, int32_t reward_method, int64_t* policy, float* value, rb_stream_t stream) {
	return adi_targets_impl(values, solved_children, solved_states, n, depth, reward_method, policy, value, nullptr, 0.0, 1.0, stream);
}

int rb_adi_targets_weights(const float* values, const uint8_t* solved_children, const uint8_t* solved_states, int32_t games,
                           int32_t depth, int32_t reward_method, double alpha, double ws, int64_t* policy, float* value,
                           float* loss_weights, rb_stream_t stream) {
	RB_REQUIRE(games >= 0 && loss_weights, "bad size or null loss_weights");
	return adi_targets_impl(values, solved_children, solved_states, (int64_t)games * depth, depth, reward_method, policy, value,
	                        loss_weights, alpha, ws, stream);
}

double rb_adi_weight_sum(int32_t games, int32_t depth) {
	if (games <= 0 || depth <= 0) return 0.0;
	const int64_t n = (int64_t)games * depth;
	double* w = new double[n];
	for (int64_t i = 0; i < n; ++i) w[i] = 1.0 / (double)(1 + i % depth);
	const double s = rbadi::pairwise_sum(w, n);
	delete[] w;
	return s;
}

int rb_adi_loss_weights(float* out, int32_t games, int32_t depth, double alpha, double ws, rb_stream_t stream) {
	RB_REQUIRE(games >= 0 && depth >= 0, "bad size");
	const int64_t n = (int64_t)games * depth;
	if (n == 0) return RB_OK;
	RB_REQUIRE(out, "null pointer");
	rbadi::k_loss_weights<<<rb_grid(n, rbadi::kThreads, 8), rbadi::kThreads, 0, S(stream)>>>(out, n, depth, alpha, ws);
	RB_LAUNCHED("adi_loss_weights");
	return RB_OK;
}

// ---- search frontier ----------------------------------------------------------------------------------------
int64_t rb_hashset_bytes(int64_t capacity) { return capacity > 0 ? capacity * (int64_t)sizeof(rbf::Slot) : 0; }

static bool pow2(int64_t x) { return x > 0 && (x & (x - 1)) == 0; }
// a table the kernels can address: power-of-two capacity, slot numbers in 30 bits, 32-byte aligned slots
#define RB_REQUIRE_TABLE(table, capacity)                                                                              \
	do {                                                                                                               \
		RB_REQUIRE((table) && pow2(capacity) && aligned((table), 32), "table must be 32-byte aligned with a power-of-two capacity"); \
		if ((capacity) > rbf::kMaxCapacity) return rb_fail(RB_ERR_CAPACITY, "hash set capacity above 2^30 slots is not supported%s%s"); \
	} while (0)

int rb_hashset_clear(void* table, int64_t capacity, rb_stream_t stream) {
	RB_REQUIRE_TABLE(table, capacity);
	rbf::k_clear<<<rb_grid(2 * capacity, rbf::kThreads * 4, kGridUncapped), rbf::kThreads, 0, S(stream)>>>(table, capacity);
	RB_LAUNCHED("hashset_clear");
	return RB_OK;
}

int rb_hashset_rehash(void* src, int64_t src_capacity, void* dst, int64_t dst_capacity, rb_stream_t stream) {
	RB_REQUIRE_TABLE(src, src_capacity);
	RB_REQUIRE_TABLE(dst, dst_capacity);
	RB_REQUIRE(dst_capacity >= src_capacity, "the new table must not be smaller");
	int rc = rb_hashset_clear(dst, dst_capacity, stream);
	if (rc != RB_OK) return rc;
	rbf::k_rehash<<<rb_grid(src_capacity, rbf::kThreads * 4, 8), rbf::kThreads, 0, S(stream)>>>(src, src_capacity, dst, dst_capacity);
	RB_LAUNCHED("hashset_rehash");
	return RB_OK;
}

int64_t rb_hashset_scratch_bytes(int64_t n) { return n >= 0 ? rbf::scratch_bytes(n, true) : 0; }

int64_t rb_frontier_scratch_bytes(int rep, int64_t n) {
	if (n < 0) return 0;
	const int64_t items = 12 * n;
	int64_t b = rbf::scratch_bytes(items, rep == RB_REP_686);
	if (rep == RB_REP_686) b += items * 288 + ((items + 3) / 4) * 16;     // children + new item ids
	return b;
}

int rb_hashset_insert_unique(int rep, void* table, int64_t capacity, const int8_t* states, int64_t n, int32_t* count_dev,
                             uint8_t* seen, uint8_t* first, int32_t* index, void* scratch, rb_stream_t stream) {
	RB_REQUIRE(rep_ok(rep) && n >= 0 && n < (1ll << 31), "bad rep or size");
	if (n == 0) return RB_OK;
	RB_REQUIRE_TABLE(table, capacity);
	RB_REQUIRE(states && count_dev && scratch && aligned(scratch, 16), "bad pointers");
	RB_INIT();
	const rbf::Scratch sc = rbf::scratch_of(scratch, n);
	cudaStream_t st = S(stream);
	RB_CUDA(cudaMemsetAsync(sc.lost, 0, (size_t)rbf::control_bytes(n), st));
	const int need_first = first != nullptr;
	if (rep == RB_REP_2024) {
		rbf::k_probe2024<<<(unsigned)sc.nb, rbf::kThreads, 0, st>>>(rbf::FromArray2024{states}, table, capacity, n, need_first, sc.word, sc.lost, sc.ctl, seen, index, nullptr, 1);
		RB_LAUNCHED("frontier_probe_2024");
	} else {
		RB_REQUIRE(aligned(states, 4), "6x8x6 states must be 4-byte aligned");
		rbf::k_pack686<<<(unsigned)((n + 7) / 8), rbf::kThreads, 0, st>>>(states, n, sc.keys);
		RB_LAUNCHED("frontier_pack_686");
		rbf::k_probe_keys<<<(unsigned)sc.nb, rbf::kThreads, 0, st>>>(sc.keys, table, capacity, n, need_first, sc.word, sc.lost, sc.ctl, seen, index);
		RB_LAUNCHED("frontier_probe_keys");
	}
	rbf::k_resolve<rbf::NoProvider, false><<<(unsigned)sc.nb, rbf::kThreads, 0, st>>>(
		rbf::NoProvider{}, table, capacity, n, need_first, sc.word, sc.lost, sc.status, sc.ctl, count_dev, nullptr, first, index, nullptr, nullptr, nullptr,
		nullptr, nullptr, nullptr, 1);
	RB_LAUNCHED("frontier_resolve");
	if (index) {
		rbf::k_index_rest<<<(unsigned)sc.nb, rbf::kThreads, 0, st>>>(table, capacity, n, sc.word, first, index);
		RB_LAUNCHED("frontier_index_rest");
	}
	return RB_OK;
}

int rb_hashset_lookup(int rep, const void* table, int64_t capacity, const int8_t* states, int64_t n, int32_t* index,
                      void* scratch, rb_stream_t stream) {
	RB_REQUIRE(rep_ok(rep) && n >= 0 && n < (1ll << 31), "bad rep or size");
	if (n == 0) return RB_OK;
	RB_REQUIRE_TABLE(table, capacity);
	RB_REQUIRE(states && index, "bad pointers");
	RB_INIT();
	cudaStream_t st = S(stream);
	const unsigned nb = (unsigned)rbf::n_blocks(n);
	if (rep == RB_REP_2024) {
		rbf::k_lookup2024<<<nb, rbf::kThreads, 0, st>>>(states, table, capacity, n, index);
		RB_LAUNCHED("frontier_lookup_2024");
	} else {
		RB_REQUIRE(scratch && aligned(scratch, 16) && aligned(states, 4), "6x8x6 lookup needs 16-byte aligned scratch");
		const rbf::Scratch sc = rbf::scratch_of(scratch, n);
		rbf::k_pack686<<<(unsigned)((n + 7) / 8), rbf::kThreads, 0, st>>>(states, n, sc.keys);
		RB_LAUNCHED("frontier_pack_686");
		rbf::k_lookup_keys<<<nb, rbf::kThreads, 0, st>>>(sc.keys, table, capacity, n, index);
		RB_LAUNCHED("frontier_lookup_keys");
	}
	return RB_OK;
}

static int frontier_expand_impl(int rep, void* table, int64_t capacity, const int8_t* frontier, int64_t n, const int32_t* n_dev, int32_t* count_dev,
                                int8_t* next_frontier, int32_t* parent, uint8_t* action, uint8_t* solved, uint8_t* seen, uint8_t* first,
                                int32_t* index, int32_t* n_new_dev, void* scratch, rb_stream_t stream) {
	RB_REQUIRE(rep_ok(rep) && n >= 0 && 12 * n < (1ll << 31), "bad rep or size");
	if (n == 0) {
		if (n_new_dev) RB_CUDA(cudaMemsetAsync(n_new_dev, 0, sizeof(int32_t), S(stream)));
		return RB_OK;
	}
	RB_REQUIRE_TABLE(table, capacity);
	RB_REQUIRE(frontier && count_dev && scratch && aligned(scratch, 16), "bad pointers");
	RB_REQUIRE(aligned(next_frontier, 4), "next_frontier must be 4-byte aligned");
	RB_INIT();
	const int64_t items = 12 * n;
	const rbf::Scratch sc = rbf::scratch_of(scratch, items);
	cudaStream_t st = S(stream);
	RB_CUDA(cudaMemsetAsync(sc.lost, 0, (size_t)rbf::control_bytes(items), st));
	const int need_first = first != nullptr;
	if (rep == RB_REP_2024) {
		const rbf::FromParent2024 prov{frontier};
		rbf::k_probe2024<<<(unsigned)sc.nb, rbf::kThreads, 0, st>>>(prov, table, capacity, items, need_first, sc.word, sc.lost, sc.ctl, seen, index, n_dev, 12);
		RB_LAUNCHED("frontier_probe_2024");
		rbf::k_resolve<rbf::FromParent2024, true><<<(unsigned)sc.nb, rbf::kThreads, 0, st>>>(
			prov, table, capacity, items, need_first, sc.word, sc.lost, sc.status, sc.ctl, count_dev, n_new_dev, first, index, nullptr, next_frontier, parent,
			action, solved, n_dev, 12);
		RB_LAUNCHED("frontier_resolve_2024");
	} else {
		RB_REQUIRE(aligned(frontier, 16) && aligned(next_frontier, 16), "6x8x6 states must be 16-byte aligned");
		RB_REQUIRE(!n_dev, "a device-side frontier size is supported for the 20x24 representation only");
		int8_t* children = reinterpret_cast<int8_t*>(sc.keys + items);
		int32_t* new_items = reinterpret_cast<int32_t*>(children + items * 288);
		int32_t* n_new = n_new_dev ? n_new_dev : reinterpret_cast<int32_t*>(sc.ctl + 2);
		int rc = rb_expand12(RB_REP_686, frontier, children, nullptr, nullptr, n, stream);
		if (rc != RB_OK) return rc;
		rbf::k_pack686<<<(unsigned)((items + 7) / 8), rbf::kThreads, 0, st>>>(children, items, sc.keys);
		RB_LAUNCHED("frontier_pack_686");
		rbf::k_probe_keys<<<(unsigned)sc.nb, rbf::kThreads, 0, st>>>(sc.keys, table, capacity, items, need_first, sc.word, sc.lost, sc.ctl, seen, index);
		RB_LAUNCHED("frontier_probe_keys");
		rbf::k_resolve<rbf::NoProvider, false><<<(unsigned)sc.nb, rbf::kThreads, 0, st>>>(
			rbf::NoProvider{}, table, capacity, items, need_first, sc.word, sc.lost, sc.status, sc.ctl, count_dev, n_new, first, index, new_items, nullptr,
			nullptr, nullptr, nullptr, nullptr, 1);
		RB_LAUNCHED("frontier_resolve");
		rbf::k_gather686<<<rb_grid(items, 8, 8), rbf::kThreads, 0, st>>>(children, new_items, n_new, next_frontier, parent, action, solved);
		RB_LAUNCHED("frontier_gather_686");
	}
	if (index) {
		rbf::k_index_rest<<<(unsigned)sc.nb, rbf::kThreads, 0, st>>>(table, capacity, items, sc.word, first, index);
		RB_LAUNCHED("frontier_index_rest");
	}
	return RB_OK;
}

int rb_frontier_expand(int rep, void* table, int64_t capacity, const int8_t* frontier, int64_t n, int32_t* count_dev,
                       int8_t* next_frontier, int32_t* parent, uint8_t* action, uint8_t* solved, uint8_t* seen, uint8_t* first,
                       int32_t* index, int32_t* n_new_dev, void* scratch, rb_stream_t stream) {
	return frontier_expand_impl(rep, table, capacity, frontier, n, nullptr, count_dev, next_frontier, parent, action, solved, seen, first, index,
	                            n_new_dev, scratch, stream);
}

int rb_frontier_expand_dev(int rep, void* table, int64_t capacity, const int8_t* frontier, int64_t n_max, const int32_t* n_dev,
                           int32_t* count_dev, int8_t* next_frontier, int32_t* parent, uint8_t* action, uint8_t* solved,
                           int32_t* n_new_dev, void* scratch, rb_stream_t stream) {
	RB_REQUIRE(n_dev, "null device-side frontier size");
	return frontier_expand_impl(rep, table, capacity, frontier, n_max, n_dev, count_dev, next_frontier, parent, action, solved, nullptr, nullptr, nullptr,
	                            n_new_dev, scratch, stream);
}

int rb_frontier_expand_chain(int rep, void* table, int64_t capacity, int8_t* buf_a, int8_t* buf_b, int64_t n0, int32_t layers,
                             int32_t* sizes_dev, int32_t* count_dev, void* scratch, rb_stream_t stream) {
	RB_REQUIRE(rep == RB_REP_2024 && n0 > 0 && layers >= 0 && layers <= 8, "20x24 representation, 1..8 layers");
	RB_REQUIRE(buf_a && buf_b && sizes_dev, "null buffer");
	int64_t bound = n0;
	for (int d = 0; d < layers; ++d) {
		RB_REQUIRE(12 * bound < (1ll << 28), "chained layers are for small frontiers (upper bound 12^d)");
		int rc = frontier_expand_impl(rep, table, capacity, (d & 1) ? buf_b : buf_a, bound, sizes_dev + d, count_dev, (d & 1) ? buf_a : buf_b, nullptr,
		                              nullptr, nullptr, nullptr, nullptr, nullptr, sizes_dev + d + 1, scratch, stream);
		if (rc != RB_OK) return rc;
		bound *= 12;
	}
	return RB_OK;
}

int rb_check_range(int rep, const int8_t* states, int64_t n_states, const uint8_t* faces, const uint8_t* dirs,
                   int64_t n_actions, int32_t* scratch_dev, rb_stream_t stream) {
	RB_REQUIRE(rep_ok(rep) && n_states >= 0 && n_actions >= 0 && scratch_dev, "bad argument");
	const int64_t state_bytes = (states && rep == RB_REP_2024) ? n_states * 20 : 0;
	if ((!faces || n_actions == 0) && state_bytes == 0) return RB_OK;
	RB_CUDA(cudaMemsetAsync(scratch_dev, 0, sizeof(int32_t), S(stream)));
	const int64_t work = state_bytes > n_actions ? state_bytes : n_actions;
	rbh::k_check_range<<<rb_grid(work, 256 * 8, 8), 256, 0, S(stream)>>>(rep, reinterpret_cast<const uint8_t*>(states), state_bytes,
	                                                                   faces, dirs, faces ? n_actions : 0, scratch_dev);
	RB_LAUNCHED("check_range");
	int32_t flag = 0;
	RB_CUDA(cudaMemcpyAsync(&flag, scratch_dev, sizeof(flag), cudaMemcpyDeviceToHost, S(stream)));
	RB_CUDA(cudaStreamSynchronize(S(stream)));
	if (flag) return rb_fail(RB_ERR_RANGE, "index out of range: face >= 6, direction >= 2, action >= 12 or state value >= 24%s%s");
	return RB_OK;
}

// ---- batched searches: view checks and scratch layouts ------------------------------------------------------------------
// A search's scratch: its arrays one after the other at 16-byte boundaries, then 64 spare bytes.  With a null base only the
// size is counted, so sizing and carving share one layout per search.
extern "C++" {
template <class T> static void carve(T*& dst, uint8_t* base, int64_t& used, int64_t n) {
	dst = base ? reinterpret_cast<T*>(base + used) : nullptr;
	used += rbf::up16(n * (int64_t)sizeof(T));
}

static int64_t carve_expansion(rbl::Core& v, uint8_t* base) {
	const int64_t K = v.K, P = 12 * (int64_t)v.N;
	int64_t used = 0;
	carve(v.slot, base, used, K * P);
	carve(v.flags, base, used, K * P);
	carve(v.block_new, base, used, K * ((P + rbl::kThreads - 1) / rbl::kThreads));
	carve(v.n_new, base, used, K);
	carve(v.off, base, used, K + 1);
	return used;
}

static int64_t scratch(rba::View& v, uint8_t* base) {
	int64_t used = carve_expansion(v, base);
	carve(v.tmp, base, used, (int64_t)v.K * 12 * v.N);
	return used + 64;
}

static int64_t scratch(rbb::View& v, uint8_t* base) {
	int64_t used = carve_expansion(v, base);
	carve(v.n_sel, base, used, v.K);
	carve(v.sel, base, used, (int64_t)v.K * v.N);
	carve(v.cut, base, used, v.K);
	carve(v.first_solved, base, used, v.K);
	carve(v.n_new_total, base, used, 0);                        // written by k_totals, unused: the first of the spare bytes
	return used + 64;
}

// The checks both views share, in order; then the Core is filled and the scratch carved.  An entry point checks its own
// arguments only after this, so a bad view is what a call reports first.  keys: slots one search can claim (a full table drops
// a child without an error word, k_probe stores slot -1: 2 K keys slots keep every search at load <= 1/2).
template <class AbiView, class View>
static int core_view(const AbiView* a, bool n_ok, int64_t keys, bool own_set, bool own_aligned, View& v) {
	RB_REQUIRE(a->K > 0 && a->K <= 65535 && a->M > 1 && a->N > 0 && n_ok, "bad K / M / N (K <= 65535; N <= 1024 for A*, 2^20 for BFS)");
	RB_REQUIRE(a->states && a->parents && a->parent_actions && a->count && a->won && a->table && a->scratch && own_set, "null buffer in view");
	RB_REQUIRE_TABLE(a->table, a->capacity);
	if (a->capacity < 2 * (int64_t)a->K * keys)
		return rb_fail(RB_ERR_CAPACITY, "table capacity must be at least 2 K M slots for A*, 2 K (M + 12 N) for BFS%s%s");
	RB_REQUIRE(aligned(a->scratch, 16) && aligned(a->states, 4) && own_aligned, "misaligned buffer");
	v.K = a->K; v.M = a->M; v.N = a->N;
	v.states = a->states; v.parents = a->parents; v.parent_actions = a->parent_actions; v.count = a->count; v.won = a->won;
	v.table = a->table; v.capacity = a->capacity;
	scratch(v, static_cast<uint8_t*>(a->scratch));
	return RB_OK;
}
}  // extern "C++"

// ---- batched A* ----------------------------------------------------------------------------------------------------------
int64_t rb_astar_scratch_bytes(int32_t K, int32_t N) {
	rba::View v{{K, 0, N}};
	return K > 0 && N > 0 ? scratch(v, nullptr) : 0;
}

static int astar_view(const rb_astar_view* a, rba::View& v) {
	RB_REQUIRE(a, "null view");
	v.G = a->G; v.cost = a->cost; v.in_open = a->in_open; v.n_sel = a->n_sel; v.sel = a->sel; v.solved_index = a->solved_index;
	return core_view(a, a->N <= 1024, a->M, a->G && a->cost && a->in_open && a->n_sel && a->sel && a->solved_index,
	                 aligned(a->G, 8) && aligned(a->cost, 8), v);
}

int rb_astar_init(const rb_astar_view* a, const int8_t* roots, rb_stream_t stream) {
	rba::View v;
	int rc = astar_view(a, v);
	if (rc != RB_OK) return rc;
	RB_REQUIRE(roots && aligned(roots, 4), "roots must be a 4-byte aligned device pointer");
	RB_INIT();
	rba::k_init<<<(v.K + rbl::kThreads - 1) / rbl::kThreads, rbl::kThreads, 0, S(stream)>>>(v, roots);
	RB_LAUNCHED("astar_init");
	return RB_OK;
}

int rb_astar_expand(const rb_astar_view* a, int64_t max_states, int8_t* new_states, int32_t* new_search, int32_t* new_index,
                    int32_t* n_new_total, int32_t* n_active, rb_stream_t stream) {
	rba::View v;
	int rc = astar_view(a, v);
	if (rc != RB_OK) return rc;
	RB_REQUIRE(new_states && new_search && new_index && n_new_total && n_active && aligned(new_states, 4), "null or misaligned output");
	RB_REQUIRE(max_states < v.M, "M must exceed max_states (index 0 is unused)");
	RB_INIT();
	cudaStream_t st = S(stream);
	const dim3 grid(v.nbx(), v.K);
	RB_CUDA(cudaMemsetAsync(n_active, 0, sizeof(int32_t), st));
	{
		static std::mutex mu;                                    // once per device, and never inside a stream capture of the step
		static bool done[64] = {};
		int dev = 0;
		RB_CUDA(cudaGetDevice(&dev));
		std::lock_guard<std::mutex> lock(mu);
		if (dev >= 0 && dev < 64 && !done[dev]) {
			RB_CUDA(cudaFuncSetAttribute(rba::k_select, cudaFuncAttributeMaxDynamicSharedMemorySize, rba::kSelSmem));
			done[dev] = true;
		}
	}
	rba::k_select<<<v.K, rba::kSelThreads, rba::kSelSmem, st>>>(v, max_states, n_active);
	RB_LAUNCHED("astar_select");
	rbl::k_probe<<<grid, rbl::kThreads, 0, st>>>(v);
	RB_LAUNCHED("astar_probe");
	rbl::k_flag<<<grid, rbl::kThreads, 0, st>>>(v);
	RB_LAUNCHED("astar_flag");
	rbl::k_totals<<<1, 1024, 0, st>>>(v, n_new_total);
	RB_LAUNCHED("astar_totals");
	rba::k_assign<<<grid, rbl::kThreads, 0, st>>>(v, new_states, new_search, new_index);
	RB_LAUNCHED("astar_assign");
	return RB_OK;
}

int rb_astar_commit(const rb_astar_view* a, const float* values, double lambda, const int32_t* new_search, const int32_t* new_index,
                    const int32_t* n_new_total, rb_stream_t stream) {
	rba::View v;
	int rc = astar_view(a, v);
	if (rc != RB_OK) return rc;
	RB_REQUIRE(values && new_search && new_index && n_new_total, "null input");
	cudaStream_t st = S(stream);
	const dim3 grid(v.nbx(), v.K);
	const int64_t worst = (int64_t)v.K * v.P();
	rba::k_push<<<(unsigned)((worst + rbl::kThreads - 1) / rbl::kThreads), rbl::kThreads, 0, st>>>(v, values, lambda, new_search, new_index, n_new_total);
	RB_LAUNCHED("astar_push");
	rba::k_relax_eval<<<grid, rbl::kThreads, 0, st>>>(v, 0);
	RB_LAUNCHED("astar_relax_eval0");
	rba::k_relax_new_ways<<<grid, rbl::kThreads, 0, st>>>(v);
	RB_LAUNCHED("astar_relax_new_ways");
	rba::k_relax_eval<<<grid, rbl::kThreads, 0, st>>>(v, 1);
	RB_LAUNCHED("astar_relax_eval1");
	rba::k_relax_shortcuts<<<dim3((v.N + rbl::kThreads - 1) / rbl::kThreads, v.K), rbl::kThreads, 0, st>>>(v);
	RB_LAUNCHED("astar_relax_shortcuts");
	rba::k_finish<<<grid, rbl::kThreads, 0, st>>>(v);
	RB_LAUNCHED("astar_finish");
	return RB_OK;
}

// ---- batched BFS ---------------------------------------------------------------------------------------------------------
int64_t rb_bfs_scratch_bytes(int32_t K, int32_t N) {
	rbb::View v{{K, 0, N}};
	return K > 0 && N > 0 ? scratch(v, nullptr) : 0;
}

static int bfs_view(const rb_bfs_view* b, rbb::View& v) {
	RB_REQUIRE(b, "null view");
	v.head = b->head; v.done = b->done; v.solved_parent = b->solved_parent; v.solved_action = b->solved_action;
	// the children of parents dropped by the budget are claimed before the cut is known: a search holds up to M + 12 N keys
	return core_view(b, b->N <= (1 << 20), b->M + 12 * (int64_t)b->N, b->head && b->done && b->solved_parent && b->solved_action, true, v);
}

int rb_bfs_init(const rb_bfs_view* b, const int8_t* roots, rb_stream_t stream) {
	rbb::View v;
	int rc = bfs_view(b, v);
	if (rc != RB_OK) return rc;
	RB_REQUIRE(roots && aligned(roots, 4), "roots must be a 4-byte aligned device pointer");
	RB_INIT();
	rbb::k_init<<<(v.K + rbl::kThreads - 1) / rbl::kThreads, rbl::kThreads, 0, S(stream)>>>(v, roots);
	RB_LAUNCHED("bfs_init");
	return RB_OK;
}

int rb_bfs_step(const rb_bfs_view* b, int64_t max_states, int32_t* n_active, rb_stream_t stream) {
	rbb::View v;
	int rc = bfs_view(b, v);
	if (rc != RB_OK) return rc;
	RB_REQUIRE(n_active, "null n_active");
	RB_REQUIRE(max_states >= 1 && max_states < v.M, "M must exceed max_states (index 0 is unused)");
	RB_INIT();
	cudaStream_t st = S(stream);
	const dim3 grid(v.nbx(), v.K);
	rbb::k_pop<<<dim3((v.N + rbl::kThreads - 1) / rbl::kThreads, v.K), rbl::kThreads, 0, st>>>(v, max_states, n_active);
	RB_LAUNCHED("bfs_pop");
	rbl::k_probe<<<grid, rbl::kThreads, 0, st>>>(v);
	RB_LAUNCHED("bfs_probe");
	rbl::k_flag<<<grid, rbl::kThreads, 0, st>>>(v);
	RB_LAUNCHED("bfs_flag");
	rbl::k_totals<<<1, 1024, 0, st>>>(v, v.n_new_total);
	RB_LAUNCHED("bfs_totals");
	rbb::k_assign<<<grid, rbl::kThreads, 0, st>>>(v, max_states);
	RB_LAUNCHED("bfs_assign");
	rbb::k_finish<<<grid, rbl::kThreads, 0, st>>>(v, max_states, n_active);
	RB_LAUNCHED("bfs_finish");
	return RB_OK;
}

int rb_bfs_paths(const rb_bfs_view* b, uint8_t* queues, int32_t* lengths, int32_t L, rb_stream_t stream) {
	rbb::View v;
	int rc = bfs_view(b, v);
	if (rc != RB_OK) return rc;
	RB_REQUIRE(queues && lengths && L > 0, "null output or L <= 0");
	RB_INIT();
	rbb::k_paths<<<(v.K + rbl::kThreads - 1) / rbl::kThreads, rbl::kThreads, 0, S(stream)>>>(v, queues, lengths, L);
	RB_LAUNCHED("bfs_paths");
	return RB_OK;
}

// ---- device-seeded and packed scrambles --------------------------------------------------------------------------------------
int rb_scramble_seeded(int rep, uint64_t seed, uint64_t first_cube, const int8_t* start, int8_t* out, int64_t n, int32_t depth,
                       rb_stream_t stream) {
	RB_REQUIRE(rep_ok(rep) && n >= 0 && depth >= 0, "bad rep or size");
	if (n == 0) return RB_OK;
	RB_REQUIRE(out && start != out, "null output (or start aliases out)");
	RB_INIT();
	if (rep != RB_REP_2024) {
		RB_REQUIRE(aligned(out, 16) && aligned(start, 16), "6x8x6 states must be 16-byte aligned");
		RB_REQUIRE(rbt::host().stickers_ok, "sticker tables: the 20x24 and 6x8x6 move tables disagree");
	}
	int rc = rbs::launch_seeded(seed, first_cube, out, n, depth, S(stream), scramble_pitch(rep));
	return rc != RB_OK ? rc : scramble_finish(rep, start, out, n, S(stream));
}

int rb_as2024(const int8_t* states686, int8_t* states2024, uint8_t* ok, int64_t n, rb_stream_t stream) {
	RB_REQUIRE(n >= 0, "bad size");
	if (n == 0) return RB_OK;
	RB_REQUIRE(states686 && states2024, "null pointer");
	RB_REQUIRE(rbt::host().stickers_ok, "sticker tables: the 20x24 and 6x8x6 move tables disagree");
	RB_INIT();
	if (ok) RB_CUDA(cudaMemsetAsync(ok, 1, (size_t)n, S(stream)));
	rb686::k_as2024<<<rb_grid(n * 20, rb686::kThreads, 8), rb686::kThreads, 0, S(stream)>>>(states686, states2024, ok, n);
	RB_LAUNCHED("as2024");
	return RB_OK;
}

int rb_as686(const int8_t* states2024, int8_t* states686, int64_t n, rb_stream_t stream) {
	RB_REQUIRE(n >= 0, "bad size");
	if (n == 0) return RB_OK;
	RB_REQUIRE(states2024 && states686 && aligned(states2024, 4) && aligned(states686, 16), "null or misaligned pointer");
	RB_REQUIRE(rbt::host().stickers_ok, "sticker tables: the 20x24 and 6x8x6 move tables disagree");
	RB_INIT();
	rb686::k_render_from2024<<<rb_grid((n + 31) / 32, rb686::kWarps, 8), rb686::kThreads, 0, S(stream)>>>(states686, nullptr, n, states2024);
	RB_LAUNCHED("render_686");
	return RB_OK;
}

int rb_seeded_actions(uint64_t seed, uint64_t first_cube, uint8_t* actions, int64_t n, int32_t depth, rb_stream_t stream) {
	RB_REQUIRE(n >= 0 && depth >= 0, "bad size");
	if (n == 0 || depth == 0) return RB_OK;
	RB_REQUIRE(actions, "null output");
	return rbs::launch_seeded_actions(seed, first_cube, actions, n, depth, S(stream));
}

int rb_unpack_actions(const uint8_t* packed, uint8_t* actions, int64_t n, int32_t depth, rb_stream_t stream) {
	RB_REQUIRE(n >= 0 && depth >= 0, "bad size");
	if (n == 0 || depth == 0) return RB_OK;
	RB_REQUIRE(packed && actions, "null pointer");
	const int vec_ok = depth % 2 == 0 && aligned(packed, 16) && aligned(actions, 16);
	const int64_t work = n * ((depth + 1) / 2);
	rbh::k_unpack_actions<<<rb_grid(vec_ok ? work / 8 + 1 : work, 256, 8), 256, 0, S(stream)>>>(packed, actions, n, depth, vec_ok);
	RB_LAUNCHED("unpack_actions");
	return RB_OK;
}

// ---- host-buffer entry points ------------------------------------------------------------------------------
extern "C++" {
// Runs enqueue(slot, stream, base, count) over [0, n) in chunks, alternating the two staging slots; always drains both streams
// before returning (no copy to or from the caller's host buffers is left in flight, error or not).
template <class Enqueue>
static int rbh_run_chunks(int64_t n, int64_t chunk, Enqueue enqueue) {
	rbh::Staging& st = rbh::g_stage;
	int rc = RB_OK, k = 0;
	for (int64_t base = 0; base < n && rc == RB_OK; base += chunk, k ^= 1)
		rc = enqueue(k, st.stream[k], base, n - base < chunk ? n - base : chunk);
	return rbh::stage_sync(rc);
}
// chunks of <= cap items (a multiple of 256 so every chunk base stays 16-byte aligned), at least 4 chunks
static int64_t rbh_chunk(int64_t n, int64_t cap) {
	int64_t chunk = ((n + 3) / 4 + 255) / 256 * 256;
	return chunk > cap ? cap : chunk;
}
}  // extern "C++"

int rbh_scramble(int rep, const uint8_t* actions, int8_t* out, int64_t n, int32_t depth) {
	RB_REQUIRE(rep_ok(rep) && n >= 0 && depth >= 0, "bad rep or size");
	if (n == 0) return RB_OK;
	RB_REQUIRE(out && (actions || depth == 0), "null pointer");
	RB_INIT();
	std::lock_guard<std::mutex> lock(rbh::g_stage_mu);
	const int64_t sb = rep == RB_REP_2024 ? 20 : 288, chunk = rbh_chunk(n, 1 << 20);
	int rc = rbh::stage_reserve((size_t)chunk * (depth > 0 ? depth : 1), 0, (size_t)chunk * sb);
	if (rc != RB_OK) return rc;
	rbh::Staging& st = rbh::g_stage;
	return rbh_run_chunks(n, chunk, [&](int k, cudaStream_t s, int64_t base, int64_t cnt) -> int {
		if (depth > 0) RB_CUDA(cudaMemcpyAsync(st.buf[k][0], actions + base * depth, (size_t)cnt * depth, cudaMemcpyHostToDevice, s));
		int r = rb_scramble(rep, reinterpret_cast<const uint8_t*>(st.buf[k][0]), depth, 1, nullptr, reinterpret_cast<int8_t*>(st.buf[k][2]), cnt, depth, s);
		if (r != RB_OK) return r;
		RB_CUDA(cudaMemcpyAsync(out + base * sb, st.buf[k][2], (size_t)cnt * sb, cudaMemcpyDeviceToHost, s));
		return RB_OK;
	});
}

int rbh_scramble_packed(int rep, const uint8_t* packed, int8_t* out, int64_t n, int32_t depth) {
	RB_REQUIRE(rep_ok(rep) && n >= 0 && depth >= 0, "bad rep or size");
	if (n == 0) return RB_OK;
	RB_REQUIRE(out && (packed || depth == 0), "null pointer");
	RB_INIT();
	std::lock_guard<std::mutex> lock(rbh::g_stage_mu);
	const int64_t sb = rep == RB_REP_2024 ? 20 : 288, pb = (depth + 1) / 2, chunk = rbh_chunk(n, 1 << 20);
	int rc = rbh::stage_reserve((size_t)chunk * (pb > 0 ? pb : 1), 0, (size_t)chunk * sb, (size_t)chunk * (depth > 0 ? depth : 1));
	if (rc != RB_OK) return rc;
	rbh::Staging& st = rbh::g_stage;
	return rbh_run_chunks(n, chunk, [&](int k, cudaStream_t s, int64_t base, int64_t cnt) -> int {
		uint8_t* acts = reinterpret_cast<uint8_t*>(st.buf[k][3]);
		if (depth > 0) {
			RB_CUDA(cudaMemcpyAsync(st.buf[k][0], packed + base * pb, (size_t)cnt * pb, cudaMemcpyHostToDevice, s));
			int r = rb_unpack_actions(reinterpret_cast<const uint8_t*>(st.buf[k][0]), acts, cnt, depth, s);
			if (r != RB_OK) return r;
		}
		int r = rb_scramble(rep, acts, depth, 1, nullptr, reinterpret_cast<int8_t*>(st.buf[k][2]), cnt, depth, s);
		if (r != RB_OK) return r;
		RB_CUDA(cudaMemcpyAsync(out + base * sb, st.buf[k][2], (size_t)cnt * sb, cudaMemcpyDeviceToHost, s));
		return RB_OK;
	});
}

int rbh_scramble_seeded(int rep, uint64_t seed, uint64_t first_cube, int8_t* out, int64_t n, int32_t depth) {
	RB_REQUIRE(rep_ok(rep) && n >= 0 && depth >= 0, "bad rep or size");
	if (n == 0) return RB_OK;
	RB_REQUIRE(out, "null pointer");
	RB_INIT();
	std::lock_guard<std::mutex> lock(rbh::g_stage_mu);
	const int64_t sb = rep == RB_REP_2024 ? 20 : 288, chunk = rbh_chunk(n, 1 << 20);
	int rc = rbh::stage_reserve(0, 0, (size_t)chunk * sb);
	if (rc != RB_OK) return rc;
	rbh::Staging& st = rbh::g_stage;
	return rbh_run_chunks(n, chunk, [&](int k, cudaStream_t s, int64_t base, int64_t cnt) -> int {
		int r = rb_scramble_seeded(rep, seed, first_cube + (uint64_t)base, nullptr, reinterpret_cast<int8_t*>(st.buf[k][2]), cnt, depth, s);
		if (r != RB_OK) return r;
		RB_CUDA(cudaMemcpyAsync(out + base * sb, st.buf[k][2], (size_t)cnt * sb, cudaMemcpyDeviceToHost, s));
		return RB_OK;
	});
}

int rbh_multi_rotate(int rep, const int8_t* states, const uint8_t* faces, const uint8_t* dirs, int8_t* out, int64_t n) {
	RB_REQUIRE(rep_ok(rep) && n >= 0, "bad rep or size");
	if (n == 0) return RB_OK;
	RB_REQUIRE(states && faces && out, "null pointer");
	RB_INIT();
	std::lock_guard<std::mutex> lock(rbh::g_stage_mu);
	const int64_t sb = rep == RB_REP_2024 ? 20 : 288, chunk = rbh_chunk(n, 1 << 22);
	int rc = rbh::stage_reserve((size_t)chunk * sb, (size_t)chunk * 2, (size_t)chunk * sb);
	if (rc != RB_OK) return rc;
	rbh::Staging& st = rbh::g_stage;
	return rbh_run_chunks(n, chunk, [&](int k, cudaStream_t s, int64_t base, int64_t cnt) -> int {
		uint8_t* f_dev = reinterpret_cast<uint8_t*>(st.buf[k][1]);
		uint8_t* d_dev = dirs ? f_dev + chunk : nullptr;
		RB_CUDA(cudaMemcpyAsync(st.buf[k][0], states + base * sb, (size_t)cnt * sb, cudaMemcpyHostToDevice, s));
		RB_CUDA(cudaMemcpyAsync(f_dev, faces + base, (size_t)cnt, cudaMemcpyHostToDevice, s));
		if (dirs) RB_CUDA(cudaMemcpyAsync(d_dev, dirs + base, (size_t)cnt, cudaMemcpyHostToDevice, s));
		int r = rb_multi_rotate(rep, reinterpret_cast<const int8_t*>(st.buf[k][0]), f_dev, d_dev, reinterpret_cast<int8_t*>(st.buf[k][2]), cnt, s);
		if (r != RB_OK) return r;
		RB_CUDA(cudaMemcpyAsync(out + base * sb, st.buf[k][2], (size_t)cnt * sb, cudaMemcpyDeviceToHost, s));
		return RB_OK;
	});
}

// Pinned host memory for the rbh_* calls.  huge != 0: anonymous mapping advised to transparent huge pages before it is touched
// and registered (2 MB pages keep the IOMMU / DMA translation working set of a multi-GB transfer small; several GPUs copying
// at once into 4 KB-paged buffers are translation-bound on some hosts).  Free with rbh_host_free(ptr, bytes).
void* rbh_host_alloc(int64_t bytes, int huge) {
	if (bytes <= 0) return nullptr;
	const size_t sz = ((size_t)bytes + (2u << 20) - 1) & ~((size_t)(2u << 20) - 1);
	void* p = mmap(nullptr, sz, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
	if (p == MAP_FAILED) { rb_fail(RB_ERR_BAD_ARG, "mmap of the host buffer failed%s%s"); return nullptr; }
	if (huge) madvise(p, sz, MADV_HUGEPAGE);
	memset(p, 0, sz);                                      // touch: pages (huge ones where the kernel grants them) exist before pinning
	if (cudaHostRegister(p, sz, cudaHostRegisterPortable) != cudaSuccess) {
		cudaGetLastError();
		munmap(p, sz);
		rb_fail(RB_ERR_CUDA, "cudaHostRegister of the host buffer failed%s%s");
		return nullptr;
	}
	return p;
}

int rbh_host_free(void* ptr, int64_t bytes) {
	if (!ptr) return RB_OK;
	const size_t sz = ((size_t)bytes + (2u << 20) - 1) & ~((size_t)(2u << 20) - 1);
	RB_CUDA(cudaHostUnregister(ptr));
	munmap(ptr, sz);
	return RB_OK;
}

int rbh_release(void) {
	std::lock_guard<std::mutex> lock(rbh::g_stage_mu);
	return rbh::stage_release();
}

}  // extern "C"
