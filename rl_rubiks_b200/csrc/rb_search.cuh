// Lockstep expansion core of the batched searches (rb_astar.cuh, rb_bfs.cuh).  K searches select up to N parents each per
// step; the children are generated in (parent, action) order and deduplicated against the search's own seen-set with the
// reference's batch-order numbering (same probe / flag / assign scheme as rb_frontier.cuh).  The key carries the search id in
// the 24 free bits of its high word, so all searches share one table.  A step is the search's select, k_probe, k_flag,
// k_totals, the search's assign kernel (number_new_child first) and its finish kernel (rearm_firstpos first).
// 20x24 representation only.
#pragma once
#include "rb_common.cuh"
#include "rb_frontier.cuh"

namespace rbl {

constexpr int kThreads = 256;

struct Core {                       // the fields every lockstep search has (rba::View and rbb::View add their own)
	int K, M, N;
	int8_t* states;                 // [K][M][20]
	int32_t* parents;               // [K][M]
	uint8_t* parent_actions;        // [K][M]
	int32_t* count;                 // [K] states stored
	uint8_t* won;                   // [K]
	int32_t* n_sel;                 // [K] parents selected in the running step
	int32_t* sel;                   // [K][N] their indices
	void* table;
	int64_t capacity;
	// expansion scratch, [K][P] with P = 12 N
	int32_t* slot;
	uint8_t* flags;                 // bit 0 new, bit 1 old (first & seen); A* keeps its relaxation flag in bit 2
	int32_t* block_new;             // [K][nbx]
	int32_t* n_new;                 // [K]
	int32_t* off;                   // [K + 1]
	__host__ __device__ int P() const { return 12 * N; }
	__host__ __device__ int nbx() const { return (12 * N + kThreads - 1) / kThreads; }
};

// the key of a state in search s: the packed 20x24 state (100 bits) with the search id in bits 40-55 of the high word
__device__ __forceinline__ rbf::Key key(const uint32_t (&w)[5], int s) {
	rbf::Key k = rbf::pack2024(w);
	k.hi |= (unsigned long long)s << 40;
	return k;
}

__device__ __forceinline__ bool is_solved(const uint32_t (&w)[5]) {
	const uint32_t* sv = reinterpret_cast<const uint32_t*>(g_solved2024);
	return (w[0] == sv[0]) & (w[1] == sv[1]) & (w[2] == sv[2]) & (w[3] == sv[3]) & (w[4] == sv[4]);
}

// child i of search s: action i % 12 applied to the selected parent i / 12
__device__ __forceinline__ void child_words(const Core& v, int s, int i, const uint8_t* s_lut, uint32_t (&w)[5], int& parent) {
	parent = v.sel[(int64_t)s * v.N + i / 12];
	const uint32_t* p = reinterpret_cast<const uint32_t*>(v.states + ((int64_t)s * v.M + parent) * 20);
#pragma unroll
	for (int k = 0; k < 5; ++k) w[k] = p[k];
	rb_move2024(s_lut, (uint32_t)(i % 12), w);
}

// The root of search s becomes its state 1: stored without parent, entered into the table with index 1.  Returns whether it
// is solved, and marks the search won if so.
__device__ __forceinline__ bool init_root(const Core& v, int s, const int8_t* __restrict__ roots) {
	uint32_t w[5];
	const uint32_t* p = reinterpret_cast<const uint32_t*>(roots + (int64_t)s * 20);
	uint32_t* dst = reinterpret_cast<uint32_t*>(v.states + ((int64_t)s * v.M + 1) * 20);
#pragma unroll
	for (int k = 0; k < 5; ++k) { w[k] = p[k]; dst[k] = w[k]; }
	const rbf::Table t = rbf::table_of(v.table, v.capacity);
	const int64_t slot = rbf::find_or_claim(t, key(w, s));
	if (slot >= 0) t.val(slot) = 1;
	const int64_t row = (int64_t)s * v.M + 1;
	v.parents[row] = 0;
	v.parent_actions[row] = 0;
	const bool solved = is_solved(w);
	v.won[s] = solved ? 1 : 0;
	return solved;
}

// ---- probe / flag / totals ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) k_probe(Core v) {
	__shared__ __align__(16) uint8_t s_lut[RB_LUT_BYTES];
	rb_stage_lut2024(s_lut);
	__syncthreads();
	const int s = blockIdx.y, i = blockIdx.x * kThreads + threadIdx.x;
	if (i >= v.n_sel[s] * 12) return;
	uint32_t w[5]; int parent;
	child_words(v, s, i, s_lut, w, parent);
	const rbf::Table t = rbf::table_of(v.table, v.capacity);
	const int64_t slot = rbf::find_or_claim(t, key(w, s));
	v.slot[(int64_t)s * v.P() + i] = (int32_t)slot;
	if (slot >= 0) atomicMin(&t.firstpos(slot), (uint32_t)i);
}

__global__ void __launch_bounds__(kThreads) k_flag(Core v) {
	const int s = blockIdx.y, i = blockIdx.x * kThreads + threadIdx.x;
	const rbf::Table t = rbf::table_of(v.table, v.capacity);
	bool is_new = false;
	if (i < v.n_sel[s] * 12) {
		const int32_t slot = v.slot[(int64_t)s * v.P() + i];
		bool seen = false, first = false;
		if (slot >= 0) { seen = t.val(slot) != 0; first = t.firstpos(slot) == (uint32_t)i; }
		is_new = first && !seen;
		v.flags[(int64_t)s * v.P() + i] = (uint8_t)((is_new ? 1 : 0) | ((first && seen) ? 2 : 0));
	}
	const int c = __syncthreads_count(is_new);
	if (threadIdx.x == 0) v.block_new[s * v.nbx() + blockIdx.x] = c;
}

// n_new[s], exclusive offsets over the searches, grand total.  One block.
__global__ void __launch_bounds__(1024) k_totals(Core v, int32_t* __restrict__ n_new_total) {
	__shared__ int32_t s_carry, s_warp[32];
	if (threadIdx.x == 0) s_carry = 0;
	__syncthreads();
	for (int base = 0; base < v.K; base += 1024) {
		const int s = base + threadIdx.x;
		int32_t x = 0;
		if (s < v.K) {
			const int nb = (v.n_sel[s] * 12 + kThreads - 1) / kThreads;
			for (int b = 0; b < nb; ++b) x += v.block_new[s * v.nbx() + b];
			v.n_new[s] = x;
		}
		int32_t incl = x;
#pragma unroll
		for (int o = 1; o < 32; o <<= 1) {
			const int32_t y = __shfl_up_sync(0xffffffffu, incl, o);
			if ((threadIdx.x & 31) >= o) incl += y;
		}
		if ((threadIdx.x & 31) == 31) s_warp[threadIdx.x >> 5] = incl;
		__syncthreads();
		if (threadIdx.x < 32) {
			int32_t wv = s_warp[threadIdx.x];
#pragma unroll
			for (int o = 1; o < 32; o <<= 1) {
				const int32_t y = __shfl_up_sync(0xffffffffu, wv, o);
				if (threadIdx.x >= o) wv += y;
			}
			s_warp[threadIdx.x] = wv;
		}
		__syncthreads();
		incl += threadIdx.x >= 32 ? s_warp[(threadIdx.x >> 5) - 1] : 0;
		const int32_t carry = s_carry;
		if (s < v.K) v.off[s] = carry + incl - x;
		__syncthreads();
		if (threadIdx.x == 1023) s_carry = carry + incl;
		__syncthreads();
	}
	if (threadIdx.x == 0) { v.off[v.K] = s_carry; *n_new_total = s_carry; }
}

// ---- assign / finish ------------------------------------------------------------------------------------------------------
struct NewChild {
	int k;                          // rank among the search's new children of the step, in batch order
	int idx;                        // its state index, count + k + 1
	int parent;
	uint32_t w[5];                  // its state
};

// Start of an assign kernel (grid nbx x K): child i of search s, if new, gets index count + rank + 1 in its slot, and its state
// is regenerated.  Every thread of the block must call it (it holds barriers); it returns false for a child that is not new.
__device__ __forceinline__ bool number_new_child(const Core& v, int s, int i, NewChild& c) {
	__shared__ __align__(16) uint8_t s_lut[RB_LUT_BYTES];
	__shared__ int32_t s_warp[kThreads / 32];
	rb_stage_lut2024(s_lut);
	const bool is_new = i < v.n_sel[s] * 12 && (v.flags[(int64_t)s * v.P() + i] & 1);
	const int r = rbf::block_rank(is_new, s_warp);               // also orders the LUT staging before use
	if (!is_new) return false;
	int32_t prefix = 0;
	for (int b = 0; b < (int)blockIdx.x; ++b) prefix += v.block_new[s * v.nbx() + b];
	c.k = prefix + r;
	c.idx = v.count[s] + c.k + 1;
	rbf::table_of(v.table, v.capacity).val(v.slot[(int64_t)s * v.P() + i]) = c.idx;
	child_words(v, s, i, s_lut, c.w, c.parent);
	return true;
}

// Start of a finish kernel: the slot child i of search s probed (one of n_sel * 12) is idle for the next step's race again.
__device__ __forceinline__ void rearm_firstpos(const Core& v, int s, int i, int n_sel) {
	if (i < n_sel * 12) {
		const int32_t slot = v.slot[(int64_t)s * v.P() + i];
		if (slot >= 0) rbf::table_of(v.table, v.capacity).firstpos(slot) = 0xffffffffu;
	}
}

}  // namespace rbl
