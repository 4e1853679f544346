// Batched breadth-first search on the device: K independent searches advance in lockstep, up to N FIFO pops per search and
// step.
//
// Replaces BFS.search (reference: librubiks/solving/agents.py:96-123) -- the FIFO, the dict, the budget test before every
// pop -- for many cubes at once.  Every search reproduces the reference's trace exactly:
//   * the FIFO is the stored states themselves: state i of a search is the i-th state its dict records (root = 1, children
//     numbered in (parent, action) order), so popping is taking head, head + 1, ...; a step pops
//     take = min(N, count - head + 1) of them;
//   * children are deduplicated and numbered by the lockstep expansion core the batched A* uses too (rb_search.cuh: probe,
//     flag, totals, then k_assign here);
//   * the budget `len(states) < max_states` is tested before every pop (agents.py:104): parent j of the step is admitted iff
//     count + (new states recorded by the step's parents before j) < max_states.  The admitted parents are a prefix, and the
//     last one records new state number max_states - count (the cut); later parents' children are dropped;
//   * a child already in the dict is skipped before the solved test; the first new child in batch order that is solved and
//     has an admitted parent ends the search before it is recorded: len = count + its rank among the step's new children.
// States numbered >= max_states are never popped: they are counted and entered into the table, not stored.
// 20x24 representation only.  Buffers are caller-owned (rb_bfs_view, include/rubiks_b200.h).
#pragma once
#include "rb_search.cuh"

namespace rbb {

using rbl::kThreads;
constexpr int32_t kNoCut = 0x7fffffff;
constexpr unsigned long long kNoSolved = ~0ull;

struct View : rbl::Core {           // device-side copy of rb_bfs_view; n_sel, sel, cut, first_solved, n_new_total: scratch
	int32_t* head;
	uint8_t* done;
	int32_t* solved_parent;
	uint8_t* solved_action;
	int32_t* cut;                   // [K] batch position of the child numbered max_states (kNoCut: none this step)
	unsigned long long* first_solved;   // [K] (rank << 32 | batch position) of the first solved new child
	int32_t* n_new_total;           // [1] written by rbl::k_totals, unused here
};

// roots: state 1 of every search; a solved root is found at once with len 0 (agents.py:99-100)
__global__ void __launch_bounds__(kThreads) k_init(View v, const int8_t* __restrict__ roots) {
	const int s = blockIdx.x * kThreads + threadIdx.x;
	if (s >= v.K) return;
	const bool solved = rbl::init_root(v, s, roots);
	v.count[s] = solved ? 0 : 1;
	v.head[s] = 1;
	v.done[s] = solved ? 1 : 0;
	v.solved_parent[s] = 0;
	v.solved_action[s] = 0;
}

// pop: sel[s][j] = head + j for j < take; per-step state of the search re-armed.  A search that cannot pop (budget spent,
// FIFO dry) is done.  Block (0, 0) zeroes the active counter that k_finish fills.
__global__ void __launch_bounds__(kThreads) k_pop(View v, int64_t max_states, int32_t* __restrict__ n_active) {
	const int s = blockIdx.y, j = blockIdx.x * kThreads + threadIdx.x;
	const int cnt = v.count[s], head = v.head[s];
	const bool active = !v.done[s] && (int64_t)cnt < max_states && head <= cnt;
	const int take = active ? min(v.N, cnt - head + 1) : 0;
	if (j < take) v.sel[(int64_t)s * v.N + j] = head + j;
	if (j == 0) {
		v.n_sel[s] = take;
		v.cut[s] = kNoCut;
		v.first_solved[s] = kNoSolved;
		if (!active) v.done[s] = 1;
		if (s == 0) *n_active = 0;
	}
}

// New children get index count + rank + 1 in batch order; those that can be popped later (index < M) are stored with parent
// and action.  The child numbered max_states marks the cut, and the first solved new child is kept by (rank, position).
__global__ void __launch_bounds__(kThreads) k_assign(View v, int64_t max_states) {
	const int s = blockIdx.y, i = blockIdx.x * kThreads + threadIdx.x;
	rbl::NewChild c;
	if (!rbl::number_new_child(v, s, i, c)) return;
	if (c.idx < v.M) {
		const int64_t row = (int64_t)s * v.M + c.idx;
		uint32_t* dst = reinterpret_cast<uint32_t*>(v.states + row * 20);
#pragma unroll
		for (int q = 0; q < 5; ++q) dst[q] = c.w[q];
		v.parents[row] = c.parent;
		v.parent_actions[row] = (uint8_t)(i % 12);
	}
	if ((int64_t)c.idx == max_states) v.cut[s] = i;
	if (rbl::is_solved(c.w)) atomicMin(&v.first_solved[s], ((unsigned long long)c.k << 32) | (unsigned)i);
}

// Firstpos re-arm of every probed slot; one thread per search applies the cut and the first-solved rule, advances count and
// head and counts the searches still running.
__global__ void __launch_bounds__(kThreads) k_finish(View v, int64_t max_states, int32_t* __restrict__ n_active) {
	const int s = blockIdx.y, i = blockIdx.x * kThreads + threadIdx.x;
	const int take = v.n_sel[s];
	rbl::rearm_firstpos(v, s, i, take);
	if (i != 0 || take == 0) return;
	const int cnt = v.count[s];
	const int cut = v.cut[s];
	const unsigned long long fs = v.first_solved[s];
	if (fs != kNoSolved) {
		const int pos = (int)(uint32_t)fs, rank = (int)(fs >> 32);
		if (cut == kNoCut || pos / 12 <= cut / 12) {             // its parent was popped: found before it is recorded
			v.count[s] = cnt + rank;
			v.won[s] = 1;
			v.done[s] = 1;
			v.solved_parent[s] = v.sel[(int64_t)s * v.N + pos / 12];
			v.solved_action[s] = (uint8_t)(pos % 12);
			return;
		}
	}
	if (cut != kNoCut) {
		// the parent of the cut records all its new children; no later parent is popped
		int adm = (int)(max_states - cnt);
		const uint8_t* f = v.flags + (int64_t)s * v.P();
		for (int q = cut + 1; q < (cut / 12 + 1) * 12; ++q) adm += f[q] & 1;
		v.count[s] = cnt + adm;
		v.done[s] = 1;
		return;
	}
	const int c2 = cnt + v.n_new[s], h2 = v.head[s] + take;
	v.count[s] = c2;
	v.head[s] = h2;
	if ((int64_t)c2 >= max_states || h2 > c2) { v.done[s] = 1; return; }
	atomicAdd(n_active, 1);
}

// Action queue of every won search: the path to the solved child's parent plus its action, uint8 [K][L]; lengths[s] is its
// length (0 for an unsolved search or a solved start), or -1 when it does not fit in L.
__global__ void __launch_bounds__(kThreads) k_paths(View v, uint8_t* __restrict__ queues, int32_t* __restrict__ lengths, int L) {
	const int s = blockIdx.x * kThreads + threadIdx.x;
	if (s >= v.K) return;
	if (!v.won[s] || v.solved_parent[s] == 0) { lengths[s] = 0; return; }
	const int32_t* par = v.parents + (int64_t)s * v.M;
	const uint8_t* act = v.parent_actions + (int64_t)s * v.M;
	int d = 1;
	for (int p = v.solved_parent[s]; p != 1 && d <= L; p = par[p]) ++d;
	if (d > L) { lengths[s] = -1; return; }
	uint8_t* q = queues + (int64_t)s * L;
	q[d - 1] = v.solved_action[s];
	int p = v.solved_parent[s];
	for (int e = d - 2; e >= 0; --e) { q[e] = act[p]; p = par[p]; }
	lengths[s] = d;
}

}  // namespace rbb
