// Batched Monte Carlo tree search on the device: K independent searches advance in lockstep, one leaf expansion per search
// and step.
//
// Replaces the host side of MCTS.search (reference: librubiks/solving/agents.py:461-633) -- the node arrays, the sequential
// UCB walk, the backup, the graph completion and the BFS that shortens the action queue -- for many cubes at once.  Every
// search reproduces the reference's trace node for node (tests/agent_harness.py::MCTS is the statement-by-statement replay):
//   * the leaf's 12 children are deduplicated and numbered by the lockstep expansion core with N = 1 (rb_search.cuh: probe,
//     flag, totals, then k_assign here), so new nodes are numbered in action order;
//   * the walk scores U + (W - L) with U = ((c P) sqrt(sum N)) / (1 + N) in double, rounded op by op (no FMA), and takes the
//     first maximum with numpy's argmax rule (the first NaN wins);
//   * the backup follows numpy's fancy-index semantics: W = maximum(W, max of the step's new values) (NaN propagates),
//     N += 1 once per distinct (node, action) pair of the walk, then L = 0 on the walk's pairs and their reverses.  L counts
//     the virtual loss in units of nu = 100 and is zero everywhere outside the running walk.
// A node's row is written in full when the node is numbered, so reused buffers need no clearing.
// 20x24 representation only.  Buffers are caller-owned (rb_mcts_view, include/rubiks_b200.h).
#pragma once
#include "rb_search.cuh"

namespace rbm {

using rbl::kThreads;
constexpr int kWalkWarps = kThreads / 32;         // searches per block of k_walk (one warp each)
constexpr int kNotFound = 0x7fffffff;             // discovery key of a node the shortening BFS has not reached

struct View : rbl::Core {           // device-side copy of rb_mcts_view; N = 1 (the leaf), n_sel / sel: scratch
	int32_t* neighbors;             // [K][M][12]
	uint8_t* leaves;                // [K][M]
	float* Pv;                      // [K][M][12] P (Core::P() is the expansion width)
	float* V;                       // [K][M]
	int32_t* Nv;                    // [K][M][12]
	float* W;                       // [K][M][12]
	int32_t* L;                     // [K][M][12] virtual loss, in units of nu
	int32_t* solved_index;          // [K]
	int32_t* path_node;             // [K][max_path] the walk: node j and the action taken there
	uint8_t* path_action;           // [K][max_path]
	int32_t* path_len;              // [K]
	int32_t* order;                 // [K][M] FIFO of the graph shortening
	int max_path;
};

// W, N, L and the neighbours zero, leaf flag set: the row of a node just numbered (P and V come from the net)
__device__ __forceinline__ void clear_row(const View& v, int64_t row) {
#pragma unroll
	for (int a = 0; a < 12; ++a) {
		v.neighbors[row * 12 + a] = 0;
		v.Nv[row * 12 + a] = 0;
		v.W[row * 12 + a] = 0.f;
		v.L[row * 12 + a] = 0;
	}
	v.leaves[row] = 1;
}

// np.maximum: NaN if either is NaN
__device__ __forceinline__ float nan_max(float a, float b) { return (a != a || b != b) ? __int_as_float(0x7fc00000) : (a >= b ? a : b); }

// (y, j) beats (x, i) under numpy's argmax: the first NaN, else the first maximum.  Index -1: no candidate.
__device__ __forceinline__ bool beats(double x, int i, double y, int j) {
	if (j < 0) return false;
	if (i < 0) return true;
	const bool xn = x != x, yn = y != y;
	if (xn || yn) return yn && (!xn || j < i);
	return y > x || (y == x && j < i);
}

// roots: state 1 of every search (a solved start is found at once with len 1, agents.py:466-468); rows 0 and 1 are cleared
// (row 0 is the reference's unused node: leaf flag set, no neighbours).  The first commit writes P and V of the roots.
__global__ void __launch_bounds__(kThreads) k_init(View v, const int8_t* __restrict__ roots) {
	const int s = blockIdx.x * kThreads + threadIdx.x;
	if (s >= v.K) return;
	const bool solved = rbl::init_root(v, s, roots);
	const int64_t base = (int64_t)s * v.M;
	clear_row(v, base);
	clear_row(v, base + 1);
	v.count[s] = 1;
	v.solved_index[s] = 0;
	v.path_len[s] = 0;
	v.sel[s] = 1;
	v.n_sel[s] = solved ? 0 : 1;
}

// ---- expansion: assign, after rbl::k_probe / k_flag / k_totals (grid 1 x K) ------------------------------------------------
// agents.py:511-544.  New children get index count + rank + 1 in action order, a full row and a place in the contiguous batch
// (state + search + index) the net runs on; all 12 children become the leaf's neighbours and the leaf theirs.
__global__ void __launch_bounds__(kThreads)
k_assign(View v, int8_t* __restrict__ new_states, int32_t* __restrict__ new_search, int32_t* __restrict__ new_index) {
	const int s = blockIdx.y, i = threadIdx.x;
	rbl::NewChild c;
	const bool is_new = rbl::number_new_child(v, s, i, c);
	if (i >= v.n_sel[s] * 12) return;
	const int64_t base = (int64_t)s * v.M;
	const int leaf = v.sel[s];
	int idx;
	if (is_new) {
		idx = c.idx;
		const int64_t row = base + idx;
		uint32_t* dst = reinterpret_cast<uint32_t*>(v.states + row * 20);
		const int64_t j = (int64_t)v.off[s] + c.k;
		uint32_t* dst2 = reinterpret_cast<uint32_t*>(new_states + j * 20);
#pragma unroll
		for (int q = 0; q < 5; ++q) { dst[q] = c.w[q]; dst2[q] = c.w[q]; }
		new_search[j] = s;
		new_index[j] = idx;
		v.parents[row] = leaf;
		v.parent_actions[row] = (uint8_t)i;
		clear_row(v, row);
		if (rbl::is_solved(c.w)) {                                  // at most one child is the solved state
			v.won[s] = 1;
			v.solved_index[s] = idx;
		}
	} else {
		idx = rbf::table_of(v.table, v.capacity).val(v.slot[(int64_t)s * v.P() + i]);
	}
	v.neighbors[(base + leaf) * 12 + i] = idx;
	v.neighbors[(base + idx) * 12 + (i ^ 1)] = leaf;
	if (i == 0) v.leaves[base + leaf] = 0;
}

// ---- commit ------------------------------------------------------------------------------------------------------------
// P (softmax already applied) and V of the new nodes, W = v on their rows.  The root's W row stays zero until its expansion,
// as in the reference.  Thread 0 re-arms the counters k_walk fills.
__global__ void __launch_bounds__(kThreads)
k_values(View v, const float* __restrict__ probs, const float* __restrict__ values, const int32_t* __restrict__ new_search,
         const int32_t* __restrict__ new_index, const int32_t* __restrict__ n_total, int32_t* __restrict__ n_active,
         int32_t* __restrict__ overflow) {
	const int64_t j = (int64_t)blockIdx.x * kThreads + threadIdx.x;
	if (j == 0) { *n_active = 0; *overflow = 0; }
	if (j >= *n_total) return;
	const int idx = new_index[j];
	const int64_t row = (int64_t)new_search[j] * v.M + idx;
	const float val = values[j];
	v.V[row] = val;
#pragma unroll
	for (int a = 0; a < 12; ++a) {
		v.Pv[row * 12 + a] = probs[j * 12 + a];
		if (idx != 1) v.W[row * 12 + a] = val;
	}
}

// One warp per search that ran this step: the backup of the expanded leaf (agents.py:546-573), then, unless the search is
// won, the next walk (agents.py:575-595) and the budget test len + 12 <= max_states for the next step.
__global__ void __launch_bounds__(kThreads)
k_walk(View v, double c, int64_t max_states, int32_t* __restrict__ n_active, int32_t* __restrict__ overflow) {
	const int lane = threadIdx.x & 31;
	const int s = blockIdx.x * kWalkWarps + (threadIdx.x >> 5);
	if (s >= v.K || !v.n_sel[s]) return;
	const int64_t base = (int64_t)s * v.M;
	const int leaf = v.sel[s];
	if (!v.leaves[base + leaf]) {                                    // expanded this step (the roots' first call expands nothing)
		const int cnt = v.count[s], nn = v.n_new[s];
		const int64_t lr = (base + leaf) * 12;
		if (lane < 12) v.W[lr + lane] = v.V[base + v.neighbors[lr + lane]];
		float m = lane < nn ? v.V[base + cnt + 1 + lane] : -INFINITY;
#pragma unroll
		for (int o = 16; o > 0; o >>= 1) m = nan_max(m, __shfl_xor_sync(0xffffffffu, m, o));
		if (lane == 0) {
			v.count[s] = cnt + nn;
			const int len = v.path_len[s];
			const int32_t* pn = v.path_node + (int64_t)s * v.max_path;
			const uint8_t* pa = v.path_action + (int64_t)s * v.max_path;
			// every pair of the walk holds L > 0 until this pass zeroes it: N counts each distinct pair once
			for (int j = 0; j < len; ++j) {
				const int64_t e = (base + pn[j]) * 12 + pa[j];
				if (v.L[e] != 0) {
					v.L[e] = 0;
					v.Nv[e] += 1;
					if (nn) v.W[e] = nan_max(v.W[e], m);
				}
			}
			for (int j = 0; j < len; ++j) {
				const int next = j + 1 < len ? pn[j + 1] : leaf;
				v.L[(base + next) * 12 + (pa[j] ^ 1)] = 0;
			}
		}
		__syncwarp();
	}
	if (v.won[s]) {
		if (lane == 0) v.n_sel[s] = 0;
		return;
	}
	int cur = 1, len = 0;
	while (!v.leaves[base + cur] && len < v.max_path) {
		const int64_t r = (base + cur) * 12;
		const int n = lane < 12 ? v.Nv[r + lane] : 0;
		int sum = n;
#pragma unroll
		for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
		double score = 0.0;
		int arg = -1;
		if (lane < 12) {
			const double u = __ddiv_rn(__dmul_rn(__dmul_rn(c, (double)v.Pv[r + lane]), __dsqrt_rn((double)sum)), (double)(1 + n));
			const double q = __dsub_rn((double)v.W[r + lane], __dmul_rn((double)v.L[r + lane], 100.0));
			score = __dadd_rn(u, q);
			arg = lane;
		}
#pragma unroll
		for (int o = 16; o > 0; o >>= 1) {
			const double y = __shfl_xor_sync(0xffffffffu, score, o);
			const int j = __shfl_xor_sync(0xffffffffu, arg, o);
			if (beats(score, arg, y, j)) { score = y; arg = j; }
		}
		const int nxt = v.neighbors[r + arg];
		if (lane == 0) {
			v.L[r + arg] += 1;
			v.L[(base + nxt) * 12 + (arg ^ 1)] += 1;
			v.path_node[(int64_t)s * v.max_path + len] = cur;
			v.path_action[(int64_t)s * v.max_path + len] = (uint8_t)arg;
		}
		__syncwarp();
		cur = nxt;
		++len;
	}
	if (lane == 0) {
		const bool over = !v.leaves[base + cur];                   // the walk would need more than max_path moves
		v.path_len[s] = len;
		v.sel[s] = cur;
		const bool active = !over && (int64_t)v.count[s] + 12 <= max_states;
		v.n_sel[s] = active ? 1 : 0;
		if (active) atomicAdd(n_active, 1);
		if (over) atomicExch(overflow, 1);
	}
}

// ---- finish --------------------------------------------------------------------------------------------------------------
// agents.py:597-611 for the won searches (graph mode): the children of every leaf looked up in the search's own keys (0 when
// absent), entered into the neighbour table both ways.  Both assignments agree wherever they meet (child * a^-1 is the leaf),
// so the writes need no order; the reference's stray writes to row 0 are never made.
__global__ void __launch_bounds__(kThreads) k_complete(View v) {
	__shared__ __align__(16) uint8_t s_lut[RB_LUT_BYTES];
	const int s = blockIdx.y;
	if (!v.won[s]) return;
	rb_stage_lut2024(s_lut);
	__syncthreads();
	const int64_t base = (int64_t)s * v.M;
	const rbf::Table t = rbf::table_of(v.table, v.capacity);
	const int64_t items = 12 * (int64_t)v.count[s];
	for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < items; i += (int64_t)gridDim.x * kThreads) {
		const int node = (int)(i / 12) + 1, a = (int)(i % 12);
		if (!v.leaves[base + node]) continue;
		uint32_t w[5];
		const uint32_t* p = reinterpret_cast<const uint32_t*>(v.states + (base + node) * 20);
#pragma unroll
		for (int k = 0; k < 5; ++k) w[k] = p[k];
		rb_move2024(s_lut, (uint32_t)a, w);
		const int64_t slot = rbf::find_only(t, rbl::key(w, s));
		const int idx = slot >= 0 ? t.val(slot) : 0;
		v.neighbors[(base + node) * 12 + a] = idx;
		if (idx) v.neighbors[(base + idx) * 12 + (a ^ 1)] = node;
	}
}

// Action queue of every search, uint8 [K][Lq]; lengths[s] its length, or -1 when it does not fit.  One block per search.
//   graph mode, won: agents.py:613-633, the BFS over the neighbour table from node 1, layer by layer.  A node's discovery key
//     is the least (FIFO position of the discoverer) * 12 + action over its discoverers (atomicMin, the firstpos race), which
//     is the sequential FIFO's first discovery; the winners of a layer are appended in key order.  The BFS stops at the first
//     layer that discovers the solved node.  `parents` holds the keys.
//   otherwise: the actions of the last walk, plus the solving action when won (a solved start: empty).
__global__ void __launch_bounds__(kThreads)
k_queue(View v, int graph, uint8_t* __restrict__ queues, int32_t* __restrict__ lengths, int Lq) {
	__shared__ int32_t s_warp[kThreads / 32];
	const int s = blockIdx.x, t = threadIdx.x;
	const int64_t base = (int64_t)s * v.M;
	const int target = v.solved_index[s];
	uint8_t* out = queues + (int64_t)s * Lq;
	if (!(graph && v.won[s] && target > 1)) {
		if (t != 0) return;
		const int len = v.path_len[s];                              // 0 for a solved start
		const int d = len + (target > 1 ? 1 : 0);
		if (d > Lq) { lengths[s] = -1; return; }
		for (int j = 0; j < len; ++j) out[j] = v.path_action[(int64_t)s * v.max_path + j];
		if (target > 1) out[len] = v.parent_actions[base + target];
		lengths[s] = d;
		return;
	}
	int32_t* key = v.parents + base;
	int32_t* q = v.order + base;
	const int32_t* nb = v.neighbors + base * 12;
	const int cnt = v.count[s];
	for (int i = t; i <= cnt; i += kThreads) key[i] = kNotFound;
	__syncthreads();
	if (t == 0) { key[1] = -1; q[0] = 1; }
	__syncthreads();
	int lo = 0, hi = 1;
	bool found = false;
	while (lo < hi) {
		const int64_t end = (int64_t)hi * 12;
		for (int64_t j = (int64_t)lo * 12 + t; j < end; j += kThreads) {
			const int n = nb[(int64_t)q[j / 12] * 12 + j % 12];
			if (n) atomicMin(&key[n], (int)j);
		}
		__syncthreads();
		found = __ldcg(&key[target]) != kNotFound;
		if (found) break;
		int tail = hi;
		for (int64_t j0 = (int64_t)lo * 12; j0 < end; j0 += kThreads) {
			const int64_t j = j0 + t;
			int n = 0;
			if (j < end) n = nb[(int64_t)q[j / 12] * 12 + j % 12];
			const bool win = n && __ldcg(&key[n]) == (int)j;
			int total;
			const int r = rbf::block_rank(win, s_warp, &total);
			if (win) q[tail + r] = n;
			tail += total;
			__syncthreads();                                        // s_warp is reused by the next chunk
		}
		lo = hi;
		hi = tail;
		__syncthreads();                                            // the new layer is in q
	}
	if (t != 0) return;
	if (!found) { lengths[s] = 0; return; }
	int d = 0;
	for (int n = target; n != 1; n = q[__ldcg(&key[n]) / 12]) ++d;
	if (d > Lq) { lengths[s] = -1; return; }
	int n = target;
	for (int e = d - 1; e >= 0; --e) {
		const int k = __ldcg(&key[n]);
		out[e] = (uint8_t)(k % 12);
		n = q[k / 12];
	}
	lengths[s] = d;
}

}  // namespace rbm
