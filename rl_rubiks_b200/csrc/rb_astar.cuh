// Batched weighted A* on the device: K independent searches advance in lockstep, one expansion step per call sequence.
//
// Replaces the host side of AStar.search / expand_batch / relax_seen_states (reference:
// librubiks/solving/agents.py:221-367) -- the heapq open list, the dict, the numpy bookkeeping -- for many cubes at once
// (SURVEY 8f rows N2 + N3).  Every search reproduces the reference's trace exactly:
//   * the open list is one (cost f64, in_open) pair per stored state (a state is pushed once, when it is created, and
//     relaxations never re-push: agents.py:316-317, 333-367); popping the N smallest (cost, index) tuples of a heapq is
//     selecting and sorting the N smallest keys, done per search by one block (chunked bitonic sort + merge with a running
//     threshold);
//   * children of the popped parents are deduplicated and numbered by the lockstep expansion core (rb_search.cuh: probe,
//     flag, totals, then k_assign here);
//   * costs are lambda * G (f64) + H (f32 widened), H = -value, as agents.py:380-383;
//   * the two relaxation passes are vectorised numpy statements: all right-hand sides are evaluated before any write, and a
//     duplicate target keeps the LAST assignment (numpy fancy assignment).  They are therefore four small kernels:
//     evaluate / write "new ways" (targets unique), evaluate "shortcuts", write them per parent in action order.
// 20x24 representation only.  Buffers are caller-owned (rb_astar_view, include/rubiks_b200.h).
#pragma once
#include "rb_search.cuh"

namespace rba {

using rbl::kThreads;
constexpr int kSelThreads = 1024;
constexpr unsigned long long kInfKey = ~0ull;

// f64 -> u64 whose unsigned order is the numeric order (-0.0 is folded into +0.0; NaN sorts last, like nothing the reference
// could pop before finite costs).
__device__ __forceinline__ unsigned long long sortable(double c) {
	if (c == 0.0) c = 0.0;
	if (c != c) return kInfKey - 1;
	const unsigned long long b = (unsigned long long)__double_as_longlong(c);
	return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

struct View : rbl::Core {           // device-side copy of rb_astar_view
	double* G;
	double* cost;
	uint8_t* in_open;
	int32_t* solved_index;
	double* tmp;                    // scratch, [K][P]: the relaxation passes' right-hand sides
};

__device__ __forceinline__ bool lex_less(unsigned long long ka, uint32_t ia, unsigned long long kb, uint32_t ib) {
	return ka < kb || (ka == kb && ia < ib);
}

// ---- pop: the N smallest (cost, index) of the open list, ascending ------------------------------------------------------
// One block per search.  The open list is scanned once, 2048 entries per round (two coalesced loads in flight per thread);
// an entry that beats the running threshold -- the N-th best (key, index) so far, INF until N candidates were merged -- is
// appended to a staging buffer in shared memory.  Only when 1024 candidates are staged (or the scan ends) are they sorted
// (bitonic, descending) and merged into the running best 1024 (ascending): [best | chunk] is then bitonic and one merge
// network keeps the lower half.  With a tightening threshold the number of sort + merge rounds is ~(N / 1024)(1 + ln(n / N))
// instead of one per 1024 open entries.  Ties are broken by index, so the result does not depend on the staging order.
constexpr int kStage = 3072;                     // < 1024 left over + at most 2048 staged per round
constexpr int kSelSmem = (2048 + kStage) * (8 + 4) + 16;

__device__ __forceinline__ void sort_merge_1024(unsigned long long* s_key, uint32_t* s_idx, int t) {
	// bitonic sort of [1024, 2048), descending
	for (int size = 2; size <= 1024; size <<= 1)
		for (int stride = size >> 1; stride > 0; stride >>= 1) {
			const int j = t ^ stride;
			if (j > t) {
				const bool up = (t & size) != 0;                // mirrored direction bits => descending overall
				const int a = 1024 + t, b = 1024 + j;
				const bool a_gt_b = lex_less(s_key[b], s_idx[b], s_key[a], s_idx[a]);
				if (a_gt_b == up) {
					const unsigned long long tk = s_key[a]; s_key[a] = s_key[b]; s_key[b] = tk;
					const uint32_t ti = s_idx[a]; s_idx[a] = s_idx[b]; s_idx[b] = ti;
				}
			}
			__syncthreads();
		}
	// [best ascending | chunk descending] is bitonic: merge to ascending over all 2048, keep the lower half
	for (int stride = 1024; stride > 0; stride >>= 1) {
#pragma unroll
		for (int r = 0; r < 2; ++r) {
			const int e = t + 1024 * r, j = e ^ stride;
			if (j > e) {
				if (lex_less(s_key[j], s_idx[j], s_key[e], s_idx[e])) {
					const unsigned long long tk = s_key[e]; s_key[e] = s_key[j]; s_key[j] = tk;
					const uint32_t ti = s_idx[e]; s_idx[e] = s_idx[j]; s_idx[j] = ti;
				}
			}
		}
		__syncthreads();
	}
}

__global__ void __launch_bounds__(kSelThreads)
k_select(View v, int64_t max_states, int32_t* __restrict__ n_active) {
	extern __shared__ __align__(16) uint8_t sel_smem[];
	unsigned long long* s_key = reinterpret_cast<unsigned long long*>(sel_smem);               // [2048]: best | sort area
	unsigned long long* st_key = s_key + 2048;                                                  // [kStage]
	uint32_t* s_idx = reinterpret_cast<uint32_t*>(st_key + kStage);                             // [2048]
	uint32_t* st_idx = s_idx + 2048;                                                            // [kStage]
	int* s_cnt = reinterpret_cast<int*>(st_idx + kStage);
	const int s = blockIdx.x, t = threadIdx.x;
	const int cnt = v.count[s];
	const bool active = !v.won[s] && cnt > 0 && (int64_t)cnt + v.P() <= max_states;
	if (!active) {
		if (t == 0) v.n_sel[s] = 0;
		return;
	}
	const double* cost = v.cost + (int64_t)s * v.M;
	uint8_t* in_open = v.in_open + (int64_t)s * v.M;
	s_key[t] = kInfKey; s_idx[t] = 0xffffffffu;
	if (t == 0) *s_cnt = 0;
	__syncthreads();
	// moves the last min(staged, 1024) candidates into the sort area (INF padded) and merges them into the best
	auto flush = [&](int staged) {
		const int take = staged < 1024 ? staged : 1024, from = staged - take;
		if (t < take) { s_key[1024 + t] = st_key[from + t]; s_idx[1024 + t] = st_idx[from + t]; }
		else { s_key[1024 + t] = kInfKey; s_idx[1024 + t] = 0xffffffffu; }
		__syncthreads();
		if (t == 0) *s_cnt = from;
		sort_merge_1024(s_key, s_idx, t);                          // ends with a barrier
	};
	for (int base = 1; base <= cnt; base += 2 * kSelThreads) {
		const unsigned long long thr_k = s_key[v.N - 1];
		const uint32_t thr_i = s_idx[v.N - 1];
		const int i0 = base + t, i1 = base + kSelThreads + t;
		const bool o0 = i0 <= cnt && in_open[i0], o1 = i1 <= cnt && in_open[i1];
		const double c0 = o0 ? cost[i0] : 0.0, c1 = o1 ? cost[i1] : 0.0;
		if (o0) {
			const unsigned long long k = sortable(c0);
			if (lex_less(k, (uint32_t)i0, thr_k, thr_i)) { const int p = atomicAdd(s_cnt, 1); st_key[p] = k; st_idx[p] = (uint32_t)i0; }
		}
		if (o1) {
			const unsigned long long k = sortable(c1);
			if (lex_less(k, (uint32_t)i1, thr_k, thr_i)) { const int p = atomicAdd(s_cnt, 1); st_key[p] = k; st_idx[p] = (uint32_t)i1; }
		}
		__syncthreads();
		int staged = *s_cnt;
		__syncthreads();                                           // everyone has read the count before thread 0 rewrites it
		while (staged >= 1024) { flush(staged); staged -= 1024; }
	}
	{
		const int staged = *s_cnt;
		__syncthreads();
		if (staged > 0) flush(staged);
	}
	// pop
	if (t < v.N && s_key[t] != kInfKey) {
		v.sel[(int64_t)s * v.N + t] = (int32_t)s_idx[t];
		in_open[s_idx[t]] = 0;
	}
	const int n = __syncthreads_count(t < v.N && s_key[t] != kInfKey);
	if (t == 0) {
		v.n_sel[s] = n;
		if (n) atomicAdd(n_active, 1);
	}
}

// ---- expansion: assign, after rbl::k_probe / k_flag / k_totals ------------------------------------------------------------
// New children get index count + rank + 1 in batch order, are stored with G / parent / action, tested for solved and
// appended to the contiguous cost batch (state + search + index) the value net runs on.
__global__ void __launch_bounds__(kThreads)
k_assign(View v, int8_t* __restrict__ new_states, int32_t* __restrict__ new_search, int32_t* __restrict__ new_index) {
	const int s = blockIdx.y, i = blockIdx.x * kThreads + threadIdx.x;
	rbl::NewChild c;
	if (!rbl::number_new_child(v, s, i, c)) return;
	const int64_t row = (int64_t)s * v.M + c.idx;
	uint32_t* dst = reinterpret_cast<uint32_t*>(v.states + row * 20);
	const int64_t j = (int64_t)v.off[s] + c.k;
	uint32_t* dst2 = reinterpret_cast<uint32_t*>(new_states + j * 20);
#pragma unroll
	for (int q = 0; q < 5; ++q) { dst[q] = c.w[q]; dst2[q] = c.w[q]; }
	v.G[row] = v.G[(int64_t)s * v.M + c.parent] + 1.0;
	v.parent_actions[row] = (uint8_t)(i % 12);
	v.parents[row] = c.parent;
	new_search[j] = s;
	new_index[j] = c.idx;
	if (rbl::is_solved(c.w)) {
		v.won[s] = 1;
		v.solved_index[s] = c.idx;
	}
}

// cost = lambda * G + H, H = -value (agents.py:380-383: f64 * f64 + f32 widened), and the state enters the open list.
__global__ void __launch_bounds__(kThreads)
k_push(View v, const float* __restrict__ values, double lambda, const int32_t* __restrict__ new_search,
       const int32_t* __restrict__ new_index, const int32_t* __restrict__ n_total) {
	const int64_t j = (int64_t)blockIdx.x * kThreads + threadIdx.x;
	if (j >= *n_total) return;
	const int64_t row = (int64_t)new_search[j] * v.M + new_index[j];
	v.cost[row] = __dadd_rn(__dmul_rn(lambda, v.G[row]), (double)(-values[j]));
	v.in_open[row] = 1;
}

// ---- relaxation (agents.py:333-367) -----------------------------------------------------------------------------------------
// pass 1, evaluate: new_ways = G[parent] + 1 < G[state] for the seen first-occurrence children, on the G of before the pass
__global__ void __launch_bounds__(kThreads) k_relax_eval(View v, int pass) {
	const int s = blockIdx.y, i = blockIdx.x * kThreads + threadIdx.x;
	if (v.won[s] || i >= v.n_sel[s] * 12) return;
	const int64_t it = (int64_t)s * v.P() + i;
	uint8_t f = v.flags[it] & 3;
	if (f & 2) {
		const rbf::Table t = rbf::table_of(v.table, v.capacity);
		const int st = t.val(v.slot[it]), par = v.sel[(int64_t)s * v.N + i / 12];
		const double gs = v.G[(int64_t)s * v.M + st], gp = v.G[(int64_t)s * v.M + par];
		const double val = pass == 0 ? gp + 1.0 : gs + 1.0;     // new way to the state / shortcut to the parent
		if (pass == 0 ? val < gs : val < gp) { f |= 4; v.tmp[it] = val; }
	}
	v.flags[it] = f;
}
// pass 1, write: the targets (seen states) are unique within a search
__global__ void __launch_bounds__(kThreads) k_relax_new_ways(View v) {
	const int s = blockIdx.y, i = blockIdx.x * kThreads + threadIdx.x;
	if (v.won[s] || i >= v.n_sel[s] * 12) return;
	const int64_t it = (int64_t)s * v.P() + i;
	if (!(v.flags[it] & 4)) return;
	const rbf::Table t = rbf::table_of(v.table, v.capacity);
	const int64_t row = (int64_t)s * v.M + t.val(v.slot[it]);
	v.G[row] = v.tmp[it];
	v.parent_actions[row] = (uint8_t)(i % 12);
	v.parents[row] = v.sel[(int64_t)s * v.N + i / 12];
}
// pass 2, write: a parent may be the target of several of its 12 children; numpy keeps the last one
__global__ void __launch_bounds__(kThreads) k_relax_shortcuts(View v) {
	const int s = blockIdx.y, j = blockIdx.x * kThreads + threadIdx.x;
	if (v.won[s] || j >= v.n_sel[s]) return;
	const rbf::Table t = rbf::table_of(v.table, v.capacity);
	const int par = v.sel[(int64_t)s * v.N + j];
	const int64_t row = (int64_t)s * v.M + par;
	for (int a = 0; a < 12; ++a) {
		const int64_t it = (int64_t)s * v.P() + j * 12 + a;
		if (v.flags[it] & 4) {
			v.G[row] = v.tmp[it];
			v.parent_actions[row] = (uint8_t)(a ^ 1);               // rev_action
			v.parents[row] = t.val(v.slot[it]);
		}
	}
}

__global__ void __launch_bounds__(kThreads) k_finish(View v) {
	const int s = blockIdx.y, i = blockIdx.x * kThreads + threadIdx.x;
	const int n = v.n_sel[s];
	rbl::rearm_firstpos(v, s, i, n);
	if (i == 0) v.count[s] += n ? v.n_new[s] : 0;
}

// roots: state 1 of every search, G = 0, in the open list with cost 0 (agents.py:233-234)
__global__ void __launch_bounds__(kThreads) k_init(View v, const int8_t* __restrict__ roots) {
	const int s = blockIdx.x * kThreads + threadIdx.x;
	if (s >= v.K) return;
	const bool solved = rbl::init_root(v, s, roots);            // agents.py:230: a solved start returns True at once
	const int64_t row = (int64_t)s * v.M + 1;
	v.G[row] = 0.0;
	v.cost[row] = 0.0;
	v.in_open[row] = solved ? 0 : 1;
	v.count[s] = 1;
	v.solved_index[s] = solved ? 1 : 0;
	v.n_sel[s] = 0;
}

}  // namespace rba
