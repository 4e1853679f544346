"""
Search frontier on the device: the seen-set, child expansion and dedup that `BFS`, `AStar` and `MCTS` do with a
Python dict keyed on `state.tostring()` (reference: librubiks/solving/agents.py:96-123, 254-331, 511-544, 597-611).

`StateHashSet` is an open-addressing hash set on the packed state in caller-owned (torch) device memory with the
reference's index semantics: states are numbered 1, 2, ... in insertion order, a batch is numbered in batch order,
in-batch duplicates resolve to their first occurrence (agents.py:286-306).  `BFS` (layer-synchronous), `BFSBatch` (K
breadth-first searches in lockstep on the device), `AStarBatch` (K searches in lockstep, open list and relaxation on the
device) and `MCTSBatch` (K Monte Carlo tree searches in lockstep, node arrays and UCB walk on the device; the three batched
agents share their host driver, `_BatchAgent`) carry the reference agents' interface (`search(state, time_limit, max_states)
-> bool`, `action_queue`, `len(agent)`).  The reference's single-search host loops (A* around a heapq, MCTS' UCB walk) are
replayed statement by statement in tests/agent_harness.py around `StateHashSet`, as the test reference of the device
primitives and the batched agents.
"""
from __future__ import annotations

import ctypes as C
from collections import deque
from time import perf_counter

import numpy as np
import torch

from . import _native as N
from . import cube


def _pow2_at_least(x: int) -> int:
	return 1 << max(4, int(x - 1).bit_length())


def read_count(t: torch.Tensor) -> int:
	"""Host read of a device counter of the frontier kernels (`count`, `n_new`): -1 means a batch found the hash table full
	(include/rubiks_b200.h, RB_ERR_CAPACITY semantics without a sync inside the call)."""
	n = int(t.item())
	if n < 0:
		raise N.RubiksError(f"librubiks_b200 error {N.RB_ERR_CAPACITY}: the state hash set overflowed (table full); its contents are undefined")
	return n


class StateHashSet:
	def __init__(self, capacity: int = 1 << 16, is2024: bool | None = None):
		N.require_cuda()
		self.is2024 = cube.get_is2024() if is2024 is None else is2024
		self.rep = N.REP_2024 if self.is2024 else N.REP_686
		self.shape = (20,) if self.is2024 else (6, 8, 6)
		self.dev = torch.device("cuda", torch.cuda.current_device())
		self.capacity = _pow2_at_least(capacity)
		self.table = torch.empty(N.lib.rb_hashset_bytes(self.capacity), dtype=torch.uint8, device=self.dev)
		self.count = torch.zeros(1, dtype=torch.int32, device=self.dev)
		self.n_new = torch.zeros(1, dtype=torch.int32, device=self.dev)
		self._upper = 0                      # host-side upper bound of the set size (no sync needed)
		self._scratch = None
		self.clear()

	def clear(self):
		N.check(N.lib.rb_hashset_clear(N.ptr(self.table), self.capacity, N.stream_handle()))
		self.count.zero_()
		self._upper = 0

	def __len__(self) -> int:
		n = read_count(self.count)
		self._upper = n
		return n

	def _reserve(self, incoming: int):
		"""Keeps the load factor <= 1/2 using the host-side upper bound (exact size read back only when needed)."""
		if 2 * (self._upper + incoming) <= self.capacity:
			return
		len(self)
		if 2 * (self._upper + incoming) <= self.capacity:
			return
		new_cap = _pow2_at_least(4 * (self._upper + incoming))
		new_table = torch.empty(N.lib.rb_hashset_bytes(new_cap), dtype=torch.uint8, device=self.dev)
		N.check(N.lib.rb_hashset_rehash(N.ptr(self.table), self.capacity, N.ptr(new_table), new_cap, N.stream_handle()))
		self.table, self.capacity = new_table, new_cap

	def _scratch_for(self, nbytes: int) -> torch.Tensor:
		if self._scratch is None or self._scratch.numel() < nbytes:
			self._scratch = torch.empty(int(nbytes * 1.25) + 256, dtype=torch.uint8, device=self.dev)
		return self._scratch

	def _states(self, states):
		if isinstance(states, torch.Tensor):
			t, was_np = states.to(device=self.dev, dtype=torch.int8), False
		else:
			arr = np.ascontiguousarray(states, dtype=np.int8)
			t, was_np = torch.from_numpy(arr if arr.flags.writeable else arr.copy()).to(self.dev), True
		if t.dim() == len(self.shape):
			t = t.unsqueeze(0)
		if tuple(t.shape[1:]) != self.shape:
			raise IndexError(f"states of shape {tuple(t.shape)} do not match {self.shape}")
		return t.contiguous(), was_np

	def insert_unique(self, states):
		"""-> (seen bool (n,), first bool (n,), index int32 (n,)) with the semantics of agents.py:286-306."""
		s, was_np = self._states(states)
		n = s.shape[0]
		self._reserve(n)
		seen = torch.empty(n, dtype=torch.uint8, device=self.dev)
		first = torch.empty(n, dtype=torch.uint8, device=self.dev)
		index = torch.empty(n, dtype=torch.int32, device=self.dev)
		scratch = self._scratch_for(N.lib.rb_hashset_scratch_bytes(n))
		N.check(N.lib.rb_hashset_insert_unique(self.rep, N.ptr(self.table), self.capacity, N.ptr(s), n, N.ptr(self.count), N.ptr(seen),
											   N.ptr(first), N.ptr(index), N.ptr(scratch), N.stream_handle()))
		self._upper += n
		out = (seen.bool(), first.bool(), index)
		return tuple(x.cpu().numpy() for x in out) if was_np else out

	def lookup(self, states):
		"""Index of every state, 0 when absent (agents.py:606-607)."""
		s, was_np = self._states(states)
		n = s.shape[0]
		index = torch.empty(n, dtype=torch.int32, device=self.dev)
		scratch = self._scratch_for(N.lib.rb_hashset_scratch_bytes(n))
		N.check(N.lib.rb_hashset_lookup(self.rep, N.ptr(self.table), self.capacity, N.ptr(s), n, N.ptr(index), N.ptr(scratch), N.stream_handle()))
		return index.cpu().numpy() if was_np else index

	def expand(self, frontier: torch.Tensor, flags: bool = False, parents: bool = True, solved: bool = True, index: bool = False,
			   states: bool = True):
		"""One frontier step: 12 children of every frontier state, dedup against the set and within the batch, new states
		compacted in batch order.  Returns a dict of device tensors sized for the worst case (12 n rows); the first
		`n_new` rows are valid.  `n_new` itself stays on the device (`out['n_new']`) until the caller reads it.
		`states=False` (20x24 only): the new states are counted and entered into the set but not written out (the last layer of
		a closure)."""
		f, _ = self._states(frontier)
		n = f.shape[0]
		m = 12 * n
		self._reserve(m)
		out = {"next": torch.empty(m, *self.shape, dtype=torch.int8, device=self.dev) if states or not self.is2024 else None}
		out["parent"] = torch.empty(m, dtype=torch.int32, device=self.dev) if parents else None
		out["action"] = torch.empty(m, dtype=torch.uint8, device=self.dev) if parents else None
		out["solved"] = torch.empty(m, dtype=torch.uint8, device=self.dev) if solved else None
		out["seen"] = torch.empty(m, dtype=torch.uint8, device=self.dev) if flags else None
		out["first"] = torch.empty(m, dtype=torch.uint8, device=self.dev) if flags else None
		out["index"] = torch.empty(m, dtype=torch.int32, device=self.dev) if index else None
		scratch = self._scratch_for(N.lib.rb_frontier_scratch_bytes(self.rep, n))
		N.check(N.lib.rb_frontier_expand(self.rep, N.ptr(self.table), self.capacity, N.ptr(f), n, N.ptr(self.count), N.ptr(out["next"]),
										 N.ptr(out["parent"]), N.ptr(out["action"]), N.ptr(out["solved"]), N.ptr(out["seen"]),
										 N.ptr(out["first"]), N.ptr(out["index"]), N.ptr(self.n_new), N.ptr(scratch), N.stream_handle()))
		self._upper += m
		out["n_new"] = self.n_new
		return out


LAST_LAYER_MS = []


def bfs_layers(max_depth: int, start=None, is2024: bool | None = None, capacity: int | None = None, chain_items: int = 1 << 18):
	"""Layer-synchronous BFS closure from `start` (default solved): per-depth counts of newly discovered states
	(1, 12, 114, 1068, ... for the 20x24 cube) and the StateHashSet.  Everything but one int per layer stays on the device."""
	is2024 = cube.get_is2024() if is2024 is None else is2024
	hs = StateHashSet(capacity or (1 << 16), is2024)
	if start is None:
		start = cube._solved[hs.rep]
	frontier, _ = hs._states(start)
	hs.insert_unique(frontier)
	counts = [1]
	events = [torch.cuda.Event(enable_timing=True) for _ in range(max_depth + 1)]
	events[0].record()
	d = 0
	if is2024 and chain_items > 0:
		# the first layers are tiny: they are enqueued back to back with their sizes left on the device (the size of layer d+1 is
		# the n_new of layer d; grids and buffers are sized for the upper bound 12^d) and all counts are read with one sync
		n0, layers, bound = frontier.shape[0], 0, frontier.shape[0]
		while layers < max_depth - 1 and 12 * bound <= chain_items:
			layers, bound = layers + 1, 12 * bound
		if layers:
			sizes = torch.zeros(layers + 1, dtype=torch.int32, device=hs.dev)
			sizes[0] = n0
			hs._reserve(2 * bound)
			bufs = [torch.empty(bound, 20, dtype=torch.int8, device=hs.dev) for _ in range(2)]
			bufs[0][:n0] = frontier
			scratch = hs._scratch_for(N.lib.rb_frontier_scratch_bytes(hs.rep, bound // 12))
			N.check(N.lib.rb_frontier_expand_chain(hs.rep, N.ptr(hs.table), hs.capacity, N.ptr(bufs[0]), N.ptr(bufs[1]), n0, layers, N.ptr(sizes),
												   N.ptr(hs.count), N.ptr(scratch), N.stream_handle()))
			hs._upper += 2 * bound
			frontier, d = bufs[layers & 1], layers
			for k in range(1, d + 1):
				events[k].record()
		if d:
			got = sizes[1:d + 1].tolist()
			if min(got) < 0:
				read_count(sizes[1:d + 1].min())
			counts += [int(x) for x in got]
			frontier = frontier[:counts[-1]]
	while d < max_depth:
		last = d == max_depth - 1                    # nobody expands the last layer's states: they are entered into the set and counted only
		out = hs.expand(frontier, parents=False, solved=False, states=not last)
		events[d + 1].record()
		n_new = read_count(out["n_new"])
		frontier = out["next"][:n_new] if out["next"] is not None else None
		counts.append(n_new)
		d += 1
	global LAST_LAYER_MS
	LAST_LAYER_MS = [events[d].elapsed_time(events[d + 1]) for d in range(max_depth)]      # device time per layer (diagnostics)
	return counts, hs


class Agent:
	"""Interface of the reference agents (agents.py:14-64)."""

	def __init__(self):
		self.action_queue = deque()
		self._explored_states = 0

	def reset(self, time_limit, max_states):
		self._explored_states = 0
		self.action_queue = deque()
		if hasattr(self, "net"):
			self.net.eval()
		assert time_limit or max_states
		return time_limit or 1e10, max_states or int(1e10)

	def __len__(self):
		return self._explored_states


class BFS(Agent):
	"""Breadth-first search (agents.py:92-129) as layer-synchronous kernel sequences instead of one dict probe per child.

	The reference pops ONE parent at a time and tests its budget `len(self) < max_states` before every pop (agents.py:104),
	so a search that runs out of budget stops in the middle of a layer.  Parents are expanded here a slice of the FIFO
	frontier at a time; new children come back compacted in FIFO order with their parent position, so the parent at which
	the reference would have stopped is found by position: the last admitted parent is the one that records the
	(budget)-th new state, every later parent's children are dropped, and a solved child only counts under an admitted
	parent.  `len(agent)`, the found flag and the action queue are the reference's for any budget
	(tests/golden/bfs_budget.npz).  The time limit is tested once per slice, not once per parent."""

	_min_slice = 4096                              # parents per expansion when the budget is small

	def __init__(self, is2024: bool | None = None):
		super().__init__()
		self.is2024 = is2024

	def search(self, state, time_limit: float = None, max_states: int = None) -> bool:
		time_limit, max_states = self.reset(time_limit, max_states)
		t0 = perf_counter()
		is2024 = cube.get_is2024() if self.is2024 is None else self.is2024
		hs = StateHashSet(1 << 16, is2024)
		frontier, _ = hs._states(state)
		if bool((frontier[0].cpu().numpy() == cube._solved[hs.rep]).all()):
			return True
		hs.insert_unique(frontier)
		total = self._explored_states = 1
		layers = []                                   # per layer: (position of the parent in the previous layer, action)
		while frontier.shape[0] and total < max_states:
			nxt, par, act, done = [], [], [], 0
			while done < frontier.shape[0] and total < max_states and perf_counter() - t0 < time_limit:
				# never more parents than the remaining budget could admit if each recorded a single new state ...
				take = min(frontier.shape[0] - done, max(self._min_slice, max_states - total))
				out = hs.expand(frontier[done:done + take])
				n_new = read_count(out["n_new"])
				parent = out["parent"][:n_new]
				n_adm = n_new
				if total + n_new >= max_states:
					# ... and the parent that records new state number (max_states - total) is the last one popped
					last = parent[max_states - total - 1]
					n_adm = int(torch.searchsorted(parent, last, right=True).item())
				hit = torch.nonzero(out["solved"][:n_adm])
				par.append(parent[:n_adm] + done); act.append(out["action"][:n_adm])
				if hit.numel():
					k = int(hit[0].item())                # first solved new child in FIFO order
					# the reference returns before recording it: the dict holds the states discovered before it
					self._explored_states = total + k
					layers.append((torch.cat(par), torch.cat(act)))
					pos = sum(p.shape[0] for p in par[:-1]) + k
					for parent, action in reversed(layers):
						self.action_queue.appendleft(int(action[pos].item()))
						pos = int(parent[pos].item())
					return True
				total += n_adm
				self._explored_states = total
				nxt.append(out["next"][:n_adm])
				done += take
			if done < frontier.shape[0]:
				return False                              # budget or time ran out inside the layer
			layers.append((torch.cat(par), torch.cat(act)))
			frontier = torch.cat(nxt)
		return False

	def __str__(self):
		return "Breadth-first search"


def _roots2024(states, is2024: bool, dev) -> torch.Tensor:
	"""Start states (K, *shape) of a batched search as 20-byte device rows: the searches run on the 20x24 form, 6x8x6 starts
	are converted (`cube.to_2024`: an unreachable start is an IndexError)."""
	s = states if isinstance(states, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(states, dtype=np.int8))
	s = s.to(device=dev, dtype=torch.int8)
	return s.reshape(-1, 20).contiguous() if is2024 else cube.to_2024(s)


class _BatchAgent(Agent):
	"""K searches in lockstep on the device (csrc/rb_search.cuh), the part every such search has: the state rows, parents,
	counts and shared seen-set, the one-cube `search` of the reference agents' interface and the step loop of `search_many`.
	Both representations (the module flag, or `is2024`): the searches run on the 20-byte states, 6x8x6 starts are converted
	on the way in.  A subclass brings its buffers and C view (`_alloc`), its C calls for the scratch size and the init
	(`_c_scratch_bytes`, `_c_init`), one step (`_advance`) and the read-back (`_results`)."""

	_default_max_states = 1 << 20              # buffers are sized by the state budget: a search limited by time only gets this one

	def __init__(self, is2024: bool | None = None):
		super().__init__()
		N.require_cuda()
		self.is2024 = cube.get_is2024() if is2024 is None else bool(is2024)
		self.dev = torch.device("cuda", torch.cuda.current_device())

	def search(self, state, time_limit: float = None, max_states: int = None) -> bool:
		"""The reference agent's `search(state, time_limit, max_states)` for one cube on the batched machinery (K = 1): fills
		`action_queue`, and `len(agent)` is the number of states stored (0 for a solved start).  The time limit is tested before
		every step."""
		assert time_limit or max_states
		won, queues, count = self.search_many(np.asarray(state)[None] if not isinstance(state, torch.Tensor) else state[None],
											  int(max_states or self._default_max_states), time_limit=time_limit)
		self.action_queue = deque(queues[0])
		self._explored_states = 0 if won[0] and not queues[0] and count[0] <= 1 else int(count[0])
		return bool(won[0])

	def _alloc_core(self, K: int, M: int, Nx: int, keys: int) -> bool:
		"""The buffers every search has, for K searches of M state rows and up to Nx parents per step; `keys`: entries one search
		can hold in the seen-set, which is kept at load <= 1/2.  False when the previous call's buffers (same K, M, Nx) are
		reused: every field a search reads is re-initialised by its init and `rb_hashset_clear`."""
		if getattr(self, "_shape", None) == (K, M, Nx):
			return False
		self._shape = (K, M, Nx)
		self.K, self.M = K, M
		dev = self.dev
		self.states = torch.empty(K, M, 20, dtype=torch.int8, device=dev)
		self.parents = torch.zeros(K, M, dtype=torch.int32, device=dev)
		self.parent_actions = torch.zeros(K, M, dtype=torch.uint8, device=dev)
		self.count = torch.zeros(K, dtype=torch.int32, device=dev)
		self.won = torch.zeros(K, dtype=torch.uint8, device=dev)
		self.capacity = _pow2_at_least(2 * K * keys)
		self.table = torch.empty(N.lib.rb_hashset_bytes(self.capacity), dtype=torch.uint8, device=dev)
		self.scratch = torch.empty(self._c_scratch_bytes(K, Nx), dtype=torch.uint8, device=dev)
		self.counters = torch.zeros(2, dtype=torch.int32, device=dev)          # new states of the step (A* only), searches active
		self.counters_host = torch.zeros(2, dtype=torch.int32, pin_memory=True)
		return True

	def _start(self, roots: torch.Tensor, max_states: int):
		sh = N.stream_handle()
		N.check(N.lib.rb_hashset_clear(N.ptr(self.table), self.capacity, sh))
		N.check(self._c_init(C.byref(self.view), N.ptr(roots), sh))

	def _read(self):
		"""The one host read of a step: `counters` through the pinned buffer."""
		self.counters_host.copy_(self.counters, non_blocking=True)
		torch.cuda.current_stream().synchronize()
		return self.counters_host.tolist()

	@torch.no_grad()
	def _run(self, states, max_states: int, max_steps: int | None, time_limit: float | None):
		"""`search_many`: steps until `_advance` reports no search active, or `max_steps` / the time limit ends the call.
		`steps` counts the steps that ran, `launches` the library's kernel launches outside CUDA graphs from the first step to
		the end of the read-back."""
		t0 = perf_counter()
		max_states = int(max_states)
		roots = _roots2024(states, self.is2024, self.dev)
		self._alloc(roots.shape[0], max_states)
		self._start(roots, max_states)
		self.steps = 0
		l0 = N.lib.rb_launch_count()
		while (max_steps is None or self.steps < max_steps) and (time_limit is None or perf_counter() - t0 < time_limit):
			ran, active = self._advance(max_states)
			self.steps += ran
			if not active:
				break
		out = self._results()
		self.launches = N.lib.rb_launch_count() - l0
		return out


class AStarBatch(_BatchAgent):
	"""Batched weighted A* (agents.py:171-413) for K cubes at once, entirely on the device (SURVEY 8f rows N2 + N3): open
	list, seen-set, G / parent relaxation and the pop of the N cheapest states per search are kernels (csrc/rb_astar.cuh);
	the host only runs the value net on the contiguous batch of new states of all searches and reads two counters per step.
	Every search follows the reference's trace exactly (same pops, same state numbering, same G / parents / action queue).

	Both representations describe the same cube and children come in the same action order, so the trace is the same; with
	the 6x8x6 representation the new states are rendered as 6x8x6 rows (`rb_as686`) only to feed the value net its 288-wide
	one-hot.

	The launches of a step are two CUDA graphs (expand: 6 kernels + 1 memset, commit: 6 kernels), captured once per buffer set."""

	_c_scratch_bytes, _c_init = N.lib.rb_astar_scratch_bytes, N.lib.rb_astar_init

	def __init__(self, net, lambda_: float, expansions: int, oh_dtype=torch.float32, is2024: bool | None = None, use_graphs: bool = True):
		super().__init__(is2024)
		if not 0 < expansions <= 1024:
			raise ValueError("expansions must be in 1..1024")
		self.net, self.lambda_, self.expansions = net, float(lambda_), int(expansions)
		# torch.bfloat16 (opt-in, not the reference's dtype): bf16 one-hot rows and a bf16-autocast forward of the value net
		self.oh_dtype = oh_dtype
		self._as_oh = cube._oh_fn("rb_as_oh", oh_dtype)
		self.use_graphs = use_graphs

	def __str__(self):
		return f"AStar (lambda={self.lambda_}, N={self.expansions})"

	def _alloc(self, K: int, max_states: int):
		dev, Nx = self.dev, self.expansions
		M = max_states + 1
		if not self._alloc_core(K, M, Nx, M):    # a search stores at most M states
			self.parents.zero_(); self.parent_actions.zero_()     # reused buffers: rb_astar_init does not clear these
			self.in_open.zero_()
			return
		self.G = torch.empty(K, M, dtype=torch.float64, device=dev)
		self.cost = torch.empty(K, M, dtype=torch.float64, device=dev)
		self.in_open = torch.zeros(K, M, dtype=torch.uint8, device=dev)
		self.n_sel = torch.zeros(K, dtype=torch.int32, device=dev)
		self.sel = torch.zeros(K, Nx, dtype=torch.int32, device=dev)
		self.solved_index = torch.zeros(K, dtype=torch.int32, device=dev)
		P = 12 * Nx
		self.new_states = torch.empty(K * P, 20, dtype=torch.int8, device=dev)
		self.new_search = torch.empty(K * P, dtype=torch.int32, device=dev)
		self.new_index = torch.empty(K * P, dtype=torch.int32, device=dev)
		self.values = torch.zeros(K * P, dtype=torch.float32, device=dev)      # the net's output lands here: fixed address for the commit graph
		self.oh = torch.empty(K * P, 480 if self.is2024 else 288, dtype=self.oh_dtype, device=dev)
		self.new_states686 = None if self.is2024 else torch.empty(K * P, 6, 8, 6, dtype=torch.int8, device=dev)
		self.view = N.AStarView(K, M, Nx, *(N.ptr(t) for t in (self.states, self.G, self.parents, self.parent_actions, self.cost, self.in_open,
																 self.count, self.n_sel, self.sel, self.won, self.solved_index, self.table)),
								self.capacity, N.ptr(self.scratch))
		self._graphs = None

	def _start(self, roots: torch.Tensor, max_states: int):
		"""Also readies the two halves of a step: plain C-ABI calls, or replays of their CUDA graphs (captured once per buffer set;
		the graphs hold kernel launches only -- the value net runs between them, on however many new states there are)."""
		v = C.byref(self.view)
		n_total, n_active = N.ptr(self.counters[:1]), N.ptr(self.counters[1:])

		def expand():
			N.check(N.lib.rb_astar_expand(v, max_states, N.ptr(self.new_states), N.ptr(self.new_search), N.ptr(self.new_index), n_total, n_active,
										  N.stream_handle()))

		def commit():
			N.check(N.lib.rb_astar_commit(v, N.ptr(self.values), self.lambda_, N.ptr(self.new_search), N.ptr(self.new_index), n_total,
										  N.stream_handle()))

		if self.use_graphs and self._graphs is None:
			# one plain expansion before the capture (tables uploaded, function attributes set: nothing of that may happen inside
			# a capture), then everything is initialised again
			super()._start(roots, max_states)
			expand()
			torch.cuda.current_stream().synchronize()
		super()._start(roots, max_states)
		if self.use_graphs:
			if self._graphs is None:
				ge, gc = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
				with torch.cuda.graph(ge):
					expand()
				with torch.cuda.graph(gc):
					commit()
				self._graphs = ge, gc
			expand, commit = self._graphs[0].replay, self._graphs[1].replay
		self._expand, self._commit = expand, commit

	def search_many(self, states, max_states: int, max_steps: int | None = None, time_limit: float | None = None):
		"""states: (K, *shape) int8 (numpy or CUDA tensor).  Returns (solved bool (K,), action queues: list of K lists,
		len per search int (K,)), the three things `AStar.search` leaves behind for one cube."""
		self.net.eval()
		return self._run(states, max_states, max_steps, time_limit)

	def _advance(self, max_states: int):
		self._expand()
		n_total, n_active = self._read()
		if n_active == 0:
			return False, False
		self._values(n_total)
		self._commit()
		return True, True

	def _values(self, n: int):
		"""agents.py:379-381: one-hot born on the device, value head only; the f32 values land in `self.values[:n]`."""
		if n == 0:
			return
		oh = self.oh[:n]
		src = self.new_states
		rep = N.REP_2024
		if not self.is2024:
			N.check(N.lib.rb_as686(N.ptr(self.new_states), N.ptr(self.new_states686), n, N.stream_handle()))
			src, rep = self.new_states686, N.REP_686
		N.check(self._as_oh(rep, N.ptr(src), N.ptr(oh), n, N.stream_handle()))
		with torch.autocast("cuda", dtype=torch.bfloat16, enabled=self.oh_dtype == torch.bfloat16):
			val = self.net(oh, value=True, policy=False)
		self.values[:n].copy_(val.reshape(-1))

	def _results(self):
		won = self.won.bool().cpu().numpy()
		count = self.count.cpu().numpy().astype(int)
		solved_index = self.solved_index.cpu().numpy()
		queues = []
		for s in range(self.K):
			q = []
			if won[s] and solved_index[s] > 1:
				n = count[s] + 1
				parents, actions = self.parents[s, :n].cpu().numpy(), self.parent_actions[s, :n].cpu().numpy()
				i = int(solved_index[s])
				while i != 1:                                            # agents.py:245-251
					q.insert(0, int(actions[i]))
					i = int(parents[i])
			queues.append(q)
		return won, queues, count


class BFSBatch(_BatchAgent):
	"""Breadth-first search (agents.py:92-129) for K cubes at once, entirely on the device (csrc/rb_bfs.cuh): every search pops
	up to `_step` parents of its FIFO per step, with the reference's budget test before every pop, and all searches share one
	seen-set.  The host reads one counter per step (searches still running).  Each search's found flag, `len(agent)` and
	action queue are `BFS.search`'s for the same start and `max_states` (tests/golden/bfs_budget.npz)."""

	_step = 2048                                   # parents popped per search and step (changes no result)
	_queue_len = 16                                # a FIFO index below 2^29 has BFS depth <= 9
	_c_scratch_bytes, _c_init = N.lib.rb_bfs_scratch_bytes, N.lib.rb_bfs_init

	def __str__(self):
		return "Breadth-first search (batched)"

	def _alloc(self, K: int, max_states: int):
		dev, Nx = self.dev, self._step
		M = max_states + 1
		# a search holds at most M states plus the children of one step's dropped parents
		if not self._alloc_core(K, M, Nx, M + 12 * Nx):
			return
		self.head = torch.zeros(K, dtype=torch.int32, device=dev)
		self.done = torch.zeros(K, dtype=torch.uint8, device=dev)
		self.solved_parent = torch.zeros(K, dtype=torch.int32, device=dev)
		self.solved_action = torch.zeros(K, dtype=torch.uint8, device=dev)
		self.queues = torch.zeros(K, self._queue_len, dtype=torch.uint8, device=dev)
		self.lengths = torch.zeros(K, dtype=torch.int32, device=dev)
		self.view = N.BFSView(K, M, Nx, *(N.ptr(t) for t in (self.states, self.parents, self.parent_actions, self.count, self.head, self.won,
															 self.done, self.solved_parent, self.solved_action, self.table)),
							  self.capacity, N.ptr(self.scratch))

	def search_many(self, states, max_states: int, time_limit: float | None = None):
		"""states: (K, *shape) int8 (numpy or CUDA tensor).  Returns (found bool (K,), action queues: list of K lists,
		len per search int (K,)), the three things `BFS.search` leaves behind for one cube (len 0 for a solved start)."""
		return self._run(states, max_states, None, time_limit)

	def _advance(self, max_states: int):
		N.check(N.lib.rb_bfs_step(C.byref(self.view), max_states, N.ptr(self.counters[1:]), N.stream_handle()))
		return True, self._read()[1] > 0

	def _results(self):
		N.check(N.lib.rb_bfs_paths(C.byref(self.view), N.ptr(self.queues), N.ptr(self.lengths), self._queue_len, N.stream_handle()))
		won = self.won.bool().cpu().numpy()
		count = self.count.cpu().numpy().astype(int)
		lengths = self.lengths.cpu().numpy()
		if (lengths < 0).any():
			raise N.RubiksError(f"an action queue is longer than {self._queue_len} moves")
		queues = self.queues.cpu().numpy()
		return won, [queues[s, :lengths[s]].tolist() for s in range(len(won))], count


class MCTSBatch(_BatchAgent):
	"""Monte Carlo tree search (agents.py:415-645) for K cubes at once, entirely on the device (csrc/rb_mcts.cuh): every search
	expands one leaf per step, and the node arrays, the UCB walk with its virtual loss, the backup and, in graph mode
	(`search_graph`), the graph completion and the BFS that shortens the action queue are kernels.  The host runs the net on
	the contiguous batch of new states of all searches (`p, v = net(oh)`, P = `p.softmax(dim=1)`) and reads three counters
	per step.  Every search equals `MCTS.search` for the same start, net, `c`, `search_graph` and `max_states` node for node
	(`states`, `neighbors`, `leaves`, `N`, `W`, `V`, `P`; `L` counts the virtual loss in units of nu = 100), found flag,
	`len(agent)` and action queue.  Both representations, as `AStarBatch`: 6x8x6 rows are rendered only for the net's
	288-wide one-hot.

	A walk longer than `max_path` moves raises RubiksError.  A step is 6 plain kernel launches (expand: 4, commit: 2): capturing
	the two halves as CUDA graphs, as A* does, measured no faster (tools/mcts_batch_bench.py), since the net and the host read
	of each step dominate."""

	def __init__(self, net, c: float, search_graph: bool, is2024: bool | None = None, max_path: int = 1024):
		super().__init__(is2024)
		if max_path < 1:
			raise ValueError("max_path must be at least 1")
		self.net, self.c, self.search_graph, self.max_path = net, float(c), bool(search_graph), int(max_path)

	def __str__(self):
		return ("BFS" if self.search_graph else "Naive") + f" MCTS (c={self.c}, batched)"

	@staticmethod
	def _c_scratch_bytes(K: int, Nx: int):
		return N.lib.rb_mcts_scratch_bytes(K)

	_c_init = N.lib.rb_mcts_init

	def _alloc(self, K: int, max_states: int):
		dev = self.dev
		M = max_states + 1
		if not self._alloc_core(K, M, 1, M):        # a search stores at most M nodes; every row is written when numbered
			return
		self.neighbors = torch.empty(K, M, 12, dtype=torch.int32, device=dev)
		self.leaves = torch.empty(K, M, dtype=torch.uint8, device=dev)
		self.P = torch.empty(K, M, 12, dtype=torch.float32, device=dev)
		self.V = torch.empty(K, M, dtype=torch.float32, device=dev)
		self.N = torch.empty(K, M, 12, dtype=torch.int32, device=dev)
		self.W = torch.empty(K, M, 12, dtype=torch.float32, device=dev)
		self.L = torch.empty(K, M, 12, dtype=torch.int32, device=dev)
		self.solved_index = torch.zeros(K, dtype=torch.int32, device=dev)
		self.path_node = torch.zeros(K, self.max_path, dtype=torch.int32, device=dev)
		self.path_action = torch.zeros(K, self.max_path, dtype=torch.uint8, device=dev)
		self.path_len = torch.zeros(K, dtype=torch.int32, device=dev)
		self.order = torch.empty(K, M, dtype=torch.int32, device=dev)
		self.new_states = torch.empty(12 * K, 20, dtype=torch.int8, device=dev)
		self.new_search = torch.empty(12 * K, dtype=torch.int32, device=dev)
		self.new_index = torch.empty(12 * K, dtype=torch.int32, device=dev)
		self.new_states686 = None if self.is2024 else torch.empty(12 * K, 6, 8, 6, dtype=torch.int8, device=dev)
		self.oh = torch.empty(12 * K, 480 if self.is2024 else 288, dtype=torch.float32, device=dev)
		self.probs = torch.zeros(12 * K, 12, dtype=torch.float32, device=dev)       # the net's outputs land here
		self.values = torch.zeros(12 * K, dtype=torch.float32, device=dev)
		self.root_search = torch.arange(K, dtype=torch.int32, device=dev)
		self.root_index = torch.ones(K, dtype=torch.int32, device=dev)
		self.root_total = torch.full((1,), K, dtype=torch.int32, device=dev)
		self.queues = torch.zeros(K, self.max_path + 1, dtype=torch.uint8, device=dev)
		self.lengths = torch.zeros(K, dtype=torch.int32, device=dev)
		# new states of the step, searches expanding in the next step, walk overflow
		self.counters = torch.zeros(3, dtype=torch.int32, device=dev)
		self.counters_host = torch.zeros(3, dtype=torch.int32, pin_memory=True)
		self.view = N.MCTSView(K, M, self.max_path, *(N.ptr(t) for t in (
			self.states, self.parents, self.parent_actions, self.neighbors, self.leaves, self.P, self.V, self.N, self.W, self.L, self.count,
			self.won, self.solved_index, self.path_node, self.path_action, self.path_len, self.order, self.table)), self.capacity, N.ptr(self.scratch))

	def _net_rows(self, src: torch.Tensor, n: int):
		"""agents.py:470-472, 546-552: the net on the 20-byte rows src[:n]; softmax(policy) and value land in `probs[:n]` and
		`values[:n]`."""
		if n == 0:
			return
		oh, rep = self.oh[:n], N.REP_2024
		if not self.is2024:
			N.check(N.lib.rb_as686(N.ptr(src), N.ptr(self.new_states686), n, N.stream_handle()))
			src, rep = self.new_states686, N.REP_686
		N.check(N.lib.rb_as_oh(rep, N.ptr(src), N.ptr(oh), n, N.stream_handle()))
		p, v = self.net(oh)
		self.probs[:n].copy_(p.softmax(dim=1))
		self.values[:n].copy_(v.reshape(-1))

	def _start(self, roots: torch.Tensor, max_states: int):
		"""Roots, their net call, their P and V and the first walks."""
		self._max_states = max_states
		super()._start(roots, max_states)
		self._net_rows(roots, roots.shape[0])
		self._commit(self.root_search, self.root_index, self.root_total)

	def _expand(self):
		N.check(N.lib.rb_mcts_expand(C.byref(self.view), N.ptr(self.new_states), N.ptr(self.new_search), N.ptr(self.new_index),
									 N.ptr(self.counters[0:1]), N.stream_handle()))

	def _commit(self, search: torch.Tensor, index: torch.Tensor, total: torch.Tensor):
		N.check(N.lib.rb_mcts_commit(C.byref(self.view), N.ptr(self.probs), N.ptr(self.values), N.ptr(search), N.ptr(index), N.ptr(total), self.c,
									 self._max_states, N.ptr(self.counters[1:2]), N.ptr(self.counters[2:3]), N.stream_handle()))

	def search_many(self, states, max_states: int, max_steps: int | None = None, time_limit: float | None = None):
		"""states: (K, *shape) int8 (numpy or CUDA tensor).  Returns (found bool (K,), action queues: list of K lists, len per
		search int (K,)), the three things `MCTS.search` leaves behind for one cube (len 1 for a solved start).  A search cut
		off by the budget returns the actions of its last walk."""
		self.net.eval()
		return self._run(states, max_states, max_steps, time_limit)

	def search(self, state, time_limit: float = None, max_states: int = None) -> bool:
		"""`_BatchAgent.search`, with MCTS' len: the nodes stored, 1 for a solved start (agents.py:466-468 store the root first)."""
		won = super().search(state, time_limit, max_states)
		self._explored_states = int(self._count[0])
		return won

	def _check_overflow(self, flag: int):
		if flag:
			raise N.RubiksError(f"an MCTS walk needs more than max_path = {self.max_path} moves")

	def _advance(self, max_states: int):
		self._expand()
		n_total, n_active, overflow = self._read()
		self._check_overflow(overflow)
		if n_active == 0:
			return False, False
		self._net_rows(self.new_states, n_total)
		self._commit(self.new_search, self.new_index, self.counters[0:1])
		return True, True

	def _results(self):
		N.check(N.lib.rb_mcts_finish(C.byref(self.view), int(self.search_graph), N.ptr(self.queues), N.ptr(self.lengths), self.max_path + 1,
									 N.stream_handle()))
		self._check_overflow(int(self.counters[2].item()))
		won = self.won.bool().cpu().numpy()
		self._count = count = self.count.cpu().numpy().astype(int)
		lengths = self.lengths.cpu().numpy()
		if (lengths < 0).any():
			raise N.RubiksError(f"an action queue is longer than {self.max_path + 1} moves")
		queues = self.queues.cpu().numpy()
		return won, [queues[s, :lengths[s]].tolist() for s in range(len(won))], count
