"""
Search frontier on the device: the seen-set, child expansion and dedup that `BFS`, `AStar` and `MCTS` do with a
Python dict keyed on `state.tostring()` (reference: librubiks/solving/agents.py:96-123, 254-331, 511-544, 597-611).

`StateHashSet` is an open-addressing hash set on the packed state in caller-owned (torch) device memory with the
reference's index semantics: states are numbered 1, 2, ... in insertion order, a batch is numbered in batch order,
in-batch duplicates resolve to their first occurrence (agents.py:286-306).  `BFS` (layer-synchronous), `BFSBatch` (K
breadth-first searches in lockstep on the device) and `AStarBatch` (K searches in lockstep, open list and relaxation on the
device) carry the reference agents' interface
(`search(state, time_limit, max_states) -> bool`, `action_queue`, `len(agent)`).  The reference's host-side agent loops
(single-search A* around a heapq, MCTS' UCB walk) are not part of the product: tests/agent_harness.py replays them around
`StateHashSet` to check the device primitives against traces recorded from the reference.
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
	are converted (`rb_as2024`); an unreachable 6x8x6 start is an IndexError."""
	s = states if isinstance(states, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(states, dtype=np.int8))
	s = s.to(device=dev, dtype=torch.int8)
	if is2024:
		return s.reshape(-1, 20).contiguous()
	s = s.reshape(-1, 6, 8, 6).contiguous()
	roots = torch.empty(s.shape[0], 20, dtype=torch.int8, device=dev)
	ok = torch.empty(s.shape[0], dtype=torch.uint8, device=dev)
	N.check(N.lib.rb_as2024(N.ptr(s), N.ptr(roots), N.ptr(ok), s.shape[0], N.stream_handle()))
	if not bool(ok.all().item()):
		raise IndexError("a 6x8x6 start state is not a reachable cube")
	return roots


class AStarBatch:
	"""Batched weighted A* (agents.py:171-413) for K cubes at once, entirely on the device (SURVEY 8f rows N2 + N3): open
	list, seen-set, G / parent relaxation and the pop of the N cheapest states per search are kernels (csrc/rb_astar.cuh);
	the host only runs the value net on the contiguous batch of new states of all searches and reads two counters per step.
	Every search follows the reference's trace exactly (same pops, same state numbering, same G / parents / action queue).

	Both representations (the module flag, or `is2024`): the searches always run on the 20-byte states -- the two
	representations describe the same cube, children come in the same action order, so the trace is the same -- and with the
	6x8x6 representation the roots are converted on the way in (`rb_as2024`) and the new states are rendered as 6x8x6 rows
	(`rb_as686`) only to feed the value net its 288-wide one-hot.

	The launches of a step are two CUDA graphs (expand: 6 kernels + 1 memset, commit: 6 kernels), captured once per buffer set."""

	def __init__(self, net, lambda_: float, expansions: int, oh_dtype=torch.float32, is2024: bool | None = None, use_graphs: bool = True):
		N.require_cuda()
		if not 0 < expansions <= 1024:
			raise ValueError("expansions must be in 1..1024")
		self.net, self.lambda_, self.expansions = net, float(lambda_), int(expansions)
		self.is2024 = cube.get_is2024() if is2024 is None else bool(is2024)
		# torch.bfloat16 (opt-in, not the reference's dtype): bf16 one-hot rows and a bf16-autocast forward of the value net
		self.oh_dtype = oh_dtype
		self._as_oh = cube._oh_fn("rb_as_oh", oh_dtype)
		self.dev = torch.device("cuda", torch.cuda.current_device())
		self.use_graphs = use_graphs
		self.action_queue = deque()

	def _alloc(self, K: int, max_states: int):
		dev, Nx = self.dev, self.expansions
		M = max_states + 1
		if getattr(self, "_shape", None) == (K, M, Nx):           # buffers of the previous search_many are reused (everything that
			self.parents.zero_(); self.parent_actions.zero_()     # matters is re-initialised by rb_astar_init / rb_hashset_clear)
			self.in_open.zero_()
			return
		self._shape = (K, M, Nx)
		self.K, self.M = K, M
		self.states = torch.empty(K, M, 20, dtype=torch.int8, device=dev)
		self.G = torch.empty(K, M, dtype=torch.float64, device=dev)
		self.parents = torch.zeros(K, M, dtype=torch.int32, device=dev)
		self.parent_actions = torch.zeros(K, M, dtype=torch.uint8, device=dev)
		self.cost = torch.empty(K, M, dtype=torch.float64, device=dev)
		self.in_open = torch.zeros(K, M, dtype=torch.uint8, device=dev)
		self.count = torch.zeros(K, dtype=torch.int32, device=dev)
		self.n_sel = torch.zeros(K, dtype=torch.int32, device=dev)
		self.sel = torch.zeros(K, Nx, dtype=torch.int32, device=dev)
		self.won = torch.zeros(K, dtype=torch.uint8, device=dev)
		self.solved_index = torch.zeros(K, dtype=torch.int32, device=dev)
		self.capacity = _pow2_at_least(2 * K * M)                 # load <= 1/2 by construction: a search stores at most M states
		self.table = torch.empty(N.lib.rb_hashset_bytes(self.capacity), dtype=torch.uint8, device=dev)
		self.scratch = torch.empty(N.lib.rb_astar_scratch_bytes(K, Nx), dtype=torch.uint8, device=dev)
		P = 12 * Nx
		self.new_states = torch.empty(K * P, 20, dtype=torch.int8, device=dev)
		self.new_search = torch.empty(K * P, dtype=torch.int32, device=dev)
		self.new_index = torch.empty(K * P, dtype=torch.int32, device=dev)
		self.counters = torch.zeros(2, dtype=torch.int32, device=dev)          # n_new_total, n_active
		self.counters_host = torch.zeros(2, dtype=torch.int32, pin_memory=True)
		self.values = torch.zeros(K * P, dtype=torch.float32, device=dev)      # the net's output lands here: fixed address for the commit graph
		self.oh = torch.empty(K * P, 480 if self.is2024 else 288, dtype=self.oh_dtype, device=dev)
		self.new_states686 = None if self.is2024 else torch.empty(K * P, 6, 8, 6, dtype=torch.int8, device=dev)
		self.view = N.AStarView(K, M, Nx, *(N.ptr(t) for t in (self.states, self.G, self.parents, self.parent_actions, self.cost, self.in_open,
																 self.count, self.n_sel, self.sel, self.won, self.solved_index, self.table)),
								self.capacity, N.ptr(self.scratch))
		self._graphs = None

	# ---- the reference agents' interface, one cube (agents.py:221-252) ----
	_default_max_states = 1 << 20              # buffers are sized by the state budget: a search limited by time only gets this one

	def search(self, state, time_limit: float = None, max_states: int = None) -> bool:
		"""`AStar.search(state, time_limit, max_states)` for one cube on the batched machinery (K = 1): fills `action_queue`,
		`len(agent)` is the number of states stored.  The time limit is tested before every expansion step, like
		agents.py:238."""
		assert time_limit or max_states
		won, queues, count = self.search_many(np.asarray(state)[None] if not isinstance(state, torch.Tensor) else state[None],
											  int(max_states or self._default_max_states), time_limit=time_limit)
		self.action_queue = deque(queues[0])
		self._explored_states = int(count[0]) if not (won[0] and count[0] == 1 and not queues[0]) else 0      # solved start: nothing stored
		return bool(won[0])

	def __len__(self):
		return getattr(self, "_explored_states", 0)

	def __str__(self):
		return f"AStar (lambda={self.lambda_}, N={self.expansions})"

	def _step_calls(self, max_states: int):
		"""The two halves of a step as callables: plain C-ABI calls, or replays of their CUDA graphs (captured once per buffer set
		and budget; the graphs hold kernel launches only -- the value net runs between them, on however many new states there are)."""
		v = C.byref(self.view)
		n_total_ptr, n_active_ptr = C.c_void_p(self.counters.data_ptr()), C.c_void_p(self.counters.data_ptr() + 4)

		def expand():
			N.check(N.lib.rb_astar_expand(v, int(max_states), N.ptr(self.new_states), N.ptr(self.new_search), N.ptr(self.new_index),
										  n_total_ptr, n_active_ptr, N.stream_handle()))

		def commit():
			N.check(N.lib.rb_astar_commit(v, N.ptr(self.values), self.lambda_, N.ptr(self.new_search), N.ptr(self.new_index), n_total_ptr,
										  N.stream_handle()))

		if not self.use_graphs:
			return expand, commit
		if self._graphs is None or self._graphs[0] != int(max_states):
			ge, gc = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
			with torch.cuda.graph(ge):
				expand()
			with torch.cuda.graph(gc):
				commit()
			self._graphs = (int(max_states), ge, gc)
		return self._graphs[1].replay, self._graphs[2].replay

	@torch.no_grad()
	def search_many(self, states, max_states: int, max_steps: int | None = None, time_limit: float | None = None):
		"""states: (K, *shape) int8 (numpy or CUDA tensor).  Returns (solved bool (K,), action queues: list of K lists,
		len per search int (K,)), the three things `AStar.search` leaves behind for one cube."""
		t0 = perf_counter()
		roots = _roots2024(states, self.is2024, self.dev)
		self._alloc(roots.shape[0], int(max_states))
		self.net.eval()
		sh = N.stream_handle()
		def start():
			N.check(N.lib.rb_hashset_clear(N.ptr(self.table), self.capacity, sh))
			N.check(N.lib.rb_astar_init(C.byref(self.view), N.ptr(roots), sh))

		if self.use_graphs and self._graphs is None:
			# one plain expansion before the capture (tables uploaded, function attributes set: nothing of that may happen inside
			# a capture), then everything is initialised again
			start()
			N.check(N.lib.rb_astar_expand(C.byref(self.view), int(max_states), N.ptr(self.new_states), N.ptr(self.new_search), N.ptr(self.new_index),
										  C.c_void_p(self.counters.data_ptr()), C.c_void_p(self.counters.data_ptr() + 4), sh))
			torch.cuda.current_stream().synchronize()
		start()
		expand, commit = self._step_calls(max_states)
		self.steps = self.launches = 0
		l0 = N.lib.rb_launch_count()
		while (max_steps is None or self.steps < max_steps) and (time_limit is None or perf_counter() - t0 < time_limit):
			expand()
			self.counters_host.copy_(self.counters, non_blocking=True)           # the one host sync of a step
			torch.cuda.current_stream().synchronize()
			n_total, n_active = (int(x) for x in self.counters_host.tolist())
			if n_active == 0:
				break
			self._values(n_total)
			commit()
			self.steps += 1
		self.launches = N.lib.rb_launch_count() - l0
		return self._results()

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


class BFSBatch:
	"""Breadth-first search (agents.py:92-129) for K cubes at once, entirely on the device (csrc/rb_bfs.cuh): every search pops
	up to `_step` parents of its FIFO per step, with the reference's budget test before every pop, and all searches share one
	seen-set.  The host reads one counter per step (searches still running).  Each search's found flag, `len(agent)` and
	action queue are `BFS.search`'s for the same start and `max_states` (tests/golden/bfs_budget.npz).

	Both representations (the module flag, or `is2024`): the searches run on the 20-byte states, 6x8x6 starts are converted
	on the way in (`rb_as2024`)."""

	_step = 2048                                   # parents popped per search and step (changes no result)
	_queue_len = 16                                # a FIFO index below 2^29 has BFS depth <= 9
	_default_max_states = 1 << 20                  # buffers are sized by the state budget: a search limited by time only gets this one

	def __init__(self, is2024: bool | None = None):
		N.require_cuda()
		self.is2024 = cube.get_is2024() if is2024 is None else bool(is2024)
		self.dev = torch.device("cuda", torch.cuda.current_device())
		self.action_queue = deque()
		self._explored_states = 0

	def __len__(self):
		return self._explored_states

	def __str__(self):
		return "Breadth-first search (batched)"

	def _alloc(self, K: int, max_states: int):
		dev, Nx = self.dev, self._step
		M = max_states + 1
		if getattr(self, "_shape", None) == (K, M, Nx):           # every field a search reads is re-initialised by rb_bfs_init /
			return                                                # rb_hashset_clear
		self._shape = (K, M, Nx)
		self.K, self.M = K, M
		self.states = torch.empty(K, M, 20, dtype=torch.int8, device=dev)
		self.parents = torch.zeros(K, M, dtype=torch.int32, device=dev)
		self.parent_actions = torch.zeros(K, M, dtype=torch.uint8, device=dev)
		self.count = torch.zeros(K, dtype=torch.int32, device=dev)
		self.head = torch.zeros(K, dtype=torch.int32, device=dev)
		self.won = torch.zeros(K, dtype=torch.uint8, device=dev)
		self.done = torch.zeros(K, dtype=torch.uint8, device=dev)
		self.solved_parent = torch.zeros(K, dtype=torch.int32, device=dev)
		self.solved_action = torch.zeros(K, dtype=torch.uint8, device=dev)
		# load <= 1/2: a search holds at most M states plus the children of one step's dropped parents
		self.capacity = _pow2_at_least(2 * K * (M + 12 * Nx))
		self.table = torch.empty(N.lib.rb_hashset_bytes(self.capacity), dtype=torch.uint8, device=dev)
		self.scratch = torch.empty(N.lib.rb_bfs_scratch_bytes(K, Nx), dtype=torch.uint8, device=dev)
		self.n_active = torch.zeros(1, dtype=torch.int32, device=dev)
		self.n_active_host = torch.zeros(1, dtype=torch.int32, pin_memory=True)
		self.queues = torch.zeros(K, self._queue_len, dtype=torch.uint8, device=dev)
		self.lengths = torch.zeros(K, dtype=torch.int32, device=dev)
		self.view = N.BFSView(K, M, Nx, *(N.ptr(t) for t in (self.states, self.parents, self.parent_actions, self.count, self.head, self.won,
															 self.done, self.solved_parent, self.solved_action, self.table)),
							  self.capacity, N.ptr(self.scratch))

	def search(self, state, time_limit: float = None, max_states: int = None) -> bool:
		"""`BFS.search(state, time_limit, max_states)` for one cube on the batched machinery (K = 1): fills `action_queue` and
		`len(agent)`.  The time limit is tested before every step."""
		assert time_limit or max_states
		won, queues, count = self.search_many(np.asarray(state)[None] if not isinstance(state, torch.Tensor) else state[None],
											  int(max_states or self._default_max_states), time_limit=time_limit)
		self.action_queue = deque(queues[0])
		self._explored_states = int(count[0])
		return bool(won[0])

	@torch.no_grad()
	def search_many(self, states, max_states: int, time_limit: float | None = None):
		"""states: (K, *shape) int8 (numpy or CUDA tensor).  Returns (found bool (K,), action queues: list of K lists,
		len per search int (K,)), the three things `BFS.search` leaves behind for one cube (len 0 for a solved start)."""
		t0 = perf_counter()
		roots = _roots2024(states, self.is2024, self.dev)
		self._alloc(roots.shape[0], int(max_states))
		sh = N.stream_handle()
		v = C.byref(self.view)
		N.check(N.lib.rb_hashset_clear(N.ptr(self.table), self.capacity, sh))
		N.check(N.lib.rb_bfs_init(v, N.ptr(roots), sh))
		self.steps = 0
		l0 = N.lib.rb_launch_count()
		while time_limit is None or perf_counter() - t0 < time_limit:
			N.check(N.lib.rb_bfs_step(v, int(max_states), N.ptr(self.n_active), sh))
			self.steps += 1
			self.n_active_host.copy_(self.n_active, non_blocking=True)          # the one host read of a step
			torch.cuda.current_stream().synchronize()
			if int(self.n_active_host[0]) == 0:
				break
		N.check(N.lib.rb_bfs_paths(v, N.ptr(self.queues), N.ptr(self.lengths), self._queue_len, sh))
		self.launches = N.lib.rb_launch_count() - l0
		won = self.won.bool().cpu().numpy()
		count = self.count.cpu().numpy().astype(int)
		lengths = self.lengths.cpu().numpy()
		if (lengths < 0).any():
			raise N.RubiksError(f"an action queue is longer than {self._queue_len} moves")
		queues = self.queues.cpu().numpy()
		return won, [queues[s, :lengths[s]].tolist() for s in range(len(won))], count
