"""CPU checks of the batched BFS (csrc/rb_bfs.cuh): a numpy emulation of its sliced step equals BFS.search (agents.py:96-123,
restated by oracle.bfs_search) for every step size, and the C ABI refuses bad views before it launches anything."""
import ctypes

import numpy as np
import pytest

from oracle import cube_oracle as O


def sliced_bfs(start, max_states: int, N: int, is2024: bool = True):
	"""One step of every search in rb_bfs_step, restated: pop up to N parents from the FIFO (the stored states), number the
	new children in batch order, admit the parents before the one that records new state number max_states - count (the
	cut), and end at the first solved new child under an admitted parent.  -> (found, len, action queue)."""
	start = np.asarray(start)
	if O.is_solved(start, is2024):
		return True, 0, []
	seen = O.SeenSet()
	seen.insert_unique(start[None])
	states, parents, actions = [None, start], [0, 0], [0, 0]
	count, head = 1, 1
	while count < max_states and head <= count:
		take = min(N, count - head + 1)
		par = np.arange(head, head + take)
		children = O.expand12(np.stack([states[p] for p in par]), is2024)
		was_seen, first, _ = seen.insert_unique(children)
		new = np.flatnonzero(first & ~was_seen)                    # batch positions, in rank order
		rest = max_states - count
		cut = int(new[rest - 1]) if len(new) >= rest else None
		solved = [k for k, i in enumerate(new) if O.is_solved(children[i], is2024)]
		if solved:
			k = solved[0]
			i = int(new[k])
			if cut is None or i // 12 <= cut // 12:
				queue, p = [i % 12], int(par[i // 12])
				while p != 1:
					queue.insert(0, actions[p])
					p = parents[p]
				return True, count + k, queue
		if cut is not None:
			return False, count + int(np.count_nonzero(new // 12 <= cut // 12)), []
		for i in new:
			states.append(children[i]); parents.append(int(par[i // 12])); actions.append(int(i % 12))
		count += len(new)
		head += take
	return False, count, []


def test_sliced_step_equals_reference_on_golden_budgets(golden):
	"""The 152 searches recorded from the reference under binding budgets, both representations, at three step sizes."""
	g = golden("bfs_budget")
	for c in range(int(g["n_cases"])):
		start, max_states = g[f"start_{c}"], int(g[f"max_{c}"])
		is2024 = start.shape == (20,)
		want = (bool(g[f"found_{c}"]), int(g[f"len_{c}"]), g[f"queue_{c}"].tolist())
		for N in (1, 7, 4096):
			if N == 1 and max_states > 2000:
				continue                                               # one pop per step: slow in Python, nothing new
			assert sliced_bfs(start, max_states, N, is2024) == want, (c, N)


@pytest.mark.parametrize("N", [1, 7, 4096])
def test_sliced_step_equals_oracle_at_random(N):
	"""Random scrambles of depth 2-5, budgets that end in the first layers, inside a layer, at the solved child's step and
	just around it; a solved start."""
	rng = np.random.RandomState(5)
	for depth in (2, 3, 4, 5):
		for _ in range(2):
			start = O.scramble(rng.randint(0, 6, depth), rng.randint(0, 2, depth), True)
			found, length, _ = O.bfs_search(start, 10 ** 6)
			budgets = {1, 2, 12, 13, 14, 100, 127, max(1, length - 1), length, length + 1, length + 12}
			for m in sorted(b for b in budgets if b <= 3000):
				assert sliced_bfs(start, m, N) == O.bfs_search(start, m), (depth, m, N)
	assert sliced_bfs(O.solved(True), 5, N) == (True, 0, [])


def _view(N, K, M, Nx, capacity, fake):
	return N.BFSView(K, M, Nx, *([fake] * 10), capacity, fake)


def test_bfs_view_is_checked_before_any_launch():
	"""The table must hold 2 K (M + 12 N) slots (the children of dropped parents are claimed before the cut is known), computed
	without 32-bit overflow; K is at most 65535 (the grid's y dimension); no buffer may be null.  Every pointer is fake and
	never dereferenced: the checks come first."""
	from rl_rubiks_b200 import _native as N
	fake = ctypes.c_void_p(1 << 20)
	out = ctypes.c_void_p(1 << 21)
	K, M, Nx = 3, 1000, 4
	need = 2 * K * (M + 12 * Nx)                                       # 6288: a 4096-slot table is too small, 8192 is enough
	assert N.lib.rb_bfs_scratch_bytes(K, Nx) > 0 and N.lib.rb_bfs_scratch_bytes(0, Nx) == 0
	v = _view(N, K, M, Nx, 4096, fake)
	assert 4096 < need <= 8192
	assert N.lib.rb_bfs_init(ctypes.byref(v), fake, None) == N.RB_ERR_CAPACITY
	assert N.lib.rb_bfs_step(ctypes.byref(v), M - 1, out, None) == N.RB_ERR_CAPACITY
	assert N.lib.rb_bfs_paths(ctypes.byref(v), out, out, 16, None) == N.RB_ERR_CAPACITY
	# 2 K M alone (the A* rule) would fit in 8192 with a larger N: the 12 N term counts
	v = _view(N, K, M, 100, 8192, fake)
	assert N.lib.rb_bfs_init(ctypes.byref(v), fake, None) == N.RB_ERR_CAPACITY
	# 2 K (M + 12 N) above 2^31 (and above any table the library accepts)
	v = _view(N, 65535, 1 << 14, 1, 1 << 30, fake)
	assert N.lib.rb_bfs_init(ctypes.byref(v), fake, None) == N.RB_ERR_CAPACITY
	v = _view(N, 65535, 1 << 14, 1 << 20, 1 << 30, fake)               # 12 N K alone is above 2^39
	assert N.lib.rb_bfs_step(ctypes.byref(v), 10, out, None) == N.RB_ERR_CAPACITY
	# K beyond the grid's y dimension
	v = _view(N, 65536, 2, 1, 1 << 30, fake)
	assert N.lib.rb_bfs_init(ctypes.byref(v), fake, None) == N.RB_ERR_BAD_ARG
	# null buffers: each field of the view, and the call's own arguments
	for field in ("states", "parents", "parent_actions", "count", "head", "won", "done", "solved_parent", "solved_action", "table", "scratch"):
		v = _view(N, K, M, Nx, 8192, fake)
		setattr(v, field, None)
		assert N.lib.rb_bfs_init(ctypes.byref(v), fake, None) == N.RB_ERR_BAD_ARG, field
	v = _view(N, K, M, Nx, 8192, fake)
	assert N.lib.rb_bfs_init(ctypes.byref(v), None, None) == N.RB_ERR_BAD_ARG
	assert N.lib.rb_bfs_step(ctypes.byref(v), M - 1, None, None) == N.RB_ERR_BAD_ARG
	assert N.lib.rb_bfs_step(ctypes.byref(v), M, out, None) == N.RB_ERR_BAD_ARG           # M must exceed max_states
	assert N.lib.rb_bfs_paths(ctypes.byref(v), None, out, 16, None) == N.RB_ERR_BAD_ARG
	assert N.lib.rb_bfs_paths(ctypes.byref(v), out, None, 16, None) == N.RB_ERR_BAD_ARG
	assert N.lib.rb_bfs_init(None, fake, None) == N.RB_ERR_BAD_ARG
