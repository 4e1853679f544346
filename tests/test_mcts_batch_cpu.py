"""CPU checks of the batched MCTS's C ABI (csrc/rb_mcts.cuh, include/rubiks_b200.h): a bad view is refused before anything is
launched, as for the batched A* and BFS."""
import ctypes

FIELDS = ("states", "parents", "parent_actions", "neighbors", "leaves", "P", "V", "N", "W", "L", "count", "won", "solved_index",
		  "path_node", "path_action", "path_len", "order", "table", "scratch")


def _view(N, K, M, max_path, capacity, fake):
	return N.MCTSView(K, M, max_path, *([fake] * 18), capacity, fake)


def _calls(N, v, fake, out):
	"""Every entry point that takes a view, called with valid-looking other arguments."""
	v = ctypes.byref(v)
	return {
		"init": lambda: N.lib.rb_mcts_init(v, fake, None),
		"expand": lambda: N.lib.rb_mcts_expand(v, out, out, out, out, None),
		"commit": lambda: N.lib.rb_mcts_commit(v, fake, fake, fake, fake, fake, 1.0, 10, out, out, None),
		"finish": lambda: N.lib.rb_mcts_finish(v, 1, out, out, 16, None),
	}


def test_mcts_view_is_checked_before_any_launch():
	"""K is at most 65535 (the grid's y dimension); the table must hold 2 K M slots (computed without 32-bit overflow); no
	buffer may be null; max_path is at least 1.  Every pointer is fake and never dereferenced: the checks come first."""
	from rl_rubiks_b200 import _native as N
	fake = ctypes.c_void_p(1 << 20)
	out = ctypes.c_void_p(1 << 21)
	K, M = 3, 1000
	assert N.lib.rb_mcts_scratch_bytes(K) > 0 and N.lib.rb_mcts_scratch_bytes(0) == 0
	assert 4096 < 2 * K * M <= 8192
	for name, call in _calls(N, _view(N, K, M, 64, 4096, fake), fake, out).items():
		assert call() == N.RB_ERR_CAPACITY, name
	v = _view(N, 65535, 1 << 14, 64, 1 << 30, fake)                     # 2 K M overflows 32 bits
	assert N.lib.rb_mcts_init(ctypes.byref(v), fake, None) == N.RB_ERR_CAPACITY
	for bad in (_view(N, 65536, 2, 64, 1 << 30, fake), _view(N, 0, 2, 64, 1 << 30, fake), _view(N, K, M, 0, 8192, fake),
				_view(N, K, M, -1, 8192, fake), _view(N, 1, (1 << 27) + 1, 64, 1 << 30, fake)):
		for name, call in _calls(N, bad, fake, out).items():
			assert call() == N.RB_ERR_BAD_ARG, (bad.K, bad.M, bad.max_path, name)
	for field in FIELDS:
		v = _view(N, K, M, 64, 8192, fake)
		setattr(v, field, None)
		for name, call in _calls(N, v, fake, out).items():
			assert call() == N.RB_ERR_BAD_ARG, (field, name)
	v = _view(N, K, M, 64, 8192, fake)
	vp = ctypes.byref(v)
	assert N.lib.rb_mcts_init(vp, None, None) == N.RB_ERR_BAD_ARG
	assert N.lib.rb_mcts_expand(vp, None, out, out, out, None) == N.RB_ERR_BAD_ARG
	assert N.lib.rb_mcts_expand(vp, out, out, out, None, None) == N.RB_ERR_BAD_ARG
	assert N.lib.rb_mcts_commit(vp, None, fake, fake, fake, fake, 1.0, 10, out, out, None) == N.RB_ERR_BAD_ARG
	assert N.lib.rb_mcts_commit(vp, fake, fake, fake, fake, fake, 1.0, 10, out, None, None) == N.RB_ERR_BAD_ARG
	assert N.lib.rb_mcts_commit(vp, fake, fake, fake, fake, fake, 1.0, M, out, out, None) == N.RB_ERR_BAD_ARG   # M must exceed max_states
	assert N.lib.rb_mcts_finish(vp, 0, None, out, 16, None) == N.RB_ERR_BAD_ARG
	assert N.lib.rb_mcts_finish(vp, 0, out, out, 0, None) == N.RB_ERR_BAD_ARG
	assert N.lib.rb_mcts_init(None, fake, None) == N.RB_ERR_BAD_ARG
	assert N.lib.rb_mcts_expand(None, out, out, out, out, None) == N.RB_ERR_BAD_ARG
	assert N.lib.rb_mcts_commit(None, fake, fake, fake, fake, fake, 1.0, 10, out, out, None) == N.RB_ERR_BAD_ARG
	assert N.lib.rb_mcts_finish(None, 1, out, out, 16, None) == N.RB_ERR_BAD_ARG
