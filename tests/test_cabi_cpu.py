"""CPU-side checks of the C-ABI library: it loads, exports every symbol include/rubiks_b200.h declares, its
host-generated tables equal the reference's (golden fixtures) and the host helpers agree with numpy.
No kernel is launched here."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
	text = open(os.path.join(ROOT, "include", "rubiks_b200.h")).read()
	text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
	return sorted(set(re.findall(r"\b(rbh?_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
	from rl_rubiks_b200 import _native as N
	syms = _declared_symbols()
	assert len(syms) >= 25
	raw = ctypes.CDLL(N.LIB_PATH)
	for s in syms:
		assert hasattr(raw, s), f"{s} declared in include/rubiks_b200.h but not exported"
		assert s in N.SIGNATURES, f"{s} has no ctypes signature in _native.py"
	assert sorted(N.SIGNATURES) == syms
	assert N.lib.rb_version() >= 100


def test_host_tables_equal_reference(golden):
	from rl_rubiks_b200 import cube
	g = golden("tables")
	t = cube.tables()
	assert (t["delta_maps"] == g["delta_maps"]).all()
	assert (t["perm686"] == g["perm686"]).all()
	s = np.arange(24)
	for a in range(12):
		f, d = a // 2, 1 - a % 2
		assert (t["lut2024"][a] == s + g["delta_maps"][d, f]).all()
	assert (cube.get_solved() == g["solved2024"]).all()
	cube.set_is2024(False)
	try:
		assert (cube.get_solved() == g["solved686"]).all() and cube.shape() == (6, 8, 6) and cube.get_oh_shape() == 288
	finally:
		cube.set_is2024(True)
	assert cube.shape() == (20,) and cube.get_oh_shape() == 480


def test_action_helpers_match_reference_literals(golden):
	"""reference tests/test_cube.py:116-127 and the golden action tables."""
	from rl_rubiks_b200 import cube
	g = golden("tables")
	assert (cube.iter_actions(2) == g["iter_actions2"]).all() and cube.iter_actions(2).dtype == np.uint8
	f, d = cube.indices_to_actions(np.arange(12))
	assert (f == g["idx2act_faces"]).all() and (d == g["idx2act_dirs"]).all()
	assert (cube.rev_actions(np.arange(12)) == g["rev_actions"]).all()
	assert [cube.rev_action(a) for a in range(12)] == g["rev_actions"].tolist()
	assert (np.array(cube.action_space) == g["action_space"]).all() and cube.action_dim == 12
	assert (cube.repeat_state(cube.get_solved()) == np.tile(cube.get_solved(), (12, 1))).all()


def test_representation_flag_and_decorator():
	"""reference tests/test_rubiks.py:10-38."""
	from rl_rubiks_b200 import cube

	class Holder:
		is2024 = False

		@cube.with_used_repr
		def which(self):
			return cube.get_is2024()

	assert cube.get_is2024() is True
	assert Holder().which() is False and cube.get_is2024() is True
	cube.store_repr(); cube.set_is2024(False); assert not cube.get_is2024()
	cube.restore_repr(); assert cube.get_is2024()
	with pytest.raises(AssertionError):
		cube.set_is2024(1)


def test_stringify_literals():
	"""Presentation helpers against the reference's solved layout (tests/test_cube.py:33-43)."""
	from rl_rubiks_b200 import cube
	from oracle import cube_oracle as O
	for is2024 in (True, False):
		cube.set_is2024(is2024)
		try:
			assert cube.stringify(cube.get_solved()) == O.stringify(O.solved(is2024), is2024)
			s = O.scramble([0, 3, 5, 2], [1, 0, 0, 1], is2024)
			assert cube.stringify(s) == O.stringify(s, is2024) and (cube.as69(s) == O.as633(s, is2024).reshape(6, 9)).all()
		finally:
			cube.set_is2024(True)


@pytest.mark.parametrize("games,depth", [(1, 1), (3, 7), (6, 5), (1000, 25), (7500, 30), (17, 999), (5, 128), (2, 129)])
def test_weight_sum_is_numpy_pairwise(games, depth):
	from rl_rubiks_b200 import _native as N
	want = np.tile(1 / np.arange(1, depth + 1), games).sum()
	assert N.lib.rb_adi_weight_sum(games, depth) == want


def test_missing_gpu_fails_loudly():
	import torch
	from rl_rubiks_b200 import cube, _native as N
	if torch.cuda.is_available():
		pytest.skip("GPU present")
	with pytest.raises(N.RubiksError):
		cube.multi_rotate(np.zeros((1, 20), np.int8), [0], [1])


def test_hashset_capacity_limits_are_errors():
	"""Slot numbers travel in 30 bits: a larger table is refused (RB_ERR_CAPACITY) before anything is launched."""
	from rl_rubiks_b200 import _native as N
	assert N.lib.rb_hashset_bytes(1 << 20) == 32 << 20
	fake = ctypes.c_void_p(1 << 20)                                   # aligned, never dereferenced: the checks come first
	assert N.lib.rb_hashset_clear(fake, 1 << 31, None) == N.RB_ERR_CAPACITY
	assert N.lib.rb_hashset_clear(fake, (1 << 20) + 1, None) == N.RB_ERR_BAD_ARG
	assert N.lib.rb_hashset_clear(ctypes.c_void_p((1 << 20) + 16), 1 << 20, None) == N.RB_ERR_BAD_ARG
	assert N.lib.rb_hashset_rehash(fake, 1 << 10, fake, 1 << 31, None) == N.RB_ERR_CAPACITY
	# A* shares one table among K searches of up to M states: below 2 K M slots a full table would drop children silently.
	# roots / new_states / values are NULL, so no call can get past its argument checks to a launch.
	K, M, Nx = 3, 1000, 4
	v = N.AStarView(K, M, Nx, *([fake] * 12), 2048, fake)              # 2048 < 2 K M = 6000
	out = [fake] * 4
	assert N.lib.rb_astar_init(ctypes.byref(v), None, None) == N.RB_ERR_CAPACITY
	assert N.lib.rb_astar_expand(ctypes.byref(v), M - 1, None, *out, None) == N.RB_ERR_CAPACITY
	assert N.lib.rb_astar_commit(ctypes.byref(v), None, 0.5, *out[:3], None) == N.RB_ERR_CAPACITY
	v.K, v.M = 65535, 1 << 14                                           # 2 K M overflows 32 bits
	v.capacity = 1 << 30
	assert N.lib.rb_astar_init(ctypes.byref(v), None, None) == N.RB_ERR_CAPACITY
