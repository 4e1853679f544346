"""The deduplicated 3-move table of k_scramble_macro3 (rl_rubiks_b200/csrc/rb_scramble_macro.cuh): 1080 distinct elements
in eight copies, and a remap that gives, for every row index the kernel can form, the twist|flip word and the element.  Checked
against the raw 3-move and 2-move tables the library exports, without a GPU."""
import numpy as np

N_ELEMS, SINGLE, N_REMAP, COPIES = 1080, 2356, 2372, 8
IDX_MAX = 15 + 12 * 15 + 144 * 15          # largest index of 4-bit masked action bytes


def _tables():
	from rl_rubiks_b200 import _native as N
	elems = np.empty((N_ELEMS, 4), dtype=np.uint32)
	remap = np.empty((N_REMAP, 2), dtype=np.uint32)
	N.check(N.lib.rb_get_macro3_dedup(elems.ctypes.data, remap.ctypes.data))
	rows3 = np.empty((12 ** 3, 5), dtype=np.uint32)
	N.check(N.lib.rb_get_macro3_table(rows3.ctypes.data))
	rows2 = np.empty((13 ** 2, 5), dtype=np.uint32)
	N.check(N.lib.rb_get_macro_table(rows2.ctypes.data))
	return elems, remap, rows3, rows2


def _row(elems, remap, i):
	"""The five row words the kernel reads for remap index i (LDS.64 of the remap, LDS.128 of the element)."""
	tf, e = remap[i]
	return np.concatenate([elems[e], [tf]]).astype(np.uint32)


def test_1080_distinct_elements():
	elems, remap, rows3, _ = _tables()
	assert len({tuple(r) for r in elems}) == N_ELEMS
	assert len({tuple(r) for r in rows3[:, :4]}) == N_ELEMS          # the 1728 rows have no more selector parts than that
	assert set(remap[:12 ** 3, 1]) == set(range(N_ELEMS))


def test_remap_reproduces_every_row_of_the_raw_table():
	elems, remap, rows3, _ = _tables()
	inv = lambda a: a ^ 1
	for a2 in range(12):
		for a1 in range(12):
			for a0 in range(12):
				i = a0 + 12 * a1 + 144 * a2
				want = rows3[inv(a0) + 12 * inv(a1) + 144 * inv(a2)]
				assert (_row(elems, remap, i) == want).all(), (a0, a1, a2)


def test_single_move_entries_equal_the_one_move_elements():
	elems, remap, rows3, rows2 = _tables()
	for a in range(12):
		got = _row(elems, remap, SINGLE + a)
		assert (got == rows2[(a ^ 1) + 13 * 12]).all(), a          # 2-move row (a ^ 1, identity)
		assert (got == rows3[a + 12 * a + 144 * a]).all(), a        # a a a = a^-1 = a ^ 1
	for a in range(12, 16):
		assert remap[SINGLE + a, 0] == 0 and remap[SINGLE + a, 1] < N_ELEMS


def test_every_formable_index_stays_inside_the_staged_bytes():
	_, remap, _, _ = _tables()
	elem_bytes = N_ELEMS * COPIES * 16
	image_bytes = elem_bytes + N_REMAP * 8
	assert image_bytes % 16 == 0                                   # one bulk copy
	idx = np.concatenate([np.arange(IDX_MAX + 1), SINGLE + np.arange(16)])
	assert idx.max() < N_REMAP
	e = remap[idx, 1].astype(np.int64)
	assert (e * COPIES * 16 + (COPIES - 1) * 16 + 16 <= elem_bytes).all()
	invalid = np.arange(12 ** 3, IDX_MAX + 1)
	assert (remap[invalid, 0] == 0).all()                         # invalid actions: memory-safe, no twist or flip
