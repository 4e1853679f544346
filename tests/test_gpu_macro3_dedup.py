"""k_scramble_macro3 on the deduplicated table against the oracle, in every kMode, with the depth % 3 trailing moves taken as
single-move rows of the remap: depth % 3 == 1 and == 2, and depth % 24 on each remainder branch (one or two single rows after
the 3-move rows, unaligned rows taken byte by byte).  One size spans more than one pass of the grid, so warps take a second
chunk after the table is staged."""
import numpy as np
import pytest

from oracle import cube_oracle as O

pytestmark = pytest.mark.gpu

# kMode 0 (depth % 4 != 0), 1 (depth % 4 == 0), 2 (depth % 16 == 0), 3 (depth % 128 == 0); each with depth % 3 == 1 and 2
DEPTHS = {
	0: [25, 26, 101, 103],
	1: [20, 44, 52, 100],
	2: [32, 64, 80, 112],
	3: [128, 256],
}
CASES = [pytest.param(m, d, id=f"mode{m}-d{d}") for m, ds in DEPTHS.items() for d in ds]


def _scramble(is2024, n, depth, seed):
	from rl_rubiks_b200 import cube
	cube.set_is2024(is2024)
	try:
		g = np.random.RandomState(seed)
		acts = g.randint(0, 12, (n, depth)).astype(np.uint8)
		f, d = O.indices_to_actions(acts)
		assert (cube.scramble_batch(acts) == O.scramble_many(f, d, is2024)).all(), (is2024, n, depth)
	finally:
		cube.set_is2024(True)


def test_depths_cover_every_mode_and_tail():
	for mode, depths in DEPTHS.items():
		for d in depths:
			assert mode == (0 if d % 4 else 3 if d % 128 == 0 else 2 if d % 16 == 0 else 1)
		assert {d % 3 for d in depths} == {1, 2}, mode


@pytest.mark.parametrize("is2024", [True, False], ids=["2024", "686"])
@pytest.mark.parametrize("mode, depth", CASES)
def test_dedup_table_depths_vs_oracle(mode, depth, is2024):
	_scramble(is2024, 4099, depth, seed=depth)


@pytest.mark.parametrize("depth", [100, 101])
def test_dedup_table_more_than_one_pass(depth):
	_scramble(True, 250_001, depth, seed=7)
