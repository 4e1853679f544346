"""The shapes of tests/test_gpu_launch_shapes.py against the launcher formulas as they stand in the sources: grid caps
(rb_grid arguments and RB_NUM_SMS), the units per SM of sequence_chunk, the 2 GiB store-policy threshold and the 1024-wide
A* rounds.  If a cap is retuned, this fails on the CPU instead of the GPU tests quietly going back to a single pass."""
import os
import re

import pytest

from tests import test_gpu_launch_shapes as S

CSRC = os.path.join(S.ROOT, "rl_rubiks_b200", "csrc")
NAMESPACES = {"rb_cube2024.cuh": "rb2024", "rb_cube686.cuh": "rb686", "rb_adi.cuh": "rbadi", "rb_astar.cuh": "rba"}

# launch in GRIDS -> the kernel launch in rubiks_b200.cu it names (first occurrence)
LAUNCHES = {
	"multi_rotate_2024_aligned": "rb2024::k_multi_rotate<<<",
	"multi_rotate_2024_unaligned": "rb2024::k_multi_rotate_any<<<",
	"is_solved_2024_aligned": "rb2024::k_is_solved<<<",
	"is_solved_2024_unaligned": "rb2024::k_is_solved_any<<<",
	"multi_rotate_686": "rb686::k_multi_rotate<<<",
	"is_solved_686": "rb686::k_is_solved<<<",
	"as_correct_686": "rb686::k_as_correct<<<",
	"scramble_2024_strided": "rb2024::k_scramble<<<",
	"scramble_686_strided": "rb686::k_scramble<<<",
	"render_686": "rb686::k_render_from2024<<<",
	"sequence_states_2024": "rb2024::k_sequence_states<<<",
	"adi_targets": "rbadi::k_targets<<<",
	"adi_loss_weights": "rbadi::k_loss_weights<<<",
}


def _read(name):
	with open(os.path.join(CSRC, name)) as f:
		return re.sub(r"//[^\n]*", "", f.read())


def _c_eval(expr, env):
	expr = re.sub(r"\b(\w+)::(k\w+)\b", lambda m: str(env[m.group(1)][m.group(2)]), expr)
	return eval(expr.replace("/", "//"), {}, {})


def _constants():
	env = {}
	for fname, ns in NAMESPACES.items():
		env[ns] = {}
		for name, expr in re.findall(r"constexpr int (k\w+) = ([^;]+);", _read(fname)):
			try:
				env[ns][name] = eval(re.sub(r"\b(k\w+)\b", lambda m: str(env[ns][m.group(1)]), expr).replace("/", "//"), {}, {})
			except (KeyError, SyntaxError, NameError):
				pass
	return env


def _args(call):
	"""Top-level comma-separated arguments of the first parenthesised call in `call`."""
	depth, cur, out = 0, "", []
	for ch in call[call.index("(") + 1:]:
		if ch == "(":
			depth += 1
		elif ch == ")":
			if depth == 0:
				out.append(cur.strip())
				return out
			depth -= 1
		elif ch == "," and depth == 0:
			out.append(cur.strip()); cur = ""
			continue
		cur += ch
	raise AssertionError(call)


@pytest.fixture(scope="module")
def src():
	return _read("rubiks_b200.cu")


def test_num_sms_matches():
	m = re.search(r"#define RB_NUM_SMS (\d+)", _read("rb_common.cuh"))
	assert int(m.group(1)) == S.NUM_SMS


@pytest.mark.parametrize("launch", list(LAUNCHES))
def test_grid_caps_put_shapes_past_one_pass(src, launch):
	env = _constants()
	i = src.index(LAUNCHES[launch])
	work, per_block, bps = _args(src[i:src.index("\n", i)])
	per_block, bps = _c_eval(per_block, env), _c_eval(bps, env)
	var = "games" if "games" in work else "n"
	items = lambda n: _c_eval(re.sub(rf"\b{var}\b", str(n), work), env)
	cap_items = S.NUM_SMS * bps * per_block
	lo, hi = 1, 1 << 40                                            # largest state count one grid pass covers
	while lo < hi:
		mid = (lo + hi + 1) // 2
		lo, hi = (mid, hi) if items(mid) <= cap_items else (lo, mid - 1)
	assert S.pass_states(launch) in (lo, lo + 1) and items(S.pass_states(launch) + 1) > cap_items, launch
	if launch.startswith("adi_"):
		games, depth = S.ADI_TARGETS_SHAPE
		assert items(games * depth) > cap_items
		return
	sizes = S.wrap_sizes(launch)
	assert items(sizes[0]) > cap_items and sizes[0] <= lo + 1            # one item (or one block) into the second pass
	assert items(sizes[1]) > 2 * cap_items and items(sizes[1]) % per_block != 0                 # third pass, ragged last block


def test_sequence_chunk_units_and_shapes(src):
	body = src[src.index("static int sequence_units_per_sm"):]
	body = body[:body.index("\n}\n")]
	adi = int(re.search(r'atoi\(e\) : (\d+)', body).group(1))
	one_hot = int(re.search(r"with_oh \? (\d+) : (\d+)", body).group(1))
	assert (one_hot, adi) == (S.SEQ_UNITS_ONE_HOT, S.SEQ_UNITS_ADI)
	chunk_src = src[src.index("static int sequence_chunk"):]
	assert "(int64_t)RB_NUM_SMS * units_per_sm" in chunk_src[:chunk_src.index("\n}\n")]
	for (games, depth), chunk in S.SEQ_ONE_HOT_SHAPES.items():
		assert S.sequence_chunk(games, depth, one_hot) == chunk
	for (games, depth), chunk in S.ADI_SHAPES.items():
		assert S.sequence_chunk(games, depth, adi) == chunk
	for (games, depth), chunk in S.ADI_UNITS1_SHAPES.items():
		assert S.sequence_chunk(games, depth, 1) == chunk
	chunks = set(S.SEQ_ONE_HOT_SHAPES.values()) | set(S.ADI_SHAPES.values()) | set(S.ADI_UNITS1_SHAPES.values())
	assert {2, 3, 6} <= chunks and max(chunks) > 32
	assert any(d % c for (g, d), c in S.SEQ_ONE_HOT_SHAPES.items()) and any(d % c for (g, d), c in S.ADI_UNITS1_SHAPES.items())
	# the ADI shape of the write-back case is also a multi-position one
	assert (8000, 30) in S.ADI_SHAPES


def test_store_policy_threshold_and_big_outputs():
	m = re.search(r"out_bytes >= \(int64_t\(1\) << (\d+)\) \? RB_STORE_WB : RB_STORE_CS", _read("rb_common.cuh"))
	assert m and (1 << int(m.group(1))) == S.STORE_WB_BYTES
	for name, (rows, width, esz) in S.BIG_ONE_HOT.items():
		assert rows * width * esz >= S.STORE_WB_BYTES, name
	for name in ("as_oh_2024_f32", "expand12_2024_bf16"):
		rows, width, _ = S.BIG_ONE_HOT[name]
		assert rows * width > 1 << 31, name                       # element offsets past int32
	games, depth = next(k for k, c in S.ADI_SHAPES.items() if c == 2)
	assert 12 * games * depth == S.BIG_ONE_HOT["adi_generate_2024_f32"][0]


def test_astar_rounds_in_search_core():
	"""k_totals lives in the lockstep expansion core both batched searches share (rb_search.cuh)."""
	src = _read("rb_astar.cuh")
	body = _read("rb_search.cuh")
	body = body[body.index("k_totals("):]
	step = int(re.search(r"for \(int base = 0; base < v\.K; base \+= (\d+)\)", body).group(1))
	assert step == 1024
	assert [-(-k // step) for k in (1100, 2085)] == [2, 3]
	assert re.search(r"a->N <= 1024", _read("rubiks_b200.cu")) and re.search(r"constexpr int kSelThreads = 1024;", src)
