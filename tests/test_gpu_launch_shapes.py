"""GPU parity at the launch shapes the small-size suite never reaches: second (and third) grid-stride passes of every capped
launch in rubiks_b200.cu, the write-back store policy and one-hot element offsets past 2^31, multi-position work units of the
sequence / ADI kernels, A* batches wider than one block of k_totals and the full 1024-wide pop, and the kernel variants that
environment knobs select.  Outputs too large for the numpy oracle are compared on the first and last 1024 rows, every row
within 64 of each pass boundary (or element-offset boundary) and a seeded sample of 4096 rows; size-independent properties
(inverse moves, row sums, argmax, f32 == bf16) are checked on the whole output on the device.

The shapes are derived from the launcher formulas below; tests/test_launch_shapes_cpu.py re-derives the formulas from the
sources and fails if a retuned cap or threshold moves a shape off its intended branch."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import cube_oracle as O

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NUM_SMS = 148

# capped launch -> (work items per state, items per block, blocks per SM) of its rb_grid(...) call; the grid covers
# NUM_SMS * blocks_per_sm * per_block / items_per_state states in one pass
GRIDS = {
	"multi_rotate_2024_aligned": (1, 256, 5),
	"multi_rotate_2024_unaligned": (1, 1024, 2),
	"is_solved_2024_aligned": (1, 256, 8),
	"is_solved_2024_unaligned": (1, 1024, 2),
	"multi_rotate_686": (1, 32, 5),
	"is_solved_686": (1, 32, 8),
	"as_correct_686": (48, 256, 8),
	"scramble_2024_strided": (1, 256, 8),
	"scramble_686_strided": (1, 8, 6),
	"render_686": (1, 8 * 32, 8),
	"sequence_states_2024": (1, 256, 24),
	"adi_targets": (1, 256, 8),
	"adi_loss_weights": (1, 256, 8),
}


def pass_states(launch):
	"""States (games for sequence_states, games * depth for the ADI launches) one grid pass covers."""
	per_state, per_block, bps = GRIDS[launch]
	return NUM_SMS * bps * per_block // per_state


def wrap_sizes(launch):
	"""Just past one pass, and about 2.3 passes with a ragged tail."""
	cap = pass_states(launch)
	return [cap + 1, (int(2.3 * cap) + 37) | 1]                  # odd: never a whole number of blocks


WRAP_CASES = [(launch, n) for launch in GRIDS if not launch.startswith("adi_") and launch != "sequence_states_2024"
			  for n in wrap_sizes(launch)]
SEQ_STATES_DEPTH = 2

# sequence_chunk(games, depth, units_per_sm) of the launcher, and the units per SM it is called with
SEQ_UNITS_ONE_HOT, SEQ_UNITS_ADI = 256, 1024


def sequence_chunk(games, depth, units_per_sm):
	target = NUM_SMS * units_per_sm
	per_game = min(max(-(-target // games), 1), depth)
	return -(-depth // per_game)


# (games, depth) -> the chunk the launcher must pick
SEQ_ONE_HOT_SHAPES = {(2000, 30): 2, (5000, 20): 3, (2000, 100): 6, (37888, 33): 33}
ADI_SHAPES = {(8000, 30): 2, (15000, 31): 3}
ADI_UNITS1_SHAPES = {(25, 35): 6, (148, 40): 40, (300, 33): 33}     # under RB_SEQ_UNITS_PER_SM=1
ADI_TARGETS_SHAPE = (10000, 31)

STORE_WB_BYTES = 1 << 31
# one-hot outputs of >= 2 GiB (write-back stores); name -> (rows, row width, element bytes)
BIG_ONE_HOT = {
	"as_oh_2024_f32": (4_600_000, 480, 4),
	"as_oh_686_f32": (2_000_000, 288, 4),
	"expand12_2024_bf16": (12 * 400_000, 480, 2),
	"expand12_2024_f32": (12 * 100_000, 480, 4),
	"adi_generate_2024_f32": (12 * 8000 * 30, 480, 4),
}

GiB = 1 << 30


@pytest.fixture(autouse=True)
def _guard():
	from rl_rubiks_b200 import cube
	cube.set_is2024(True)
	torch.cuda.empty_cache()
	torch.cuda.reset_peak_memory_stats()
	yield
	cube.set_is2024(True)
	peak = torch.cuda.max_memory_allocated()
	print(f"peak device memory {peak / GiB:.2f} GiB")
	assert peak < 20 * GiB


def _cube(is2024):
	from rl_rubiks_b200 import cube
	cube.set_is2024(is2024)
	return cube


def check_rows(n, boundaries=(), seed=0, sample=4096):
	"""First and last 1024 rows, rows within 64 of every boundary, a seeded sample: sorted unique int64 row numbers < n."""
	parts = [np.arange(min(n, 1024)), np.arange(max(0, n - 1024), n)]
	for b in boundaries:
		parts.append(np.arange(max(0, b - 64), min(n, b + 65)))
	parts.append(np.random.RandomState(seed).randint(0, n, sample))
	return np.unique(np.concatenate(parts)).astype(np.int64)


def pass_bounds(launch, n):
	cap = pass_states(launch)
	return list(range(cap, n, cap))


def _dev_rows(t, rows):
	return t.index_select(0, torch.from_numpy(rows).cuda()).cpu().numpy()


def _rand_actions(n, depth, seed):
	g = torch.Generator(device="cuda")
	g.manual_seed(seed)
	return torch.randint(0, 12, (n, depth), dtype=torch.uint8, device="cuda", generator=g)


def _device_states(n, is2024, seed, depth=24):
	cube = _cube(is2024)
	return cube.scramble_batch(_rand_actions(n, depth, seed))


def _oh_rows_equal(oh, rows, states, is2024):
	got = oh.index_select(0, torch.from_numpy(rows).cuda()).float().cpu().numpy()
	return (got == O.as_oh(states, is2024)).all()


def _oh_argmax_ok_2024(oh, states, step=1 << 20):
	"""Every 480-wide row of a 20x24 one-hot (f32 or bf16) has one 1 per cubie, at the cubie's value."""
	for i in range(0, oh.shape[0], step):
		o = oh[i:i + step].view(-1, 20, 24)
		s = states[i:i + step].long()
		if not bool(((o != 0).sum(2) == 1).all()) or not bool((o.amax(2) == 1).all()):
			return False
		if not bool((o.argmax(2) == s).all()):
			return False
	return True


# ---- 1. grid-stride wraps ---------------------------------------------------------------------------------------------
def _wrap_multi_rotate(launch, n):
	from rl_rubiks_b200 import _native as N
	is2024 = "2024" in launch
	cube = _cube(is2024)
	states = _device_states(n, is2024, seed=n)
	g = torch.Generator(device="cuda"); g.manual_seed(n + 1)
	faces = torch.randint(0, 6, (n,), dtype=torch.uint8, device="cuda", generator=g)
	dirs = torch.randint(0, 2, (n,), dtype=torch.uint8, device="cuda", generator=g)
	src = states
	if launch.endswith("unaligned"):                      # a view one byte into an allocation: the tile kernel
		buf = torch.empty(states.numel() + 4, dtype=torch.int8, device="cuda")
		src = buf[1:1 + states.numel()].view(states.shape)
		src.copy_(states)
	out = torch.empty_like(states)
	N.check(N.lib.rb_multi_rotate(cube._rep(), N.ptr(src), N.ptr(faces), N.ptr(dirs), N.ptr(out), n, N.stream_handle()))
	rows = check_rows(n, pass_bounds(launch, n), seed=n)
	want = O.multi_rotate(_dev_rows(states, rows), _dev_rows(faces, rows), _dev_rows(dirs, rows), is2024)
	assert (_dev_rows(out, rows) == want).all()
	# the inverse action (same face, other direction) returns every state to its parent, through the same launch
	back, inv_dirs = torch.empty_like(states), 1 - dirs
	if launch.endswith("unaligned"):
		src.copy_(out)
		N.check(N.lib.rb_multi_rotate(cube._rep(), N.ptr(src), N.ptr(faces), N.ptr(inv_dirs), N.ptr(back), n, N.stream_handle()))
	else:
		N.check(N.lib.rb_multi_rotate(cube._rep(), N.ptr(out), N.ptr(faces), N.ptr(inv_dirs), N.ptr(back), n, N.stream_handle()))
	assert torch.equal(back, states)


def _wrap_is_solved(launch, n):
	from rl_rubiks_b200 import _native as N
	is2024 = "2024" in launch
	cube = _cube(is2024)
	states = _device_states(n, is2024, seed=n, depth=3)
	solved = torch.from_numpy(O.solved(is2024)).cuda()
	states[:: 97] = solved                                # solved states spread over every pass
	states[-1] = solved
	src = states
	if launch.endswith("unaligned"):
		buf = torch.empty(states.numel() + 4, dtype=torch.int8, device="cuda")
		src = buf[1:1 + states.numel()].view(states.shape)
		src.copy_(states)
	flags = torch.empty(n, dtype=torch.uint8, device="cuda")
	N.check(N.lib.rb_multi_is_solved(cube._rep(), N.ptr(src), N.ptr(flags), n, N.stream_handle()))
	want_dev = (states.view(n, -1) == solved.view(1, -1)).all(1)
	assert torch.equal(flags.bool(), want_dev)
	rows = check_rows(n, pass_bounds(launch, n), seed=n)
	assert (_dev_rows(flags, rows).astype(bool) == O.multi_is_solved(_dev_rows(states, rows), is2024)).all()


def _wrap_as_correct(launch, n):
	cube = _cube(False)
	states = _device_states(n, False, seed=n)
	oh = cube.as_oh(states)
	got = cube.as_correct(oh)
	rows = check_rows(n, pass_bounds(launch, n), seed=n)
	assert (_dev_rows(got, rows) == O.as_correct_686(_dev_rows(oh, rows))).all()
	# a solved cube is correct everywhere; the whole output agrees with the solved pattern where the state does
	solved_oh = cube.as_oh(torch.from_numpy(O.solved_686()[None]).cuda())
	assert torch.equal(cube.as_correct(solved_oh.expand(n, -1).contiguous()), cube.as_correct(solved_oh).expand(n, -1, -1))


def _wrap_scramble(launch, n):
	"""The strided kernels (actions in a misaligned move-major view), or the macro-move kernel + render for 6x8x6."""
	from rl_rubiks_b200 import _native as N
	is2024 = "2024" in launch
	cube = _cube(is2024)
	depth = 24
	acts = _rand_actions(n, depth, seed=n)                               # (n, depth) cube-major
	out = torch.empty(n, *cube.shape(), dtype=torch.int8, device="cuda")
	if launch == "render_686":
		N.check(N.lib.rb_scramble(cube._rep(), N.ptr(acts), depth, 1, None, N.ptr(out), n, depth, N.stream_handle()))
	else:
		pad = torch.empty(depth * n + 16, dtype=torch.uint8, device="cuda")
		view = pad[4:4 + depth * n].view(depth, n)                        # 4 bytes in: not 16-byte aligned
		view.copy_(acts.t())
		N.check(N.lib.rb_scramble(cube._rep(), N.ptr(view), 1, n, None, N.ptr(out), n, depth, N.stream_handle()))
	rows = check_rows(n, pass_bounds(launch, n), seed=n)
	f, d = O.indices_to_actions(_dev_rows(acts, rows))
	assert (_dev_rows(out, rows) == O.scramble_many(f, d, is2024)).all()
	# the reversed inverse sequence, applied from the scrambled states through the same launch, solves every cube
	inv = (acts ^ 1).flip(1).contiguous()
	back = torch.empty_like(out)
	if launch == "render_686":
		N.check(N.lib.rb_scramble(cube._rep(), N.ptr(inv), depth, 1, N.ptr(out), N.ptr(back), n, depth, N.stream_handle()))
	else:
		view.copy_(inv.t())
		N.check(N.lib.rb_scramble(cube._rep(), N.ptr(view), 1, n, N.ptr(out), N.ptr(back), n, depth, N.stream_handle()))
	assert bool(cube.multi_is_solved(back).all())
	# with start states: start, then the sequence
	start = _device_states(n, is2024, seed=n + 7, depth=5)
	if launch == "render_686":
		N.check(N.lib.rb_scramble(cube._rep(), N.ptr(acts), depth, 1, N.ptr(start), N.ptr(back), n, depth, N.stream_handle()))
	else:
		view.copy_(acts.t())
		N.check(N.lib.rb_scramble(cube._rep(), N.ptr(view), 1, n, N.ptr(start), N.ptr(back), n, depth, N.stream_handle()))
	want = _dev_rows(start, rows)
	for m in range(depth):
		want = O.multi_rotate(want, f[:, m], d[:, m], is2024)
	assert (_dev_rows(back, rows) == want).all()


_WRAP_FN = {
	"multi_rotate_2024_aligned": _wrap_multi_rotate, "multi_rotate_2024_unaligned": _wrap_multi_rotate, "multi_rotate_686": _wrap_multi_rotate,
	"is_solved_2024_aligned": _wrap_is_solved, "is_solved_2024_unaligned": _wrap_is_solved, "is_solved_686": _wrap_is_solved,
	"as_correct_686": _wrap_as_correct,
	"scramble_2024_strided": _wrap_scramble, "scramble_686_strided": _wrap_scramble, "render_686": _wrap_scramble,
}


@pytest.mark.parametrize("launch,n", [pytest.param(l, n, id=f"{l}-{n}") for l, n in WRAP_CASES])
def test_grid_stride_wrap(launch, n):
	_WRAP_FN[launch](launch, n)


def _seq_states_oracle(faces, dirs, ws, is2024, games=None):
	"""O.sequence_scrambler without the one-hot, for the game columns `games` (all by default): (len(games) * depth, *shape)."""
	if games is not None:
		faces, dirs = faces[:, games], dirs[:, games]
	depth, g = faces.shape
	cur = np.repeat(O.solved(is2024)[None], g, axis=0)
	seq = [cur] if ws else []
	for d in range(depth - int(ws)):
		cur = O.multi_rotate(cur, faces[d], dirs[d], is2024)
		seq.append(cur)
	return np.stack(seq, axis=1).reshape(g * depth, *cur.shape[1:])


@pytest.mark.parametrize("games", [pytest.param(n, id=f"sequence_states_2024-{n}") for n in wrap_sizes("sequence_states_2024")])
def test_grid_stride_wrap_sequence_states(games):
	cube = _cube(True)
	depth = SEQ_STATES_DEPTH
	g = np.random.RandomState(games)
	faces, dirs = g.randint(0, 6, (depth, games)), g.randint(0, 2, (depth, games))
	faces[:, ::501], dirs[:, ::501] = 3, np.array([1, 0])[:, None]         # these games return to solved at position 1
	cols = check_rows(games, pass_bounds("sequence_states_2024", games), seed=games)
	for ws in (False, True):
		states, _, flags = cube.sequence_scrambler_from(faces, dirs, ws, with_oh=False, with_flags=True, device_out=True)
		rows = (cols[:, None] * depth + np.arange(depth)).reshape(-1)
		want = _seq_states_oracle(faces, dirs, ws, True, cols)
		assert (_dev_rows(states, rows) == want).all()
		assert (_dev_rows(flags, rows) == O.multi_is_solved(want, True)).all()
		solved = torch.from_numpy(O.solved_2024()).cuda()
		assert torch.equal(flags, (states == solved).all(1))


# ---- 2. write-back stores, element offsets past 2^31 ------------------------------------------------------------------
def _offset_rows(rows, width, esz):
	"""Rows holding element 2^31 and byte 2^32 (and 2^31 bytes) of a one-hot output, when it has them."""
	out = set()
	for el in ((1 << 31), (1 << 32) // esz, (1 << 31) // esz):
		if el // width < rows:
			out.add(el // width)
	return sorted(out)


@pytest.mark.parametrize("is2024,n", [pytest.param(True, BIG_ONE_HOT["as_oh_2024_f32"][0], id="as_oh_2024_f32"),
									   pytest.param(False, BIG_ONE_HOT["as_oh_686_f32"][0], id="as_oh_686_f32")])
def test_as_oh_write_back_large(is2024, n):
	cube = _cube(is2024)
	states = _device_states(n, is2024, seed=3, depth=20)
	oh = cube.as_oh(states)
	width = cube.get_oh_shape()
	rows = check_rows(n, _offset_rows(n, width, 4), seed=4)
	assert _oh_rows_equal(oh, rows, _dev_rows(states, rows), is2024)
	if is2024:
		assert _oh_argmax_ok_2024(oh, states)
	else:
		for i in range(0, n, 1 << 20):
			assert torch.equal(oh[i:i + (1 << 20)], states[i:i + (1 << 20)].view(-1, 288).float())
	del oh
	# f32 and bf16 rows are the same values
	ob = cube.as_oh(states, dtype=torch.bfloat16)
	sub = torch.from_numpy(rows).cuda()
	assert (ob.index_select(0, sub).float().cpu().numpy() == O.as_oh(_dev_rows(states, rows), is2024)).all()
	if is2024:
		assert _oh_argmax_ok_2024(ob, states)


@pytest.mark.parametrize("dtype,parents", [pytest.param(torch.bfloat16, BIG_ONE_HOT["expand12_2024_bf16"][0] // 12, id="expand12_2024_bf16"),
											pytest.param(torch.float32, BIG_ONE_HOT["expand12_2024_f32"][0] // 12, id="expand12_2024_f32")])
def test_expand12_write_back_large(dtype, parents):
	cube = _cube(True)
	states = _device_states(parents, True, seed=5, depth=20)
	one = torch.from_numpy(O.rotate_2024(O.solved_2024(), 2, 1)).cuda()
	states[::1000] = one                                          # one child of each is solved
	children, oh, flags = cube.expand12(states, with_oh=True, with_solved=True, oh_dtype=dtype)
	n = 12 * parents
	esz = 2 if dtype == torch.bfloat16 else 4
	rows = check_rows(n, _offset_rows(n, 480, esz), seed=6)
	want = O.expand12(_dev_rows(states, np.unique(rows // 12)), True)
	pos = np.searchsorted(np.unique(rows // 12), rows // 12) * 12 + rows % 12
	want = want[pos]
	assert (_dev_rows(children, rows) == want).all()
	assert (oh.index_select(0, torch.from_numpy(rows).cuda()).float().cpu().numpy() == O.as_oh(want, True)).all()
	assert (_dev_rows(flags, rows) == O.multi_is_solved(want, True)).all()
	assert _oh_argmax_ok_2024(oh, children)
	solved = torch.from_numpy(O.solved_2024()).cuda()
	assert torch.equal(flags, (children == solved).all(1)) and int(flags.sum()) >= len(range(0, parents, 1000))
	# child a moved by a ^ 1 is its parent
	inv = torch.arange(12, device="cuda", dtype=torch.uint8).repeat(parents) ^ 1
	back = cube.multi_rotate(children, inv // 2, 1 - inv % 2)
	assert torch.equal(back.view(parents, 12, 20), states[:, None].expand(parents, 12, 20))


# ---- 3. sequence / ADI work units of several positions ----------------------------------------------------------------
@pytest.mark.parametrize("games,depth", [pytest.param(g, d, id=f"chunk{c}-{g}x{d}") for (g, d), c in SEQ_ONE_HOT_SHAPES.items()])
def test_sequence_one_hot_multi_position_chunks(games, depth):
	cube = _cube(True)
	g = np.random.RandomState(games + depth)
	faces, dirs = g.randint(0, 6, (depth, games)), g.randint(0, 2, (depth, games))
	faces[:2, ::17], dirs[:2, ::17] = 3, np.array([1, 0])[:, None]        # back to solved after two moves
	n = games * depth
	for ws in (False, True):
		want = _seq_states_oracle(faces, dirs, ws, True)
		states, oh, flags = cube.sequence_scrambler_from(faces, dirs, ws, with_flags=True, device_out=True)
		assert (states.cpu().numpy() == want).all()
		assert (flags.cpu().numpy() == O.multi_is_solved(want, True)).all()
		rows = check_rows(n, seed=int(ws))
		assert _oh_rows_equal(oh, rows, want[rows], True)
		assert _oh_argmax_ok_2024(oh, states)
		del oh
		_, ob = cube.sequence_scrambler_from(faces, dirs, ws, oh_dtype=torch.bfloat16, device_out=True)
		assert _oh_rows_equal(ob, rows, want[rows], True) and _oh_argmax_ok_2024(ob, states)
		del ob


class _IntNet(torch.nn.Module):
	"""Integer value net: floor((one-hot @ w) / quant), exact in f32 and bf16 for |w| <= 3 (sums of 20 terms)."""

	def __init__(self, w, quant=4.0):
		super().__init__()
		self.w, self.quant = torch.from_numpy(np.asarray(w, dtype=np.float32)).cuda(), quant

	def forward(self, x, policy=True, value=True):
		return torch.floor((x @ self.w.to(x.dtype)).float() / self.quant).unsqueeze(1)


def _int_values_2024(children, w, quant=4.0):
	"""_IntNet on 20x24 states without building the one-hot: oh @ w = sum over cubies of w[24 i + value]."""
	s = (w[np.arange(20) * 24 + children.astype(np.int64)]).sum(1, dtype=np.float32)
	return np.floor(s / np.float32(quant)).astype(np.float32)


def run_adi_case(games, depth, oh_dtype, methods=O.REWARD_METHODS, alphas=(0.0, 0.3), seed=0):
	"""ADIGenerator + adi_traindata with the integer net against the oracle: states, children, flags in full, one-hot rows
	sampled and checked whole on the device, targets and loss weights in full for every method and alpha."""
	from rl_rubiks_b200 import adi
	cube = _cube(True)
	g = np.random.RandomState(seed + games + depth)
	faces, dirs = g.randint(0, 6, (depth, games)), g.randint(0, 2, (depth, games))
	faces[:2, ::13], dirs[:2, ::13] = 3, np.array([1, 0])[:, None]
	w = g.randint(-3, 4, 480).astype(np.float32)
	net = _IntNet(w)
	n = games * depth
	rows = check_rows(n, seed=seed)
	crow = check_rows(12 * n, [], seed=seed + 1)
	for ws in (False, True):
		want = _seq_states_oracle(faces, dirs, ws, True)
		children = O.expand12(want, True)
		ss, sc = O.multi_is_solved(want, True), O.multi_is_solved(children, True)
		gen = adi.ADIGenerator(games, depth, "lapanfix" if ws else "paper", keep_states=True, keep_children=True, oh_dtype=oh_dtype)
		gen.set_actions(faces, dirs)
		oh_s, oh_c = gen.generate()
		assert (gen.states.cpu().numpy() == want).all() and (gen.children.cpu().numpy() == children).all()
		assert (gen.solved_states.cpu().numpy() == ss).all() and (gen.solved_children.cpu().numpy() == sc).all()
		assert _oh_rows_equal(oh_s, rows, want[rows], True) and _oh_rows_equal(oh_c, crow, children[crow], True)
		assert _oh_argmax_ok_2024(oh_s, gen.states) and _oh_argmax_ok_2024(oh_c, gen.children)
		values = _int_values_2024(children, w)
		del gen, oh_s, oh_c
		for method in methods:
			if (method == "lapanfix") != ws:
				continue
			gen = adi.ADIGenerator(games, depth, method, oh_dtype=oh_dtype)
			for alpha in alphas:
				oh, policy, value, lw = adi.adi_traindata(net, games, depth, method, alpha, faces, dirs, ff_batches=4, generator=gen)
				wp, wv = O.adi_targets(values, sc, ss, method, depth)
				assert (policy.cpu().numpy() == wp).all(), (method, alpha)
				assert (value.cpu().numpy() == wv).all(), (method, alpha)
				assert (lw.cpu().numpy() == O.adi_loss_weights(games, depth, alpha)).all(), (method, alpha)
				assert _oh_rows_equal(oh, rows, want[rows], True)
			del gen


@pytest.mark.parametrize("games,depth", [pytest.param(g, d, id=f"chunk{c}-{g}x{d}") for (g, d), c in ADI_SHAPES.items()])
def test_adi_multi_position_chunks(games, depth):
	"""8000 x 30 in f32 (6 GB of one-hot: write-back stores, two positions per unit); 15000 x 31 in bf16 (three positions)."""
	run_adi_case(games, depth, torch.float32 if ADI_SHAPES[(games, depth)] == 2 else torch.bfloat16)


def test_adi_targets_weights_second_pass_ties_nan_inf():
	from rl_rubiks_b200 import _native as N
	games, depth = ADI_TARGETS_SHAPE
	n = games * depth
	g = np.random.RandomState(9)
	values = (np.round(g.randn(12 * n) * 2) / 2).astype(np.float32)           # many exact ties
	values[g.randint(0, 12 * n, 5000)] = np.nan
	values[g.randint(0, 12 * n, 5000)] = np.inf
	values[g.randint(0, 12 * n, 5000)] = -np.inf
	values[12 * (n - 1):] = np.nan                                            # the last state of the last pass
	sc = g.rand(12 * n) < 0.05
	ss = g.rand(n) < 0.05
	v_d = torch.from_numpy(values).cuda()
	sc_d, ss_d = torch.from_numpy(sc.astype(np.uint8)).cuda(), torch.from_numpy(ss.astype(np.uint8)).cuda()
	p = torch.empty(n, dtype=torch.int64, device="cuda")
	v = torch.empty(n, dtype=torch.float32, device="cuda")
	lw = torch.empty(n, dtype=torch.float32, device="cuda")
	ws = float(np.tile(1 / np.arange(1, depth + 1), games).sum())
	for method in O.REWARD_METHODS:
		for alpha in (0.0, 0.3):
			N.check(N.lib.rb_adi_targets_weights(N.ptr(v_d), N.ptr(sc_d), N.ptr(ss_d), games, depth, N.REWARD_METHODS[method], alpha, ws,
												 N.ptr(p), N.ptr(v), N.ptr(lw), N.stream_handle()))
			wp, wv = O.adi_targets(values, sc, ss, method, depth)
			assert (p.cpu().numpy() == wp).all(), method
			assert np.array_equal(v.cpu().numpy(), wv, equal_nan=True), method
			assert (lw.cpu().numpy() == O.adi_loss_weights(games, depth, alpha)).all(), (method, alpha)
			lw2 = torch.empty_like(lw)
			N.check(N.lib.rb_adi_loss_weights(N.ptr(lw2), games, depth, alpha, ws, N.stream_handle()))
			assert torch.equal(lw2, lw)


# ---- 4. wide A* batches -------------------------------------------------------------------------------------------------
class _AStarNet(torch.nn.Module):
	"""floor((one-hot @ w) / quant); values >= hi become +inf and values <= lo -inf (costs -inf / +inf)."""

	def __init__(self, w, quant=4.0, lo=None, hi=None, const=None):
		super().__init__()
		self.w, self.quant, self.lo, self.hi, self.const = torch.from_numpy(np.asarray(w, np.float32)).cuda(), quant, lo, hi, const

	def forward(self, x, policy=True, value=True):
		if self.const is not None:
			return torch.full((x.shape[0], 1), self.const, device=x.device)
		v = torch.floor((x @ self.w) / self.quant)
		if self.hi is not None:
			v = torch.where(v >= self.hi, torch.full_like(v, np.inf), v)
		if self.lo is not None:
			v = torch.where(v <= self.lo, torch.full_like(v, -np.inf), v)
		return v.unsqueeze(1)

	def h(self, states):
		"""Minus the value, on the host (agents.py:380-381)."""
		if self.const is not None:
			return np.full(len(states), -np.float32(self.const), np.float32)
		w = self.w.cpu().numpy()
		v = np.floor((O.as_oh_2024(states) @ w) / np.float32(self.quant)).astype(np.float32)
		if self.hi is not None:
			v[v >= self.hi] = np.inf
		if self.lo is not None:
			v[v <= self.lo] = -np.inf
		return -v


def _oracle_astar(start, lam, n_exp, h, max_states):
	"""AStar.search (agents.py:221-252) on the oracle's bookkeeping (as in test_gpu_frontier.py)."""
	a = O.AStarFrontier(lam, n_exp, h)
	a.reset(start, capacity=max_states + 12 * n_exp + 2)
	if O.is_solved(start, True):
		return True, a
	while len(a) + 12 * n_exp <= max_states:
		won, _ = a.expand_batch(a.pop_batch())
		if won:
			return True, a
	return False, a


def _astar_roots(K, seed, depth=12):
	g = np.random.RandomState(seed)
	roots = O.scramble_many(g.randint(0, 6, (K, depth)), g.randint(0, 2, (K, depth)), True)
	roots[::7] = O.solved_2024()
	for k in range(3, K, 5):
		a = g.randint(0, 12)
		roots[k] = O.rotate_2024(O.solved_2024(), a // 2, 1 - a % 2)
	return roots


def _astar_check(net, lam, n_exp, roots, max_states):
	from rl_rubiks_b200 import cube
	from rl_rubiks_b200.frontier import AStarBatch
	_cube(True)
	agent = AStarBatch(net, lambda_=lam, expansions=n_exp)
	won, queues, count = agent.search_many(roots, max_states)
	L_max = int(count.max()) + 1
	st, G = agent.states[:, :L_max].cpu().numpy(), agent.G[:, :L_max].cpu().numpy()
	par, pact = agent.parents[:, :L_max].cpu().numpy(), agent.parent_actions[:, :L_max].cpu().numpy()
	in_open, cost = agent.in_open[:, :L_max].bool().cpu().numpy(), agent.cost[:, :L_max].cpu().numpy()
	sidx = agent.solved_index.cpu().numpy()
	for s, start in enumerate(roots):
		ok, a = _oracle_astar(start, lam, n_exp, net.h, max_states)
		L = len(a)
		assert bool(won[s]) == ok and count[s] == L, (s, won[s], ok, count[s], L)
		assert (st[s, 1:L + 1] == a.states[1:L + 1]).all(), s
		assert (G[s, 1:L + 1] == a.G[1:L + 1]).all(), s
		assert (par[s, 2:L + 1] == a.parents[2:L + 1]).all(), s
		assert (pact[s, 2:L + 1] == a.parent_actions[2:L + 1]).all(), s
		if not ok:
			mine = sorted((float(cost[s, i]), int(i)) for i in np.where(in_open[s, :L + 1])[0])
			assert mine == sorted((float(c), int(i)) for c, i in a.open), s
		if ok:
			want_idx = int(a.seen.lookup(O.solved_2024()[None])[0])
			assert sidx[s] == want_idx, (s, sidx[s], want_idx)
			i, q = want_idx, []
			while i != 1:
				q.insert(0, int(a.parent_actions[i])); i = int(a.parents[i])
			assert q == queues[s], s
			state = start
			for act in queues[s]:
				state = O.rotate_2024(state, *cube.action_space[act])
			assert O.is_solved(state, True)
		else:
			assert queues[s] == []


@pytest.mark.parametrize("K,n_exp", [pytest.param(1100, 1, id="K1100-N1"), pytest.param(2085, 3, id="K2085-N3")])
def test_astar_totals_several_chunks(K, n_exp):
	"""k_totals sums the new-state counts of 1024 searches per round with a carry: K = 1100 / 2085 gives two / three rounds."""
	g = np.random.RandomState(K)
	_astar_check(_AStarNet(g.randint(-3, 4, 480)), 0.16, n_exp, _astar_roots(K, K), 150)


def test_astar_full_width_pop():
	"""N = 1024: the pop threshold is the last slot of the 1024-entry best list."""
	g = np.random.RandomState(1024)
	roots = np.stack([O.scramble(g.randint(0, 6, 40), g.randint(0, 2, 40), True) for _ in range(3)])
	_astar_check(_AStarNet(g.randint(-3, 4, 480)), 0.16, 1024, roots, 40000)


@pytest.mark.parametrize("case", ["constant-lambda0", "inf-values"])
def test_astar_cost_ties_and_infinities(case):
	"""lambda = 0 with a constant net: every open entry has the same cost and pops go by index alone; a net with +-inf values
	gives -inf / +inf costs that tie among themselves."""
	g = np.random.RandomState(11)
	if case == "constant-lambda0":
		net, lam = _AStarNet(np.zeros(480), const=3.0), 0.0
	else:
		net, lam = _AStarNet(g.randint(-3, 4, 480), lo=-2, hi=2), 0.16
	roots = _astar_roots(1100, 12, depth=10)
	_astar_check(net, lam, 3, roots, 150)
	_astar_check(net, lam, 1024, roots[:3], 13000)


# ---- 5. kernel variants selected by environment variables (read once per process: run in a child) --------------------
def _child_store_policy():
	from rl_rubiks_b200 import adi
	for is2024 in (True, False):
		cube = _cube(is2024)
		n = 4099
		g = np.random.RandomState(1)
		states = O.scramble_many(g.randint(0, 6, (n, 6)), g.randint(0, 2, (n, 6)), is2024)
		want_ch = O.expand12(states, is2024)
		for dt in (torch.float32, torch.bfloat16):
			assert (cube.as_oh(states, dtype=dt).float().cpu().numpy() == O.as_oh(states, is2024)).all()
			ch, oh, fl = cube.expand12(states, with_oh=True, with_solved=True, oh_dtype=dt)
			assert (ch == want_ch).all() and (oh.float().cpu().numpy() == O.as_oh(want_ch, is2024)).all()
			assert (fl == O.multi_is_solved(want_ch, is2024)).all()
			g = np.random.RandomState(2)
			for games, depth in ((300, 25), (7, 33)):
				faces, dirs = g.randint(0, 6, (depth, games)), g.randint(0, 2, (depth, games))
				for ws in (False, True):
					want_s, want_oh = O.sequence_scrambler(faces, dirs, ws, is2024)
					s, oh = cube.sequence_scrambler_from(faces, dirs, ws, oh_dtype=dt)
					assert (s == want_s).all() and (oh.float().cpu().numpy() == want_oh).all()
					gen = adi.ADIGenerator(games, depth, "lapanfix" if ws else "paper", keep_states=True, keep_children=True, oh_dtype=dt)
					gen.set_actions(faces, dirs)
					oh_s, oh_c = gen.generate()
					wc = O.expand12(want_s, is2024)
					assert (oh_s.float().cpu().numpy() == want_oh).all() and (gen.children.cpu().numpy() == wc).all()
					assert (oh_c.float().cpu().numpy() == O.as_oh(wc, is2024)).all()
					assert (gen.solved_children.cpu().numpy() == O.multi_is_solved(wc, is2024)).all()
	cube.set_is2024(True)


def _child_seq_units():
	for (games, depth), chunk in ADI_UNITS1_SHAPES.items():
		assert sequence_chunk(games, depth, 1) == chunk
		run_adi_case(games, depth, torch.float32, seed=chunk)


ENV_CASES = {
	"RB_STORE_POLICY=0": ({"RB_STORE_POLICY": "0"}, _child_store_policy),
	"RB_STORE_POLICY=1": ({"RB_STORE_POLICY": "1"}, _child_store_policy),
	"RB_SEQ_UNITS_PER_SM=1": ({"RB_SEQ_UNITS_PER_SM": "1"}, _child_seq_units),
}


def _child(name):
	"""Entry point of the child process: runs the checks of one ENV_CASES entry, exits non-zero on a mismatch."""
	env, fn = ENV_CASES[name]
	for k, v in env.items():
		assert os.environ.get(k) == v, f"{k} is not set in the child"
	torch.cuda.set_device(0)
	fn()
	torch.cuda.synchronize()
	print(f"{name}: ok")


@pytest.mark.parametrize("name", list(ENV_CASES))
def test_env_selected_variants(name):
	env = dict(os.environ, **ENV_CASES[name][0])
	code = f"import sys; sys.path.insert(0, {ROOT!r}); from tests.test_gpu_launch_shapes import _child; _child({name!r})"
	r = subprocess.run([sys.executable, "-c", code], env=env, cwd=ROOT, timeout=900, capture_output=True, text=True)
	assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
	assert f"{name}: ok" in r.stdout
