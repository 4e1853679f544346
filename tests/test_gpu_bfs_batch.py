"""GPU parity tests of the batched BFS (frontier.BFSBatch, csrc/rb_bfs.cuh): K breadth-first searches in lockstep must each
give BFS.search's found flag, len(agent) and action queue (agents.py:96-123) -- against the reference's recordings, the
literal oracle, the single-search BFS mirror through the evaluator, and themselves at other batch shapes."""
import numpy as np
import pytest

from oracle import cube_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _repr_guard():
	from rl_rubiks_b200 import cube
	cube.set_is2024(True)
	yield
	cube.set_is2024(True)


def _agent(step=None, is2024=True):
	from rl_rubiks_b200.frontier import BFSBatch
	agent = BFSBatch(is2024=is2024)
	if step is not None:
		agent._step = step
	return agent


def _golden_groups(g, is2024):
	"""Recorded cases of one representation grouped by budget: {max_states: [case, ...]}."""
	groups = {}
	for c in range(int(g["n_cases"])):
		if (g[f"start_{c}"].shape == (20,)) == is2024:
			groups.setdefault(int(g[f"max_{c}"]), []).append(c)
	return groups


def _check(g, cases, won, queues, lens, tag):
	for k, c in enumerate(cases):
		assert bool(won[k]) == bool(g[f"found_{c}"]), (tag, c)
		assert int(lens[k]) == int(g[f"len_{c}"]), (tag, c, int(lens[k]), int(g[f"len_{c}"]))
		assert queues[k] == g[f"queue_{c}"].tolist(), (tag, c)


@pytest.mark.parametrize("step", [1, 7, None], ids=["N1", "N7", "default"])
def test_golden_budgets_2024(golden, step):
	"""The 144 20x24 searches recorded from the reference under binding budgets: one search_many of K = 12 per budget."""
	g = golden("bfs_budget")
	groups = _golden_groups(g, True)
	assert sum(len(c) for c in groups.values()) == 144 and all(len(c) == 12 for c in groups.values())
	agent = _agent(step)
	for max_states, cases in groups.items():
		won, queues, lens = agent.search_many(np.stack([g[f"start_{c}"] for c in cases]), max_states)
		_check(g, cases, won, queues, lens, (step, max_states))


@pytest.mark.parametrize("step", [1, 7, None], ids=["N1", "N7", "default"])
def test_golden_budgets_686(golden, step):
	"""The 8 6x8x6 recordings, searched from 6x8x6 roots."""
	from rl_rubiks_b200 import cube
	g = golden("bfs_budget")
	groups = _golden_groups(g, False)
	assert sum(len(c) for c in groups.values()) == 8
	cube.set_is2024(False)
	agent = _agent(step, is2024=None)
	assert not agent.is2024
	for max_states, cases in groups.items():
		won, queues, lens = agent.search_many(np.stack([g[f"start_{c}"] for c in cases]), max_states)
		_check(g, cases, won, queues, lens, (step, max_states))


def test_unreachable_686_root_is_an_index_error():
	agent = _agent(is2024=False)
	bad = np.zeros_like(O.solved(False))                               # no sticker shows any colour
	with pytest.raises(IndexError):
		agent.search_many(bad[None], 10)


def test_one_cube_search_matches_reference(golden):
	"""BFS.search's interface on one cube: search.npz's recording, and a solved start (found, len 0)."""
	from rl_rubiks_b200 import cube
	g = golden("search")
	agent = _agent()
	assert agent.search(g["bfs_start"], None, 10 ** 6) == bool(g["bfs_found"])
	assert len(agent) == int(g["bfs_len"])
	assert list(agent.action_queue) == g["bfs_queue"].tolist()
	s = g["bfs_start"]
	for a in agent.action_queue:
		s = cube.rotate(s, *cube.action_space[a])
	assert cube.is_solved(s)
	assert agent.search(cube.get_solved(), None, 10) is True
	assert len(agent) == 0 and list(agent.action_queue) == []
	assert agent.search(g["bfs_start"], 60.0, None) == bool(g["bfs_found"]) and len(agent) == int(g["bfs_len"])


@pytest.mark.parametrize("max_states", [700, 4000])
def test_evaluator_parity_fixed_depths(max_states):
	"""eval_batched(BFSBatch()) and eval(BFS()) draw the same cubes and give the same turns and states; 700 ends the deeper
	searches in the middle of a layer."""
	from rl_rubiks_b200.evaluation import Evaluator
	from rl_rubiks_b200.frontier import BFS
	ev = Evaluator(6, range(1, 6), max_states=max_states)
	np.random.seed(11)
	res, states, _ = ev.eval(BFS())
	np.random.seed(11)
	res_b, states_b, _ = ev.eval_batched(_agent())
	assert (res_b == res).all() and (states_b == states).all()
	assert (res[0] == 1).all()
	if max_states == 700:
		assert (res == -1).any() and (states[res == -1] >= 700).all()


def test_evaluator_parity_deep_mode():
	from rl_rubiks_b200.evaluation import Evaluator
	from rl_rubiks_b200.frontier import BFS
	ev = Evaluator(5, range(0), max_states=300)
	np.random.seed(3)
	res, states, _ = ev.eval(BFS())
	np.random.seed(3)
	res_b, states_b, _ = ev.eval_batched(_agent())
	assert (res == -1).all() and (res_b == -1).all()
	assert (states_b == states).all()


def test_oracle_at_random():
	"""Random scrambles of depth 2-6; budgets that end inside a layer, on a parent boundary (a parent's last new child is the
	budget's state) and with the solved child's step just inside or outside the cut; N = 7 and the default."""
	rng = np.random.RandomState(21)
	starts = [O.scramble(rng.randint(0, 6, d), rng.randint(0, 2, d), True) for d in (2, 3, 3, 4, 4, 5, 5, 6)]
	budgets = {1, 12, 13, 50, 127, 128, 600, 1196, 2500}
	for s in starts:
		found, length, _ = O.bfs_search(s, 2500)
		if found:
			budgets |= {max(1, length - 1), length, length + 1}
	want = {m: [O.bfs_search(s, m) for s in starts] for m in sorted(budgets)}
	for step in (7, None):
		agent = _agent(step)
		for m, w in want.items():
			won, queues, lens = agent.search_many(np.stack(starts), m)
			for k in range(len(starts)):
				assert (bool(won[k]), int(lens[k]), queues[k]) == w[k], (step, m, k)


def test_isolation_at_k1100(golden):
	"""K = 1100 searches in one table: golden starts repeated, interleaved with solved starts and duplicate roots (k_totals
	walks the searches in chunks of 1024).  Every search gives its own single-search answer."""
	g = golden("bfs_budget")
	max_states = 1000
	cases = _golden_groups(g, True)[max_states]
	solved = O.solved(True)
	starts, want = [], []
	for k in range(1100):
		if k % 5 == 4:
			starts.append(solved); want.append((True, 0, []))
		else:
			c = cases[(k * 7) % len(cases)]
			starts.append(g[f"start_{c}"]); want.append((bool(g[f"found_{c}"]), int(g[f"len_{c}"]), g[f"queue_{c}"].tolist()))
	agent = _agent()
	won, queues, lens = agent.search_many(np.stack(starts), max_states)
	for k in range(1100):
		assert (bool(won[k]), int(lens[k]), queues[k]) == want[k], k


def test_determinism_and_reuse(golden):
	"""Two runs are bit-identical; a search_many after a different one of the same shape (reused buffers and table) answers
	as a fresh agent does."""
	g = golden("bfs_budget")
	groups = _golden_groups(g, True)
	a, b = np.stack([g[f"start_{c}"] for c in groups[2000]]), np.stack([g[f"start_{c}"] for c in groups[5000]])
	agent = _agent()
	r1 = agent.search_many(a, 5000)
	r2 = agent.search_many(a, 5000)
	assert (r1[0] == r2[0]).all() and r1[1] == r2[1] and (r1[2] == r2[2]).all()
	assert (agent.count.cpu().numpy() == r1[2]).all()
	agent.search_many(b, 5000)
	r3 = agent.search_many(a, 5000)
	fresh = _agent().search_many(a, 5000)
	assert (r3[0] == fresh[0]).all() and r3[1] == fresh[1] and (r3[2] == fresh[2]).all()
	assert (fresh[0] == r1[0]).all() and fresh[1] == r1[1] and (fresh[2] == r1[2]).all()
