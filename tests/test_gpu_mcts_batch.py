"""GPU parity tests of the batched MCTS (frontier.MCTSBatch, csrc/rb_mcts.cuh): K Monte Carlo tree searches in lockstep must
each equal MCTS.search (agents.py:461-633) node for node -- against the reference's recorded traces, the numpy oracle, the
statement-by-statement harness (tests/agent_harness.py::MCTS) and the sequential evaluator.

Every net here is batch-invariant (the batched agent runs the net on all searches' new states at once, the harness on at most
12 rows): one-hot rows times small-integer weights are exact in any summation order, and the policies go through torch's
softmax on both sides."""
import numpy as np
import pytest
import torch

from oracle import cube_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _repr_guard():
	from rl_rubiks_b200 import cube
	cube.set_is2024(True)
	yield
	cube.set_is2024(True)


class _CountNet(torch.nn.Module):
	"""The golden MCTS runs' net: uniform policy logits, value = number of cubies in their solved place."""

	def __init__(self, is2024=True):
		super().__init__()
		w = O.as_oh_2024(O.solved_2024()[None])[0] if is2024 else O.as_oh_686(O.solved_686()[None])[0]
		self.w = torch.from_numpy(w).cuda()

	def forward(self, x, policy=True, value=True):
		return torch.zeros(x.shape[0], 12, device=x.device), torch.floor(x @ self.w).unsqueeze(1)


def _count_net_np(oh):
	w = O.as_oh_2024(O.solved_2024()[None])[0]
	return np.zeros((len(oh), 12), np.float32), np.floor(oh @ w)


class _IntNet(torch.nn.Module):
	"""Integer policy logits (a non-uniform softmax) and integer values from small-integer weights."""

	def __init__(self, width=480, seed=0):
		super().__init__()
		g = np.random.RandomState(seed)
		self.wp = torch.from_numpy(g.randint(-3, 4, (width, 12)).astype(np.float32)).cuda()
		self.wv = torch.from_numpy(g.randint(-2, 3, width).astype(np.float32)).cuda()

	def forward(self, x, policy=True, value=True):
		return torch.floor((x @ self.wp) / 2.0), torch.floor((x @ self.wv) / 2.0).unsqueeze(1)


class _PoisonNet(_CountNet):
	"""_CountNet with NaN, +inf and -inf values and all-NaN policy rows for a few states (an integer hash of the one-hot picks
	them).  NaN and +inf scores ignore the virtual loss, so such a net can walk in circles forever: the starts below were chosen
	so that the reference's walks end."""

	def __init__(self):
		super().__init__()
		self.wh = torch.from_numpy(np.random.RandomState(7).randint(-3, 4, 480).astype(np.float32)).cuda()

	def forward(self, x, policy=True, value=True):
		p, v = super().forward(x)
		h = torch.remainder(x @ self.wh + 1000, 61).unsqueeze(1)
		v = torch.where(h == 1, float("nan"), torch.where(h == 2, float("inf"), torch.where(h == 3, float("-inf"), v)))
		return torch.where(h == 4, float("nan"), p), v


def _agent(net, c, graph, **kw):
	from rl_rubiks_b200.frontier import MCTSBatch
	return MCTSBatch(net, c=c, search_graph=graph, **kw)


def _scrambles(seed, depths):
	rng = np.random.RandomState(seed)
	return [O.scramble(rng.randint(0, 6, d), rng.randint(0, 2, d), True) for d in depths]


class _Host:
	"""The batched agent's node arrays on the host, one copy per search_many."""

	def __init__(self, agent):
		self.a = agent
		for name in ("states", "neighbors", "leaves", "N", "W", "V", "P", "L", "count", "path_len", "path_node", "path_action", "won"):
			setattr(self, name, getattr(agent, name).cpu().numpy())


def _same(x, y):
	return np.array_equal(np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64), equal_nan=True)


def _check_L_invariant(h, k):
	"""L is zero outside the running walk: nothing for a won search, exactly the last walk's virtual loss otherwise (each move
	raises its pair and the reverse pair by one nu)."""
	n = int(h.count[k])
	L = h.L[k, :n + 1]
	if h.won[k]:
		assert not L.any(), k
		return
	ln = int(h.path_len[k])
	assert int(L.sum()) == 2 * ln, k
	walk = set()
	for node, a in zip(h.path_node[k, :ln], h.path_action[k, :ln]):
		walk |= {(int(node), int(a)), (int(h.neighbors[k, node, a]), int(a) ^ 1)}
	assert {(int(x), int(a)) for x, a in zip(*np.nonzero(L))} <= walk, k


def _check_vs_harness(h, k, m, ok, is2024=True, queue=None):
	"""Search k of the batched run against a finished harness (or oracle) search: found, len, queue and every node array."""
	L = len(m)
	assert bool(h.won[k]) == bool(ok), k
	assert int(h.count[k]) == L, (k, int(h.count[k]), L)
	assert queue == list(m.action_queue), (k, queue, list(m.action_queue))
	states = m.states[1:L + 1]
	if isinstance(states, torch.Tensor):
		from rl_rubiks_b200 import cube
		states = (states if is2024 else cube.to_2024(states)).cpu().numpy()
	assert (h.states[k, 1:L + 1] == states).all(), k
	assert (h.neighbors[k, :L + 1] == m.neighbors[:L + 1]).all(), k
	assert (h.leaves[k, :L + 1].astype(bool) == m.leaves[:L + 1]).all(), k
	assert (h.N[k, :L + 1] == m.N[:L + 1]).all(), k
	assert _same(h.W[k, 1:L + 1], m.W[1:L + 1]), k
	assert _same(h.L[k, :L + 1] * 100.0, m.L[:L + 1]), k
	if not (ok and L == 1):                      # a solved start stores no P / V
		assert _same(h.V[k, 1:L + 1], m.V[1:L + 1]), k
		assert _same(h.P[k, 1:L + 1], m.P[1:L + 1]), k
	_check_L_invariant(h, k)


def _solves(start, queue):
	s = np.asarray(start)
	for a in queue:
		s = O.expand12(s[None], True)[a]
	return O.is_solved(s, True)


def _harness(net, c, graph, start, max_states, is2024=None):
	from tests.agent_harness import MCTS
	m = MCTS(net, c=c, search_graph=graph, is2024=is2024)
	ok = m.search(start, None, max_states)
	return m, ok


GOLDEN = [("a", 5.0, True, 3000), ("b", 0.6, False, 400)]


def _check_golden(g, tag, h, k, queue):
	L = int(g[f"mcts{tag}_len"])
	assert bool(h.won[k]) == bool(g[f"mcts{tag}_ok"]) and int(h.count[k]) == L
	assert queue == g[f"mcts{tag}_queue"].tolist()
	assert (h.states[k, 1:L + 1] == g[f"mcts{tag}_states"]).all()
	assert (h.neighbors[k, :L + 1] == g[f"mcts{tag}_neighbors"]).all()
	assert (h.leaves[k, :L + 1].astype(bool) == g[f"mcts{tag}_leaves"]).all()
	assert (h.N[k, :L + 1] == g[f"mcts{tag}_N"]).all()
	assert (h.W[k, 1:L + 1] == g[f"mcts{tag}_W"]).all() and (h.V[k, 1:L + 1] == g[f"mcts{tag}_V"]).all()
	_check_L_invariant(h, k)
	if bool(g[f"mcts{tag}_ok"]):
		assert _solves(g[f"mcts{tag}_start"], queue)


@pytest.mark.parametrize("tag,c,graph,max_states", GOLDEN)
def test_golden_trace_alone(golden, tag, c, graph, max_states):
	"""The two traces recorded from the reference, K = 1: node arrays, len and queue."""
	g = golden("search")
	agent = _agent(_CountNet(), c, graph)
	won, queues, count = agent.search_many(g[f"mcts{tag}_start"][None], max_states)
	_check_golden(g, tag, _Host(agent), 0, queues[0])


@pytest.mark.parametrize("tag,c,graph,max_states", GOLDEN)
def test_golden_trace_in_batch(golden, tag, c, graph, max_states):
	"""The recorded trace as search 17 of 40, among random starts (checked against the oracle)."""
	g = golden("search")
	starts = _scrambles(3, [1 + k % 8 for k in range(40)])
	starts[17] = g[f"mcts{tag}_start"]
	agent = _agent(_CountNet(), c, graph)
	won, queues, count = agent.search_many(np.stack(starts), max_states)
	h = _Host(agent)
	_check_golden(g, tag, h, 17, queues[17])
	for k in range(0, 40, 3):
		m = O.MCTSOracle(_count_net_np, c, graph)
		ok = m.search(starts[k], max_states)
		_check_vs_harness(h, k, m, ok, queue=queues[k])


@pytest.mark.parametrize("c,graph,max_states", [(0.6, False, 300), (5.0, True, 600), (1.5, True, 150)])
def test_oracle_k1100(c, graph, max_states):
	"""K = 1100 (more than one 1024-search round of k_totals), depths 1-8: every search equals the oracle node for node; the
	budget ends some searches before their solve and lets others solve."""
	starts = _scrambles(int(c * 10) + max_states, [1 + k % 8 for k in range(1100)])
	agent = _agent(_CountNet(), c, graph)
	won, queues, count = agent.search_many(np.stack(starts), max_states)
	h = _Host(agent)
	assert won.any() and not won.all()
	for k in range(1100):
		m = O.MCTSOracle(_count_net_np, c, graph)
		ok = m.search(starts[k], max_states)
		_check_vs_harness(h, k, m, ok, queue=queues[k])
		if ok:
			assert _solves(starts[k], queues[k])


@pytest.mark.parametrize("graph", [False, True], ids=["tree", "graph"])
def test_policy_net_vs_harness(graph):
	"""32 starts, an integer-weight net whose policy is not uniform."""
	net = _IntNet(seed=2)
	starts = _scrambles(8, [2 + k % 7 for k in range(32)])
	c = 0.9 if graph else 2.5
	agent = _agent(net, c, graph)
	won, queues, count = agent.search_many(np.stack(starts), 400)
	h = _Host(agent)
	assert np.unique(h.P[0, 1]).size > 1
	for k in range(32):
		m, ok = _harness(net, c, graph, starts[k], 400)
		_check_vs_harness(h, k, m, ok, queue=queues[k])


POISON_STARTS = [5, 21, 24, 44, 59, 87, 108, 127, 134, 143]


@pytest.mark.parametrize("graph", [False, True], ids=["tree", "graph"])
def test_nan_inf_net_vs_harness(graph):
	"""NaN and +-inf values and NaN policies: numpy's argmax (the first NaN wins) and np.maximum (NaN propagates)."""
	rng = np.random.RandomState(31)
	pool = []
	for t in range(144):
		d = 3 + t % 5
		pool.append(O.scramble(rng.randint(0, 6, d), rng.randint(0, 2, d), True))
	starts = [pool[t] for t in POISON_STARTS]
	c = 3.0 if graph else 0.6
	net = _PoisonNet()
	agent = _agent(net, c, graph)
	won, queues, count = agent.search_many(np.stack(starts), 300)
	h = _Host(agent)
	n_nan = n_inf = 0
	for k in range(len(starts)):
		m, ok = _harness(net, c, graph, starts[k], 300)
		_check_vs_harness(h, k, m, ok, queue=queues[k])
		n_nan += int(np.isnan(m.V[1:len(m) + 1]).sum() + np.isnan(m.P[1:len(m) + 1]).sum())
		n_inf += int(np.isinf(m.V[1:len(m) + 1]).sum())
	assert n_nan and n_inf


@pytest.mark.parametrize("graph", [False, True], ids=["tree", "graph"])
def test_686_vs_harness(graph):
	"""6x8x6 roots and a 288-wide net, against the harness on the 6x8x6 representation."""
	from rl_rubiks_b200 import cube
	cube.set_is2024(False)
	net = _IntNet(width=288, seed=4)
	rng = np.random.RandomState(40)
	starts = [O.scramble(rng.randint(0, 6, d), rng.randint(0, 2, d), False) for d in range(2, 10)]
	agent = _agent(net, 1.2, graph)
	assert not agent.is2024
	won, queues, count = agent.search_many(np.stack(starts), 300)
	h = _Host(agent)
	for k in range(len(starts)):
		m, ok = _harness(net, 1.2, graph, starts[k], 300)
		_check_vs_harness(h, k, m, ok, is2024=False, queue=queues[k])


def test_solved_duplicate_roots_and_small_budgets(golden):
	"""Solved starts (found, len 1, empty queue), duplicate roots (same answers, separate searches), and budgets below 13 that
	allow no expansion (not found, len 1, empty queue)."""
	g = golden("search")
	a = g["mctsb_start"]
	solved = O.solved(True)
	starts = np.stack([a, solved, a, solved, a])
	agent = _agent(_CountNet(), 0.6, False)
	won, queues, count = agent.search_many(starts, 400)
	want = (bool(g["mctsb_ok"]), g["mctsb_queue"].tolist(), int(g["mctsb_len"]))
	for k in (0, 2, 4):
		assert (bool(won[k]), queues[k], int(count[k])) == want
	for k in (1, 3):
		assert (bool(won[k]), queues[k], int(count[k])) == (True, [], 1)
	h = _Host(agent)
	for k in (0, 2, 4):
		_check_golden(g, "b", h, k, queues[k])
	for graph in (False, True):
		agent = _agent(_CountNet(), 0.6, graph)
		for max_states in (1, 12):
			won, queues, count = agent.search_many(starts, max_states)
			h = _Host(agent)
			for k in range(5):
				m, ok = _harness(_CountNet(), 0.6, graph, starts[k], max_states)
				_check_vs_harness(h, k, m, ok, queue=queues[k])
			assert list(won) == [False, True, False, True, False] and list(count) == [1] * 5 and queues == [[]] * 5


def test_one_cube_search(golden):
	"""MCTS.search's interface on one cube: the graph trace, and a solved start (found, len 1)."""
	g = golden("search")
	agent = _agent(_CountNet(), 5.0, True)
	assert agent.search(g["mctsa_start"], None, 3000) == bool(g["mctsa_ok"])
	assert len(agent) == int(g["mctsa_len"]) and list(agent.action_queue) == g["mctsa_queue"].tolist()
	assert agent.search(O.solved(True), None, 100) is True
	assert len(agent) == 1 and list(agent.action_queue) == []


def test_determinism_and_reuse():
	"""Two runs are identical; a call on reused buffers after one with other starts equals a fresh agent."""
	a = np.stack(_scrambles(12, [3, 5, 7, 8] * 6))
	b = np.stack(_scrambles(13, [2, 4, 6, 8] * 6))

	def run(agent, starts):
		out = agent.search_many(starts, 500)
		h = _Host(agent)
		return out, [getattr(h, n).copy() for n in ("count", "states", "neighbors", "leaves", "N", "W", "V", "P", "L")]

	def same(x, y):
		(w1, q1, c1), a1 = x
		(w2, q2, c2), a2 = y
		assert (w1 == w2).all() and q1 == q2 and (c1 == c2).all()
		for k, n in enumerate(a1[0]):                       # the rows in use; rows past count keep an earlier call's data
			for u, v in zip(a1[1:], a2[1:]):
				assert _same(u[k, 1:n + 1], v[k, 1:n + 1]), k

	agent = _agent(_CountNet(), 2.0, True)
	r1 = run(agent, a)
	same(r1, run(agent, a))
	run(agent, b)
	same(r1, run(agent, a))
	same(r1, run(_agent(_CountNet(), 2.0, True), a))


def test_max_path_overflow_raises():
	"""A walk longer than max_path is an error naming the cap, not a silently shortened walk."""
	from rl_rubiks_b200 import _native as N
	agent = _agent(_CountNet(), 0.6, False, max_path=1)
	with pytest.raises(N.RubiksError, match="max_path = 1"):
		agent.search_many(np.stack(_scrambles(5, [6, 7])), 2000)
	with pytest.raises(ValueError):
		_agent(_CountNet(), 0.6, False, max_path=0)


@pytest.mark.parametrize("graph", [False, True], ids=["tree", "graph"])
def test_evaluator_parity(graph):
	"""eval_batched(MCTSBatch) and eval(MCTS) draw the same cubes and give the same turns and states, at fixed depths and in
	deep mode."""
	from rl_rubiks_b200.evaluation import Evaluator
	from tests.agent_harness import MCTS
	net = _CountNet()
	ev = Evaluator(4, range(1, 6), max_states=250)
	np.random.seed(17)
	res, states, _ = ev.eval(MCTS(net, 0.6, graph))
	np.random.seed(17)
	res_b, states_b, _ = ev.eval_batched(_agent(net, 0.6, graph))
	assert (res_b == res).all() and (states_b == states).all()
	assert (res[0] >= 1).all()
	ev = Evaluator(3, range(0), max_states=120)
	np.random.seed(5)
	res, states, _ = ev.eval(MCTS(net, 0.6, graph))
	np.random.seed(5)
	res_b, states_b, _ = ev.eval_batched(_agent(net, 0.6, graph))
	assert (res_b == res).all() and (states_b == states).all()
