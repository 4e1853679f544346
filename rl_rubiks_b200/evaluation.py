"""
Evaluation driver: mirror of `Evaluator` (reference: librubiks/solving/evaluation.py:15-94) plus a batched variant
(SURVEY 8f row N3).

`Evaluator.eval(agent)` is the reference's sequential loop -- per scrambling depth and game: `cube.scramble(depth, True)`
then `agent.search(state, max_time, max_states)` -- and returns the same three (len(depths), n_games) arrays: turns to
solve (-1 unsolved), states explored (`len(agent)`) and seconds per game.

`Evaluator.eval_batched(agent)` draws exactly the same scrambles from the global numpy stream (same order of
`np.random` calls, evaluation.py:74-76 and cube.py:206-216), then hands ALL cubes of the evaluation to a batched agent
(`frontier.AStarBatch`, `frontier.BFSBatch` or `frontier.MCTSBatch`, through `search_many`) in one call, so that a B200
advances every search in lockstep instead of one cube at a time.  A* and MCTS (given the net) and BFS are deterministic given
the start state and a `max_states` budget, so `results` and `states` equal the sequential loop's; `times` is the wall time of the batch divided
evenly.  With one process per GPU the cubes are sharded by rank (searches are independent, no collective on the path) and
the three arrays gathered at the end.
"""
from __future__ import annotations

import time

import numpy as np
import torch

from . import cube, sharding


class Evaluator:
	def __init__(self, n_games, scrambling_depths, max_time=None, max_states=None):
		self.n_games, self.max_time, self.max_states = n_games, max_time, max_states
		# evaluation.py:30: an empty range means "deep": depths sampled uniformly in [100, 999]
		self.scrambling_depths = np.array(scrambling_depths) if scrambling_depths != range(0) else np.array([0])

	def _isdeep(self) -> bool:
		return self.scrambling_depths.size == 1 and self.scrambling_depths[0] == 0

	def approximate_time(self):
		return self.max_time * self.n_games * len(self.scrambling_depths)

	def _draw(self):
		"""The scrambles of one evaluation, [(state, depth)] * (len(depths) * n_games), consuming the global numpy stream exactly as
		the reference's loop does (evaluation.py:74-76 draws a depth in deep mode, cube.py:206-216 draws faces then directions and
		draws again when `force_not_solved` finds the cube solved) -- but scrambled in batches: all draws are made first, cubes of
		equal depth go through one `scramble_batch`, and only if some cube came out solved (possible at shallow depths only) is
		the stream rewound to just after that cube's draw and the remainder drawn again."""
		games = [int(d) for d in self.scrambling_depths for _ in range(self.n_games)]        # depth per game (0 = to be drawn)
		deep = self._isdeep()
		states, depths = [None] * len(games), list(games)
		first, pending = 0, False                       # `pending`: game `first` has its depth already and must redraw faces / dirs only
		while first < len(games):
			after, draws = [], []
			for j in range(first, len(games)):
				if deep and not (pending and j == first):
					depths[j] = int(np.random.randint(100, 1000))                              # evaluation.py:75-76
				faces = np.random.randint(6, size=(depths[j],))                                 # cube.py:208-209
				dirs = np.random.randint(2, size=(depths[j],))
				draws.append(cube._actions_u8(faces, dirs))
				after.append(np.random.get_state())
			out = [None] * len(draws)
			for d in sorted(set(depths[first:])):
				idx = [k for k in range(len(draws)) if depths[first + k] == d]
				batch = cube.scramble_batch(np.stack([draws[k] for k in idx])) if d else np.stack([cube.get_solved()] * len(idx))
				for k, st in zip(idx, batch):
					out[k] = st
			solved = [k for k in range(len(draws)) if depths[first + k] != 0 and bool((out[k] == cube.get_solved_instance()).all())]
			stop = solved[0] if solved else len(draws)
			states[first:first + stop] = out[:stop]
			first += stop
			pending = bool(solved)
			if solved:
				np.random.set_state(after[stop])                                                # the redraw continues right after that cube's draw
		return list(zip(states, depths))

	def eval(self, agent):
		"""evaluation.py:54-94, one `agent.search` per cube (the searches of the reference's agents draw nothing from the numpy
		stream, so making all scrambles first leaves every draw where the reference has it)."""
		res, states, times = [], [], []
		for state, _ in self._draw():
			t0 = time.perf_counter()
			solved = agent.search(state, self.max_time, self.max_states)
			times.append(time.perf_counter() - t0)
			res.append(len(agent.action_queue) if solved else -1)
			states.append(len(agent))
		shape = (len(self.scrambling_depths), self.n_games)
		return np.reshape(res, shape), np.reshape(states, shape), np.reshape(times, shape)

	def eval_batched(self, agent, shard: bool = True):
		"""All cubes of the evaluation in one `agent.search_many(states, max_states)` call (`AStarBatch`, `BFSBatch`, `MCTSBatch`; this rank's
		share of them when a process group is up and `shard` is set).  Requires `max_states` (a wall-clock limit has no batched
		meaning)."""
		if not self.max_states:
			raise ValueError("eval_batched needs max_states: batched searches advance in lockstep and have no per-game time limit")
		starts = np.stack([s for s, _ in self._draw()])                    # same draws on every rank (same numpy seed)
		n = len(starts)
		rank, ws = sharding.world() if shard else (0, 1)
		lo, hi = sharding.shard_bounds(n, ws, rank)
		torch.cuda.synchronize()
		t0 = time.perf_counter()
		won, queues, count = agent.search_many(starts[lo:hi], self.max_states)
		torch.cuda.synchronize()
		dt = time.perf_counter() - t0
		res = np.array([len(q) if w else -1 for w, q in zip(won, queues)], dtype=np.int64)
		local = torch.from_numpy(np.stack([res, np.asarray(count, dtype=np.int64)], axis=1))
		if ws > 1:
			local = sharding.gather_rows(local.cuda(), n).cpu()
			dt = sharding.reduce_stats({"s": dt}, op="max", device=torch.device("cuda", torch.cuda.current_device()))["s"]
		shape = (len(self.scrambling_depths), self.n_games)
		out = local.numpy()
		return out[:, 0].reshape(shape), out[:, 1].reshape(shape), np.full(shape, dt / max(n, 1))

	@staticmethod
	def states_per_sec(states: np.ndarray, times: np.ndarray) -> np.ndarray:
		"""evaluation.py:120-121: the reference's per-game throughput statistic."""
		safe = times != 0
		return states[safe] / times[safe]
