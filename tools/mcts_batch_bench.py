#!/usr/bin/env python
"""One MCTS evaluation run both ways: `Evaluator.eval(MCTS)` (the statement-by-statement replay of the reference's agent in
tests/agent_harness.py, one search per cube) and `Evaluator.eval_batched(MCTSBatch)` (every cube in one batched search), from
the same numpy seed and with an exact net (uniform policy, value = cubies in their solved place; its outputs do not depend on
the batch).  Asserts that the two give identical results and states arrays, then prints the wall time of each, the batched
run's steps, kernel launches and host reads per step, and the card's name and power limit.
Then times the batched agent alone at an evaluation size: random-init fc_small (model.py:117-161: 480 -> 4096 -> 2048 ->
{512 -> 12, 512 -> 1}, ELU + BatchNorm1d) in eval mode with TF32, timing only.

Default size: 10 games x depths 1-10 (100 searches), c = 0.6, graph search, max_states = 3000; then 1000 cubes at depth 30
with max_states = 2000."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import cube_oracle as O  # noqa: E402
from rl_rubiks_b200 import _native as N  # noqa: E402
from rl_rubiks_b200 import cube  # noqa: E402
from rl_rubiks_b200.evaluation import Evaluator  # noqa: E402
from rl_rubiks_b200.frontier import MCTSBatch  # noqa: E402
from tests.agent_harness import MCTS  # noqa: E402


def card() -> str:
	try:
		q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
							"--format=csv,noheader"], capture_output=True, text=True, timeout=60)
		return q.stdout.strip() or f"{torch.cuda.get_device_name()} (power limit not readable)"
	except (OSError, subprocess.SubprocessError):
		return f"{torch.cuda.get_device_name()} (power limit not readable)"


class CountNet(torch.nn.Module):
	def __init__(self):
		super().__init__()
		self.w = torch.from_numpy(O.as_oh_2024(O.solved_2024()[None])[0]).cuda()

	def forward(self, x, policy=True, value=True):
		return torch.zeros(x.shape[0], 12, device=x.device), torch.floor(x @ self.w).unsqueeze(1)


class FCSmall(torch.nn.Module):
	def __init__(self):
		super().__init__()
		def block(a, b):
			return [torch.nn.Linear(a, b), torch.nn.ELU(), torch.nn.BatchNorm1d(b)]
		self.body = torch.nn.Sequential(*block(480, 4096), *block(4096, 2048))
		self.policy = torch.nn.Sequential(*block(2048, 512), torch.nn.Linear(512, 12))
		self.value = torch.nn.Sequential(*block(2048, 512), torch.nn.Linear(512, 1))

	def forward(self, x, policy=True, value=True):
		h = self.body(x)
		return self.policy(h), self.value(h)


class Counting:
	"""The agent's `search`, with the library's launches counted."""

	def __init__(self, agent):
		self.agent, self.launches = agent, 0

	def search(self, *a):
		l0 = N.lib.rb_launch_count()
		ok = self.agent.search(*a)
		self.launches += N.lib.rb_launch_count() - l0
		return ok

	def __getattr__(self, name):
		return getattr(self.agent, name)

	def __len__(self):
		return len(self.agent)


def main():
	ap = argparse.ArgumentParser()
	ap.add_argument("--games", type=int, default=10)
	ap.add_argument("--depths", type=str, default="1-10", help="first-last scrambling depth")
	ap.add_argument("--max-states", type=int, default=3000)
	ap.add_argument("--c", type=float, default=0.6)
	ap.add_argument("--tree", action="store_true", help="tree search instead of graph search")
	ap.add_argument("--seed", type=int, default=0)
	ap.add_argument("--eval-cubes", type=int, default=1000)
	ap.add_argument("--eval-depth", type=int, default=30)
	ap.add_argument("--eval-max-states", type=int, default=2000)
	args = ap.parse_args()
	graph = not args.tree
	lo, hi = (int(x) for x in args.depths.split("-"))
	ev = Evaluator(args.games, range(lo, hi + 1), max_states=args.max_states)
	print(f"card: {card()}")
	print(f"evaluation: {args.games} games x depths {lo}-{hi} = {args.games * (hi - lo + 1)} searches, max_states {args.max_states}, "
		  f"c {args.c}, {'graph' if graph else 'tree'} search, seed {args.seed}, exact net (uniform policy, cubies in place)")
	net = CountNet()

	np.random.seed(args.seed)
	agent = Counting(MCTS(net, args.c, graph))
	torch.cuda.synchronize()
	t0 = time.perf_counter()
	res, states, _ = ev.eval(agent)
	torch.cuda.synchronize()
	dt = time.perf_counter() - t0
	print(f"eval(MCTS):              {dt:8.3f} s  launches {agent.launches}; host reads: several per step of every search")

	batched = MCTSBatch(net, args.c, graph)
	for run in ("first", "again"):
		np.random.seed(args.seed)
		t0 = time.perf_counter()
		res_b, states_b, _ = ev.eval_batched(batched)
		dt_b = time.perf_counter() - t0
		assert (res_b == res).all(), "batched MCTS results differ from the sequential ones"
		assert (states_b == states).all(), "batched MCTS states differ from the sequential ones"
		print(f"eval_batched(MCTSBatch): {dt_b:8.3f} s  ({run} call) steps {batched.steps} launches {batched.launches} "
			  f"({batched.launches / max(batched.steps, 1):.1f} per step), host reads per step 1; {dt / dt_b:.1f}x the sequential eval")
	print(f"identical: results and states arrays ({int((res >= 0).sum())} of {res.size} solved, {int(states.sum())} states)")

	torch.backends.cuda.matmul.allow_tf32 = True
	torch.backends.cudnn.allow_tf32 = True
	fc = FCSmall().cuda().eval()
	rng = np.random.RandomState(args.seed)
	acts = rng.randint(0, 12, (args.eval_cubes, args.eval_depth)).astype(np.uint8)
	starts = cube.scramble_batch(acts)
	print(f"timing only: {args.eval_cubes} cubes at depth {args.eval_depth}, max_states {args.eval_max_states}, random-init fc_small "
		  f"(eval mode, TF32), c {args.c}, {'graph' if graph else 'tree'} search")
	batched = MCTSBatch(fc, args.c, graph)
	for run in ("first", "again"):
		torch.cuda.synchronize()
		t0 = time.perf_counter()
		won, _, count = batched.search_many(starts, args.eval_max_states)
		torch.cuda.synchronize()
		dt_b = time.perf_counter() - t0
		print(f"MCTSBatch: {dt_b:8.3f} s  ({run} call) steps {batched.steps} ({1e3 * dt_b / max(batched.steps, 1):.3f} ms per step) "
			  f"states {int(count.sum())} ({count.sum() / dt_b / 1e6:.3f} M states/s) solved {int(won.sum())}")


if __name__ == "__main__":
	main()
