#!/usr/bin/env python
"""One BFS evaluation run both ways: `Evaluator.eval(BFS())` (one search per cube, sequential) and
`Evaluator.eval_batched(BFSBatch())` (every cube in one batched search), from the same numpy seed.  Asserts that the two give
identical results and states arrays, then prints wall time, steps, kernel launches and host reads per step of each run and the
card's name and power limit.  The batched path runs once per step size in --steps (the first run of each allocates its
buffers; a second, timed again, reuses them).

Default size: 100 games x depths 1-6 (600 searches) with max_states = 50 000."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rl_rubiks_b200 import _native as N  # noqa: E402
from rl_rubiks_b200.evaluation import Evaluator  # noqa: E402
from rl_rubiks_b200.frontier import BFS, BFSBatch  # noqa: E402


def card() -> str:
	try:
		q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
							"--format=csv,noheader"], capture_output=True, text=True, timeout=60)
		return q.stdout.strip() or f"{torch.cuda.get_device_name()} (power limit not readable)"
	except (OSError, subprocess.SubprocessError):
		return f"{torch.cuda.get_device_name()} (power limit not readable)"


class Counting:
	"""The agent's `search`, with the library's launches and the searches counted."""

	def __init__(self, agent):
		self.agent, self.launches, self.searches = agent, 0, 0

	def search(self, *a):
		l0 = N.lib.rb_launch_count()
		ok = self.agent.search(*a)
		self.launches += N.lib.rb_launch_count() - l0
		self.searches += 1
		return ok

	def __getattr__(self, name):
		return getattr(self.agent, name)

	def __len__(self):
		return len(self.agent)


def main():
	ap = argparse.ArgumentParser()
	ap.add_argument("--games", type=int, default=100)
	ap.add_argument("--depths", type=str, default="1-6", help="first-last scrambling depth")
	ap.add_argument("--max-states", type=int, default=50000)
	ap.add_argument("--seed", type=int, default=0)
	ap.add_argument("--steps", type=str, default=str(BFSBatch._step), help="comma-separated pops per search and step to run")
	args = ap.parse_args()
	lo, hi = (int(x) for x in args.depths.split("-"))
	ev = Evaluator(args.games, range(lo, hi + 1), max_states=args.max_states)
	print(f"card: {card()}")
	print(f"evaluation: {args.games} games x depths {lo}-{hi} = {args.games * (hi - lo + 1)} searches, max_states {args.max_states}, seed {args.seed}")

	np.random.seed(args.seed)
	agent = Counting(BFS())
	torch.cuda.synchronize()
	t0 = time.perf_counter()
	res, states, _ = ev.eval(agent)
	torch.cuda.synchronize()
	dt = time.perf_counter() - t0
	print(f"eval(BFS()):              {dt:8.3f} s  launches {agent.launches} ({agent.launches / agent.searches:.1f} per search); "
		  f"host reads: 2 or more per slice of every search")

	for step in (int(x) for x in args.steps.split(",")):
		batched = BFSBatch()
		batched._step = step
		for run in ("first", "again"):
			np.random.seed(args.seed)
			t0 = time.perf_counter()
			res_b, states_b, _ = ev.eval_batched(batched)
			dt_b = time.perf_counter() - t0
			assert (res_b == res).all(), "batched BFS results differ from the sequential ones"
			assert (states_b == states).all(), "batched BFS states differ from the sequential ones"
			print(f"eval_batched(BFSBatch()): {dt_b:8.3f} s  N {step} ({run} call) steps {batched.steps} launches {batched.launches} "
				  f"host reads per step 1; {dt / dt_b:.1f}x the sequential eval")
	print(f"identical: results and states arrays ({int((res >= 0).sum())} of {res.size} solved, {int(states.sum())} states)")


if __name__ == "__main__":
	main()
