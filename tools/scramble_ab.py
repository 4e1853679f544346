#!/usr/bin/env python
"""A/B timing of the scramble between two builds of librubiks_b200.so loaded into one process: rounds alternate the two builds
(ROUNDS rounds of REPS launches each), and the outputs are compared byte for byte with each other and on a subsample with the
oracle.  One line per depth: median ms per launch [min-max] of each build, their ratio.

  python tools/scramble_ab.py OLD.so NEW.so        env: LAYOUT=cube  DEPTHS=100,200  CUBES=16777216  ROUNDS=7  REPS=20  TAG=label

LAYOUT picks the kernel family: cube = rb_scramble on cube-major actions [n][depth], move = the same actions transposed to
move-major [depth][n], seeded = rb_scramble_seeded (moves drawn on the device; parity replays rb_seeded_actions on the oracle)."""
import ctypes as C
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import cube_oracle as O  # noqa: E402

libs = {}
for name, path in (("old", os.path.abspath(sys.argv[1])), ("new", os.path.abspath(sys.argv[2]))):
	L = C.CDLL(path)
	L.rb_scramble.restype = C.c_int
	L.rb_scramble.argtypes = [C.c_int, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]
	L.rb_scramble_seeded.restype = C.c_int
	L.rb_scramble_seeded.argtypes = [C.c_int, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]
	L.rb_seeded_actions.restype = C.c_int
	L.rb_seeded_actions.argtypes = [C.c_uint64, C.c_uint64, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]
	L.rb_last_error.restype = C.c_char_p
	libs[name] = L

dev = torch.device("cuda", 0)
torch.cuda.set_device(0)
sh = C.c_void_p(torch.cuda.current_stream().cuda_stream)
depths = [int(x) for x in os.environ.get("DEPTHS", "100").split(",")]
n = int(os.environ.get("CUBES", str(1 << 24)))
rounds, reps = int(os.environ.get("ROUNDS", "7")), int(os.environ.get("REPS", "20"))
tag = os.environ.get("TAG", "")
layout = os.environ.get("LAYOUT", "cube")
assert layout in ("cube", "move", "seeded"), layout
SEED = 3
for depth in depths:
	if layout == "seeded":
		acts = torch.empty(n, depth, dtype=torch.uint8, device=dev)       # the stream the kernel draws, for the oracle
		if libs["new"].rb_seeded_actions(SEED, 0, C.c_void_p(acts.data_ptr()), n, depth, sh):
			raise RuntimeError(libs["new"].rb_last_error().decode())
	else:
		g = torch.Generator(device=dev); g.manual_seed(SEED)
		acts = torch.randint(0, 12, (n, depth), dtype=torch.uint8, device=dev, generator=g)
	acts_mm = acts.t().contiguous() if layout == "move" else None
	outs = {k: torch.empty(n, 20, dtype=torch.int8, device=dev) for k in libs}

	def run(k):
		o = C.c_void_p(outs[k].data_ptr())
		if layout == "cube":
			rc = libs[k].rb_scramble(0, C.c_void_p(acts.data_ptr()), depth, 1, None, o, n, depth, sh)
		elif layout == "move":
			rc = libs[k].rb_scramble(0, C.c_void_p(acts_mm.data_ptr()), 1, n, None, o, n, depth, sh)
		else:
			rc = libs[k].rb_scramble_seeded(0, SEED, 0, None, o, n, depth, sh)
		if rc:
			raise RuntimeError(libs[k].rb_last_error().decode())

	for k in libs:
		for _ in range(3):
			run(k)
	torch.cuda.synchronize()
	ms = {k: [] for k in libs}
	for r in range(rounds):
		for k in (("old", "new") if r % 2 == 0 else ("new", "old")):
			a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
			a.record()
			for _ in range(reps):
				run(k)
			b.record(); torch.cuda.synchronize()
			ms[k].append(a.elapsed_time(b) / reps)
	same = bool(torch.equal(outs["old"], outs["new"]))
	sub = torch.arange(0, n, max(1, n // 4096), device=dev)
	f, d = O.indices_to_actions(acts[sub].cpu().numpy())
	ok = bool((outs["new"][sub].cpu().numpy() == O.scramble_many(f, d, True)).all())
	mo, mn = float(np.median(ms["old"])), float(np.median(ms["new"]))
	print(f"{tag} {layout} depth {depth} n {n} old {mo:.4f} [{min(ms['old']):.4f}-{max(ms['old']):.4f}] new {mn:.4f} "
		  f"[{min(ms['new']):.4f}-{max(ms['new']):.4f}] new/old {mn / mo:.4f} identical {same} parity {ok}", flush=True)
	del acts, acts_mm, outs
	torch.cuda.empty_cache()
