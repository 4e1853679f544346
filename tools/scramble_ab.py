#!/usr/bin/env python
"""A/B timing of rb_scramble (cube-major actions, 20x24 states) between two builds of librubiks_b200.so loaded into one process:
rounds alternate the two builds (ROUNDS rounds of REPS launches each), and the outputs are compared byte for byte with each other
and on a subsample with the oracle.  One line per depth: median ms per launch [min-max] of each build, their ratio.

  python tools/scramble_ab.py OLD.so NEW.so        env: DEPTHS=100,200  CUBES=16777216  ROUNDS=7  REPS=20  TAG=label

Environment knobs (RB_SCRAMBLE_*) apply to both builds."""
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
	L.rb_last_error.restype = C.c_char_p
	libs[name] = L

dev = torch.device("cuda", 0)
torch.cuda.set_device(0)
sh = C.c_void_p(torch.cuda.current_stream().cuda_stream)
depths = [int(x) for x in os.environ.get("DEPTHS", "100").split(",")]
n = int(os.environ.get("CUBES", str(1 << 24)))
rounds, reps = int(os.environ.get("ROUNDS", "7")), int(os.environ.get("REPS", "20"))
tag = os.environ.get("TAG", "")
for depth in depths:
	g = torch.Generator(device=dev); g.manual_seed(3)
	acts = torch.randint(0, 12, (n, depth), dtype=torch.uint8, device=dev, generator=g)
	outs = {k: torch.empty(n, 20, dtype=torch.int8, device=dev) for k in libs}

	def run(k):
		rc = libs[k].rb_scramble(0, C.c_void_p(acts.data_ptr()), depth, 1, None, C.c_void_p(outs[k].data_ptr()), n, depth, sh)
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
	print(f"{tag} depth {depth} n {n} old {mo:.4f} [{min(ms['old']):.4f}-{max(ms['old']):.4f}] new {mn:.4f} "
		  f"[{min(ms['new']):.4f}-{max(ms['new']):.4f}] new/old {mn / mo:.4f} identical {same} parity {ok}", flush=True)
	del acts, outs
	torch.cuda.empty_cache()
