#!/usr/bin/env python
"""
bench.py -- headline benchmark of the cube-dynamics hot path (BASELINE.json configs[1]):
raw scramble throughput, 2^24 cubes x 100 random moves, 20x24 representation, per GPU (weak scaling).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --gpus N ...            # the reference's numpy algorithm on the host cores
  python bench.py ... --dump-outputs DIR                   # also write the last timed step's states to DIR/states.npy

One JSON line on stdout (rank 0).  A "step" is one pass of the scramble kernel over the whole batch of
host-supplied action sequences already resident in HBM (`value`), and the same pass through the host-buffer C-ABI
call `rbh_scramble` with the H2D/D2H copies inside the timed region (`e2e`).  `roofline` is the scramble kernel's
algorithmic bytes (100 B actions in + 20 B state out per cube, SURVEY 8d C2) over its CUDA-event time against the
measured HBM copy peak; `extra.adi` reports the fused ADI generator (configs[0]) the same way.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_CUBES = 1 << 24
DEPTH = 100
BYTES_PER_CUBE = DEPTH + 20          # uint8 actions in + int8[20] state out (SURVEY 8d, C2)
# ncu --set full capture of the shipped scramble kernel (one 2^24-cube launch), summarised by tools/ncu_summary.py: bench.py reads
# `roofline.traffic` (dram read + write) and the limiter percentages from this file at run time.
NCU_SUMMARY = os.path.join(ROOT, "profiles", "r2_scramble_macro3_ncu.json")
DUMP_ROWS = 1 << 19          # --dump-outputs: a fixed sample of the final states (2^19 x 20 float32 = 40 MB)
METRIC, UNIT = "cube_moves_per_sec", "moves/s"
WORKLOAD = "raw scramble: 2^24 cubes x 100 random moves per GPU, 20x24 rep, packed int8 (BASELINE configs[1])"


def measured_peaks():
	path = os.path.join(ROOT, "MEASURED_PEAKS.json")
	if os.path.exists(path):
		return json.load(open(path)), "measured (MEASURED_PEAKS.json)"
	return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


def ncu_capture():
	"""-> (dram bytes per cube, limiter dict, source) from the committed ncu summary, or (None, None, why)."""
	try:
		m = json.load(open(NCU_SUMMARY))["launches"][0]["metrics"]
		per_cube = (m["dram__bytes_read.sum"] + m["dram__bytes_write.sum"]) / (1 << 24)
		lim = {"l1tex_pct": m["l1tex__throughput.avg.pct_of_peak_sustained_elapsed"],
			   "alu_pipe_pct": m["sm__pipe_alu_cycles_active.avg.pct_of_peak_sustained_active"],
			   "fma_pipe_pct": m["sm__pipe_fma_cycles_active.avg.pct_of_peak_sustained_active"],
			   "issue_active_pct": m["smsp__issue_active.avg.pct_of_peak_sustained_active"],
			   "dram_pct": m["gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed"],
			   "shared_wavefronts": m["l1tex__data_pipe_lsu_wavefronts_mem_shared.sum"],
			   "shared_bank_conflict_replays": m["l1tex__data_bank_conflicts_pipe_lsu_mem_shared.sum"],
			   "mio_throttle_stall_per_issue": m["smsp__average_warps_issue_stalled_mio_throttle_per_issue_active.ratio"],
			   "resource": "shared-memory wavefronts of the table gathers (l1tex 95 %, MIO throttle the top stall; half are bank-conflict "
						   "replays), with the integer ALU pipe right behind: conflict-free table reads (throw-away builds) reach 0.72 ms "
						   "= 0.43 of the roofline, where the ALU pipe takes over: profiles/r2_scramble_pipe_experiments.txt"}
		return per_cube, lim, "ncu --set full, " + os.path.relpath(NCU_SUMMARY, ROOT)
	except (OSError, KeyError, IndexError, ValueError) as e:
		return None, None, f"no ncu summary ({e})"


class ClockSampler:
	"""Samples SM clocks and throttle reasons through NVML (a polling thread, ~1 kHz) while the timed regions run; falls
	back to `nvidia-smi -lms` when the NVML binding is missing."""
	Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
		"clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

	def __init__(self, index: int):
		self.index, self.sm, self.reasons, self.max_mhz = index, [], set(), None
		self.proc, self.stop, self.thread, self.rows = None, threading.Event(), None, []

	def _poll_nvml(self, nv, h):
		bits = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
				"sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
		while not self.stop.is_set():
			try:
				self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
				r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
				self.reasons.update(k for k, b in bits.items() if r & b)
			except Exception:
				break
			time.sleep(0.001)

	def __enter__(self):
		try:
			import pynvml as nv
			nv.nvmlInit()
			vis, phys = os.environ.get("CUDA_VISIBLE_DEVICES", ""), self.index      # CUDA_VISIBLE_DEVICES may renumber
			parts = [x.strip() for x in vis.split(",")] if vis else []
			if self.index < len(parts) and parts[self.index].isdigit():
				phys = int(parts[self.index])
			h = nv.nvmlDeviceGetHandleByIndex(phys)
			self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
			self.thread = threading.Thread(target=self._poll_nvml, args=(nv, h), daemon=True)
			self.thread.start()
			return self
		except Exception:
			pass
		try:
			self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
										 stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
			self.thread = threading.Thread(target=self._pump, daemon=True)
			self.thread.start()
		except OSError:
			self.proc = None
		return self

	def _pump(self):
		names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
		for line in self.proc.stdout:
			r = [x.strip() for x in line.split(",")]
			if len(r) >= 6 and r[0].replace(".", "").isdigit():
				self.sm.append(float(r[0]))
				self.max_mhz = max(self.max_mhz or 0.0, float(r[1])) if r[1].replace(".", "").isdigit() else self.max_mhz
				self.reasons.update(n for n, v in zip(names, r[2:6]) if v.lower().startswith("active"))

	def __exit__(self, *exc):
		self.stop.set()
		if self.proc:
			time.sleep(0.05)
			self.proc.terminate()
		if self.thread:
			self.thread.join(timeout=2)

	def summary(self):
		return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
				"samples": len(self.sm)}


# ------------------------------------------------------------------------------------------------------------
# CPU legs, fanned out over the host cores.  kind "reference": the reference's OWN librubiks.cube (unmodified copy under
# baseline/_ref, made by baseline/make_ref.py; travels to the GPU box with the working tree) running the loop of cube.py:229-231,
# `states = multi_rotate(states, faces[d], dirs[d])` for d in range(depth).  kind "port": the numpy oracle (the restatement used
# as the parity checker), about 2.3 x faster per core than the reference because it looks moves up in one direct table.
# ------------------------------------------------------------------------------------------------------------
CPU_CHUNK = 1 << 14          # cubes per numpy call: the (depth, n) int64 draws of a chunk stay cache/RAM friendly
REF_DIR = os.path.join(ROOT, "baseline", "_ref")


def ref_available() -> bool:
	return os.path.exists(os.path.join(REF_DIR, "librubiks", "cube", "cube.py"))


def _cpu_worker(args):
	seed, chunks, depth, kind = args
	os.environ["CUDA_VISIBLE_DEVICES"] = ""          # CPU legs: the reference picks its device at import time (librubiks/__init__.py:5-6)
	g = np.random.RandomState(seed)
	faces, dirs = g.randint(0, 6, (depth, CPU_CHUNK)), g.randint(0, 2, (depth, CPU_CHUNK))
	if kind == "reference":
		if REF_DIR not in sys.path:
			sys.path.insert(0, REF_DIR)
		from librubiks import cube as ref_cube
		ref_cube.set_is2024(True)
		t0 = time.perf_counter()
		for _ in range(chunks):
			states = np.array([ref_cube.get_solved()] * CPU_CHUNK)
			for d in range(depth):
				states = ref_cube.multi_rotate(states, faces[d], dirs[d])
		return time.perf_counter() - t0
	from oracle import cube_oracle as O
	faces, dirs = np.ascontiguousarray(faces.T), np.ascontiguousarray(dirs.T)
	t0 = time.perf_counter()
	for _ in range(chunks):
		O.scramble_many(faces, dirs, True)
	return time.perf_counter() - t0


def cpu_scramble_throughput(chunks_per_core: int, depth: int, cores: int, kind: str, pool=None):
	"""moves/s of the CPU path: `cores` processes, each scrambling `chunks_per_core` x 2^14 cubes (wall clock of the slowest)."""
	own = pool is None
	if own:
		pool = cpu_pool(cores, depth, kind)
	try:
		t0 = time.perf_counter()
		pool.map(_cpu_worker, [(s, chunks_per_core, depth, kind) for s in range(cores)], chunksize=1)
		dt = time.perf_counter() - t0
	finally:
		if own:
			pool.close()
	return cores * chunks_per_core * CPU_CHUNK * depth / dt, dt


def cpu_pool(cores: int, depth: int, kind: str):
	"""Worker processes started with `spawn` (the parent may hold a CUDA context, which a forked child must not touch) and warmed
	up: every worker has imported numpy / torch / the CPU implementation before anything is timed."""
	import multiprocessing as mp
	pool = mp.get_context("spawn").Pool(cores)
	pool.map(_cpu_worker, [(s, 0, depth, kind) for s in range(4 * cores)], chunksize=1)
	return pool


def cpu_sample_text(kind, cores, chunks, depth, dt=None):
	what = ("the reference's own librubiks.cube.multi_rotate loop (cube.py:229-231, unmodified copy in baseline/_ref)" if kind == "reference"
			else "numpy oracle port of cube.py:206-263")
	return f"{cores} processes x {chunks * CPU_CHUNK} cubes x {depth} moves, {what}" + (f", {dt:.1f} s" if dt is not None else "") + \
		"; throughput per move, the GPU arm runs 2^24 cubes"


def run_reference(args):
	"""--impl reference: the reference's CPU implementation of the path on all host cores, a bounded sample per step."""
	rank = int(os.environ.get("RANK", "0"))
	if rank != 0:
		return
	cores = os.cpu_count() or 1
	kind = "reference" if ref_available() else "port"
	per_core = 2 if kind == "reference" else 4            # chunks of 2^14 cubes per core and step: ~1.3 s of CPU work per step
	pool = cpu_pool(cores, DEPTH, kind)
	try:
		for _ in range(args.warmup):
			cpu_scramble_throughput(per_core, DEPTH, cores, kind, pool)
		t0 = time.perf_counter()
		for _ in range(args.steps):
			cpu_scramble_throughput(per_core, DEPTH, cores, kind, pool)
		dt = time.perf_counter() - t0
	finally:
		pool.close()
	value = args.steps * cores * per_core * CPU_CHUNK * DEPTH / dt
	sample = cpu_sample_text(kind, cores, per_core, DEPTH) + " per step"
	print(json.dumps({
		"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
		"warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
		"vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": {"workload": WORKLOAD, "sample": sample},
		"cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
		"e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
	}), flush=True)


# ------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------
def run_gpu(args):
	import torch
	import torch.distributed as dist
	rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
	local = int(os.environ.get("LOCAL_RANK", "0"))
	torch.cuda.set_device(local)
	dev = torch.device("cuda", local)
	if world > 1:
		# stdout carries ONE JSON line: NCCL_DEBUG=VERSION makes NCCL printf its version to stdout, INFO / TRACE go to the debug file
		if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
			os.environ["NCCL_DEBUG"] = "WARN"
		os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
		dist.init_process_group("nccl", device_id=dev)
	import rl_rubiks_b200  # noqa: F401  (raises if the CUDA library is missing: no CPU fallback)
	from rl_rubiks_b200 import _native as N, adi, cube, sharding

	n, depth = args.cubes, DEPTH
	gen = torch.Generator(device=dev)
	gen.manual_seed(sharding.rank_seed(1234, rank))   # each rank scrambles its own shard of cubes (weak scaling, no collective)
	actions = torch.randint(0, 12, (n, depth), dtype=torch.uint8, device=dev, generator=gen)
	out = torch.empty(n, 20, dtype=torch.int8, device=dev)
	stream = N.stream_handle()

	def step():
		N.check(N.lib.rb_scramble(N.REP_2024, N.ptr(actions), depth, 1, None, N.ptr(out), n, depth, stream))

	def barrier():
		if world > 1:
			dist.barrier()
		torch.cuda.synchronize()

	for _ in range(max(args.warmup, 3)):
		step()
	barrier()
	launches0 = N.lib.rb_launch_count()
	ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
	with ClockSampler(local) as clocks:
		barrier()
		ev[0].record()
		for k in range(args.steps):
			step()
			ev[k + 1].record()
		barrier()
	launches = N.lib.rb_launch_count() - launches0
	if args.dump_outputs and rank == 0:
		# the states the last timed step returned (`out` is reused further down): the same seeded rows on every run, so that two
		# builds can be compared output for output
		rows = np.sort(np.random.RandomState(0).choice(n, min(n, DUMP_ROWS), replace=False))
		states = out[torch.from_numpy(rows).to(dev)].cpu().numpy().astype(np.float32)
		os.makedirs(args.dump_outputs, exist_ok=True)
		np.save(os.path.join(args.dump_outputs, "states.npy"), states)
	ms_total = ev[0].elapsed_time(ev[-1])
	per_launch_ms = [ev[k].elapsed_time(ev[k + 1]) for k in range(args.steps)]
	t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
	if world > 1:
		dist.all_reduce(t, op=dist.ReduceOp.MAX)
	ms_total = float(t.item())
	ms_step = ms_total / args.steps
	value = world * n * depth / (ms_step * 1e-3)

	# parity spot check of what was just timed (bit-exact vs the oracle on a subsample), outside the timed region
	from oracle import cube_oracle as O
	sub = torch.arange(0, n, max(1, n // 2048), device=dev)[:2048]
	f, d = O.indices_to_actions(actions[sub].cpu().numpy())
	parity_ok = bool((out[sub].cpu().numpy() == O.scramble_many(f, d, True)).all())
	out_ref = out[:4096].cpu().numpy()

	# ---- end to end: host buffers through the C-ABI calls, copies inside the timed region ----
	# (a) rbh_scramble_seeded: the reference's own call shape -- cube.scramble draws its moves itself (cube.py:206-211), so the
	#     inputs are (seed, first cube, n, depth) and the results come back as int8[n][20]: 20 B per cube over PCIe.  HEADLINE e2e.
	# (b) rbh_scramble: host-drawn actions uint8[n][100] in, states out: 120 B per cube over PCIe.
	# (c) rbh_scramble_packed: host-drawn actions, two moves per byte: 70 B per cube over PCIe.
	host_out = torch.empty(n, 20, dtype=torch.int8, pin_memory=True)
	e2e_steps = max(1, min(args.steps, 5))
	seed, first_cube = 20241018, rank * n                      # rank r owns cubes [r n, (r + 1) n) of ONE stream: no collective

	def timed_e2e(call):
		N.check(call())
		barrier()
		t0 = time.perf_counter()
		for _ in range(e2e_steps):
			N.check(call())
		barrier()
		te = torch.tensor([(time.perf_counter() - t0) / e2e_steps], dtype=torch.float64, device=dev)
		if world > 1:
			dist.all_reduce(te, op=dist.ReduceOp.MAX)
		return float(te.item())

	seeded_s = timed_e2e(lambda: N.lib.rbh_scramble_seeded(N.REP_2024, seed, first_cube, N.ptr(host_out), n, depth))
	# parity of what was just timed: replay the dumped moves of a subsample on the oracle
	sub_n = 2048
	sub_first = first_cube + (n - sub_n)
	sub_actions = cube.seeded_actions(sub_n, depth, seed, sub_first).cpu().numpy()
	assert (sub_actions == O.seeded_actions(seed, sub_first, sub_n, depth)).all()
	f, d = O.indices_to_actions(sub_actions)
	seeded_ok = bool((host_out[n - sub_n:].numpy() == O.scramble_many(f, d, True)).all())
	# device-timed seeded kernel alone (20 B per cube leave the chip)
	for _ in range(3):
		N.check(N.lib.rb_scramble_seeded(N.REP_2024, seed, first_cube, None, N.ptr(out), n, depth, stream))
	sa, sb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
	barrier()
	sa.record()
	for _ in range(args.steps):
		N.check(N.lib.rb_scramble_seeded(N.REP_2024, seed, first_cube, None, N.ptr(out), n, depth, stream))
	sb.record()
	barrier()
	ts = torch.tensor([sa.elapsed_time(sb) / args.steps], dtype=torch.float64, device=dev)
	if world > 1:
		dist.all_reduce(ts, op=dist.ReduceOp.MAX)
	seeded_kernel_ms = float(ts.item())

	host_actions = torch.empty(n, depth, dtype=torch.uint8, pin_memory=True)
	host_actions.copy_(actions)
	host_s = timed_e2e(lambda: N.lib.rbh_scramble(N.REP_2024, N.ptr(host_actions), N.ptr(host_out), n, depth))
	e2e_ok = bool((host_out[:4096].numpy() == out_ref[:4096]).all())
	host_packed = torch.empty(n, depth // 2, dtype=torch.uint8, pin_memory=True)
	host_packed.copy_(actions[:, 0::2] + 13 * actions[:, 1::2])
	packed_s = timed_e2e(lambda: N.lib.rbh_scramble_packed(N.REP_2024, N.ptr(host_packed), N.ptr(host_out), n, depth))
	packed_ok = bool((host_out[:4096].numpy() == out_ref[:4096]).all())
	N.check(N.lib.rbh_release())
	del host_actions, host_out, host_packed

	# ---- secondary: fused ADI generator at BASELINE configs[0] (1000 games x depth 25, lapanfix) ----
	games, adepth = 1000, 25
	gadi = adi.ADIGenerator(games, adepth, "lapanfix", keep_states=True)
	gadi.set_actions(torch.randint(0, 12, (adepth, games), dtype=torch.uint8, device=dev, generator=gen))
	values = torch.randn(12 * games * adepth, device=dev)
	flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # > 126 MB L2
	for _ in range(3):
		gadi.generate(); gadi.targets(values, 0.3)
	adi_ms = []
	for _ in range(10):
		flush.zero_()
		a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
		a.record(); gadi.generate(); gadi.targets(values, 0.3); b.record()
		torch.cuda.synchronize()
		adi_ms.append(a.elapsed_time(b))
	def over_ranks(seconds):
		"""(max over ranks, this rank's): every rank generates its own batch, the aggregate rate is world * batch / slowest rank."""
		t = torch.tensor([seconds], dtype=torch.float64, device=dev)
		if world > 1:
			dist.all_reduce(t, op=dist.ReduceOp.MAX)
		return float(t.item())

	adi_t_rank = float(np.median(adi_ms)) * 1e-3
	adi_t = over_ranks(adi_t_rank)
	nst = games * adepth
	# same batch with bf16 one-hot rows (opt-in dtype, not the reference's: half the write traffic, input of a bf16 forward)
	gadi16 = adi.ADIGenerator(games, adepth, "lapanfix", keep_states=True, oh_dtype=torch.bfloat16)
	gadi16.actions.copy_(gadi.actions)
	for _ in range(3):
		gadi16.generate(); gadi16.targets(values, 0.3)
	adi16_ms = []
	for _ in range(10):
		flush.zero_()
		a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
		a.record(); gadi16.generate(); gadi16.targets(values, 0.3); b.record()
		torch.cuda.synchronize()
		adi16_ms.append(a.elapsed_time(b))
	adi16_t = over_ranks(float(np.median(adi16_ms)) * 1e-3)
	adi16_bytes = 960 * 13 * nst + 20 * nst + 13 * nst + 4 * 12 * nst + 16 * nst + nst
	adi_bytes = 1920 * 13 * nst + 20 * nst + 13 * nst + 4 * 12 * nst + 16 * nst + nst      # SURVEY 8d C1: 626 450 000 B

	peaks, peak_src = measured_peaks()
	peak = float(peaks["hbm_gbs"])
	kernel_ms = float(np.mean(per_launch_ms))
	achieved = BYTES_PER_CUBE * n / (kernel_ms * 1e-3) / 1e9
	if rank != 0:
		if world > 1:
			dist.destroy_process_group()
		return
	cores = os.cpu_count() or 1
	cpu_kind = "reference" if ref_available() else "port"
	cpu_chunks = 12 if cpu_kind == "reference" else 32     # ~8-10 s of work on every host core
	cpu_value, cpu_dt = cpu_scramble_throughput(cpu_chunks, depth, cores, cpu_kind)
	port_value, port_dt = cpu_scramble_throughput(16, depth, cores, "port")
	one_value, one_dt = cpu_scramble_throughput(4, depth, 1, cpu_kind)          # the reference as it runs: one process (BASELINE.md 4.2a)
	ncu_per_cube, limiter, ncu_src = ncu_capture()
	result = {
		"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
		"ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
		"data": "synthetic",
		"config": {"workload": WORKLOAD, "cubes_per_gpu": n, "depth": depth, "actions": "host-supplied uint8 [n][100], resident in HBM",
				   "l2": "inputs (1.68 GB actions) larger than the 126 MB L2, no reuse between steps", "parity_subsample_ok": parity_ok},
		"roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
					 "traffic": int(ncu_per_cube * n) if ncu_per_cube is not None else None,
					 "traffic_source": ncu_src + " (dram read + write of one 2^24-cube launch, scaled by cubes)",
					 "peak_source": peak_src, "kernel": "rbs::k_scramble_macro3<1, 1>", "kernel_ms": kernel_ms,
					 "algorithmic_bytes_per_launch": BYTES_PER_CUBE * n,
					 "note": "100 dependent moves per 120 bytes: the multi-move scramble is bound by the shared-memory table gathers with the integer ALU pipe right behind (measured floor of the design 0.72 ms = 0.43), not HBM-bound: DESIGN.md 3.1",
					 "limiter": dict(limiter, source=ncu_src) if limiter else None},
		"cpu_baseline": {"value": cpu_value, "unit": UNIT, "cores": cores, "kind": cpu_kind, "sample": cpu_sample_text(cpu_kind, cores, cpu_chunks, depth, cpu_dt),
						 "single_process": {"value": one_value, "cores": 1, "kind": cpu_kind, "sample": cpu_sample_text(cpu_kind, 1, 4, depth, one_dt)},
						 "port": {"value": port_value, "kind": "port", "sample": cpu_sample_text("port", cores, 16, depth, port_dt)}},
		"e2e": {"value": world * n * depth / seeded_s, "unit": UNIT, "h2d_bytes_per_step": 16, "d2h_bytes_per_step": n * 20,
				"ms_per_step": seeded_s * 1e3, "parity_ok": seeded_ok,
				"api": "rbh_scramble_seeded (C ABI): the moves are drawn on the device (Philox4x32-10, one subsequence per cube) as cube.scramble "
					   "draws its own (cube.py:206-211); in: seed + first cube id (16 B), out: int8[n][20] to pinned host memory",
				"algorithmic_bytes_per_cube": 20,
				"note": "PCIe-bound: 20 B per cube come back at ~56 GB/s on one GPU; the N GPUs of one box share one path into host memory "
						"(71 / 75 / 95 GB/s in total at N = 2 / 4 / 8 on this pool's VM hosts, DESIGN.md 6), so the end-to-end rate does not scale with N "
						"while the device-timed value does",
				"host_actions": {"value": world * n * depth / host_s, "ms_per_step": host_s * 1e3, "h2d_bytes_per_step": n * depth,
								 "d2h_bytes_per_step": n * 20, "api": "rbh_scramble: host-drawn uint8[n][100] actions in", "parity_ok": e2e_ok,
								 "algorithmic_bytes_per_cube": 120},
				"packed_actions": {"value": world * n * depth / packed_s, "ms_per_step": packed_s * 1e3, "h2d_bytes_per_step": n * depth // 2,
								   "d2h_bytes_per_step": n * 20, "api": "rbh_scramble_packed: host-drawn actions, two moves per byte", "parity_ok": packed_ok,
								   "algorithmic_bytes_per_cube": 70}},
		"gpu_launches": int(launches),
		"clocks": clocks.summary(),
		"extra": {"note": "adi / adi_bf16_rows: every rank generates its own batch (weak scaling); samples_per_sec = n_gpus x batch / slowest rank",
				  "seeded_kernel": {"workload": "rb_scramble_seeded, device-resident: Philox draw + scramble in one kernel, 20 B per cube written",
									"moves_per_sec": world * n * depth / (seeded_kernel_ms * 1e-3), "ms": seeded_kernel_ms},
				  "adi": {"workload": "fused ADI batch 1000 games x depth 25 (BASELINE configs[0]): generate + targets kernels",
						  "samples_per_sec": world * nst / adi_t, "children_per_sec": world * 12 * nst / adi_t, "ms": adi_t * 1e3,
							  "samples_per_sec_per_gpu": nst / adi_t, "n_gpus": world,
						  "roofline": {"bound": "hbm", "achieved": adi_bytes / adi_t / 1e9, "peak": peak, "unit": "GB/s",
									   "frac": adi_bytes / adi_t / 1e9 / peak, "algorithmic_bytes": adi_bytes},
						  "l2": "256 MB flush buffer written between timed iterations"},
				  "adi_bf16_rows": {"workload": "same batch, one-hot rows emitted as bfloat16 (opt-in; the reference's dtype is f32)",
									"samples_per_sec": world * nst / adi16_t, "samples_per_sec_per_gpu": nst / adi16_t, "ms": adi16_t * 1e3,
									"roofline": {"bound": "hbm", "achieved": adi16_bytes / adi16_t / 1e9, "peak": peak, "unit": "GB/s",
												 "frac": adi16_bytes / adi16_t / 1e9 / peak, "algorithmic_bytes": adi16_bytes}}},
	}
	print(json.dumps(result), flush=True)
	if world > 1:
		dist.destroy_process_group()


def main():
	ap = argparse.ArgumentParser()
	ap.add_argument("--gpus", type=int, default=1)
	ap.add_argument("--steps", type=int, default=20)
	ap.add_argument("--warmup", type=int, default=3)
	ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
	ap.add_argument("--cubes", type=int, default=N_CUBES, help="cubes per GPU (default 2^24, the BASELINE size)")
	ap.add_argument("--dump-outputs", metavar="DIR", default=None,
					help="after the timed steps, write the int8[20] states of the last step as float32 to DIR/states.npy: "
						 f"rank 0's cubes, at most {DUMP_ROWS} rows drawn with a fixed seed, in cube order")
	args = ap.parse_args()
	if args.steps < 1:
		ap.error("--steps must be at least 1")
	if args.dump_outputs and args.impl == "reference":
		ap.error("--dump-outputs applies to the CUDA arm (--impl b200)")
	if args.impl == "reference":
		run_reference(args)
		return
	world = int(os.environ.get("WORLD_SIZE", "1"))
	if args.gpus > 1 and world == 1:
		# convenience: re-launch under torchrun, one process per GPU
		cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
			   "--master-port", os.environ.get("MASTER_PORT", "29531"), os.path.abspath(__file__), "--gpus", str(args.gpus),
			   "--steps", str(args.steps), "--warmup", str(args.warmup), "--cubes", str(args.cubes)]
		if args.dump_outputs:
			cmd += ["--dump-outputs", os.path.abspath(args.dump_outputs)]
		sys.exit(subprocess.call(cmd))
	run_gpu(args)


if __name__ == "__main__":
	main()
