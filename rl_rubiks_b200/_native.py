"""ctypes binding of librubiks_b200.so (C ABI: include/rubiks_b200.h).

The product path has no CPU fallback: importing this module without the built library, or calling into it
without a CUDA device, raises."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RB_LIB_PATH") or os.path.join(_HERE, "librubiks_b200.so")      # RB_LIB_PATH: kernel experiments (tools/)

RB_OK, RB_ERR_BAD_ARG, RB_ERR_CUDA, RB_ERR_RANGE, RB_ERR_CAPACITY = 0, 1, 2, 3, 4
REP_2024, REP_686 = 0, 1
REWARD_METHODS = {"paper": 0, "lapanfix": 1, "schultzfix": 2, "reward0": 3}

if not os.path.exists(LIB_PATH):
	raise ImportError(
		f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
		"(nvcc, sm_100a).  rl_rubiks_b200 has no CPU fallback.")

lib = C.CDLL(LIB_PATH)

_p, _i32, _i64, _f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_double

# name -> (restype, argtypes); mirrors include/rubiks_b200.h one to one
SIGNATURES = {
	"rb_version": (C.c_int, []),
	"rb_last_error": (C.c_char_p, []),
	"rb_launch_count": (_i64, []),
	"rb_get_delta_maps": (C.c_int, [_p]),
	"rb_get_lut2024": (C.c_int, [_p]),
	"rb_get_perm686": (C.c_int, [_p]),
	"rb_get_macro_table": (C.c_int, [_p]),
	"rb_get_macro3_table": (C.c_int, [_p]),
	"rb_get_macro3_dedup": (C.c_int, [_p, _p]),
	"rb_get_stickers686": (C.c_int, [_p, _p, _p, _p]),
	"rb_get_solved": (C.c_int, [C.c_int, _p]),
	"rb_multi_rotate": (C.c_int, [C.c_int, _p, _p, _p, _p, _i64, _p]),
	"rb_multi_is_solved": (C.c_int, [C.c_int, _p, _p, _i64, _p]),
	"rb_as_oh": (C.c_int, [C.c_int, _p, _p, _i64, _p]),
	"rb_as_correct_686": (C.c_int, [_p, _p, _i64, _p]),
	"rb_expand12": (C.c_int, [C.c_int, _p, _p, _p, _p, _i64, _p]),
	"rb_check_range": (C.c_int, [C.c_int, _p, _i64, _p, _p, _i64, _p, _p]),
	"rb_scramble": (C.c_int, [C.c_int, _p, _i64, _i64, _p, _p, _i64, _i32, _p]),
	"rb_sequence_scramble": (C.c_int, [C.c_int, _p, _p, _i32, _i32, _i32, _p, _p, _p, _p]),
	"rb_adi_generate": (C.c_int, [C.c_int, _p, _p, _i32, _i32, _i32, _p, _p, _p, _p, _p, _p, _p]),
	"rb_as_oh_bf16": (C.c_int, [C.c_int, _p, _p, _i64, _p]),
	"rb_expand12_bf16": (C.c_int, [C.c_int, _p, _p, _p, _p, _i64, _p]),
	"rb_sequence_scramble_bf16": (C.c_int, [C.c_int, _p, _p, _i32, _i32, _i32, _p, _p, _p, _p]),
	"rb_adi_generate_bf16": (C.c_int, [C.c_int, _p, _p, _i32, _i32, _i32, _p, _p, _p, _p, _p, _p, _p]),
	"rb_adi_targets": (C.c_int, [_p, _p, _p, _i64, _i32, _i32, _p, _p, _p]),
	"rb_adi_targets_weights": (C.c_int, [_p, _p, _p, _i32, _i32, _i32, _f64, _f64, _p, _p, _p, _p]),
	"rb_adi_weight_sum": (_f64, [_i32, _i32]),
	"rb_adi_loss_weights": (C.c_int, [_p, _i32, _i32, _f64, _f64, _p]),
	"rb_hashset_bytes": (_i64, [_i64]),
	"rb_hashset_clear": (C.c_int, [_p, _i64, _p]),
	"rb_hashset_rehash": (C.c_int, [_p, _i64, _p, _i64, _p]),
	"rb_hashset_scratch_bytes": (_i64, [_i64]),
	"rb_hashset_insert_unique": (C.c_int, [C.c_int, _p, _i64, _p, _i64, _p, _p, _p, _p, _p, _p]),
	"rb_hashset_lookup": (C.c_int, [C.c_int, _p, _i64, _p, _i64, _p, _p, _p]),
	"rb_frontier_expand": (C.c_int, [C.c_int, _p, _i64, _p, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
	"rb_frontier_expand_dev": (C.c_int, [C.c_int, _p, _i64, _p, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
	"rb_frontier_expand_chain": (C.c_int, [C.c_int, _p, _i64, _p, _p, _i64, _i32, _p, _p, _p, _p]),
	"rb_frontier_scratch_bytes": (_i64, [C.c_int, _i64]),
	"rb_astar_scratch_bytes": (_i64, [_i32, _i32]),
	"rb_astar_init": (C.c_int, [_p, _p, _p]),
	"rb_astar_expand": (C.c_int, [_p, _i64, _p, _p, _p, _p, _p, _p]),
	"rb_astar_commit": (C.c_int, [_p, _p, _f64, _p, _p, _p, _p]),
	"rb_bfs_scratch_bytes": (_i64, [_i32, _i32]),
	"rb_bfs_init": (C.c_int, [_p, _p, _p]),
	"rb_bfs_step": (C.c_int, [_p, _i64, _p, _p]),
	"rb_bfs_paths": (C.c_int, [_p, _p, _p, _i32, _p]),
	"rb_mcts_scratch_bytes": (_i64, [_i32]),
	"rb_mcts_init": (C.c_int, [_p, _p, _p]),
	"rb_mcts_expand": (C.c_int, [_p, _p, _p, _p, _p, _p]),
	"rb_mcts_commit": (C.c_int, [_p, _p, _p, _p, _p, _p, _f64, _i64, _p, _p, _p]),
	"rb_mcts_finish": (C.c_int, [_p, _i32, _p, _p, _i32, _p]),
	"rb_as686": (C.c_int, [_p, _p, _i64, _p]),
	"rb_as2024": (C.c_int, [_p, _p, _p, _i64, _p]),
	"rb_scramble_seeded": (C.c_int, [C.c_int, C.c_uint64, C.c_uint64, _p, _p, _i64, _i32, _p]),
	"rb_seeded_actions": (C.c_int, [C.c_uint64, C.c_uint64, _p, _i64, _i32, _p]),
	"rb_unpack_actions": (C.c_int, [_p, _p, _i64, _i32, _p]),
	"rbh_scramble": (C.c_int, [C.c_int, _p, _p, _i64, _i32]),
	"rbh_scramble_packed": (C.c_int, [C.c_int, _p, _p, _i64, _i32]),
	"rbh_scramble_seeded": (C.c_int, [C.c_int, C.c_uint64, C.c_uint64, _p, _i64, _i32]),
	"rbh_multi_rotate": (C.c_int, [C.c_int, _p, _p, _p, _p, _i64]),
	"rbh_host_alloc": (_p, [_i64, C.c_int]),
	"rbh_host_free": (C.c_int, [_p, _i64]),
	"rbh_release": (C.c_int, []),
}

for _name, (_res, _args) in SIGNATURES.items():
	_fn = getattr(lib, _name)          # AttributeError here = the .so does not match the header
	_fn.restype, _fn.argtypes = _res, _args


class AStarView(C.Structure):
	"""rb_astar_view (include/rubiks_b200.h)."""
	_fields_ = [("K", _i32), ("M", _i32), ("N", _i32), ("states", _p), ("G", _p), ("parents", _p), ("parent_actions", _p),
				("cost", _p), ("in_open", _p), ("count", _p), ("n_sel", _p), ("sel", _p), ("won", _p), ("solved_index", _p),
				("table", _p), ("capacity", _i64), ("scratch", _p)]


class BFSView(C.Structure):
	"""rb_bfs_view (include/rubiks_b200.h)."""
	_fields_ = [("K", _i32), ("M", _i32), ("N", _i32), ("states", _p), ("parents", _p), ("parent_actions", _p), ("count", _p),
				("head", _p), ("won", _p), ("done", _p), ("solved_parent", _p), ("solved_action", _p), ("table", _p),
				("capacity", _i64), ("scratch", _p)]


class MCTSView(C.Structure):
	"""rb_mcts_view (include/rubiks_b200.h)."""
	_fields_ = [("K", _i32), ("M", _i32), ("max_path", _i32), ("states", _p), ("parents", _p), ("parent_actions", _p), ("neighbors", _p),
				("leaves", _p), ("P", _p), ("V", _p), ("N", _p), ("W", _p), ("L", _p), ("count", _p), ("won", _p), ("solved_index", _p),
				("path_node", _p), ("path_action", _p), ("path_len", _p), ("order", _p), ("table", _p), ("capacity", _i64), ("scratch", _p)]


class RubiksError(RuntimeError):
	pass


def check(rc: int):
	"""Maps the C status to the exceptions the reference would raise (SURVEY 8b, Errors)."""
	if rc == RB_OK:
		return
	msg = lib.rb_last_error().decode()
	if rc == RB_ERR_RANGE:
		raise IndexError(msg)
	raise RubiksError(f"librubiks_b200 error {rc}: {msg}")


def ptr(t):
	"""Device (or pinned host) address of a torch tensor, or None."""
	return None if t is None else C.c_void_p(t.data_ptr())


def stream_handle():
	import torch
	return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda():
	import torch
	if not torch.cuda.is_available():
		raise RubiksError("rl_rubiks_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
