"""The seen-set (csrc/rb_frontier.cuh) on crafted probe chains, read back slot by slot.

Random states in a table kept at load <= 1/2 give probe chains of a few slots, so the long walks of `find_or_claim` and
`find_only` run only by chance elsewhere in the suite.  Here the hash is ported to numpy and pinned against the device; with it
states are chosen by their home slot to build what the table must survive: one home slot shared by hundreds of states, a
chain that wraps from slot C-1 to slot 0, a table exactly full, one slot raced for by 64k items, a frontier expanded into a
crowded table, and the A* table shared by up to 65535 searches.  Every result is compared with the dict oracle and every
table is dumped and checked for the invariants of a settled table (`check_table`)."""
import numpy as np
import pytest
import torch

from oracle import cube_oracle as O

pytestmark = pytest.mark.gpu

REPS = [pytest.param(True, id="2024"), pytest.param(False, id="686")]
GiB = 1 << 30
EMPTY = np.uint64(0xFFFFFFFFFFFFFFFF)
IDLE = np.uint32(0xFFFFFFFF)
SLOT = np.dtype([("lo", "<u8"), ("hi", "<u8"), ("val", "<i4"), ("firstpos", "<u4"), ("spare", "<u8")])     # rbf::Slot, 32 B
POOL_N, POOL_DEPTH, POOL_SEED = 1 << 19, 40, 20261020


@pytest.fixture(autouse=True)
def _guard():
	from rl_rubiks_b200 import cube
	cube.set_is2024(True)
	torch.cuda.empty_cache()
	torch.cuda.reset_peak_memory_stats()
	yield
	cube.set_is2024(True)
	print(f"peak device memory {torch.cuda.max_memory_allocated() / GiB:.2f} GiB")


# ---- numpy port of the key packing and the hash --------------------------------------------------------------------------
def key2024(states):
	"""pack2024: cubie j (5 bits) at bit 5j, cubies 0-11 in lo, 12-19 in hi."""
	s = np.asarray(states).reshape(-1, 20).astype(np.uint64)
	sh = np.arange(12, dtype=np.uint64) * np.uint64(5)
	lo = np.bitwise_or.reduce(s[:, :12] << sh, axis=1)
	hi = np.bitwise_or.reduce(s[:, 12:] << sh[:8], axis=1)
	return lo, hi


def key686(states):
	"""k_pack686: face f -> sum_j c_j 6^j over its 8 sticker colours; faces 0-2 in lo, 3-5 in hi, 21 bits apart."""
	c = np.asarray(states).reshape(-1, 6, 8, 6).argmax(axis=3).astype(np.uint64)
	face = (c * (np.uint64(6) ** np.arange(8, dtype=np.uint64))).sum(axis=2)
	sh = np.arange(3, dtype=np.uint64) * np.uint64(21)
	return np.bitwise_or.reduce(face[:, :3] << sh, axis=1), np.bitwise_or.reduce(face[:, 3:] << sh, axis=1)


def keys(states, is2024):
	return key2024(states) if is2024 else key686(states)


def astar_key(states, search):
	"""rbl::key (k_probe, root init): the search id in bits 40-55 of the 20x24 key's high word."""
	lo, hi = key2024(states)
	return lo, hi | (np.asarray(search, dtype=np.uint64) << np.uint64(40))


def hash_key(lo, hi):
	"""rbf::hash_key in uint64 arithmetic (wraps like the device's)."""
	lo, hi = np.asarray(lo, np.uint64), np.asarray(hi, np.uint64)
	with np.errstate(over="ignore"):
		h = (lo * np.uint64(0x9E3779B97F4A7C15)) ^ ((hi + np.uint64(0x7F4A7C15)) * np.uint64(0xC2B2AE3D27D4EB4F))
		h ^= h >> np.uint64(32)
		h *= np.uint64(0xD6E8FEB86659FD93)
		h ^= h >> np.uint64(29)
	return h


def home(lo, hi, C):
	return (hash_key(lo, hi) & np.uint64(C - 1)).astype(np.int64)


# ---- candidates: distinct reachable states, picked by home slot --------------------------------------------------------
_POOLS = {}


def pool(is2024):
	"""2^19 seeded 40-move scrambles (the same cubes in both representations), deduplicated, with their keys and hashes."""
	if is2024 not in _POOLS:
		from rl_rubiks_b200 import cube
		cube.set_is2024(is2024)
		try:
			st = cube.scramble_seeded(POOL_N, POOL_DEPTH, POOL_SEED).cpu().numpy()
		finally:
			cube.set_is2024(True)
		lo, hi = keys(st, is2024)
		_, first = np.unique(np.stack([lo, hi], 1), axis=0, return_index=True)
		first.sort()
		_POOLS[is2024] = {"states": st[first], "lo": lo[first], "hi": hi[first], "hash": hash_key(lo[first], hi[first])}
	return _POOLS[is2024]


class Picker:
	"""Hands out pool states by home slot at capacity C, each state at most once."""

	def __init__(self, is2024, C):
		self.p, self.C = pool(is2024), C
		self.home = (self.p["hash"] & np.uint64(C - 1)).astype(np.int64)
		self.used = np.zeros(len(self.home), bool)
		self.order = np.argsort(self.home, kind="stable")
		self.start = np.searchsorted(self.home[self.order], np.arange(C + 1))

	def at(self, slot, k):
		cand = self.order[self.start[slot]:self.start[slot + 1]]
		idx = cand[~self.used[cand]][:k]
		assert len(idx) == k, f"pool has {len(idx)} unused states homed at {slot}, {k} wanted"
		self.used[idx] = True
		return self.p["states"][idx]

	def any(self, k):
		idx = np.nonzero(~self.used)[0][:k]
		self.used[idx] = True
		return self.p["states"][idx]

	def fullest(self):
		return int(np.bincount(self.home, minlength=self.C).argmax())


# ---- a table at a fixed capacity, through the C ABI (the Python mirror would grow it) ----------------------------------
class Table:
	def __init__(self, C, is2024, count=None):
		from rl_rubiks_b200 import _native as N
		self.N, self.C, self.is2024 = N, C, is2024
		self.rep = N.REP_2024 if is2024 else N.REP_686
		self.shape = (20,) if is2024 else (6, 8, 6)
		self.t = torch.empty(N.lib.rb_hashset_bytes(C), dtype=torch.uint8, device="cuda")
		self.count = torch.zeros(1, dtype=torch.int32, device="cuda") if count is None else count.clone()
		N.check(N.lib.rb_hashset_clear(N.ptr(self.t), C, N.stream_handle()))

	def _dev(self, states):
		return torch.from_numpy(np.ascontiguousarray(states, dtype=np.int8).reshape(-1, *self.shape)).cuda()

	def insert(self, states):
		"""rb_hashset_insert_unique with every per-item output: (seen, first, index) as numpy."""
		N, s = self.N, self._dev(states)
		n = s.shape[0]
		seen, first = (torch.full((n,), 7, dtype=torch.uint8, device="cuda") for _ in range(2))
		index = torch.full((n,), -7, dtype=torch.int32, device="cuda")
		scratch = torch.empty(N.lib.rb_hashset_scratch_bytes(n), dtype=torch.uint8, device="cuda")
		N.check(N.lib.rb_hashset_insert_unique(self.rep, N.ptr(self.t), self.C, N.ptr(s), n, N.ptr(self.count), N.ptr(seen), N.ptr(first),
											   N.ptr(index), N.ptr(scratch), N.stream_handle()))
		return seen.cpu().numpy(), first.cpu().numpy(), index.cpu().numpy()

	def lookup(self, states):
		N, s = self.N, self._dev(states)
		n = s.shape[0]
		index = torch.full((n,), -7, dtype=torch.int32, device="cuda")
		scratch = torch.empty(N.lib.rb_hashset_scratch_bytes(n), dtype=torch.uint8, device="cuda")
		N.check(N.lib.rb_hashset_lookup(self.rep, N.ptr(self.t), self.C, N.ptr(s), n, N.ptr(index), N.ptr(scratch), N.stream_handle()))
		return index.cpu().numpy()

	def rehash(self, C2):
		dst = Table(C2, self.is2024, self.count)
		self.N.check(self.N.lib.rb_hashset_rehash(self.N.ptr(self.t), self.C, self.N.ptr(dst.t), C2, self.N.stream_handle()))
		return dst

	def expand(self, frontier):
		"""rb_frontier_expand with every output, as numpy."""
		N, f = self.N, self._dev(frontier)
		m = 12 * f.shape[0]
		out = {"next": torch.empty(m, *self.shape, dtype=torch.int8, device="cuda"), "parent": torch.empty(m, dtype=torch.int32, device="cuda"),
			   "action": torch.empty(m, dtype=torch.uint8, device="cuda"), "solved": torch.empty(m, dtype=torch.uint8, device="cuda"),
			   "seen": torch.empty(m, dtype=torch.uint8, device="cuda"), "first": torch.empty(m, dtype=torch.uint8, device="cuda"),
			   "index": torch.empty(m, dtype=torch.int32, device="cuda"), "n_new": torch.empty(1, dtype=torch.int32, device="cuda")}
		scratch = torch.empty(N.lib.rb_frontier_scratch_bytes(self.rep, f.shape[0]), dtype=torch.uint8, device="cuda")
		N.check(N.lib.rb_frontier_expand(self.rep, N.ptr(self.t), self.C, N.ptr(f), f.shape[0], N.ptr(self.count), *(N.ptr(out[k]) for k in (
			"next", "parent", "action", "solved", "seen", "first", "index", "n_new")), N.ptr(scratch), N.stream_handle()))
		return {k: v.cpu().numpy() for k, v in out.items()}

	def size(self):
		return int(self.count.item())

	def dump(self):
		return self.t.cpu().numpy().view(SLOT)


# ---- invariants of a settled table -------------------------------------------------------------------------------------
def check_table(tab, lo, hi, val, count):
	"""`tab` (a dump) holds exactly the keys (lo, hi) with indices `val`, `count` of them, and is what a correct sequence of
	batches leaves behind: keys unique, every firstpos idle, empty slots untouched, and every key reachable by linear probing
	from its home slot (no empty slot between home and key, cyclically)."""
	C = len(tab)
	occ = ~((tab["lo"] == EMPTY) & (tab["hi"] == EMPTY))
	assert int(occ.sum()) == count == len(lo), (int(occ.sum()), count, len(lo))
	olo, ohi, oval = tab["lo"][occ], tab["hi"][occ], tab["val"][occ]
	o = np.lexsort((olo, ohi))
	dup = (olo[o][1:] == olo[o][:-1]) & (ohi[o][1:] == ohi[o][:-1])
	assert not dup.any(), f"{int(dup.sum())} keys stored twice"
	e = np.lexsort((lo, hi))
	assert (olo[o] == lo[e]).all() and (ohi[o] == hi[e]).all(), "stored keys differ from the oracle's states"
	bad = oval[o] != np.asarray(val)[e]
	assert not bad.any(), f"{int(bad.sum())} slots carry another index than the oracle's"
	assert (tab["firstpos"] == IDLE).all(), f"{int((tab['firstpos'] != IDLE).sum())} slots keep a firstpos"
	assert (tab["val"][~occ] == 0).all() and (tab["spare"][~occ] == 0).all(), "an empty slot was written"
	slots = np.nonzero(occ)[0]
	h = home(olo, ohi, C)
	d = (slots - h) % C
	cs = np.concatenate([[0], np.cumsum(np.concatenate([occ, occ]))])
	broken = cs[h + d] - cs[h] != d
	assert not broken.any(), f"{int(broken.sum())} keys sit behind an empty slot of their probe chain"


def check_against(tbl, ref):
	"""check_table against the dict oracle, whose indices must be 1..len."""
	shape = tbl.shape
	st = np.frombuffer(b"".join(ref.index.keys()), np.int8).reshape(-1, *shape) if len(ref) else np.zeros((0, *shape), np.int8)
	val = np.fromiter(ref.index.values(), np.int64, len(ref))
	assert (np.sort(val) == np.arange(1, len(ref) + 1)).all()
	lo, hi = keys(st, tbl.is2024)
	check_table(tbl.dump(), lo, hi, val, tbl.size())


def insert_both(tbl, ref, states):
	seen, first, idx = tbl.insert(states)
	w_seen, w_first, w_idx = ref.insert_unique(states)
	assert (seen == w_seen).all() and (first == w_first).all() and (idx == w_idx).all()
	assert tbl.size() == len(ref)
	check_against(tbl, ref)
	return seen, first, idx


def shuffled(rng, *parts):
	a = np.concatenate(parts)
	return a[rng.permutation(len(a))]


def check_rehashes(tbl, ref):
	"""Rehash into the same, twice and four times the capacity: indices kept, invariants hold, the source untouched."""
	before = tbl.dump().copy()
	every = np.frombuffer(b"".join(ref.index.keys()), np.int8).reshape(-1, *tbl.shape)
	for f in (1, 2, 4):
		dst = tbl.rehash(f * tbl.C)
		assert dst.size() == len(ref)
		check_against(dst, ref)
		assert (dst.lookup(every) == ref.lookup(every)).all()
	assert (tbl.dump().view(np.uint8) == before.view(np.uint8)).all()


# ---- 1. the port ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("is2024", REPS)
def test_key_and_hash_port_matches_device(is2024):
	"""3000 states with pairwise different home slots in a sparse table: each sits in its home slot with its batch index."""
	C = 1 << 16
	p = pool(is2024)
	h = home(p["lo"], p["hi"], C)
	_, one = np.unique(h, return_index=True)
	pick = np.sort(one)[:3000]
	tbl = Table(C, is2024)
	seen, first, idx = tbl.insert(p["states"][pick])
	assert not seen.any() and first.all() and (idx == np.arange(1, 3001)).all()
	tab = tbl.dump()
	slot = tab[h[pick]]
	assert (slot["lo"] == p["lo"][pick]).all() and (slot["hi"] == p["hi"][pick]).all()
	assert (slot["val"] == np.arange(1, 3001)).all()
	check_table(tab, p["lo"][pick], p["hi"][pick], np.arange(1, 3001), tbl.size())


# ---- 2. crafted chains ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("is2024", REPS)
def test_cluster_on_one_home_slot(is2024):
	"""320 states share one home slot at C = 1024 (a 320-slot walk for the last of them), each inserted 4x in one shuffled
	batch; then seen cluster states (3x each) mixed with new cluster states and states homed just behind the cluster."""
	C, rng = 1024, np.random.RandomState(1)
	pk = Picker(is2024, C)
	h0 = pk.fullest()
	cluster, fresh, absent = pk.at(h0, 320), pk.at(h0, 40), pk.at(h0, 40)
	behind = np.concatenate([pk.at((h0 + k) % C, 2) for k in range(1, 40, 3)])
	tbl, ref = Table(C, is2024), O.SeenSet()
	insert_both(tbl, ref, shuffled(rng, *[cluster] * 4))
	seen_part = cluster[rng.permutation(320)[:100]]
	insert_both(tbl, ref, shuffled(rng, seen_part, seen_part, seen_part, fresh, fresh, behind))
	# absent: homed inside the cluster (at its home and along it), never inserted -- a scan down the whole chain
	inside = np.concatenate([pk.at((h0 + k) % C, 1) for k in range(0, 400, 7)])
	probe = np.concatenate([absent, inside])
	assert (tbl.lookup(probe) == 0).all()
	every = np.concatenate([cluster, fresh, behind])
	assert (tbl.lookup(every) == ref.lookup(every)).all()
	check_rehashes(tbl, ref)


@pytest.mark.parametrize("is2024", REPS)
def test_chain_wraps_from_last_slot_to_slot_zero(is2024):
	"""12 states homed at each of the last 8 slots run past slot C-1 into slots 0, 1, ...; states homed at slots 0-3 queue
	behind the wrapped chain."""
	C, rng = 1024, np.random.RandomState(2)
	pk = Picker(is2024, C)
	tail = np.concatenate([pk.at(C - 8 + k, 12) for k in range(8)])
	head = np.concatenate([pk.at(k, 6) for k in range(4)])
	absent = np.concatenate([pk.at(s, 3) for s in list(range(C - 8, C)) + [0, 1, 2, 3]])
	tbl, ref = Table(C, is2024), O.SeenSet()
	insert_both(tbl, ref, shuffled(rng, tail, tail))
	insert_both(tbl, ref, shuffled(rng, head, head, tail[::5]))
	tab = tbl.dump()
	occ = ~((tab["lo"] == EMPTY) & (tab["hi"] == EMPTY))
	h = home(tab["lo"], tab["hi"], C)
	# 96 keys from slot C-8 on fill slots C-8 .. 87 whatever the order they came in; the 24 homed at 0-3 then fill 88 .. 111
	assert occ[C - 8:].all() and occ[:112].all() and not occ[112:C - 8].any()
	assert (h[:88] >= C - 8).all() and (h[88:112] < 4).all()
	assert (tbl.lookup(absent) == 0).all()
	every = np.concatenate([tail, head])
	assert (tbl.lookup(every) == ref.lookup(every)).all()
	check_rehashes(tbl, ref)


@pytest.mark.parametrize("C", [64, 1024])
@pytest.mark.parametrize("is2024", REPS)
def test_exactly_full_table(is2024, C):
	"""C - 1 distinct states over three batches with duplicates succeed; the C-th, homed just past the last empty slot, walks
	all C slots to it; then C absent lookups each scan the whole table and return 0, the table is rehashed, and one more
	distinct state overflows: count -1 and index -1, sticky, with the table unchanged."""
	rng = np.random.RandomState(C)
	pk = Picker(is2024, C)
	states = pk.any(C - 1)
	tbl, ref = Table(C, is2024), O.SeenSet()
	parts = np.array_split(np.arange(C - 1), 3)
	for b, part in enumerate(parts):
		old = states[np.concatenate(parts[:b])] if b else states[:0]
		old = old[rng.permutation(len(old))[:C // 8]]
		insert_both(tbl, ref, shuffled(rng, states[part], states[part], old))
	assert tbl.size() == C - 1
	tab = tbl.dump()
	empty = np.nonzero((tab["lo"] == EMPTY) & (tab["hi"] == EMPTY))[0]
	assert len(empty) == 1
	last = pk.at((int(empty[0]) + 1) % C, 1)                            # its probe reaches the empty slot on the C-th try
	seen, first, idx = insert_both(tbl, ref, shuffled(rng, last, last, states[:5]))
	assert tbl.size() == C and (idx >= 1).all()
	assert tbl.lookup(last)[0] == C
	absent = pk.any(C)
	assert (tbl.lookup(absent) == 0).all()
	check_rehashes(tbl, ref)
	before = tbl.dump().copy()
	one = pk.any(1)
	seen, first, idx = tbl.insert(np.concatenate([one, states[:3]]))
	assert tbl.size() == -1 and idx[0] == -1 and not seen[0]
	assert (idx[1:] == ref.lookup(states[:3])).all()
	tbl.insert(states[3:6])
	assert tbl.size() == -1
	assert (tbl.dump().view(np.uint8) == before.view(np.uint8)).all()


@pytest.mark.parametrize("is2024", REPS)
def test_one_home_slot_contention_is_deterministic(is2024):
	"""65536 items drawn from 8 states that share one home slot: every item races for the same slot and then the same
	7-slot chain.  Dict semantics, and the same arrays on each of 3 fresh tables."""
	C, rng = 1024, np.random.RandomState(3)
	pk = Picker(is2024, C)
	eight = pk.at(pk.fullest(), 8)
	batch = eight[rng.randint(0, 8, 1 << 16)]
	runs = []
	for _ in range(3):
		tbl, ref = Table(C, is2024), O.SeenSet()
		runs.append(insert_both(tbl, ref, batch))
		seen, first, idx = insert_both(tbl, ref, batch[::-1])
		assert seen.all() and (idx == runs[-1][2][::-1]).all()
	for r in runs[1:]:
		assert all((a == b).all() for a, b in zip(r, runs[0]))


@pytest.mark.parametrize("is2024", REPS)
def test_frontier_expand_on_crowded_table(is2024):
	"""rb_frontier_expand (and, 20x24, rb_frontier_expand_chain) two layers deep into a table pre-filled with two states on
	every home slot the children will probe (load ~0.5, every child walks past fillers)."""
	from rl_rubiks_b200 import _native as N
	C, rng = 1 << 14, np.random.RandomState(4)
	g = np.random.RandomState(5)
	start = O.scramble_many(g.randint(0, 6, (24, 3)), g.randint(0, 2, (24, 3)), is2024)
	sim = O.SeenSet()
	_, first, _ = sim.insert_unique(start)
	frontier0 = start[first]
	frontiers, children = [frontier0], []
	for _ in range(2):
		ch = O.expand12(frontiers[-1], is2024)
		seen, first, _ = sim.insert_unique(ch)
		children.append(ch)
		frontiers.append(ch[first & ~seen])
	clo, chi = keys(np.concatenate(children), is2024)
	pk = Picker(is2024, C)
	fill = np.concatenate([pk.at(s, 2) for s in np.unique(home(clo, chi, C))])
	flo, fhi = keys(fill, is2024)
	assert not set(zip(flo.tolist(), fhi.tolist())) & set(zip(clo.tolist(), chi.tolist()))

	tbl, ref = Table(C, is2024), O.SeenSet()
	insert_both(tbl, ref, shuffled(rng, fill))
	insert_both(tbl, ref, frontier0)
	frontier = frontier0
	sizes = []
	for _ in range(2):
		out = tbl.expand(frontier)
		ch = O.expand12(frontier, is2024)
		seen, first, idx = ref.insert_unique(ch)
		new = first & ~seen
		n_new = int(out["n_new"][0])
		assert n_new == new.sum() and tbl.size() == len(ref)
		assert (out["next"][:n_new] == ch[new]).all()
		assert (out["parent"][:n_new] == np.repeat(np.arange(len(frontier)), 12)[new]).all()
		assert (out["action"][:n_new] == np.tile(np.arange(12), len(frontier))[new]).all()
		assert (out["solved"][:n_new].astype(bool) == O.multi_is_solved(ch[new], is2024)).all()
		assert (out["seen"].astype(bool) == seen).all() and (out["first"].astype(bool) == first).all() and (out["index"] == idx).all()
		check_against(tbl, ref)
		frontier = ch[new]
		sizes.append(n_new)
	if not is2024:
		return
	# the same two layers chained on the device (sizes never leave it) into an identically pre-filled table
	chain, ref2 = Table(C, True), O.SeenSet()
	insert_both(chain, ref2, shuffled(np.random.RandomState(4), fill))
	insert_both(chain, ref2, frontier0)
	n0 = len(frontier0)
	bufs = [torch.zeros(n0 * 144, 20, dtype=torch.int8, device="cuda") for _ in range(2)]
	bufs[0][:n0] = torch.from_numpy(frontier0).cuda()
	layer_sizes = torch.zeros(3, dtype=torch.int32, device="cuda")
	layer_sizes[0] = n0
	scratch = torch.empty(N.lib.rb_frontier_scratch_bytes(N.REP_2024, 12 * n0), dtype=torch.uint8, device="cuda")
	N.check(N.lib.rb_frontier_expand_chain(N.REP_2024, N.ptr(chain.t), C, N.ptr(bufs[0]), N.ptr(bufs[1]), n0, 2, N.ptr(layer_sizes),
										   N.ptr(chain.count), N.ptr(scratch), N.stream_handle()))
	assert layer_sizes[1:].tolist() == sizes and chain.size() == len(ref)
	assert (bufs[0][:sizes[1]].cpu().numpy() == frontier).all()
	every = np.concatenate([fill, frontier0, *children])
	assert (chain.lookup(every) == ref.lookup(every)).all()
	check_against(chain, ref)


# ---- 3. A*: K searches on one table --------------------------------------------------------------------------------------
class _IntNet(torch.nn.Module):
	"""floor(one-hot @ w / 4) with integer w: exact values that do not depend on a row's position in the batch."""

	def __init__(self, w):
		super().__init__()
		self.w = torch.from_numpy(np.asarray(w, np.float32)).cuda()

	def forward(self, x, policy=True, value=True):
		return torch.floor((x @ self.w) / 4.0).unsqueeze(1)


ASTAR_W = np.random.RandomState(13).randint(-3, 4, 480)
ASTAR_LAMBDA = 0.16


def astar_pool():
	"""A cube r and its 12 neighbours: roots that differ but share most of their nearby states."""
	g = np.random.RandomState(12)
	r = O.scramble(g.randint(0, 6, 9), g.randint(0, 2, 9), True)
	return np.concatenate([r[None], O.expand12(r[None], True)])


def root_ids(K):
	"""Search s starts from pool cube (s * 0x9E3779B1 >> 11) % 13: searches whose ids differ in high bits only start apart."""
	return ((np.arange(K, dtype=np.uint64) * np.uint64(0x9E3779B1)) >> np.uint64(11)).astype(np.int64) % 13


_HARNESS = {}


def harness_trace(j, n_exp, max_states):
	"""tests.agent_harness.AStar (the reference's single search) from pool cube j: won, queue, len, states, G, parents."""
	if (j, n_exp, max_states) not in _HARNESS:
		from tests.agent_harness import AStar
		a = AStar(_IntNet(ASTAR_W), lambda_=ASTAR_LAMBDA, expansions=n_exp, is2024=True)
		ok = a.search(astar_pool()[j], None, max_states)
		L = len(a)
		_HARNESS[(j, n_exp, max_states)] = (ok, list(a.action_queue), L, a.states[1:L + 1].cpu().numpy(), a.G[1:L + 1].copy(),
											a.parents[2:L + 1].copy(), a.parent_actions[2:L + 1].copy())
	return _HARNESS[(j, n_exp, max_states)]


@pytest.mark.parametrize("K,n_exp,max_states", [pytest.param(13, 4, 600, id="K13"), pytest.param(300, 4, 600, id="K300"),
												pytest.param(65535, 1, 100, id="K65535")])
def test_astar_searches_share_one_table(K, n_exp, max_states):
	"""K searches from the 13-cube pool: each follows the harness's trace from its root, and the shared table holds, per
	search id, exactly that search's states numbered 1..count with the id in bits 40-55 of the key.  K = 65535 is the
	gridDim.y limit and uses every search-id bit."""
	from rl_rubiks_b200.frontier import AStarBatch
	pool13, ids = astar_pool(), root_ids(K)
	if K > 256:
		assert (ids[256:] != ids[:K - 256]).any()                          # ids equal in their low 8 bits start apart
	agent = AStarBatch(_IntNet(ASTAR_W), lambda_=ASTAR_LAMBDA, expansions=n_exp, is2024=True)
	won, queues, count = agent.search_many(pool13[ids], max_states)
	for j in range(13):
		ok, q, L, st, G, par, pact = harness_trace(j, n_exp, max_states)
		S = np.nonzero(ids == j)[0]
		if not len(S):
			continue
		Sd = torch.from_numpy(S).cuda()
		assert (won[S] == ok).all() and (count[S] == L).all(), j
		assert all(queues[s] == q for s in S), j
		assert (agent.states.index_select(0, Sd)[:, 1:L + 1].cpu().numpy() == st).all(), j
		assert (agent.G.index_select(0, Sd)[:, 1:L + 1].cpu().numpy() == G).all(), j
		assert (agent.parents.index_select(0, Sd)[:, 2:L + 1].cpu().numpy() == par).all(), j
		assert (agent.parent_actions.index_select(0, Sd)[:, 2:L + 1].cpu().numpy() == pact).all(), j
	# the table: every search's states, keyed with its id, numbered 1..count[s]
	tab = agent.table.cpu().numpy().view(SLOT)
	L_max = int(count.max())
	states = agent.states[:, 1:L_max + 1].cpu().numpy()
	sid = np.repeat(np.arange(K), L_max)
	row = np.tile(np.arange(1, L_max + 1), K)
	live = row <= count[sid]
	lo, hi = astar_key(states.reshape(-1, 20)[live], sid[live])
	check_table(tab, lo, hi, row[live], int(count.sum()))
	occ = ~((tab["lo"] == EMPTY) & (tab["hi"] == EMPTY))
	assert (np.bincount((tab["hi"][occ] >> np.uint64(40)).astype(np.int64), minlength=K) == count).all()
