// Fast multi-move scramble for the 20x24 representation (BASELINE configs[1]: 2^24 cubes x 100 moves).
//
// The byte-LUT kernel (rb2024::k_scramble) does 20 data-dependent shared-memory lookups per move and is bound by
// shared-memory bank conflicts at ~2 % of the HBM roofline (profiles/r1a_scramble_v1_ncu.txt).  The kernels here change the
// representation instead of the table: inside the kernel a cube is kept "slot-major" -- which cubie sits in each of
// the 8 corner / 12 edge positions -- so that a move is a FIXED byte permutation of registers (PRMT with a selector
// that depends only on the action) plus an additive orientation update:
//   corners: 8 bytes (C0,C1), byte = twist accumulator (bits 0-4, value mod 3 is the twist) | cubie id << 5
//   edges  : 12 bytes (E0,E1,E2), byte = cubie id (bits 0-3) | three partial flip bits (4-6) whose parity is the flip
// Permutation + additive orientation is closed under composition, so k consecutive moves are fused into one table row of
// five words: corner selectors, three edge selector words and one word carrying the 8 twist increments and 12 flip bits.
//
//   k_scramble_macro3 (the one that runs for depth <= 400): rows of THREE moves (12^3), the product taken backwards (inverse
//     moves, reverse order) so that the registers end up cubie-major -- see the comments at the kernel.  Up to depth 195 the
//     table is deduplicated to its 1080 distinct elements in 8 conflict-free copies (0.757 ms for 2^24 x 100 moves), for
//     longer sequences it is the 1728 rows in four copies of the 16-byte part (0.82 ms at depth 100).
//   k_scramble_macro (fallback for longer sequences): rows of TWO moves (13^2 with identity padding), the table replicated
//     so that every fetch is bank-conflict free (64 KB), forward product, scatter to cubie-major at the end.
//
// The corner twist t relates to the reference's orientation o (the axis the tracked sticker faces, maps.py:128)
// by t = o for positions {1,3,4,6} and t = -o mod 3 for positions {0,2,5,7} (the corner's chirality, the same split
// cube.py:292 uses); with that labelling every quarter turn adds a constant per slot.  rbs::host() derives all
// rows from the 20x24 LUT and verifies the additivity for every (action, position, orientation).
//
// Action tiles ([32 cubes][depth] bytes per warp, contiguous in HBM) are brought into shared memory with 1-D bulk
// async copies (cp.async.bulk, TMA engine, completion on the warp's mbarrier).
#pragma once
#include "rb_common.cuh"
#include "rb_tables.cuh"
#include <cuda.h>              // CUtensorMap (types only: the encoder is fetched through cudaGetDriverEntryPoint)
#include <array>
#include <map>

namespace rbs {

constexpr int kA = 13;                          // 12 actions + identity
constexpr int kRows = kA * kA;                  // 169
constexpr int kRowWords = 5;                    // s_corner, s_edge0, s_edge1, s_edge2, twists|flips
constexpr int kDevRows = 256;                   // actions are masked to 4 bits in the kernel (index <= 210); rows >= 169 are the identity
constexpr int kP1Bytes = kDevRows * 8 * 16;     // 16-byte part, 8 copies (one per bank group)
constexpr int kP2Bytes = kDevRows * 32 * 4;     // 4-byte part, 32 copies (one per bank)
constexpr int kTableBytes = kP1Bytes + kP2Bytes;        // 65,536
constexpr int kMaxThreads = 1024;               // 32 warps (CUDA limit per CTA)
constexpr int kSmemBudget = 227 * 1024;
constexpr int kReduceEvery = 10;                // rows between twist folds (5 action words): 10 + 10 * 2 <= 31

__device__ __align__(16) uint32_t g_macro[kRows * kRowWords + 3];
// The 3-move kernel applies INVERSE moves (a ^ 1); its two device tables are stored pre-permuted -- entry (a0, a1, a2) holds the
// row of (a0 ^ 1, a1 ^ 1, a2 ^ 1) -- so that the kernel indexes them with the raw action bytes (no XOR per action word).
__device__ __align__(16) uint32_t g_macro3[12 * 12 * 12 * kRowWords + 3];
__device__ __align__(16) uint32_t g_macro_tail_inv[13 * 13 * kRowWords + 3];

struct Elem {                                   // one cube-group element in slot-major gather form
	uint8_t csrc[8], ctw[8], esrc[12], efl[12];
};

static inline bool neg_chirality(int pos) { return pos == 0 || pos == 2 || pos == 5 || pos == 7; }
static inline int twist_of(int pos, int ori) { return neg_chirality(pos) ? (3 - ori) % 3 : ori; }

// Single move as a gather element, derived from the direct LUT (and checked for additivity).
static bool single(const rbt::Tables& t, int a, Elem& e) {
	for (int q = 0; q < 8; ++q) { e.csrc[q] = (uint8_t)q; e.ctw[q] = 0; }
	for (int q = 0; q < 12; ++q) { e.esrc[q] = (uint8_t)q; e.efl[q] = 0; }
	if (a == 12) return true;
	for (int p = 0; p < 8; ++p) {
		int delta = -1, dst = -1;
		for (int o = 0; o < 3; ++o) {
			const int v = t.lut[a][0][3 * p + o], p2 = v / 3, o2 = v % 3;
			const int d = (twist_of(p2, o2) - twist_of(p, o) + 3) % 3;
			if (o == 0) { delta = d; dst = p2; }
			else if (d != delta || p2 != dst) return false;
		}
		e.csrc[dst] = (uint8_t)p;
		e.ctw[dst] = (uint8_t)delta;
	}
	for (int p = 0; p < 12; ++p) {
		const int v0 = t.lut[a][1][2 * p], v1 = t.lut[a][1][2 * p + 1];
		if (v0 / 2 != v1 / 2 || ((v0 % 2) ^ 0) != ((v1 % 2) ^ 1)) return false;
		e.esrc[v0 / 2] = (uint8_t)p;
		e.efl[v0 / 2] = (uint8_t)(v0 % 2);
	}
	return true;
}

// r = "first x, then y"
static void compose(const Elem& x, const Elem& y, Elem& r) {
	for (int q = 0; q < 8; ++q) {
		r.csrc[q] = x.csrc[y.csrc[q]];
		r.ctw[q] = (uint8_t)((x.ctw[y.csrc[q]] + y.ctw[q]) % 3);
	}
	for (int q = 0; q < 12; ++q) {
		r.esrc[q] = x.esrc[y.esrc[q]];
		r.efl[q] = (uint8_t)(x.efl[y.esrc[q]] ^ y.efl[q]);
	}
}

// Register layout: C0 = corner slots 0-3 (byte i = slot i), C1 = slots 4-7; E0,E1,E2 = edge slots 0-3, 4-7, 8-11.
// Row word 4, byte i: bits 0-1 twist increment of corner slot i, bits 2-3 of slot 4+i, bits 4/5/6 flip of edge slot
// i / 4+i / 8+i.
static void encode(const Elem& e, uint32_t* row) {
	uint32_t sc = 0, tf = 0;
	for (int q = 0; q < 8; ++q) sc |= (uint32_t)e.csrc[q] << (4 * q);       // low 16: selector of C0', high 16: of C1'
	for (int i = 0; i < 4; ++i) tf |= ((uint32_t)e.ctw[i] | ((uint32_t)e.ctw[4 + i] << 2)) << (8 * i);
	row[0] = sc;
	for (int d = 0; d < 3; ++d) {
		uint32_t sa = 0, sb = 0;
		for (int i = 0; i < 4; ++i) {
			const int s = e.esrc[4 * d + i];
			sa |= (uint32_t)(s < 8 ? s : 0) << (4 * i);                     // x  = prmt(E0, E1, sa)
			sb |= (uint32_t)(s < 8 ? i : 4 + (s - 8)) << (4 * i);           // Ed' = prmt(x, E2, sb)
			tf |= (uint32_t)e.efl[4 * d + i] << (8 * i + 4 + d);            // Ed' ^= tf & (0x10101010 << d)
		}
		row[1 + d] = sa | (sb << 16);
	}
	row[4] = tf;
}

constexpr int kRows3 = 12 * 12 * 12;            // 3-move rows, index a0 + 12 a1 + 144 a2 (no identity padding: the tail uses the 2-move table)

// Deduplicated 3-move table (k_scramble_macro3 for depths up to 195, see launch()): a row is a function of the group element its three moves
// multiply to, and the 1728 sequences give only 1080 elements (1068 at distance 3, plus the 12 single moves: x x x = x^-1).
// The 16-byte part of each element is stored once per lane of a quarter-warp phase (8 copies, [element][copy], copy = lane % 8:
// conflict-free LDS.128); a remap indexed like g_macro3 gives {twist|flip word, element}.  Entries past the 1728 valid indices
// (4-bit masked invalid actions, up to kIdxMax3) point at element 0 with no twist or flip; entries kSingle3 + a (a = 0..15, the
// raw action masked to 4 bits) are the single inverse move a ^ 1 for the depth % 3 tail (a >= 12: element 0 again).
constexpr int kElems3 = 1080;
constexpr int kRepDedup = 8;
constexpr int kSingle3 = 15 + 12 * 15 + 144 * 15 + 1;          // 2356 = kIdxMax3 + 1
constexpr int kRemap3 = kSingle3 + 16;                          // 2372
constexpr int kElemBytes3 = kElems3 * kRepDedup * 16;           // 138,240
constexpr int kImageBytes3 = kElemBytes3 + kRemap3 * 8;          // 157,216: staged with one bulk copy (multiple of 16)
__device__ __align__(16) uint32_t g_macro3_image[kImageBytes3 / 4];       // Host::image3

struct Host {
	uint32_t rows[kRows * kRowWords + 3];
	uint32_t rows3[kRows3 * kRowWords + 3];
	uint32_t rows3_inv[kRows3 * kRowWords + 3];          // rows3 re-indexed by the inverse actions (device layout of g_macro3)
	uint32_t rows_inv[kRows * kRowWords + 3];             // rows re-indexed likewise (identity 12 stays 12): g_macro_tail_inv
	uint32_t elems3[kElems3 * 4];                         // distinct 16-byte parts of rows3_inv
	uint32_t remap3[kRemap3 * 2];                         // {twist|flip word, element index}, indexed like rows3_inv, then kSingle3 + a
	uint32_t image3[kImageBytes3 / 4];                    // shared-memory image of the deduplicated table (8 copies | remap)
	bool ok;
};

static const Host& host() {
	static Host h;
	static std::once_flag once;
	std::call_once(once, [] {
		memset(&h, 0, sizeof(h));
		const rbt::Tables& t = rbt::host();
		Elem s[kA];
		h.ok = true;
		for (int a = 0; a < kA; ++a) h.ok = single(t, a, s[a]) && h.ok;
		for (int a1 = 0; a1 < kA; ++a1)
			for (int a0 = 0; a0 < kA; ++a0) {
				Elem x;
				compose(s[a0], s[a1], x);
				encode(x, h.rows + (a0 + kA * a1) * kRowWords);
				if (a0 < 12 && a1 < 12)
					for (int a2 = 0; a2 < 12; ++a2) {
						Elem y;
						compose(x, s[a2], y);
						encode(y, h.rows3 + (a0 + 12 * a1 + 144 * a2) * kRowWords);
					}
			}
		auto inv = [](int a) { return a < 12 ? a ^ 1 : a; };
		for (int i = 0; i < kRows3; ++i) {
			const int j = inv(i % 12) + 12 * inv(i / 12 % 12) + 144 * inv(i / 144);
			memcpy(h.rows3_inv + i * kRowWords, h.rows3 + j * kRowWords, sizeof(uint32_t) * kRowWords);
		}
		for (int i = 0; i < kRows; ++i) {
			const int j = inv(i % kA) + kA * inv(i / kA);
			memcpy(h.rows_inv + i * kRowWords, h.rows + j * kRowWords, sizeof(uint32_t) * kRowWords);
		}

		std::map<std::array<uint32_t, 4>, uint32_t> elem;
		auto element_of = [&](const uint32_t* r) {                        // index of r's 16-byte part, appended when new
			const std::array<uint32_t, 4> key{r[0], r[1], r[2], r[3]};
			auto it = elem.find(key);
			if (it != elem.end()) return it->second;
			const uint32_t e = (uint32_t)elem.size();
			if (e < (uint32_t)kElems3) memcpy(h.elems3 + 4 * e, r, 16);
			elem.emplace(key, e);
			return e;
		};
		for (int i = 0; i < kRows3; ++i) {
			const uint32_t* r = h.rows3_inv + i * kRowWords;
			h.remap3[2 * i] = r[4];
			h.remap3[2 * i + 1] = element_of(r);
		}
		for (int a = 0; a < 12; ++a) {
			uint32_t r[kRowWords];
			encode(s[a ^ 1], r);
			h.remap3[2 * (kSingle3 + a)] = r[4];
			h.remap3[2 * (kSingle3 + a) + 1] = element_of(r);
		}
		h.ok = h.ok && elem.size() == (size_t)kElems3;
		// every index the kernel can form reproduces the row it stands for, word for word
		auto same = [&](int i, const uint32_t* r) {
			const uint32_t e = h.remap3[2 * i + 1];
			return e < (uint32_t)kElems3 && memcmp(h.elems3 + 4 * e, r, 16) == 0 && h.remap3[2 * i] == r[4];
		};
		for (int i = 0; i < kRows3; ++i) h.ok = h.ok && same(i, h.rows3_inv + i * kRowWords);
		for (int a = 0; a < 12; ++a) h.ok = h.ok && same(kSingle3 + a, h.rows_inv + (a + kA * 12) * kRowWords);
		for (int e = 0; e < kElems3; ++e)
			for (int c = 0; c < kRepDedup; ++c) memcpy(h.image3 + (e * kRepDedup + c) * 4, h.elems3 + 4 * e, 16);
		memcpy(h.image3 + kElemBytes3 / 4, h.remap3, sizeof(h.remap3));
	});
	return h;
}

// ---- device side ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
	asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
	asm volatile(
		"{\n\t"
		".reg .pred p;\n\t"
		"WAIT_%=:\n\t"
		"mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
		"@p bra DONE_%=;\n\t"
		"bra WAIT_%=;\n\t"
		"DONE_%=:\n\t"
		"}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// 1-D bulk async copy global -> shared (TMA engine; SASS UBLKCP), completion counted in bytes on `bar`.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
	             "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
	             : "memory");
}

// 2-D tensor copy global -> shared (TMA; SASS UTMALDG): box {32 cubes, h moves} of the move-major action array at (x = first
// cube, y = first move), written row by row (32 bytes per move), completion counted in bytes on `bar`.
__device__ __forceinline__ void tma_2d_g2s(void* dst_smem, const CUtensorMap* map, int32_t x, int32_t y, uint64_t* bar) {
	asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(smem_u32(dst_smem)),
	             "l"(map), "r"(x), "r"(y), "r"(smem_u32(bar))
	             : "memory");
}

struct Slots {
	uint32_t C0, C1, E0, E1, E2;
};

// PRMT straight from PTX: __byte_perm() masks the selector with 0x7777 first (one extra LOP3 per permute); the table's
// selector nibbles are always < 8, so the mask is dead weight on the ALU pipe that bounds this kernel.
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
	uint32_t r;
	asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(sel));
	return r;
}
// x >> k on the FMA pipe (IMAD.HI by 2^(32-k)) instead of SHF on the ALU pipe.
template <int k>
__device__ __forceinline__ uint32_t shr_fma(uint32_t x) {
	uint32_t r;
	asm("mul.hi.u32 %0, %1, %2;" : "=r"(r) : "r"(x), "r"(1u << (32 - k)));
	return r;
}

// x >> 16 as a 2-way dot product (IDP.2A: x.hi16 * 1 + x.lo16 * 0): half the pipe time of the quarter-rate IMAD.HI
__device__ __forceinline__ uint32_t shr16(uint32_t x) {
	uint32_t r;
	asm("dp2a.hi.u32.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(x), "r"(0x01000000u), "r"(0u));
	return r;
}

// One table row applied to the slot-major state.  p1 = {corner selectors, edge selectors 0..2}, tf = twists | flips.
__device__ __forceinline__ void apply_row(const uint4 p1, const uint32_t tf, Slots& s) {
	const uint32_t tf2 = shr_fma<2>(tf);
	const uint32_t c0 = prmt(s.C0, s.C1, p1.x), c1 = prmt(s.C0, s.C1, shr16(p1.x));
	s.C0 = c0 + (tf & 0x03030303u);
	s.C1 = c1 + (tf2 & 0x03030303u);
	const uint32_t x0 = prmt(s.E0, s.E1, p1.y), x1 = prmt(s.E0, s.E1, p1.z), x2 = prmt(s.E0, s.E1, p1.w);
	const uint32_t e0 = prmt(x0, s.E2, shr16(p1.y)), e1 = prmt(x1, s.E2, shr16(p1.z)), e2 = prmt(x2, s.E2, shr16(p1.w));
	s.E0 = e0 ^ (tf & 0x10101010u);                  // three partial flip bits per edge byte (4, 5, 6): no shifts needed,
	s.E1 = e1 ^ (tf & 0x20202020u);                  // the flip is their parity (bytes wander between E0, E1, E2)
	s.E2 = e2 ^ (tf & 0x40404040u);
}

// Table offset of row `idx` for this lane: idx * 128 + off (one IMAD, FMA pipe).
__device__ __forceinline__ uint32_t row_offset(uint32_t idx, uint32_t off) {
	uint32_t o;
	asm("mad.lo.u32 %0, %1, 128, %2;" : "=r"(o) : "r"(idx), "r"(off));
	return o;
}

// Row at byte offset `o1` (16-byte part, this lane's bank group) / `o1 + d2` (4-byte part, this lane's bank).
__device__ __forceinline__ void apply_at(const uint8_t* table, uint32_t o1, uint32_t d2, Slots& s) {
	apply_row(*reinterpret_cast<const uint4*>(table + o1), *reinterpret_cast<const uint32_t*>(table + o1 + d2), s);
}

__device__ __forceinline__ void fill_table(uint8_t* table, const uint32_t* g_rows) {
	for (int i = threadIdx.x; i < kDevRows * 32; i += blockDim.x) {
		const int row = i >> 5, c = i & 31;
		const uint32_t* r = g_rows + (row < kRows ? row : kRows - 1) * kRowWords;          // last row = (12, 12) = identity
		if (c < 8) *reinterpret_cast<uint4*>(table + (row * 8 + c) * 16) = make_uint4(r[0], r[1], r[2], r[3]);
		*reinterpret_cast<uint32_t*>(table + kP1Bytes + (row * 32 + c) * 4) = r[4];
	}
}

// One base-4 digit fold of every twist accumulator (bits 0-4 of a corner byte): value mod 3 unchanged (4 == 1 mod 3),
// any accumulator <= 31 becomes <= 3 + 7 = 10.  Between folds kReduceEvery rows add at most 2 each: 10 + 2 * 10 <= 31.
__device__ __forceinline__ uint32_t fold_twists(uint32_t c) {
	// acc = 4 q + r  ->  q + r = acc - 3 q, per byte, without touching the id bits: one shift (IMAD.HI) and one multiply-add on
	// the FMA pipe, one LOP3 on the ALU pipe (the masked form (c & 0xe0..) | ((c & 3..) + (c >> 2 & 7..)) costs three)
	const uint32_t q = shr_fma<2>(c) & 0x07070707u;
	uint32_t r;
	asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(q), "r"(0xfffffffdu), "r"(c));
	return r;
}

// Slot-major -> the reference's cubie-major int8[20] (written to this thread's 20-byte row in shared memory).
__device__ __forceinline__ void store_state(uint8_t* __restrict__ o, const Slots& s) {
#pragma unroll
	for (int q = 0; q < 8; ++q) {
		const uint32_t b = ((q < 4 ? s.C0 : s.C1) >> (8 * (q & 3))) & 0xffu;
		const uint32_t acc = b & 31u, t = acc - 3u * ((acc * 11u) >> 5);          // acc % 3 for acc < 32
		const bool neg = q == 0 || q == 2 || q == 5 || q == 7;
		const uint32_t ori = neg ? (t ? 3u - t : 0u) : t;
		o[b >> 5] = (uint8_t)(3 * q + ori);
	}
#pragma unroll
	for (int q = 0; q < 12; ++q) {
		const uint32_t b = ((q < 4 ? s.E0 : (q < 8 ? s.E1 : s.E2)) >> (8 * (q & 3))) & 0xffu;
		o[8 + (b & 15u)] = (uint8_t)(2 * q + (__popc(b & 0x70u) & 1u));
	}
}

// Work unit = chunk of 32 consecutive cubes = one warp.  Dynamic shared memory: [macro table | one mbarrier per warp |
// one action buffer (32 * depth bytes) per warp].  Each warp streams its own chunks: lane 0 starts the bulk copy of the
// warp's next chunk as soon as the warp has copied the previous result out, so a warp waits for HBM only once per chunk
// while the other ~35 resident warps of the SM keep both math pipes busy -- no block-wide barrier after start-up, and
// one buffer per warp (100 B per thread) leaves room for 40 warps per SM instead of 24 with block-wide double buffering.
// The finished state overwrites the first 20 bytes of the thread's own (consumed) action row.
template <bool kWordAligned>
__global__ void __launch_bounds__(kMaxThreads, 1)
k_scramble_macro(const uint8_t* __restrict__ actions, int8_t* __restrict__ out, int64_t n, int depth, int out_pitch) {
	extern __shared__ __align__(128) uint8_t smem[];
	uint8_t* table = smem;
	uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kTableBytes);
	const uint32_t lane = threadIdx.x & 31, wib = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
	const int chunk_bytes = 32 * depth;                       // multiple of 32: every chunk base stays 16-byte aligned
	uint8_t* buf = smem + kTableBytes + kMaxThreads / 32 * 8 + (size_t)wib * chunk_bytes;
	uint64_t* bar = &bars[wib];
	const uint32_t lane_off = (lane & 7u) * 16u, d2 = (uint32_t)kP1Bytes + lane * 4u - lane_off;

	const int64_t n_chunks = (n + 31) / 32;
	const int64_t stride = (int64_t)gridDim.x * n_warps;
	int64_t chunk = (int64_t)blockIdx.x * n_warps + wib;       // a CTA's warps take consecutive chunks: one contiguous span per round

	auto issue = [&](int64_t c) {                             // lane 0: start the bulk copy of chunk c into this warp's buffer
		const int cnt = (int)min((int64_t)32, n - c * 32);
		const uint32_t bulk = (uint32_t)(cnt * depth) & ~15u;
		if (bulk) {
			mbar_expect_tx(bar, bulk);
			bulk_g2s(buf, actions + c * chunk_bytes, bulk, bar);
		}
	};
	if (lane == 0) mbar_init(bar, 1);
	asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
	__syncwarp();
	if (lane == 0 && chunk < n_chunks) issue(chunk);
	fill_table(table, g_macro);
	__syncthreads();

	uint32_t parity = 0;
	for (; chunk < n_chunks; chunk += stride) {
		const int cnt = (int)min((int64_t)32, n - chunk * 32);
		const int bytes = cnt * depth, bulk = bytes & ~15;
		if (bulk < bytes) {                                            // ragged last chunk: < 16 trailing bytes by hand
			if ((int)lane < bytes - bulk) buf[bulk + lane] = actions[chunk * chunk_bytes + bulk + lane];
			__syncwarp();
		}
		if (bulk) { mbar_wait(bar, parity); parity ^= 1u; }

		if ((int)lane < cnt) {
			uint8_t* row = buf + lane * depth;
			Slots s{0x60402000u, 0xe0c0a080u, 0x03020100u, 0x07060504u, 0x0b0a0908u};
			// 4 moves = 1 action word = 2 table rows.  Groups of 5 words are fully unrolled (immediate offsets, no loop
			// bookkeeping on the ALU pipe that bounds this kernel) and end with the twist fold: 10 rows add at most 20.
			auto word_at = [&](int m) -> uint32_t {
				if (kWordAligned) return *reinterpret_cast<const uint32_t*>(row + m);
				return row[m] | (row[m + 1] << 8) | (row[m + 2] << 16) | ((uint32_t)row[m + 3] << 24);
			};
			auto apply_word = [&](uint32_t w) {
				w &= 0x0f0f0f0fu;                                       // any byte stays inside the 256-row table (valid input: 0..11)
				apply_at(table, row_offset(__dp4a(w, 0x00000D01u, 0u), lane_off), d2, s);
				apply_at(table, row_offset(__dp4a(w, 0x0D010000u, 0u), lane_off), d2, s);
			};
			int m = 0;
			for (; m + 20 <= depth; m += 20) {
				const uint32_t w0 = word_at(m), w1 = word_at(m + 4), w2 = word_at(m + 8), w3 = word_at(m + 12), w4 = word_at(m + 16);
				apply_word(w0); apply_word(w1); apply_word(w2); apply_word(w3); apply_word(w4);
				s.C0 = fold_twists(s.C0); s.C1 = fold_twists(s.C1);
			}
			if (m < depth) {
				for (; m + 4 <= depth; m += 4) apply_word(word_at(m));     // at most 4 words = 8 rows
				s.C0 = fold_twists(s.C0); s.C1 = fold_twists(s.C1);
				for (; m < depth; m += 2) {                                // up to 3 trailing moves, identity padded
					const uint32_t a0 = row[m], a1 = m + 1 < depth ? row[m + 1] : 12u;
					apply_at(table, row_offset((a0 & 15u) + 13u * (a1 & 15u), lane_off), d2, s);
				}
			}
			store_state(row, s);                                       // depth >= 20: the row is consumed, reuse its head
		}
		__syncwarp();
		// copy out: word k of cube c sits at buf + c*depth + 4k; consecutive lanes write consecutive global words
		{
			// out_pitch = 20 for the 20x24 output; 288 when the state is parked at the head of a 6x8x6 row (rb686 render)
			uint8_t* dst = reinterpret_cast<uint8_t*>(out) + chunk * 32 * out_pitch;
			if (kWordAligned && (reinterpret_cast<uintptr_t>(out) & 3u) == 0) {
				for (int i = lane; i < cnt * 5; i += 32) {
					const int c = i / 5, k = i - 5 * c;
					*reinterpret_cast<uint32_t*>(dst + c * out_pitch + 4 * k) = *reinterpret_cast<const uint32_t*>(buf + c * depth + 4 * k);
				}
			} else {
				for (int i = lane; i < cnt * 20; i += 32) {
					const int c = i / 20, k = i - 20 * c;
					dst[c * out_pitch + k] = buf[c * depth + k];
				}
			}
		}
		// generic-proxy writes (store_state) and reads of the buffer are ordered before the async-proxy refill
		asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
		__syncwarp();
		if (lane == 0 && chunk + stride < n_chunks) issue(chunk + stride);
	}
}

// ---- 3-move rows --------------------------------------------------------------------------------------------------------
// Same state, same row format, but one row = three consecutive moves (12^3 = 1728 rows): a third fewer PRMT / LOP3 / IMAD
// per move on the math pipes that bound the 2-move kernel.  The price is the table: 8 conflict-free copies of the 16-byte
// part would need 221 KB, so it is kept in kRep1 = 4 copies laid out row-major [row][copy] -- copy k = lane % 4 lives in
// bank groups {k, k + 4}, so within one quarter-warp phase of the LDS.128 only the two lanes that share a copy can collide
// (when their rows have the same parity): ~1.9 wavefronts per phase instead of 2.6 for an unreplicated table.  The 4-byte
// twist|flip word comes from a second array, one per row.  Trailing depth % 3 moves use the 2-move table (one copy).
// Where the action buffers leave room for it, the deduplicated table (Host::image3, kDedup) replaces both arrays: 8 copies fit
// for 1080 elements, and the depth % 3 moves are single-move rows of the same table.
// Action bytes are masked to 4 bits, so an out-of-range action forms a row index <= kIdxMax3 that still lies inside the
// CTA's shared memory (the launch always requests at least that much): an unspecified but memory-safe result.
constexpr int kRep1 = 4;
constexpr int kIdxMax3 = 15 + 12 * 15 + 144 * 15;           // 2355
constexpr int kP1Bytes3 = kRows3 * kRep1 * 16;              // 110,592
constexpr int kP2Rows3 = 2368;                              // > kIdxMax3
constexpr int kP2Bytes3 = kP2Rows3 * 4;                     // one twist|flip word per row
constexpr int kTailBytes = kDevRows * 32;                   // 2-move rows padded to 32 bytes, one copy
constexpr int kTableBytes3 = kP1Bytes3 + kP2Bytes3 + kTailBytes;      // the 4-copy table: [P1 | P2 | tail]
constexpr int kMinSmem3 = (kIdxMax3 + 1) * kRep1 * 16 + 128;

__device__ __forceinline__ uint32_t mad_u32(uint32_t a, uint32_t b, uint32_t c) {
	uint32_t o;
	asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(o) : "r"(a), "r"(b), "r"(c));
	return o;
}

// Shared-memory loads by 32-bit shared-space address (no generic-to-shared base add per row).
__device__ __forceinline__ uint4 lds128(uint32_t a) {
	uint4 v;
	asm("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
	return v;
}
__device__ __forceinline__ uint32_t lds32(uint32_t a) {
	uint32_t v;
	asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
	return v;
}
__device__ __forceinline__ uint2 lds64(uint32_t a) {
	uint2 v;
	asm("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
	return v;
}

// The 4-copy table, staged by the whole CTA (the caller synchronises): kRep1 copies of each row's 16-byte part, the rows'
// twist|flip words (zero up to kP2Rows3), then the 2-move rows for the depth % 3 moves.
__device__ __forceinline__ void stage_table3(uint8_t* table) {
	for (int i = threadIdx.x; i < kP2Rows3 * kRep1; i += blockDim.x) {
		const int row = i / kRep1, c = i % kRep1;
		if (row < kRows3) {
			const uint32_t* r = g_macro3 + row * kRowWords;
			*reinterpret_cast<uint4*>(table + (row * kRep1 + c) * 16) = make_uint4(r[0], r[1], r[2], r[3]);
			if (c == 0) *reinterpret_cast<uint32_t*>(table + kP1Bytes3 + row * 4) = r[4];
		} else if (c == 0) {
			*reinterpret_cast<uint32_t*>(table + kP1Bytes3 + row * 4) = 0u;
		}
	}
	uint8_t* tail = table + kP1Bytes3 + kP2Bytes3;
	for (int i = threadIdx.x; i < kDevRows; i += blockDim.x) {
		const uint32_t* r = g_macro_tail_inv + (i < kRows ? i : kRows - 1) * kRowWords;
		*reinterpret_cast<uint4*>(tail + i * 32) = make_uint4(r[0], r[1], r[2], r[3]);
		*reinterpret_cast<uint32_t*>(tail + i * 32 + 16) = r[4];
	}
}

__device__ __forceinline__ void fold(Slots& s) { s.C0 = fold_twists(s.C0); s.C1 = fold_twists(s.C1); }

// The row primitives of the 3-move kernels on one lane's view of the table at `table` (the 4-copy table, or kDedup: the
// deduplicated one).  p1_stride / p2_stride arrive as kernel arguments: see k_scramble_macro3.
// The kernels multiply the INVERSE moves in REVERSE order: the slot-major product is then the inverse group element, whose
// byte q holds the position (and minus the twist) of CUBIE q -- the reference's cubie-major state up to a per-byte formula,
// so the result needs no scatter by cubie id (20 conflicting STS.U8 per cube otherwise).  The inversion a ^ 1 is folded into
// the tables' layout, the action bytes are only masked to 4 bits; the row index a0 + 12 a1 + 144 a2 (a0 = the later move) is
// one or two dp4a.
template <bool kDedup>
struct Rows3 {
	uint32_t off1, off2, tail, p1_stride, p2_stride;

	__device__ __forceinline__ Rows3(const uint8_t* table, uint32_t lane, uint32_t p1, uint32_t p2)
		: off1(smem_u32(table) + (lane & ((kDedup ? kRepDedup : kRep1) - 1)) * 16u),
		  off2(smem_u32(table) + (kDedup ? (uint32_t)kElemBytes3 : (uint32_t)kP1Bytes3)),
		  tail(smem_u32(table + kP1Bytes3 + kP2Bytes3)), p1_stride(p1), p2_stride(p2) {}

	__device__ __forceinline__ void apply3(Slots& s, uint32_t r) const {
		if (kDedup) {
			const uint2 e = lds64(mad_u32(r, p2_stride, off2));                 // {twist|flip, element}
			apply_row(lds128(mad_u32(e.y, p1_stride, off1)), e.x, s);
		} else {
			const uint32_t o1 = mad_u32(r, 16u * kRep1, off1), o2 = mad_u32(r, p2_stride, off2);
			apply_row(lds128(o1), lds32(o2), s);
		}
	}
	// kDedup: the single inverse move a ^ 1 (a masked to 4 bits)
	__device__ __forceinline__ void apply1(Slots& s, uint32_t a) const { apply3(s, (uint32_t)kSingle3 + a); }
	// 4-copy table: a 2-move row (the second move may be the identity, 12)
	__device__ __forceinline__ void apply_tail(Slots& s, uint32_t idx2) const {
		const uint32_t r = tail + idx2 * 32u;
		apply_row(lds128(r), lds32(r + 16u), s);
	}
	// 12 moves = 3 action words = 4 rows, last move first
	__device__ __forceinline__ void apply_words(Slots& s, uint32_t w0, uint32_t w1, uint32_t w2) const {
		w0 &= 0x0f0f0f0fu; w1 &= 0x0f0f0f0fu; w2 &= 0x0f0f0f0fu;
		apply3(s, __dp4a(w2, 0x010C9000u, 0u));
		apply3(s, __dp4a(w2, 0x00000001u, __dp4a(w1, 0x0C900000u, 0u)));
		apply3(s, __dp4a(w1, 0x0000010Cu, __dp4a(w0, 0x90000000u, 0u)));
		apply3(s, __dp4a(w0, 0x00010C90u, 0u));
	}
	// 8 moves, bytes 7..0: (7,6,5) (4,3,2) then the pair (1,0)
	__device__ __forceinline__ void rem8(Slots& s, uint32_t wa, uint32_t wb) const {
		wa &= 0x0f0f0f0fu; wb &= 0x0f0f0f0fu;
		apply3(s, __dp4a(wb, 0x010C9000u, 0u));
		apply3(s, __dp4a(wb, 0x00000001u, __dp4a(wa, 0x0C900000u, 0u)));
		if (kDedup) { apply1(s, (wa >> 8) & 0xffu); apply1(s, wa & 0xffu); }
		else apply_tail(s, __dp4a(wa, 0x0000010Du, 0u));
	}
	// 4 moves, bytes 3..0: (3,2,1) then the single move 0
	__device__ __forceinline__ void rem4(Slots& s, uint32_t wa) const {
		wa &= 0x0f0f0f0fu;
		apply3(s, __dp4a(wa, 0x010C9000u, 0u));
		if (kDedup) apply1(s, wa & 0xffu);
		else apply_tail(s, (wa & 0xffu) + 13u * 12u);
	}
	// 24 moves: 8 rows add at most 16 to a twist accumulator <= 10
	__device__ __forceinline__ void group24(Slots& s, uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3, uint32_t w4, uint32_t w5) const {
		apply_words(s, w3, w4, w5); apply_words(s, w0, w1, w2);
		fold(s);
	}
};

// The whole sequence from word loads: word_at(m) = action bytes m .. m+3 (m % 4 == 0), inv_at(m) = action byte m masked to 4 bits
// (the tables are indexed by the raw action).  The depth % 24 moves at the end of the sequence come first -- at most 4 + 3 + 1
// rows, 8 byte-fetched rows when !kWords (depth % 4 != 0) -- then 24-move groups from the end, two (48 moves) per loop trip:
// half the loop bookkeeping.
template <bool kWords, bool kDedup, class WordAt, class InvAt>
__device__ __forceinline__ void walk3(const Rows3<kDedup>& t, Slots& s, int depth, WordAt word_at, InvAt inv_at) {
	const int M = depth - depth % 24;
	int pos = depth;
	if (pos > M) {
		if (kWords) {                                               // 4, 8, ..., 20 moves: whole words, indices by dp4a
			if (pos - 12 >= M) { t.apply_words(s, word_at(pos - 12), word_at(pos - 8), word_at(pos - 4)); pos -= 12; }
			if (pos - 8 >= M) t.rem8(s, word_at(pos - 8), word_at(pos - 4));
			else if (pos - 4 >= M) t.rem4(s, word_at(pos - 4));
		} else {
			for (; pos - 3 >= M; pos -= 3) t.apply3(s, inv_at(pos - 1) + 12u * inv_at(pos - 2) + 144u * inv_at(pos - 3));
			if (kDedup) {
				for (; pos > M; --pos) t.apply1(s, inv_at(pos - 1));
			} else if (pos > M) {
				t.apply_tail(s, inv_at(pos - 1) + 13u * (pos - 2 >= M ? inv_at(pos - 2) : 12u));
			}
		}
		fold(s);
	}
	auto group24 = [&](int m) { t.group24(s, word_at(m), word_at(m + 4), word_at(m + 8), word_at(m + 12), word_at(m + 16), word_at(m + 20)); };
	int m = M - 24;
	for (; m >= 24; m -= 48) { group24(m); group24(m - 24); }
	if (m >= 0) group24(m);
}

// Writes the packed [cube][20] results of cnt <= kCubes cubes starting at cube `first`: thread tid holds words tid + kCubes * t
// of the span in w[t].  out_pitch = 20: contiguous in HBM; 288: each state parked at the head of a 6x8x6 row for the rb686
// render; bytes where out or the pitch is not word aligned.
template <int kCubes>
__device__ __forceinline__ void store_results(int8_t* out, int64_t first, int out_pitch, int cnt, uint32_t tid, const uint32_t (&w)[5]) {
	uint8_t* dst = reinterpret_cast<uint8_t*>(out) + first * out_pitch;
	if (out_pitch == 20 && (reinterpret_cast<uintptr_t>(out) & 3u) == 0) {
#pragma unroll
		for (int t = 0; t < 5; ++t) {
			const int j = (int)tid + kCubes * t;
			if (j < cnt * 5) reinterpret_cast<uint32_t*>(dst)[j] = w[t];
		}
	} else if ((reinterpret_cast<uintptr_t>(out) & 3u) == 0 && (out_pitch & 3) == 0) {
#pragma unroll
		for (int t = 0; t < 5; ++t) {
			const int j = (int)tid + kCubes * t, c = j / 5, k = j - 5 * c;
			if (j < cnt * 5) *reinterpret_cast<uint32_t*>(dst + c * out_pitch + 4 * k) = w[t];
		}
	} else {
#pragma unroll
		for (int t = 0; t < 5; ++t) {
			const int j = (int)tid + kCubes * t, c = j / 5, k = j - 5 * c;
			if (j < cnt * 5)
				for (int q = 0; q < 4; ++q) dst[c * out_pitch + 4 * k + q] = (uint8_t)(w[t] >> (8 * q));
		}
	}
}

// Per byte: twist accumulator (bits 0-4) -> its value mod 3, by base-4 digit folds (4 == 1 mod 3); other bits ignored.
// The accumulators have just been folded (<= 10, fits 4 bits): two digit folds suffice.
__device__ __forceinline__ uint32_t mod3_bytes_folded(uint32_t c) {
	uint32_t t = (c & 0x03030303u) + ((c >> 2) & 0x03030303u);       // <= 3 + 2
	t = (t & 0x03030303u) + ((t >> 2) & 0x01010101u);                 // 0..3, 3 == 0
	const uint32_t x = t & (t >> 1) & 0x01010101u;
	return t ^ (x * 3u);
}

// Inverse-element form (see Rows3): byte q of the slot-major registers describes CUBIE q -- id field = its position, twist
// accumulator = minus its twist, flip bits = its flip.  Per byte: corner value 3 * pos + ori with ori = acc mod 3 where the
// position has negative chirality (0, 2, 5, 7: bit 0 == bit 2), its negation elsewhere; edge value 2 * pos + flip.  The five
// words are the reference's int8[20] state.
__device__ __forceinline__ void cubie_major(const Slots& s, uint32_t (&w)[5]) {
#pragma unroll
	for (int h = 0; h < 2; ++h) {
		const uint32_t c = h ? s.C1 : s.C0;
		const uint32_t t = mod3_bytes_folded(c);
		const uint32_t sw = ((t << 1) & 0x02020202u) | ((t >> 1) & 0x01010101u);        // 1 <-> 2: minus t mod 3
		const uint32_t p = (c >> 5) & 0x07070707u;
		const uint32_t neg = (((p ^ (p >> 2)) & 0x01010101u) ^ 0x01010101u) * 255u;      // 0xff where bit 0 == bit 2
		w[h] = p * 3u + ((t & neg) | (sw & ~neg));
	}
#pragma unroll
	for (int d = 0; d < 3; ++d) {
		const uint32_t e = d == 0 ? s.E0 : (d == 1 ? s.E1 : s.E2);
		const uint32_t f = ((e >> 4) ^ (e >> 5) ^ (e >> 6)) & 0x01010101u;
		w[2 + d] = ((e & 0x0f0f0f0fu) << 1) + f;
	}
}

// kMode: 0 = any depth (unaligned rows, funnel-shifted words), 1 = depth % 4 == 0 (word loads), 2 = depth % 16 == 0 (16-byte
// loads in the main loop), 3 = depth % 128 == 0 (16-byte loads from padded rows).  Separate instantiations keep the common
// mode-1 kernel (depth 100) free of the other modes' code.
// n_work <= blockDim.x / 32 warps take chunks (small n is spread over all SMs).
// kDedup: the deduplicated table (kImageBytes3, see Host::image3), staged by one bulk copy; a row is an LDS.64 of the remap
// {twist|flip, element} and an LDS.128 of the element's copy for this lane, both conflict free in the element part: 4 + ~6
// wavefronts per row against 7.75 + 3.5 for the 4-copy table, whose rows are two independent loads.  Otherwise the 4-copy
// table, staged by the whole CTA.
template <int kMode, bool kDedup>
__global__ void __launch_bounds__(kMaxThreads, 1)
k_scramble_macro3(const uint8_t* __restrict__ actions, int8_t* __restrict__ out, int64_t n, int depth, int out_pitch,
                  uint32_t p1_stride, uint32_t p2_stride, uint32_t n_work) {
	// p2_stride = 4 (8 for kDedup: the remap entry) and p1_stride = 128 (kDedup: the element stride) arrive as kernel arguments
	// so that the addresses are IMADs (FMA pipe) rather than the LEA (ALU pipe, the binding one) ptxas emits for a power-of-two
	// constant
	constexpr bool kWordAligned = kMode >= 1;
	extern __shared__ __align__(128) uint8_t smem[];
	uint8_t* table = smem;                                              // [P1 | P2 | tail | mbarriers | action buffers]
	uint64_t* tbar = reinterpret_cast<uint64_t*>(smem + kImageBytes3);  // kDedup: [elements | remap | table mbarrier | mbarriers | ...]
	uint64_t* bars = reinterpret_cast<uint64_t*>(kDedup ? smem + kImageBytes3 + 16 : smem + kTableBytes3);
	const uint32_t lane = threadIdx.x & 31, wib = threadIdx.x >> 5, n_warps = n_work;
	const int chunk_bytes = 32 * depth;
	// depth % 16 == 0: the main loop reads the action rows with 16-byte loads (a16).  depth % 128 == 0: the rows are 128 bytes
	// apart or a multiple, every lane in the same bank group (8-way conflicts even for 16-byte loads, 32-way for words); those
	// chunks are copied row by row (32 bulk copies, one per lane -- dearer than one 3200-byte copy, worth it only here) into
	// rows of pitch depth + 16, whose 16-byte stride is odd: conflict free.  Measured, 2^24 cubes: depth 64 1.00 -> 0.76 ms,
	// 96 1.08 -> 0.82 ms (16-byte loads), 128 2.91 -> 1.33 ms (padded rows).
	constexpr bool a16 = kMode >= 2, pad16 = kMode == 3;
	const int pitch = depth + (pad16 ? 16 : 0);
	uint8_t* buf = reinterpret_cast<uint8_t*>(bars) + kMaxThreads / 32 * 8 + (size_t)wib * (32 * pitch);
	uint64_t* bar = &bars[wib];
	const Rows3<kDedup> t(table, lane, p1_stride, p2_stride);

	const int64_t n_chunks = (n + 31) / 32;
	const int64_t stride = (int64_t)gridDim.x * n_warps;
	int64_t chunk = (int64_t)blockIdx.x * n_warps + wib;

	auto issue = [&](int64_t c) {                             // warp-wide: starts the bulk copy (copies) of chunk c into this warp's buffer
		if (c >= n_chunks) return;
		const int cnt = (int)min((int64_t)32, n - c * 32);
		if (pad16) {
			if (lane == 0) mbar_expect_tx(bar, (uint32_t)(cnt * depth));
			__syncwarp();
			if ((int)lane < cnt) bulk_g2s(buf + lane * pitch, actions + c * chunk_bytes + (int64_t)lane * depth, (uint32_t)depth, bar);
		} else if (lane == 0) {
			const uint32_t bulk = (uint32_t)(cnt * depth) & ~15u;
			if (bulk) {
				mbar_expect_tx(bar, bulk);
				bulk_g2s(buf, actions + c * chunk_bytes, bulk, bar);
			}
		}
	};
	if (kDedup && threadIdx.x == 0) mbar_init(tbar, 1);
	if (lane == 0) mbar_init(bar, 1);
	asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
	__syncwarp();
	if (kDedup && threadIdx.x == 0) {
		mbar_expect_tx(tbar, (uint32_t)kImageBytes3);
		bulk_g2s(table, g_macro3_image, (uint32_t)kImageBytes3, tbar);
	}
	if (wib < n_work) issue(chunk);
	if (!kDedup) stage_table3(table);
	__syncthreads();                                                    // kDedup: the table mbarrier is initialised for every warp
	if (wib >= n_work) return;
	if (kDedup) mbar_wait(tbar, 0);

	uint32_t parity = 0;
	for (; chunk < n_chunks; chunk += stride) {
		const int cnt = (int)min((int64_t)32, n - chunk * 32);
		const int bytes = cnt * depth, bulk = bytes & ~15;
		if (bulk < bytes) {
			if ((int)lane < bytes - bulk) buf[bulk + lane] = actions[chunk * chunk_bytes + bulk + lane];
			__syncwarp();
		}
		if (bulk) { mbar_wait(bar, parity); parity ^= 1u; }

		uint32_t res[5] = {0u, 0u, 0u, 0u, 0u};
		if ((int)lane < cnt) {
			uint8_t* row = buf + lane * pitch;
			Slots s{0x60402000u, 0xe0c0a080u, 0x03020100u, 0x07060504u, 0x0b0a0908u};
			// depth % 4 != 0: rows start at any byte; two aligned words and one funnel shift give the four action bytes at m
			// (m is a multiple of 4 here; the word after the row's last one may belong to the next row or to the 16 bytes of
			// slack behind the last buffer)
			const uint32_t* arow = reinterpret_cast<const uint32_t*>(buf + ((lane * depth) & ~3));
			const uint32_t ashift = ((lane * depth) & 3) * 8;
			auto word_at = [&](int m) -> uint32_t {
				if (kWordAligned) return *reinterpret_cast<const uint32_t*>(row + m);
				return __funnelshift_r(arow[m >> 2], arow[(m >> 2) + 1], ashift);
			};
			if (a16) {
				// depth % 16 == 0 (so depth % 24 is 0, 8 or 16): rows whose word stride is a multiple of 8 (depth 32, 64, 96, ...) would
				// read single words with 8- to 32-way bank conflicts, 16-byte loads cut that four-fold.  Pairs of groups are anchored at
				// multiples of 48 from the row start; what lies above them -- an odd group and / or the remainder -- is at most 40 bytes
				// starting 16-byte aligned and is taken with two or three 16-byte loads as well (the last may run 8 bytes past the row).
				const int M = depth - depth % 24;
				int m = M - 24;
				const int rem = depth - M, top = (M / 48) * 48;
				const bool odd = (M / 24) & 1;
				const uint4* q = reinterpret_cast<const uint4*>(row + top);
				if (odd) {
					const uint4 q0 = q[0], q1 = q[1];
					if (rem == 8) { t.rem8(s, q1.z, q1.w); fold(s); }
					else if (rem == 16) { const uint4 q2 = q[2]; t.apply_words(s, q1.w, q2.x, q2.y); t.rem4(s, q1.z); fold(s); }
					t.group24(s, q0.x, q0.y, q0.z, q0.w, q1.x, q1.y);
					m -= 24;
				} else if (rem) {
					const uint4 q0 = q[0];
					if (rem == 8) t.rem8(s, q0.x, q0.y);
					else { t.apply_words(s, q0.y, q0.z, q0.w); t.rem4(s, q0.x); }
					fold(s);
				}
				for (; m >= 24; m -= 48) {
					const uint4* p = reinterpret_cast<const uint4*>(row + (m - 24));
					const uint4 q0 = p[0], q1 = p[1], q2 = p[2];
					t.apply_words(s, q2.y, q2.z, q2.w); t.apply_words(s, q1.z, q1.w, q2.x);
					fold(s);
					t.apply_words(s, q0.w, q1.x, q1.y); t.apply_words(s, q0.x, q0.y, q0.z);
					fold(s);
				}
			} else {
				walk3<kWordAligned>(t, s, depth, word_at, [&](int m) -> uint32_t { return row[m] & 15u; });
			}
			cubie_major(s, res);
		}
		__syncwarp();                                                     // every lane's action row is consumed: the buffer head is free
		if ((int)lane < cnt) {
			uint32_t* dst_row = reinterpret_cast<uint32_t*>(buf + lane * 20);   // results packed [cube][20] at the head of the warp's buffer
#pragma unroll
			for (int k = 0; k < 5; ++k) dst_row[k] = res[k];
		}
		__syncwarp();
		// 32 cubes = 640 contiguous bytes in shared memory: each lane takes its five words into registers, the buffer is then
		// free for the bulk copy of the warp's next chunk, which is started BEFORE the results leave for HBM (the stores, and
		// their completion, are off the path that refills the buffer).
		uint32_t outw[5];
#pragma unroll
		for (int k = 0; k < 5; ++k) {
			const int j = lane + 32 * k;
			outw[k] = j < cnt * 5 ? reinterpret_cast<const uint32_t*>(buf)[j] : 0u;
		}
		// generic-proxy reads / writes of the buffer are ordered before the async-proxy refill
		asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
		__syncwarp();
		issue(chunk + stride);
		store_results<32>(out, chunk * 32, out_pitch, cnt, lane, outw);
	}
}

// ---- move-major actions ---------------------------------------------------------------------------------------------------------
// The reference draws its scrambles as faces / dirs of shape (depth, games) (cube.py:226-227): MOVE-major, uint8 [depth][n].
// Work unit = a span of 128 consecutive cubes = one quad of four warps.  The quad's tile is depth rows of 128 bytes fetched
// by 2-D tensor copies (TMA, box {128 cubes, <= 256 moves}; 32-byte rows -- a tile per warp -- cap the copy engine at one
// row request per ~8 clocks and cost 1.49 ms for 2^24 x 100 moves).  Shared-memory banks are the word COLUMN of the tile
// whatever the row, so the conflict-free read is a whole row per instruction: lane l takes word l of rows m .. m+3 (four
// LDS.32) and holds moves m .. m+3 of cubes 4 l .. 4 l + 3 as a 4 x 4 byte matrix; warp k of the quad transposes out column
// k (three PRMT with warp-uniform selectors) and works on cube 4 l + k.  The rest is walk3 on the 4-copy table.
constexpr int kSpan = 128;
__device__ __forceinline__ void quad_sync(uint32_t quad) {
	asm volatile("bar.sync %0, 128;" ::"r"(quad + 1u) : "memory");
}

template <bool kWords>                                   // depth % 4 == 0: the remainder is whole action words too
__global__ void __launch_bounds__(kMaxThreads, 1)
k_scramble_mm(const __grid_constant__ CUtensorMap tmap, int8_t* __restrict__ out, int64_t n, int depth, int out_pitch, uint32_t p2_stride,
              uint32_t n_quads, int box_h) {
	extern __shared__ __align__(128) uint8_t smem[];
	uint8_t* table = smem;                                              // [P1 | P2 | tail | mbarriers | one tile per quad]
	uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kTableBytes3);
	const uint32_t lane = threadIdx.x & 31, wib = threadIdx.x >> 5, quad = wib >> 2, k = wib & 3u, tq = threadIdx.x & 127u;
	const int span_bytes = kSpan * depth;
	uint8_t* tile = reinterpret_cast<uint8_t*>(bars) + kMaxThreads / 32 * 8 + (size_t)quad * span_bytes;
	uint64_t* bar = &bars[quad];
	const Rows3<false> t(table, lane, 0u, p2_stride);
	const int64_t n_spans = (n + kSpan - 1) / kSpan, stride = (int64_t)gridDim.x * n_quads;
	int64_t span = (int64_t)blockIdx.x * n_quads + quad;

	auto issue = [&](int64_t sp) {                            // one thread of the quad; cubes past n are zero filled (action 0)
		if (sp >= n_spans) return;
		mbar_expect_tx(bar, (uint32_t)span_bytes);
		for (int y = 0; y < depth; y += box_h) tma_2d_g2s(tile + y * kSpan, &tmap, (int32_t)(sp * kSpan), y, bar);
	};
	if (tq == 0) mbar_init(bar, 1);
	asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
	if (tq == 0 && quad < n_quads) issue(span);                            // the thread that initialised the barrier; the others meet it after the block barrier
	stage_table3(table);
	__syncthreads();
	if (quad >= n_quads) return;

	const uint32_t sel1 = k < 2 ? 0x5140u : 0x7362u, sel2 = (k & 1u) ? 0x7632u : 0x5410u;   // column k of a 4 x 4 byte matrix
	const uint32_t my_cube = 4u * lane + k;                                                 // within the span
	const uint32_t* tilew = reinterpret_cast<const uint32_t*>(tile);
	uint32_t parity = 0;
	for (; span < n_spans; span += stride) {
		const int cnt = (int)min((int64_t)kSpan, n - span * kSpan);
		mbar_wait(bar, parity); parity ^= 1u;

		uint32_t res[5];
		{
			Slots s{0x60402000u, 0xe0c0a080u, 0x03020100u, 0x07060504u, 0x0b0a0908u};
			auto word_at = [&](int m) -> uint32_t {                            // action bytes m .. m+3 of this lane's cube (m % 4 == 0)
				const uint32_t* p = tilew + m * 32 + (int)lane;
				const uint32_t x = prmt(p[0], p[32], sel1), y = prmt(p[64], p[96], sel1);
				return prmt(x, y, sel2);
			};
			walk3<kWords>(t, s, depth, word_at, [&](int m) -> uint32_t { return tile[m * kSpan + (int)my_cube] & 15u; });
			cubie_major(s, res);
		}
		quad_sync(quad);                                                  // the whole tile is consumed
		{
			uint32_t* dst_row = reinterpret_cast<uint32_t*>(tile + my_cube * 20);   // results packed [cube][20] at the head of the tile
#pragma unroll
			for (int j = 0; j < 5; ++j) dst_row[j] = res[j];
		}
		quad_sync(quad);
		uint32_t outw[5];
#pragma unroll
		for (int j = 0; j < 5; ++j) {
			const int i = (int)tq + kSpan * j;
			outw[j] = i < cnt * 5 ? tilew[i] : 0u;
		}
		asm volatile("fence.proxy.async.shared::cta;" ::: "memory");        // generic reads / writes of the tile before its async refill
		quad_sync(quad);
		if (tq == 0) issue(span + stride);
		store_results<kSpan>(out, span * kSpan, out_pitch, cnt, tq, outw);
	}
}

// Defined in rb_scramble_seeded.cuh; its shared-memory attribute is set with the others in ensure_device().
struct PhiloxKeys;
__global__ void k_scramble_seeded(PhiloxKeys keys, uint64_t first_cube, int8_t* __restrict__ out, int64_t n, int depth, int out_pitch,
                                  uint32_t p2_stride, uint32_t n_warps);

static int ensure_device() {
	static std::mutex mu;
	static bool done[64] = {};
	int dev = 0;
	RB_CUDA(cudaGetDevice(&dev));
	std::lock_guard<std::mutex> lock(mu);
	if (dev < 0 || dev >= 64) return rb_fail(RB_ERR_BAD_ARG, "device ordinal out of range%s%s");
	if (done[dev]) return RB_OK;
	const Host& h = host();
	if (!h.ok) return rb_fail(RB_ERR_BAD_ARG, "macro-move tables: a host check failed (twist additivity or the deduplicated 3-move table)%s%s");
	RB_CUDA(cudaMemcpyToSymbol(g_macro, h.rows, sizeof(h.rows)));
	RB_CUDA(cudaMemcpyToSymbol(g_macro3, h.rows3_inv, sizeof(h.rows3_inv)));
	RB_CUDA(cudaMemcpyToSymbol(g_macro_tail_inv, h.rows_inv, sizeof(h.rows_inv)));
	RB_CUDA(cudaMemcpyToSymbol(g_macro3_image, h.image3, sizeof(h.image3)));
	RB_CUDA(cudaFuncSetAttribute(k_scramble_macro3<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget));
	RB_CUDA(cudaFuncSetAttribute(k_scramble_macro3<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget));
	RB_CUDA(cudaFuncSetAttribute(k_scramble_macro3<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget));
	RB_CUDA(cudaFuncSetAttribute(k_scramble_macro3<3, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget));
	RB_CUDA(cudaFuncSetAttribute(k_scramble_macro3<0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget));
	RB_CUDA(cudaFuncSetAttribute(k_scramble_macro3<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget));
	RB_CUDA(cudaFuncSetAttribute(k_scramble_macro3<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget));
	RB_CUDA(cudaFuncSetAttribute(k_scramble_macro3<3, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget));
	RB_CUDA(cudaFuncSetAttribute(k_scramble_mm<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget));
	RB_CUDA(cudaFuncSetAttribute(k_scramble_mm<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget));
	RB_CUDA(cudaFuncSetAttribute(k_scramble_macro<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget));
	RB_CUDA(cudaFuncSetAttribute(k_scramble_macro<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget));
	RB_CUDA(cudaFuncSetAttribute(k_scramble_seeded, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget));
	done[dev] = true;
	return RB_OK;
}

constexpr int64_t kFixedSmem = kTableBytes + kMaxThreads / 32 * 8;        // table + one mbarrier per warp

// Warps per CTA (one 32-cube chunk buffer each) for a given depth, 0 when the fast path does not apply.
static int warps_for(int64_t n, int depth) {
	if (depth < 20) return 0;                   // the result is written over the head of the 20+ byte action row
	int64_t w = (kSmemBudget - 1024 - kFixedSmem) / (32 * (int64_t)depth);
	if (w > kMaxThreads / 32) w = kMaxThreads / 32;
	const int64_t spread = ((n + 31) / 32 + RB_NUM_SMS - 1) / RB_NUM_SMS;      // small n: use every SM
	if (w > spread) w = spread;
	return (int)w;
}

// 3-move kernels: fixed shared memory (4-copy table + one mbarrier per warp) and warps per CTA for a given depth (0: use the
// 2-move kernel)
constexpr int64_t kFixedSmem3 = kTableBytes3 + kMaxThreads / 32 * 8;
constexpr int kStageThreads = 1024;             // threads that fill the table, whatever the number of working warps
// row pitch of the action buffers (see the kernel): depth % 128 == 0 rows are padded by 16 bytes
static int pitch3(int depth) { return depth % 128 == 0 ? depth + 16 : depth; }
constexpr int64_t kFixedSmemDedup = kImageBytes3 + 16 + kMaxThreads / 32 * 8;   // image + table mbarrier + one per warp
// Warps per CTA that the shared memory beside the table holds (the deduplicated table: in multiples of 4 so that the four
// sub-partitions get equal shares -- 2^24 x 100 moves on B200: 23 warps 0.771 ms, 20 warps 0.757 ms).
static int64_t smem_warps3(int depth, bool dedup) {
	const int64_t w = (kSmemBudget - 16 - (dedup ? kFixedSmemDedup : kFixedSmem3)) / (32 * (int64_t)pitch3(depth));
	return dedup ? w & ~3 : w;
}
static int warps_for3(int64_t n, int depth, bool dedup) {
	if (depth < 20) return 0;
	int64_t w = smem_warps3(depth, dedup);
	if (w > kMaxThreads / 32) w = kMaxThreads / 32;
	if (w < 8) return 0;                         // long sequences: too few resident warps to hide the table latency
	const int64_t spread = ((n + 31) / 32 + RB_NUM_SMS - 1) / RB_NUM_SMS;
	if (w > spread) w = spread;
	return (int)w;
}

// cuTensorMapEncodeTiled through the runtime (no link against libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
	static EncodeTiledFn fn = [] {
		void* p = nullptr;
		cudaDriverEntryPointQueryResult q;
		if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) p = nullptr;
		return reinterpret_cast<EncodeTiledFn>(p);
	}();
	return fn;
}

// Box height of the move-major tile copies: the whole depth when it fits one box (<= 256 rows), else an even split into boxes
// whose height is a multiple of 4 rows (every box must land 128-byte aligned in shared memory); 0 = none.
static int box_height(int depth) {
	if (depth <= 256) return depth;
	for (int k = (depth + 255) / 256; k <= 16; ++k)
		if (depth % k == 0 && (depth / k) % 4 == 0) return depth / k;
	return 0;
}

// Can the move-major ([depth][n]) fast path take this call?
static bool can_transposed(const uint8_t* actions, int64_t n, int depth) {
	return depth >= 20 && n % 16 == 0 && n < (int64_t(1) << 31) && (reinterpret_cast<uintptr_t>(actions) & 15u) == 0 && box_height(depth) > 0 &&
	       encode_tiled_fn() != nullptr;
}

// quads (tiles of 128 cubes x depth bytes) per CTA for the move-major kernel; 0 = does not apply
static int quads_for(int64_t n, int depth) {
	if (depth < 20) return 0;
	int64_t q = (kSmemBudget - 16 - kFixedSmem3) / ((int64_t)kSpan * depth);
	if (q > kMaxThreads / 128) q = kMaxThreads / 128;
	if (q < 2) return 0;
	const int64_t spread = ((n + kSpan - 1) / kSpan + RB_NUM_SMS - 1) / RB_NUM_SMS;
	if (q > spread) q = spread;
	return (int)q;
}

// move-major actions uint8 [depth][n] (see can_transposed / quads_for)
static int launch_mm(const uint8_t* actions, int8_t* out, int64_t n, int depth, cudaStream_t st, int out_pitch) {
	int rc = ensure_device();
	if (rc != RB_OK) return rc;
	const int Q = quads_for(n, depth), bh = box_height(depth);
	if (Q <= 0 || bh <= 0) return rb_fail(RB_ERR_BAD_ARG, "move-major fast path does not apply%s%s");
	CUtensorMap tmap;
	const cuuint64_t gdim[2] = {(cuuint64_t)n, (cuuint64_t)depth}, gstride[1] = {(cuuint64_t)n};
	const cuuint32_t box[2] = {(cuuint32_t)kSpan, (cuuint32_t)bh}, estride[2] = {1u, 1u};
	const CUresult cr = encode_tiled_fn()(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<uint8_t*>(actions), gdim, gstride, box, estride,
	                                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
	                                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
	if (cr != CUDA_SUCCESS) return rb_fail(RB_ERR_CUDA, "cuTensorMapEncodeTiled failed for the move-major action array%s%s");
	const int64_t spans = (n + kSpan - 1) / kSpan, ctas = (spans + Q - 1) / Q;
	const int grid = (int)(ctas < RB_NUM_SMS ? ctas : RB_NUM_SMS);
	size_t smem = (size_t)kFixedSmem3 + (size_t)Q * kSpan * depth + 16;
	if (smem < (size_t)kMinSmem3) smem = kMinSmem3;
	if (depth % 4 == 0) k_scramble_mm<true><<<grid, kStageThreads, smem, st>>>(tmap, out, n, depth, out_pitch, 4u, (uint32_t)Q, bh);
	else k_scramble_mm<false><<<grid, kStageThreads, smem, st>>>(tmap, out, n, depth, out_pitch, 4u, (uint32_t)Q, bh);
	RB_LAUNCHED("scramble_mm_2024");
	return RB_OK;
}

// The 3-move kernel on W3 warps per CTA, its mode picked by the depth.
template <bool kDedup>
static int launch3(const uint8_t* actions, int8_t* out, int64_t n, int depth, cudaStream_t st, int out_pitch, int W3) {
	const int64_t ctas = ((n + 31) / 32 + W3 - 1) / W3;
	const int grid = (int)(ctas < RB_NUM_SMS ? ctas : RB_NUM_SMS);
	// the 4-copy table is staged by a full CTA however few warps have work (4096 cubes: 128 single-warp CTAs took 70 us to fill it)
	const int threads = kDedup || W3 * 32 >= kStageThreads ? W3 * 32 : kStageThreads;
	size_t smem = (size_t)(kDedup ? kFixedSmemDedup : kFixedSmem3) + (size_t)W3 * 32 * pitch3(depth) + 16;
	if (smem < (size_t)kMinSmem3) smem = kMinSmem3;
	// element / row stride and remap entry / twist|flip word stride (the 4-copy table's 16-byte stride is a constant)
	const uint32_t p1 = kDedup ? kRepDedup * 16u : 0u, p2 = kDedup ? 8u : 4u, nw = (uint32_t)W3;
	if (depth % 4 != 0) k_scramble_macro3<0, kDedup><<<grid, threads, smem, st>>>(actions, out, n, depth, out_pitch, p1, p2, nw);
	else if (depth % 128 == 0) k_scramble_macro3<3, kDedup><<<grid, threads, smem, st>>>(actions, out, n, depth, out_pitch, p1, p2, nw);
	else if (depth % 16 == 0) k_scramble_macro3<2, kDedup><<<grid, threads, smem, st>>>(actions, out, n, depth, out_pitch, p1, p2, nw);
	else k_scramble_macro3<1, kDedup><<<grid, threads, smem, st>>>(actions, out, n, depth, out_pitch, p1, p2, nw);
	RB_LAUNCHED("scramble_macro3_2024");
	return RB_OK;
}

// actions: cube-major uint8 [n][depth]
static int launch(const uint8_t* actions, int8_t* out, int64_t n, int depth, cudaStream_t st, int out_pitch) {
	int rc = ensure_device();
	if (rc != RB_OK) return rc;
	// The deduplicated table where it leaves room for at least 12 warps (pitch <= 195: every depth from 20 to 195), else the
	// 4-copy table.  2^24 cubes on B200, deduplicated / 4-copy: depth 100 (20 warps) 0.757 / 0.818 ms, 144 (16) 1.059 / 1.172,
	// 176 (12) 1.319 / 1.450; with 8 warps it loses at some depths (200: 1.737 / 1.655, 256: 2.222 / 2.170).
	const bool dedup = smem_warps3(depth, true) >= 12;
	const int W3 = warps_for3(n, depth, dedup);
	if (W3 > 0) return dedup ? launch3<true>(actions, out, n, depth, st, out_pitch, W3) : launch3<false>(actions, out, n, depth, st, out_pitch, W3);
	const int W = warps_for(n, depth);
	const int64_t ctas = ((n + 31) / 32 + W - 1) / W;
	const int grid = (int)(ctas < RB_NUM_SMS ? ctas : RB_NUM_SMS);
	const size_t smem = (size_t)kFixedSmem + (size_t)W * 32 * depth;
	if (depth % 4 == 0) k_scramble_macro<true><<<grid, W * 32, smem, st>>>(actions, out, n, depth, out_pitch);
	else k_scramble_macro<false><<<grid, W * 32, smem, st>>>(actions, out, n, depth, out_pitch);
	RB_LAUNCHED("scramble_macro_2024");
	return RB_OK;
}

}  // namespace rbs
